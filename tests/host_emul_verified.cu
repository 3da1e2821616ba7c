// tests/host_emul_verified.cu -- TEST SCAFFOLDING, never shipped.
//
// Runs the verify-then-release flavours of the engine's per-thread device code on the CPU: the tag-only pass of the
// shared-key lane code (ag_batch_lane<..., VERIFY>), the flat slot mapping of the gated GCTR pass (ag_gated_ctr_slot,
// with the offsets form's warp-level binary search) and the two-phase per-key message (ag_perkey_message<..., VERIFY>).
// The cross-thread steps the kernels do with shuffles are restated with plain loops.  Built by
// tests/test_batch_verified.py with `nvcc -x cu` (host code only).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../aes-gcm-128-192-256-bits_b200/csrc/gcm_core.cuh"
#include "../aes-gcm-128-192-256-bits_b200/csrc/perkey_core.cuh"

namespace {

struct TeHost {
    const uint32_t* te0;
    __host__ __device__ uint32_t operator()(int tab, uint32_t w, int k) const
    {
        const uint32_t t = te0[(w >> (8 * k)) & 0xff];
        return tab ? ag_rotl32(t, 8 * tab) : t;
    }
};

struct GhHost {
    const uint4* tab;
    __host__ __device__ uint4 operator()(uint32_t w, int k) const { return tab[(w >> (8 * k)) & 0xff]; }
};

struct SubWordHost {
    const uint8_t* sbox;
    __host__ __device__ uint32_t operator()(uint32_t w) const
    {
        return (uint32_t)sbox[w & 0xff] | ((uint32_t)sbox[(w >> 8) & 0xff] << 8) | ((uint32_t)sbox[(w >> 16) & 0xff] << 16) |
               ((uint32_t)sbox[w >> 24] << 24);
    }
};

struct SubCacheHost {
    uint32_t v[12];
    void put(int j, uint32_t x) { v[j] = x; }
    uint32_t get(int j) const { return v[j]; }
};

struct Rows4Host {
    uint4 r[16];
    __host__ __device__ void put(int n, uint4 v) { r[n] = v; }
    __host__ __device__ uint4 get(uint32_t w, int k) const { return r[(w >> (4 * k)) & 0xf]; }
};

gf128 gf_pow(gf128 h, uint64_t e)
{
    gf128 r = gf_one();
    while (e) {
        if (e & 1) r = gf_mul(r, h);
        h = gf_mul(h, h);
        e >>= 1;
    }
    return r;
}

void build_table(const gf128& c, std::vector<uint4>& tab)
{
    gf128 basis[8];
    basis[0] = c;
    for (int k = 1; k < 8; ++k) basis[k] = gf_mulx(basis[k - 1]);
    tab.resize(256);
    for (uint32_t b = 0; b < 256; ++b) tab[b] = gf_table_row(basis, b);
}

struct Tables {
    uint8_t sbox[256];
    uint32_t te0[256];
    Tables() { ag_build_sbox_te0(sbox, te0); }
};
const Tables& tables()
{
    static Tables t;
    return t;
}

}  // namespace

// ---- verify-then-release batch decrypt --------------------------------------------------------------------------
// Pass 1: the tag-only flavour of ag_batch_lane (G lanes per message, S segments weighted as a GHASH-only pass, the
// partials combined as in batch_nr): writes ok[] only.
template <int NR>
static void batch_verify_nr(const BatchParams& p, uint32_t G, uint32_t S, const gf128& H)
{
    std::vector<uint4> tab_g, tab_1;
    build_table(gf_pow(H, G), tab_g);
    build_table(H, tab_1);
    TeHost te{tables().te0};
    GhHost gh_g{tab_g.data()}, gh_1{tab_1.data()};
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        MsgDesc whole = ag_batch_msg(p, m);
        uint32_t iv[3];
        ag_batch_iv(p, m, iv, &whole.j0ctr);
        const AesCtrConst cc = aes_ctr_precompute(p.rk, iv[0], iv[1], iv[2], te);
        gf128 total = gf_zero();
        uint32_t e[4] = {0, 0, 0, 0};
        for (uint32_t seg = 0; seg < S; ++seg) {
            uint64_t after = 0;
            const MsgDesc d = S > 1 ? ag_batch_segment(whole, seg, S, &after, 1) : whole;
            gf128 r = gf_zero();
            AesCtrSeqCache cache;
            cache.key = 0xFFFFFFFFu;
            for (uint32_t t = 0; t < G; ++t) {
                uint32_t el[4] = {0, 0, 0, 0};
                const gf128 y = ag_batch_lane<NR, true, false, true>(p.rk, cc, cache, d, t, G, te, gh_g, el);
                if (t == G - 1 && d.last) memcpy(e, el, 16);
                r = gf_mul_table(gf_xor(r, y), gh_1);
            }
            if (after) r = gf_mul(r, gf_pow(H, after));
            total = gf_xor(total, r);
        }
        uint32_t x[4];
        ag_load_block(p.tag + 16 * m, 16, x);
        uint32_t diff = 0;
        for (int k = 0; k < 4; ++k) diff |= x[k] ^ ag_bswap32(total.w[k]) ^ e[k];
        p.ok[m] = diff ? 0 : 1;
    }
}

// Pass 2: k_batch_ctr_gated's slot mapping on a virtual grid of n_warps warps (chunks of 32 x AG_GATED_ROWS slots
// round-robin, the offsets form's warp-level binary search, every lane walking forward).
template <int NR>
static void ctr_gated_nr(const BatchParams& p, uint64_t n_slots, uint64_t bpr, uint64_t n_warps)
{
    TeHost te{tables().te0};
    if (p.in_off) n_slots = (p.in_off[p.n_msgs] - p.in_off[0] + 15) >> 4;
    const uint64_t CH = 32ull * AG_GATED_ROWS, n_chunks = (n_slots + CH - 1) / CH;
    for (uint64_t w = 0; w < n_warps; ++w)
        for (uint64_t c = w; c < n_chunks; c += n_warps) {
            const uint64_t m0 = p.in_off ? ag_gated_first_msg(p, c * CH) : 0;
            for (uint32_t lane = 0; lane < 32; ++lane) {
                uint64_t m = m0;
                for (uint32_t k = 0; k < AG_GATED_ROWS; ++k) {
                    const uint64_t s = c * CH + 32 * k + lane;
                    if (s < n_slots) ag_gated_ctr_slot<NR>(p, s, bpr, m, te);
                }
            }
        }
}

extern "C" {

// offsets (in_off) or uniform (len, stride) or slots (len_arr, stride) batch; iv_is_j0 as in BatchParams
int emul_batch_verify(const uint8_t* rk_bytes, int nr, int G, int S, const uint8_t* iv, int iv_is_j0, const uint8_t* aad,
                      const uint64_t* aad_off, uint64_t aad_len, uint64_t aad_stride, const uint8_t* in, const uint64_t* in_off,
                      uint64_t len, uint64_t stride, const uint32_t* len_arr, const uint8_t* tag, uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    p.iv = iv;
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.aad = aad;
    p.aad_off = aad_off;
    p.aad_len = aad_len;
    p.aad_stride = aad_stride;
    p.in = in;
    p.in_off = in_off;
    p.len = len;
    p.stride = stride;
    p.len_arr = len_arr;
    p.tag = const_cast<uint8_t*>(tag);
    p.ok = ok;
    p.n_msgs = n_msgs;
    const TeHost te{tables().te0};
    uint32_t h[4];
    aes_encrypt_words(p.rk, nr, 0, 0, 0, 0, te, h);
    const gf128 H = gf_from_le_words(h[0], h[1], h[2], h[3]);
    switch (nr) {
        case 10: batch_verify_nr<10>(p, G, S, H); break;
        case 12: batch_verify_nr<12>(p, G, S, H); break;
        case 14: batch_verify_nr<14>(p, G, S, H); break;
        default: return -1;
    }
    return 0;
}

int emul_batch_ctr_gated(const uint8_t* rk_bytes, int nr, const uint8_t* iv, int iv_is_j0, const uint8_t* in, const uint64_t* in_off,
                         uint64_t len, uint64_t stride, const uint32_t* len_arr, uint8_t* out, uint8_t* ok, uint64_t n_msgs,
                         uint64_t n_warps)
{
    BatchParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    p.iv = iv;
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.in = in;
    p.in_off = in_off;
    p.len = len;
    p.stride = stride;
    p.len_arr = len_arr;
    p.out = out;
    p.ok = ok;
    p.n_msgs = n_msgs;
    // as agcm_batch_decrypt_verified*: blocks per whole slot (slots form) or per record (uniform form)
    const uint64_t bpr = len_arr ? (stride + 15) >> 4 : (len + 15) >> 4;
    switch (nr) {
        case 10: ctr_gated_nr<10>(p, bpr * n_msgs, bpr, n_warps); break;
        case 12: ctr_gated_nr<12>(p, bpr * n_msgs, bpr, n_warps); break;
        case 14: ctr_gated_nr<14>(p, bpr * n_msgs, bpr, n_warps); break;
        default: return -1;
    }
    return 0;
}

// the verified flavour of the per-key message (phase 1 tag check, phase 2 GCTR only on a match)
int emul_batch_perkey_verified(const uint8_t* keys, int key_bytes, const uint8_t* iv, const uint8_t* aad, const uint64_t* aad_off,
                               const uint8_t* in, const uint64_t* in_off, uint8_t* out, const uint8_t* tag, uint8_t* ok,
                               uint64_t n_msgs)
{
    BatchParams p;
    memset(&p, 0, sizeof(p));
    p.keys = keys;
    p.iv = iv;
    p.aad = aad;
    p.aad_off = aad_off;
    p.in = in;
    p.in_off = in_off;
    p.out = out;
    p.n_msgs = n_msgs;
    TeHost te{tables().te0};
    SubWordHost sb{tables().sbox};
    const int nk = key_bytes / 4;
    if (nk != 4 && nk != 6 && nk != 8) return -1;
    for (uint64_t m = 0; m < n_msgs; ++m) {
        const MsgDesc d = ag_batch_msg(p, m);
        uint32_t key[8] = {0}, ivw[3] = {0, 0, 0}, tg[4], x[4];
        for (int j = 0; j < key_bytes; ++j) key[j >> 2] |= (uint32_t)keys[m * key_bytes + j] << (8 * (j & 3));
        for (int j = 0; j < 12; ++j) ivw[j >> 2] |= (uint32_t)iv[12 * m + j] << (8 * (j & 3));
        ag_load_block(tag + 16 * m, 16, x);
        memcpy(tg, x, 16);
        Rows4Host rows;
        SubCacheHost subc;
        if (nk == 4) ag_perkey_message<4, true, false, true>(key, ivw[0], ivw[1], ivw[2], d, te, sb, rows, subc, tg);
        if (nk == 6) ag_perkey_message<6, true, false, true>(key, ivw[0], ivw[1], ivw[2], d, te, sb, rows, subc, tg);
        if (nk == 8) ag_perkey_message<8, true, false, true>(key, ivw[0], ivw[1], ivw[2], d, te, sb, rows, subc, tg);
        ok[m] = ((x[0] ^ tg[0]) | (x[1] ^ tg[1]) | (x[2] ^ tg[2]) | (x[3] ^ tg[3])) ? 0 : 1;
    }
    return 0;
}

}  // extern "C"

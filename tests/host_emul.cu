// tests/host_emul.cu -- TEST SCAFFOLDING, never shipped.
//
// Runs the engine's per-thread device code (csrc/gcm_core.cuh, aes_core.cuh,
// gf128.cuh -- the very functions the CUDA kernels call) on the CPU, looping over
// the "threads" of a small virtual grid, so that the CPU test-suite can check the
// index arithmetic (front padding, strided Horner weights, ragged last block,
// lane combine) against the oracle without a GPU.  The cross-thread steps that
// the kernels do with shuffles / shared memory are restated here with plain
// loops.  Built by tests/conftest.py with `nvcc -x cu` (host code only).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../aes-gcm-128-192-256-bits_b200/csrc/gcm_core.cuh"
#include "../aes-gcm-128-192-256-bits_b200/csrc/perkey_core.cuh"
#include "../aes-gcm-128-192-256-bits_b200/csrc/host_sched.h"

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

gf128 gf_from_bytes(const uint8_t b[16])
{
    gf128 r;
    for (int i = 0; i < 4; ++i)
        r.w[i] = ((uint32_t)b[4 * i] << 24) | ((uint32_t)b[4 * i + 1] << 16) | ((uint32_t)b[4 * i + 2] << 8) | b[4 * i + 3];
    return r;
}

void gf_to_bytes(const gf128& v, uint8_t b[16])
{
    for (int i = 0; i < 4; ++i) {
        b[4 * i] = (uint8_t)(v.w[i] >> 24);
        b[4 * i + 1] = (uint8_t)(v.w[i] >> 16);
        b[4 * i + 2] = (uint8_t)(v.w[i] >> 8);
        b[4 * i + 3] = (uint8_t)v.w[i];
    }
}

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

template <int NR>
void stream_nr(const StreamParams& p, int mode, uint64_t ncta, uint64_t nt, const gf128& H, gf128& total)
{
    const uint32_t Gt = (uint32_t)(ncta * nt);
    std::vector<uint4> tab;
    build_table(gf_pow(H, Gt), tab);
    TeHost te{tables().te0};
    GhHost gh{tab.data()};
    total = gf_zero();
    for (uint32_t g = 0; g < Gt; ++g) {
        gf128 y;
        switch (mode) {
            case AG_MODE_ENC: y = ag_stream_lane<NR, AG_MODE_ENC, false>(p, g, Gt, te, gh); break;
            case AG_MODE_DEC: y = ag_stream_lane<NR, AG_MODE_DEC, true>(p, g, Gt, te, gh); break;
            case AG_MODE_GHASH_ONLY: y = ag_stream_lane<NR, AG_MODE_GHASH_ONLY, true>(p, g, Gt, te, gh); break;
            default: y = ag_stream_lane<NR, AG_MODE_CTR_ONLY, false>(p, g, Gt, te, gh); break;
        }
        // kernel: y *= hpow_thread[nt - tid]; CTA xor; *= hpow_cta[ncta-1-cta]
        const uint64_t cta = g / nt, tid = g % nt;
        y = gf_mul(y, gf_pow(H, nt - tid));
        y = gf_mul(y, gf_pow(gf_pow(H, nt), ncta - 1 - cta));
        total = gf_xor(total, y);
    }
}

template <int NR, bool DEC>
void batch_nr(const BatchParams& p, uint32_t G, const gf128& H, uint32_t S = 1)
{
    std::vector<uint4> tab_g, tab_1;
    build_table(gf_pow(H, G), tab_g);
    build_table(H, tab_1);
    TeHost te{tables().te0};
    GhHost gh_g{tab_g.data()}, gh_1{tab_1.data()};
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        const MsgDesc whole = ag_batch_msg(p, m);
        const uint8_t* ivp = p.iv + 12 * m;
        uint32_t iv[3] = {0, 0, 0};
        for (int j = 0; j < 12; ++j) iv[j >> 2] |= (uint32_t)ivp[j] << (8 * (j & 3));
        const AesCtrConst cc = aes_ctr_precompute(p.rk, iv[0], iv[1], iv[2], te);
        gf128 total = gf_zero();
        uint32_t e[4] = {0, 0, 0, 0};
        // S > 1: the message as S counter-range segments (k_batch_cta's split layout), each partial
        // scaled by H^after and XORed, as k_batch_split_finish does
        for (uint32_t seg = 0; seg < S; ++seg) {
            uint64_t after = 0;
            const MsgDesc d = S > 1 ? ag_batch_segment(whole, seg, S, &after) : whole;
            gf128 r = gf_zero();
            AesCtrSeqCache cache;
            cache.key = 0xFFFFFFFFu;
            for (uint32_t t = 0; t < G; ++t) {
                uint32_t el[4] = {0, 0, 0, 0};
                gf128 y = ag_batch_lane<NR, DEC>(p.rk, cc, cache, d, t, G, te, gh_g, el);
                if (t == G - 1 && d.last) { e[0] = el[0]; e[1] = el[1]; e[2] = el[2]; e[3] = el[3]; }
                r = gf_xor(r, y);
                r = gf_mul_table(r, gh_1);
            }
            if (after) r = gf_mul(r, gf_pow(H, after));
            total = gf_xor(total, r);
        }
        const gf128 r = total;
        uint32_t tg[4] = {ag_bswap32(r.w[0]) ^ e[0], ag_bswap32(r.w[1]) ^ e[1], ag_bswap32(r.w[2]) ^ e[2],
                          ag_bswap32(r.w[3]) ^ e[3]};
        uint8_t* tp = p.tag + 16 * m;
        if (DEC) {
            uint32_t x[4];
            ag_load_block(tp, 16, x);
            p.ok[m] = ((x[0] ^ tg[0]) | (x[1] ^ tg[1]) | (x[2] ^ tg[2]) | (x[3] ^ tg[3])) ? 0 : 1;
        } else {
            ag_store_block(tp, 16, tg);
        }
    }
}

template <int NK, bool DEC>
void perkey_nk(const BatchParams& p)
{
    TeHost te{tables().te0};
    SubWordHost sb{tables().sbox};
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        const MsgDesc d = ag_batch_msg(p, m);
        uint32_t key[8] = {0}, iv[3] = {0, 0, 0};
        const uint8_t* kp = p.keys + m * (uint64_t)(4 * NK);
        for (int j = 0; j < 4 * NK; ++j) key[j >> 2] |= (uint32_t)kp[j] << (8 * (j & 3));
        const uint8_t* ivp = p.iv + 12 * m;
        for (int j = 0; j < 12; ++j) iv[j >> 2] |= (uint32_t)ivp[j] << (8 * (j & 3));
        Rows4Host rows;
        SubCacheHost subc;
        uint32_t tg[4];
        ag_perkey_message<NK, DEC>(key, iv[0], iv[1], iv[2], d, te, sb, rows, subc, tg);
        uint8_t* tp = p.tag + 16 * m;
        if (DEC) {
            uint32_t x[4];
            ag_load_block(tp, 16, x);
            p.ok[m] = ((x[0] ^ tg[0]) | (x[1] ^ tg[1]) | (x[2] ^ tg[2]) | (x[3] ^ tg[3])) ? 0 : 1;
        } else {
            ag_store_block(tp, 16, tg);
        }
    }
}

}  // namespace

// k_batch_warp's BALANCED partition on a virtual grid of n_warps warps (uniform records): warp w
// owns the w-th equal share of the AAD axis and of the payload axis of the concatenated messages; every unit's 32 lane
// accumulators are combined as k_batch_warp's combine rounds do (serial Horner with H, times H^after) and
// XORed into the message accumulator; the tag step of the same kernel at the end.
template <int NR, bool DEC>
static void batch_balanced_nr(const BatchParams& p, uint32_t n_warps, const gf128& H)
{
    std::vector<uint4> tab_g, tab_1;
    build_table(gf_pow(H, 32), tab_g);
    build_table(H, tab_1);
    TeHost te{tables().te0};
    GhHost gh_g{tab_g.data()}, gh_1{tab_1.data()};
    const uint64_t ax_a = p.aad ? (p.aad_len + 15) >> 4 : 0, ax_p = ((p.len + 15) >> 4) + AG_FINISH_WEIGHT;
    uint64_t quota_aad = ((ax_a * p.n_msgs + n_warps - 1) / n_warps + 31) & ~31ull;
    const uint64_t quota_pt = ((ax_p * p.n_msgs + n_warps - 1) / n_warps + 31) & ~31ull;
    if (!quota_aad) quota_aad = 32;
    std::vector<gf128> acc(p.n_msgs, gf_zero());
    std::vector<uint32_t> ej0(4 * p.n_msgs, 0);
    std::vector<int> closed(p.n_msgs, 0), arrived(p.n_msgs, 0);
    for (uint64_t w = 0; w < n_warps; ++w) {
        for (int axis = ax_a ? 0 : 1; axis < 2; ++axis) {
            const uint64_t per = axis ? ax_p : ax_a, quota = axis ? quota_pt : quota_aad, total = per * p.n_msgs;
            const uint64_t g0 = w * quota;
            uint64_t g1 = g0 + quota;
            if (g1 > total) g1 = total;
            for (uint64_t m = g0 / per; m * per < g1; ++m) {
                const uint64_t lo = m * per, r0 = (g0 > lo ? g0 : lo) - lo, r1 = (g1 < lo + per ? g1 : lo + per) - lo;
                uint64_t after = 0;
                MsgDesc d = ag_batch_range(ag_batch_msg(p, m), axis ? ax_a + r0 : r0, axis ? ax_a + r1 : r1, &after, 1);
                arrived[m]++;
                if (!d.last && d.len == 0 && d.aad_len == 0) continue;
                const uint8_t* ivp = p.iv + 12 * m;
                uint32_t iv[3] = {0, 0, 0};
                for (int j = 0; j < 12; ++j) iv[j >> 2] |= (uint32_t)ivp[j] << (8 * (j & 3));
                const AesCtrConst cc = aes_ctr_precompute(p.rk, iv[0], iv[1], iv[2], te);
                gf128 r = gf_zero();
                for (uint32_t t = 0; t < 32; ++t) {
                    AesCtrSeqCache cache;
                    cache.key = 0xFFFFFFFFu;
                    uint32_t el[4] = {0, 0, 0, 0};
                    gf128 y = ag_batch_lane<NR, DEC>(p.rk, cc, cache, d, t, 32u, te, gh_g, el);
                    if (t == 31 && d.last) { memcpy(&ej0[4 * m], el, 16); closed[m]++; }
                    r = gf_xor(r, y);
                    r = gf_mul_table(r, gh_1);
                }
                if (after) r = gf_mul(r, gf_pow(H, after));
                acc[m] = gf_xor(acc[m], r);
            }
        }
    }
    // the kernel's count of units per message (arrive) must agree with the pairs actually visited
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        uint64_t units = ((m + 1) * ax_p - 1) / quota_pt - (m * ax_p) / quota_pt + 1;
        if (ax_a) units += ((m + 1) * ax_a - 1) / quota_aad - (m * ax_a) / quota_aad + 1;
        if (units != (uint64_t)arrived[m]) closed[m] = -1;
    }
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        const gf128 r = acc[m];
        uint32_t tg[4] = {ag_bswap32(r.w[0]) ^ ej0[4 * m], ag_bswap32(r.w[1]) ^ ej0[4 * m + 1], ag_bswap32(r.w[2]) ^ ej0[4 * m + 2],
                          ag_bswap32(r.w[3]) ^ ej0[4 * m + 3]};
        if (closed[m] != 1) tg[0] ^= 0xDEADBEEFu;   // every message is closed by exactly one unit
        uint8_t* tp = p.tag + 16 * m;
        if (DEC) {
            uint32_t x[4];
            ag_load_block(tp, 16, x);
            p.ok[m] = ((x[0] ^ tg[0]) | (x[1] ^ tg[1]) | (x[2] ^ tg[2]) | (x[3] ^ tg[3])) ? 0 : 1;
        } else {
            ag_store_block(tp, 16, tg);
        }
    }
}

extern "C" {

int emul_batch_perkey(const uint8_t* keys, int key_bytes, int decrypt, const uint8_t* iv, const uint8_t* aad,
                      const uint64_t* aad_off, const uint8_t* in, const uint64_t* in_off, uint8_t* out, uint8_t* tag,
                      uint8_t* ok, uint64_t n_msgs)
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
    p.tag = tag;
    p.ok = ok;
    p.n_msgs = n_msgs;
    switch (key_bytes) {
        case 16: decrypt ? perkey_nk<4, true>(p) : perkey_nk<4, false>(p); break;
        case 24: decrypt ? perkey_nk<6, true>(p) : perkey_nk<6, false>(p); break;
        case 32: decrypt ? perkey_nk<8, true>(p) : perkey_nk<8, false>(p); break;
        default: return -1;
    }
    return 0;
}


// rk_bytes: (nr+1)*16 expanded key bytes.  Returns the un-finished GHASH partial
// sum_i C_i H^(n-i) (natural byte order) and writes `out`.
int emul_stream(const uint8_t* rk_bytes, int nr, const uint8_t iv[12], uint32_t ctr0, const uint8_t* in, uint8_t* out,
                uint64_t n_bytes, int mode, int ncta, int nt, uint8_t partial16[16])
{
    StreamParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    for (int j = 0; j < 12; ++j) p.iv[j >> 2] |= (uint32_t)iv[j] << (8 * (j & 3));
    p.ctr0 = ctr0;
    p.n_bytes = n_bytes;
    p.in = in;
    p.out = out;
    const TeHost te{tables().te0};
    uint32_t h[4];
    aes_encrypt_words(p.rk, nr, 0, 0, 0, 0, te, h);
    const gf128 H = gf_from_le_words(h[0], h[1], h[2], h[3]);
    gf128 total;
    switch (nr) {
        case 10: stream_nr<10>(p, mode, ncta, nt, H, total); break;
        case 12: stream_nr<12>(p, mode, ncta, nt, H, total); break;
        case 14: stream_nr<14>(p, mode, ncta, nt, H, total); break;
        default: return -1;
    }
    gf_to_bytes(total, partial16);
    return 0;
}

int emul_batch_split(const uint8_t* rk_bytes, int nr, int decrypt, int G, int S, const uint8_t* iv, const uint8_t* aad,
                     const uint64_t* aad_off, const uint8_t* in, const uint64_t* in_off, uint8_t* out, uint8_t* tag,
                     uint8_t* ok, uint64_t n_msgs);

int emul_batch(const uint8_t* rk_bytes, int nr, int decrypt, int G, const uint8_t* iv, const uint8_t* aad,
               const uint64_t* aad_off, const uint8_t* in, const uint64_t* in_off, uint8_t* out, uint8_t* tag, uint8_t* ok,
               uint64_t n_msgs)
{
    return emul_batch_split(rk_bytes, nr, decrypt, G, 1, iv, aad, aad_off, in, in_off, out, tag, ok, n_msgs);
}

int emul_batch_split(const uint8_t* rk_bytes, int nr, int decrypt, int G, int S, const uint8_t* iv, const uint8_t* aad,
                     const uint64_t* aad_off, const uint8_t* in, const uint64_t* in_off, uint8_t* out, uint8_t* tag,
                     uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    p.iv = iv;
    p.aad = aad;
    p.aad_off = aad_off;
    p.in = in;
    p.in_off = in_off;
    p.out = out;
    p.tag = tag;
    p.ok = ok;
    p.n_msgs = n_msgs;
    const TeHost te{tables().te0};
    uint32_t h[4];
    aes_encrypt_words(p.rk, nr, 0, 0, 0, 0, te, h);
    const gf128 H = gf_from_le_words(h[0], h[1], h[2], h[3]);
    switch (nr) {
        case 10: decrypt ? batch_nr<10, true>(p, G, H, S) : batch_nr<10, false>(p, G, H, S); break;
        case 12: decrypt ? batch_nr<12, true>(p, G, H, S) : batch_nr<12, false>(p, G, H, S); break;
        case 14: decrypt ? batch_nr<14, true>(p, G, H, S) : batch_nr<14, false>(p, G, H, S); break;
        default: return -1;
    }
    return 0;
}

int emul_batch_balanced(const uint8_t* rk_bytes, int nr, int decrypt, int n_warps, const uint8_t* iv, const uint8_t* aad,
                        uint64_t aad_len, uint64_t aad_stride, const uint8_t* in, uint8_t* out, uint64_t len, uint64_t stride,
                        uint8_t* tag, uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    p.iv = iv;
    p.aad = aad_len ? aad : nullptr;
    p.in = in;
    p.out = out;
    p.tag = tag;
    p.ok = ok;
    p.n_msgs = n_msgs;
    p.len = len;
    p.stride = stride;
    p.aad_len = aad_len;
    p.aad_stride = aad_stride;
    const TeHost te{tables().te0};
    uint32_t h[4];
    aes_encrypt_words(p.rk, nr, 0, 0, 0, 0, te, h);
    const gf128 H = gf_from_le_words(h[0], h[1], h[2], h[3]);
    switch (nr) {
        case 10: decrypt ? batch_balanced_nr<10, true>(p, n_warps, H) : batch_balanced_nr<10, false>(p, n_warps, H); break;
        case 12: decrypt ? batch_balanced_nr<12, true>(p, n_warps, H) : batch_balanced_nr<12, false>(p, n_warps, H); break;
        case 14: decrypt ? batch_balanced_nr<14, true>(p, n_warps, H) : batch_balanced_nr<14, false>(p, n_warps, H); break;
        default: return -1;
    }
    return 0;
}

int emul_key_expand(const uint8_t* key, int key_bytes, uint8_t* out)
{
    uint32_t rk[60];
    const uint8_t* sb = tables().sbox;
    const int nr = aes_key_expand_words(key, key_bytes, [&](uint32_t b) { return (uint32_t)sb[b & 0xff]; }, rk);
    memcpy(out, rk, (size_t)16 * (nr + 1));
    return nr;
}

void emul_gf_mul(const uint8_t a[16], const uint8_t b[16], uint8_t out[16])
{
    gf_to_bytes(gf_mul(gf_from_bytes(a), gf_from_bytes(b)), out);
}

// product through the Shoup-table path used on the per-block hot loop
void emul_gf_mul_table(const uint8_t x[16], const uint8_t c[16], uint8_t out[16])
{
    std::vector<uint4> tab;
    build_table(gf_from_bytes(c), tab);
    GhHost gh{tab.data()};
    gf_to_bytes(gf_mul_table(gf_from_bytes(x), gh), out);
}

void emul_gf_sqr(const uint8_t a[16], uint8_t out[16]) { gf_to_bytes(gf_sqr(gf_from_bytes(a)), out); }

void emul_sbox(uint8_t out[256]) { memcpy(out, tables().sbox, 256); }

// granule schedule of the host-buffer pipeline (csrc/host_sched.h)
uint32_t emul_chunk_schedule(uint64_t n, uint64_t peak, uint64_t base, uint64_t* sz, uint32_t cap)
{
    return ag_chunk_schedule(n, peak, base, sz, cap);
}

}  // extern "C"

// tests/host_emul.cu -- TEST SCAFFOLDING, never shipped.
//
// Runs the engine's per-thread device code (csrc/gcm_core.cuh, aes_core.cuh, gf128.cuh, perkey_core.cuh -- the very
// functions the CUDA kernels call) on the CPU, looping over the "threads" of a small virtual grid, so that the CPU
// test-suite can check the index arithmetic (front padding, strided Horner weights, ragged last block, lane combine)
// against the oracle without a GPU.  That includes the verify-then-release flavours: the tag-only pass of the
// shared-key lane code (ag_batch_lane<..., VERIFY>), the flat slot mapping of the gated GCTR pass (ag_gated_ctr_slot,
// with the offsets form's warp-level binary search) and the two-phase per-key message (ag_perkey_message<..., VERIFY>).
// The cross-thread steps that the kernels do with shuffles / shared memory are restated here with plain loops.
// Built by tests/batch_cases.py with `nvcc -x cu` (host code only).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <type_traits>
#include <vector>

#include "../aes-gcm-128-192-256-bits_b200/csrc/gcm_core.cuh"
#include "../aes-gcm-128-192-256-bits_b200/csrc/perkey_core.cuh"
#include "../aes-gcm-128-192-256-bits_b200/csrc/host_sched.h"
#include "../aes-gcm-128-192-256-bits_b200/csrc/kernels.h"

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

// n little-endian words from bytes
void le_words(const uint8_t* b, int n, uint32_t* w)
{
    for (int i = 0; i < n; ++i)
        w[i] = (uint32_t)b[4 * i] | ((uint32_t)b[4 * i + 1] << 8) | ((uint32_t)b[4 * i + 2] << 16) |
               ((uint32_t)b[4 * i + 3] << 24);
}

// H = E_K(0^128)
gf128 hash_key(const uint32_t* rk, int nr)
{
    uint32_t h[4];
    aes_encrypt_words(rk, nr, 0, 0, 0, 0, TeHost{tables().te0}, h);
    return gf_from_le_words(h[0], h[1], h[2], h[3]);
}

// The tag from a message's GHASH accumulator r and E_K(J0)
void tag_words(const gf128& r, const uint32_t e[4], uint32_t tg[4])
{
    for (int k = 0; k < 4; ++k) tg[k] = ag_bswap32(r.w[k]) ^ e[k];
}

// f(std::integral_constant<int, V>) for the V of Vs equal to v, -1 if there is none
template <int... Vs, class F>
int with(int v, F&& f)
{
    int rc = -1;
    (void)((v == Vs && ((rc = f(std::integral_constant<int, Vs>{})), true)) || ...);
    return rc;
}

// The fields every batch entry point sets; the layout fields are the caller's
BatchParams batch_params(const uint8_t* rk_bytes, int nr, const uint8_t* iv, const uint8_t* in, uint8_t* out, uint8_t* tag,
                         uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p{};
    if (rk_bytes) memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    p.iv = iv;
    p.in = in;
    p.out = out;
    p.tag = tag;
    p.ok = ok;
    p.n_msgs = n_msgs;
    return p;
}

template <int NR>
void stream_nr(const StreamParams& p, int mode, uint64_t ncta, uint64_t nt, gf128& total)
{
    const gf128 H = hash_key(p.rk, NR);
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

// One G-lane group on unit d (a message or a part of one): R = sum_t Y_t H^(G-t) by serial Horner with H, as the
// narrow groups of batch_groups and the combine round of k_batch_warp do.  E_K(J0) into e when the unit ends the message.
template <int NR, bool DEC, bool VERIFY>
gf128 lane_group(const uint32_t* rk, const AesCtrConst& cc, const MsgDesc& d, uint32_t G, const TeHost& te,
                 const GhHost& gh_g, const GhHost& gh_1, uint32_t e[4])
{
    gf128 r = gf_zero();
    for (uint32_t t = 0; t < G; ++t) {
        AesCtrSeqCache cache;
        cache.key = 0xFFFFFFFFu;
        uint32_t el[4] = {0, 0, 0, 0};
        r = gf_xor(r, ag_batch_lane<NR, DEC, false, VERIFY>(rk, cc, cache, d, t, G, te, gh_g, el));
        r = gf_mul_table(r, gh_1);
        if (t == G - 1 && d.last) memcpy(e, el, 16);
    }
    return r;
}

// batch_groups<NR, DEC, G, VERIFY>, one message after the other.  S > 1: the message as S counter-range segments (the
// split layout of k_batch_cta, the ticket units of k_batch_warp), each partial scaled by H^after and XORed.
template <int NR, bool DEC, bool VERIFY>
void batch_nr(const BatchParams& p, uint32_t G, uint32_t S)
{
    const gf128 H = hash_key(p.rk, NR);
    std::vector<uint4> tab_g, tab_1;
    build_table(gf_pow(H, G), tab_g);
    build_table(H, tab_1);
    const TeHost te{tables().te0};
    const GhHost gh_g{tab_g.data()}, gh_1{tab_1.data()};
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        MsgDesc whole = ag_batch_msg(p, m);
        uint32_t iv[3];
        ag_batch_iv(p, m, iv, &whole.j0ctr);
        const AesCtrConst cc = aes_ctr_precompute(p.rk, iv[0], iv[1], iv[2], te);
        gf128 total = gf_zero();
        uint32_t e[4] = {0, 0, 0, 0};
        for (uint32_t seg = 0; seg < S; ++seg) {
            uint64_t after = 0;
            const MsgDesc d = S > 1 ? ag_batch_segment(whole, seg, S, &after, VERIFY ? 1 : 4) : whole;
            gf128 r = lane_group<NR, DEC, VERIFY>(p.rk, cc, d, G, te, gh_g, gh_1, e);
            if (after) r = gf_mul(r, gf_pow(H, after));
            total = gf_xor(total, r);
        }
        uint32_t tg[4];
        tag_words(total, e, tg);
        ag_tag_out<DEC || VERIFY>(p, m, tg);
    }
}

// k_batch_warp's BALANCED partition on a virtual grid of n_warps warps (uniform records): warp w owns the w-th equal
// share of the AAD axis and of the payload axis of the concatenated messages; every unit's 32 lane accumulators are
// combined as k_batch_warp's combine rounds do (lane_group, times H^after) and XORed into the message accumulator;
// the tag step of the same kernel at the end.
template <int NR, bool DEC>
void batch_balanced_nr(const BatchParams& p, uint32_t n_warps)
{
    const gf128 H = hash_key(p.rk, NR);
    std::vector<uint4> tab_g, tab_1;
    build_table(gf_pow(H, 32), tab_g);
    build_table(H, tab_1);
    const TeHost te{tables().te0};
    const GhHost gh_g{tab_g.data()}, gh_1{tab_1.data()};
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
                uint32_t iv[3];
                ag_batch_iv(p, m, iv, &d.j0ctr);
                const AesCtrConst cc = aes_ctr_precompute(p.rk, iv[0], iv[1], iv[2], te);
                if (d.last) closed[m]++;
                gf128 r = lane_group<NR, DEC, false>(p.rk, cc, d, 32, te, gh_g, gh_1, &ej0[4 * m]);
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
        uint32_t tg[4];
        tag_words(acc[m], &ej0[4 * m], tg);
        if (closed[m] != 1) tg[0] ^= 0xDEADBEEFu;   // every message is closed by exactly one unit
        ag_tag_out<DEC>(p, m, tg);
    }
}

// Pass 2 of the verify-then-release decrypt: k_batch_ctr_gated's slot mapping on a virtual grid of n_warps warps
// (chunks of 32 x AG_GATED_ROWS slots round-robin, the offsets form's warp-level binary search, every lane walking
// forward).
template <int NR>
void ctr_gated_nr(const BatchParams& p, uint64_t n_slots, uint64_t bpr, uint64_t n_warps)
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

// batch_perkey<NK, DEC, WIDE, VERIFY>, one message after the other
template <int NK, bool DEC, bool VERIFY>
void perkey_nk(const BatchParams& p)
{
    const TeHost te{tables().te0};
    const SubWordHost sb{tables().sbox};
    for (uint64_t m = 0; m < p.n_msgs; ++m) {
        const MsgDesc d = ag_batch_msg(p, m);
        uint32_t key[8], iv[3], tg[4];
        le_words(p.keys + m * (uint64_t)(4 * NK), NK, key);
        le_words(p.iv + 12 * m, 3, iv);
        Rows4Host rows;
        SubCacheHost subc;
        if (VERIFY) {
            uint32_t x[4];
            ag_load_block(p.tag + 16 * m, 16, x);   // expected tag in, computed tag out
            memcpy(tg, x, 16);
            ag_perkey_message<NK, true, false, true>(key, iv[0], iv[1], iv[2], d, te, sb, rows, subc, tg);
            p.ok[m] = ag_tag_eq(x, tg);
        } else {
            ag_perkey_message<NK, DEC>(key, iv[0], iv[1], iv[2], d, te, sb, rows, subc, tg);
            ag_tag_out<DEC>(p, m, tg);
        }
    }
}

}  // namespace

extern "C" {

// Shared-key batch in the offsets (in_off), uniform (len, stride) or slots (len_arr, stride) form; iv_is_j0 as in
// BatchParams.  decrypt: 0 encrypt, 1 decrypt, AG_DECRYPT_VERIFIED the tag-only pass (writes ok[] only).
int emul_batch(const uint8_t* rk_bytes, int nr, int decrypt, int G, int S, const uint8_t* iv, int iv_is_j0, const uint8_t* aad,
               const uint64_t* aad_off, uint64_t aad_len, uint64_t aad_stride, const uint8_t* in, const uint64_t* in_off,
               uint64_t len, uint64_t stride, const uint32_t* len_arr, uint8_t* out, uint8_t* tag, uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p = batch_params(rk_bytes, nr, iv, in, out, tag, ok, n_msgs);
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.aad = aad;
    p.aad_off = aad_off;
    p.aad_len = aad_len;
    p.aad_stride = aad_stride;
    p.in_off = in_off;
    p.len = len;
    p.stride = stride;
    p.len_arr = len_arr;
    return with<10, 12, 14>(nr, [&](auto NR) {
        return with<0, 1, AG_DECRYPT_VERIFIED>(decrypt, [&](auto D) {
            batch_nr<NR, D != 0, D == AG_DECRYPT_VERIFIED>(p, G, S);
            return 0;
        });
    });
}

// Pass 2 of the verify-then-release decrypt over the same layouts (iv_is_j0 as above): writes the payload of the
// messages whose ok[m] is 1
int emul_batch_ctr_gated(const uint8_t* rk_bytes, int nr, const uint8_t* iv, int iv_is_j0, const uint8_t* in, const uint64_t* in_off,
                         uint64_t len, uint64_t stride, const uint32_t* len_arr, uint8_t* out, uint8_t* ok, uint64_t n_msgs,
                         uint64_t n_warps)
{
    BatchParams p = batch_params(rk_bytes, nr, iv, in, out, nullptr, ok, n_msgs);
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.in_off = in_off;
    p.len = len;
    p.stride = stride;
    p.len_arr = len_arr;
    // as agcm_batch_decrypt_verified*: blocks per whole slot (slots form) or per record (uniform form)
    const uint64_t bpr = len_arr ? (stride + 15) >> 4 : (len + 15) >> 4;
    return with<10, 12, 14>(nr, [&](auto NR) {
        ctr_gated_nr<NR>(p, bpr * n_msgs, bpr, n_warps);
        return 0;
    });
}

int emul_batch_balanced(const uint8_t* rk_bytes, int nr, int decrypt, int n_warps, const uint8_t* iv, int iv_is_j0,
                        const uint8_t* aad, uint64_t aad_len, uint64_t aad_stride, const uint8_t* in, uint8_t* out, uint64_t len,
                        uint64_t stride, uint8_t* tag, uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p = batch_params(rk_bytes, nr, iv, in, out, tag, ok, n_msgs);
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.aad = aad_len ? aad : nullptr;
    p.aad_len = aad_len;
    p.aad_stride = aad_stride;
    p.len = len;
    p.stride = stride;
    return with<10, 12, 14>(nr, [&](auto NR) {
        return with<0, 1>(decrypt, [&](auto D) {
            batch_balanced_nr<NR, D != 0>(p, n_warps);
            return 0;
        });
    });
}

// Per-key batch in the offsets form; decrypt as in emul_batch (AG_DECRYPT_VERIFIED: payload written only on a match)
int emul_batch_perkey(const uint8_t* keys, int key_bytes, int decrypt, const uint8_t* iv, const uint8_t* aad,
                      const uint64_t* aad_off, const uint8_t* in, const uint64_t* in_off, uint8_t* out, uint8_t* tag,
                      uint8_t* ok, uint64_t n_msgs)
{
    BatchParams p = batch_params(nullptr, 0, iv, in, out, tag, ok, n_msgs);
    p.keys = keys;
    p.aad = aad;
    p.aad_off = aad_off;
    p.in_off = in_off;
    return with<16, 24, 32>(key_bytes, [&](auto KB) {
        return with<0, 1, AG_DECRYPT_VERIFIED>(decrypt, [&](auto D) {
            perkey_nk<KB / 4, D != 0, D == AG_DECRYPT_VERIFIED>(p);
            return 0;
        });
    });
}

// Keystream blocks of the counters ctr0, ctr0 + stride, ... (n_blocks of them, mod 2^32) under the 12 IV bytes, as one
// lane makes them with one counter cache: which = 0 the sequential cache of the batch lanes (AesCtrSeqCache), 1 the
// stream kernel's (AesCtrCache).  The kernels' strides never move the counter's top byte alone; a stride of 2^24 does.
int emul_ctr_cached(const uint8_t* rk_bytes, int nr, const uint8_t iv12[12], uint32_t ctr0, uint32_t stride, uint64_t n_blocks,
                    int which, uint8_t* out)
{
    uint32_t rk[60], iv[3];
    memcpy(rk, rk_bytes, (size_t)16 * (nr + 1));
    le_words(iv12, 3, iv);
    const TeHost te{tables().te0};
    const AesCtrConst cc = aes_ctr_precompute(rk, iv[0], iv[1], iv[2], te);
    AesCtrSeqCache seq;
    seq.key = 0xFFFFFFFFu;
    AesCtrCache str;
    str.key = 0x00FFFF00u;
    return with<10, 12, 14>(nr, [&](auto NR) {
        for (uint64_t b = 0; b < n_blocks; ++b) {
            uint32_t ks[4];
            const uint32_t ctr = ctr0 + (uint32_t)b * stride;
            if (which) aes_ctr_block_cached<NR>(rk, cc, str, ctr, te, ks);
            else aes_ctr_block_seq<NR>(rk, cc, seq, ctr, te, ks);
            ag_store_block(out + 16 * b, 16, ks);
        }
        return 0;
    });
}

// The per-key kernels' counter mode (perkey_ctr_init + perkey_ctr_block: the key schedule on the fly, their own copy of the
// sequential cache) from the raw key, over the counters ctr0, ctr0 + stride, ... as in emul_ctr_cached
int emul_perkey_ctr(const uint8_t* key, int key_bytes, const uint8_t iv12[12], uint32_t ctr0, uint32_t stride,
                    uint64_t n_blocks, uint8_t* out)
{
    const TeHost te{tables().te0};
    const SubWordHost sb{tables().sbox};
    uint32_t kw[8], iv[3];
    le_words(key, key_bytes / 4, kw);
    le_words(iv12, 3, iv);
    return with<16, 24, 32>(key_bytes, [&](auto KB) {
        PerKeyCtr<KB / 4> st;
        SubCacheHost subc;
        perkey_ctr_init<KB / 4>(kw, iv[0], iv[1], iv[2], te, sb, subc, st);
        for (uint64_t b = 0; b < n_blocks; ++b) {
            uint32_t ks[4];
            perkey_ctr_block(st, ctr0 + (uint32_t)b * stride, te, subc, ks);
            ag_store_block(out + 16 * b, 16, ks);
        }
        return 0;
    });
}

// rk_bytes: (nr+1)*16 expanded key bytes.  Returns the un-finished GHASH partial
// sum_i C_i H^(n-i) (natural byte order) and writes `out`.
int emul_stream(const uint8_t* rk_bytes, int nr, const uint8_t iv[12], uint32_t ctr0, const uint8_t* in, uint8_t* out,
                uint64_t n_bytes, int mode, int ncta, int nt, uint8_t partial16[16])
{
    StreamParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, rk_bytes, (size_t)16 * (nr + 1));
    le_words(iv, 3, p.iv);
    p.ctr0 = ctr0;
    p.n_bytes = n_bytes;
    p.in = in;
    p.out = out;
    gf128 total;
    const int rc = with<10, 12, 14>(nr, [&](auto NR) {
        stream_nr<NR>(p, mode, ncta, nt, total);
        return 0;
    });
    if (rc == 0) gf_to_bytes(total, partial16);
    return rc;
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

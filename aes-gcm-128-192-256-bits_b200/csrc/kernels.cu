// sm_100a kernels of the AES-GCM engine, part 1: one message / one counter-range shard (k_stream), the tag
// finish, the peer-memory exchange, the key schedule and per-key setup.  Shared-memory plan and lookup
// functors: smem_tables.cuh.  Batches: kernels_batch.cu, kernels_perkey.cu.
//
// Reference blocks replaced: gcm_gctr (aes_icb + aes_ecb + xor, src/gcm_gctr.vhd:150),
// gcm_ghash + ghash_gfmul (src/gcm_ghash.vhd:225-293, src/ghash_gfmul.vhd:42-63),
// aes_kexp (config/config_aes_kexp.py:128-159, tb/key_exp.py:79-114).
#include <cuda_runtime.h>
#include <stdint.h>
#include "gcm_core.cuh"
#include "kernels.h"
#include "smem_tables.cuh"

// ===========================================================================
// aes_kexp on the device: one thread per key (tb/key_exp.py:118 semantics;
// output bytes identical to its list, stage r at bytes 16r..16r+15).
// ===========================================================================
__global__ void k_key_expand(const uint8_t* __restrict__ keys, uint64_t n_keys, int key_bytes,
                             const uint32_t* __restrict__ te0, uint8_t* __restrict__ round_keys)
{
    __shared__ uint32_t sbox_s[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sbox_s[i] = (__ldg(te0 + i) >> 8) & 0xff;
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_keys) return;
    uint8_t key[32];
    for (int j = 0; j < key_bytes; ++j) key[j] = keys[i * key_bytes + j];
    uint32_t rk[60];
    auto sb = [&](uint32_t b) { return sbox_s[b & 0xff]; };
    const int nr = aes_key_expand_words(key, key_bytes, sb, rk);
    uint32_t* dst = reinterpret_cast<uint32_t*>(round_keys + i * (uint64_t)(16 * (nr + 1)));
    for (int j = 0; j < 4 * (nr + 1); ++j) dst[j] = rk[j];  // LE words == the byte string
}

// ===========================================================================
// Per-key setup: stage keys, H, H^(2^k), per-thread / per-CTA weights, Shoup
// tables.  One CTA of 256 threads, one launch per agcm_set_key: the key (raw,
// or the Nr+1 user-loaded stages of config/config_aes_kprexp.py:66-95) rides
// in the kernel parameters, so the host does no H2D copy.
// ===========================================================================
__global__ void __launch_bounds__(256) k_key_setup(KeyDev* kd, const __grid_constant__ KeyIn in,
                                                   const uint32_t* __restrict__ te0, uint32_t nt_stream, uint32_t ncta)
{
    const uint32_t tid = threadIdx.x;
    __shared__ gf128 s_pow2[64];
    __shared__ uint32_t s_rk[60];
    __shared__ uint32_t s_te0[256];                      // the serial parts below look up shared memory, not L2
    __shared__ gf128 s_hthr[AG_STREAM_NT_MAX + 1];       // H^k, k <= NT: built here, written out once
    __shared__ gf128 s_hcta[AG_MAX_CTA + 1];             // (H^NT)^k, k <= ncta
    s_te0[tid] = __ldg(te0 + tid);                       // blockDim.x == 256
    __syncthreads();
    struct TeShared {
        const uint32_t* t;
        __device__ __forceinline__ uint32_t operator()(int tab, uint32_t w, int k) const
        {
            const uint32_t v = t[(w >> (8 * k)) & 0xff];
            return tab ? ag_rotl32(v, 8 * tab) : v;
        }
    };
    if (in.pre_expanded) {
        if (tid < 4 * (in.nr + 1)) s_rk[tid] = in.w[tid];
    } else if (tid == 0) {
        uint8_t key[32];
        for (uint32_t j = 0; j < in.key_bytes; ++j) key[j] = (uint8_t)(in.w[j >> 2] >> (8 * (j & 3)));
        auto sb = [&](uint32_t b) { return (s_te0[b & 0xff] >> 8) & 0xff; };
        aes_key_expand_words(key, (int)in.key_bytes, sb, s_rk);
    }
    __syncthreads();
    if (tid < 60) kd->rk[tid] = tid < 4 * (in.nr + 1) ? s_rk[tid] : 0u;
    if (tid == 0) {
        TeShared te{s_te0};
        uint32_t h[4];
        aes_encrypt_words(s_rk, (int)in.nr, 0, 0, 0, 0, te, h);  // H = E_K(0^128), gcm_gctr.vhd:141-144
        gf128 p = gf_from_le_words(h[0], h[1], h[2], h[3]);
        kd->H = p;
        kd->nr = in.nr;
        kd->nt_stream = nt_stream;
        kd->ncta = ncta;
        for (int k = 0; k < 64; ++k) {
            s_pow2[k] = p;
            p = gf_sqr(p);
        }
        s_hthr[0] = gf_one();
        s_hthr[1] = s_pow2[0];
        s_hcta[0] = gf_one();
    }
    __syncthreads();
    if (tid < 64) kd->pow2[tid] = s_pow2[tid];
    // H^k for k = 2..nt_stream by doubling: H^(2^s + j) = H^j * H^(2^s), j = 1..2^s
    for (uint32_t s = 0; (1u << s) < nt_stream; ++s) {
        const uint32_t half = 1u << s;
        for (uint32_t j = tid; j < half; j += blockDim.x) {
            const uint32_t dst = half + 1 + j;
            if (dst <= nt_stream) s_hthr[dst] = gf_mul(s_hthr[1 + j], s_pow2[s]);
        }
        __syncthreads();
    }
    // (H^NT)^k for k = 1..ncta, same doubling with base powers pow2[log2(NT) + s]
    uint32_t lg = 0;
    while ((1u << lg) < nt_stream) ++lg;
    if (tid == 0) s_hcta[1] = s_pow2[lg];
    __syncthreads();
    for (uint32_t s = 0; (1u << s) < ncta; ++s) {
        const uint32_t half = 1u << s;
        for (uint32_t j = tid; j < half; j += blockDim.x) {
            const uint32_t dst = half + 1 + j;
            if (dst <= ncta) s_hcta[dst] = gf_mul(s_hcta[1 + j], s_pow2[lg + s]);
        }
        __syncthreads();
    }
    for (uint32_t k = tid; k <= nt_stream; k += blockDim.x) kd->hpow_thread[k] = s_hthr[k];
    for (uint32_t k = tid; k <= ncta; k += blockDim.x) kd->hpow_cta[k] = s_hcta[k];
    // Shoup tables, row b per thread (blockDim.x == 256)
    for (int j = 0; j < 8; ++j) {
        gf128 c;
        if (j < 6) c = s_pow2[j];
        else if (j == 6) c = s_pow2[lg];
        else c = s_hcta[ncta];
        gf128 basis[8];
        basis[0] = c;
#pragma unroll
        for (int k = 1; k < 8; ++k) basis[k] = gf_mulx(basis[k - 1]);
        for (uint32_t b = tid; b < 256; b += blockDim.x) kd->tab[j][b] = gf_table_row(basis, b);
    }
}

// One full warp.  s = xor of the shard partials (natural GHASH domain, BE words).
struct FinishArgs {
    const uint32_t* rk;
    uint32_t nr;
    const uint32_t* iv;
    uint32_t j0w;         // counter word of J0 (byte-swapped)
    const KeyDev* key;
    const uint32_t* te0;
    const uint8_t* aad;
    uint64_t aad_len, ct_len;
    uint8_t* tag_calc;
    const uint8_t* tag_expected;
    uint8_t* ok;
    const uint32_t* hn;   // H^(ct blocks) precomputed by k_pow (4 BE words), or null: compute here
    bool smem_tables;     // the CTA's shared T-tables are valid (called from k_stream)
};

__device__ void finish_warp(const FinishArgs& p, gf128 s)
{
    const uint32_t lane = threadIdx.x & 31;
    const KeyDev* kd = p.key;
    const uint64_t n = (p.ct_len + 15) >> 4;
    // the constants of the serial chain below, requested up front (each is a global-memory round trip otherwise)
    const gf128 hkey = kd->H;
    uint32_t exp_tag[4] = {0, 0, 0, 0};
    if (lane == 0 && p.tag_expected && p.ok) ag_load_block(p.tag_expected, 16, exp_tag);
    gf128 hn_pre = gf_zero();
    const bool have_aad = p.aad && p.aad_len;
    if (have_aad && p.hn) { hn_pre.w[0] = __ldcg(p.hn + 0); hn_pre.w[1] = __ldcg(p.hn + 1); hn_pre.w[2] = __ldcg(p.hn + 2); hn_pre.w[3] = __ldcg(p.hn + 3); }
    const gf128 w_lane = have_aad ? kd->hpow_thread[32 - lane] : gf_zero();
    if (have_aad) {  // uniform
        // short AAD (host routes long AAD through k_stream<GHASH_ONLY>): the warp
        // runs the same front-padded strided Horner with G = 32 and generic products.
        const uint64_t a = (p.aad_len + 15) >> 4;
        const uint64_t rows = (a + 31) >> 5, pad = rows * 32 - a;
        const gf128 h32 = kd->pow2[5];
        gf128 qa = gf_zero();
        for (uint64_t u = 0; u < rows; ++u) {
            const uint64_t v = u * 32 + lane;
            if (u) qa = gf_mul(qa, h32);
            if (v >= pad) {
                const uint64_t i = v - pad;
                const uint64_t left = p.aad_len - 16 * i;
                uint32_t x[4];
                ag_load_block(p.aad + 16 * i, left < 16 ? (uint32_t)left : 16u, x);
                qa = gf_xor(qa, gf_from_le_words(x[0], x[1], x[2], x[3]));
            }
        }
        qa = gf_mul(qa, w_lane);
        qa = warp_xor(qa);                     // QA = sum A_i H^(a-i)
        const gf128 hn = p.hn ? hn_pre : warp_gf_pow(kd, n);
        if (lane == 0) s = gf_xor(s, gf_mul(qa, hn));
    }
    if (lane == 0) {
        const uint64_t ab = p.aad_len * 8, cb = p.ct_len * 8;
        s.w[0] ^= (uint32_t)(ab >> 32); s.w[1] ^= (uint32_t)ab; s.w[2] ^= (uint32_t)(cb >> 32); s.w[3] ^= (uint32_t)cb;
        s = gf_mul(s, hkey);
        uint32_t e[4];
        if (p.smem_tables) {
            TeSmem te{ag_smem, 0};
            aes_encrypt_words(p.rk, (int)p.nr, p.iv[0], p.iv[1], p.iv[2], p.j0w, te, e);  // J0 (= IV || 00000001 for a 96-bit IV)
        } else {
            TeGlobal te{p.te0};
            aes_encrypt_words(p.rk, (int)p.nr, p.iv[0], p.iv[1], p.iv[2], p.j0w, te, e);
        }
        uint32_t t[4] = {ag_bswap32(s.w[0]) ^ e[0], ag_bswap32(s.w[1]) ^ e[1], ag_bswap32(s.w[2]) ^ e[2],
                         ag_bswap32(s.w[3]) ^ e[3]};
        ag_store_block(p.tag_calc, 16, t);
        if (p.tag_expected && p.ok) *p.ok = ag_tag_eq(exp_tag, t);
    }
}

// One tiny all-to-all over NVLink peer memory instead of a collective library call (one warp):
// lane w stores this rank's scaled partial into its slot of rank w's exchange buffer, fences at
// system scope and raises the slot's epoch flag.  Nobody waits here: the bulk kernel of the next
// message may start while the flags of this one are still in flight (k_peer_finish, on a side
// stream, is the only waiter).
__device__ __forceinline__ void ag_peer_post(uint8_t* const* peer_bufs, uint32_t rank, uint32_t world, uint32_t epoch,
                                             const gf128& s)
{
    const uint32_t w = threadIdx.x & 31, slot = epoch % AG_PEER_RING;
    if (w < world) {
        uint8_t* dst = peer_bufs[w];
        __stcg(reinterpret_cast<uint4*>(dst + (slot * AG_PEER_MAX + rank) * 16), make_uint4(s.w[0], s.w[1], s.w[2], s.w[3]));
        __threadfence_system();
        *reinterpret_cast<volatile uint32_t*>(dst + AG_PEER_FLAGS + (slot * AG_PEER_MAX + rank) * 4) = epoch;
    }
}

// Posts a partial computed by earlier launches (the host-buffer pipeline: 16 B in natural GHASH
// byte order) or, with a null pointer, the zero partial of a rank whose counter range is empty
// (fewer blocks than ranks): such a rank still takes part in the exchange.
__global__ void __launch_bounds__(32) k_peer_post(uint8_t* const* peer_bufs, uint32_t rank, uint32_t world, uint32_t epoch,
                                                  const uint8_t* __restrict__ partial16)
{
    gf128 s = gf_zero();
    if (partial16) {
        uint32_t x[4];
        ag_load_block(partial16, 16, x);
        s = gf_from_le_words(x[0], x[1], x[2], x[3]);
    }
    ag_peer_post(peer_bufs, rank, world, epoch, s);
}

// Waits (bounded by the global timer) for the world's flags of `epoch` in this rank's own buffer,
// XORs the slots and finishes the tag.  FAILS CLOSED: if a peer never shows up the tag is
// zeroed, ok = 0, and both status words are raised (the host-mapped one turns every later peer
// call into AGCM_E_PEER_TIMEOUT).
__global__ void __launch_bounds__(32) k_peer_finish(const __grid_constant__ PeerFinishParams p)
{
    const uint32_t w = threadIdx.x, slot = p.epoch % AG_PEER_RING;
    const uint8_t* mine = p.peer_bufs[p.rank];
    bool arrived = true;
    if (w < p.world) {
        const volatile uint32_t* f = reinterpret_cast<const volatile uint32_t*>(mine + AG_PEER_FLAGS + (slot * AG_PEER_MAX + w) * 4);
        uint64_t t0 = 0;
        uint32_t spins = 0;
        while (*f != p.epoch) {
            __nanosleep(64);
            if ((++spins & 255u) == 0) {
                uint64_t now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (!t0) t0 = now;
                else if (now - t0 > p.timeout_ns) { arrived = false; break; }
            }
        }
    }
    __threadfence_system();
    gf128 t = gf_zero();
    if (w < p.world) {
        const uint4 q = __ldcv(reinterpret_cast<const uint4*>(mine + (slot * AG_PEER_MAX + w) * 16));
        t.w[0] = q.x; t.w[1] = q.y; t.w[2] = q.z; t.w[3] = q.w;
    }
    const gf128 s = warp_xor(t);
    if (!__all_sync(0xffffffffu, arrived)) {
        if (w == 0) {
            const uint32_t z[4] = {0, 0, 0, 0};
            ag_store_block(p.f.tag_calc, 16, z);
            if (p.f.ok) *p.f.ok = 0;
            if (p.status_dev) *p.status_dev = 1;
            if (p.status_host) *p.status_host = 1;
            __threadfence_system();
        }
        return;
    }
    FinishArgs a{p.f.rk, p.f.nr, p.f.iv, p.f.j0w, p.f.key, p.f.te0, p.f.aad, p.f.aad_len, p.f.ct_len, p.f.tag_calc,
                 p.f.tag_expected, p.f.ok, p.f.hn, false};
    finish_warp(a, s);
}

__global__ void __launch_bounds__(32) k_stream_finish(const __grid_constant__ FinishParams p)
{
    const uint32_t lane = threadIdx.x;
    gf128 s = gf_zero();
    for (uint32_t j = lane; j < p.n_parts; j += 32) {
        uint32_t x[4];
        ag_load_block(p.parts + 16 * j, 16, x);
        s = gf_xor(s, gf_from_le_words(x[0], x[1], x[2], x[3]));
    }
    s = warp_xor(s);
    FinishArgs a{p.rk, p.nr, p.iv, p.j0w, p.key, p.te0, p.aad, p.aad_len, p.ct_len, p.tag_calc, p.tag_expected, p.ok, p.hn, false};
    finish_warp(a, s);
}

// ===========================================================================
// Single stream: fused GCTR + GHASH, grid-wide strided Horner.
// grid = kd->ncta CTAs x kd->nt_stream threads; writes one 16 B partial per CTA.
// ===========================================================================
template <int NR, int MODE, bool ALIGNED>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_stream(const __grid_constant__ StreamParams p)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31, nt = blockDim.x;
    if (MODE == AG_MODE_CTR_ONLY && p.gate && __ldcg(p.gate) == 0) return;   // tag did not verify: release nothing
    if (MODE != AG_MODE_GHASH_ONLY) stage_te0(p.te0);
    if (MODE != AG_MODE_CTR_ONLY) fill_gh_tables(p.key->tab[7], nullptr);
    __syncthreads();
    if (MODE != AG_MODE_GHASH_ONLY) expand_aes_tables();
    __syncthreads();

    TeSmem te{ag_smem, lane * 4};
    GhSmem gh{ag_smem + SM_GH, (lane & 7) * 16};
    const uint32_t Gt = gridDim.x * nt;
    const uint32_t g = blockIdx.x * nt + tid;
    gf128 y = ag_stream_lane<NR, MODE, ALIGNED>(p, g, Gt, te, gh);
    if (MODE == AG_MODE_CTR_ONLY) return;

    // lane weight H^(Gt-g) = (H^NT)^(ncta-1-cta) * H^(NT-tid); lanes that absorbed nothing (short
    // messages leave most of the grid idle) skip the bit-serial product
    gf128 w_cta = gf_zero();
    if (tid == 0) w_cta = p.key->hpow_cta[gridDim.x - 1 - blockIdx.x];   // in flight during the per-thread product
    if (__any_sync(0xffffffffu, (y.w[0] | y.w[1] | y.w[2] | y.w[3]) != 0)) y = gf_mul(y, p.key->hpow_thread[nt - tid]);
    y = warp_xor(y);
    gf128* red = reinterpret_cast<gf128*>(ag_smem + SM_MISC);
    if (lane == 0) red[tid >> 5] = y;
    __syncthreads();
    if (tid < 32) {
        gf128 v = (tid < (nt >> 5)) ? red[tid] : gf_zero();
        v = warp_xor(v);
        if (tid == 0) {
            v = gf_mul(v, w_cta);
            uint32_t* dst = p.partials + 4 * blockIdx.x;
            dst[0] = v.w[0]; dst[1] = v.w[1]; dst[2] = v.w[2]; dst[3] = v.w[3];
        }
        // The last CTA to get here folds the per-CTA partials (and, for a single-shard
        // message, finishes the tag) so that one launch does the whole message.
        uint32_t ticket = 0;
        if (p.done_counter) {
            if (tid == 0) {
                __threadfence();
                ticket = atomicAdd(p.done_counter, 1u);
            }
            ticket = __shfl_sync(0xffffffffu, ticket, 0);
            if (ticket == gridDim.x - 1) {
                __threadfence();
                gf128 s = gf_zero();
                for (uint32_t j = tid; j < gridDim.x; j += 32) {
                    const uint4 q = __ldcg(reinterpret_cast<const uint4*>(p.partials) + j);
                    s.w[0] ^= q.x; s.w[1] ^= q.y; s.w[2] ^= q.z; s.w[3] ^= q.w;
                }
                s = warp_xor(s);
                if (p.scale_e) {
                    gf128 he;
                    if (p.scale_pow) {
                        he.w[0] = __ldcg(p.scale_pow + 0); he.w[1] = __ldcg(p.scale_pow + 1);
                        he.w[2] = __ldcg(p.scale_pow + 2); he.w[3] = __ldcg(p.scale_pow + 3);
                    } else {
                        he = warp_gf_pow(p.key, p.scale_e);
                    }
                    s = gf_mul(s, he);
                }
                if (p.out16 && tid == 0) {
                    const uint32_t o[4] = {ag_bswap32(s.w[0]), ag_bswap32(s.w[1]), ag_bswap32(s.w[2]), ag_bswap32(s.w[3])};
                    ag_store_block(p.out16, 16, o);  // natural GHASH byte order
                }
                if (p.peer_world) ag_peer_post(p.peer_bufs, p.peer_rank, p.peer_world, p.peer_epoch, s);
                if (p.fuse_finish) {
                    FinishArgs a{p.rk, (uint32_t)NR, p.iv, p.j0w, p.key, p.te0, p.aad, p.aad_len, p.ct_len, p.tag_calc,
                                 p.tag_expected, p.ok, p.hn, MODE != AG_MODE_GHASH_ONLY};
                    finish_warp(a, s);
                }
                if (tid == 0) *p.done_counter = 0;  // ready for the next launch on this context
            }
        }
    }
}

// out[0..3] = H^e (BE words); cached per (key, e) by the host so that the tag finish
// does not recompute it for every message of the same length
__global__ void __launch_bounds__(32) k_pow(const KeyDev* kd, uint64_t e, uint32_t* __restrict__ out)
{
    const gf128 r = warp_gf_pow(kd, e);
    if (threadIdx.x == 0) { out[0] = r.w[0]; out[1] = r.w[1]; out[2] = r.w[2]; out[3] = r.w[3]; }
}

// out16 = xor of n 16-byte partials (natural byte order in and out)
__global__ void __launch_bounds__(32) k_xor_parts(const uint8_t* __restrict__ parts, uint32_t n, uint8_t* __restrict__ out)
{
    const uint32_t lane = threadIdx.x;
    gf128 s = gf_zero();
    for (uint32_t j = lane; j < n; j += 32) {
        uint32_t x[4];
        ag_load_block(parts + 16 * j, 16, x);
        s.w[0] ^= x[0]; s.w[1] ^= x[1]; s.w[2] ^= x[2]; s.w[3] ^= x[3];
    }
    s = warp_xor(s);
    if (lane == 0) ag_store_block(out, 16, s.w);
}

// Tag finish (gcm_ghash.vhd:257,293 + tb/gcm_model.py:33-51):
//   S = xor parts (each already aligned so that the last CT block weighs H^1)
//   QA = sum A_i H^(a-i) over the (short) AAD given here, if any
//   TAG = ((QA * H^n) xor S xor LEN) * H xor E_K(J0)
// decrypt: constant-time compare with the expected tag -> ok flag; the computed
// tag is always written to tag_calc.

// ===========================================================================
// launchers (called from capi.cu)
// ===========================================================================
size_t ag_smem_bytes() { return kSmemBytes; }

cudaError_t ag_launch_stream(const StreamParams& p, int nr, int mode, int ncta, int nt, cudaStream_t st)
{
    // 128-bit path when both buffers are 16-byte aligned (GHASH-only has no output buffer)
    const bool aligned = (((uintptr_t)p.in | (uintptr_t)p.out) & 15) == 0;
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with<AG_MODE_ENC, AG_MODE_DEC, AG_MODE_GHASH_ONLY, AG_MODE_CTR_ONLY>(mode, [&](auto MODE) {
            return aligned ? ag_launch_smem(k_stream<NR, MODE, true>, ncta, nt, kSmemBytes, st, p)
                           : ag_launch_smem(k_stream<NR, MODE, false>, ncta, nt, kSmemBytes, st, p);
        });
    });
}

cudaError_t ag_launch_key_expand(const uint8_t* keys, uint64_t n_keys, int key_bytes, const uint32_t* te0,
                                 uint8_t* round_keys, cudaStream_t st)
{
    if (n_keys == 0) return cudaSuccess;
    const int nt = 128;
    const uint64_t nb = (n_keys + nt - 1) / nt;
    k_key_expand<<<(unsigned)nb, nt, 0, st>>>(keys, n_keys, key_bytes, te0, round_keys);
    return cudaGetLastError();
}

cudaError_t ag_launch_key_setup(KeyDev* kd, const KeyIn& in, const uint32_t* te0, int nt_stream, int ncta,
                                cudaStream_t st)
{
    k_key_setup<<<1, 256, 0, st>>>(kd, in, te0, (uint32_t)nt_stream, (uint32_t)ncta);
    return cudaGetLastError();
}

cudaError_t ag_launch_pow(const KeyDev* kd, uint64_t e, uint32_t* out, cudaStream_t st)
{
    k_pow<<<1, 32, 0, st>>>(kd, e, out);
    return cudaGetLastError();
}

cudaError_t ag_launch_xor_parts(const uint8_t* parts, uint32_t n, uint8_t* out, cudaStream_t st)
{
    k_xor_parts<<<1, 32, 0, st>>>(parts, n, out);
    return cudaGetLastError();
}

// CUDA loads a kernel lazily at its first launch, and that load can wait for running kernels to
// drain.  A first launch of k_peer_post / k_peer_finish while a finish kernel of the same process
// spins for a peer flag would then stall until the timeout: load them at agcm_peer_setup instead.
cudaError_t ag_preload_peer_kernels()
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, k_peer_post);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, k_peer_finish);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, k_pow);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, k_xor_parts);
    return e;
}

cudaError_t ag_launch_peer_finish(const PeerFinishParams& p, cudaStream_t st)
{
    k_peer_finish<<<1, 32, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t ag_launch_peer_post(uint8_t* const* peer_bufs, uint32_t rank, uint32_t world, uint32_t epoch,
                                const uint8_t* partial16, cudaStream_t st)
{
    k_peer_post<<<1, 32, 0, st>>>(peer_bufs, rank, world, epoch, partial16);
    return cudaGetLastError();
}

cudaError_t ag_launch_finish(const FinishParams& p, cudaStream_t st)
{
    k_stream_finish<<<1, 32, 0, st>>>(p);
    return cudaGetLastError();
}

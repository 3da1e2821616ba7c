// sm_100a kernels of the AES-GCM engine, part 3: one DISTINCT key per message (BASELINE config 4).
#include <cuda_runtime.h>
#include <stdint.h>
#include "gcm_core.cuh"
#include "kernels.h"
#include "smem_tables.cuh"
#include "perkey_core.cuh"
#include "tma_util.cuh"

// ===========================================================================
// Batched messages, one DISTINCT key per message (BASELINE config 4): one thread
// per message, key schedule on the fly (aes_kexp expand variant), private 4-bit
// GHASH table.  512 threads (128 registers each); shared memory: Te0|Te1 (64 KB,
// Te2/Te3 by a 16-bit rotate) + 512 x 256 B private tables.
// ===========================================================================
namespace {

constexpr uint32_t PK_NT = 512;
constexpr uint32_t PK_GH4 = 65536;          // + up to 2 KB alignment pad
constexpr uint32_t PK_SUBC = 12 * PK_NT * 4;   // SubWord outputs of the schedule: 12 words per thread, [j][tid]
constexpr uint32_t PK_SMEM = PK_GH4 + 2048 + PK_NT * 256 + PK_SUBC;

struct TeSmem2 {
    const uint8_t* base;
    uint32_t lane4;
    __device__ __forceinline__ uint32_t operator()(int tab, uint32_t w, int k) const
    {
        const uint32_t off = __byte_perm(w, lane4, 0x5504 | (k << 4));
        const uint32_t v = *reinterpret_cast<const uint32_t*>(base + off + (tab & 1) * 128);
        return (tab & 2) ? __byte_perm(v, 0, 0x1032) : v;
    }
};

// SubWord through byte 1 of the lane-private Te0 rows (Te0 = {2S, S, S, 3S})
struct SubWordSmem {
    const uint8_t* base;
    uint32_t lane4;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const
    {
        const uint32_t b0 = *(base + __byte_perm(w, lane4, 0x5504) + 1);
        const uint32_t b1 = *(base + __byte_perm(w, lane4, 0x5514) + 1);
        const uint32_t b2 = *(base + __byte_perm(w, lane4, 0x5524) + 1);
        const uint32_t b3 = *(base + __byte_perm(w, lane4, 0x5534) + 1);
        return b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
    }
};

// thread-private column: row n at base + n*128 (8 threads interleave 16 B slots in a
// 128 B row, so the 8 lanes of a quarter-warp never share a bank group)
struct Rows4Smem {
    uint32_t base;  // 32-bit shared address, bits 7..10 clear
    __device__ __forceinline__ void put(int n, uint4 r) const
    {
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(base + n * 128), "r"(r.x), "r"(r.y), "r"(r.z), "r"(r.w)
                     : "memory");
    }
    __device__ __forceinline__ uint4 get(uint32_t w, int k) const
    {
        const uint32_t n7 = (4 * k >= 7) ? (w >> (4 * k - 7)) : (w << (7 - 4 * k));
        const uint32_t addr = (n7 & 0x780u) | base;
        uint4 r;
        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr) : "memory");
        return r;
    }
};

// thread-private word column: word j at base + j * (4 * PK_NT) (a warp reads 128 consecutive bytes)
template <uint32_t NT>
struct SubCacheT {
    uint32_t base;  // 32-bit shared address of this thread's word 0
    __device__ __forceinline__ void put(int j, uint32_t v) const
    {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(base + j * (4 * NT)), "r"(v) : "memory");
    }
    __device__ __forceinline__ uint32_t get(int j) const
    {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base + j * (4 * NT)) : "memory");
        return v;
    }
};
using SubCacheSmem = SubCacheT<PK_NT>;

// Te0 alone (the even 128 B halves of the 256 B rows); Te1..Te3 by a byte rotate of the looked-up word
struct TeSmem1 {
    const uint8_t* base;
    uint32_t lane4;
    __device__ __forceinline__ uint32_t operator()(int tab, uint32_t w, int k) const
    {
        const uint32_t off = __byte_perm(w, lane4, 0x5504 | (k << 4));
        const uint32_t v = *reinterpret_cast<const uint32_t*>(base + off);
        return tab == 0 ? v : __byte_perm(v, 0, tab == 1 ? 0x2103 : tab == 2 ? 0x1032 : 0x0321);   // rotl 8 / 16 / 24
    }
};

// The SubWord columns in the ODD 128 B halves of the Te0 rows (where Te1 used to be): word j of thread
// (warp, lane) in half-row j*16 + warp -- 12 x 16 = 192 of the 256 half-rows, a warp reads 128 consecutive bytes
struct SubCacheRows {
    uint32_t base;  // 32-bit shared address of (half-row `warp`, lane)
    __device__ __forceinline__ void put(int j, uint32_t v) const
    {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(base + j * 4096), "r"(v) : "memory");
    }
    __device__ __forceinline__ uint32_t get(int j) const
    {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base + j * 4096) : "memory");
        return v;
    }
};

__device__ __forceinline__ void load_words(const uint8_t* p, int n_words, uint32_t* w)
{
    if (((uintptr_t)p & 3) == 0) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < n_words) w[i] = q[i];
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < n_words)
                w[i] = (uint32_t)p[4 * i] | ((uint32_t)p[4 * i + 1] << 8) | ((uint32_t)p[4 * i + 2] << 16) |
                       ((uint32_t)p[4 * i + 3] << 24);
    }
}

}  // namespace

// One lane per message.  VERIFY: the verify-then-release form (k_batch_perkey_verified, agcm_batch_decrypt_verified_perkey*):
// each lane checks its message's tag first and decrypts it only if it matched (ag_perkey_message<.., VERIFY>), ok[m]
// either way.
template <int NK, bool DEC, bool WIDE, bool VERIFY>
// (tid is read in the kernel, whose launch bounds give the compiler its range)
__device__ __forceinline__ void batch_perkey(const BatchParams& p, uint32_t tid)
{
    const uint32_t lane = tid & 31;
    // Te0 | Te1 only
    for (uint32_t idx = tid; idx < 256 * 32; idx += blockDim.x) {
        const uint32_t x = idx >> 5, l = idx & 31;
        const uint32_t t = __ldg(p.te0 + x);
        uint32_t* a = reinterpret_cast<uint32_t*>(ag_smem + SM_AES_A + x * 256 + l * 4);
        a[0] = t;
        a[32] = ag_rotl32(t, 8);
    }
    __syncthreads();
    TeSmem2 te{ag_smem, lane * 4};
    SubWordSmem sb{ag_smem, lane * 4};
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(ag_smem) + PK_GH4;
    const uint32_t s_al = (s0 + 2047u) & ~2047u;
    Rows4Smem rows{s_al + (tid >> 3) * 2048u + (tid & 7) * 16u};
    SubCacheSmem subc{s_al + PK_NT * 256u + tid * 4u};

    // Static stride, or (p.ticket: offset batches in length order) the next 32 messages of the order to whichever warp
    // is free: a warp that drew long messages must not also own a fixed share of all the later ones.
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + tid;
    for (;; g += (uint64_t)gridDim.x * blockDim.x) {
        if (p.ticket) {
            uint32_t t = 0;
            if (lane == 0) t = atomicAdd(p.ticket, 1u);
            t = __shfl_sync(0xffffffffu, t, 0);
            if ((uint64_t)t * 32 >= p.n_msgs) break;
            g = (uint64_t)t * 32 + lane;
            if (g >= p.n_msgs) continue;   // the last group may be short (the warp's next draw ends the loop)
        } else if (g >= p.n_msgs) {
            break;
        }
        const uint64_t m = p.perm ? p.perm[g] : g;   // length order for offset batches: a warp's 32 messages are equally long
        const MsgDesc d = ag_batch_msg(p, m);
        uint32_t key[8], iv[3];
        load_words(p.keys + m * (uint64_t)(4 * NK), NK, key);
        load_words(p.iv + 12 * m, 3, iv);
        if (VERIFY) {
            uint32_t x[4], tg[4];
            ag_load_block(p.tag + 16 * m, 16, x);   // expected tag in, computed tag out
            tg[0] = x[0]; tg[1] = x[1]; tg[2] = x[2]; tg[3] = x[3];
            ag_perkey_message<NK, true, WIDE, true>(key, iv[0], iv[1], iv[2], d, te, sb, rows, subc, tg);
            p.ok[m] = ag_tag_eq(x, tg);
        } else {
            uint32_t tg[4];
            ag_perkey_message<NK, DEC, WIDE>(key, iv[0], iv[1], iv[2], d, te, sb, rows, subc, tg);
            ag_tag_out<DEC>(p, m, tg);
        }
    }
}

template <int NK, bool DEC, bool WIDE>
__global__ void __launch_bounds__(PK_NT, 1) k_batch_perkey(const __grid_constant__ BatchParams p)
{
    batch_perkey<NK, DEC, WIDE, false>(p, threadIdx.x);
}

template <int NK, bool WIDE>
__global__ void __launch_bounds__(PK_NT, 1) k_batch_perkey_verified(const __grid_constant__ BatchParams p)
{
    batch_perkey<NK, true, WIDE, true>(p, threadIdx.x);
}


// ---------------------------------------------------------------------------
// The same kernel for FIXED-SIZE records, staged by TMA like k_batch_tile: one lane per message,
// box {32 bytes x 32 messages} per warp and tile, two tiles per warp, groups of 32 messages by
// atomic ticket.  Removes the thread-per-message LDG.128 / STG.128 (32 lines per request: ~17 % of
// the binding L1/shared data pipe and 1.29x DRAM over-fetch, profiles/r1_ncu_perkey.md).
// To keep 16 warps next to 32 KB of tiles, Te1 goes: the AES region holds Te0 alone (Te1..Te3 by a byte
// rotate of the looked-up word, one PRMT more on three lookups in four -- the ALU pipe has the room, the
// lookup pipe is the binding one), and the SubWord columns move into the half-rows Te1 used to fill.
// Shared memory: 64 KB Te0 + SubWord | 32 KB tiles | 128 KB private 4-bit GHASH tables.
// ---------------------------------------------------------------------------
namespace {
constexpr uint32_t PKT_NT = 512;
constexpr uint32_t PKT_TILES = 65536;                               // 16 warps x 2 x 1 KB
constexpr uint32_t PKT_BARS = PKT_TILES + (PKT_NT / 32) * 2 * TILE_BYTES;   // 16 x 2 mbarriers
constexpr uint32_t PKT_GH4 = PKT_BARS + 256;                        // + up to 2 KB alignment pad
constexpr uint32_t PKT_SMEM = 232448;                               // all of it (227 KB); the layout is checked at run time
}  // namespace

template <int NK, bool DEC>
__global__ void __launch_bounds__(PKT_NT, 1) k_batch_perkey_tile(const __grid_constant__ TileParams P)
{
    const BatchParams& p = P.b;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t idx = tid; idx < 256 * 32; idx += blockDim.x) {   // Te0 only
        const uint32_t x = idx >> 5, l = idx & 31;
        *reinterpret_cast<uint32_t*>(ag_smem + SM_AES_A + x * 256 + l * 4) = __ldg(p.te0 + x);
    }
    const uint32_t bar0 = ag_smem_addr(ag_smem + PKT_BARS + warp * 16), bar1 = bar0 + 8;
    if (lane == 0) {
        ag_mbar_init(bar0, 1);
        ag_mbar_init(bar1, 1);
        ag_fence_barrier_init();
        ag_prefetch_tmap(&P.tm_in);
        ag_prefetch_tmap(&P.tm_out);
    }
    __syncthreads();
    TeSmem1 te{ag_smem, lane * 4};
    SubWordSmem sb{ag_smem, lane * 4};
    const uint32_t s0 = ag_smem_addr(ag_smem) + PKT_GH4;
    const uint32_t s_al = (s0 + 2047u) & ~2047u;
    Rows4Smem rows{s_al + (tid >> 3) * 2048u + (tid & 7) * 16u};
    SubCacheRows subc{ag_smem_addr(ag_smem) + SM_AES_A + warp * 256u + 128u + lane * 4u};
    if (s_al + PKT_NT * 256u > ag_smem_addr(ag_smem) + PKT_SMEM) __trap();   // layout does not fit

    uint8_t* tiles = ag_smem + PKT_TILES + warp * (2 * TILE_BYTES);
    const uint32_t tile_sa = ag_smem_addr(tiles);
    const uint32_t sw = (lane >> 2) & 1;
    const uint32_t coff0 = lane * 32 + ((0 ^ sw) << 4), coff1 = lane * 32 + ((1 ^ sw) << 4);
    uint32_t par0 = 0, par1 = 0;
    const uint32_t n_blocks = (uint32_t)((p.len + 15) >> 4), tail = (uint32_t)(p.len & 15), n_full = (uint32_t)(p.len >> 4);
    const uint32_t n_tiles = (n_blocks + 1) >> 1;
    const uint32_t a_blocks = (uint32_t)((p.aad_len + 15) >> 4), atail = (uint32_t)(p.aad_len & 15);
    const uint32_t n_groups = (uint32_t)((p.n_msgs + 31) >> 5);
    for (;;) {
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(P.ticket, 1u);
        g = __shfl_sync(0xffffffffu, g, 0);
        if (g >= n_groups) break;
        const int32_t row0 = (int32_t)(g * 32);
        if (lane == 0 && n_tiles) {
            ag_mbar_expect_tx(bar0, TILE_BYTES);
            ag_tma_load_2d(tile_sa, &P.tm_in, 0, row0, bar0);
        }
        const uint64_t m_raw = (uint64_t)g * 32 + lane;
        const bool valid = m_raw < p.n_msgs;
        const uint64_t m = valid ? m_raw : p.n_msgs - 1;
        uint32_t key[8], iv[3];
        load_words(p.keys + m * (uint64_t)(4 * NK), NK, key);
        load_words(p.iv + 12 * m, 3, iv);
        uint32_t e[4];
        aes_encrypt_otf<NK>(key, 0, 0, 0, 0, te, sb, e);  // H = E_K(0^128)  (gcm_gctr.vhd:141-144)
        gf_build_table4(gf_from_le_words(e[0], e[1], e[2], e[3]), rows);
        PerKeyCtr<NK> st;
        perkey_ctr_init<NK>(key, iv[0], iv[1], iv[2], te, sb, subc, st);
        perkey_ctr_block<NK>(st, 1u, te, subc, e);  // E_K(J0)
        gf128 y = gf_zero();
        if (a_blocks) {
            const uint8_t* ap = p.aad + m * p.aad_stride;
            for (uint32_t i = 0; i < a_blocks; ++i) {
                uint32_t x[4];
                ag_load_block(ap + 16 * (uint64_t)i, (i == a_blocks - 1 && atail) ? atail : 16u, x);
                y = gf_xor(y, gf_from_le_words(x[0], x[1], x[2], x[3]));
                y = gf_mul_table4(y, rows);
            }
        }
        for (uint32_t t = 0; t < n_tiles; ++t) {
            const uint32_t b = t & 1;
            if (lane == 0 && t + 1 < n_tiles) {
                ag_bulk_wait_read0();
                ag_mbar_expect_tx(b ? bar0 : bar1, TILE_BYTES);
                ag_tma_load_2d(tile_sa + (b ^ 1) * TILE_BYTES, &P.tm_in, (int32_t)((t + 1) * 32), row0, b ? bar0 : bar1);
            }
            if (b) { ag_mbar_wait(bar1, par1); par1 ^= 1; } else { ag_mbar_wait(bar0, par0); par0 ^= 1; }
            uint8_t* tb = tiles + b * TILE_BYTES;
#pragma unroll 1
            for (int k = 0; k < 2; ++k) {
                const uint32_t j = 2 * t + k;
                if (j < n_blocks) {   // uniform
                    uint4* cp = reinterpret_cast<uint4*>(tb + (k ? coff1 : coff0));
                    const uint4 xv = *cp;
                    uint32_t x[4] = {xv.x, xv.y, xv.z, xv.w};
                    const bool ragged = (j == n_full);
                    if (ragged) ag_mask_block(x, tail);
                    uint32_t ks[4];
                    perkey_ctr_block<NK>(st, 2u + j, te, subc, ks);
                    uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
                    if (!ragged) {
                        *cp = make_uint4(o[0], o[1], o[2], o[3]);
                    } else {
                        if (valid) ag_store_block(p.out + m * p.stride + 16 * (uint64_t)j, tail, o);
                        ag_mask_block(o, tail);
                    }
                    if (DEC) y = gf_xor(y, gf_from_le_words(x[0], x[1], x[2], x[3]));
                    else y = gf_xor(y, gf_from_le_words(o[0], o[1], o[2], o[3]));
                    y = gf_mul_table4(y, rows);
                }
            }
            if (2 * t < n_full) {
                ag_fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    ag_tma_store_2d(&P.tm_out, (int32_t)(t * 32), row0, tile_sa + b * TILE_BYTES);
                    ag_bulk_commit();
                }
            } else {
                __syncwarp();
            }
        }
        const uint64_t ab = p.aad_len * 8, cb = p.len * 8;
        y.w[0] ^= (uint32_t)(ab >> 32); y.w[1] ^= (uint32_t)ab; y.w[2] ^= (uint32_t)(cb >> 32); y.w[3] ^= (uint32_t)cb;
        y = gf_mul_table4(y, rows);
        const uint32_t tg[4] = {ag_bswap32(y.w[0]) ^ e[0], ag_bswap32(y.w[1]) ^ e[1], ag_bswap32(y.w[2]) ^ e[2],
                                ag_bswap32(y.w[3]) ^ e[3]};
        if (valid) ag_tag_out<DEC>(p, m, tg);
        if (lane == 0) ag_bulk_wait_read0();
        __syncwarp();
    }
    if (lane == 0) ag_bulk_wait0();
}

cudaError_t ag_launch_batch_perkey_tile(const TileParams& p, int nr, int decrypt, int max_cta, cudaStream_t st)
{
    const uint64_t groups = (p.b.n_msgs + 31) / 32, per_cta = PKT_NT / 32;
    const uint64_t need = (groups + per_cta - 1) / per_cta;
    const int ncta = (int)(need < (uint64_t)max_cta ? need : (uint64_t)max_cta);
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with_dec(decrypt, [&](auto DEC) { return ag_launch_smem(k_batch_perkey_tile<NR - 6, DEC>, ncta, PKT_NT, PKT_SMEM, st, p); });
    });
}

cudaError_t ag_launch_batch_perkey(const BatchParams& p, int nr, int decrypt, int max_cta, cudaStream_t st)
{
    const uint64_t need = (p.n_msgs + PK_NT - 1) / PK_NT;
    const int ncta = (int)(need < (uint64_t)max_cta ? need : (uint64_t)max_cta);
    // realigned wide access when a message may sit at an odd address: batches packed by offsets, or records whose
    // buffers or pitch are not 16-byte aligned
    const bool wide = p.in_off || p.aad_off || ((((uintptr_t)p.in | (uintptr_t)p.out) | p.stride) & 15) != 0;
    return ag_with_nr(nr, [&](auto NR) {
        constexpr int NK = NR - 6;   // key words
        auto go = [&](auto kernel) { return ag_launch_smem(kernel, ncta, PK_NT, PK_SMEM, st, p); };
        if (decrypt == AG_DECRYPT_VERIFIED) return wide ? go(k_batch_perkey_verified<NK, true>) : go(k_batch_perkey_verified<NK, false>);
        return ag_with_dec(decrypt, [&](auto DEC) { return wide ? go(k_batch_perkey<NK, DEC, true>) : go(k_batch_perkey<NK, DEC, false>); });
    });
}

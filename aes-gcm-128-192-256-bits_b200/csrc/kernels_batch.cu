// sm_100a kernels of the AES-GCM engine, part 2: many independent messages under ONE shared key
// (BASELINE configs 1, 3, 5): lane groups (k_batch), TMA-staged fixed-size records (k_batch_tile), a warp
// per balanced unit (k_batch_warp), a CTA per message / segment (k_batch_cta), and the per-message J0 of
// IVs that are not 96 bits (k_batch_j0).  Replaces the testbench's -n N loops over the model
// (tb/gcm_testbench.py:25); datapath as in kernels.cu.
#include <cuda_runtime.h>
#include <stdint.h>
#include "gcm_core.cuh"
#include "kernels.h"
#include "smem_tables.cuh"
#include "tma_util.cuh"

// J0 per message for IVs of any length (SP 800-38D 7.1 step 2), one thread per IV: a 96-bit IV
// gives IV || 0^31 1 (src/aes_icb.vhd:34,118), any other length GHASH_H(IV || 0^(s+64) || [len(IV)]_64)
// with the serial recurrence of src/gcm_ghash.vhd:269-272.  16 bytes out per message.
__global__ void k_batch_j0(const KeyDev* kd, const uint8_t* __restrict__ iv, const uint64_t* __restrict__ iv_off,
                           uint64_t iv_len, uint64_t n, uint8_t* __restrict__ j0)
{
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    const uint64_t off = iv_off ? iv_off[m] : m * iv_len;
    const uint64_t len = iv_off ? iv_off[m + 1] - off : iv_len;
    const uint8_t* p = iv + off;
    uint8_t* dst = j0 + 16 * m;
    if (len == 12) {
        for (int j = 0; j < 12; ++j) dst[j] = p[j];
        dst[12] = dst[13] = dst[14] = 0;
        dst[15] = 1;
        return;
    }
    const gf128 h = kd->H;
    gf128 y = gf_zero();
    for (uint64_t o = 0; o < len; o += 16) {
        uint32_t x[4];
        ag_load_block(p + o, (len - o) < 16 ? (uint32_t)(len - o) : 16u, x);
        y = gf_mul(gf_xor(y, gf_from_le_words(x[0], x[1], x[2], x[3])), h);
    }
    const uint64_t bits = len * 8;
    y.w[2] ^= (uint32_t)(bits >> 32);
    y.w[3] ^= (uint32_t)bits;
    y = gf_mul(y, h);
    const uint32_t o4[4] = {ag_bswap32(y.w[0]), ag_bswap32(y.w[1]), ag_bswap32(y.w[2]), ag_bswap32(y.w[3])};
    ag_store_block(dst, 16, o4);
}

// ===========================================================================
// Batched messages under one shared key: G lanes per message, persistent grid.
// Tables: T_a = H^G (row Horner), T_b = H (lane combine).
// VERIFY: the tag-only pass of the verify-then-release decrypt (k_batch_verify): writes ok[] and nothing else.
// ===========================================================================
template <int NR, bool DEC, int G, bool VERIFY>
// (tid / nt are read in the kernel, whose launch bounds give the compiler their range)
__device__ __forceinline__ void batch_groups(const BatchParams& p, uint32_t tid, uint32_t nt)
{
    const uint32_t lane = tid & 31;
    constexpr int LG = (G == 1) ? 0 : (G == 2) ? 1 : (G == 4) ? 2 : (G == 8) ? 3 : (G == 16) ? 4 : 5;
    if (p.range && p.range[0] >= p.range[1]) return;   // an empty length class: not even the tables
    stage_te0(p.te0);
    fill_gh_tables(p.key->tab[LG], p.key->tab[0]);
    __syncthreads();
    expand_aes_tables();
    __syncthreads();

    TeSmem te{ag_smem, lane * 4};
    GhSmem gh_g{ag_smem + SM_GH, (lane & 7) * 16};
    GhSmem gh_1{ag_smem + SM_GH + 128, (lane & 7) * 16};

    const uint32_t t = lane & (G - 1);
    const uint32_t gbase = lane & ~(uint32_t)(G - 1);
    gf128 lane_weight = gf_one();
    if (G >= 16) lane_weight = p.key->hpow_thread[G - t];   // H^(G-t), G <= nt_stream
    const uint64_t groups_per_cta = nt / G;
    const uint64_t n_groups = (uint64_t)gridDim.x * groups_per_cta;
    const uint64_t gid = (uint64_t)blockIdx.x * groups_per_cta + tid / G;
    // every warp runs the same trip count; lanes past the end are predicated off.  With a ticket (zero at
    // launch) each warp draws its next 32/G messages when it is done with the last: messages of different
    // lengths (an offset batch) then no longer pin the grid to the warps that drew the long ones.
    const uint64_t warp_first = (uint64_t)blockIdx.x * groups_per_cta + (tid & ~31u) / G;
    const uint64_t r0 = p.range ? p.range[0] : 0, r1 = p.range ? p.range[1] : p.n_msgs;   // this launch's slice of the order
    for (uint64_t w0 = r0 + warp_first, m = r0 + gid;; w0 += n_groups, m += n_groups) {
        if (p.ticket) {
            uint32_t tk = 0;
            if (lane == 0) tk = atomicAdd(p.ticket, 32u / G);
            w0 = r0 + __shfl_sync(0xffffffffu, tk, 0);
            m = w0 + lane / G;
        }
        if (w0 >= r1) break;
        const bool valid = m < r1;
        if (valid && p.perm) m = p.perm[m];
        gf128 y = gf_zero();
        AesCtrConst cc;
        AesCtrSeqCache cache;
        cache.key = 0xFFFFFFFFu;  // invalid: the key only ever holds 24 bits
        uint32_t e[4] = {0, 0, 0, 0};  // E_K(J0): produced by lane G-1 (the one that meets the length block)
        if (valid) {
            MsgDesc d = ag_batch_msg(p, m);
            uint32_t iv0, iv1, iv2;
            if (!p.iv_is_j0 && ((uintptr_t)(p.iv + 12 * m) & 3) == 0) {
                const uint32_t* q = reinterpret_cast<const uint32_t*>(p.iv + 12 * m);
                iv0 = q[0]; iv1 = q[1]; iv2 = q[2];
            } else {
                uint32_t ivw[3];
                ag_batch_iv(p, m, ivw, &d.j0ctr);
                iv0 = ivw[0]; iv1 = ivw[1]; iv2 = ivw[2];
            }
            cc = aes_ctr_precompute(p.rk, iv0, iv1, iv2, te);
            y = ag_batch_lane<NR, DEC, G == 1, VERIFY>(p.rk, cc, cache, d, t, (uint32_t)G, te, gh_g, e);
        }
        __syncwarp();
        // R = sum_t Y_t H^(G-t)
        gf128 r = gf_zero();
        if (G >= 16) {
            // wide groups: every lane applies its own weight with one generic product (integer
            // pipe only), then a butterfly XOR -- G-1 serial table products would keep the lookup
            // pipe, the binding one, busy for G x 64 wavefronts per warp
            r = gf_mul(y, lane_weight);
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) {
                r.w[0] ^= __shfl_xor_sync(0xffffffffu, r.w[0], o);
                r.w[1] ^= __shfl_xor_sync(0xffffffffu, r.w[1], o);
                r.w[2] ^= __shfl_xor_sync(0xffffffffu, r.w[2], o);
                r.w[3] ^= __shfl_xor_sync(0xffffffffu, r.w[3], o);
            }
        } else {
            // narrow groups: serial Horner over the group's lanes with T_b = H
#pragma unroll 1
            for (int k = 0; k < G; ++k) {
                gf128 yk;
                yk.w[0] = __shfl_sync(0xffffffffu, y.w[0], gbase + k);
                yk.w[1] = __shfl_sync(0xffffffffu, y.w[1], gbase + k);
                yk.w[2] = __shfl_sync(0xffffffffu, y.w[2], gbase + k);
                yk.w[3] = __shfl_sync(0xffffffffu, y.w[3], gbase + k);
                r = gf_xor(r, yk);
                r = gf_mul_table(r, gh_1);
            }
        }
        if (valid && t == G - 1) {
            const uint32_t tg[4] = {ag_bswap32(r.w[0]) ^ e[0], ag_bswap32(r.w[1]) ^ e[1], ag_bswap32(r.w[2]) ^ e[2],
                                    ag_bswap32(r.w[3]) ^ e[3]};
            ag_tag_out<DEC>(p, m, tg);
        }
        __syncwarp();
    }
}

template <int NR, bool DEC, int G>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch(const __grid_constant__ BatchParams p)
{
    batch_groups<NR, DEC, G, false>(p, threadIdx.x, blockDim.x);
}

template <int NR, int G>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_verify(const __grid_constant__ BatchParams p)
{
    batch_groups<NR, true, G, true>(p, threadIdx.x, blockDim.x);
}

// ===========================================================================
// Batched FIXED-SIZE records under the shared key, one lane per message, records staged through
// shared memory by TMA (BASELINE config 3: 2^20 x 1500 B at a 1504 B stride).
//
// Why: with a message per lane the compute layout is the cheapest there is (no lane combine, no
// front padding, the Horner constant is H itself), but every 128-bit global load/store of a warp
// touches 32 different lines -- ncu: ~48 of ~277 L1/shared data-pipe wavefronts per 32 blocks
// (profiles/r1_ncu_batch.md), on the pipe that binds the kernel.  Here the batch is a 2-D tensor
// [message][byte] (row pitch = the record stride); one elected lane per warp asks the TMA unit for
// the box {32 bytes x 32 messages}: two blocks of each of the warp's 32 messages land as a dense,
// 32B-swizzled 1 KB tile (conflict-free LDS.128/STS.128: 4 + 4 wavefronts per 32 blocks), the lanes
// XOR the keystream in place, and the same box goes back with a TMA store.  The async proxy moves
// the bytes; the LSU pipe only sees the tile accesses.  Both tensors have 16-byte-granular extents:
// the load tensor covers the record rounded UP to whole blocks (it reaches into the caller's
// padding, which the lane masks off: src/gcm_ghash.vhd:228-246), the store tensor the record
// rounded DOWN (a ragged tail leaves by byte stores of its own lane); rows past the last message
// arrive as zeros and are clipped on the way out.
// Two tiles per warp (load of tile t+1 in flight while tile t is processed); groups of 32
// messages are handed out by an atomic ticket, so no warp idles while another still has a queue.
//
// GATHER = true: messages of DIFFERENT lengths in fixed-pitch slots (agcm_batch_crypt_slots), taken in
// the length-sorted order perm[].  A warp's 32 messages are then 32 arbitrary rows of the tensor, which
// the Blackwell TMA addresses directly: tile::gather4 loads four named rows x 32 bytes (box {32, 1}),
// tile::scatter4 stores them; eight lanes issue one each per tile, all completing on the warp's
// mbarrier.  A row index past the tensor reads zeros and writes nothing (tools/gather4_probe.cu), which
// is how lanes without a message, and rows whose 32 bytes are not both whole blocks of their message,
// are kept out of the store: those last one or two blocks leave by the lane's own stores, so no byte
// past a message's length is written.  The tile loop runs to the longest of the 32 messages.
// ===========================================================================
namespace {
constexpr uint32_t SM_TILE_BAR = SM_MISC + 1024;          // 16 warps x 2 mbarriers
constexpr uint32_t SM_TILE = SM_MISC + 2048;              // 16 warps x 2 tiles x 1 KB
constexpr size_t kTileSmemBytes = SM_TILE + (AG_STREAM_NT_MAX / 32) * 2 * TILE_BYTES;
}  // namespace

template <int NR, bool DEC, bool GATHER>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_tile(const __grid_constant__ TileParams P)
{
    const BatchParams& p = P.b;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    stage_te0(p.te0);
    fill_gh_tables(p.key->tab[0], nullptr);   // Horner constant H (a message per lane)
    const uint32_t bar0 = ag_smem_addr(ag_smem + SM_TILE_BAR + warp * 16), bar1 = bar0 + 8;
    if (lane == 0) {
        ag_mbar_init(bar0, 1);
        ag_mbar_init(bar1, 1);
        ag_fence_barrier_init();
        ag_prefetch_tmap(&P.tm_in);
        ag_prefetch_tmap(&P.tm_out);
        if (P.aad_tiled) ag_prefetch_tmap(&P.tm_aad);
    }
    __syncthreads();
    expand_aes_tables();
    __syncthreads();

    TeSmem te{ag_smem, lane * 4};
    GhSmem gh{ag_smem + SM_GH, (lane & 7) * 16};
    uint8_t* tiles = ag_smem + SM_TILE + warp * (2 * TILE_BYTES);
    const uint32_t tile_sa = ag_smem_addr(tiles);
    // this lane's two 16-byte chunks inside a tile (CU_TENSOR_MAP_SWIZZLE_32B: address bit 4 ^= bit 7)
    const uint32_t sw = (lane >> 2) & 1;
    const uint32_t coff0 = lane * 32 + ((0 ^ sw) << 4), coff1 = lane * 32 + ((1 ^ sw) << 4);
    uint32_t par0 = 0, par1 = 0;

    // uniform records: the same for every lane; GATHER: this lane's message, set per group
    uint64_t len = p.len, aad_len = p.aad_len;
    uint32_t n_blocks = (uint32_t)((len + 15) >> 4), tail = (uint32_t)(len & 15), n_full = (uint32_t)(len >> 4);
    uint32_t a_blocks = (uint32_t)((aad_len + 15) >> 4), atail = (uint32_t)(aad_len & 15);
    // the unified sequence AAD | CT (gcm_ghash.vhd:259-272) as ONE stream of tiles through the two buffers
    // (tiled AAD has one length for all messages, also with GATHER)
    const uint32_t a_tiles = P.aad_tiled ? (a_blocks + 1) >> 1 : 0;
    uint32_t tot_tiles = a_tiles + ((n_blocks + 1) >> 1);
    const uint32_t n_groups = (uint32_t)((p.n_msgs + 31) >> 5);
    const bool issuer = GATHER ? (lane & 3) == 0 : lane == 0;   // lanes that talk to the TMA unit
    const int32_t row_none = (int32_t)p.n_msgs;                 // the first row past the tensors
    for (;;) {
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(P.ticket, 1u);
        g = __shfl_sync(0xffffffffu, g, 0);
        if (g >= n_groups) break;
        const int32_t row0 = (int32_t)(g * 32);
        const uint64_t m_raw = (uint64_t)g * 32 + lane;
        const bool valid = m_raw < p.n_msgs;
        uint64_t m = valid ? m_raw : p.n_msgs - 1;   // idle lanes of the last group shadow a real message
        int32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0;     // GATHER: the rows of this lane's quad
        if constexpr (GATHER) {
            if (p.perm) m = p.perm[m];
            const MsgDesc d = ag_batch_msg(p, m);
            len = d.len;
            aad_len = d.aad_len;
            n_blocks = (uint32_t)((len + 15) >> 4); tail = (uint32_t)(len & 15); n_full = (uint32_t)(len >> 4);
            a_blocks = (uint32_t)((aad_len + 15) >> 4); atail = (uint32_t)(aad_len & 15);
            tot_tiles = a_tiles + __reduce_max_sync(0xffffffffu, (n_blocks + 1) >> 1);
            const int32_t row = valid ? (int32_t)m : row_none;
            r0 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 0);
            r1 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 1);
            r2 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 2);
            r3 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 3);
        }
        auto issue = [&](uint32_t T, uint32_t buf) {   // issuer lanes only
            const uint32_t bar = buf ? bar1 : bar0;
            if (lane == 0) ag_mbar_expect_tx(bar, TILE_BYTES);
            const CUtensorMap* tm = T < a_tiles ? &P.tm_aad : &P.tm_in;
            const int32_t col = (int32_t)((T < a_tiles ? T : T - a_tiles) * 32);
            if constexpr (GATHER) ag_tma_gather4(tile_sa + buf * TILE_BYTES + lane * 32, tm, col, r0, r1, r2, r3, bar);
            else ag_tma_load_2d(tile_sa + buf * TILE_BYTES, tm, col, row0, bar);
        };
        if (issuer && tot_tiles) issue(0, 0);
        uint32_t ivw[3], j0ctr;
        ag_batch_iv(p, m, ivw, &j0ctr);
        const AesCtrConst cc = aes_ctr_precompute(p.rk, ivw[0], ivw[1], ivw[2], te);
        AesCtrSeqCache cache;
        cache.key = 0xFFFFFFFFu;
        gf128 y = gf_zero();
        if (a_blocks && !P.aad_tiled) {   // AAD the TMA cannot address (alignment): read in place
            const uint8_t* ap = p.aad + m * p.aad_stride;
            for (uint32_t i = 0; i < a_blocks; ++i) {
                uint32_t x[4];
                ag_load_block(ap + 16 * (uint64_t)i, (i == a_blocks - 1 && atail) ? atail : 16u, x);
                y.w[0] ^= ag_bswap32(x[0]); y.w[1] ^= ag_bswap32(x[1]); y.w[2] ^= ag_bswap32(x[2]); y.w[3] ^= ag_bswap32(x[3]);
                y = gf_mul_table(y, gh);
            }
        }
        for (uint32_t T = 0; T < tot_tiles; ++T) {
            const uint32_t b = T & 1;
            if (issuer && T + 1 < tot_tiles) {
                ag_bulk_wait_read0();   // the store of tile T-1 has read the buffer tile T+1 lands in
                issue(T + 1, b ^ 1);
            }
            if (b) { ag_mbar_wait(bar1, par1); par1 ^= 1; } else { ag_mbar_wait(bar0, par0); par0 ^= 1; }
            uint8_t* tb = tiles + b * TILE_BYTES;
            if (T < a_tiles) {   // uniform: an AAD tile is absorbed, nothing goes back
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const uint32_t j = 2 * T + k;
                    if (j < a_blocks) {
                        const uint4 xv = *reinterpret_cast<const uint4*>(tb + (k ? coff1 : coff0));
                        uint32_t x[4] = {xv.x, xv.y, xv.z, xv.w};
                        if (j == a_blocks - 1 && atail) ag_mask_block(x, atail);
                        y.w[0] ^= ag_bswap32(x[0]); y.w[1] ^= ag_bswap32(x[1]); y.w[2] ^= ag_bswap32(x[2]); y.w[3] ^= ag_bswap32(x[3]);
                        y = gf_mul_table(y, gh);
                    }
                }
                __syncwarp();
                continue;
            }
            const uint32_t t = T - a_tiles;
            // GATHER: this row leaves through the TMA only if both of its blocks in the tile are whole
            const bool row_by_tma = !GATHER || 2 * t + 2 <= n_full;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint32_t j = 2 * t + k;
                if (j < n_blocks) {   // uniform unless GATHER
                    uint4* cp = reinterpret_cast<uint4*>(tb + (k ? coff1 : coff0));
                    const uint4 xv = *cp;
                    uint32_t x[4] = {xv.x, xv.y, xv.z, xv.w};
                    const bool ragged = (j == n_full);   // the record's short last block
                    if (ragged) ag_mask_block(x, tail);  // the load box reaches into the caller's padding
                    uint32_t ks[4];
                    aes_ctr_block_seq<NR>(p.rk, cc, cache, j0ctr + 1u + j, te, ks);
                    uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
                    if (!ragged && row_by_tma) {
                        *cp = make_uint4(o[0], o[1], o[2], o[3]);
                    } else {
                        // the store tensor ends at the last WHOLE block (GATHER: the row is left out of the
                        // scatter): these bytes go out by the lane's own stores, once per message, so that
                        // the padding between records is never written
                        if (valid) ag_store_block(p.out + m * p.stride + 16 * (uint64_t)j, ragged ? tail : 16u, o);
                        if (ragged) ag_mask_block(o, tail);
                    }
                    if (DEC) {
                        y.w[0] ^= ag_bswap32(x[0]); y.w[1] ^= ag_bswap32(x[1]); y.w[2] ^= ag_bswap32(x[2]); y.w[3] ^= ag_bswap32(x[3]);
                    } else {
                        y.w[0] ^= ag_bswap32(o[0]); y.w[1] ^= ag_bswap32(o[1]); y.w[2] ^= ag_bswap32(o[2]); y.w[3] ^= ag_bswap32(o[3]);
                    }
                    y = gf_mul_table(y, gh);
                }
            }
            if constexpr (GATHER) {
                const int32_t row = (valid && row_by_tma) ? (int32_t)m : row_none;
                const int32_t s0 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 0), s1 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 1);
                const int32_t s2 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 2), s3 = __shfl_sync(0xffffffffu, row, (lane & ~3u) + 3);
                ag_fence_async_smem();
                __syncwarp();
                if (issuer && (s0 != row_none || s1 != row_none || s2 != row_none || s3 != row_none)) {
                    ag_tma_scatter4(&P.tm_out, (int32_t)(t * 32), s0, s1, s2, s3, tile_sa + b * TILE_BYTES + lane * 32);
                    ag_bulk_commit();
                }
            } else if (2 * t < n_full) {   // uniform: the tile holds at least one whole block
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
        // length block (gcm_ghash.vhd:257), last multiply, E_K(J0) (gcm_ghash.vhd:293)
        {
            const uint64_t ab = aad_len * 8, cb = len * 8;
            y.w[0] ^= (uint32_t)(ab >> 32); y.w[1] ^= (uint32_t)ab; y.w[2] ^= (uint32_t)(cb >> 32); y.w[3] ^= (uint32_t)cb;
            y = gf_mul_table(y, gh);
            uint32_t e[4];
            aes_ctr_block_seq<NR>(p.rk, cc, cache, j0ctr, te, e);
            const uint32_t tg[4] = {ag_bswap32(y.w[0]) ^ e[0], ag_bswap32(y.w[1]) ^ e[1], ag_bswap32(y.w[2]) ^ e[2],
                                    ag_bswap32(y.w[3]) ^ e[3]};
            if (valid) ag_tag_out<DEC>(p, m, tg);
        }
        if (issuer) ag_bulk_wait_read0();   // both tiles are free again for the next group
        __syncwarp();
    }
    if (issuer) ag_bulk_wait0();
}

// ===========================================================================
// Batched LONG messages under the shared key: one CTA per message (G = blockDim.x
// lanes).  Same front-padded strided Horner as k_batch, constant H^NT (tab[6]); lane
// weights H^(NT-tid) by one bit-serial product per lane per message, then a CTA
// XOR-reduce.  Used when messages are too few to give every warp its own message.
// ===========================================================================
template <int NR, bool DEC>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_cta(const __grid_constant__ BatchParams p)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31, nt = blockDim.x;
    stage_te0(p.te0);
    fill_gh_tables(p.key->tab[6], nullptr);
    __syncthreads();
    expand_aes_tables();
    __syncthreads();
    TeSmem te{ag_smem, lane * 4};
    GhSmem gh_g{ag_smem + SM_GH, (lane & 7) * 16};
    gf128* red = reinterpret_cast<gf128*>(ag_smem + SM_MISC);
    const gf128 wgt = p.key->hpow_thread[nt - tid];
    // H^after cache of the split layout, 32 direct-mapped entries (key 0 = empty): with equal-length
    // messages a CTA meets S / gcd(gridDim, S) distinct segment indices (S/4 on 148 CTAs, 4 apart),
    // and one exponentiation by a single warp (seven dependent generic products, the rest of the
    // CTA waiting) costs ~20 us
    uint64_t* pow_keys = reinterpret_cast<uint64_t*>(ag_smem + SM_MISC + 1056);   // 32 x 8 B
    gf128* pow_vals = reinterpret_cast<gf128*>(ag_smem + SM_MISC + 1312);         // 32 x 16 B
    if (tid < 32) pow_keys[tid] = 0;
    __syncthreads();
    // One unit per CTA pass: a whole message, or (split > 1) one counter-range segment of it --
    // a few long messages would otherwise leave the grid idle in the last round (256 messages on
    // 148 CTAs: 2 rounds, 86 % busy).  A segment's partial is scaled by H^(blocks after it), the
    // S partials and E_K(J0) go to seg_parts, and k_batch_split_finish XORs them into the tag.
    const uint32_t S = p.split;
    const uint64_t n_units = p.n_msgs * S;
    // units go to whichever CTA is free next (atomic ticket): with static round-robin every CTA
    // waits for the one that drew the most (or the longest) units
    uint32_t* s_unit = reinterpret_cast<uint32_t*>(ag_smem + SM_MISC + 1824);
    for (uint64_t it = 0;; ++it) {
        uint64_t u;
        if (p.ticket) {
            if (tid == 0) *s_unit = atomicAdd(p.ticket, 1u);
            __syncthreads();
            u = *s_unit;
        } else {
            u = blockIdx.x + it * gridDim.x;
        }
        if (u >= n_units) break;
        const uint64_t m = u / S;
        const uint32_t seg = (uint32_t)(u - m * S);
        uint64_t after = 0;
        MsgDesc d = ag_batch_msg(p, m);
        if (S > 1) d = ag_batch_segment(d, seg, S, &after);
        uint32_t ivw[3];
        ag_batch_iv(p, m, ivw, &d.j0ctr);
        const uint32_t iv0 = ivw[0], iv1 = ivw[1], iv2 = ivw[2];
        const AesCtrConst cc = aes_ctr_precompute(p.rk, iv0, iv1, iv2, te);
        // lanes step their counter by nt (512: a multiple of 256): the stream kernel's cache fits
        AesCtrCache cache;
        cache.key = 0x00FFFF00u;  // invalid: a valid key has those bits clear
        uint32_t e[4] = {0, 0, 0, 0};
        gf128 y = ag_batch_lane<NR, DEC>(p.rk, cc, cache, d, tid, nt, te, gh_g, e);
        if (tid == nt - 1) {   // the lane that met the length block also produced E_K(J0)
            uint32_t* ej = reinterpret_cast<uint32_t*>(ag_smem + SM_MISC + 1024);
            ej[0] = e[0]; ej[1] = e[1]; ej[2] = e[2]; ej[3] = e[3];
        }
        if (__any_sync(0xffffffffu, (y.w[0] | y.w[1] | y.w[2] | y.w[3]) != 0)) y = gf_mul(y, wgt);
        y = warp_xor(y);
        if (lane == 0) red[tid >> 5] = y;
        __syncthreads();
        if (tid < 32) {
            gf128 r = (tid < (nt >> 5)) ? red[tid] : gf_zero();
            r = warp_xor(r);
            const uint32_t* ej = reinterpret_cast<const uint32_t*>(ag_smem + SM_MISC + 1024);
            if (S > 1) {
                if (after) {  // uniform
                    const uint32_t slot = (seg >> 2) & 31u;
                    gf128 ha;
                    if (pow_keys[slot] == after) {
                        ha = pow_vals[slot];
                    } else {
                        ha = warp_gf_pow(p.key, after);
                        __syncwarp();
                        if (tid == 0) {
                            pow_vals[slot] = ha;
                            pow_keys[slot] = after;
                        }
                        __syncwarp();
                    }
                    r = gf_mul(r, ha);
                }
                if (tid == 0) {
                    uint32_t* dst = p.seg_parts + 4 * u;
                    dst[0] = r.w[0]; dst[1] = r.w[1]; dst[2] = r.w[2]; dst[3] = r.w[3];
                    if (d.last) {
                        uint32_t* de = p.seg_parts + 4 * (n_units + m);
                        de[0] = ej[0]; de[1] = ej[1]; de[2] = ej[2]; de[3] = ej[3];
                    }
                }
            } else if (tid == 0) {
                const uint32_t tg[4] = {ag_bswap32(r.w[0]) ^ ej[0], ag_bswap32(r.w[1]) ^ ej[1], ag_bswap32(r.w[2]) ^ ej[2],
                                        ag_bswap32(r.w[3]) ^ ej[3]};
                ag_tag_out<DEC>(p, m, tg);
            }
        }
        __syncthreads();
    }
}

// ===========================================================================
// Batched MID-SIZE and LONG messages under the shared key: one WARP per unit, where a unit is a
// message or a counter-range part of it (ag_batch_range, the single-GPU form of the shards of
// parallel.py).  Two ways of cutting:
//   * uniform batches: a static BALANCED partition.  The AAD blocks of all messages are laid end
//     to end on one axis, their payload blocks (+ 8 positions per message for the length block and
//     E_K(J0)) on a second one, and warp w owns the w-th equal share of EACH: every warp gets the
//     same number of GHASH-only rows and the same number of AES rows to within one, whatever the
//     number and size of the messages (a single weighted axis would hand some warps only AAD and
//     others only payload, and those advance at different speeds next to each other: measured).
//     At most 2 x (n_warps + n_msgs) units, so the per-unit overhead is paid a few times per warp;
//   * offset (ragged) batches: `split` equal-work segments per message, handed out by ticket.
// The per-unit epilogue is deferred: a warp DUMPS its 32 raw lane accumulators (512 B, coalesced).
// The lane weights H^(32-t) -- one ~1100-instruction generic product per lane and unit when done in
// place, which is what made fine cuts unaffordable for k_batch / k_batch_cta -- are applied in
// combine rounds with one LANE per unit (a 32-step Horner with the H table, up to 16 units side by
// side), which also scale by H^after and XOR the unit into its message's accumulator; the lane
// that completes a message's last unit writes (or checks) the tag.  One launch.  Linearity of GHASH
// in its input, as in src/gcm_ghash.vhd:317-344.  Tables: T_a = H^32, T_b = H.
// VERIFY: the tag-only pass of the verify-then-release decrypt (k_batch_warp_verify).
// ===========================================================================
template <int NR, bool DEC, bool VERIFY>
__device__ __forceinline__ void batch_warp_units(const BatchParams& p)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    stage_te0(p.te0);
    fill_gh_tables(p.key->tab[5], p.key->tab[0]);   // T_a = H^32 (rows), T_b = H (unit combine)
    __syncthreads();
    expand_aes_tables();
    __syncthreads();
    TeSmem te{ag_smem, lane * 4};
    GhSmem gh{ag_smem + SM_GH, (lane & 7) * 16};
    GhSmem gh_1{ag_smem + SM_GH + 128, (lane & 7) * 16};
    // units this warp has dumped but not yet combined (ids), 16 per warp
    uint32_t* pend = reinterpret_cast<uint32_t*>(ag_smem + SM_MISC + 1024) + warp * 16;
    uint32_t n_pend = 0;
    const uint32_t S = p.split;
    const uint64_t ax_a = p.aad ? (p.aad_len + 15) >> 4 : 0;               // positions per message on the AAD axis
    const uint64_t ax_p = ((p.len + 15) >> 4) + AG_FINISH_WEIGHT;            // ... and on the payload axis

    // One more unit of message m is done (combined, or a cut that owned no block); whoever completes
    // the count turns the accumulator into the tag.
    auto arrive = [&](uint64_t m) {
        uint32_t units = S;   // how many units the message was cut into
        if (p.quota_pt) {
            units = (uint32_t)(((m + 1) * ax_p - 1) / p.quota_pt - (m * ax_p) / p.quota_pt + 1);
            if (ax_a) units += (uint32_t)(((m + 1) * ax_a - 1) / p.quota_aad - (m * ax_a) / p.quota_aad + 1);
        }
        __threadfence();
        const uint32_t done = atomicAdd(p.msg_cnt + m, 1u) + 1;
        if (done != units) return;
        __threadfence();
        uint32_t* dst = p.msg_acc + 4 * m;
        const uint32_t a0 = atomicOr(dst + 0, 0u), a1 = atomicOr(dst + 1, 0u), a2 = atomicOr(dst + 2, 0u), a3 = atomicOr(dst + 3, 0u);
        const uint4 e = __ldcg(reinterpret_cast<const uint4*>(p.msg_ej0 + 4 * m));
        const uint32_t tg[4] = {ag_bswap32(a0) ^ e.x, ag_bswap32(a1) ^ e.y, ag_bswap32(a2) ^ e.z, ag_bswap32(a3) ^ e.w};
        ag_tag_out<DEC>(p, m, tg);
    };

    // Combine round: lane i takes pending unit i.  R = sum_t Y_t H^(32-t) by a serial Horner over the
    // dumped accumulators with the H table, times H^(blocks after the unit) (product of the H^(2^k)
    // of the set bits), XOR into the message's accumulator; the lane that completes a message's last
    // unit turns the accumulator into the tag.
    auto combine = [&]() {
        __syncwarp();
        if (lane < n_pend) {
            const uint64_t id = pend[lane];
            const uint64_t m = __ldcg(p.unit_desc + 2 * id) - 1, after = __ldcg(p.unit_desc + 2 * id + 1);
            gf128 r = gf_zero();
            const uint4* acc = p.seg_acc + id * 32;
#pragma unroll 1
            for (int t = 0; t < 32; ++t) {
                const uint4 q = __ldcg(acc + t);
                r.w[0] ^= q.x; r.w[1] ^= q.y; r.w[2] ^= q.z; r.w[3] ^= q.w;
                r = gf_mul_table(r, gh_1);
            }
            if (after) {
                // H^after left to right: a GF(2)-linear squaring (~130 integer ops) per bit and, for a set
                // bit, one product with H through the shared table -- no generic products, no loads
                gf128 f = gf_one();
#pragma unroll 1
                for (int k = 63 - __clzll((long long)after); k >= 0; --k) {
                    f = gf_sqr(f);
                    if ((after >> k) & 1) f = gf_mul_table(f, gh_1);
                }
                r = gf_mul(r, f);
            }
            uint32_t* dst = p.msg_acc + 4 * m;
            atomicXor(dst + 0, r.w[0]); atomicXor(dst + 1, r.w[1]); atomicXor(dst + 2, r.w[2]); atomicXor(dst + 3, r.w[3]);
            arrive(m);
        }
        __syncwarp();
        n_pend = 0;
    };

    auto run_unit = [&](uint64_t id, uint64_t m, const MsgDesc& d, uint64_t after) {
        uint32_t ivw[3];
        MsgDesc du = d;
        ag_batch_iv(p, m, ivw, &du.j0ctr);
        const AesCtrConst cc = aes_ctr_precompute(p.rk, ivw[0], ivw[1], ivw[2], te);
        AesCtrSeqCache cache;
        cache.key = 0xFFFFFFFFu;
        uint32_t e[4] = {0, 0, 0, 0};
        const gf128 y = ag_batch_lane<NR, DEC, false, VERIFY>(p.rk, cc, cache, du, lane, 32u, te, gh, e);
        __stcg(p.seg_acc + id * 32 + lane, make_uint4(y.w[0], y.w[1], y.w[2], y.w[3]));
        if (lane == 0) {
            __stcg(p.unit_desc + 2 * id, m + 1);
            __stcg(p.unit_desc + 2 * id + 1, after);
            pend[n_pend] = (uint32_t)id;
        }
        if (du.last && lane == 31)   // the lane that met the length block also produced E_K(J0)
            __stcg(reinterpret_cast<uint4*>(p.msg_ej0 + 4 * m), make_uint4(e[0], e[1], e[2], e[3]));
        if (++n_pend == 16) combine();
    };

    if (p.quota_pt) {
        const uint64_t w = (uint64_t)blockIdx.x * (blockDim.x >> 5) + warp;
        const uint64_t id_half = (uint64_t)gridDim.x * (blockDim.x >> 5) + p.n_msgs;
        // axis 0: AAD blocks (positions 0 .. a of a message), axis 1: payload blocks + finish (positions a .. )
        for (int axis = ax_a ? 0 : 1; axis < 2; ++axis) {
            const uint64_t per = axis ? ax_p : ax_a, quota = axis ? p.quota_pt : p.quota_aad, total = per * p.n_msgs;
            const uint64_t g0 = w * quota;
            uint64_t g1 = g0 + quota;
            if (g1 > total) g1 = total;
            for (uint64_t m = g0 / per; m * per < g1; ++m) {   // uniform per warp
                const uint64_t lo = m * per, r0 = (g0 > lo ? g0 : lo) - lo, r1 = (g1 < lo + per ? g1 : lo + per) - lo;
                uint64_t after = 0;
                const MsgDesc d = ag_batch_range(ag_batch_msg(p, m), axis ? ax_a + r0 : r0, axis ? ax_a + r1 : r1, &after, 1);
                if (!d.last && d.len == 0 && d.aad_len == 0) {   // a cut inside the finish positions: no block of it is mine
                    if (lane == 0) arrive(m);
                    continue;
                }
                run_unit((axis ? id_half : 0) + w + m, m, d, after);
            }
        }
    } else {
        const uint64_t n_units = p.n_msgs * S;
        for (;;) {
            uint32_t tk = 0;
            if (lane == 0) tk = atomicAdd(p.ticket, 1u);
            const uint64_t u = __shfl_sync(0xffffffffu, tk, 0);
            if (u >= n_units) break;
            const uint64_t m = u / S;
            uint64_t after = 0;
            MsgDesc d = ag_batch_msg(p, m);
            if (S > 1) d = ag_batch_segment(d, (uint32_t)(u - m * S), S, &after, VERIFY ? 1 : 4);
            run_unit(u, m, d, after);
        }
    }
    if (n_pend) combine();
}

template <int NR, bool DEC>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_warp(const __grid_constant__ BatchParams p)
{
    batch_warp_units<NR, DEC, false>(p);
}

template <int NR>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_warp_verify(const __grid_constant__ BatchParams p)
{
    batch_warp_units<NR, true, true>(p);
}

// ===========================================================================
// Pass 2 of the verify-then-release batch decrypt: GCTR over the payload blocks of the whole batch cut flat into
// slots (ag_gated_ctr_slot), skipping every message whose tag pass 1 rejected -- the batch analogue of
// k_stream<CTR_ONLY> with its gate.  A warp takes 32 x AG_GATED_ROWS consecutive slots per chunk, lane l the slots
// l, l + 32, ...; in an offset batch lane 0 finds the chunk's first message by binary search over in_off and every
// lane walks forward from there.  A slot that falls in a rejected message costs one flag load.
// ===========================================================================
// n_slots: slots of the uniform / slots forms (offsets: from in_off, which lives on the device)
template <int NR>
__global__ void __launch_bounds__(AG_STREAM_NT_MAX, 1) k_batch_ctr_gated(const __grid_constant__ BatchParams p, uint64_t n_slots,
                                                                       uint64_t bpr)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    stage_te0(p.te0);
    __syncthreads();
    expand_aes_tables();
    __syncthreads();
    TeSmem te{ag_smem, lane * 4};
    constexpr uint64_t CH = 32ull * AG_GATED_ROWS;
    if (p.in_off) n_slots = (p.in_off[p.n_msgs] - p.in_off[0] + 15) >> 4;
    const uint64_t n_chunks = (n_slots + CH - 1) / CH;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t c = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (tid >> 5); c < n_chunks; c += warps) {
        uint64_t m = 0;
        if (p.in_off) {
            if (lane == 0) m = ag_gated_first_msg(p, c * CH);
            m = __shfl_sync(0xffffffffu, m, 0);
        }
#pragma unroll 1
        for (uint32_t k = 0; k < AG_GATED_ROWS; ++k) {
            const uint64_t s = c * CH + 32 * k + lane;
            if (s < n_slots) ag_gated_ctr_slot<NR>(p, s, bpr, m, te);
        }
    }
}

// Tag finish of the split layout: one thread per message XORs its S scaled partials
// (linearity of GHASH in its input, the same algebra as gcm_ghash.vhd:330-332) and E_K(J0).
template <bool DEC>
__global__ void k_batch_split_finish(const __grid_constant__ BatchParams p)
{
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= p.n_msgs) return;
    const uint32_t S = p.split;
    uint32_t r[4] = {0, 0, 0, 0};
    for (uint32_t k = 0; k < S; ++k) {
        const uint4 q = *reinterpret_cast<const uint4*>(p.seg_parts + 4 * (m * S + k));
        r[0] ^= q.x; r[1] ^= q.y; r[2] ^= q.z; r[3] ^= q.w;
    }
    const uint4 e = *reinterpret_cast<const uint4*>(p.seg_parts + 4 * (p.n_msgs * S + m));
    const uint32_t tg[4] = {ag_bswap32(r[0]) ^ e.x, ag_bswap32(r[1]) ^ e.y, ag_bswap32(r[2]) ^ e.z, ag_bswap32(r[3]) ^ e.w};
    ag_tag_out<DEC>(p, m, tg);
}

// ===========================================================================
// Length sort of an offset batch (counting sort, longest first).  A warp works on 32/G messages side by
// side in lock step, so a row costs the warp as much as its LONGEST message needs: with mixed lengths in
// arrival order (an IMIX of 64 / 576 / 1500 B packets) three quarters of the lane-rows are idle.  Keys are
// the work of a message in blocks (payload + a quarter of the AAD), clipped to AG_SORT_BUCKETS - 1.
// ===========================================================================
namespace {
constexpr uint32_t AG_SORT_BUCKETS = 4096;
constexpr uint32_t AG_SORT_LONG = 1024, AG_SORT_MID = 256;   // class limits in blocks of work: long >= 1024 > medium >= 256 > short
__device__ __forceinline__ uint32_t ag_sort_bucket(const BatchParams& p, uint64_t m)
{
    const MsgDesc d = ag_batch_msg(p, m);
    const uint64_t n = (d.len + 15) >> 4, a = (d.aad_len + 15) >> 4;
    const uint64_t w = n + (a + 3) / 4;
    return AG_SORT_BUCKETS - 1 - (uint32_t)(w < AG_SORT_BUCKETS - 1 ? w : AG_SORT_BUCKETS - 1);   // bucket 0 = longest
}
}  // namespace

__global__ void __launch_bounds__(256) k_len_hist(const __grid_constant__ BatchParams p, uint32_t* __restrict__ hist)
{
    __shared__ uint32_t h[AG_SORT_BUCKETS];
    for (uint32_t i = threadIdx.x; i < AG_SORT_BUCKETS; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; m < p.n_msgs; m += (uint64_t)gridDim.x * blockDim.x)
        atomicAdd(&h[ag_sort_bucket(p, m)], 1u);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < AG_SORT_BUCKETS; i += blockDim.x)
        if (h[i]) atomicAdd(hist + i, h[i]);
}

// exclusive scan of the 4096 bucket counts, in place (one CTA of 1024 threads, 4 buckets each)
__global__ void __launch_bounds__(1024) k_len_scan(uint32_t* __restrict__ hist, uint32_t* __restrict__ ranges)
{
    __shared__ uint32_t part[1024];
    const uint32_t t = threadIdx.x;
    uint32_t v[4], s = 0;
    for (int k = 0; k < 4; ++k) { v[k] = hist[4 * t + k]; s += v[k]; }
    part[t] = s;
    __syncthreads();
    for (uint32_t d = 1; d < 1024; d <<= 1) {
        const uint32_t x = t >= d ? part[t - d] : 0;
        __syncthreads();
        part[t] += x;
        __syncthreads();
    }
    uint32_t run = part[t] - s;
    for (int k = 0; k < 4; ++k) { hist[4 * t + k] = run; run += v[k]; }
    __syncthreads();
    // three length classes of the sorted order, one k_batch launch each (long: 32 lanes per message, medium: 4,
    // short: 1): ranges[2c], ranges[2c+1].  Bucket b holds work 4095 - b blocks; the order is longest first.
    if (t == 0) {
        const uint32_t end_long = hist[AG_SORT_BUCKETS - AG_SORT_LONG], end_mid = hist[AG_SORT_BUCKETS - AG_SORT_MID];
        ranges[0] = 0;        ranges[1] = end_long;
        ranges[2] = end_long; ranges[3] = end_mid;
        ranges[4] = end_mid;  ranges[5] = part[1023];
    }
}

// Scatter, chunk by chunk of 2048 messages per CTA: a shared-memory histogram of the chunk, ONE global atomic per
// (chunk, non-empty bucket) to reserve that bucket's range, then ranks inside the chunk from shared-memory
// atomics.  (A global atomic per message serialises on the handful of buckets a real packet mix uses: an IMIX of
// three lengths spent more time here than in the cipher.)
__global__ void __launch_bounds__(256) k_len_scatter(const __grid_constant__ BatchParams p, uint32_t* __restrict__ cursor,
                                                     uint32_t* __restrict__ perm)
{
    constexpr uint32_t CH = 2048;
    __shared__ uint32_t cnt[AG_SORT_BUCKETS];    // count, then the chunk's base in the bucket's global range
    __shared__ uint32_t rank[AG_SORT_BUCKETS];
    const uint64_t n_chunks = (p.n_msgs + CH - 1) / CH;
    for (uint64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        for (uint32_t i = threadIdx.x; i < AG_SORT_BUCKETS; i += blockDim.x) { cnt[i] = 0; rank[i] = 0; }
        __syncthreads();
        const uint64_t m0 = c * CH, m1 = (m0 + CH < p.n_msgs) ? m0 + CH : p.n_msgs;
        uint32_t bk[CH / 256];
#pragma unroll
        for (uint32_t k = 0; k < CH / 256; ++k) {
            const uint64_t m = m0 + k * 256 + threadIdx.x;
            bk[k] = m < m1 ? ag_sort_bucket(p, m) : 0xFFFFFFFFu;
            if (m < m1) atomicAdd(&cnt[bk[k]], 1u);
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < AG_SORT_BUCKETS; i += blockDim.x)
            if (cnt[i]) cnt[i] = atomicAdd(cursor + i, cnt[i]);
        __syncthreads();
#pragma unroll
        for (uint32_t k = 0; k < CH / 256; ++k)
            if (bk[k] != 0xFFFFFFFFu) perm[cnt[bk[k]] + atomicAdd(&rank[bk[k]], 1u)] = (uint32_t)(m0 + k * 256 + threadIdx.x);
        __syncthreads();
    }
}

cudaError_t ag_launch_len_sort(const BatchParams& p, uint32_t* hist4096, uint32_t* ranges6, uint32_t* perm, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(hist4096, 0, sizeof(uint32_t) * AG_SORT_BUCKETS, st);
    if (e != cudaSuccess) return e;
    const unsigned nb = (unsigned)((p.n_msgs + 255) / 256 < 1184 ? (p.n_msgs + 255) / 256 : 1184);
    k_len_hist<<<nb, 256, 0, st>>>(p, hist4096);
    k_len_scan<<<1, 1024, 0, st>>>(hist4096, ranges6);
    k_len_scatter<<<nb, 256, 0, st>>>(p, hist4096, perm);
    return cudaGetLastError();
}

// ===========================================================================
// launchers (called from capi.cu)
// ===========================================================================
cudaError_t ag_launch_batch_tile(const TileParams& p, int nr, int decrypt, int gather, int ncta, cudaStream_t st)
{
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with_dec(decrypt, [&](auto DEC) {
            return gather ? ag_launch_smem(k_batch_tile<NR, DEC, true>, ncta, AG_STREAM_NT_MAX, kTileSmemBytes, st, p)
                          : ag_launch_smem(k_batch_tile<NR, DEC, false>, ncta, AG_STREAM_NT_MAX, kTileSmemBytes, st, p);
        });
    });
}

static cudaError_t launch_batch_warp_verify(const BatchParams& p, int nr, int ncta, cudaStream_t st);

cudaError_t ag_launch_batch_warp(const BatchParams& p, int nr, int decrypt, int ncta, cudaStream_t st)
{
    if (decrypt == AG_DECRYPT_VERIFIED) return launch_batch_warp_verify(p, nr, ncta, st);
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with_dec(decrypt, [&](auto DEC) { return ag_launch_smem(k_batch_warp<NR, DEC>, ncta, AG_STREAM_NT_MAX, kSmemBytes, st, p); });
    });
}

cudaError_t ag_launch_batch_cta(const BatchParams& p, int nr, int decrypt, int ncta, int nt, cudaStream_t st)
{
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with_dec(decrypt, [&](auto DEC) {
            cudaError_t e = ag_launch_smem(k_batch_cta<NR, DEC>, ncta, nt, kSmemBytes, st, p);
            if (e != cudaSuccess || p.split <= 1) return e;
            k_batch_split_finish<DEC><<<(unsigned)((p.n_msgs + 127) / 128), 128, 0, st>>>(p);
            return cudaGetLastError();
        });
    });
}

cudaError_t ag_launch_batch(const BatchParams& p, int nr, int decrypt, int g, int ncta, int nt, cudaStream_t st)
{
    return ag_with_nr(nr, [&](auto NR) {
        return ag_with<1, 2, 4, 8, 16, 32>(g, [&](auto G) {
            if (decrypt == AG_DECRYPT_VERIFIED) return ag_launch_smem(k_batch_verify<NR, G>, ncta, nt, kSmemBytes, st, p);
            return ag_with_dec(decrypt, [&](auto DEC) { return ag_launch_smem(k_batch<NR, DEC, G>, ncta, nt, kSmemBytes, st, p); });
        });
    });
}

// Defined past ag_launch_batch, so that k_batch_warp_verify is instantiated after k_batch_verify (and k_batch_warp before
// k_batch).  The order of instantiation moves the register allocation of the AES-128 warp-unit kernels; in this order
// they spill no more than they did with a launcher per kernel.
static cudaError_t launch_batch_warp_verify(const BatchParams& p, int nr, int ncta, cudaStream_t st)
{
    return ag_with_nr(nr, [&](auto NR) { return ag_launch_smem(k_batch_warp_verify<NR>, ncta, AG_STREAM_NT_MAX, kSmemBytes, st, p); });
}

cudaError_t ag_launch_batch_ctr_gated(const BatchParams& p, int nr, uint64_t n_slots, uint64_t bpr, int max_cta, cudaStream_t st)
{
    const uint64_t chunks = (n_slots + 32ull * AG_GATED_ROWS - 1) / (32ull * AG_GATED_ROWS), per_cta = AG_STREAM_NT_MAX / 32;
    const uint64_t need = (chunks + per_cta - 1) / per_cta;
    const int ncta = p.in_off ? max_cta : (int)(need < (uint64_t)max_cta ? need : (uint64_t)max_cta);
    if (ncta == 0) return cudaSuccess;
    return ag_with_nr(nr, [&](auto NR) {
        return ag_launch_smem(k_batch_ctr_gated<NR>, ncta, AG_STREAM_NT_MAX, kSmemBytes, st, p, n_slots, bpr);
    });
}

cudaError_t ag_launch_batch_j0(const KeyDev* kd, const uint8_t* iv, const uint64_t* iv_off, uint64_t iv_len, uint64_t n,
                               uint8_t* j0, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    k_batch_j0<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(kd, iv, iv_off, iv_len, n, j0);
    return cudaGetLastError();
}


// Per-thread AES-GCM work items, written once as host+device code.
//
// The CUDA kernels (kernels*.cu) call these with shared-memory lookup functors;
// tests/host_emul.cu calls the SAME functions on the CPU with plain-array
// functors and loops over "threads" to check the index arithmetic (front
// padding, strided Horner weights, partial last block) against the oracle
// before any GPU time is spent.  This is test scaffolding: the product library
// exports no CPU path.
//
// GHASH decomposition (replaces the serial recurrence Y <- (Y xor X)*H of
// src/gcm_ghash.vhd:269-272 by the equivalent polynomial, using the linearity the
// reference itself relies on at gcm_ghash.vhd:317-344):
//
//   a group of G lanes shares one block sequence S_0..S_{m-1}; it is front-padded
//   with `pad` virtual zero blocks to rows*G; lane t owns virtual blocks
//   t, t+G, t+2G, ... and runs  Y_t <- Y_t * H^G  xor  S   per row.
//   Then  sum_i S_i H^(m-i) = sum_t Y_t * H^(G-t).
#pragma once
#include <stdint.h>
#include <string.h>
#include "aes_core.cuh"
#include "gf128.cuh"

enum : int {
    AG_MODE_ENC = 0,         // out = in ^ KS ; GHASH over out   (src/aes_gcm.vhd:207-211, enc)
    AG_MODE_DEC = 1,         // out = in ^ KS ; GHASH over in    (src/aes_gcm.vhd:207-211, dec)
    AG_MODE_GHASH_ONLY = 2,  // GHASH over in (bulk AAD)
    AG_MODE_CTR_ONLY = 3     // out = in ^ KS ; no GHASH (profiling aid)
};

constexpr int AG_MAX_CTA = 256;       // upper bound on persistent-grid size
// Threads per persistent CTA.  512 (128 registers per thread, no spills) measured 1-2 % faster than
// 1024 (64 registers, a few spills) on every path: 16 warps already keep > 200 lookups in flight per SM.
#ifndef AG_NT_MAX
#define AG_NT_MAX 512
#endif
constexpr int AG_STREAM_NT_MAX = AG_NT_MAX;

// Per-key derived material, resident in HBM (about 53 KB).  Written by
// k_key_setup, read by every other kernel.
struct KeyDev {
    uint32_t rk[60];                        // stage keys as LE words (stage r = words 4r..4r+3)
    uint32_t nr;                            // 10 / 12 / 14
    uint32_t nt_stream;                     // threads per CTA the stream tables were built for
    uint32_t ncta;                          // persistent grid size the stream tables were built for
    uint32_t _pad;
    gf128 H;                                // E_K(0^128)            (src/gcm_gctr.vhd:141-144)
    gf128 pow2[64];                         // H^(2^k)
    gf128 hpow_thread[AG_STREAM_NT_MAX + 1];// H^k, k = 0..NT
    gf128 hpow_cta[AG_MAX_CTA + 1];         // (H^NT)^k, k = 0..ncta
    uint4 tab[8][256];                      // Shoup tables: [j]=H^(2^j), j=0..5; [6]=H^NT; [7]=H^(NT*ncta)
};

// ---- 16-byte block I/O ------------------------------------------------------
// nvalid in 1..16; bytes past nvalid read as zero.  Vector path when aligned.
AG_HD void ag_load_block(const uint8_t* p, uint32_t nvalid, uint32_t x[4])
{
    if (nvalid == 16) {
#if defined(__CUDA_ARCH__)
        const uintptr_t a = (uintptr_t)p;
        if ((a & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(p);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
            return;
        }
        if ((a & 3) == 0) {
            const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
            x[0] = q[0]; x[1] = q[1]; x[2] = q[2]; x[3] = q[3];
            return;
        }
#endif
    }
    // ragged / unaligned path; static register indexing (no local-memory array)
    x[0] = x[1] = x[2] = x[3] = 0;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j)
        if (j < nvalid) x[j >> 2] |= (uint32_t)p[j] << (8 * (j & 3));
}

AG_HD void ag_store_block(uint8_t* p, uint32_t nvalid, const uint32_t x[4])
{
    if (nvalid == 16) {
#if defined(__CUDA_ARCH__)
        const uintptr_t a = (uintptr_t)p;
        if ((a & 15) == 0) {
            *reinterpret_cast<uint4*>(p) = make_uint4(x[0], x[1], x[2], x[3]);
            return;
        }
        if ((a & 3) == 0) {
            uint32_t* q = reinterpret_cast<uint32_t*>(p);
            q[0] = x[0]; q[1] = x[1]; q[2] = x[2]; q[3] = x[3];
            return;
        }
#endif
    }
#if defined(__CUDA_ARCH__)
    if (((uintptr_t)p & 3) == 0) {   // ragged tail at a word-aligned address: whole words first, then the odd bytes
        uint32_t* q = reinterpret_cast<uint32_t*>(p);
#pragma unroll
        for (uint32_t w = 0; w < 4; ++w) {
            if (nvalid >= 4 * w + 4) {
                q[w] = x[w];
            } else {
#pragma unroll
                for (uint32_t j = 4 * w; j < 4 * w + 3; ++j)
                    if (j < nvalid) p[j] = (uint8_t)(x[w] >> (8 * (j & 3)));
            }
        }
        return;
    }
#endif
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j)
        if (j < nvalid) p[j] = (uint8_t)(x[j >> 2] >> (8 * (j & 3)));
}

// zero bytes nvalid..15 of a block held as LE words (gcm_ghash.vhd:228-246 mask)
AG_HD void ag_mask_block(uint32_t x[4], uint32_t nvalid)
{
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const int lo = 4 * w;
        if ((int)nvalid <= lo) x[w] = 0;
        else if ((int)nvalid < lo + 4) x[w] &= (1u << (8 * (nvalid - lo))) - 1u;
    }
}

// ---- 16-byte blocks at addresses that are NOT 16-byte aligned (device only) -----------------
// Byte-wise access costs 16 load and 16 store instructions per block, each of them scattered over the
// warp; these helpers use whole aligned 16-byte granules instead.
#if defined(__CUDA_ARCH__)
// bytes r .. r+15 of the 32-byte string a | b (1 <= r <= 15): a three-stage barrel shifter
__device__ __forceinline__ uint4 ag_realign(const uint4& a, const uint4& b, uint32_t r)
{
    uint32_t c0 = a.x, c1 = a.y, c2 = a.z, c3 = a.w, c4 = b.x, c5 = b.y, c6 = b.z;
    if (r & 8) { c0 = c2; c1 = c3; c2 = c4; c3 = c5; c4 = c6; c5 = b.w; }
    if (r & 4) { c0 = c1; c1 = c2; c2 = c3; c3 = c4; c4 = c5; }
    const uint32_t sh = (r & 3) * 8;
    return make_uint4(__funnelshift_r(c0, c1, sh), __funnelshift_r(c1, c2, sh), __funnelshift_r(c2, c3, sh),
                      __funnelshift_r(c3, c4, sh));
}
#endif

// Load like ag_load_block; a whole block at an unaligned address comes from the two aligned granules that
// hold it when both lie inside [lo, hi) -- the unit's own bytes, so nothing outside the caller's data is read.
// Only for addresses that are not even word-aligned (k_stream's strided lanes: a word-aligned block is cheaper as four
// 32-bit loads).
AG_HD void ag_load_block_in(const uint8_t* p, uint32_t nvalid, uint32_t x[4], const uint8_t* lo, const uint8_t* hi)
{
#if defined(__CUDA_ARCH__)
    const uintptr_t a = (uintptr_t)p;
    const uint32_t r = (uint32_t)(a & 15);
    if (nvalid == 16 && (r & 3) != 0) {
        const uint8_t* base = p - r;
        if (base >= lo && base + 32 <= hi) {
            const uint4 w0 = *reinterpret_cast<const uint4*>(base), w1 = *reinterpret_cast<const uint4*>(base + 16);
            const uint4 v = ag_realign(w0, w1, r);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
            return;
        }
    }
#else
    (void)lo; (void)hi;
#endif
    ag_load_block(p, nvalid, x);
}

// The same decision hoisted out of a message's block loop, for a lane that walks its message alone (k_batch<G = 1>):
// blocks 1 .. n_wide of a buffer whose base sits r != 0 bytes past a 16-byte boundary are read as two aligned granules
// inside the buffer; the loop pays one unsigned compare per block.  Here the two granules also beat four 32-bit loads
// of a word-aligned block (1500 B records at a 1500 B pitch, AES-192: 450 vs 404 GB/s).
struct AgWideWindow {
    uint32_t r;        // base & 15
    uint32_t n_wide;   // blocks 1 .. n_wide qualify (0: none)
    AG_HD static AgWideWindow make(const uint8_t* base, uint64_t len)
    {
        AgWideWindow w;
        w.r = (uint32_t)((uintptr_t)base & 15);
        // block j (j >= 1) spans granules [16j - r, 16j - r + 32) of the buffer: inside it while 16j - r + 32 <= len
        w.n_wide = 0;
        if (w.r != 0 && len + w.r >= 48) {
            const uint64_t q = (len + w.r - 32) >> 4;
            w.n_wide = q > 0xFFFFFFFEull ? 0xFFFFFFFEu : (uint32_t)q;
        }
        return w;
    }
};

// The upper granule of block j is the lower granule of block j + 1: a lane that reads consecutive blocks keeps it.
struct AgLoadCarry {
    uint4 g;
    uint32_t j;   // g is the lower granule of block j (0xFFFFFFFF: nothing kept)
};

template <bool WIDE>
AG_HD void ag_load_block_win(const uint8_t* base, uint32_t j, uint32_t nvalid, uint32_t x[4], const AgWideWindow& w, AgLoadCarry& c)
{
#if defined(__CUDA_ARCH__)
    if (WIDE && j - 1u < w.n_wide) {   // 1 <= j <= n_wide: a whole block (the last, possibly short, block is index >= n_wide + 1)
        const uint8_t* g = base + 16 * (uint64_t)j - w.r;
        const uint4 w1 = *reinterpret_cast<const uint4*>(g + 16);
        const uint4 w0 = (c.j == j) ? c.g : *reinterpret_cast<const uint4*>(g);
        const uint4 v = ag_realign(w0, w1, w.r);
        x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
        c.g = w1;
        c.j = j + 1;
        return;
    }
#else
    (void)w; (void)c;
#endif
    ag_load_block(base + 16 * (uint64_t)j, nvalid, x);
}

#if defined(__CUDA_ARCH__)
// Stores of CONSECUTIVE whole blocks at unaligned addresses by one thread: the granule that holds the tail of
// the previous block and the head of this one leaves with one 128-bit store; only the head of the first block
// and the tail of the last one go out byte by byte (flush).  Writes exactly the bytes of the blocks it is given.
struct AgStoreCarry {
    uint4 prev;
    uint8_t* prev_addr;
    bool have;
    __device__ __forceinline__ void init() { have = false; prev_addr = nullptr; prev = make_uint4(0, 0, 0, 0); }
    __device__ __forceinline__ void flush()
    {
        if (!have) return;
        const uint32_t ro = (uint32_t)((uintptr_t)prev_addr & 15);
        const uint32_t w[4] = {prev.x, prev.y, prev.z, prev.w};
        uint8_t* q = prev_addr + 16 - ro;   // aligned: the last ro bytes of the block
        for (uint32_t j = 16 - ro; j < 16; ++j) q[j - (16 - ro)] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
        have = false;
    }
    // q: unaligned address of this whole block
    __device__ __forceinline__ void put(uint8_t* q, const uint32_t o[4])
    {
        const uint32_t ro = (uint32_t)((uintptr_t)q & 15);
        const uint4 cur = make_uint4(o[0], o[1], o[2], o[3]);
        if (have && prev_addr + 16 == q) {
            *reinterpret_cast<uint4*>(q - ro) = ag_realign(prev, cur, 16 - ro);
        } else {
            flush();
            for (uint32_t j = 0; j < 16 - ro; ++j) q[j] = (uint8_t)(o[j >> 2] >> (8 * (j & 3)));
        }
        prev = cur;
        prev_addr = q;
        have = true;
    }
};
#endif

// ---- single stream: one lane of the grid-wide strided Horner ----------------
struct StreamParams {
    uint32_t rk[60];
    uint32_t iv[3];       // the 12 IV bytes as LE words
    uint32_t ctr0;        // counter of this shard's block 0 = J0 counter + 1 + first_block (mod 2^32; = 2 + first_block
                          // for a 96-bit IV, aes_icb.vhd:100)
    uint32_t j0w;         // counter word of J0 as the AES state holds it (byte-swapped; 0x01000000 for a 96-bit IV)
    uint64_t n_bytes;     // bytes in this shard
    const uint8_t* in;
    uint8_t* out;
    const KeyDev* key;
    const uint32_t* te0;  // 256-entry Te0 in HBM (per context)
    uint32_t* partials;   // gridDim.x x 4 BE words: per-CTA GHASH partial, last block weighted H^1
    // fused tail, run by the last CTA to finish (null done_counter = off)
    uint32_t* done_counter;       // zero before the launch; reset by the kernel
    uint64_t scale_e;             // partial *= H^scale_e (blocks after this shard)
    const uint32_t* scale_pow;    // H^scale_e precomputed by k_pow (4 BE words), or null: compute in the tail
    uint8_t* out16;               // scaled partial in natural byte order (may be null)
    uint32_t fuse_finish;         // also finish the tag (single-shard message, short AAD)
    const uint8_t* aad;
    uint64_t aad_len, ct_len;
    uint8_t* tag_calc;
    const uint8_t* tag_expected;
    uint8_t* ok;
    const uint32_t* hn;           // H^(ct blocks), precomputed (k_pow) or null
    // exchange of the shard partials over peer memory (NVLink): the tail POSTS this rank's scaled
    // partial into slot (peer_epoch % AG_PEER_RING, peer_rank) of every peer's exchange buffer and
    // raises the slot's epoch flag; k_peer_finish (side stream) waits for the world's flags.
    // peer_bufs[w] = rank w's exchange buffer mapped in this process (AG_PEER_* layout)
    uint8_t* const* peer_bufs;
    uint32_t peer_rank, peer_world, peer_epoch;
    // verify-then-release decrypt: the whole grid returns at once, output untouched, when *gate == 0
    const uint8_t* gate;
};

// Exchange buffer of one rank: a ring of AG_PEER_RING epochs x AG_PEER_MAX slots of 16 B written
// by the peers, then the matching 4-byte epoch flags.  A rank posts epoch e only after its own
// finish of epoch e - AG_PEER_AHEAD completed (which proves every peer posted e - AG_PEER_AHEAD,
// hence finished e - 2*AG_PEER_AHEAD): with RING >= 2*AHEAD a slot is never overwritten before
// its reader is done, and a rank runs at most AHEAD messages ahead of the slowest one.
constexpr uint32_t AG_PEER_MAX = 16;
constexpr uint32_t AG_PEER_RING = 8;
constexpr uint32_t AG_PEER_AHEAD = 4;
constexpr uint32_t AG_PEER_FLAGS = AG_PEER_RING * AG_PEER_MAX * 16;
constexpr uint32_t AG_PEER_BYTES = AG_PEER_FLAGS + AG_PEER_RING * AG_PEER_MAX * 4;

#if defined(__CUDA_ARCH__)
// Warp-cooperative store of one WHOLE block per lane at consecutive unaligned addresses (lane l writes q + 16 l, r = q & 15
// != 0, the same for all; `whole`: this lane has such a block).  Byte stores would cost sixteen requests per block; here
// lane l fetches the block of lane l - 1 by shuffle and writes the ALIGNED granule that holds its neighbour's last r bytes
// and its own first 16 - r: one 128-bit store per block.  Only the first lane of a run writes its head, and the last one
// its tail, byte by byte.  Called by all 32 lanes; writes exactly the bytes of the whole blocks.
__device__ __forceinline__ void ag_store_row_coop(uint8_t* dst, const uint32_t o[4], bool whole, uint32_t r)
{
    const uint32_t lane = threadIdx.x & 31;
    uint4 prev;
    prev.x = __shfl_up_sync(0xffffffffu, o[0], 1);
    prev.y = __shfl_up_sync(0xffffffffu, o[1], 1);
    prev.z = __shfl_up_sync(0xffffffffu, o[2], 1);
    prev.w = __shfl_up_sync(0xffffffffu, o[3], 1);
    const bool prev_whole = __shfl_up_sync(0xffffffffu, (int)whole, 1) != 0 && lane > 0;
    const bool next_whole = __shfl_down_sync(0xffffffffu, (int)whole, 1) != 0 && lane < 31;
    if (!whole) return;
    if (prev_whole) {
        *reinterpret_cast<uint4*>(dst - r) = ag_realign(prev, make_uint4(o[0], o[1], o[2], o[3]), 16 - r);
    } else {
        ag_store_block(dst, 16 - r, o);                    // head: the first 16 - r bytes (dst + 16 - r is aligned)
    }
    if (!next_whole) {
        const uint4 t = ag_realign(make_uint4(o[0], o[1], o[2], o[3]), make_uint4(0, 0, 0, 0), 16 - r);
        const uint32_t tw[4] = {t.x, t.y, t.z, t.w};
        ag_store_block(dst + 16 - r, r, tw);               // tail: the last r bytes, at an aligned address
    }
}
#endif

// Returns Y_g for global lane g of Gt lanes; the caller multiplies by H^(Gt-g).
// Block indices fit 32 bits (a counter range holds < 2^32 blocks).
// ALIGNED: `in`/`out` are 16-byte aligned, so every full block moves with one 128-bit
// load/store and only the owner of a ragged last block takes the byte path.
template <int NR, int MODE, bool ALIGNED, class TE, class GH>
AG_HD gf128 ag_stream_lane(const StreamParams& p, uint32_t g, uint32_t Gt, TE&& te, GH&& gh)
{
    const uint32_t n_blocks = (uint32_t)((p.n_bytes + 15) >> 4);
    const uint32_t n_full = (uint32_t)(p.n_bytes >> 4);               // blocks that are whole
    const uint32_t rows = (uint32_t)(((uint64_t)n_blocks + Gt - 1) / Gt);
    const uint32_t pad = (uint32_t)((uint64_t)rows * Gt - n_blocks);   // < Gt
    const uint32_t tail = (uint32_t)(p.n_bytes & 15);                  // bytes in a short last block

    AesCtrConst cc;
    AesCtrCache cache;
    // row 0 may start inside the front padding: i is the block index of this lane in the
    // current row, valid when `have`.
    bool have = rows && g >= pad;
    uint32_t i = g - pad;  // wraps when !have; row 1 then lands on g + Gt - pad
    if (MODE != AG_MODE_GHASH_ONLY) {
        cc = aes_ctr_precompute(p.rk, p.iv[0], p.iv[1], p.iv[2], te);
        aes_ctr_cache_fill(p.rk, cc, ag_bswap32(p.ctr0 + i) ^ p.rk[3], te, cache);
    }

    auto load = [&](uint32_t bi, uint32_t x[4]) {
        const uint8_t* src = p.in + 16 * (uint64_t)bi;
        if (ALIGNED && bi < n_full) {
#if defined(__CUDA_ARCH__)
            const uint4 v = *reinterpret_cast<const uint4*>(src);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
#else
            ag_load_block(src, 16, x);
#endif
        } else {
            ag_load_block_in(src, bi < n_full ? 16u : tail, x, p.in, p.in + p.n_bytes);
        }
    };

    gf128 y = gf_zero();
    uint32_t xn[4] = {0, 0, 0, 0};
#if defined(__CUDA_ARCH__)
    // output at an odd address: the lanes of a warp hold consecutive blocks, so whole blocks leave as aligned granules
    // assembled across neighbouring lanes (ag_store_row_coop) instead of byte by byte
    const uint32_t r_out = (uint32_t)((uintptr_t)p.out & 15);
    // (a word-aligned output does better with four 32-bit stores per block: 460 vs 429 GB/s)
    const bool coop = !ALIGNED && MODE != AG_MODE_GHASH_ONLY && (r_out & 3) != 0;
#endif
    // software prefetch: row u+1's block is requested before row u is processed
    if (have) load(i, xn);
    for (uint32_t u = 0; u < rows; ++u) {
        uint32_t x[4] = {xn[0], xn[1], xn[2], xn[3]};
        if (u + 1 < rows) load(i + Gt, xn);  // rows >= 1 are never padding
        if (MODE != AG_MODE_CTR_ONLY && u) y = gf_mul_table(y, gh);
        uint32_t o[4] = {0, 0, 0, 0};
        bool whole_out = false;   // coop: this lane's whole block is stored after the branch, by the warp together
        if (have) {
            uint32_t s[4];
            if (MODE == AG_MODE_GHASH_ONLY) {
                s[0] = x[0]; s[1] = x[1]; s[2] = x[2]; s[3] = x[3];
            } else {
                uint32_t ks[4];
                aes_ctr_block_cached<NR>(p.rk, cc, cache, p.ctr0 + i, te, ks);
                o[0] = x[0] ^ ks[0]; o[1] = x[1] ^ ks[1]; o[2] = x[2] ^ ks[2]; o[3] = x[3] ^ ks[3];
                uint8_t* dst = p.out + 16 * (uint64_t)i;
                if (ALIGNED && i < n_full) {
#if defined(__CUDA_ARCH__)
                    *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
#else
                    ag_store_block(dst, 16, o);
#endif
                } else {
                    const uint32_t nv = i < n_full ? 16u : tail;
#if defined(__CUDA_ARCH__)
                    if (coop && nv == 16) whole_out = true;
                    else
#endif
                        ag_store_block(dst, nv, o);
                    if (MODE == AG_MODE_ENC && nv != 16) ag_mask_block(o, nv);
                }
                if (MODE == AG_MODE_ENC) {
                    s[0] = o[0]; s[1] = o[1]; s[2] = o[2]; s[3] = o[3];
                } else {
                    s[0] = x[0]; s[1] = x[1]; s[2] = x[2]; s[3] = x[3];
                }
            }
            if (MODE != AG_MODE_CTR_ONLY) {
                y.w[0] ^= ag_bswap32(s[0]);
                y.w[1] ^= ag_bswap32(s[1]);
                y.w[2] ^= ag_bswap32(s[2]);
                y.w[3] ^= ag_bswap32(s[3]);
            }
        }
#if defined(__CUDA_ARCH__)
        if (coop) ag_store_row_coop(p.out + 16 * (uint64_t)i, o, whole_out, r_out);   // all lanes of the warp, every row
#endif
        have = true;
        i += Gt;
    }
    return y;
}

// ---- batched messages: one lane of a G-lane group ----------------------------
struct BatchParams {
    uint32_t rk[60];
    const KeyDev* key;
    const uint32_t* te0;
    const uint8_t* keys;       // per-message raw keys (n_msgs x key_bytes) for k_batch_perkey, else null
    const uint8_t* iv;         // n_msgs x 12 (96-bit IVs), or n_msgs x 16 pre-counter blocks J0 when iv_is_j0
    uint32_t iv_is_j0;         // 1: `iv` holds J0 per message (any IV length, SP 800-38D 7.1; agcm_batch_derive_j0)
    const uint8_t* aad;        // may be null when there is no AAD
    const uint64_t* aad_off;   // n_msgs+1 offsets, or null => uniform (aad_stride, aad_len)
    const uint8_t* in;
    const uint64_t* in_off;    // n_msgs+1 offsets, or null => uniform (stride, len)
    uint8_t* out;              // same offsets as `in`
    uint8_t* tag;              // n_msgs x 16: produced (enc) / expected (dec)
    uint8_t* ok;               // n_msgs, dec only: 1 = authentic
    uint64_t n_msgs;
    uint64_t len, stride, aad_len, aad_stride;  // uniform layout
    // fixed-pitch SLOTS holding messages of different lengths (agcm_batch_crypt_slots): message m is
    // len_arr[m] bytes at m * stride (clamped to the pitch); null => `len` for all.  AAD likewise.
    const uint32_t* len_arr;
    const uint32_t* aad_len_arr;
    // k_batch_cta only: every message is cut into `split` counter-range segments, one CTA each
    // (1 = whole messages); seg_parts holds n_msgs x split scaled partials then n_msgs x E_K(J0)
    uint32_t split;
    uint32_t* seg_parts;
    // k_batch_cta: units (messages or segments) are handed out by this counter (zero at launch);
    // null = static round-robin over the CTAs
    uint32_t* ticket;
    // k_batch, offset batches: the order in which the lane groups take the messages -- sorted by length
    // (longest first) so that the messages a warp works on side by side are equally long; null = 0, 1, 2, ...
    const uint32_t* perm;
    // ... and the slice [range[0], range[1]) of that order this launch works on (device words written by the sort:
    // one launch per length class, each with its own lane-group width); null = all n_msgs
    const uint32_t* range;
    // k_batch_warp (a warp per unit): raw lane accumulators (32 x 16 B per unit id, BE words), unit
    // descriptors {message + 1 (0 = unused id), blocks after the unit}, per-message XOR accumulators
    // and E_K(J0) (n_msgs x 16 B each)
    uint4* seg_acc;
    uint64_t* unit_desc;
    uint32_t* msg_acc;
    uint32_t* msg_cnt;         // units of message m combined so far (the last one writes the tag)
    uint32_t* msg_ej0;
    // uniform batches: static BALANCED partition on two axes -- the AAD blocks of all messages laid end to
    // end, and their payload blocks (+ AG_FINISH_WEIGHT positions per message for the length block and
    // E_K(J0)); warp w owns positions [w*quota_aad, (w+1)*quota_aad) of the first and
    // [w*quota_pt, (w+1)*quota_pt) of the second.  quota_pt == 0: units of `split` segments by ticket.
    uint64_t quota_aad, quota_pt;
    uint64_t n_ids;            // unit ids in use: 2 x (n_warps + n_msgs) (balanced) or n_msgs * split (ticket)
};

// 1 if the computed tag equals the expected one, else 0; every word is compared (no early exit)
AG_HD uint8_t ag_tag_eq(const uint32_t x[4], const uint32_t tg[4])
{
    const uint32_t diff = (x[0] ^ tg[0]) | (x[1] ^ tg[1]) | (x[2] ^ tg[2]) | (x[3] ^ tg[3]);
    return diff ? 0 : 1;
}

// The computed tag of batch message m: decrypt, checked against the expected tag into ok[m]; encrypt, stored
template <bool DEC>
AG_HD void ag_tag_out(const BatchParams& p, uint64_t m, const uint32_t tg[4])
{
    uint8_t* tp = p.tag + 16 * m;
    if (DEC) {
        uint32_t x[4];
        ag_load_block(tp, 16, x);
        p.ok[m] = ag_tag_eq(x, tg);
    } else {
        ag_store_block(tp, 16, tg);
    }
}

// One message, or one counter-range segment of it (ag_batch_segment).
struct MsgDesc {
    const uint8_t* in;
    uint8_t* out;
    const uint8_t* aad;
    uint64_t len, aad_len;              // what THIS unit reads: payload bytes, AAD bytes
    uint64_t total_len, total_aad_len;  // the whole message (the length block, gcm_ghash.vhd:257)
    uint32_t ctr_off;                   // payload block index of the unit's first block (counter = j0ctr + 1 + ctr_off + j)
    uint32_t j0ctr;                     // counter field of J0: 1 for a 96-bit IV (src/aes_icb.vhd:34,99)
    uint32_t last;                      // the unit ends the message: it absorbs the length block and makes E_K(J0)
};

AG_HD MsgDesc ag_batch_msg(const BatchParams& p, uint64_t m)
{
    MsgDesc d;
    uint64_t o, l;
    if (p.in_off) { o = p.in_off[m]; l = p.in_off[m + 1] - o; }
    else { o = m * p.stride; l = p.len_arr ? (p.len_arr[m] < p.stride ? p.len_arr[m] : p.stride) : p.len; }
    d.in = p.in + o;
    d.out = p.out + o;
    d.len = l;
    if (p.aad_off) { o = p.aad_off[m]; l = p.aad_off[m + 1] - o; }
    else { o = m * p.aad_stride; l = p.aad_len_arr ? (p.aad_len_arr[m] < p.aad_stride ? p.aad_len_arr[m] : p.aad_stride) : p.aad_len; }
    d.aad = p.aad ? p.aad + o : nullptr;
    d.aad_len = p.aad ? l : 0;
    d.total_len = d.len;
    d.total_aad_len = d.aad_len;
    d.ctr_off = 0;
    d.j0ctr = 1;
    d.last = 1;
    return d;
}

// Message m's counter-block prefix as three LE words, and (J0 mode) the counter field of its J0.
AG_HD void ag_batch_iv(const BatchParams& p, uint64_t m, uint32_t iv[3], uint32_t* j0ctr)
{
    const uint8_t* ivp = p.iv + (p.iv_is_j0 ? 16 : 12) * m;
    iv[0] = iv[1] = iv[2] = 0;
    for (int j = 0; j < 4; ++j) {
        iv[0] |= (uint32_t)ivp[j] << (8 * j);
        iv[1] |= (uint32_t)ivp[4 + j] << (8 * j);
        iv[2] |= (uint32_t)ivp[8 + j] << (8 * j);
    }
    *j0ctr = p.iv_is_j0 ? (((uint32_t)ivp[12] << 24) | ((uint32_t)ivp[13] << 16) | ((uint32_t)ivp[14] << 8) | (uint32_t)ivp[15]) : 1u;
}

// A unit of work smaller than a message: the part of message w whose WEIGHT positions fall in
// [w0, w1), the single-GPU form of the counter-range shards of parallel.py.  Positions run over the
// unified sequence AAD | CT (so bulk AAD is shared out too) with an AAD block (GHASH only) weighing
// 1 and a payload block (AES + GHASH) 4, followed by AG_FINISH_WEIGHT positions that stand for the
// length block and E_K(J0): the unit whose range reaches the end of them closes the message
// (d.last).  *after = blocks of the unified sequence that follow the unit: its GHASH partial is
// scaled by H^after before the partials of a message are XORed.  AAD and CT are each zero-padded
// to whole blocks by the reference (gcm_ghash.vhd:228-244), so cutting at block boundaries changes
// nothing; adjacent ranges share their boundary block index, so units tile a message exactly.
constexpr uint64_t AG_FINISH_WEIGHT = 8;

AG_HD uint64_t ag_msg_weight(uint64_t aad_len, uint64_t len, uint64_t ptw = 4)
{
    return ((aad_len + 15) >> 4) + ptw * ((len + 15) >> 4) + AG_FINISH_WEIGHT;
}

// ptw = weight of a payload block (an AAD block weighs 1)
AG_HD MsgDesc ag_batch_range(const MsgDesc& w, uint64_t w0, uint64_t w1, uint64_t* after, uint64_t ptw = 4)
{
    const uint64_t a = (w.aad_len + 15) >> 4, n = (w.len + 15) >> 4, tot = a + n, W = a + ptw * n;
    const bool last = w1 >= W + AG_FINISH_WEIGHT;
    if (w0 > W) w0 = W;
    if (w1 > W) w1 = W;
    uint64_t u0 = w0 <= a ? w0 : a + (w0 - a + ptw - 1) / ptw;
    uint64_t u1 = w1 <= a ? w1 : a + (w1 - a + ptw - 1) / ptw;
    if (u0 > tot) u0 = tot;
    if (u1 > tot || last) u1 = tot;
    const uint64_t a0 = u0 < a ? u0 : a, a1 = u1 < a ? u1 : a;          // AAD blocks [a0, a1)
    const uint64_t c0 = (u0 > a ? u0 : a) - a, c1 = (u1 > a ? u1 : a) - a;  // CT blocks [c0, c1)
    MsgDesc d = w;
    d.aad = (a1 > a0) ? w.aad + 16 * a0 : nullptr;
    d.aad_len = (a1 > a0) ? ((a1 == a) ? w.aad_len - 16 * a0 : 16 * (a1 - a0)) : 0;
    d.in = w.in + 16 * c0;
    d.out = w.out + 16 * c0;
    d.len = (c1 > c0) ? ((c1 == n) ? w.len - 16 * c0 : 16 * (c1 - c0)) : 0;
    d.ctr_off = (uint32_t)c0;
    d.last = last ? 1u : 0u;
    *after = last ? 0 : (tot - u1) + 1;
    return d;
}

// Segment `seg` of S equal-WORK segments of message w (the length block and E_K(J0) with segment S-1).
// ptw as in ag_batch_range (1: a tag-only pass, where a payload block costs what an AAD block costs).
AG_HD MsgDesc ag_batch_segment(const MsgDesc& w, uint32_t seg, uint32_t S, uint64_t* after, uint64_t ptw = 4)
{
    const uint64_t a = (w.aad_len + 15) >> 4, n = (w.len + 15) >> 4;
    const uint64_t W = a + ptw * n, per = (W + S - 1) / S;
    uint64_t w0 = (uint64_t)seg * per, w1 = w0 + per;
    if (w0 > W) w0 = W;
    if (w1 > W) w1 = W;
    if (seg == S - 1) w1 = W + AG_FINISH_WEIGHT;
    return ag_batch_range(w, w0, w1, after, ptw);
}

// Lane t of G over the unified sequence [AAD blocks | CT blocks | length block]
// (gcm_ghash.vhd:259-272 order; length block gcm_ghash.vhd:257).  DEC selects the
// GHASH source (aes_gcm.vhd:207-211).  Returns Y_t (weight H^(G-t) still to apply).
// CACHE: AesCtrSeqCache when G is small (a lane's counters are near-consecutive), AesCtrCache when
// G is a multiple of 256 (one CTA per message: the lane's low counter byte never changes).
// An AAD row has no AES pass to hide its load behind, so the AAD block of row u+1 is fetched
// before row u is processed (one row of software prefetch); a payload block is loaded at the top
// of its own row and consumed after the AES rounds.
// SEQ: the lane walks CONSECUTIVE payload blocks (G == 1), so unaligned output can leave granule by granule.
// VERIFY: the tag-only flavour of a decrypt (pass 1 of the verify-then-release batch): payload blocks are absorbed
// like AAD rows -- no keystream, no store -- and only the lane that meets the length block runs AES (E_K(J0)).
template <int NR, bool DEC, bool SEQ = false, bool VERIFY = false, class CACHE, class TE, class GH>
AG_HD gf128 ag_batch_lane(const uint32_t* rk, const AesCtrConst& cc, CACHE& cache, const MsgDesc& d, uint32_t t,
                          uint32_t G, TE&& te, GH&& gh_g, uint32_t ej0[4])
{
    // block counts fit 32 bits (a message is < 2^32 blocks; AAD + payload + 1 likewise)
    const uint32_t a = (uint32_t)((d.aad_len + 15) >> 4), n = (uint32_t)((d.len + 15) >> 4);
    const uint32_t mb = a + n + (d.last ? 1u : 0u);
    const uint32_t rows = (mb + G - 1) / G;
    const uint32_t pad = rows * G - mb;   // < G
    const uint32_t atail = (uint32_t)(d.aad_len & 15), tail = (uint32_t)(d.len & 15);
    const uint32_t a_gh = VERIFY ? a + n : a;   // blocks of the GHASH-only prefix of the unified sequence
    gf128 y = gf_zero();
    uint32_t i = t - pad;                 // wraps while inside the front padding (row 0 only)
    bool have = t >= pad;
    uint32_t nxt[4] = {0, 0, 0, 0};
    // Realigned wide loads only where a lane walks its message alone (SEQ).  For lane groups they were measured too:
    // +3 % on a heavy-tailed packed mix (long messages at odd addresses), but the extra path in the block loop cost
    // every ALIGNED lane-group batch about 1 % (1500 B records, G = 2: 536 vs 529 GB/s) -- not kept.
    const AgWideWindow win_aad = SEQ ? AgWideWindow::make(d.aad, d.aad ? d.aad_len : 0) : AgWideWindow{0, 0};
    const AgWideWindow win_in = SEQ ? AgWideWindow::make(d.in, d.len) : AgWideWindow{0, 0};
    AgLoadCarry lc_aad, lc_in;
    lc_aad.j = lc_in.j = 0xFFFFFFFFu;
    lc_aad.g = lc_in.g = make_uint4(0, 0, 0, 0);
#if defined(__CUDA_ARCH__)
    AgStoreCarry carry;
    carry.init();
    const bool wide_st = SEQ && (((uintptr_t)d.out & 15) != 0);
#endif
    // block i < a_gh of the GHASH-only prefix: an AAD block or (VERIFY) a payload block
#define AG_LOAD_GH(i, x)                                                                                                 \
    if constexpr (VERIFY) {                                                                                              \
        if ((i) >= a) ag_load_block_win<SEQ>(d.in, (i) - a, ((i) == a + n - 1 && tail) ? tail : 16u, x, win_in, lc_in);    \
        else ag_load_block_win<SEQ>(d.aad, (i), ((i) == a - 1 && atail) ? atail : 16u, x, win_aad, lc_aad);             \
    } else ag_load_block_win<SEQ>(d.aad, (i), ((i) == a - 1 && atail) ? atail : 16u, x, win_aad, lc_aad)
    if (rows && have && i < a_gh) { AG_LOAD_GH(i, nxt); }
    // Rows 0 .. aad_rows-1 hold AAD blocks only (row u spans blocks uG-pad .. uG+G-1-pad): they run in
    // a loop of their own -- prefetch, one table product, one XOR, like k_stream<GHASH_ONLY> -- so
    // that bulk AAD is not dragged through the AES-sized body of the general loop below.
    const uint32_t aad_rows = (uint32_t)(((uint64_t)a_gh + pad) / G);
    uint32_t u = 0;
#if defined(__CUDA_ARCH__)
    // 16-byte aligned AAD: whole blocks move with one 128-bit load each, TWO rows ahead of the product
    // that consumes them (a GHASH-only row is short: one row of prefetch does not cover a DRAM round trip)
    // (VERIFY: any alignment -- the prefix spans two buffers, and ag_load_block_win picks the access per block)
    if (aad_rows > 2 && (VERIFY || ((uintptr_t)d.aad & 15) == 0)) {
        const uint32_t a_full = (uint32_t)(d.aad_len >> 4);   // blocks below this index are whole
        auto ldq = [&](uint32_t bi) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if constexpr (VERIFY) {
                if (bi < a_gh) {
                    uint32_t x[4];
                    AG_LOAD_GH(bi, x);
                    v = make_uint4(x[0], x[1], x[2], x[3]);
                }
            } else if (bi < a_full) {
                v = *reinterpret_cast<const uint4*>(d.aad + 16 * (uint64_t)bi);
            } else if (bi < a) {
                uint32_t x[4];
                ag_load_block(d.aad + 16 * (uint64_t)bi, atail, x);
                v = make_uint4(x[0], x[1], x[2], x[3]);
            }
            return v;
        };
        uint4 q1 = ldq(i + G);   // row 1 (rows >= 1 never touch the front padding)
        for (; u < aad_rows; ++u) {
            const bool hv = have;
            const uint32_t s0 = nxt[0], s1 = nxt[1], s2 = nxt[2], s3 = nxt[3];
            nxt[0] = q1.x; nxt[1] = q1.y; nxt[2] = q1.z; nxt[3] = q1.w;
            i += G;
            have = true;
            q1 = ldq(i + G);   // two rows ahead; past the AAD it returns zeros that are never used
            if (u) y = gf_mul_table(y, gh_g);
            if (hv) {
                y.w[0] ^= ag_bswap32(s0);
                y.w[1] ^= ag_bswap32(s1);
                y.w[2] ^= ag_bswap32(s2);
                y.w[3] ^= ag_bswap32(s3);
            }
        }
        // hand over to the general loop with its one-row prefetch: nxt holds row aad_rows' AAD block (if it is one)
        if (!(u < rows && i < a_gh)) { nxt[0] = nxt[1] = nxt[2] = nxt[3] = 0; }
    }
#endif
    for (; u < aad_rows; ++u) {
        const bool hv = have;
        const uint32_t s0 = nxt[0], s1 = nxt[1], s2 = nxt[2], s3 = nxt[3];
        i += G;
        have = true;
        if (u + 1 < rows && i < a_gh) { AG_LOAD_GH(i, nxt); }
        if (u) y = gf_mul_table(y, gh_g);
        if (hv) {
            y.w[0] ^= ag_bswap32(s0);
            y.w[1] ^= ag_bswap32(s1);
            y.w[2] ^= ag_bswap32(s2);
            y.w[3] ^= ag_bswap32(s3);
        }
    }
    for (; u < rows; ++u) {
        const uint32_t ic = i;
        const bool hv = have;
        uint32_t s[4] = {nxt[0], nxt[1], nxt[2], nxt[3]};
        i += G;
        have = true;
        if (u + 1 < rows && i < a_gh) { AG_LOAD_GH(i, nxt); }
        if (u) y = gf_mul_table(y, gh_g);
        if (!hv) continue;
        if (ic >= a_gh) {
            // The length block always lands on lane G-1 of the last row.  That lane has no payload
            // block in this row, so it spends the row's AES pass on E_K(J0) (counter 1,
            // src/aes_icb.vhd:34,99): the tag mask costs no pass of its own.  (VERIFY: past the
            // GHASH-only prefix there is nothing but the length block.)
            const bool is_len = VERIFY || (d.last && (ic == a + n));
            const uint32_t j = ic - a;
            const uint32_t nv = (j == n - 1 && tail) ? tail : 16u;
            uint32_t x[4] = {0, 0, 0, 0};
            if (!is_len) ag_load_block_win<SEQ>(d.in, j, nv, x, win_in, lc_in);   // in flight during the AES rounds
            uint32_t ks[4];
            aes_ctr_block_auto<NR>(rk, cc, cache, is_len ? d.j0ctr : d.j0ctr + 1u + d.ctr_off + j, te, ks);   // inc32: wraps mod 2^32
            if (is_len) {
                ej0[0] = ks[0]; ej0[1] = ks[1]; ej0[2] = ks[2]; ej0[3] = ks[3];
                // [len(A)]64 || [len(C)]64 in bits, big-endian (gcm_ghash.vhd:257)
                const uint64_t ab = d.total_aad_len * 8, cb = d.total_len * 8;
                y.w[0] ^= (uint32_t)(ab >> 32);
                y.w[1] ^= (uint32_t)ab;
                y.w[2] ^= (uint32_t)(cb >> 32);
                y.w[3] ^= (uint32_t)cb;
                continue;
            }
            uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
#if defined(__CUDA_ARCH__)
            if (wide_st && nv == 16) {
                carry.put(d.out + 16 * (uint64_t)j, o);
            } else {
                if (SEQ) carry.flush();
                ag_store_block(d.out + 16 * (uint64_t)j, nv, o);
            }
#else
            ag_store_block(d.out + 16 * (uint64_t)j, nv, o);
#endif
            if (DEC) {
                s[0] = x[0]; s[1] = x[1]; s[2] = x[2]; s[3] = x[3];
            } else {
                if (nv != 16) ag_mask_block(o, nv);
                s[0] = o[0]; s[1] = o[1]; s[2] = o[2]; s[3] = o[3];
            }
        }
        y.w[0] ^= ag_bswap32(s[0]);
        y.w[1] ^= ag_bswap32(s[1]);
        y.w[2] ^= ag_bswap32(s[2]);
        y.w[3] ^= ag_bswap32(s[3]);
    }
#if defined(__CUDA_ARCH__)
    if (SEQ) carry.flush();
#endif
#undef AG_LOAD_GH
    return y;
}

// ---- pass 2 of the verify-then-release batch: GCTR gated by the ok flags of pass 1 ---------------
// Counter mode needs no per-message combine, so the payload blocks of the whole batch are cut FLAT into slots, and
// neighbouring threads take neighbouring slots -- neighbouring blocks of one record, so that 128-bit accesses
// coalesce without any staging.  A message whose ok[m] is 0 is skipped: its output range is never written.
//   uniform / slots: slot s = block s % bpr of message s / bpr (bpr = blocks per record pitch); slot blocks past
//                    the message's length are skipped;
//   offsets:         slot s = the bytes [in_off[0] + 16 s, + 16) of the input: it owns every block whose first byte
//                    lies there (at most one per message; several when messages are shorter than a block).
constexpr uint32_t AG_GATED_ROWS = 8;   // slots per lane and warp chunk (a warp works 32 x AG_GATED_ROWS slots)

// First message of an offset batch that ends past input byte in_off[0] + 16 s (n_msgs if none): binary search.
AG_HD uint64_t ag_gated_first_msg(const BatchParams& p, uint64_t s)
{
    const uint64_t lo = p.in_off[0] + 16 * s;
    uint64_t l = 0, h = p.n_msgs;   // answer in [l, h]
    while (l < h) {
        const uint64_t mid = l + ((h - l) >> 1);
        if (p.in_off[mid + 1] <= lo) l = mid + 1;
        else h = mid;
    }
    return l;
}

// Block j of message m (payload at byte offset off of in / out, len bytes), if ok[m] says so.
template <int NR, class TE>
AG_HD void ag_gated_ctr_block(const BatchParams& p, uint64_t m, uint32_t j, uint64_t off, uint64_t len, TE&& te)
{
    if (p.ok[m] == 0) return;
    uint32_t iv[3], j0ctr;
    ag_batch_iv(p, m, iv, &j0ctr);
    const uint64_t left = len - 16 * (uint64_t)j;
    const uint32_t nv = left < 16 ? (uint32_t)left : 16u;
    uint32_t x[4], ks[4];
    ag_load_block(p.in + off + 16 * (uint64_t)j, nv, x);
    aes_rounds_from<1, NR>(p.rk, iv[0] ^ p.rk[0], iv[1] ^ p.rk[1], iv[2] ^ p.rk[2], ag_bswap32(j0ctr + 1u + j) ^ p.rk[3], te,
                           ks);   // inc32: wraps mod 2^32
    const uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
    ag_store_block(p.out + off + 16 * (uint64_t)j, nv, o);   // nv < 16: exactly the message's last bytes
}

// Slot s.  m: offsets form only -- a message index at or before the slot's first one (from ag_gated_first_msg or the
// lane's previous slot); advanced past the messages that end before the slot.
template <int NR, class TE>
AG_HD void ag_gated_ctr_slot(const BatchParams& p, uint64_t s, uint64_t bpr, uint64_t& m, TE&& te)
{
    if (p.in_off) {
        const uint64_t lo = p.in_off[0] + 16 * s, hi = lo + 16;
        while (m < p.n_msgs && p.in_off[m + 1] <= lo) ++m;
        for (uint64_t q = m; q < p.n_msgs; ++q) {
            const uint64_t o0 = p.in_off[q], o1 = p.in_off[q + 1];
            if (o0 >= hi) break;
            const uint64_t j = lo > o0 ? (lo - o0 + 15) >> 4 : 0;   // the message's block that starts in [lo, hi)
            const uint64_t b = o0 + 16 * j;
            if (b < hi && b < o1) ag_gated_ctr_block<NR>(p, q, (uint32_t)j, o0, o1 - o0, te);
        }
        return;
    }
    const uint64_t mm = ((s | bpr) >> 32) ? s / bpr : (uint64_t)((uint32_t)s / (uint32_t)bpr);
    const uint32_t j = (uint32_t)(s - mm * bpr);
    const uint64_t len = p.len_arr ? (p.len_arr[mm] < p.stride ? p.len_arr[mm] : p.stride) : p.len;
    if (16 * (uint64_t)j < len) ag_gated_ctr_block<NR>(p, mm, j, mm * p.stride, len, te);
}

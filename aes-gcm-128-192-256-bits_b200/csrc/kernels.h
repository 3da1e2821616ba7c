// Internal launcher interface between the kernel translation units (kernels*.cu) and capi.cu (not installed).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "gcm_core.cuh"

// Tag finish (gcm_ghash.vhd:257,293 + tb/gcm_model.py:33-51); see k_stream_finish.
struct FinishParams {
    uint32_t rk[60];
    uint32_t nr;
    uint32_t iv[3];
    uint32_t j0w;                 // counter word of J0, byte-swapped (0x01000000 for a 96-bit IV)
    const KeyDev* key;
    const uint32_t* te0;
    const uint8_t* parts;         // n_parts x 16 B in natural GHASH byte order
    uint32_t n_parts;
    const uint8_t* aad;           // null: no AAD, or AAD already folded into parts
    uint64_t aad_len;             // true AAD length (length block)
    uint64_t ct_len;
    uint8_t* tag_calc;            // 16 B out, always written
    const uint8_t* tag_expected;  // 16 B in (decrypt) or null
    uint8_t* ok;                  // 1 B out (decrypt) or null
    const uint32_t* hn;           // H^(ct blocks) from k_pow, or null
};

// Tag finish of a sharded message whose partials arrive over peer memory (k_peer_finish).
struct PeerFinishParams {
    FinishParams f;               // parts / n_parts unused
    uint8_t* const* peer_bufs;    // device array: rank w's exchange buffer mapped in this process
    uint32_t rank, world, epoch;
    uint64_t timeout_ns;          // give up (fail closed) when a peer's flag is this late
    uint32_t* status_dev;         // set to 1 on timeout
    volatile uint32_t* status_host;  // same, in mapped pinned host memory (read by the next call without a sync)
};

cudaError_t ag_launch_stream(const StreamParams& p, int nr, int mode, int ncta, int nt, cudaStream_t st);
cudaError_t ag_launch_batch(const BatchParams& p, int nr, int decrypt, int g, int ncta, int nt, cudaStream_t st);
// k_batch_tile: fixed-size records as a 2-D tensor [message][byte], staged by TMA
struct TileParams {
    BatchParams b;
    CUtensorMap tm_in, tm_out;   // box {32 bytes, 32 messages}, CU_TENSOR_MAP_SWIZZLE_32B
    CUtensorMap tm_aad;          // the AAD records as a tensor of their own (k_batch_tile, when aad_tiled)
    uint32_t aad_tiled;
    uint32_t* ticket;            // zero at launch: next group of 32 messages
};
constexpr uint32_t AG_TILE_BOX_BYTES = 32, AG_TILE_BOX_MSGS = 32;
// gather = 1: rows named one by one (tile::gather4 / scatter4; tensor maps with box {32 bytes, 1 message}), messages
// of different lengths in fixed-pitch slots, taken in the order b.perm
cudaError_t ag_launch_batch_tile(const TileParams& p, int nr, int decrypt, int gather, int ncta, cudaStream_t st);
cudaError_t ag_launch_batch_perkey_tile(const TileParams& p, int nr, int decrypt, int max_cta, cudaStream_t st);
// k_batch_warp, units combined in the same launch (p.split, p.seg_acc, p.unit_desc, p.msg_*, p.ticket set)
cudaError_t ag_launch_batch_warp(const BatchParams& p, int nr, int decrypt, int ncta, cudaStream_t st);
// counting sort of a ragged batch by message length (longest first): perm[n_msgs], scratch hist[4096], and the
// [start, end) slices of the order that hold the long / medium / short messages (ranges6)
cudaError_t ag_launch_len_sort(const BatchParams& p, uint32_t* hist4096, uint32_t* ranges6, uint32_t* perm, cudaStream_t st);
cudaError_t ag_launch_batch_cta(const BatchParams& p, int nr, int decrypt, int ncta, int nt, cudaStream_t st);
// decrypt == 2: verify-then-release (k_batch_perkey_verified: the payload is written only where the tag matched)
cudaError_t ag_launch_batch_perkey(const BatchParams& p, int nr, int decrypt, int max_cta, cudaStream_t st);
// verify-then-release batch decrypt under the shared key: pass 1 = the tag-only flavour of k_batch (lane groups of g) or
// k_batch_warp (writes ok[] only); pass 2 = k_batch_ctr_gated over n_slots flat slots (bpr: blocks per record pitch of
// the uniform / slots forms; both unused for offsets), which writes only the messages whose ok[m] is 1
cudaError_t ag_launch_batch_verify(const BatchParams& p, int nr, int g, int ncta, int nt, cudaStream_t st);
cudaError_t ag_launch_batch_warp_verify(const BatchParams& p, int nr, int ncta, cudaStream_t st);
cudaError_t ag_launch_batch_ctr_gated(const BatchParams& p, int nr, uint64_t n_slots, uint64_t bpr, int max_cta, cudaStream_t st);
cudaError_t ag_launch_key_expand(const uint8_t* keys, uint64_t n_keys, int key_bytes, const uint32_t* te0,
                                 uint8_t* round_keys, cudaStream_t st);
// The key as k_key_setup takes it: raw key bytes, or the Nr+1 pre-expanded stages, as LE words.
struct KeyIn {
    uint32_t w[60];
    uint32_t key_bytes;     // 16 / 24 / 32 (raw key length; unused when pre_expanded)
    uint32_t nr;            // 10 / 12 / 14
    uint32_t pre_expanded;  // w holds 4*(nr+1) stage-key words, used as they are
};
cudaError_t ag_launch_key_setup(KeyDev* kd, const KeyIn& in, const uint32_t* te0, int nt_stream, int ncta,
                                cudaStream_t st);
cudaError_t ag_launch_pow(const KeyDev* kd, uint64_t e, uint32_t* out4, cudaStream_t st);
cudaError_t ag_launch_finish(const FinishParams& p, cudaStream_t st);
cudaError_t ag_launch_peer_finish(const PeerFinishParams& p, cudaStream_t st);
cudaError_t ag_preload_peer_kernels();
cudaError_t ag_launch_peer_post(uint8_t* const* peer_bufs, uint32_t rank, uint32_t world, uint32_t epoch,
                                const uint8_t* partial16, cudaStream_t st);
cudaError_t ag_launch_batch_j0(const KeyDev* kd, const uint8_t* iv, const uint64_t* iv_off, uint64_t iv_len, uint64_t n,
                               uint8_t* j0, cudaStream_t st);
cudaError_t ag_launch_xor_parts(const uint8_t* parts16, uint32_t n, uint8_t* out16, cudaStream_t st);
size_t ag_smem_bytes();

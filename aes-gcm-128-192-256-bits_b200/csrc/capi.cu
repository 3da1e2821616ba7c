// C ABI of the engine (include/aesgcm_b200.h).  Host-side glue only: argument
// checks, kernel parameter blocks, scratch buffers, and the chunked
// host<->device pipeline.  All arithmetic happens in the kernels (kernels*.cu); there is no
// CPU implementation of the datapath in this library.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <vector>

#include "../../include/aesgcm_b200.h"
#include "kernels.h"
#include "host_sched.h"

namespace {

constexpr int kSlots = 3;
constexpr size_t kChunkBytesMax = 64u << 20;  // host pipeline granule (upper bound; AGCM_CHUNK_MB tunes it)
constexpr size_t kMaxChunks = 8192;
constexpr uint64_t kAadInlineMax = 4096;   // bytes of AAD folded inside k_stream_finish
constexpr uint64_t kMaxBlocks = 0xFFFFFFFEull;

// scratch layout (bytes) inside ctx->d_scratch
constexpr size_t SC_PART_CT = 0;     // 16
constexpr size_t SC_TAGCALC = 32;    // 16
constexpr size_t SC_OK = 48;         // 1
constexpr size_t SC_TAG = 64;        // 16 (host API)
constexpr size_t SC_J0 = 80;         // 16: J0 of a non-96-bit IV
constexpr size_t SC_KEY = 96;        // 32 raw key upload
constexpr size_t SC_PARTS = 256;     // list of 16 B partials for finish (user parts + AAD part)
constexpr size_t SC_PARTS_MAX = 1024;
constexpr size_t SC_BYTES = SC_PARTS + 16 * (SC_PARTS_MAX + 1);

// device buffer grown on demand (grow()): the capacity only grows, and the contents are not preserved
template <class T>
struct GrownBuf {
    T* p = nullptr;
    size_t cap = 0;   // bytes
};

// A power of H cached on the device.  It is produced asynchronously by k_pow on whichever stream asked
// first; a later consumer on a DIFFERENT stream (a user stream, the library's pipeline or side streams)
// must not read it before that launch ran.
struct PowCache {
    uint32_t* d = nullptr;       // 4 BE words
    uint64_t e = ~0ull;          // exponent it was computed for (~0 = none)
    cudaEvent_t ev = nullptr;    // recorded after the producing launch
    cudaStream_t st = nullptr;   // the producer's stream
};

}  // namespace

struct agcm_ctx {
    int device = 0, sm_count = 0, ncta = 0, nt = 0;
    uint32_t* d_te0 = nullptr;
    KeyDev* d_key = nullptr;
    uint32_t* d_parts = nullptr;  // 2 x AG_MAX_CTA x 4 words: [0] CT partials, [1] AAD partials
    GrownBuf<uint32_t> seg_parts;    // split batch layouts: segment partials and unit scratch
    uint8_t* d_scratch = nullptr;
    uint32_t* d_counters = nullptr;  // last-CTA tickets: [0] context scratch, [1+s] pipeline slot s
    PowCache pow_n;                  // H^n for the tag finish
    PowCache pow_scale;              // H^blocks_after of the last shard call
    uint32_t j0ctr = 1;              // counter field of J0 for the call in progress (1 for a 96-bit IV)
    GrownBuf<uint8_t> iv_stage;      // padded long IV for the J0 derivation
    // peer-memory exchange (multi-GPU)
    uint8_t** d_peer_bufs = nullptr; // device array of world pointers
    uint32_t* d_peer_status = nullptr;
    uint32_t* h_peer_status = nullptr;   // mapped pinned word raised by k_peer_finish on a timeout
    int peer_rank = 0, peer_world = 0;
    uint32_t peer_epoch = 0;             // exchanges issued so far
    uint64_t peer_timeout_ns = 10000000000ull;   // 10 s (AGCM_PEER_TIMEOUT_MS)
    cudaStream_t peer_side = nullptr;    // the finishes wait for the world's flags here, off the caller's stream
    cudaEvent_t peer_bulk_ev[AG_PEER_RING] = {};
    cudaEvent_t peer_fin_ev[AG_PEER_RING] = {};
    uint32_t h_rk[60];
    uint8_t h_H[16];
    uint8_t h_key_in[240];           // the key as it was loaded, to recognise a reload of the same key
    size_t key_in_len = 0;
    int key_in_mode = 0, key_in_pre = 0;
    int nr = 0;
    bool key_set = false;
    cudaError_t last_err = cudaSuccess;
    uint64_t launches = 0;
    // optional per-launch timing of the dominant kernel (bench.py roofline)
    bool timing = false;
    static constexpr int kTimingRing = 64;
    cudaEvent_t tev[2 * kTimingRing] = {};
    int tev_pending = 0;
    double t_total_ms = 0.0;
    uint64_t t_count = 0;
    // host pipeline (lazy)
    cudaStream_t hs[kSlots] = {nullptr, nullptr, nullptr};
    uint8_t* d_stage[kSlots] = {nullptr, nullptr, nullptr};
    uint8_t* d_stage_aux[kSlots] = {nullptr, nullptr, nullptr};  // iv / aad / tag / ok for batch chunks
    uint32_t* d_stage_parts[kSlots] = {nullptr, nullptr, nullptr};
    uint8_t* d_chunk_partials = nullptr;
    GrownBuf<uint8_t> aad_stage;         // host-supplied AAD
    uint32_t* d_tile_ticket = nullptr;   // k_batch_tile / _warp / _cta: next unit (zeroed before each launch)
    bool no_ticket = false;              // set while the host batch pipeline runs chunks on several streams at once
    GrownBuf<uint32_t> sort;             // length sort of an offset batch: 4096 bucket counters, then perm[n_msgs]
    void* tmap_encode = nullptr;         // cuTensorMapEncodeTiled, resolved through the runtime (no link-time libcuda)
    GrownBuf<uint8_t> verify;            // whole ciphertext of a verify-then-release host decrypt
    bool pipeline_ready = false;
    size_t chunk_bytes = 32u << 20;
    size_t ramp_base = 1u << 20;         // first and last granule of the host pipeline (host_sched.h)
};

namespace {

int cuda_fail(agcm_ctx* c, cudaError_t e)
{
    if (c) c->last_err = e;
    return AGCM_E_CUDA;
}

#define AG_CUDA(ctx, call)                              \
    do {                                                \
        cudaError_t _e = (call);                        \
        if (_e != cudaSuccess) return cuda_fail(ctx, _e); \
    } while (0)

int mode_to_nr(int mode)
{
    switch (mode) {
        case 128: return 10;
        case 192: return 12;
        case 256: return 14;
    }
    return 0;
}

void iv_words(const uint8_t iv[12], uint32_t w[3])
{
    for (int i = 0; i < 3; ++i)
        w[i] = (uint32_t)iv[4 * i] | ((uint32_t)iv[4 * i + 1] << 8) | ((uint32_t)iv[4 * i + 2] << 16) |
               ((uint32_t)iv[4 * i + 3] << 24);
}

// fold finished (event pair) timings of the stream kernel into the running total
int timing_drain(agcm_ctx* c)
{
    for (int i = 0; i < c->tev_pending; ++i) {
        AG_CUDA(c, cudaEventSynchronize(c->tev[2 * i + 1]));
        float ms = 0.f;
        AG_CUDA(c, cudaEventElapsedTime(&ms, c->tev[2 * i], c->tev[2 * i + 1]));
        c->t_total_ms += ms;
        c->t_count++;
    }
    c->tev_pending = 0;
    return AGCM_OK;
}

template <class T>
int grow(agcm_ctx* c, GrownBuf<T>& b, size_t need)
{
    if (need <= b.cap) return AGCM_OK;
    AG_CUDA(c, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    AG_CUDA(c, cudaMalloc(&b.p, need));
    b.cap = need;
    return AGCM_OK;
}

// c->d_tile_ticket with its first `words` words zeroed on `st` (allocated on first use)
int zeroed_ticket(agcm_ctx* c, size_t words, cudaStream_t st, uint32_t*& ticket)
{
    if (!c->d_tile_ticket) AG_CUDA(c, cudaMalloc(&c->d_tile_ticket, 4 * sizeof(uint32_t)));
    AG_CUDA(c, cudaMemsetAsync(c->d_tile_ticket, 0, words * sizeof(uint32_t), st));
    ticket = c->d_tile_ticket;
    return AGCM_OK;
}

// H^e in `pc` for a consumer on `st`: waits for the cached value's producer, and runs k_pow on `st` for a new exponent
int pow_get(agcm_ctx* c, PowCache& pc, uint64_t e, cudaStream_t st)
{
    if (pc.ev && pc.st != st) AG_CUDA(c, cudaStreamWaitEvent(st, pc.ev, 0));
    if (pc.e == e) return AGCM_OK;
    AG_CUDA(c, ag_launch_pow(c->d_key, e, pc.d, st));
    c->launches++;
    pc.e = e;
    if (!pc.ev) AG_CUDA(c, cudaEventCreateWithFlags(&pc.ev, cudaEventDisableTiming));
    AG_CUDA(c, cudaEventRecord(pc.ev, st));
    pc.st = st;
    return AGCM_OK;
}

// the caller's stream waits for every peer finish issued so far (they may still read pow_n)
int peer_join_stream(agcm_ctx* c, cudaStream_t st)
{
    if (c->peer_epoch && c->peer_fin_ev[0]) AG_CUDA(c, cudaStreamWaitEvent(st, c->peer_fin_ev[c->peer_epoch % AG_PEER_RING], 0));
    return AGCM_OK;
}

// H^n for the tag finish, computed once per (key, n) on the caller's stream
int ensure_pow(agcm_ctx* c, uint64_t n_blocks, cudaStream_t st)
{
    if (c->pow_n.e != n_blocks) {
        int rc = peer_join_stream(c, st);   // a deferred finish of an earlier message may still read the old power
        if (rc) return rc;
    }
    return pow_get(c, c->pow_n, n_blocks, st);   // ... and so may a consumer ordered after the old producer
}

// Fields all three forms of the tag finish share.  On decrypt the computed tag goes to scratch, never to the caller.
FinishParams finish_params(const agcm_ctx* c, int decrypt, const uint8_t iv[12], const uint8_t* d_aad, uint64_t aad_len,
                           uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok, const uint32_t* hn)
{
    FinishParams f;
    memset(&f, 0, sizeof(f));
    memcpy(f.rk, c->h_rk, sizeof(f.rk));
    f.nr = (uint32_t)c->nr;
    iv_words(iv, f.iv);
    f.j0w = __builtin_bswap32(c->j0ctr);
    f.key = c->d_key;
    f.te0 = c->d_te0;
    f.aad = d_aad;
    f.aad_len = aad_len;
    f.ct_len = ct_len;
    f.tag_calc = decrypt ? c->d_scratch + SC_TAGCALC : d_tag;
    f.tag_expected = decrypt ? d_tag : nullptr;
    f.ok = decrypt ? d_ok : nullptr;
    f.hn = hn;
    return f;
}

// GHASH partial of `n_bytes` at d_in (optionally also CTR) -> 16 B at d_partial16,
// scaled by H^blocks_after; the fold of the per-CTA partials runs in the last CTA of
// the same launch.  parts_raw: per-CTA scratch (AG_MAX_CTA x 4 words); counter: its ticket.
// ff: the tag finish fused into the same launch (single-shard message, short AAD).
int run_stream(agcm_ctx* c, int mode, const uint8_t iv[12], uint64_t first_block, const uint8_t* d_in, uint8_t* d_out,
               uint64_t n_bytes, uint64_t blocks_after, uint32_t* parts_raw, uint8_t* d_partial16, cudaStream_t st,
               uint32_t* counter, const FinishParams* ff = nullptr, uint32_t peer_epoch = 0, const uint8_t* gate = nullptr)
{
    if (n_bytes == 0) {
        if (d_partial16) AG_CUDA(c, cudaMemsetAsync(d_partial16, 0, 16, st));
        return AGCM_OK;
    }
    StreamParams p;
    memset(&p, 0, sizeof(p));
    memcpy(p.rk, c->h_rk, sizeof(p.rk));
    iv_words(iv, p.iv);
    p.ctr0 = (uint32_t)(c->j0ctr + 1 + first_block);   // inc32 from J0 (2 + first_block for a 96-bit IV)
    p.j0w = __builtin_bswap32(c->j0ctr);
    p.n_bytes = n_bytes;
    p.in = d_in;
    p.out = d_out;
    p.key = c->d_key;
    p.te0 = c->d_te0;
    p.partials = parts_raw;
    p.gate = gate;
    if (mode != AG_MODE_CTR_ONLY) {
        p.done_counter = counter;
        p.scale_e = blocks_after;
        // a shard of a long stream is called again and again with the same exponent (every
        // step of a sharded job): H^blocks_after is computed once per (key, exponent) by k_pow on
        // this stream instead of seven dependent products in the tail of every launch.  The
        // host-pipeline chunks (their own streams, a different exponent each) compute it in the tail.
        if (blocks_after && counter == c->d_counters && mode != AG_MODE_GHASH_ONLY) {
            if (!c->pow_scale.d) AG_CUDA(c, cudaMalloc(&c->pow_scale.d, 16));
            int rc = pow_get(c, c->pow_scale, blocks_after, st);
            if (rc) return rc;
            p.scale_pow = c->pow_scale.d;
        }
        p.out16 = d_partial16;
        if (ff) {
            p.fuse_finish = 1;
            p.aad = ff->aad;
            p.aad_len = ff->aad_len;
            p.ct_len = ff->ct_len;
            p.tag_calc = ff->tag_calc;
            p.tag_expected = ff->tag_expected;
            p.ok = ff->ok;
            p.hn = ff->hn;
        }
        if (peer_epoch) {   // post the scaled partial to every rank (k_peer_finish does the rest)
            p.peer_bufs = c->d_peer_bufs;
            p.peer_rank = (uint32_t)c->peer_rank;
            p.peer_world = (uint32_t)c->peer_world;
            p.peer_epoch = peer_epoch;
        }
    }
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (c->timing) {
        if (c->tev_pending == agcm_ctx::kTimingRing) {
            int rc = timing_drain(c);
            if (rc) return rc;
        }
        ev0 = c->tev[2 * c->tev_pending];
        ev1 = c->tev[2 * c->tev_pending + 1];
        AG_CUDA(c, cudaEventRecord(ev0, st));
    }
    // An input of at most one grid row (blocks <= ncta * nt) needs only the CTAs its blocks land in:
    // the lane and CTA weights are relative to the launched grid, and the row constant H^(nt*ncta)
    // is never applied.  A short message then pays for filling one CTA's tables, not 148.
    int ncta = c->ncta;
    const uint64_t blocks = (n_bytes + 15) >> 4;
    if (blocks <= (uint64_t)c->ncta * (uint64_t)c->nt) ncta = (int)((blocks + (uint64_t)c->nt - 1) / (uint64_t)c->nt);
    AG_CUDA(c, ag_launch_stream(p, c->nr, mode, ncta, c->nt, st));
    c->launches++;
    if (c->timing) {
        AG_CUDA(c, cudaEventRecord(ev1, st));
        c->tev_pending++;
    }
    return AGCM_OK;
}

// parts16: device list of n_parts partials (natural byte order), may live anywhere.
int run_finish(agcm_ctx* c, int decrypt, const uint8_t iv[12], const uint8_t* d_parts16, int n_parts, const uint8_t* d_aad,
               uint64_t aad_len, uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok, cudaStream_t st)
{
    if (n_parts < 0 || (size_t)n_parts > SC_PARTS_MAX) return AGCM_E_BAD_ARG;
    if (decrypt && (!d_tag || !d_ok)) return AGCM_E_BAD_ARG;
    if (!decrypt && !d_tag) return AGCM_E_BAD_ARG;
    const uint64_t n_ct_blocks = (ct_len + 15) >> 4;
    if (n_ct_blocks > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
    const uint8_t* parts = d_parts16;
    int np = n_parts;
    const uint8_t* aad_inline = (aad_len && d_aad) ? d_aad : nullptr;
    if (aad_len && !d_aad) return AGCM_E_BAD_ARG;
    if (aad_len > kAadInlineMax) {
        // bulk AAD: same grid-wide Horner in GHASH-only mode, weighted by H^(n_ct_blocks)
        uint8_t* list = c->d_scratch + SC_PARTS;
        if (n_parts) AG_CUDA(c, cudaMemcpyAsync(list, d_parts16, 16 * (size_t)n_parts, cudaMemcpyDeviceToDevice, st));
        int rc = run_stream(c, AG_MODE_GHASH_ONLY, iv, 0, d_aad, nullptr, aad_len, n_ct_blocks,
                            c->d_parts + 4 * AG_MAX_CTA, list + 16 * (size_t)n_parts, st, c->d_counters);
        if (rc) return rc;
        parts = list;
        np = n_parts + 1;
        aad_inline = nullptr;
    }
    if (aad_inline) {
        int rc = ensure_pow(c, n_ct_blocks, st);
        if (rc) return rc;
    }
    FinishParams f = finish_params(c, decrypt, iv, aad_inline, aad_len, ct_len, d_tag, d_ok, aad_inline ? c->pow_n.d : nullptr);
    f.parts = parts;
    f.n_parts = (uint32_t)np;
    AG_CUDA(c, ag_launch_finish(f, st));
    c->launches++;
    return AGCM_OK;
}

// J0 of an IV that is not 96 bits long (SP 800-38D 7.1 step 2): GHASH_H(IV || 0^(s+64) || [len(IV)]_64),
// computed by the device (k_stream<GHASH_ONLY>) and read back; the message then runs with the
// first 96 bits of J0 as its "IV" and J0's last 32 bits as the counter field.  Synchronises `st`.
int derive_j0(agcm_ctx* c, const uint8_t* h_iv, size_t iv_len, uint8_t j0[16], cudaStream_t st)
{
    if (!h_iv || iv_len == 0 || iv_len > (1ull << 32)) return AGCM_E_BAD_LEN;
    if (!c->key_set) return AGCM_E_NO_KEY;
    const size_t padded = ((iv_len + 15) & ~(size_t)15) + 16;
    std::vector<uint8_t> buf(padded, 0);
    memcpy(buf.data(), h_iv, iv_len);
    const uint64_t bits = (uint64_t)iv_len * 8;
    for (int i = 0; i < 8; ++i) buf[padded - 1 - i] = (uint8_t)(bits >> (8 * i));
    int rc = grow(c, c->iv_stage, padded < 4096 ? 4096 : padded);
    if (rc) return rc;
    AG_CUDA(c, cudaMemcpyAsync(c->iv_stage.p, buf.data(), padded, cudaMemcpyHostToDevice, st));
    const uint8_t iv0[12] = {0};
    rc = run_stream(c, AG_MODE_GHASH_ONLY, iv0, 0, c->iv_stage.p, nullptr, padded, 0, c->d_parts, c->d_scratch + SC_J0, st,
                    c->d_counters);
    if (rc) return rc;
    AG_CUDA(c, cudaMemcpyAsync(j0, c->d_scratch + SC_J0, 16, cudaMemcpyDeviceToHost, st));
    AG_CUDA(c, cudaStreamSynchronize(st));
    return AGCM_OK;
}

// J0 of an IV of any length: IV || 0^31 || 1 for a 96-bit IV (no launch), else derive_j0 on `st`
int resolve_j0(agcm_ctx* c, const uint8_t* h_iv, size_t iv_len, uint8_t j0[16], cudaStream_t st)
{
    if (iv_len != 12) return derive_j0(c, h_iv, iv_len, j0, st);
    memcpy(j0, h_iv, 12);
    j0[12] = j0[13] = j0[14] = 0;
    j0[15] = 1;
    return AGCM_OK;
}

// The counter field of J0 replaces the constant 1 of the 96-bit case for the duration of a call.
struct J0Scope {
    agcm_ctx* c;
    J0Scope(agcm_ctx* ctx, const uint8_t j0[16]) : c(ctx)
    {
        if (c && j0) c->j0ctr = ((uint32_t)j0[12] << 24) | ((uint32_t)j0[13] << 16) | ((uint32_t)j0[14] << 8) | (uint32_t)j0[15];
    }
    ~J0Scope() { if (c) c->j0ctr = 1; }
};

// First steps of a host-buffer call (they may allocate, so before anything is enqueued): the device, the pipeline
// (created on first use) and room for `aad_len` bytes of AAD
int host_begin(agcm_ctx* c, uint64_t aad_len)
{
    AG_CUDA(c, cudaSetDevice(c->device));
    if (c->pipeline_ready) return grow(c, c->aad_stage, aad_len);
    if (const char* e = getenv("AGCM_CHUNK_MB")) {
        const long mb = atol(e);
        if (mb >= 1 && (size_t)mb <= (kChunkBytesMax >> 20)) c->chunk_bytes = (size_t)mb << 20;
    }
    if (const char* e = getenv("AGCM_RAMP_KB")) {   // first / last granule of a host-buffer call; 0 = equal granules
        const long kb = atol(e);
        if (kb >= 0 && (size_t)kb <= (kChunkBytesMax >> 10)) c->ramp_base = (size_t)kb << 10;
    }
    for (int s = 0; s < kSlots; ++s) {
        AG_CUDA(c, cudaStreamCreateWithFlags(&c->hs[s], cudaStreamNonBlocking));
        AG_CUDA(c, cudaMalloc(&c->d_stage[s], kChunkBytesMax));
        AG_CUDA(c, cudaMalloc(&c->d_stage_aux[s], kChunkBytesMax / 8));
        AG_CUDA(c, cudaMalloc(&c->d_stage_parts[s], sizeof(uint32_t) * 4 * AG_MAX_CTA));
    }
    AG_CUDA(c, cudaMalloc(&c->d_chunk_partials, 16 * kMaxChunks));
    c->pipeline_ready = true;
    return grow(c, c->aad_stage, aad_len);
}

// Last steps of a single-message host-buffer call: the ok byte (decrypt) or the tag out, then a wait for `st`.
int host_end(agcm_ctx* c, int decrypt, uint8_t h_tag[16], int* h_ok, cudaStream_t st)
{
    uint8_t okb = 1;
    if (decrypt) AG_CUDA(c, cudaMemcpyAsync(&okb, c->d_scratch + SC_OK, 1, cudaMemcpyDeviceToHost, st));
    else AG_CUDA(c, cudaMemcpyAsync(h_tag, c->d_scratch + SC_TAG, 16, cudaMemcpyDeviceToHost, st));
    AG_CUDA(c, cudaStreamSynchronize(st));
    if (h_ok) *h_ok = okb ? 1 : 0;
    return AGCM_OK;
}

int pick_lanes(const agcm_ctx* c, int lanes, uint64_t n_msgs, uint64_t avg_len, bool aligned16 = true, uint64_t real_blocks = 0)
{
    if (lanes == 1 || lanes == 2 || lanes == 4 || lanes == 8 || lanes == 16 || lanes == 32) return lanes;
    if (lanes > 4096 && lanes <= 4096 + 65536) return lanes;  // one warp per 1/S of a message (k_batch_warp), S = lanes - 4096
    if (lanes == 1024) return 1024;  // one CTA per message
    if (lanes > 1024 && lanes <= 1024 + 256 && ((lanes - 1024) & (lanes - 1025)) == 0) return lanes;  // ... per 1/S of a message
    if (lanes != 0) return -1;
    // Measured (tools/sweep_lanes.py, profiles/r1_lane_sweep.md): the best lane count grows like
    // sqrt(blocks)/4 -- 1 below 16 blocks (64 B: 370 vs 290 GB/s for 2 lanes), 2 at 1-1.5 KB, 4 at
    // 4 KB, 8 at 16 KB, 32 from 64 KB -- the trade between coalescing (16*G contiguous bytes per
    // message per request) and the per-message lane combine and front padding.  Records that are
    // not 16-byte aligned want at least 4 lanes.  Fewer messages than lanes: widen until the
    // persistent grid is occupied, but never more lanes than blocks in a message.
    const uint64_t total_lanes = (uint64_t)c->ncta * c->nt;
    const uint64_t blocks = (avg_len + 15) / 16 + 1;
    // From 32 KiB of work per message: one WARP per unit (k_batch_warp), units handed out by ticket,
    // lane combine deferred to combine rounds of the same launch.  A unit is a message or one of S counter-range
    // segments of it; S keeps a unit near 64-256 rows of 32 blocks and gives every warp at least ~8
    // units to draw, so neither the per-unit overhead (a row or two) nor the tail matters.
    // (uniform batches say how many blocks a message really has, AAD included: bulk AAD counts in full here,
    // although it only weighs a quarter in `avg_len`)
    uint64_t warp_min = 2048;
    if (const char* e = getenv("AGCM_WARP_MIN_BLOCKS")) warp_min = (uint64_t)atol(e);   // tuning experiments
    if ((blocks >= warp_min || real_blocks >= warp_min) && !getenv("AGCM_NO_WARP_UNITS")) {
        // S only matters for offset batches (uniform ones are partitioned exactly): near 128 rows of
        // 32 blocks per unit, and at least ~16 units per warp to draw when the messages are few
        const uint64_t warps = total_lanes / 32;
        uint64_t S = 1;
        while (blocks / S > 8192 && S < 65536) S <<= 1;
        while (n_msgs * S < 16 * warps && blocks / S >= 2048 && S < 65536) S <<= 1;
        return (int)(4096 + S);
    }
    uint64_t g = 1;
    while (g < 32 && (8 * g) * (8 * g) <= 2 * blocks) g <<= 1;
    if (blocks >= 4096) g = 32;
    if (!aligned16 && blocks >= 16 && g < 4) g = 4;
    while (g < 32 && n_msgs * g * 2 <= total_lanes) g <<= 1;
    while (g > 1 && g > blocks) g >>= 1;
    // Batches of a few rounds: the persistent grid works whole lane groups, so the time is quantised -- rounds x (rows
    // per lane + ~3 rows of per-message work).  10 000 x 4 KiB on 4 lanes fills 53 % of the grid for ONE long round
    // (315 GB/s); on 32 lanes it is five short ones (365 GB/s).  Take a wider group when this count says >= 5 % less
    // (measured: 40 000 x 4 KiB 433 -> 506 GB/s with 16 lanes, 10 000 x 1500 B stays on 4).
    {
        auto cost = [&](uint64_t gg) {
            const uint64_t rounds = (n_msgs * gg + total_lanes - 1) / total_lanes;
            return (double)rounds * ((double)blocks / (double)gg + 3.0);
        };
        const double c0 = cost(g);
        uint64_t best = g;
        double cb = c0;
        for (uint64_t gg = g << 1; gg <= 32 && gg <= blocks; gg <<= 1) {
            const double cg = cost(gg);
            if (cg < cb) { cb = cg; best = gg; }
        }
        if (cb < 0.95 * c0) g = best;
    }
    // Long messages: one CTA per message (k_batch_cta) when that finishes sooner.  Both layouts
    // assign whole messages statically, so the step count is quantised: rounds x (rows per lane +
    // per-message overhead), in block-times of one lane; the overheads (2 rows for a lane group,
    // 2.5 rows for a CTA: lane weights, two barriers) are fitted to profiles/r1_lane_sweep.md.
    if (avg_len >= (uint64_t)c->nt * 16 * 4) {
        const uint64_t groups = total_lanes / g;
        const double t_g = (double)((n_msgs + groups - 1) / groups) * ((double)blocks / (double)g + 3.0);
        const double t_cta = (double)((n_msgs + (uint64_t)c->ncta - 1) / (uint64_t)c->ncta) *
                             ((double)blocks / (double)c->nt + 3.5);
        if (t_cta < t_g) {
            // few long messages: cut each into S counter-range segments so that the last round
            // of CTAs is full too
            int best = 1024;
            double t_best = t_cta;
            for (uint64_t S = 2; S <= 256; S <<= 1) {
                const double rows = (double)blocks / (double)(S * (uint64_t)c->nt);
                if (rows < 8.0) break;
                const double t = (double)((n_msgs * S + (uint64_t)c->ncta - 1) / (uint64_t)c->ncta) * (rows + 5.0);
                if (t < 0.97 * t_best) {
                    t_best = t;
                    best = 1024 + (int)S;
                }
            }
            return best;
        }
    }
    return (int)g;
}

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

const char* agcm_strerror(int rc)
{
    switch (rc) {
        case AGCM_OK: return "ok";
        case AGCM_E_BAD_MODE: return "bad mode / key length (expected 128, 192 or 256 bits)";
        case AGCM_E_BAD_LEN: return "bad length";
        case AGCM_E_COUNTER_OVERFLOW: return "more than 2^32-2 blocks under one IV";
        case AGCM_E_CUDA: return "CUDA error";
        case AGCM_E_NO_KEY: return "no key set";
        case AGCM_E_BAD_ARG: return "bad argument";
        case AGCM_E_NO_DEVICE: return "no sm_100 CUDA device (the engine has no CPU path)";
        case AGCM_E_PEER_TIMEOUT: return "a peer never posted its shard partial (the tag of that message was zeroed, ok = 0)";
    }
    return "unknown error";
}

int agcm_ctx_create_ex(agcm_ctx** out, int device, int n_cta, int threads)
{
    if (!out) return AGCM_E_BAD_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return AGCM_E_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return AGCM_E_NO_DEVICE;
    if (prop.major != 10) return AGCM_E_NO_DEVICE;
    agcm_ctx* c = new (std::nothrow) agcm_ctx();
    if (!c) return AGCM_E_BAD_ARG;
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->ncta = n_cta > 0 ? n_cta : c->sm_count;
    c->nt = threads > 0 ? threads : AG_STREAM_NT_MAX;
    if (c->ncta > AG_MAX_CTA || c->nt > AG_STREAM_NT_MAX || c->nt < 32 || (c->nt & (c->nt - 1))) {
        delete c;
        return AGCM_E_BAD_ARG;
    }
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_te0, 256 * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_key, sizeof(KeyDev));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_parts, sizeof(uint32_t) * 4 * AG_MAX_CTA * 2);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_scratch, SC_BYTES);
    if (e == cudaSuccess) e = cudaMemset(c->d_scratch, 0, SC_BYTES);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_counters, sizeof(uint32_t) * (1 + kSlots));
    if (e == cudaSuccess) e = cudaMemset(c->d_counters, 0, sizeof(uint32_t) * (1 + kSlots));
    if (e == cudaSuccess) e = cudaMalloc(&c->pow_n.d, 16);
    if (e == cudaSuccess) {
        uint8_t sbox[256];
        uint32_t te0[256];
        ag_build_sbox_te0(sbox, te0);
        e = cudaMemcpy(c->d_te0, te0, sizeof(te0), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        agcm_ctx_destroy(c);
        return AGCM_E_CUDA;
    }
    *out = c;
    return AGCM_OK;
}

int agcm_ctx_create(agcm_ctx** out, int device) { return agcm_ctx_create_ex(out, device, 0, 0); }

void agcm_ctx_destroy(agcm_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();   // a deferred peer finish or a pipeline chunk may still use the buffers freed below
    for (int s = 0; s < kSlots; ++s) {
        if (c->hs[s]) cudaStreamDestroy(c->hs[s]);
        cudaFree(c->d_stage[s]);
        cudaFree(c->d_stage_aux[s]);
        cudaFree(c->d_stage_parts[s]);
    }
    for (cudaEvent_t e : c->tev)
        if (e) cudaEventDestroy(e);
    // key hygiene: wipe the stage keys, H, its powers and tables, and the host copy
    if (c->d_key) cudaMemset(c->d_key, 0, sizeof(KeyDev));
    if (c->d_scratch) cudaMemset(c->d_scratch, 0, SC_BYTES);
    memset(c->h_rk, 0, sizeof(c->h_rk));
    memset(c->h_H, 0, sizeof(c->h_H));
    memset(c->h_key_in, 0, sizeof(c->h_key_in));
    cudaFree(c->d_chunk_partials);
    cudaFree(c->aad_stage.p);
    cudaFree(c->verify.p);
    cudaFree(c->d_tile_ticket);
    cudaFree(c->sort.p);
    cudaFree(c->d_te0);
    cudaFree(c->d_key);
    cudaFree(c->d_parts);
    cudaFree(c->seg_parts.p);
    cudaFree(c->iv_stage.p);
    cudaFree(c->d_scratch);
    cudaFree(c->d_counters);
    cudaFree(c->pow_n.d);
    cudaFree(c->pow_scale.d);
    cudaFree(c->d_peer_bufs);
    cudaFree(c->d_peer_status);
    if (c->h_peer_status) cudaFreeHost(c->h_peer_status);
    if (c->peer_side) cudaStreamDestroy(c->peer_side);
    for (uint32_t i = 0; i < AG_PEER_RING; ++i) {
        if (c->peer_bulk_ev[i]) cudaEventDestroy(c->peer_bulk_ev[i]);
        if (c->peer_fin_ev[i]) cudaEventDestroy(c->peer_fin_ev[i]);
    }
    if (c->pow_n.ev) cudaEventDestroy(c->pow_n.ev);
    if (c->pow_scale.ev) cudaEventDestroy(c->pow_scale.ev);
    delete c;
}

int agcm_last_cuda_error(const agcm_ctx* c) { return c ? (int)c->last_err : 0; }
const char* agcm_last_cuda_error_string(const agcm_ctx* c) { return cudaGetErrorString(c ? c->last_err : cudaSuccess); }
uint64_t agcm_launch_count(const agcm_ctx* c) { return c ? c->launches : 0; }

int agcm_timing_enable(agcm_ctx* c, int on)
{
    if (!c) return AGCM_E_BAD_ARG;
    AG_CUDA(c, cudaSetDevice(c->device));
    if (on && !c->tev[0])
        for (cudaEvent_t& e : c->tev) AG_CUDA(c, cudaEventCreate(&e));
    int rc = timing_drain(c);
    if (rc) return rc;
    c->timing = on != 0;
    c->t_total_ms = 0.0;
    c->t_count = 0;
    return AGCM_OK;
}

int agcm_timing_read(agcm_ctx* c, double* total_ms, uint64_t* n_launches)
{
    if (!c) return AGCM_E_BAD_ARG;
    int rc = timing_drain(c);
    if (rc) return rc;
    if (total_ms) *total_ms = c->t_total_ms;
    if (n_launches) *n_launches = c->t_count;
    return AGCM_OK;
}

int agcm_get_info(const agcm_ctx* c, int* n_cta, int* threads, int* sm_count)
{
    if (!c) return AGCM_E_BAD_ARG;
    if (n_cta) *n_cta = c->ncta;
    if (threads) *threads = c->nt;
    if (sm_count) *sm_count = c->sm_count;
    return AGCM_OK;
}

int agcm_key_expand(agcm_ctx* c, int mode, const uint8_t* d_keys, size_t n_keys, uint8_t* d_round_keys, void* stream)
{
    if (!c || (n_keys && (!d_keys || !d_round_keys))) return AGCM_E_BAD_ARG;
    if (!mode_to_nr(mode)) return AGCM_E_BAD_MODE;
    AG_CUDA(c, cudaSetDevice(c->device));
    AG_CUDA(c, ag_launch_key_expand(d_keys, n_keys, mode / 8, c->d_te0, d_round_keys, (cudaStream_t)stream));
    if (n_keys) c->launches++;
    return AGCM_OK;
}

int agcm_key_expand_host(agcm_ctx* c, int mode, const uint8_t* h_key, uint8_t* h_round_keys)
{
    if (!c || !h_key || !h_round_keys) return AGCM_E_BAD_ARG;
    const int nr = mode_to_nr(mode);
    if (!nr) return AGCM_E_BAD_MODE;
    AG_CUDA(c, cudaSetDevice(c->device));
    uint8_t* d_key = c->d_scratch + SC_KEY;
    uint8_t* d_rk = c->d_scratch + SC_PARTS;  // 240 B of the parts list area, idle outside finish
    AG_CUDA(c, cudaMemcpy(d_key, h_key, (size_t)mode / 8, cudaMemcpyHostToDevice));
    AG_CUDA(c, ag_launch_key_expand(d_key, 1, mode / 8, c->d_te0, d_rk, nullptr));
    c->launches++;
    AG_CUDA(c, cudaMemcpy(h_round_keys, d_rk, (size_t)16 * (nr + 1), cudaMemcpyDeviceToHost));
    return AGCM_OK;
}

int agcm_set_key(agcm_ctx* c, int mode, int pre_expanded, const uint8_t* h_key, size_t key_len)
{
    if (!c || !h_key) return AGCM_E_BAD_ARG;
    const int nr = mode_to_nr(mode);
    if (!nr) return AGCM_E_BAD_MODE;
    const size_t want = pre_expanded ? (size_t)16 * (nr + 1) : (size_t)mode / 8;
    if (key_len != want) return AGCM_E_BAD_MODE;
    // the same key again: H, its powers and the tables are still valid (the IP keeps H until a
    // NEW key arrives, src/gcm_ghash.vhd:123-139)
    if (c->key_set && c->key_in_mode == mode && c->key_in_pre == (pre_expanded ? 1 : 0) && c->key_in_len == key_len &&
        memcmp(c->h_key_in, h_key, key_len) == 0)
        return AGCM_OK;
    AG_CUDA(c, cudaSetDevice(c->device));
    c->key_set = false;
    c->pow_n.e = ~0ull;
    c->pow_scale.e = ~0ull;
    KeyIn in;
    memset(&in, 0, sizeof(in));
    memcpy(in.w, h_key, key_len);   // LE words == the byte string
    in.key_bytes = (uint32_t)mode / 8;
    in.nr = (uint32_t)nr;
    in.pre_expanded = pre_expanded ? 1u : 0u;
    // no kernel of an earlier call may still be reading the key material this launch overwrites
    AG_CUDA(c, cudaDeviceSynchronize());
    AG_CUDA(c, ag_launch_key_setup(c->d_key, in, c->d_te0, c->nt, c->ncta, nullptr));
    c->launches++;
    // one readback: rk[60] | nr, nt, ncta, pad | H are the first 272 bytes of KeyDev
    static_assert(offsetof(KeyDev, rk) == 0 && offsetof(KeyDev, H) == 256, "KeyDev head layout");
    uint32_t head[68];
    AG_CUDA(c, cudaMemcpy(head, c->d_key, sizeof(head), cudaMemcpyDeviceToHost));
    memset(c->h_rk, 0, sizeof(c->h_rk));
    memcpy(c->h_rk, head, (size_t)16 * (nr + 1));
    const uint32_t* hw = head + 64;
    for (int i = 0; i < 4; ++i) {
        c->h_H[4 * i + 0] = (uint8_t)(hw[i] >> 24);
        c->h_H[4 * i + 1] = (uint8_t)(hw[i] >> 16);
        c->h_H[4 * i + 2] = (uint8_t)(hw[i] >> 8);
        c->h_H[4 * i + 3] = (uint8_t)hw[i];
    }
    c->nr = nr;
    memcpy(c->h_key_in, h_key, key_len);
    c->key_in_len = key_len;
    c->key_in_mode = mode;
    c->key_in_pre = pre_expanded ? 1 : 0;
    c->key_set = true;
    return AGCM_OK;
}

int agcm_get_round_keys(const agcm_ctx* c, uint8_t* h_round_keys, size_t cap)
{
    if (!c || !h_round_keys) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    const size_t n = (size_t)16 * (c->nr + 1);
    if (cap < n) return AGCM_E_BAD_LEN;
    memcpy(h_round_keys, c->h_rk, n);
    return (int)n;
}

int agcm_get_h(const agcm_ctx* c, uint8_t h_h16[16])
{
    if (!c || !h_h16) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    memcpy(h_h16, c->h_H, 16);
    return AGCM_OK;
}

int agcm_stream_part(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in,
                     uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t* d_partial16, void* stream)
{
    if (!c || !h_iv12 || !d_partial16 || (n_bytes && (!d_in || !d_out))) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    const uint64_t nb = (n_bytes + 15) >> 4;
    if (first_block > kMaxBlocks || nb > kMaxBlocks - first_block || blocks_after > kMaxBlocks - first_block - nb)
        return AGCM_E_COUNTER_OVERFLOW;
    if (blocks_after && (n_bytes & 15)) return AGCM_E_BAD_LEN;  // only the last shard may be ragged
    AG_CUDA(c, cudaSetDevice(c->device));
    return run_stream(c, decrypt ? AG_MODE_DEC : AG_MODE_ENC, h_iv12, first_block, d_in, d_out, n_bytes, blocks_after,
                      c->d_parts, d_partial16, (cudaStream_t)stream, c->d_counters);
}

int agcm_stream_finish(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], const uint8_t* d_partials16, int n_parts,
                       const uint8_t* d_aad, uint64_t aad_len, uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok, void* stream)
{
    if (!c || !h_iv12 || (n_parts && !d_partials16)) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    AG_CUDA(c, cudaSetDevice(c->device));
    return run_finish(c, decrypt, h_iv12, d_partials16, n_parts, d_aad, aad_len, ct_len, d_tag, d_ok, (cudaStream_t)stream);
}

int agcm_stream_crypt(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], const uint8_t* d_aad, uint64_t aad_len,
                      const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint8_t* d_tag, uint8_t* d_ok, void* stream)
{
    if (!c || !h_iv12) return AGCM_E_BAD_ARG;
    uint8_t* part = c->d_scratch + SC_PART_CT;
    if (n_bytes && aad_len <= kAadInlineMax) {
        // whole message in ONE launch: the last CTA folds the partials and finishes the tag
        if (!c->key_set) return AGCM_E_NO_KEY;
        if (!d_in || !d_out || (aad_len && !d_aad) || !d_tag || (decrypt && !d_ok)) return AGCM_E_BAD_ARG;
        if (((n_bytes + 15) >> 4) > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
        AG_CUDA(c, cudaSetDevice(c->device));
        const FinishParams ff = finish_params(c, decrypt, h_iv12, aad_len ? d_aad : nullptr, aad_len, n_bytes, d_tag, d_ok, c->pow_n.d);
        if (aad_len) {
            int rc = ensure_pow(c, (n_bytes + 15) >> 4, (cudaStream_t)stream);
            if (rc) return rc;
        }
        return run_stream(c, decrypt ? AG_MODE_DEC : AG_MODE_ENC, h_iv12, 0, d_in, d_out, n_bytes, 0, c->d_parts, nullptr,
                          (cudaStream_t)stream, c->d_counters, &ff);
    }
    int rc = agcm_stream_part(c, decrypt, h_iv12, 0, d_in, d_out, n_bytes, 0, part, stream);
    if (rc) return rc;
    return agcm_stream_finish(c, decrypt, h_iv12, part, 1, d_aad, aad_len, n_bytes, d_tag, d_ok, stream);
}

int agcm_stream_crypt_iv(agcm_ctx* c, int decrypt, const uint8_t* h_iv, size_t iv_len, const uint8_t* d_aad, uint64_t aad_len,
                         const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint8_t* d_tag, uint8_t* d_ok, void* stream)
{
    if (!c || !h_iv) return AGCM_E_BAD_ARG;
    if (iv_len == 12) return agcm_stream_crypt(c, decrypt, h_iv, d_aad, aad_len, d_in, d_out, n_bytes, d_tag, d_ok, stream);
    AG_CUDA(c, cudaSetDevice(c->device));
    uint8_t j0[16];
    int rc = resolve_j0(c, h_iv, iv_len, j0, (cudaStream_t)stream);
    if (rc) return rc;
    J0Scope scope(c, j0);
    return agcm_stream_crypt(c, decrypt, j0, d_aad, aad_len, d_in, d_out, n_bytes, d_tag, d_ok, stream);
}

int agcm_peer_setup(agcm_ctx* c, int rank, int world, const uint64_t* h_peer_ptrs)
{
    if (!c || !h_peer_ptrs || world < 1 || world > (int)AG_PEER_MAX || rank < 0 || rank >= world) return AGCM_E_BAD_ARG;
    AG_CUDA(c, cudaSetDevice(c->device));
    AG_CUDA(c, cudaDeviceSynchronize());   // no finish of an earlier session may still be waiting
    if (!c->d_peer_bufs) AG_CUDA(c, cudaMalloc(&c->d_peer_bufs, sizeof(uint8_t*) * AG_PEER_MAX));
    if (!c->d_peer_status) AG_CUDA(c, cudaMalloc(&c->d_peer_status, sizeof(uint32_t)));
    if (!c->h_peer_status) AG_CUDA(c, cudaHostAlloc(reinterpret_cast<void**>(&c->h_peer_status), sizeof(uint32_t), cudaHostAllocMapped));
    AG_CUDA(c, ag_preload_peer_kernels());
    if (!c->peer_side) {
        AG_CUDA(c, cudaStreamCreateWithFlags(&c->peer_side, cudaStreamNonBlocking));
        for (uint32_t i = 0; i < AG_PEER_RING; ++i) {
            AG_CUDA(c, cudaEventCreateWithFlags(&c->peer_bulk_ev[i], cudaEventDisableTiming));
            AG_CUDA(c, cudaEventCreateWithFlags(&c->peer_fin_ev[i], cudaEventDisableTiming));
        }
    }
    if (const char* e = getenv("AGCM_PEER_TIMEOUT_MS")) {
        const long ms = atol(e);
        if (ms >= 1) c->peer_timeout_ns = (uint64_t)ms * 1000000ull;
    }
    *c->h_peer_status = 0;
    AG_CUDA(c, cudaMemset(c->d_peer_status, 0, sizeof(uint32_t)));
    AG_CUDA(c, cudaMemcpy(c->d_peer_bufs, h_peer_ptrs, sizeof(uint64_t) * (size_t)world, cudaMemcpyHostToDevice));
    // my own buffer starts with all flags clear; the caller barriers before the first exchange
    AG_CUDA(c, cudaMemset(reinterpret_cast<void*>(h_peer_ptrs[rank]), 0, AG_PEER_BYTES));
    AG_CUDA(c, cudaDeviceSynchronize());
    c->peer_rank = rank;
    c->peer_world = world;
    c->peer_epoch = 0;
    return AGCM_OK;
}

int agcm_peer_status(agcm_ctx* c, int* h_timed_out)
{
    if (!c || !h_timed_out) return AGCM_E_BAD_ARG;
    uint32_t v = 0;
    if (c->d_peer_status) {
        AG_CUDA(c, cudaSetDevice(c->device));
        if (c->peer_side) AG_CUDA(c, cudaStreamSynchronize(c->peer_side));   // every finish issued so far has run
        AG_CUDA(c, cudaMemcpy(&v, c->d_peer_status, sizeof(v), cudaMemcpyDeviceToHost));
    }
    *h_timed_out = (int)v;
    return AGCM_OK;
}

int agcm_peer_join(agcm_ctx* c, void* stream)
{
    if (!c) return AGCM_E_BAD_ARG;
    if (c->peer_world < 1) return AGCM_E_BAD_ARG;
    AG_CUDA(c, cudaSetDevice(c->device));
    return peer_join_stream(c, (cudaStream_t)stream);
}

// Common checks of the peer calls + the ring's flow control on `st`; returns the new epoch.
static int peer_begin(agcm_ctx* c, uint64_t first_block, uint64_t n_bytes, uint64_t blocks_after, uint64_t aad_len,
                      uint64_t total_len, cudaStream_t st, uint32_t* epoch_out)
{
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (c->peer_world < 1) return AGCM_E_BAD_ARG;                          // agcm_peer_setup first
    if (*(volatile uint32_t*)c->h_peer_status) return AGCM_E_PEER_TIMEOUT; // an earlier exchange failed closed
    if (aad_len > kAadInlineMax) return AGCM_E_BAD_LEN;                    // bulk AAD: use the gather path
    const uint64_t nb = (n_bytes + 15) >> 4, tb = (total_len + 15) >> 4;
    if (tb > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
    if (first_block > tb || nb > tb - first_block || blocks_after != tb - first_block - nb) return AGCM_E_BAD_LEN;
    if (blocks_after && (n_bytes & 15)) return AGCM_E_BAD_LEN;
    AG_CUDA(c, cudaSetDevice(c->device));
    const uint32_t epoch = c->peer_epoch + 1;
    // flow control of the ring (gcm_core.cuh): post epoch e only after my finish of e - AHEAD ran
    if (epoch > AG_PEER_AHEAD) AG_CUDA(c, cudaStreamWaitEvent(st, c->peer_fin_ev[(epoch - AG_PEER_AHEAD) % AG_PEER_RING], 0));
    if (aad_len) {
        int rc = ensure_pow(c, tb, st);
        if (rc) return rc;
    }
    *epoch_out = epoch;
    return AGCM_OK;
}

// The one-warp finish of `epoch` on the side stream, ordered after everything queued on `st`.
static int peer_finish(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], const uint8_t* d_aad, uint64_t aad_len,
                       uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, cudaStream_t st, uint32_t epoch, bool deferred)
{
    const uint32_t slot = epoch % AG_PEER_RING;
    c->peer_epoch = epoch;
    PeerFinishParams pf;
    memset(&pf, 0, sizeof(pf));
    pf.f = finish_params(c, decrypt, h_iv12, aad_len ? d_aad : nullptr, aad_len, total_len, d_tag, d_ok,
                         aad_len ? c->pow_n.d : nullptr);
    pf.peer_bufs = c->d_peer_bufs;
    pf.rank = (uint32_t)c->peer_rank;
    pf.world = (uint32_t)c->peer_world;
    pf.epoch = epoch;
    pf.timeout_ns = c->peer_timeout_ns;
    pf.status_dev = c->d_peer_status;
    uint32_t* mapped = nullptr;
    AG_CUDA(c, cudaHostGetDevicePointer(reinterpret_cast<void**>(&mapped), c->h_peer_status, 0));
    pf.status_host = mapped;
    // the finish waits for the world on the side stream: the caller's stream is free for the next bulk kernel
    AG_CUDA(c, cudaEventRecord(c->peer_bulk_ev[slot], st));
    AG_CUDA(c, cudaStreamWaitEvent(c->peer_side, c->peer_bulk_ev[slot], 0));
    AG_CUDA(c, ag_launch_peer_finish(pf, c->peer_side));
    c->launches++;
    AG_CUDA(c, cudaEventRecord(c->peer_fin_ev[slot], c->peer_side));
    if (!deferred) AG_CUDA(c, cudaStreamWaitEvent(st, c->peer_fin_ev[slot], 0));
    return AGCM_OK;
}

static int stream_crypt_peer(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in,
                             uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* d_aad, uint64_t aad_len,
                             uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, void* stream, bool deferred)
{
    if (!c || !h_iv12 || (n_bytes && (!d_in || !d_out)) || !d_tag || (decrypt && !d_ok) || (aad_len && !d_aad))
        return AGCM_E_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t epoch = 0;
    int rc = peer_begin(c, first_block, n_bytes, blocks_after, aad_len, total_len, st, &epoch);
    if (rc) return rc;
    if (n_bytes) {
        rc = run_stream(c, decrypt ? AG_MODE_DEC : AG_MODE_ENC, h_iv12, first_block, d_in, d_out, n_bytes, blocks_after,
                        c->d_parts, nullptr, st, c->d_counters, nullptr, epoch);
        if (rc) return rc;
    } else {   // an empty counter range (fewer blocks than ranks) still posts its zero partial
        AG_CUDA(c, ag_launch_peer_post(c->d_peer_bufs, (uint32_t)c->peer_rank, (uint32_t)c->peer_world, epoch, nullptr, st));
        c->launches++;
    }
    return peer_finish(c, decrypt, h_iv12, d_aad, aad_len, total_len, d_tag, d_ok, st, epoch, deferred);
}

int agcm_stream_crypt_peer(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in,
                           uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* d_aad, uint64_t aad_len,
                           uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, void* stream)
{
    return stream_crypt_peer(c, decrypt, h_iv12, first_block, d_in, d_out, n_bytes, blocks_after, d_aad, aad_len, total_len,
                             d_tag, d_ok, stream, false);
}

int agcm_stream_crypt_peer_async(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block,
                                 const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after,
                                 const uint8_t* d_aad, uint64_t aad_len, uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok,
                                 void* stream)
{
    return stream_crypt_peer(c, decrypt, h_iv12, first_block, d_in, d_out, n_bytes, blocks_after, d_aad, aad_len, total_len,
                             d_tag, d_ok, stream, true);
}

// ---- IVs of any length on the shard / peer / gctr entry points: the caller derives J0 once
// (agcm_derive_j0) and passes it instead of the 12 IV bytes (J0Scope).
int agcm_derive_j0(agcm_ctx* c, const uint8_t* h_iv, size_t iv_len, uint8_t h_j0[16])
{
    if (!c || !h_iv || !h_j0) return AGCM_E_BAD_ARG;
    if (iv_len != 12) AG_CUDA(c, cudaSetDevice(c->device));
    return resolve_j0(c, h_iv, iv_len, h_j0, nullptr);   // the legacy stream: this call takes none
}

int agcm_gctr_j0(agcm_ctx* c, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in, uint8_t* d_out,
                 uint64_t n_bytes, void* stream)
{
    if (!c || !h_j0) return AGCM_E_BAD_ARG;
    J0Scope scope(c, h_j0);
    return agcm_gctr(c, h_j0, first_block, d_in, d_out, n_bytes, stream);
}

int agcm_stream_part_j0(agcm_ctx* c, int decrypt, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in,
                        uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t* d_partial16, void* stream)
{
    if (!c || !h_j0) return AGCM_E_BAD_ARG;
    J0Scope scope(c, h_j0);
    return agcm_stream_part(c, decrypt, h_j0, first_block, d_in, d_out, n_bytes, blocks_after, d_partial16, stream);
}

int agcm_stream_finish_j0(agcm_ctx* c, int decrypt, const uint8_t h_j0[16], const uint8_t* d_partials16, int n_parts,
                          const uint8_t* d_aad, uint64_t aad_len, uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok, void* stream)
{
    if (!c || !h_j0) return AGCM_E_BAD_ARG;
    J0Scope scope(c, h_j0);
    return agcm_stream_finish(c, decrypt, h_j0, d_partials16, n_parts, d_aad, aad_len, ct_len, d_tag, d_ok, stream);
}

int agcm_stream_crypt_peer_j0(agcm_ctx* c, int decrypt, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in,
                              uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* d_aad, uint64_t aad_len,
                              uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, void* stream, int deferred)
{
    if (!c || !h_j0) return AGCM_E_BAD_ARG;
    J0Scope scope(c, h_j0);
    return stream_crypt_peer(c, decrypt, h_j0, first_block, d_in, d_out, n_bytes, blocks_after, d_aad, aad_len, total_len, d_tag,
                             d_ok, stream, deferred != 0);
}

int agcm_stream_decrypt_verified(agcm_ctx* c, const uint8_t* h_iv, size_t iv_len, const uint8_t* d_aad, uint64_t aad_len,
                                 const uint8_t* d_ct, uint8_t* d_pt, uint64_t n_bytes, const uint8_t* d_tag, uint8_t* d_ok,
                                 void* stream)
{
    if (!c || !h_iv || !d_tag || !d_ok || (n_bytes && (!d_ct || !d_pt)) || (aad_len && !d_aad)) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (((n_bytes + 15) >> 4) > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
    AG_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t j0[16];
    int rc = resolve_j0(c, h_iv, iv_len, j0, st);   // on `st`: the caller's earlier work there may use the same scratch
    if (rc) return rc;
    J0Scope scope(c, j0);
    // pass 1: GHASH over the ciphertext only (about 4x the rate of the fused pass), then the tag check
    uint8_t* part = c->d_scratch + SC_PART_CT;
    rc = run_stream(c, AG_MODE_GHASH_ONLY, j0, 0, d_ct, nullptr, n_bytes, 0, c->d_parts, part, st, c->d_counters);
    if (rc) return rc;
    rc = run_finish(c, 1, j0, part, 1, d_aad, aad_len, n_bytes, const_cast<uint8_t*>(d_tag), d_ok, st);
    if (rc) return rc;
    // pass 2: GCTR, gated on the device by the flag pass 1 just wrote (no host round trip)
    return run_stream(c, AG_MODE_CTR_ONLY, j0, 0, d_ct, d_pt, n_bytes, 0, c->d_parts, nullptr, st, c->d_counters, nullptr, 0, d_ok);
}

int agcm_gctr(agcm_ctx* c, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in, uint8_t* d_out,
              uint64_t n_bytes, void* stream)
{
    if (!c || !h_iv12 || (n_bytes && (!d_in || !d_out))) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    const uint64_t nb = (n_bytes + 15) >> 4;
    if (first_block > kMaxBlocks || nb > kMaxBlocks - first_block) return AGCM_E_COUNTER_OVERFLOW;
    AG_CUDA(c, cudaSetDevice(c->device));
    return run_stream(c, AG_MODE_CTR_ONLY, h_iv12, first_block, d_in, d_out, n_bytes, 0, c->d_parts, nullptr,
                      (cudaStream_t)stream, c->d_counters);
}

int agcm_ghash(agcm_ctx* c, const uint8_t* d_in, uint64_t n_bytes, uint8_t* d_y16, void* stream)
{
    if (!c || !d_y16 || (n_bytes && !d_in)) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    AG_CUDA(c, cudaSetDevice(c->device));
    const uint8_t iv0[12] = {0};
    return run_stream(c, AG_MODE_GHASH_ONLY, iv0, 0, d_in, nullptr, n_bytes, 0, c->d_parts, d_y16, (cudaStream_t)stream,
                      c->d_counters);
}

// Length order of a batch of different-length messages (device counting sort, longest first): fills the per-context
// scratch [4096-bucket histogram | 8 words of class bounds | perm[n_msgs]] and points p.perm at the order.
static int len_sort(agcm_ctx* c, BatchParams& p, size_t n_msgs, cudaStream_t st)
{
    int rc = grow(c, c->sort, sizeof(uint32_t) * (4096 + 8 + n_msgs));
    if (rc) return rc;
    AG_CUDA(c, ag_launch_len_sort(p, c->sort.p, c->sort.p + 4096, c->sort.p + 4096 + 8, st));
    c->launches += 3;
    p.perm = c->sort.p + 4096 + 8;
    return AGCM_OK;
}

// The argument check every shared-key batch kernel needs, then the context's key bound into p.
static int batch_bind_key(agcm_ctx* c, int decrypt, BatchParams& p, size_t n_msgs)
{
    if (!p.iv || !p.tag || (decrypt && !p.ok)) return AGCM_E_BAD_ARG;
    AG_CUDA(c, cudaSetDevice(c->device));
    memcpy(p.rk, c->h_rk, sizeof(p.rk));
    p.key = c->d_key;
    p.te0 = c->d_te0;
    p.n_msgs = n_msgs;
    return AGCM_OK;
}

static int batch_common(agcm_ctx* c, int decrypt, int lanes, uint64_t avg_len, BatchParams& p, size_t n_msgs, void* stream,
                        bool aligned16 = true)
{
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (n_msgs == 0) return AGCM_OK;
    int rc = batch_bind_key(c, decrypt, p, n_msgs);
    if (rc) return rc;
    const bool ragged = p.in_off || p.aad_off || p.len_arr || p.aad_len_arr;   // messages of different lengths
    const uint64_t real_blocks = !ragged ? ((p.len + 15) >> 4) + (p.aad ? (p.aad_len + 15) >> 4 : 0) : 0;
    const int g = pick_lanes(c, lanes, n_msgs, avg_len, aligned16, real_blocks);
    if (g < 0) return AGCM_E_BAD_ARG;
    if (g > 4096) {
        // a warp per unit (k_batch_warp): balanced static partition for uniform batches, `split`
        // segments per message by ticket for offset batches
        const uint64_t per_cta = (uint64_t)AG_STREAM_NT_MAX / 32;
        const bool uniform = !ragged;
        int ncta_w = c->ncta;
        if (uniform) {
            const uint64_t warps = (uint64_t)ncta_w * per_cta;
            const uint64_t ax_a = p.aad ? (p.aad_len + 15) >> 4 : 0, ax_p = ((p.len + 15) >> 4) + AG_FINISH_WEIGHT;
            p.quota_aad = ((ax_a * (uint64_t)n_msgs + warps - 1) / warps + 31) & ~31ull;   // whole rows
            p.quota_pt = ((ax_p * (uint64_t)n_msgs + warps - 1) / warps + 31) & ~31ull;
            if (!p.quota_aad) p.quota_aad = 32;
            p.n_ids = 2 * (warps + n_msgs);
            p.split = 1;
        } else {
            p.split = (uint32_t)(g - 4096);
            p.n_ids = (uint64_t)n_msgs * p.split;
            if (p.n_ids >= 0xFFFFFFFFull) return AGCM_E_BAD_LEN;
            const uint64_t need_cta = (p.n_ids + per_cta - 1) / per_cta;
            if (need_cta < (uint64_t)ncta_w) ncta_w = (int)need_cta;
        }
        // scratch: [msg_acc n_msgs x 16 | msg_cnt n_msgs x 4] (zeroed per launch) [unit_desc n_ids x 16] [msg_ej0 n_msgs x 16]
        // [seg_acc n_ids x 512]
        const size_t zero_bytes = ((size_t)n_msgs * 20 + 255) & ~(size_t)255;
        const size_t desc_bytes = ((size_t)p.n_ids * 16 + 255) & ~(size_t)255;
        const size_t ej0_bytes = ((size_t)n_msgs * 16 + 255) & ~(size_t)255;
        rc = grow(c, c->seg_parts, zero_bytes + desc_bytes + ej0_bytes + (size_t)p.n_ids * 512);
        if (rc) return rc;
        uint8_t* base = reinterpret_cast<uint8_t*>(c->seg_parts.p);
        p.msg_acc = reinterpret_cast<uint32_t*>(base);
        p.msg_cnt = reinterpret_cast<uint32_t*>(base + (size_t)n_msgs * 16);
        p.unit_desc = reinterpret_cast<uint64_t*>(base + zero_bytes);
        p.msg_ej0 = reinterpret_cast<uint32_t*>(base + zero_bytes + desc_bytes);
        p.seg_acc = reinterpret_cast<uint4*>(base + zero_bytes + desc_bytes + ej0_bytes);
        AG_CUDA(c, cudaMemsetAsync(base, 0, zero_bytes, (cudaStream_t)stream));
        if (!uniform) {
            rc = zeroed_ticket(c, 1, (cudaStream_t)stream, p.ticket);
            if (rc) return rc;
        }
        AG_CUDA(c, ag_launch_batch_warp(p, c->nr, decrypt, ncta_w, (cudaStream_t)stream));
        c->launches++;
        return AGCM_OK;
    }
    if (g >= 1024) {
        p.split = g == 1024 ? 1u : (uint32_t)(g - 1024);
        const uint64_t n_units = (uint64_t)n_msgs * p.split;
        if (p.split > 1) {
            rc = grow(c, c->seg_parts, (size_t)(n_units + n_msgs) * 16);
            if (rc) return rc;
            p.seg_parts = c->seg_parts.p;
        }
        const int ncta_m = (int)(n_units < (uint64_t)c->ncta ? n_units : (uint64_t)c->ncta);
        if (n_units > (uint64_t)ncta_m && n_units < 0xFFFFFFFFull && !c->no_ticket) {   // more units than CTAs: hand them out dynamically
            rc = zeroed_ticket(c, 1, (cudaStream_t)stream, p.ticket);
            if (rc) return rc;
        }
        AG_CUDA(c, ag_launch_batch_cta(p, c->nr, decrypt, ncta_m, c->nt, (cudaStream_t)stream));
        c->launches += p.split > 1 ? 2 : 1;
        return AGCM_OK;
    }
    // no more CTAs than there is work for
    const uint64_t groups_per_cta = (uint64_t)c->nt / g;
    uint64_t need = (n_msgs + groups_per_cta - 1) / groups_per_cta;
    int ncta = (int)(need < (uint64_t)c->ncta ? need : (uint64_t)c->ncta);
    if (ragged && n_msgs >= 1024 && n_msgs < 0xFFFFFF00ull && !c->no_ticket && !getenv("AGCM_NO_LEN_SORT")) {
        // Messages of different lengths: take them longest first, so that the 32/G messages a warp works on in
        // lock step are equally long (3 small launches; the kernels then follow perm[]), warp by warp by ticket.
        // With lanes = 0 the order is cut into three length classes, one launch each: 32 lanes per message from
        // 16 KiB of work, 4 from 4 KiB, 1 below -- a heavy tail of long messages must not crawl through one lane.
        // The class sizes stay on the device (no host round trip): an empty class costs one idle launch.
        cudaStream_t st = (cudaStream_t)stream;
        uint32_t* tickets = nullptr;
        rc = zeroed_ticket(c, 4, st, tickets);
        if (rc) return rc;
        rc = len_sort(c, p, n_msgs, st);
        if (rc) return rc;
        uint32_t* ranges = c->sort.p + 4096;
        if (lanes == 0 && !getenv("AGCM_NO_LEN_CLASSES")) {
            // short class: one lane per message with realigned wide accesses when records sit at odd addresses,
            // two lanes (32 contiguous bytes per request) when they are 16-byte aligned
            const int gs[3] = {32, 4, (aligned16 && !p.in_off) ? 2 : 1};   // packed by offsets: alignment unknown
            for (int k = 0; k < 3; ++k) {
                p.range = ranges + 2 * k;
                p.ticket = tickets + 1 + k;
                AG_CUDA(c, ag_launch_batch(p, c->nr, decrypt, gs[k], c->ncta, c->nt, st));
                c->launches++;
            }
            return AGCM_OK;
        }
        p.ticket = tickets + 1;
    }
    AG_CUDA(c, ag_launch_batch(p, c->nr, decrypt, g, ncta, c->nt, (cudaStream_t)stream));
    c->launches++;
    return AGCM_OK;
}

// ---- fixed-size records through the TMA-staged kernel (k_batch_tile) -----------------------------
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// box_rows: AG_TILE_BOX_MSGS for the one-box loads, 1 for the row-gathering form (tile::gather4 / scatter4)
static int tile_tensor_map(agcm_ctx* c, CUtensorMap* tm, const uint8_t* base, uint64_t len, uint64_t stride, uint64_t n_msgs,
                           uint32_t box_rows = AG_TILE_BOX_MSGS)
{
    if (!c->tmap_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn ||
            q != cudaDriverEntryPointSuccess)
            return AGCM_E_CUDA;
        c->tmap_encode = fn;
    }
    // the batch as a 2-D byte tensor: dim 0 = the bytes of a record (extent len), dim 1 = the messages (pitch = stride)
    const cuuint64_t dims[2] = {len, n_msgs};
    const cuuint64_t strides[1] = {stride};
    const cuuint32_t box[2] = {AG_TILE_BOX_BYTES, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<tmap_encode_fn>(c->tmap_encode)(
        tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? AGCM_OK : AGCM_E_CUDA;
}

// Can (and should) this uniform batch take the tiled kernel?  16-byte aligned buffers and pitch (TMA),
// messages short enough that a message per lane is the right compute layout, and enough of them to
// fill the persistent grid a few times over.
static bool tile_eligible(const agcm_ctx* c, int lanes, const BatchParams& p, size_t n_msgs)
{
    if (lanes != 0 && lanes != 2048) return false;
    if (p.len == 0 || p.len >= (1ull << 31) || n_msgs >= (1ull << 31) - 32) return false;
    if ((((uintptr_t)p.in | (uintptr_t)p.out) & 15) || (p.stride & 15) || p.stride >= (1ull << 40)) return false;
    if (lanes == 2048) return true;
    if (getenv("AGCM_NO_TILE")) return false;
    return p.len + p.aad_len <= 16384 && n_msgs >= (size_t)c->ncta * (size_t)c->nt;   // at least a group of 32 per warp
}

// Fixed-size, 16-byte aligned records under per-message keys: stage them by TMA (k_batch_perkey_tile) when there
// are enough messages to fill the grid; AGCM_PERKEY_TILE=0 / 1 keeps the thread-per-message loads / forces it (A/B runs)
static bool perkey_tile_eligible(const agcm_ctx* c, const BatchParams& p, size_t n_msgs)
{
    const char* ev = getenv("AGCM_PERKEY_TILE");
    if (ev && ev[0] == '0') return false;
    if (!p.len || p.len >= (1ull << 31) || n_msgs >= (1ull << 31) - 32) return false;
    if ((((uintptr_t)p.in | (uintptr_t)p.out) & 15) || (p.stride & 15) || p.stride >= (1ull << 40)) return false;
    if (ev && ev[0] == '1') return true;
    // Measured (tools/bench_variants.py --only perkey, AES-256, 64 B AAD): at a 4096 B pitch the tiled kernel wins
    // (341 vs 294 GB/s: a lane per message at a large power-of-two pitch camps on few DRAM channels), at 1504 B
    // the thread-per-message kernel does (353 vs 335: its aligned 128-bit accesses are only ~5 % of the pipe, and
    // the tiled kernel pays a PRMT more on three lookups in four for dropping Te1), at 64 B too (167 vs 164):
    // tile from 2 KiB records.
    return p.len >= 2048 && n_msgs >= (size_t)c->ncta * 448u * 2;
}

// t.b = p and in / out tensor maps of 16-byte-granular extents (the pitch is a multiple of 16 and >= len: both fit)
static int tile_records(agcm_ctx* c, TileParams& t, const BatchParams& p)
{
    memset(&t, 0, sizeof(t));
    t.b = p;
    const uint64_t len_up = (p.len + 15) & ~15ull, len_down = p.len & ~15ull;
    int rc = tile_tensor_map(c, &t.tm_in, p.in, len_up, p.stride, p.n_msgs);
    if (rc) return rc;
    return tile_tensor_map(c, &t.tm_out, p.out, len_down ? len_down : 16, p.stride, p.n_msgs);   // len < 16: never stored through
}

// The ticket zeroed, then k_batch_perkey_tile (per-key batch) or k_batch_tile on as many CTAs as its groups of 32 need
static int tile_launch(agcm_ctx* c, TileParams& t, int nr, int decrypt, int gather, cudaStream_t st)
{
    int rc = zeroed_ticket(c, 1, st, t.ticket);
    if (rc) return rc;
    if (t.b.keys) {
        AG_CUDA(c, ag_launch_batch_perkey_tile(t, nr, decrypt, c->ncta, st));
    } else {
        const uint64_t groups = (t.b.n_msgs + 31) / 32, per_cta = (uint64_t)AG_STREAM_NT_MAX / 32;
        const uint64_t need = (groups + per_cta - 1) / per_cta;
        const int ncta = (int)(need < (uint64_t)c->ncta ? need : (uint64_t)c->ncta);
        AG_CUDA(c, ag_launch_batch_tile(t, nr, decrypt, gather, ncta, st));
    }
    c->launches++;
    return AGCM_OK;
}

static int batch_tile(agcm_ctx* c, int decrypt, BatchParams& p, size_t n_msgs, cudaStream_t st)
{
    if (!c->key_set) return AGCM_E_NO_KEY;
    int rc = batch_bind_key(c, decrypt, p, n_msgs);
    if (rc) return rc;
    TileParams t;
    rc = tile_records(c, t, p);
    if (rc) return rc;
    if (p.aad && p.aad_len && !((uintptr_t)p.aad & 15) && !(p.aad_stride & 15) && p.aad_len < (1ull << 31) &&
        p.aad_stride < (1ull << 40)) {
        rc = tile_tensor_map(c, &t.tm_aad, p.aad, (p.aad_len + 15) & ~15ull, p.aad_stride, n_msgs);
        if (rc) return rc;
        t.aad_tiled = 1;
    }
    return tile_launch(c, t, c->nr, decrypt, 0, st);
}

// Slots (fixed 16-byte aligned pitch, a length per message) through the row-gathering form of the tiled kernel:
// every message fits a lane's share (pitch <= 16 KiB) and there are enough of them to fill the grid.
static bool tile_slots_eligible(const agcm_ctx* c, int lanes, const BatchParams& p, size_t n_msgs)
{
    if (lanes != 0 && lanes != 2048) return false;
    if (!p.len_arr || p.stride == 0 || p.stride >= (1ull << 31) || n_msgs >= (1ull << 30) || c->no_ticket) return false;
    if ((((uintptr_t)p.in | (uintptr_t)p.out) & 15) || (p.stride & 15)) return false;
    if (lanes == 2048) return true;   // asked for by name
    // Not a default: measured against the lane-group classes on 2^20 messages (profiles/r2_ragged.md) it is within
    // +-3 % -- with 16-byte aligned slots two lanes per message already fetch whole sectors, and the per-message work
    // that dominates short packets (IV, J0, tag) is the same in both.  AGCM_GATHER=1 makes it the choice for A/B runs.
    if (!getenv("AGCM_GATHER") || getenv("AGCM_NO_TILE")) return false;
    if (p.stride > 16384) return false;                                              // a message per lane: short messages
    if (p.aad && (p.aad_len_arr ? p.aad_stride : p.aad_len) > 4096) return false;   // long AAD: the lane-group layouts
    return n_msgs >= (size_t)c->ncta * (size_t)c->nt;
}

static int batch_tile_slots(agcm_ctx* c, int decrypt, BatchParams& p, size_t n_msgs, cudaStream_t st)
{
    if (!c->key_set) return AGCM_E_NO_KEY;
    int rc = batch_bind_key(c, decrypt, p, n_msgs);
    if (rc) return rc;
    // length order (longest first): the 32 messages a warp takes side by side are equally long
    if (n_msgs >= 64 && !getenv("AGCM_NO_LEN_SORT")) {
        rc = len_sort(c, p, n_msgs, st);
        if (rc) return rc;
    }
    TileParams t;
    memset(&t, 0, sizeof(t));
    t.b = p;
    // whole slots as rows: a lane masks what lies past its message, and rows are stored only where whole blocks are
    rc = tile_tensor_map(c, &t.tm_in, p.in, p.stride, p.stride, n_msgs, 1);
    if (rc) return rc;
    rc = tile_tensor_map(c, &t.tm_out, p.out, p.stride, p.stride, n_msgs, 1);
    if (rc) return rc;
    if (p.aad && p.aad_len && !p.aad_len_arr && !((uintptr_t)p.aad & 15) && !(p.aad_stride & 15)) {   // AAD of one length: tiled too
        rc = tile_tensor_map(c, &t.tm_aad, p.aad, (p.aad_len + 15) & ~15ull, p.aad_stride, n_msgs, 1);
        if (rc) return rc;
        t.aad_tiled = 1;
    }
    return tile_launch(c, t, c->nr, decrypt, 1, st);
}

// Checks and BatchParams of an offset batch (message i at in_off[i]) under the context's key or d_keys
static int offsets_params(BatchParams& p, const uint8_t* d_keys, const uint8_t* d_iv, int iv_is_j0, const uint8_t* d_aad,
                          const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off, uint8_t* d_out,
                          uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs)
{
    if (n_msgs && (!d_in_off || !d_in || !d_out)) return AGCM_E_BAD_ARG;
    if ((d_aad == nullptr) != (d_aad_off == nullptr)) return AGCM_E_BAD_ARG;
    memset(&p, 0, sizeof(p));
    p.keys = d_keys;
    p.iv = d_iv;
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.aad = d_aad;
    p.aad_off = d_aad_off;
    p.in = d_in;
    p.in_off = d_in_off;
    p.out = d_out;
    p.tag = d_tag;
    p.ok = d_ok;
    return AGCM_OK;
}

// Checks and BatchParams of a uniform batch (`len`-byte records at a pitch of `stride`) under the context's key or d_keys
static int uniform_params(BatchParams& p, const uint8_t* d_keys, const uint8_t* d_iv, int iv_is_j0, const uint8_t* d_aad,
                          uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                          uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs)
{
    if (n_msgs && len && (!d_in || !d_out)) return AGCM_E_BAD_ARG;
    if (stride < len || (aad_len && (!d_aad || aad_stride < aad_len))) return AGCM_E_BAD_LEN;
    // counter range AND the 32-bit block index of the unified AAD | payload | length sequence
    if (((len + 15) >> 4) > kMaxBlocks || ((aad_len + 15) >> 4) + ((len + 15) >> 4) + 1 > 0xFFFFFFFFull)
        return AGCM_E_COUNTER_OVERFLOW;
    memset(&p, 0, sizeof(p));
    p.keys = d_keys;
    p.iv = d_iv;
    p.iv_is_j0 = iv_is_j0 ? 1u : 0u;
    p.aad = aad_len ? d_aad : nullptr;
    p.in = d_in;
    p.out = d_out;
    p.tag = d_tag;
    p.ok = d_ok;
    p.len = len;
    p.stride = stride;
    p.aad_len = aad_len;
    p.aad_stride = aad_stride;
    return AGCM_OK;
}

static int batch_offsets(agcm_ctx* c, int decrypt, int lanes, uint64_t avg_len_hint, const uint8_t* d_iv, int iv_is_j0,
                         const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                         uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    if (!c) return AGCM_E_BAD_ARG;
    BatchParams p;
    int rc = offsets_params(p, nullptr, d_iv, iv_is_j0, d_aad, d_aad_off, d_in, d_in_off, d_out, d_tag, d_ok, n_msgs);
    if (rc) return rc;
    return batch_common(c, decrypt, lanes, avg_len_hint, p, n_msgs, stream);
}

static int batch_uniform(agcm_ctx* c, int decrypt, int lanes, const uint8_t* d_iv, int iv_is_j0, const uint8_t* d_aad,
                         uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                         uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    if (!c) return AGCM_E_BAD_ARG;
    BatchParams p;
    int rc = uniform_params(p, nullptr, d_iv, iv_is_j0, d_aad, aad_len, aad_stride, d_in, d_out, len, stride, d_tag, d_ok, n_msgs);
    if (rc) return rc;
    const bool aligned16 = ((((uintptr_t)d_in | (uintptr_t)d_out) | stride) & 15) == 0;
    if (lanes == 2048 && !tile_eligible(c, lanes, p, n_msgs)) return AGCM_E_BAD_ARG;
    if (n_msgs && tile_eligible(c, lanes, p, n_msgs)) return batch_tile(c, decrypt, p, n_msgs, (cudaStream_t)stream);
    // work estimate for the layout choice: an AAD block costs about a quarter of a payload block (no AES)
    return batch_common(c, decrypt, lanes, len + (d_aad ? aad_len / 4 : 0), p, n_msgs, stream, aligned16);
}

int agcm_batch_crypt(agcm_ctx* c, int decrypt, int lanes, uint64_t avg_len_hint, const uint8_t* d_iv12,
                     const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                     uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    return batch_offsets(c, decrypt, lanes, avg_len_hint, d_iv12, 0, d_aad, d_aad_off, d_in, d_in_off, d_out, d_tag, d_ok, n_msgs,
                         stream);
}

int agcm_batch_crypt_j0(agcm_ctx* c, int decrypt, int lanes, uint64_t avg_len_hint, const uint8_t* d_j0,
                        const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                        uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    return batch_offsets(c, decrypt, lanes, avg_len_hint, d_j0, 1, d_aad, d_aad_off, d_in, d_in_off, d_out, d_tag, d_ok, n_msgs,
                         stream);
}

int agcm_batch_crypt_uniform(agcm_ctx* c, int decrypt, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad,
                             uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                             uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    return batch_uniform(c, decrypt, lanes, d_iv12, 0, d_aad, aad_len, aad_stride, d_in, d_out, len, stride, d_tag, d_ok, n_msgs,
                         stream);
}

int agcm_batch_crypt_uniform_j0(agcm_ctx* c, int decrypt, int lanes, const uint8_t* d_j0, const uint8_t* d_aad,
                                uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                                uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    return batch_uniform(c, decrypt, lanes, d_j0, 1, d_aad, aad_len, aad_stride, d_in, d_out, len, stride, d_tag, d_ok, n_msgs,
                         stream);
}

int agcm_batch_crypt_slots(agcm_ctx* c, int decrypt, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad,
                           const uint32_t* d_aad_len, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out,
                           const uint32_t* d_len, uint64_t stride, uint64_t avg_len_hint, uint8_t* d_tag, uint8_t* d_ok,
                           size_t n_msgs, void* stream)
{
    if (!c || !d_len) return AGCM_E_BAD_ARG;
    if (n_msgs && stride && (!d_in || !d_out)) return AGCM_E_BAD_ARG;
    const bool has_aad = d_aad && (d_aad_len || aad_len);
    if (has_aad && (aad_stride < aad_len || aad_stride == 0)) return AGCM_E_BAD_LEN;
    if (((stride + 15) >> 4) > kMaxBlocks || ((aad_stride + 15) >> 4) + ((stride + 15) >> 4) + 1 > 0xFFFFFFFFull)
        return AGCM_E_COUNTER_OVERFLOW;   // no slot can hold a message beyond the limits
    BatchParams p;
    memset(&p, 0, sizeof(p));
    p.iv = d_iv12;
    p.aad = has_aad ? d_aad : nullptr;
    p.in = d_in;
    p.out = d_out;
    p.tag = d_tag;
    p.ok = d_ok;
    p.len = stride;
    p.stride = stride;
    p.len_arr = d_len;
    p.aad_len = has_aad ? aad_len : 0;
    p.aad_stride = has_aad ? aad_stride : 0;
    p.aad_len_arr = has_aad ? d_aad_len : nullptr;
    const bool aligned16 = ((((uintptr_t)d_in | (uintptr_t)d_out) | stride) & 15) == 0;
    if (lanes == 2048 && !tile_slots_eligible(c, lanes, p, n_msgs)) return AGCM_E_BAD_ARG;   // needs 16-byte aligned slots
    if (n_msgs && tile_slots_eligible(c, lanes, p, n_msgs)) return batch_tile_slots(c, decrypt, p, n_msgs, (cudaStream_t)stream);
    return batch_common(c, decrypt, lanes, avg_len_hint ? avg_len_hint : stride / 2, p, n_msgs, stream, aligned16);
}

int agcm_batch_derive_j0(agcm_ctx* c, const uint8_t* d_iv, const uint64_t* d_iv_off, uint64_t iv_len, size_t n_msgs,
                         uint8_t* d_j0, void* stream)
{
    if (!c || (n_msgs && (!d_iv || !d_j0))) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (!d_iv_off && iv_len == 0) return AGCM_E_BAD_LEN;
    AG_CUDA(c, cudaSetDevice(c->device));
    AG_CUDA(c, ag_launch_batch_j0(c->d_key, d_iv, d_iv_off, iv_len, n_msgs, d_j0, (cudaStream_t)stream));
    if (n_msgs) c->launches++;
    return AGCM_OK;
}

// tile: through k_batch_perkey_tile (perkey_tile_eligible); a forced tiled call goes to the launch even when empty
static int perkey_common(agcm_ctx* c, int mode, int decrypt, BatchParams& p, size_t n_msgs, bool tile, cudaStream_t st)
{
    const int nr = mode_to_nr(mode);
    if (!nr) return AGCM_E_BAD_MODE;
    if (n_msgs == 0 && !tile) return AGCM_OK;
    if (!p.keys || !p.iv || !p.tag || (decrypt && !p.ok)) return AGCM_E_BAD_ARG;
    AG_CUDA(c, cudaSetDevice(c->device));
    p.key = nullptr;
    p.te0 = c->d_te0;
    p.n_msgs = n_msgs;
    if (tile) {
        TileParams t;
        int rc = tile_records(c, t, p);
        if (rc) return rc;
        return tile_launch(c, t, nr, decrypt, 0, st);
    }
    if ((p.in_off || p.aad_off) && n_msgs >= 1024 && n_msgs < 0xFFFFFF00ull && !c->no_ticket && !getenv("AGCM_NO_LEN_SORT")) {
        // messages of different lengths, a message per lane: take them in length order (as batch_common does), so that
        // the 32 messages of a warp are equally long; thread g then works on perm[g], perm[g + grid], ...
        int rc = len_sort(c, p, n_msgs, st);
        if (rc) return rc;
        rc = zeroed_ticket(c, 1, st, p.ticket);   // groups of 32 messages, longest first, to whichever warp is free
        if (rc) return rc;
    }
    AG_CUDA(c, ag_launch_batch_perkey(p, nr, decrypt, c->ncta, st));
    c->launches++;
    return AGCM_OK;
}

int agcm_batch_crypt_perkey(agcm_ctx* c, int mode, int decrypt, const uint8_t* d_keys, const uint8_t* d_iv12,
                            const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                            uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream)
{
    if (!c) return AGCM_E_BAD_ARG;
    BatchParams p;
    int rc = offsets_params(p, d_keys, d_iv12, 0, d_aad, d_aad_off, d_in, d_in_off, d_out, d_tag, d_ok, n_msgs);
    if (rc) return rc;
    return perkey_common(c, mode, decrypt, p, n_msgs, false, (cudaStream_t)stream);
}

int agcm_batch_crypt_perkey_uniform(agcm_ctx* c, int mode, int decrypt, const uint8_t* d_keys, const uint8_t* d_iv12,
                                    const uint8_t* d_aad, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in,
                                    uint8_t* d_out, uint64_t len, uint64_t stride, uint8_t* d_tag, uint8_t* d_ok,
                                    size_t n_msgs, void* stream)
{
    if (!c) return AGCM_E_BAD_ARG;
    BatchParams p;
    int rc = uniform_params(p, d_keys, d_iv12, 0, d_aad, aad_len, aad_stride, d_in, d_out, len, stride, d_tag, d_ok, n_msgs);
    if (rc) return rc;
    return perkey_common(c, mode, decrypt, p, n_msgs, perkey_tile_eligible(c, p, n_msgs), (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------
int agcm_host_alloc(void** out, size_t bytes)
{
    if (!out) return AGCM_E_BAD_ARG;
    return cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault) == cudaSuccess ? AGCM_OK : AGCM_E_CUDA;
}

void agcm_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

// granule of the host pipeline: the tuned size, grown for very long ranges so the partial list stays bounded
static uint64_t pick_chunk(const agcm_ctx* c, uint64_t n_bytes)
{
    uint64_t b = c->chunk_bytes;
    while ((n_bytes + b - 1) / b > SC_PARTS_MAX && b < kChunkBytesMax) {
        b <<= 1;
        if (b > kChunkBytesMax) b = kChunkBytesMax;   // a non-power-of-two AGCM_CHUNK_MB must not outgrow d_stage
    }
    return b;
}

// chunked H2D -> fused kernel -> D2H of one counter range; the per-chunk partials
// (each scaled for everything after it, including `blocks_after0`) land in
// c->d_chunk_partials[0..n_chunks).  Waits for slots 1..kSlots-1 and leaves hs[0] running.
static int host_pipeline(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block0, const uint8_t* h_in,
                         uint8_t* h_out, uint64_t n_bytes, uint64_t blocks_after0, uint64_t* n_chunks_out)
{
    const uint64_t nblocks = (n_bytes + 15) >> 4;
    const uint64_t kChunkBytes = pick_chunk(c, n_bytes);
    // ramped granule sizes (host_sched.h): the first kernel starts after `ramp_base` bytes, not after a whole granule
    uint64_t sizes[SC_PARTS_MAX];
    const uint64_t n_chunks = ag_chunk_schedule(n_bytes, kChunkBytes, c->ramp_base < kChunkBytes ? c->ramp_base : 0, sizes,
                                                (uint32_t)SC_PARTS_MAX);
    if (n_bytes && !n_chunks) return AGCM_E_BAD_LEN;
    const int mode = decrypt ? AG_MODE_DEC : AG_MODE_ENC;
    uint64_t off = 0;
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const int s = (int)(k % kSlots);
        cudaStream_t st = c->hs[s];
        const uint64_t nb = sizes[k];
        const uint64_t fb = off >> 4;
        const uint64_t after = nblocks - fb - ((nb + 15) >> 4) + blocks_after0;
        AG_CUDA(c, cudaMemcpyAsync(c->d_stage[s], h_in + off, nb, cudaMemcpyHostToDevice, st));
        int rc = run_stream(c, mode, h_iv12, first_block0 + fb, c->d_stage[s], c->d_stage[s], nb,
                            after, c->d_stage_parts[s], c->d_chunk_partials + 16 * k, st, c->d_counters + 1 + s);
        if (rc) return rc;
        AG_CUDA(c, cudaMemcpyAsync(h_out + off, c->d_stage[s], nb, cudaMemcpyDeviceToHost, st));
        off += nb;
    }
    for (int s = 1; s < kSlots; ++s) AG_CUDA(c, cudaStreamSynchronize(c->hs[s]));
    *n_chunks_out = n_chunks;
    return AGCM_OK;
}

int agcm_stream_part_host(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* h_in,
                          uint8_t* h_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t h_partial16[16])
{
    if (!c || !h_iv12 || !h_partial16 || (n_bytes && (!h_in || !h_out))) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    const uint64_t nb = (n_bytes + 15) >> 4;
    if (first_block > kMaxBlocks || nb > kMaxBlocks - first_block || blocks_after > kMaxBlocks - first_block - nb)
        return AGCM_E_COUNTER_OVERFLOW;
    if (blocks_after && (n_bytes & 15)) return AGCM_E_BAD_LEN;
    int rc = host_begin(c, 0);
    if (rc) return rc;
    uint64_t n_chunks = 0;
    rc = host_pipeline(c, decrypt, h_iv12, first_block, h_in, h_out, n_bytes, blocks_after, &n_chunks);
    if (rc) return rc;
    // xor of the chunk partials = this range's partial (exponent 0: already scaled)
    uint8_t* d_p = c->d_scratch + SC_PART_CT;
    if (n_chunks == 0) {
        AG_CUDA(c, cudaMemsetAsync(d_p, 0, 16, c->hs[0]));
    } else {
        AG_CUDA(c, ag_launch_xor_parts(c->d_chunk_partials, (uint32_t)n_chunks, d_p, c->hs[0]));
        c->launches++;
    }
    AG_CUDA(c, cudaMemcpyAsync(h_partial16, d_p, 16, cudaMemcpyDeviceToHost, c->hs[0]));
    AG_CUDA(c, cudaStreamSynchronize(c->hs[0]));
    return AGCM_OK;
}

int agcm_stream_finish_host(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], const uint8_t* h_partials16, int n_parts,
                            const uint8_t* h_aad, uint64_t aad_len, uint64_t ct_len, uint8_t h_tag[16], int* h_ok)
{
    if (!c || !h_iv12 || !h_tag || (n_parts && !h_partials16) || (aad_len && !h_aad) || (decrypt && !h_ok))
        return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (n_parts < 0 || (size_t)n_parts > kMaxChunks) return AGCM_E_BAD_ARG;
    int rc = host_begin(c, aad_len);
    if (rc) return rc;
    cudaStream_t st = c->hs[0];
    if (aad_len) AG_CUDA(c, cudaMemcpyAsync(c->aad_stage.p, h_aad, aad_len, cudaMemcpyHostToDevice, st));
    if (n_parts) AG_CUDA(c, cudaMemcpyAsync(c->d_chunk_partials, h_partials16, 16 * (size_t)n_parts, cudaMemcpyHostToDevice, st));
    uint8_t* d_tag = c->d_scratch + SC_TAG;
    uint8_t* d_ok = c->d_scratch + SC_OK;
    if (decrypt) AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag, 16, cudaMemcpyHostToDevice, st));
    rc = run_finish(c, decrypt, h_iv12, c->d_chunk_partials, n_parts, c->aad_stage.p, aad_len, ct_len, d_tag, d_ok, st);
    if (rc) return rc;
    return host_end(c, decrypt, h_tag, h_ok, st);
}

int agcm_stream_crypt_peer_host(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* h_in,
                                uint8_t* h_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* h_aad, uint64_t aad_len,
                                uint64_t total_len, uint8_t h_tag[16], int* h_ok)
{
    if (!c || !h_iv12 || !h_tag || (n_bytes && (!h_in || !h_out)) || (aad_len && !h_aad) || (decrypt && !h_ok))
        return AGCM_E_BAD_ARG;
    if (c->peer_world < 1) return AGCM_E_BAD_ARG;
    int rc = host_begin(c, aad_len);
    if (rc) return rc;
    cudaStream_t st = c->hs[0];
    uint32_t epoch = 0;
    rc = peer_begin(c, first_block, n_bytes, blocks_after, aad_len, total_len, st, &epoch);
    if (rc) return rc;
    if (aad_len) AG_CUDA(c, cudaMemcpyAsync(c->aad_stage.p, h_aad, aad_len, cudaMemcpyHostToDevice, st));
    uint8_t* d_tag = c->d_scratch + SC_TAG;
    uint8_t* d_ok = c->d_scratch + SC_OK;
    if (decrypt) AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag, 16, cudaMemcpyHostToDevice, st));
    uint64_t n_chunks = 0;
    rc = host_pipeline(c, decrypt, h_iv12, first_block, h_in, h_out, n_bytes, blocks_after, &n_chunks);
    if (rc) return rc;
    const uint8_t* d_p = nullptr;   // null = the zero partial of an empty range
    if (n_chunks) {
        AG_CUDA(c, ag_launch_xor_parts(c->d_chunk_partials, (uint32_t)n_chunks, c->d_scratch + SC_PART_CT, st));
        c->launches++;
        d_p = c->d_scratch + SC_PART_CT;
    }
    AG_CUDA(c, ag_launch_peer_post(c->d_peer_bufs, (uint32_t)c->peer_rank, (uint32_t)c->peer_world, epoch, d_p, st));
    c->launches++;
    rc = peer_finish(c, decrypt, h_iv12, c->aad_stage.p, aad_len, total_len, d_tag, d_ok, st, epoch, false);
    if (rc) return rc;
    rc = host_end(c, decrypt, h_tag, h_ok, st);
    if (rc) return rc;
    if (*(volatile uint32_t*)c->h_peer_status) return AGCM_E_PEER_TIMEOUT;
    return AGCM_OK;
}

int agcm_stream_crypt_host(agcm_ctx* c, int decrypt, const uint8_t h_iv12[12], const uint8_t* h_aad, uint64_t aad_len,
                           const uint8_t* h_in, uint8_t* h_out, uint64_t n_bytes, uint8_t h_tag[16], int* h_ok)
{
    if (!c || !h_iv12 || !h_tag || (n_bytes && (!h_in || !h_out)) || (aad_len && !h_aad) || (decrypt && !h_ok))
        return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (((n_bytes + 15) >> 4) > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
    int rc = host_begin(c, aad_len);
    if (rc) return rc;
    if (aad_len) AG_CUDA(c, cudaMemcpyAsync(c->aad_stage.p, h_aad, aad_len, cudaMemcpyHostToDevice, c->hs[0]));
    uint8_t* d_tag = c->d_scratch + SC_TAG;
    uint8_t* d_ok = c->d_scratch + SC_OK;
    const uint64_t one_shot = (c->ramp_base && 2 * c->ramp_base < c->chunk_bytes) ? 2 * c->ramp_base : c->chunk_bytes;
    if (n_bytes && n_bytes <= one_shot && aad_len <= kAadInlineMax) {
        // short message: copy in, ONE launch (the kernel's last CTA finishes the tag), copy out, one wait;
        // anything longer overlaps its copies with the kernel granule by granule
        cudaStream_t st = c->hs[0];
        AG_CUDA(c, cudaMemcpyAsync(c->d_stage[0], h_in, n_bytes, cudaMemcpyHostToDevice, st));
        if (decrypt) AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag, 16, cudaMemcpyHostToDevice, st));
        rc = agcm_stream_crypt(c, decrypt, h_iv12, c->aad_stage.p, aad_len, c->d_stage[0], c->d_stage[0], n_bytes, d_tag, d_ok,
                               st);
        if (rc) return rc;
        AG_CUDA(c, cudaMemcpyAsync(h_out, c->d_stage[0], n_bytes, cudaMemcpyDeviceToHost, st));
    } else {
        uint64_t n_chunks = 0;
        rc = host_pipeline(c, decrypt, h_iv12, 0, h_in, h_out, n_bytes, 0, &n_chunks);
        if (rc) return rc;
        if (decrypt) AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag, 16, cudaMemcpyHostToDevice, c->hs[0]));
        rc = run_finish(c, decrypt, h_iv12, c->d_chunk_partials, (int)n_chunks, c->aad_stage.p, aad_len, n_bytes, d_tag, d_ok,
                        c->hs[0]);
        if (rc) return rc;
    }
    return host_end(c, decrypt, h_tag, h_ok, c->hs[0]);
}

int agcm_stream_decrypt_verified_host(agcm_ctx* c, const uint8_t* h_iv, size_t iv_len, const uint8_t* h_aad, uint64_t aad_len,
                                      const uint8_t* h_ct, uint8_t* h_pt, uint64_t n_bytes, const uint8_t h_tag[16], int* h_ok)
{
    if (!c || !h_iv || !h_tag || !h_ok || (n_bytes && (!h_ct || !h_pt)) || (aad_len && !h_aad)) return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (((n_bytes + 15) >> 4) > kMaxBlocks) return AGCM_E_COUNTER_OVERFLOW;
    int rc = host_begin(c, aad_len);
    if (rc) return rc;
    rc = grow(c, c->verify, n_bytes);   // the ciphertext stays in HBM between the two passes
    if (rc) return rc;
    uint8_t j0[16];
    rc = resolve_j0(c, h_iv, iv_len, j0, c->hs[0]);
    if (rc) return rc;
    J0Scope scope(c, j0);
    const uint64_t nblocks = (n_bytes + 15) >> 4, chunk = pick_chunk(c, n_bytes);
    const uint64_t n_chunks = (n_bytes + chunk - 1) / chunk;
    if (n_chunks > SC_PARTS_MAX) return AGCM_E_BAD_LEN;
    // pass 1: copy in and absorb, chunk by chunk (the copy of chunk k+1 overlaps the GHASH of chunk k)
    if (aad_len) AG_CUDA(c, cudaMemcpyAsync(c->aad_stage.p, h_aad, aad_len, cudaMemcpyHostToDevice, c->hs[0]));
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const int s = (int)(k % kSlots);
        const uint64_t off = k * chunk, nb = (n_bytes - off) < chunk ? (n_bytes - off) : chunk;
        const uint64_t after = nblocks - (off >> 4) - ((nb + 15) >> 4);
        AG_CUDA(c, cudaMemcpyAsync(c->verify.p + off, h_ct + off, nb, cudaMemcpyHostToDevice, c->hs[s]));
        rc = run_stream(c, AG_MODE_GHASH_ONLY, j0, 0, c->verify.p + off, nullptr, nb, after, c->d_stage_parts[s],
                        c->d_chunk_partials + 16 * k, c->hs[s], c->d_counters + 1 + s);
        if (rc) return rc;
    }
    for (int s = 1; s < kSlots; ++s) AG_CUDA(c, cudaStreamSynchronize(c->hs[s]));
    uint8_t* d_tag = c->d_scratch + SC_TAG;
    uint8_t* d_ok = c->d_scratch + SC_OK;
    AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag, 16, cudaMemcpyHostToDevice, c->hs[0]));
    rc = run_finish(c, 1, j0, c->d_chunk_partials, (int)n_chunks, c->aad_stage.p, aad_len, n_bytes, d_tag, d_ok, c->hs[0]);
    if (rc) return rc;
    rc = host_end(c, 1, nullptr, h_ok, c->hs[0]);
    if (rc || !*h_ok) return rc;   // not authentic: no plaintext byte leaves the device
    // pass 2: GCTR in place, chunk by chunk, copy out
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const int s = (int)(k % kSlots);
        const uint64_t off = k * chunk, nb = (n_bytes - off) < chunk ? (n_bytes - off) : chunk;
        rc = run_stream(c, AG_MODE_CTR_ONLY, j0, off >> 4, c->verify.p + off, c->verify.p + off, nb, 0, c->d_stage_parts[s], nullptr,
                        c->hs[s], c->d_counters + 1 + s);
        if (rc) return rc;
        AG_CUDA(c, cudaMemcpyAsync(h_pt + off, c->verify.p + off, nb, cudaMemcpyDeviceToHost, c->hs[s]));
    }
    for (int s = 0; s < kSlots; ++s) AG_CUDA(c, cudaStreamSynchronize(c->hs[s]));
    return AGCM_OK;
}

int agcm_stream_crypt_iv_host(agcm_ctx* c, int decrypt, const uint8_t* h_iv, size_t iv_len, const uint8_t* h_aad,
                              uint64_t aad_len, const uint8_t* h_in, uint8_t* h_out, uint64_t n_bytes, uint8_t h_tag[16],
                              int* h_ok)
{
    if (!c || !h_iv) return AGCM_E_BAD_ARG;
    if (iv_len == 12) return agcm_stream_crypt_host(c, decrypt, h_iv, h_aad, aad_len, h_in, h_out, n_bytes, h_tag, h_ok);
    int rc = host_begin(c, 0);
    if (rc) return rc;
    uint8_t j0[16];
    rc = resolve_j0(c, h_iv, iv_len, j0, c->hs[0]);
    if (rc) return rc;
    J0Scope scope(c, j0);
    return agcm_stream_crypt_host(c, decrypt, j0, h_aad, aad_len, h_in, h_out, n_bytes, h_tag, h_ok);
}

int agcm_batch_crypt_uniform_host(agcm_ctx* c, int decrypt, int lanes, const uint8_t* h_iv12, const uint8_t* h_aad,
                                  uint64_t aad_len, uint64_t aad_stride, const uint8_t* h_in, uint8_t* h_out,
                                  uint64_t len, uint64_t stride, uint8_t* h_tag, uint8_t* h_ok, size_t n_msgs)
{
    if (!c || !h_iv12 || !h_tag || (len && (!h_in || !h_out)) || (aad_len && !h_aad) || (decrypt && !h_ok))
        return AGCM_E_BAD_ARG;
    if (!c->key_set) return AGCM_E_NO_KEY;
    if (stride < len || (aad_len && aad_stride < aad_len)) return AGCM_E_BAD_LEN;
    if (n_msgs == 0) return AGCM_OK;
    int rc = host_begin(c, 0);
    if (rc) return rc;
    // messages per chunk: payload fits the stage buffer, side data fits the aux buffer
    const uint64_t per_msg_aux = 12 + 16 + 1 + aad_stride + 16;
    const uint64_t kChunkBytes = 32u << 20;
    uint64_t m_chunk = stride ? kChunkBytes / stride : n_msgs;
    const uint64_t m_aux = (kChunkBytes / 8) / per_msg_aux;
    if (m_chunk > m_aux) m_chunk = m_aux;
    if (m_chunk == 0) return AGCM_E_BAD_LEN;  // one record larger than the staging granule: use the stream API
    // fix the lane count once so every chunk runs the same kernel
    int g = pick_lanes(c, lanes, n_msgs < m_chunk ? n_msgs : m_chunk, len);
    if (g < 0) return AGCM_E_BAD_ARG;
    // the chunks run concurrently on the pipeline's streams and the segment layout keeps its
    // partials in one scratch buffer per context: whole-message layouts only on this path
    if (g > 4096) g = 32;     // (the warp-unit layout as well)
    if (g > 1024) g = 1024;
    // (and no ticket-driven distribution: the context has ONE ticket word)
    struct NoTicket {
        agcm_ctx* c;
        explicit NoTicket(agcm_ctx* ctx) : c(ctx) { c->no_ticket = true; }
        ~NoTicket() { c->no_ticket = false; }
    } no_ticket_scope(c);
    uint64_t k = 0;
    for (uint64_t m0 = 0; m0 < n_msgs; m0 += m_chunk, ++k) {
        const int s = (int)(k % kSlots);
        cudaStream_t st = c->hs[s];
        const uint64_t nm = (n_msgs - m0) < m_chunk ? (n_msgs - m0) : m_chunk;
        uint8_t* d_data = c->d_stage[s];
        uint8_t* aux = c->d_stage_aux[s];
        uint8_t* d_iv = aux;                          // nm x 12
        uint8_t* d_tag = aux + ((12 * m_chunk + 15) & ~15ull);  // nm x 16
        uint8_t* d_ok = d_tag + 16 * m_chunk;         // nm
        uint8_t* d_aad = d_ok + ((m_chunk + 15) & ~15ull);
        const uint64_t span = (nm - 1) * stride + len;
        if (len) AG_CUDA(c, cudaMemcpyAsync(d_data, h_in + m0 * stride, span, cudaMemcpyHostToDevice, st));
        AG_CUDA(c, cudaMemcpyAsync(d_iv, h_iv12 + 12 * m0, 12 * nm, cudaMemcpyHostToDevice, st));
        if (aad_len)
            AG_CUDA(c, cudaMemcpyAsync(d_aad, h_aad + m0 * aad_stride, (nm - 1) * aad_stride + aad_len, cudaMemcpyHostToDevice, st));
        if (decrypt) AG_CUDA(c, cudaMemcpyAsync(d_tag, h_tag + 16 * m0, 16 * nm, cudaMemcpyHostToDevice, st));
        rc = agcm_batch_crypt_uniform(c, decrypt, g, d_iv, d_aad, aad_len, aad_stride, d_data, d_data, len, stride, d_tag,
                                      d_ok, nm, st);
        if (rc) return rc;
        if (len) {
            if (stride == len) {
                AG_CUDA(c, cudaMemcpyAsync(h_out + m0 * stride, d_data, span, cudaMemcpyDeviceToHost, st));
            } else {
                // keep the caller's inter-record padding untouched
                AG_CUDA(c, cudaMemcpy2DAsync(h_out + m0 * stride, stride, d_data, stride, len, nm, cudaMemcpyDeviceToHost, st));
            }
        }
        if (decrypt) AG_CUDA(c, cudaMemcpyAsync(h_ok + m0, d_ok, nm, cudaMemcpyDeviceToHost, st));
        else AG_CUDA(c, cudaMemcpyAsync(h_tag + 16 * m0, d_tag, 16 * nm, cudaMemcpyDeviceToHost, st));
    }
    for (int s = 0; s < kSlots; ++s) AG_CUDA(c, cudaStreamSynchronize(c->hs[s]));
    return AGCM_OK;
}

}  // extern "C"
#pragma GCC visibility pop

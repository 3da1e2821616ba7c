/*
 * aesgcm_b200.h -- C ABI of the B200 (sm_100a) AES-GCM engine.
 *
 * This is the drop-in boundary for the golden-model side of
 * BLu85/AES-GCM-128-192-256-bits.  The reference has no C API: its "plugin
 * interface" is the Python surface tb/gcm_model.py (class gcm) and
 * tb/key_exp.py (aes_expand_key), which delegate to pycryptodome.  Each entry
 * point below names the reference interface it replaces (file:line relative to
 * the reference checkout).  INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.
 *
 * Conventions
 *   - Plain C: pointers and sizes only.  `d_` = DEVICE pointer, `h_` = HOST
 *     pointer.  The caller owns every buffer; the library allocates only inside
 *     the context.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Device
 *     entry points are asynchronous on that stream.  A context owns scratch
 *     buffers: use one context per concurrently active stream.
 *   - The library keeps no global mutable state.  A context is not locked internally: one
 *     host thread at a time per context; distinct contexts (same or different devices) may be
 *     used from different threads at the same time.
 *   - Return 0 on success, a negative AGCM_E_* otherwise.  Nothing throws.
 *   - mode = key size in bits: 128 / 192 / 256 (src/aes_pkg.vhd:31-33 Nr=10/12/14).
 *   - IV is 96 bits as in the IP; IVs of any other length (pycryptodome's AES.new(nonce=...), which the
 *     reference model calls at tb/gcm_model.py:18, accepts them) go through the *_iv entry points or,
 *     for shards / batches / GCTR, through agcm_derive_j0 / agcm_batch_derive_j0 + the *_j0 forms; the counter
 *     block is IV || cnt32, cnt = 1 for J0 and 2.. for data (src/aes_icb.vhd:34,99-100,118).  More than 2^32-2 data
 *     blocks per IV is AGCM_E_COUNTER_OVERFLOW (the IP raises its overflow flag,
 *     src/aes_icb.vhd:65,114,119).
 *   - There is no CPU fallback.  Every call needs a CUDA device of compute
 *     capability 10.x.
 *   - Limits: payload per IV <= (2^32-2) x 16 bytes (the 32-bit block counter); a batched
 *     message holds fewer than 2^32 blocks of AAD + payload + 1 (checked for the uniform forms; for the
 *     offset forms the offsets live in device memory and the limit is the caller's to keep: UNCHECKED);
 *     agcm_stream_finish takes up to
 *     1024 shard partials; agcm_peer_setup / agcm_peer_import up to 16 ranks; the host-buffer stream call up to
 *     1024 x 64 MiB per call.  AAD of any length (bytes 4097.. run through the grid-wide GHASH).
 *   - Device buffers may have any byte alignment; 16-byte alignment selects the 128-bit
 *     load/store path (4-byte alignment a 32-bit path, anything else bytes; batched messages that a single
 *     lane walks are read and written as realigned 16-byte granules whatever their address).  Fixed-size
 *     records at a 16-byte-aligned pitch additionally take the TMA-staged batch kernels.
 *   - Environment (read by the library, all optional; none changes a result): AGCM_CHUNK_MB (granule of
 *     the host-buffer pipeline, 1..64, default 32), AGCM_RAMP_KB (its first and last granule, default 1024;
 *     0 = equal granules), AGCM_PEER_TIMEOUT_MS (default 10000), and the A/B
 *     switches of the layout choice AGCM_NO_TILE, AGCM_PERKEY_TILE=0|1, AGCM_NO_WARP_UNITS,
 *     AGCM_WARP_MIN_BLOCKS, AGCM_NO_LEN_SORT (ragged batches in arrival order), AGCM_NO_LEN_CLASSES
 *     (sorted, but one lane count for the whole batch), AGCM_GATHER (slots: the row-gathering kernel by default).
 */
#ifndef AESGCM_B200_H
#define AESGCM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGCM_OK 0
#define AGCM_E_BAD_MODE (-1)         /* mode not 128/192/256, or key length mismatch (config/gcm_utils.py:163-171) */
#define AGCM_E_BAD_LEN (-2)          /* inconsistent lengths / offsets */
#define AGCM_E_COUNTER_OVERFLOW (-3) /* > 2^32-2 blocks under one IV (src/aes_icb.vhd:114) */
#define AGCM_E_CUDA (-4)             /* CUDA runtime error; see agcm_last_cuda_error() */
#define AGCM_E_NO_KEY (-5)           /* agcm_set_key() has not been called on this context */
#define AGCM_E_BAD_ARG (-6)          /* null pointer / unsupported argument */
#define AGCM_E_NO_DEVICE (-7)        /* no sm_100 device: the engine has no other path */
#define AGCM_E_PEER_TIMEOUT (-8)     /* a rank never posted its shard partial: that message FAILED CLOSED (tag zeroed, ok = 0) */

typedef struct agcm_ctx agcm_ctx;

/* ---- context ------------------------------------------------------------ */
int agcm_ctx_create(agcm_ctx** out, int device);
/* testing/tuning: explicit persistent-grid shape (n_cta <= 256, threads power of two <= 1024; 0 = default) */
int agcm_ctx_create_ex(agcm_ctx** out, int device, int n_cta, int threads);
void agcm_ctx_destroy(agcm_ctx* ctx);
const char* agcm_strerror(int rc);
int agcm_last_cuda_error(const agcm_ctx* ctx); /* cudaError_t of the last failure */
const char* agcm_last_cuda_error_string(const agcm_ctx* ctx);
/* persistent-grid shape and SM count actually used */
int agcm_get_info(const agcm_ctx* ctx, int* n_cta, int* threads, int* sm_count);
/* number of kernels this context has launched so far (bench.py gpu_launches) */
uint64_t agcm_launch_count(const agcm_ctx* ctx);
/* Optional CUDA-event timing of every fused stream-kernel launch, on the stream it
 * is launched on (bench.py roofline).  read: sum of durations and launch count since enable. */
int agcm_timing_enable(agcm_ctx* ctx, int on);
int agcm_timing_read(agcm_ctx* ctx, double* total_ms, uint64_t* n_launches);

/* ---- key schedule ---------------------------------------------------------
 * Replaces tb/key_exp.py:118 aes_expand_key(key_hex, size) and the on-the-fly
 * aes_kexp block (config/config_aes_kexp.py:128-159): n_keys raw keys of
 * mode/8 bytes each -> n_keys x (Nr+1)*16 bytes (176/208/240), stage r at bytes
 * 16r..16r+15, byte-identical to the reference list.  One thread per key. */
int agcm_key_expand(agcm_ctx* ctx, int mode, const uint8_t* d_keys, size_t n_keys, uint8_t* d_round_keys, void* stream);
/* host convenience over the same kernel (1 key), for the key_exp.py adapter */
int agcm_key_expand_host(agcm_ctx* ctx, int mode, const uint8_t* h_key, uint8_t* h_round_keys);

/* ---- shared key ------------------------------------------------------------
 * Replaces gcm_model.gcm.__init__'s key handling (tb/gcm_model.py:16,18) and the
 * DUT key load: raw key (tb/gcm_gctr.py:144-175, expanded on the device) or
 * pre-expanded stages (tb/gcm_gctr.py:180-214, config/config_aes_kprexp.py:66-95).
 * key_len = mode/8 when pre_expanded == 0, (Nr+1)*16 otherwise.
 * Derives on the device H = E_K(0^128) (src/gcm_gctr.vhd:141-144,
 * src/gcm_ghash.vhd:128-139), its powers and the Shoup tables; H stays valid
 * until the next agcm_set_key (src/gcm_ghash.vhd:123).  Synchronous: it first waits for all
 * work queued on the device (no earlier call may still read the old key), runs one kernel and
 * reads the stage keys and H back; about 75 us.  Loading the key that is already
 * loaded returns at once: H is kept until a NEW key arrives, as in the IP. */
int agcm_set_key(agcm_ctx* ctx, int mode, int pre_expanded, const uint8_t* h_key, size_t key_len);
int agcm_get_round_keys(const agcm_ctx* ctx, uint8_t* h_round_keys, size_t cap); /* returns byte count */
int agcm_get_h(const agcm_ctx* ctx, uint8_t h_h16[16]);

/* ---- one message, data resident in HBM ---------------------------------------
 * Replaces load_aad / load_plain_text / load_cipher_text / get_tag of
 * tb/gcm_model.py:21-51 for a whole message (the datapath of src/gcm_gctr.vhd:150
 * + src/gcm_ghash.vhd:225-293).
 *   decrypt == 0: d_out = CT, d_tag receives the 16-byte tag.
 *   decrypt == 1: d_out = PT, d_tag holds the EXPECTED tag, *d_ok = 1 if it
 *                 matches the computed tag, else 0 (tb/gcm_model.py:42-51).
 * d_in/d_out may alias exactly (in place).  16-byte alignment of d_in/d_out
 * selects the 128-bit load/store path. */
int agcm_stream_crypt(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], const uint8_t* d_aad, uint64_t aad_len,
                      const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint8_t* d_tag, uint8_t* d_ok, void* stream);

/* RELEASE OF UNVERIFIED PLAINTEXT: like the reference model (tb/gcm_model.py:29-30 hands out every
 * block at load_cipher_text time, the tag is only checked at get_tag), every decrypt call above and
 * below writes the plaintext BEFORE the tag is known to match -- on the host-buffer paths each chunk
 * is copied back while later chunks are still in flight.  Callers that must not see unauthenticated
 * plaintext use the two-pass forms: this one for a message on one GPU, agcm_batch_decrypt_verified* for
 * batches, agcm_stream_decrypt_verified_peer(_host) for a message sharded over GPUs (below).
 * agcm_stream_decrypt_verified: pass 1 = GHASH over the ciphertext + tag check (about 4x the rate of
 * the fused pass), pass 2 = GCTR gated ON THE DEVICE by the flag pass 1 wrote: when the tag does
 * not match, *d_ok = 0 and d_pt is not written at all.  IV of any length (host pointer). */
int agcm_stream_decrypt_verified(agcm_ctx* ctx, const uint8_t* h_iv, size_t iv_len, const uint8_t* d_aad, uint64_t aad_len,
                                 const uint8_t* d_ct, uint8_t* d_pt, uint64_t n_bytes, const uint8_t* d_tag, uint8_t* d_ok,
                                 void* stream);

/* VERIFY-THEN-RELEASE BATCHES: agcm_batch_decrypt_verified* take the arguments of their releasing counterparts
 * (agcm_batch_crypt, _j0, _uniform, _uniform_j0, _slots, _perkey, _perkey_uniform) minus `decrypt`, and guarantee:
 *   - d_ok[i] = 1 if message i's tag matches, else 0;
 *   - the plaintext bytes of message i are written if and only if d_ok[i] == 1;
 *   - no other byte of d_pt is ever written: not a failed message, not the gaps between offsets, not slot padding past
 *     d_len[i], not record padding past len.  d_ct == d_pt (exactly aliased) is allowed: a failed message then still
 *     holds its ciphertext.
 * Argument checks, error codes and length limits are those of the counterpart; d_tag and d_ok are required
 * (AGCM_E_BAD_ARG).  n_msgs == 0 returns AGCM_OK and launches nothing.  Shared key: two passes in stream order, no host
 * round trip -- pass 1 absorbs AAD | CT | length block with no keystream (the lane-group or warp-unit layouts; lanes
 * chooses this pass only and takes 0, 1, 2, 4, 8, 16, 32 or 4096 + S; 1024, 1024 + S and 2048 are AGCM_E_BAD_ARG),
 * pass 2 runs GCTR over the payload of the whole batch cut flat into blocks, skipping every message whose flag is 0.
 * Per key: one launch, each lane checks its message's tag and then, only if it matched, decrypts it (the TMA-staged
 * per-key kernel has no verified form).  Scratch as for the other batch calls: one such call in flight per context. */
int agcm_batch_decrypt_verified(agcm_ctx* ctx, int lanes, uint64_t avg_len_hint, const uint8_t* d_iv12, const uint8_t* d_aad,
                                const uint64_t* d_aad_off, const uint8_t* d_ct, const uint64_t* d_in_off, uint8_t* d_pt,
                                const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_j0(agcm_ctx* ctx, int lanes, uint64_t avg_len_hint, const uint8_t* d_j0, const uint8_t* d_aad,
                                   const uint64_t* d_aad_off, const uint8_t* d_ct, const uint64_t* d_in_off, uint8_t* d_pt,
                                   const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_uniform(agcm_ctx* ctx, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad, uint64_t aad_len,
                                        uint64_t aad_stride, const uint8_t* d_ct, uint8_t* d_pt, uint64_t len, uint64_t stride,
                                        const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_uniform_j0(agcm_ctx* ctx, int lanes, const uint8_t* d_j0, const uint8_t* d_aad, uint64_t aad_len,
                                           uint64_t aad_stride, const uint8_t* d_ct, uint8_t* d_pt, uint64_t len, uint64_t stride,
                                           const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_slots(agcm_ctx* ctx, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad,
                                      const uint32_t* d_aad_len, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_ct,
                                      uint8_t* d_pt, const uint32_t* d_len, uint64_t stride, uint64_t avg_len_hint,
                                      const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_perkey(agcm_ctx* ctx, int mode, const uint8_t* d_keys, const uint8_t* d_iv12, const uint8_t* d_aad,
                                       const uint64_t* d_aad_off, const uint8_t* d_ct, const uint64_t* d_in_off, uint8_t* d_pt,
                                       const uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_decrypt_verified_perkey_uniform(agcm_ctx* ctx, int mode, const uint8_t* d_keys, const uint8_t* d_iv12,
                                               const uint8_t* d_aad, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_ct,
                                               uint8_t* d_pt, uint64_t len, uint64_t stride, const uint8_t* d_tag, uint8_t* d_ok,
                                               size_t n_msgs, void* stream);

/* The same for an IV of ANY length (SP 800-38D 7.1: J0 = GHASH_H(IV || 0^(s+64) || [len(IV)]_64),
 * derived on the device; iv_len == 12 is the plain call above).  The reference IP fixes the IV at
 * 96 bits (src/gcm_pkg.vhd:17), so this goes beyond it; pycryptodome's AES.new(nonce=...), which
 * the reference model calls (tb/gcm_model.py:18), accepts such nonces.  Synchronises `stream` once
 * for the J0 readback.  h_iv is a HOST pointer. */
int agcm_stream_crypt_iv(agcm_ctx* ctx, int decrypt, const uint8_t* h_iv, size_t iv_len, const uint8_t* d_aad,
                         uint64_t aad_len, const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint8_t* d_tag,
                         uint8_t* d_ok, void* stream);

/* Counter-range shard of one message (multi-GPU, SURVEY 8(e)): blocks
 * [first_block, first_block + ceil(n_bytes/16)) of the message, counter start
 * 2 + first_block.  n_bytes must be a multiple of 16 unless this is the last
 * shard.  Writes d_partial16 = sum_i C_i * H^(n_shard - i + blocks_after) in
 * natural GHASH byte order, i.e. already scaled for the `blocks_after` CT blocks
 * that follow the shard, so the partials of all shards simply XOR. */
int agcm_stream_part(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in,
                     uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t* d_partial16, void* stream);
/* Combine n_parts gathered partials with the AAD and the length block
 * (src/gcm_ghash.vhd:257) and E_K(J0) (src/gcm_ghash.vhd:293).  ct_len is the
 * TOTAL message length in bytes.  Tag semantics as agcm_stream_crypt. */
int agcm_stream_finish(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], const uint8_t* d_partials16, int n_parts,
                       const uint8_t* d_aad, uint64_t aad_len, uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok,
                       void* stream);

/* ---- IVs that are not 96 bits on the shard / peer / GCTR / batch entry points -----------------
 * agcm_derive_j0: J0 = IV || 0^31 1 for a 96-bit IV, else GHASH_H(IV || 0^(s+64) || [len(IV)]_64)
 * computed on the device (synchronous, host pointers).  The *_j0 forms take that 16-byte J0 in
 * place of the 12 IV bytes: the counter block of data block i is inc32^(i+1)(J0), the tag mask
 * E_K(J0).  For a 96-bit IV they are identical to the plain forms. */
int agcm_derive_j0(agcm_ctx* ctx, const uint8_t* h_iv, size_t iv_len, uint8_t h_j0[16]);
int agcm_gctr_j0(agcm_ctx* ctx, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in, uint8_t* d_out,
                 uint64_t n_bytes, void* stream);
int agcm_stream_part_j0(agcm_ctx* ctx, int decrypt, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in,
                        uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t* d_partial16, void* stream);
int agcm_stream_finish_j0(agcm_ctx* ctx, int decrypt, const uint8_t h_j0[16], const uint8_t* d_partials16, int n_parts,
                          const uint8_t* d_aad, uint64_t aad_len, uint64_t ct_len, uint8_t* d_tag, uint8_t* d_ok,
                          void* stream);
/* agcm_stream_crypt_peer (deferred == 0) / agcm_stream_crypt_peer_async (deferred != 0) with a J0 */
int agcm_stream_crypt_peer_j0(agcm_ctx* ctx, int decrypt, const uint8_t h_j0[16], uint64_t first_block, const uint8_t* d_in,
                              uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* d_aad, uint64_t aad_len,
                              uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, void* stream, int deferred);

/* ---- sharded message, partials exchanged over peer memory (NVLink) ---------------------------
 * Every rank needs every rank's exchange buffer mapped in its own process.  Two ways to set that up:
 *   - agcm_peer_export / agcm_peer_import (any client, one process per GPU or several contexts in one process):
 *     the library owns the buffers and moves them between processes as CUDA IPC handles.
 *       agcm_peer_export: on the first call allocates this context's exchange buffer (cudaMalloc, 2560 bytes, on the
 *         context's device) and writes an opaque AGCM_PEER_HANDLE_BYTES handle to it; later calls write the same
 *         handle.  The caller moves the handles between the ranks by any means (a file, a socket, MPI).  The buffer
 *         lives until agcm_ctx_destroy.
 *       agcm_peer_import: h_handles = world handles, rank w's at h_handles + w * AGCM_PEER_HANDLE_BYTES; entry `rank`
 *         must be this context's own export.  Maps every other rank's buffer (cudaIpcOpenMemHandle; a buffer of this
 *         same process is used at its own address, with peer access enabled when it lives on another device), then
 *         sets up as agcm_peer_setup does.  AGCM_E_BAD_ARG for a handle that is not one (wrong magic or version), a
 *         buffer under 2560 bytes, two entries naming the same buffer, an entry `rank` that is not this context's
 *         export, and the argument checks of agcm_peer_setup.  Barrier after the import, before the first exchange.
 *         A process may import a given device's handles into one CUDA context per device (the CUDA rule); the
 *         library uses the device's primary context, so several contexts on one device may import the same handles.
 *       agcm_peer_close: unmaps what the last import mapped and leaves the world: peer calls return AGCM_E_BAD_ARG
 *         until the next set-up.  Teardown: every rank calls agcm_peer_close, the ranks barrier, then each rank
 *         calls agcm_ctx_destroy (an exported buffer must not be freed while another process still maps it).
 *         agcm_ctx_destroy also closes any mappings still open.
 *     A second import, or an agcm_peer_setup after an import, first closes the previous import's mappings.
 *   - agcm_peer_setup (callers that map the buffers themselves): h_peer_ptrs[w] = device address, valid in THIS
 *     process, of rank w's exchange buffer (>= 2560 bytes); the caller keeps the buffers mapped while the world is in
 *     use.
 * Both zero this rank's buffer -- barrier before the first exchange.  world <= 16.  AGCM_PEER_TIMEOUT_MS
 * (environment, default 10000) bounds the wait.
 * agcm_stream_crypt_peer: agcm_stream_part + the 16-byte all-to-all + agcm_stream_finish without a
 * collective library call.  The last CTA of the bulk kernel stores the scaled partial into every
 * peer's buffer (plain stores over NVLink) and raises an epoch flag; it does NOT wait.  A one-warp
 * finish kernel on a side stream of the context waits (bounded) for the world's flags in this
 * rank's buffer, XORs the slots and finishes the tag on every rank (the two-way split of
 * src/gcm_ghash.vhd:317-344 at width `world`); `stream` then waits for that finish, so d_tag / d_ok
 * are valid in stream order as for every other call.
 * agcm_stream_crypt_peer_async: the same without the last wait -- the next message's bulk kernel
 * starts while this message's flags are still arriving, so the ranks are not barriered per message
 * (a rank may run up to 4 messages ahead of the slowest one; the exchange ring holds 8).  d_tag /
 * d_ok are valid on `stream` after agcm_peer_join(ctx, stream) (a stream-side wait, no host sync).
 * All ranks must make the same sequence of peer calls; n_bytes == 0 is allowed (a rank whose
 * counter range is empty still posts); aad_len <= 4096 (else use part + gather + finish).
 * FAILS CLOSED: if a rank never posts, the finish zeroes the tag, clears ok, and every later peer
 * call on the context returns AGCM_E_PEER_TIMEOUT until the exchange is set up again;
 * agcm_peer_status (synchronises the side stream) reports it too. */
#define AGCM_PEER_HANDLE_BYTES 128
int agcm_peer_export(agcm_ctx* ctx, uint8_t h_handle[AGCM_PEER_HANDLE_BYTES]);
int agcm_peer_import(agcm_ctx* ctx, int rank, int world, const uint8_t* h_handles);
int agcm_peer_close(agcm_ctx* ctx);
int agcm_peer_setup(agcm_ctx* ctx, int rank, int world, const uint64_t* h_peer_ptrs);
int agcm_peer_status(agcm_ctx* ctx, int* h_timed_out);
int agcm_peer_join(agcm_ctx* ctx, void* stream);
int agcm_stream_crypt_peer(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in,
                           uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after, const uint8_t* d_aad, uint64_t aad_len,
                           uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok, void* stream);
int agcm_stream_crypt_peer_async(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], uint64_t first_block,
                                 const uint8_t* d_in, uint8_t* d_out, uint64_t n_bytes, uint64_t blocks_after,
                                 const uint8_t* d_aad, uint64_t aad_len, uint64_t total_len, uint8_t* d_tag, uint8_t* d_ok,
                                 void* stream);

/* VERIFY-THEN-RELEASE SHARDED DECRYPT: agcm_stream_decrypt_verified_peer decrypts this rank's shard of a message sharded as
 * for agcm_stream_crypt_peer.  Pass 1 = GHASH over this rank's ciphertext, the scaled partial posted to every rank; the
 * one-warp finish compares the WORLD's tag with d_tag; pass 2 = GCTR over this rank's shard, gated on the device by that
 * flag.  IV of any length (host pointer, as agcm_stream_decrypt_verified).  Guarantees:
 *   - on every rank, *d_ok = 1 if and only if the tag of the whole message matches the d_tag that rank was given;
 *   - a rank writes its plaintext bytes if and only if its *d_ok == 1; no other byte of d_pt is ever written, so one
 *     flipped bit in any rank's ciphertext, in the AAD or in the tag makes every rank release nothing;
 *   - d_ct == d_pt (exactly aliased) is allowed: a failed shard then still holds its ciphertext;
 *   - FAILS CLOSED as the releasing calls: if a rank never posts, *d_ok = 0, nothing is released, and every later peer
 *     call returns AGCM_E_PEER_TIMEOUT until the exchange is set up again.
 * d_ok and d_pt are valid in stream order on `stream`.  There is no deferred form: release needs the world's tag, so every
 * message is a rank-wide wait.  Argument checks, error codes and limits are those of agcm_stream_crypt_peer (aad_len <= 4096,
 * the same first_block / blocks_after / total_len consistency, an empty counter range still posts, total_len == 0 = GMAC
 * only); d_tag and d_ok are required (AGCM_E_BAD_ARG).  The call takes one epoch of the exchange ring like every other peer
 * call, so it interleaves with the releasing calls as long as every rank makes the same sequence of calls.
 * agcm_stream_decrypt_verified_peer_host: the same from host buffers, as agcm_stream_decrypt_verified_host -- the shard is
 * copied into HBM once (n_bytes of device memory, kept by the context) and absorbed chunk by chunk; only when the world's
 * tag matches does the GCTR pass run and the plaintext travel back.  On a mismatch *h_ok = 0 and h_pt is untouched; if a
 * rank never posts, the call returns AGCM_E_PEER_TIMEOUT at once (h_pt untouched).  Synchronous. */
int agcm_stream_decrypt_verified_peer(agcm_ctx* ctx, const uint8_t* h_iv, size_t iv_len, uint64_t first_block,
                                      const uint8_t* d_ct, uint8_t* d_pt, uint64_t n_bytes, uint64_t blocks_after,
                                      const uint8_t* d_aad, uint64_t aad_len, uint64_t total_len,
                                      const uint8_t* d_tag, uint8_t* d_ok, void* stream);
int agcm_stream_decrypt_verified_peer_host(agcm_ctx* ctx, const uint8_t* h_iv, size_t iv_len, uint64_t first_block,
                                           const uint8_t* h_ct, uint8_t* h_pt, uint64_t n_bytes, uint64_t blocks_after,
                                           const uint8_t* h_aad, uint64_t aad_len, uint64_t total_len,
                                           const uint8_t h_tag[16], int* h_ok);

/* ---- many independent messages under the shared key ---------------------------
 * Message i: IV d_iv12[12i..], AAD d_aad[aad_off[i]..aad_off[i+1]), payload
 * d_in[in_off[i]..in_off[i+1]) -> d_out at the same offsets, tag at d_tag[16i..]
 * (produced for encrypt, expected for decrypt), d_ok[i] (decrypt only).
 * d_aad / d_aad_off may be NULL (no AAD).  lanes = threads cooperating on one
 * message (1,2,4,8,16,32; 1024 = one whole CTA per message; 1024+S, S a power of two up to 256 =
 * one CTA per 1/S of a message: counter-range segments whose scaled GHASH partials a second launch
 * XORs into the tag; 4096+S, 1 <= S <= 65536 = one WARP per 1/S of a message, units handed out by
 * an atomic ticket and the lane combine deferred to the end of the same launch -- the layout chosen for
 * messages from about 32 KiB; 2048 = the TMA-staged message-per-lane kernel, uniform and slots forms only,
 * 16-byte aligned buffers and pitch) or 0 = choose from n_msgs and avg_len_hint.  Every choice
 * produces the same bytes.  The segment / unit layouts keep their partials in a per-context
 * scratch buffer (grown on demand, which synchronises the device the first time): one such call
 * in flight per context. */
int agcm_batch_crypt(agcm_ctx* ctx, int decrypt, int lanes, uint64_t avg_len_hint, const uint8_t* d_iv12,
                     const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                     uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
/* Same, fixed-size records: message i at d_in + i*stride (len bytes), AAD at
 * d_aad + i*aad_stride (aad_len bytes). */
int agcm_batch_crypt_uniform(agcm_ctx* ctx, int decrypt, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad,
                             uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                             uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);

/* Fixed-pitch SLOTS holding messages of different lengths (a packet ring): message i is d_len[i] bytes at
 * d_in + i*stride (a length beyond the pitch is clamped to it), its AAD d_aad_len[i] bytes at d_aad + i*aad_stride
 * (d_aad_len NULL: aad_len bytes for every message; d_aad NULL: none).  With 16-byte aligned buffers and pitch every
 * access is a 128-bit one, whatever the lengths.  From 1024 messages on, this call and agcm_batch_crypt take the
 * messages in LENGTH order (a counting sort on the device, longest first, handed out by ticket): a warp works on
 * several messages in lock step, and side by side they should be equally long (an IMIX of 64 / 576 / 1500 B
 * packets: 2-4x).  avg_len_hint as in agcm_batch_crypt (0: half the pitch).  lanes = 2048 here names the
 * row-gathering form of the TMA-staged kernel (tile::gather4 / scatter4 over the sorted rows; 16-byte aligned buffers
 * and pitch, else AGCM_E_BAD_ARG): same bytes, within a few percent of the default either way. */
int agcm_batch_crypt_slots(agcm_ctx* ctx, int decrypt, int lanes, const uint8_t* d_iv12, const uint8_t* d_aad,
                           const uint32_t* d_aad_len, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in,
                           uint8_t* d_out, const uint32_t* d_len, uint64_t stride, uint64_t avg_len_hint, uint8_t* d_tag,
                           uint8_t* d_ok, size_t n_msgs, void* stream);

/* Batches whose IVs are not all 96 bits: agcm_batch_derive_j0 turns n IVs (d_iv_off: n+1 byte
 * offsets into d_iv, or NULL = fixed iv_len bytes each) into n 16-byte J0 blocks, one thread per IV;
 * the *_j0 batch forms take d_j0 (n x 16) where the plain forms take d_iv12 (n x 12). */
int agcm_batch_derive_j0(agcm_ctx* ctx, const uint8_t* d_iv, const uint64_t* d_iv_off, uint64_t iv_len, size_t n_msgs,
                         uint8_t* d_j0, void* stream);
int agcm_batch_crypt_j0(agcm_ctx* ctx, int decrypt, int lanes, uint64_t avg_len_hint, const uint8_t* d_j0,
                        const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                        uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_crypt_uniform_j0(agcm_ctx* ctx, int decrypt, int lanes, const uint8_t* d_j0, const uint8_t* d_aad,
                                uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in, uint8_t* d_out, uint64_t len,
                                uint64_t stride, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);

/* ---- many independent messages, one DISTINCT key per message ----------------------
 * BASELINE config 4.  d_keys holds n_msgs raw keys of mode/8 bytes; each thread runs
 * the aes_kexp schedule on the fly, one stage per round (config/config_aes_kexp.py:
 * 113-159), derives its own H and E_K(J0), and absorbs GHASH with the serial
 * recurrence of src/gcm_ghash.vhd:269-272.  Does not use or change the context key.
 * Other arguments as agcm_batch_crypt / agcm_batch_crypt_uniform.
 * Messages of different lengths are taken in length order (device sort, from 1024 messages); the kernel works ONE
 * lane per message, so this call is for short messages (packets): a message of tens of KiB under its own key is
 * better served by agcm_set_key + the stream calls. */
int agcm_batch_crypt_perkey(agcm_ctx* ctx, int mode, int decrypt, const uint8_t* d_keys, const uint8_t* d_iv12,
                            const uint8_t* d_aad, const uint64_t* d_aad_off, const uint8_t* d_in, const uint64_t* d_in_off,
                            uint8_t* d_out, uint8_t* d_tag, uint8_t* d_ok, size_t n_msgs, void* stream);
int agcm_batch_crypt_perkey_uniform(agcm_ctx* ctx, int mode, int decrypt, const uint8_t* d_keys, const uint8_t* d_iv12,
                                    const uint8_t* d_aad, uint64_t aad_len, uint64_t aad_stride, const uint8_t* d_in,
                                    uint8_t* d_out, uint64_t len, uint64_t stride, uint8_t* d_tag, uint8_t* d_ok,
                                    size_t n_msgs, void* stream);

/* ---- host-buffer entry points (the call a reference-side user makes) ---------
 * Inputs and outputs live in HOST memory; the library stages them through HBM
 * in chunks, overlapping H2D, kernel and D2H on its own streams.  Pinned host
 * memory (agcm_host_alloc, or any cudaHostAlloc/registered buffer) gives full
 * PCIe rate.  Synchronous.  *h_ok is written for decrypt (may be NULL for
 * encrypt). */
int agcm_stream_crypt_host(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], const uint8_t* h_aad, uint64_t aad_len,
                           const uint8_t* h_in, uint8_t* h_out, uint64_t n_bytes, uint8_t h_tag[16], int* h_ok);
/* host buffers, IV of any length (see agcm_stream_crypt_iv) */
int agcm_stream_crypt_iv_host(agcm_ctx* ctx, int decrypt, const uint8_t* h_iv, size_t iv_len, const uint8_t* h_aad,
                              uint64_t aad_len, const uint8_t* h_in, uint8_t* h_out, uint64_t n_bytes,
                              uint8_t h_tag[16], int* h_ok);
/* Verify-then-release decrypt from host buffers (see agcm_stream_decrypt_verified): the ciphertext is
 * copied into HBM once (n_bytes of device memory, kept by the context) and absorbed chunk by chunk;
 * only when the tag matches does the GCTR pass run and the plaintext travel back.  On a mismatch
 * *h_ok = 0 and h_pt is untouched.  The default agcm_stream_crypt_host(decrypt = 1) streams instead:
 * one pass, plaintext chunks written back before the tag is known. */
int agcm_stream_decrypt_verified_host(agcm_ctx* ctx, const uint8_t* h_iv, size_t iv_len, const uint8_t* h_aad,
                                      uint64_t aad_len, const uint8_t* h_ct, uint8_t* h_pt, uint64_t n_bytes,
                                      const uint8_t h_tag[16], int* h_ok);
/* Host-buffer forms of agcm_stream_part / agcm_stream_finish (one rank's shard of a
 * sharded message; the 16-byte partials travel between ranks). */
int agcm_stream_part_host(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* h_in,
                          uint8_t* h_out, uint64_t n_bytes, uint64_t blocks_after, uint8_t h_partial16[16]);
int agcm_stream_finish_host(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], const uint8_t* h_partials16, int n_parts,
                            const uint8_t* h_aad, uint64_t aad_len, uint64_t ct_len, uint8_t h_tag[16], int* h_ok);
/* Host-buffer form of agcm_stream_crypt_peer: this rank's shard is staged through HBM in chunks
 * (the same H2D / kernel / D2H pipeline), the rank's partial is posted to the peers, and the tag /
 * ok flag come back to the host on every rank.  Synchronous; no collective library call. */
int agcm_stream_crypt_peer_host(agcm_ctx* ctx, int decrypt, const uint8_t h_iv12[12], uint64_t first_block,
                                const uint8_t* h_in, uint8_t* h_out, uint64_t n_bytes, uint64_t blocks_after,
                                const uint8_t* h_aad, uint64_t aad_len, uint64_t total_len, uint8_t h_tag[16], int* h_ok);
int agcm_batch_crypt_uniform_host(agcm_ctx* ctx, int decrypt, int lanes, const uint8_t* h_iv12, const uint8_t* h_aad,
                                  uint64_t aad_len, uint64_t aad_stride, const uint8_t* h_in, uint8_t* h_out,
                                  uint64_t len, uint64_t stride, uint8_t* h_tag, uint8_t* h_ok, size_t n_msgs);
int agcm_host_alloc(void** out, size_t bytes); /* pinned */
void agcm_host_free(void* p);

/* ---- the two halves of the datapath on their own -------------------------------
 * agcm_gctr: the gcm_gctr entity alone (src/gcm_gctr.vhd:150, aes_icb.vhd:100):
 *   d_out[i] = d_in[i] xor E_K(IV || 2 + first_block + i/16).  With a zero input
 *   it yields raw keystream (used by the streaming gcm adapter to prefetch).
 * agcm_ghash: the gcm_ghash absorb alone (src/gcm_ghash.vhd:259-272) over n_bytes
 *   (zero-padded to a block): d_y16 = sum_i X_i * H^(n-i), natural byte order,
 *   i.e. the running Y after absorbing the data from Y = 0. */
int agcm_gctr(agcm_ctx* ctx, const uint8_t h_iv12[12], uint64_t first_block, const uint8_t* d_in, uint8_t* d_out,
              uint64_t n_bytes, void* stream);
int agcm_ghash(agcm_ctx* ctx, const uint8_t* d_in, uint64_t n_bytes, uint8_t* d_y16, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AESGCM_B200_H */

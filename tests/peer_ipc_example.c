/* Plain-C client of the peer exchange (include/aesgcm_b200.h): one rank of a message sharded over processes, set up with
 * agcm_peer_export / agcm_peer_import.  The ranks exchange their handles and "ready" marks through files in a shared
 * directory (write, then rename; poll with a bounded wait).  Every rank encrypts its shard of one message, decrypts it
 * with the releasing call (good and flipped tag) and with the verify-then-release call (good and flipped tag), and writes
 * what it computed to files that tests/test_peer_ipc.py checks against OpenSSL.  Inputs: SEED through splitmix64, bytes
 * [0,32) key, [32,44) IV, [44,64) AAD, [64,64+N_BYTES) plaintext.  Built by tests with gcc only; needs a B200 to run.
 *   peer_ipc_example <dir> <rank> <world> <device>
 * Exit 0 = done, 1 = a call or a wait failed, 2 = usage, 3 = no context on the device. */
#define _POSIX_C_SOURCE 200809L
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "aesgcm_b200.h"

#define N_BYTES ((1u << 20) + 7)
#define AAD_BYTES 20
#define SEED 0x5eed5eedu
#define SENT 0x5A
#define WAIT_S 120

#define CHECK(call)                                                                                   \
    do {                                                                                              \
        int rc_ = (call);                                                                             \
        if (rc_) {                                                                                    \
            printf("rank %d: %s: %s (%s)\n", rank, #call, agcm_strerror(rc_), agcm_last_cuda_error_string(ctx)); \
            return 1;                                                                                 \
        }                                                                                             \
    } while (0)

static uint64_t splitmix64(uint64_t* s)
{
    uint64_t z = (*s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

static const char* dir;

static void path_of(char* p, size_t cap, const char* name, int rank, const char* suffix)
{
    snprintf(p, cap, "%s/%s.%d%s", dir, name, rank, suffix);
}

/* <dir>/<name>.<rank> appears complete or not at all */
static int put(const char* name, int rank, const void* data, size_t n)
{
    char tmp[4096], fin[4096];
    path_of(tmp, sizeof tmp, name, rank, ".tmp");
    path_of(fin, sizeof fin, name, rank, "");
    FILE* f = fopen(tmp, "wb");
    if (!f) return 1;
    const int bad = (n && fwrite(data, 1, n, f) != n) | (fclose(f) != 0);
    if (bad || rename(tmp, fin)) {
        printf("cannot write %s\n", fin);
        return 1;
    }
    return 0;
}

/* waits (bounded) for <dir>/<name>.<rank> and reads n bytes of it */
static int get(const char* name, int rank, void* data, size_t n)
{
    char fin[4096];
    path_of(fin, sizeof fin, name, rank, "");
    const struct timespec nap = {0, 1000000};
    for (long i = 0; i < WAIT_S * 1000L; ++i) {
        FILE* f = fopen(fin, "rb");
        if (f) {
            const size_t got = n ? fread(data, 1, n, f) : 0;
            fclose(f);
            if (got == n) return 0;
            printf("short file %s\n", fin);
            return 1;
        }
        nanosleep(&nap, NULL);
    }
    printf("timed out waiting for %s\n", fin);
    return 1;
}

/* every rank has put <name>: returns once all world marks exist */
static int barrier(const char* name, int rank, int world)
{
    if (put(name, rank, NULL, 0)) return 1;
    for (int w = 0; w < world; ++w)
        if (get(name, w, NULL, 0)) return 1;
    return 0;
}

int main(int argc, char** argv)
{
    if (argc != 5) {
        printf("usage: %s <dir> <rank> <world> <device>\n", argv[0]);
        return 2;
    }
    dir = argv[1];
    const int rank = atoi(argv[2]), world = atoi(argv[3]), device = atoi(argv[4]);
    if (world < 1 || world > 16 || rank < 0 || rank >= world) return 2;

    static uint8_t in[64 + N_BYTES];
    uint64_t s = SEED;
    for (size_t i = 0; i < sizeof in; i += 8) {
        const uint64_t r = splitmix64(&s);
        for (size_t k = 0; k < 8 && i + k < sizeof in; ++k) in[i + k] = (uint8_t)(r >> (8 * k));
    }
    const uint8_t *key = in, *iv = in + 32, *aad = in + 44, *pt = in + 64;

    /* the counter range of this rank (parallel.shard_plan) */
    const uint64_t blocks = (N_BYTES + 15) / 16, per = (blocks + world - 1) / world;
    const uint64_t fb = rank * per < blocks ? rank * per : blocks;
    const uint64_t nblk = per < blocks - fb ? per : blocks - fb;
    const uint64_t off = fb * 16, after = blocks - fb - nblk;
    const uint64_t n = off < N_BYTES ? (N_BYTES - off < nblk * 16 ? N_BYTES - off : nblk * 16) : 0;

    agcm_ctx* ctx = NULL;
    int rc = agcm_ctx_create(&ctx, device);
    if (rc) {
        printf("rank %d: agcm_ctx_create(device %d): %s\n", rank, device, agcm_strerror(rc));
        return 3;
    }
    CHECK(agcm_set_key(ctx, 256, 0, key, 32));

    static uint8_t handles[16 * AGCM_PEER_HANDLE_BYTES];
    CHECK(agcm_peer_export(ctx, handles + rank * AGCM_PEER_HANDLE_BYTES));
    if (put("handle", rank, handles + rank * AGCM_PEER_HANDLE_BYTES, AGCM_PEER_HANDLE_BYTES)) return 1;
    for (int w = 0; w < world; ++w)
        if (get("handle", w, handles + w * AGCM_PEER_HANDLE_BYTES, AGCM_PEER_HANDLE_BYTES)) return 1;
    CHECK(agcm_peer_import(ctx, rank, world, handles));
    if (barrier("imported", rank, world)) return 1;   /* every buffer is zeroed before anyone posts */

    uint8_t* ct = malloc(n + 1);
    uint8_t* out = malloc(n + 1);
    if (!ct || !out) return 1;
    uint8_t tag[16], bad_tag[16], oks[4];
    int ok = 0;
    CHECK(agcm_stream_crypt_peer_host(ctx, 0, iv, fb, pt + off, ct, n, after, aad, AAD_BYTES, N_BYTES, tag, &ok));
    if (put("ct", rank, ct, n) || put("tag", rank, tag, 16)) return 1;
    memcpy(bad_tag, tag, 16);
    bad_tag[7] ^= 0x10;

    /* releasing decrypt: writes the plaintext whatever the tag, ok says whether it matched */
    CHECK(agcm_stream_crypt_peer_host(ctx, 1, iv, fb, ct, out, n, after, aad, AAD_BYTES, N_BYTES, tag, &ok));
    oks[0] = (uint8_t)ok;
    if (put("released", rank, out, n)) return 1;
    CHECK(agcm_stream_crypt_peer_host(ctx, 1, iv, fb, ct, out, n, after, aad, AAD_BYTES, N_BYTES, bad_tag, &ok));
    oks[1] = (uint8_t)ok;

    /* verify-then-release: the output is written only if the whole message's tag matches */
    memset(out, SENT, n);
    CHECK(agcm_stream_decrypt_verified_peer_host(ctx, iv, 12, fb, ct, out, n, after, aad, AAD_BYTES, N_BYTES, tag, &ok));
    oks[2] = (uint8_t)ok;
    if (put("verified", rank, out, n)) return 1;
    memset(out, SENT, n);
    CHECK(agcm_stream_decrypt_verified_peer_host(ctx, iv, 12, fb, ct, out, n, after, aad, AAD_BYTES, N_BYTES, bad_tag, &ok));
    oks[3] = (uint8_t)ok;
    if (put("forged", rank, out, n) || put("ok", rank, oks, sizeof oks)) return 1;

    /* teardown: everyone unmaps, then barrier, then frees its own buffer */
    CHECK(agcm_peer_close(ctx));
    if (barrier("closed", rank, world)) return 1;
    agcm_ctx_destroy(ctx);
    free(ct);
    free(out);
    printf("peer_ipc_example rank %d ok\n", rank);
    return 0;
}

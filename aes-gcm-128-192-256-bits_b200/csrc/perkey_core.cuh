// One message per thread with its OWN key (BASELINE config 4): the key schedule is
// generated on the fly, one stage per round, exactly like the reference's expand
// variant of aes_kexp (config/config_aes_kexp.py:113-159,191-225 streams one
// 128-bit stage per round; word recurrence of tb/key_exp.py:98-112) -- a thread
// cannot hold 60 stage words next to the AES state, and 2^20 distinct schedules
// would not fit shared memory.  GHASH uses a thread-private 4-bit Shoup table of
// H (16 rows of 16 B in the thread's own shared-memory column) and the serial
// recurrence Y <- (Y xor X)*H of src/gcm_ghash.vhd:269-272 -- with one message
// per thread the recurrence IS the parallel form: 2^20 independent chains.
//
// The only non-linear part of the schedule is SubWord, applied to 8 / 7 / 12 words past word 11
// (AES-128 / 192 / 256).  Those SubWord outputs are computed once per message and parked in
// a 12-word thread-private shared-memory column (SUBC: put(j, v) / get(j)); per block the
// schedule is then 12 word loads and XORs instead of 48 S-box byte lookups.
//
// Host+device, exercised on the CPU by tests/host_emul.cu.
#pragma once
#include "gcm_core.cuh"

// ---- on-the-fly key schedule ------------------------------------------------
// Emits stage words in order; all indices are compile-time after unrolling.
// SB: functor uint32_t(uint32_t word) -> SubWord(word) (S-box on each byte).
template <int NK>
struct RkStream {
    uint32_t w[NK];   // sliding window: w[i % NK] = word i-NK .. i-1
    uint32_t rcon;

    AG_HD void init(const uint32_t* key)
    {
#pragma unroll
        for (int i = 0; i < NK; ++i) w[i] = key[i];
        rcon = 1;
    }

    // word i of the expanded key; must be called for i = 0, 1, 2, ... in order
    template <class SB>
    AG_HD uint32_t word(int i, SB&& sb)
    {
        if (i < NK) return w[i];
        uint32_t t = w[(i - 1) % NK];
        if (i % NK == 0) {
            t = sb((t >> 8) | (t << 24));  // SubWord(RotWord)
            t ^= rcon;
            rcon = (rcon << 1) ^ ((rcon & 0x80) ? 0x11Bu : 0u);
        } else if (NK == 8 && (i % 8) == 4) {
            t = sb(t);
        }
        w[i % NK] ^= t;
        return w[i % NK];
    }
};

// One block with the schedule generated alongside the rounds (NR = NK + 6).
template <int NK, class TE, class SB>
AG_HD void aes_encrypt_otf(const uint32_t* key, uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, TE&& te, SB&& sb,
                           uint32_t out[4])
{
    constexpr int NR = NK + 6;
    RkStream<NK> ks;
    ks.init(key);
    s0 ^= ks.word(0, sb);
    s1 ^= ks.word(1, sb);
    s2 ^= ks.word(2, sb);
    s3 ^= ks.word(3, sb);
#pragma unroll
    for (int r = 1; r < NR; ++r) {
        const uint32_t k0 = ks.word(4 * r + 0, sb), k1 = ks.word(4 * r + 1, sb), k2 = ks.word(4 * r + 2, sb),
                       k3 = ks.word(4 * r + 3, sb);
        const uint32_t t0 = te(0, s0, 0) ^ te(1, s1, 1) ^ te(2, s2, 2) ^ te(3, s3, 3) ^ k0;
        const uint32_t t1 = te(0, s1, 0) ^ te(1, s2, 1) ^ te(2, s3, 2) ^ te(3, s0, 3) ^ k1;
        const uint32_t t2 = te(0, s2, 0) ^ te(1, s3, 1) ^ te(2, s0, 2) ^ te(3, s1, 3) ^ k2;
        const uint32_t t3 = te(0, s3, 0) ^ te(1, s0, 1) ^ te(2, s1, 2) ^ te(3, s2, 3) ^ k3;
        s0 = t0;
        s1 = t1;
        s2 = t2;
        s3 = t3;
    }
    const uint32_t k0 = ks.word(4 * NR + 0, sb), k1 = ks.word(4 * NR + 1, sb), k2 = ks.word(4 * NR + 2, sb),
                   k3 = ks.word(4 * NR + 3, sb);
    out[0] = (te(2, s0, 0) & 0x000000ffu) ^ (te(3, s1, 1) & 0x0000ff00u) ^ (te(0, s2, 2) & 0x00ff0000u) ^
             (te(1, s3, 3) & 0xff000000u) ^ k0;
    out[1] = (te(2, s1, 0) & 0x000000ffu) ^ (te(3, s2, 1) & 0x0000ff00u) ^ (te(0, s3, 2) & 0x00ff0000u) ^
             (te(1, s0, 3) & 0xff000000u) ^ k1;
    out[2] = (te(2, s2, 0) & 0x000000ffu) ^ (te(3, s3, 1) & 0x0000ff00u) ^ (te(0, s0, 2) & 0x00ff0000u) ^
             (te(1, s1, 3) & 0xff000000u) ^ k2;
    out[3] = (te(2, s3, 0) & 0x000000ffu) ^ (te(3, s0, 1) & 0x0000ff00u) ^ (te(0, s1, 2) & 0x00ff0000u) ^
             (te(1, s2, 3) & 0xff000000u) ^ k3;
}

// SubWord functors for RkStream::word past word 11: record the outputs once, replay them per block.
// After unrolling, j is a compile-time constant at every call.
template <class SB, class SUBC>
struct SubRecord {
    SB& sb;
    SUBC& c;
    int j;
    AG_HD uint32_t operator()(uint32_t w)
    {
        const uint32_t v = sb(w);
        c.put(j++, v);
        return v;
    }
};
template <class SUBC>
struct SubReplay {
    SUBC& c;
    int j;
    AG_HD uint32_t operator()(uint32_t) { return c.get(j++); }
};

// ---- counter mode with the schedule on the fly, per-message constants hoisted ---------
// Stage words 0..11 (rounds 0-2) are used once per message: they go into the round-1
// constants (aes_ctr_precompute), rk[3], and the sequential-counter cache of rounds 1+2
// (aes_ctr_seq_fill, aes_core.cuh).  Per block the schedule resumes at word 12 from a saved
// copy of the sliding window, and rounds 1+2 cost 5 lookups.
template <int NK>
struct PerKeyCtr {
    RkStream<NK> at12;     // schedule state after word 11
    AesCtrConst cc;
    AesCtrSeqCache cache;
    uint32_t rk3;
    uint32_t rk8[4];
};

template <int NK, class TE, class SB, class SUBC>
AG_HD void perkey_ctr_init(const uint32_t* key, uint32_t iv0, uint32_t iv1, uint32_t iv2, TE&& te, SB&& sb, SUBC&& subc,
                           PerKeyCtr<NK>& st)
{
    RkStream<NK> ks;
    ks.init(key);
    uint32_t rk[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) rk[i] = ks.word(i, sb);
    st.at12 = ks;
    {   // run the rest of the schedule once, parking every SubWord output
        SubRecord<SB, SUBC> rec{sb, subc, 0};
        uint32_t sink = 0;
#pragma unroll
        for (int i = 12; i < 4 * (NK + 7); ++i) sink ^= ks.word(i, rec);
        (void)sink;
    }
    st.cc = aes_ctr_precompute(rk, iv0, iv1, iv2, te);
    st.rk3 = rk[3];
    st.rk8[0] = rk[8]; st.rk8[1] = rk[9]; st.rk8[2] = rk[10]; st.rk8[3] = rk[11];
    st.cache.key = 0xFFFFFFFFu;
}

template <int NK, class TE, class SUBC>
AG_HD void perkey_ctr_block(PerKeyCtr<NK>& st, uint32_t ctr, TE&& te, SUBC&& subc, uint32_t out[4])
{
    constexpr int NR = NK + 6;
    SubReplay<SUBC> sb{subc, 0};
    const uint32_t s3i = ag_bswap32(ctr) ^ st.rk3;
    if ((s3i & 0x00FFFFFFu) != st.cache.key) {
        // aes_ctr_seq_fill reads rk[3] (unused there) and rk[8..11]: hand it a view with those
        uint32_t rkv[12];
#pragma unroll
        for (int i = 0; i < 8; ++i) rkv[i] = 0;
        rkv[8] = st.rk8[0]; rkv[9] = st.rk8[1]; rkv[10] = st.rk8[2]; rkv[11] = st.rk8[3];
        aes_ctr_seq_fill(rkv, st.cc, s3i, te, st.cache);
    }
    const uint32_t a = st.cc.k[0] ^ te(3, s3i, 3);
    uint32_t s0 = st.cache.q[0] ^ te(0, a, 0);
    uint32_t s1 = st.cache.q[1] ^ te(3, a, 3);
    uint32_t s2 = st.cache.q[2] ^ te(2, a, 2);
    uint32_t s3 = st.cache.q[3] ^ te(1, a, 1);
    RkStream<NK> ks = st.at12;
#pragma unroll
    for (int r = 3; r < NR; ++r) {
        const uint32_t k0 = ks.word(4 * r + 0, sb), k1 = ks.word(4 * r + 1, sb), k2 = ks.word(4 * r + 2, sb),
                       k3 = ks.word(4 * r + 3, sb);
        const uint32_t t0 = te(0, s0, 0) ^ te(1, s1, 1) ^ te(2, s2, 2) ^ te(3, s3, 3) ^ k0;
        const uint32_t t1 = te(0, s1, 0) ^ te(1, s2, 1) ^ te(2, s3, 2) ^ te(3, s0, 3) ^ k1;
        const uint32_t t2 = te(0, s2, 0) ^ te(1, s3, 1) ^ te(2, s0, 2) ^ te(3, s1, 3) ^ k2;
        const uint32_t t3 = te(0, s3, 0) ^ te(1, s0, 1) ^ te(2, s1, 2) ^ te(3, s2, 3) ^ k3;
        s0 = t0;
        s1 = t1;
        s2 = t2;
        s3 = t3;
    }
    const uint32_t k0 = ks.word(4 * NR + 0, sb), k1 = ks.word(4 * NR + 1, sb), k2 = ks.word(4 * NR + 2, sb),
                   k3 = ks.word(4 * NR + 3, sb);
    out[0] = (te(2, s0, 0) & 0x000000ffu) ^ (te(3, s1, 1) & 0x0000ff00u) ^ (te(0, s2, 2) & 0x00ff0000u) ^
             (te(1, s3, 3) & 0xff000000u) ^ k0;
    out[1] = (te(2, s1, 0) & 0x000000ffu) ^ (te(3, s2, 1) & 0x0000ff00u) ^ (te(0, s3, 2) & 0x00ff0000u) ^
             (te(1, s0, 3) & 0xff000000u) ^ k1;
    out[2] = (te(2, s2, 0) & 0x000000ffu) ^ (te(3, s3, 1) & 0x0000ff00u) ^ (te(0, s0, 2) & 0x00ff0000u) ^
             (te(1, s1, 3) & 0xff000000u) ^ k2;
    out[3] = (te(2, s3, 0) & 0x000000ffu) ^ (te(3, s0, 1) & 0x0000ff00u) ^ (te(0, s1, 2) & 0x00ff0000u) ^
             (te(1, s2, 3) & 0xff000000u) ^ k3;
}

// ---- thread-private 4-bit Shoup table ------------------------------------------
// T[n] = n*H for the 4-bit polynomial n (bit 3 of n = x^0).  ROWS: object with
//   void put(int n, uint4 row);   uint4 get(uint32_t be_word, int nibble /*0 = low*/);
template <class ROWS>
AG_HD void gf_build_table4(const gf128& h, ROWS&& rows)
{
    gf128 b[4];
    b[0] = h;  // n = 8
    b[1] = gf_mulx(b[0]);  // n = 4
    b[2] = gf_mulx(b[1]);  // n = 2
    b[3] = gf_mulx(b[2]);  // n = 1
#pragma unroll
    for (int n = 0; n < 16; ++n) {
        uint4 r = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (n & (8 >> k)) {
                r.x ^= b[k].w[0];
                r.y ^= b[k].w[1];
                r.z ^= b[k].w[2];
                r.w ^= b[k].w[3];
            }
        rows.put(n, r);
    }
}

// X*H with the reduction deferred to the end.  X = sum over (word q, nibble k) of
// n(q,k) * x^(32q) * x^(4(7-k))  (k = 7 is the top nibble of a BE word = its lowest degrees), so
//   X*H = sum_k x^(4(7-k)) * A_k,   A_k = sum_q T[n(q,k)] * x^(32q):
// x^(32q) is a move by q words (free), and the outer sum is a Horner in x^4 over an unreduced
// 8-word accumulator: 7 shifts by one nibble and ONE fold (gf_fold256) instead of a shift and a
// reduction per nibble (about 270 integer operations per product instead of about 500).
template <class ROWS>
AG_HD gf128 gf_mul_table4(const gf128& x, ROWS&& rows)
{
    uint32_t z[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) z[m] = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (k) {
#pragma unroll
            for (int m = 7; m >= 1; --m) z[m] = ag_funnel_r(z[m], z[m - 1], 4);
            z[0] >>= 4;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 t = rows.get(x.w[q], k);
            z[q] ^= t.x;
            z[q + 1] ^= t.y;
            z[q + 2] ^= t.z;
            z[q + 3] ^= t.w;
        }
    }
    return gf_fold256(z);
}

// ---- one whole message ------------------------------------------------------------
// key: NK little-endian words of the raw key.  Returns the computed tag words (LE) and
// writes the payload.  Unified order AAD | CT | length block (gcm_ghash.vhd:259-272,257).
// WIDE: the message may sit at an odd address (batches packed by offsets): whole blocks are then read as realigned
// 16-byte granules and written through a carried granule, as in the single-lane layout of the shared-key batches
// (gcm_core.cuh: AgWideWindow, AgLoadCarry, AgStoreCarry) instead of byte by byte.
// VERIFY (verify-then-release decrypt, DEC): `tag` holds the EXPECTED tag on entry.  Phase 1 absorbs AAD | CT | length
// block without a keystream; only if the computed tag matches does phase 2 run GCTR over the same ciphertext (read a
// second time, mostly from L2) and write the payload.  Returns the computed tag in `tag` either way.  One lane does
// both phases: a second launch would rebuild the key schedule and the private GHASH table.
template <int NK, bool DEC, bool WIDE = false, bool VERIFY = false, class TE, class SB, class ROWS, class SUBC>
AG_HD void ag_perkey_message(const uint32_t* key, uint32_t iv0, uint32_t iv1, uint32_t iv2, const MsgDesc& d, TE&& te,
                             SB&& sb, ROWS&& rows, SUBC&& subc, uint32_t tag[4])
{
    uint32_t e[4];
    aes_encrypt_otf<NK>(key, 0, 0, 0, 0, te, sb, e);  // H = E_K(0^128)  (gcm_gctr.vhd:141-144)
    gf_build_table4(gf_from_le_words(e[0], e[1], e[2], e[3]), rows);
    PerKeyCtr<NK> st;
    perkey_ctr_init<NK>(key, iv0, iv1, iv2, te, sb, subc, st);
    perkey_ctr_block<NK>(st, 1u, te, subc, e);  // E_K(J0), J0 = IV || 00000001 (aes_icb.vhd:34,99)

    gf128 y = gf_zero();
    const uint64_t a = (d.aad_len + 15) >> 4, n = (d.len + 15) >> 4;   // both < 2^32 (checked / documented at the API)
    const AgWideWindow win_aad = WIDE ? AgWideWindow::make(d.aad, d.aad ? d.aad_len : 0) : AgWideWindow{0, 0};
    const AgWideWindow win_in = WIDE ? AgWideWindow::make(d.in, d.len) : AgWideWindow{0, 0};
    AgLoadCarry lc_aad, lc_in;
    lc_aad.j = lc_in.j = 0xFFFFFFFFu;
    lc_aad.g = lc_in.g = make_uint4(0, 0, 0, 0);
#if defined(__CUDA_ARCH__)
    AgStoreCarry carry;
    carry.init();
    const bool wide_st = WIDE && (((uintptr_t)d.out & 15) != 0);
#endif
    for (uint64_t i = 0; i < a; ++i) {
        const uint64_t left = d.aad_len - 16 * i;
        uint32_t s[4];
        ag_load_block_win<WIDE>(d.aad, (uint32_t)i, left < 16 ? (uint32_t)left : 16u, s, win_aad, lc_aad);
        y = gf_xor(y, gf_from_le_words(s[0], s[1], s[2], s[3]));
        y = gf_mul_table4(y, rows);
    }
    for (uint64_t j = 0; j < n; ++j) {
        const uint64_t left = d.len - 16 * j;
        const uint32_t nv = left < 16 ? (uint32_t)left : 16u;
        uint32_t x[4], ks[4];
        ag_load_block_win<WIDE>(d.in, (uint32_t)j, nv, x, win_in, lc_in);
        if constexpr (VERIFY) {
            y = gf_xor(y, gf_from_le_words(x[0], x[1], x[2], x[3]));
            y = gf_mul_table4(y, rows);
            continue;
        }
        perkey_ctr_block<NK>(st, 2u + (uint32_t)j, te, subc, ks);
        uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
#if defined(__CUDA_ARCH__)
        if (WIDE && wide_st && nv == 16) {
            carry.put(d.out + 16 * j, o);
        } else {
            if (WIDE) carry.flush();
            ag_store_block(d.out + 16 * j, nv, o);
        }
#else
        ag_store_block(d.out + 16 * j, nv, o);
#endif
        if (DEC) {
            y = gf_xor(y, gf_from_le_words(x[0], x[1], x[2], x[3]));
        } else {
            if (nv != 16) ag_mask_block(o, nv);
            y = gf_xor(y, gf_from_le_words(o[0], o[1], o[2], o[3]));
        }
        y = gf_mul_table4(y, rows);
    }
#if defined(__CUDA_ARCH__)
    if (WIDE) carry.flush();
#endif
    const uint64_t ab = d.aad_len * 8, cb = d.len * 8;
    y.w[0] ^= (uint32_t)(ab >> 32);
    y.w[1] ^= (uint32_t)ab;
    y.w[2] ^= (uint32_t)(cb >> 32);
    y.w[3] ^= (uint32_t)cb;
    y = gf_mul_table4(y, rows);
    if constexpr (VERIFY) {
        const bool match = ((tag[0] ^ ag_bswap32(y.w[0]) ^ e[0]) | (tag[1] ^ ag_bswap32(y.w[1]) ^ e[1]) |
                            (tag[2] ^ ag_bswap32(y.w[2]) ^ e[2]) | (tag[3] ^ ag_bswap32(y.w[3]) ^ e[3])) == 0;
        lc_in.j = 0xFFFFFFFFu;
        for (uint64_t j = 0; match && j < n; ++j) {   // phase 2: release
            const uint64_t left = d.len - 16 * j;
            const uint32_t nv = left < 16 ? (uint32_t)left : 16u;
            uint32_t x[4], ks[4];
            ag_load_block_win<WIDE>(d.in, (uint32_t)j, nv, x, win_in, lc_in);
            perkey_ctr_block<NK>(st, 2u + (uint32_t)j, te, subc, ks);
            const uint32_t o[4] = {x[0] ^ ks[0], x[1] ^ ks[1], x[2] ^ ks[2], x[3] ^ ks[3]};
#if defined(__CUDA_ARCH__)
            if (wide_st && nv == 16) {
                carry.put(d.out + 16 * j, o);
            } else {
                if (WIDE) carry.flush();
                ag_store_block(d.out + 16 * j, nv, o);
            }
#else
            ag_store_block(d.out + 16 * j, nv, o);
#endif
        }
#if defined(__CUDA_ARCH__)
        if (WIDE) carry.flush();
#endif
    }
    tag[0] = ag_bswap32(y.w[0]) ^ e[0];
    tag[1] = ag_bswap32(y.w[1]) ^ e[1];
    tag[2] = ag_bswap32(y.w[2]) ^ e[2];
    tag[3] = ag_bswap32(y.w[3]) ^ e[3];
}

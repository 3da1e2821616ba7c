// Shared-memory tables and warp helpers shared by every data-path kernel of the engine
// (kernels.cu: stream / key / finish / peer; kernels_batch.cu: shared-key batches; kernels_perkey.cu:
// per-message keys), and the launch and dispatch helpers of their launchers.  Everything lives in an
// anonymous namespace, one copy per translation unit.
//
// Shared-memory plan (one persistent 512-thread CTA per SM, 194 KB of the 227 KB):
//
//   [0      , 64 KB)  AES_A : 256 entries x 256 B; entry x = 32 lane-private copies
//                     of Te0[x] (128 B) then 32 copies of Te1[x] (128 B)
//   [64 KB  , 128 KB) AES_B : same for Te2 / Te3
//   [128 KB , 192 KB) GH    : 256 entries x 256 B; entry b = 8 copies of the 16 B row
//                     T_a[b] (128 B) then 8 copies of T_b[b] (128 B)
//   [192 KB , +2 KB)  reduction scratch
//
// Every data-dependent lookup is then bank-conflict free BY CONSTRUCTION: lane l
// reads word l of a 128 B row (32-bit AES lookups), or 16 B slot l%8 of a row
// (128-bit GHASH lookups, served per quarter-warp).  The 256 B entry stride makes
// the address a single PRMT: {0, 0, index byte, lane offset}; the table select is
// an immediate on the LDS.  Per 16 B block that is 16 PRMT + 16 LDS + 8 LOP3 per
// AES round and 16 PRMT + 16 LDS.128 + ~90 LOP3/SHF per GHASH multiply.
//
// Reference blocks replaced: gcm_gctr (aes_icb + aes_ecb + xor, src/gcm_gctr.vhd:150),
// gcm_ghash + ghash_gfmul (src/gcm_ghash.vhd:225-293, src/ghash_gfmul.vhd:42-63),
// aes_kexp (config/config_aes_kexp.py:128-159, tb/key_exp.py:79-114).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "gcm_core.cuh"
#include "kernels.h"

namespace {

constexpr uint32_t SM_AES_A = 0;
constexpr uint32_t SM_AES_B = 65536;
constexpr uint32_t SM_GH = 131072;
constexpr uint32_t SM_MISC = 196608;

extern __shared__ __align__(1024) uint8_t ag_smem[];

// Te_tab[(w >> 8k) & 0xff] from the lane-private replicas
struct TeSmem {
    const uint8_t* base;
    uint32_t lane4;  // (lane & 31) * 4
    __device__ __forceinline__ uint32_t operator()(int tab, uint32_t w, int k) const
    {
        const uint32_t off = __byte_perm(w, lane4, 0x5504 | (k << 4));  // (byte_k << 8) | lane4
        return *reinterpret_cast<const uint32_t*>(base + off + (tab & 1) * 128 + (tab >> 1) * 65536);
    }
};

// row T[(w >> 8k) & 0xff] of the GHASH table from the quarter-warp replicas
struct GhSmem {
    const uint8_t* base;  // ag_smem + SM_GH (+128 for T_b)
    uint32_t lane16;      // (lane & 7) * 16
    __device__ __forceinline__ uint4 operator()(uint32_t w, int k) const
    {
        const uint32_t off = __byte_perm(w, lane16, 0x5504 | (k << 4));
        return *reinterpret_cast<const uint4*>(base + off);
    }
};

// slow-path lookups straight from HBM/L2 (setup and finish kernels only)
struct TeGlobal {
    const uint32_t* te0;
    __device__ __forceinline__ uint32_t operator()(int tab, uint32_t w, int k) const
    {
        const uint32_t t = __ldg(te0 + ((w >> (8 * k)) & 0xff));
        return tab ? ag_rotl32(t, 8 * tab) : t;
    }
};

// Te0 (1 KB) is staged once through the reduction scratch with one coalesced load per thread, so
// the 16 expansion passes read shared memory instead of paying a global-load latency each: the
// table fill is most of a short message's kernel time.  Order at the call sites: stage_te0 and
// fill_gh_tables (their global loads overlap), __syncthreads, expand_aes_tables, __syncthreads.
__device__ __forceinline__ void stage_te0(const uint32_t* __restrict__ te0)
{
    uint32_t* stage = reinterpret_cast<uint32_t*>(ag_smem + SM_MISC);
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) stage[i] = __ldg(te0 + i);
}

__device__ __forceinline__ void expand_aes_tables()
{
    const uint32_t* stage = reinterpret_cast<const uint32_t*>(ag_smem + SM_MISC);
#pragma unroll 4
    for (uint32_t idx = threadIdx.x; idx < 256 * 32; idx += blockDim.x) {
        const uint32_t x = idx >> 5, l = idx & 31;
        const uint32_t t = stage[x];
        uint32_t* a = reinterpret_cast<uint32_t*>(ag_smem + SM_AES_A + x * 256 + l * 4);
        uint32_t* b = reinterpret_cast<uint32_t*>(ag_smem + SM_AES_B + x * 256 + l * 4);
        a[0] = t;
        a[32] = ag_rotl32(t, 8);
        b[0] = ag_rotl32(t, 16);
        b[32] = ag_rotl32(t, 24);
    }
}

__device__ __forceinline__ void fill_gh_tables(const uint4* __restrict__ ta, const uint4* __restrict__ tb)
{
#pragma unroll 4
    for (uint32_t idx = threadIdx.x; idx < 256 * 8; idx += blockDim.x) {
        const uint32_t b = idx >> 3, r = idx & 7;
        uint4* d = reinterpret_cast<uint4*>(ag_smem + SM_GH + b * 256 + r * 16);
        d[0] = __ldg(ta + b);
        if (tb) d[8] = __ldg(tb + b);
    }
}

__device__ __forceinline__ gf128 warp_xor(gf128 v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v.w[0] ^= __shfl_xor_sync(0xffffffffu, v.w[0], o);
        v.w[1] ^= __shfl_xor_sync(0xffffffffu, v.w[1], o);
        v.w[2] ^= __shfl_xor_sync(0xffffffffu, v.w[2], o);
        v.w[3] ^= __shfl_xor_sync(0xffffffffu, v.w[3], o);
    }
    return v;
}

// H^e for a 64-bit exponent, computed by one full warp: lane k contributes
// pow2[k]^(bit k) * pow2[k+32]^(bit k+32); the 32 factors are multiplied by a
// shuffle tree (5 generic products deep).  All lanes return the result.
__device__ gf128 warp_gf_pow(const KeyDev* kd, uint64_t e)
{
    const uint32_t lane = threadIdx.x & 31;
    gf128 f = ((e >> lane) & 1) ? kd->pow2[lane] : gf_one();
    if (e >> 32) {  // uniform
        gf128 f2 = ((e >> (lane + 32)) & 1) ? kd->pow2[lane + 32] : gf_one();
        f = gf_mul(f, f2);
    }
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        gf128 g;
        g.w[0] = __shfl_xor_sync(0xffffffffu, f.w[0], o);
        g.w[1] = __shfl_xor_sync(0xffffffffu, f.w[1], o);
        g.w[2] = __shfl_xor_sync(0xffffffffu, f.w[2], o);
        g.w[3] = __shfl_xor_sync(0xffffffffu, f.w[3], o);
        f = gf_mul(f, g);
    }
    return f;
}


// dynamic shared memory of the table kernels (AES_A | AES_B | GH | 2 KB scratch)
constexpr size_t kSmemBytes = SM_MISC + 2048;
// k_batch_tile / k_batch_perkey_tile: one TMA box = 32 messages x 32 bytes
constexpr uint32_t TILE_BYTES = 1024;

// Launch of a kernel with `smem` bytes of dynamic shared memory (past the 48 KB default, which needs the opt-in)
template <typename... KArgs, typename... Args>
cudaError_t ag_launch_smem(void (*kernel)(KArgs...), int ncta, int nt, size_t smem, cudaStream_t st, const Args&... args)
{
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<ncta, nt, smem, st>>>(args...);
    return cudaGetLastError();
}

// A run-time value as a template argument: f(std::integral_constant<int, V>) for the V of Vs equal to v,
// cudaErrorInvalidValue if there is none
template <int... Vs, typename F>
cudaError_t ag_with(int v, F&& f)
{
    cudaError_t e = cudaErrorInvalidValue;
    (void)((v == Vs && ((e = f(std::integral_constant<int, Vs>{})), true)) || ...);
    return e;
}

// NR = 10 / 12 / 14 AES rounds
template <typename F>
cudaError_t ag_with_nr(int nr, F&& f)
{
    return ag_with<10, 12, 14>(nr, f);
}

// DEC for the kernels that have no tag-only form: AG_DECRYPT_VERIFIED is refused, so that it can never select a
// decrypt that releases plaintext
template <typename F>
cudaError_t ag_with_dec(int decrypt, F&& f)
{
    if (decrypt == AG_DECRYPT_VERIFIED) return cudaErrorInvalidValue;
    return decrypt ? f(std::true_type{}) : f(std::false_type{});
}

}  // namespace

// common.cuh -- shared device helpers for libb200ssm (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200_ssm.h"

namespace b200 {

constexpr float kLog2e = 1.4426950408889634f;

// ---- error plumbing (host) ------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);
void count_launch(int n = 1);

// cudaFuncSetAttribute acts on the CURRENT device's copy of a kernel: remember (kernel, device) pairs, not just "done once",
// so a process that uses several GPUs (a model moved to cuda:1 after a run on cuda:0) opts in on each of them.
// Returns cudaSuccess when the attribute is (already) set.  Host only; defined in api.cu.
cudaError_t func_attr_per_device(const void* kernel, cudaFuncAttribute attr, int value);

#define B200_REQUIRE(cond, ...)          \
    do {                                 \
        if (!(cond)) {                   \
            b200::set_error(__VA_ARGS__); \
            return -1;                   \
        }                                \
    } while (0)

// ---- checkpoint record layout (shared by both kernel generations) ----------------------------------------------------
// One record = the 16 x 16 state entering a chunk = 256 floats: word  ckpt_state_pos(n) + 2 * (row & 7) + (row >> 3).
// States are grouped in quads of 64 words; inside ODD quads the 16-word blocks of states (0,1) and (2,3) are swapped, so a
// record copied verbatim into shared memory (one 1 KB bulk copy) is read without bank conflicts by the backward's
// [state quad][row pair] lanes (a half-warp = two quads x 8 row pairs x 8 bytes covers all 32 banks).
__host__ __device__ constexpr int ckpt_state_pos(int n) { return (n >> 2) * 64 + ((((n & 3) ^ ((n >> 2) & 1))) << 4); }

// ---- dtype helpers ---------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// ---- math ------------------------------------------------------------------------------------
// 2^x on the SFU (MUFU.EX2): the recurrence's decay a = exp(delta*A) = 2^(delta * A*log2e), the same
// identity the reference kernel uses (selective_scan_fwd_kernel.cuh:168-175,216).
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// exp(x) with a Cody-Waite split of log2(e): the error (~2 ulp of MUFU.EX2) does not grow with |x|,
// unlike __expf (ex2(x * log2e): the rounding of the product costs |x| * 2^-24 relative).
__device__ __forceinline__ float exp_acc(float x) {
    const float xc = fminf(fmaxf(x, -87.f), 88.f);  // keeps 2^n a normal number; exp(-87) ~ 1.6e-38 is 0 in effect
    const float n = rintf(xc * 1.4426950408889634f);
    float f = fmaf(xc, 1.4426950216293335f, -n);
    f = fmaf(xc, 1.9259629911266175e-8f, f);
    return ex2(f) * __int_as_float(((int)n + 127) << 23);
}

// F.softplus(beta=1, threshold=20), selective_scan_interface.py:112-113 / fwd_kernel.cuh:153-156.
__device__ __forceinline__ float softplus20(float x) { return x > 20.f ? x : log1pf(expf(x)); }

__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// softplus(x) (threshold 20, F.softplus / selective_scan_fwd_kernel.cuh:153-156) and sigmoid(x) = d softplus/dx from TWO
// MUFU operations (the libm route log1pf(expf(x)) costs ~80 instructions; the first version of this function used four MUFUs:
// ex2, lg2 and two rcp).  With e = exp(-|x|) in (0, 1]:
//     softplus(x) = max(x, 0) + log1p(e),   log1p(e) = 2 atanh(s),  s = e / (2 + e) <= 1/3  (8-term odd series, remainder < 2e-9),
//     sigmoid(x)  = x >= 0 ? 1 / (1 + e) : e / (1 + e),
// and both quotients come from ONE reciprocal r = 1 / ((1 + e)(2 + e)).  e = ex2(-|x| log2 e) without a Cody-Waite split: its
// relative error |x| 2^-24 is multiplied by e / (1 + e) in softplus, i.e. at most 1.2e-8 absolute.  Relative error of both outputs
// < 6.5e-7 for x >= -6 and < |x| 1e-7 below (where they are < 3e-3); tests/test_math_host.py restates this routine in numpy float32
// and checks it against float64.
struct SoftplusSig { float sp, sig; };
__device__ __forceinline__ SoftplusSig softplus_sigmoid(float x) {
    const float e = ex2(-fabsf(x) * kLog2e);
    const float t1 = 1.f + e, t2 = 2.f + e;
    const float r = rcp_approx(t1 * t2);
    const float inv1 = r * t2;                 // 1 / (1 + e)
    const float s = e * (r * t1);              // e / (2 + e)
    const float s2 = s * s;
    float p = fmaf(s2, 1.f / 15.f, 1.f / 13.f);
    p = fmaf(s2, p, 1.f / 11.f);
    p = fmaf(s2, p, 1.f / 9.f);
    p = fmaf(s2, p, 1.f / 7.f);
    p = fmaf(s2, p, 0.2f);
    p = fmaf(s2, p, 1.f / 3.f);
    p = fmaf(s2, p, 1.f);
    SoftplusSig o;
    o.sp = fmaf(s + s, p, fmaxf(x, 0.f));
    o.sig = x >= 0.f ? inv1 : e * inv1;
    if (x > 20.f) { o.sp = x; o.sig = 1.f; }
    return o;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// ---- vector I/O of f32 / bf16 / f16 rows (rmsnorm.cu, conv1d.cu) ----------------------------------------------
// V in {1, 2, 4} consecutive elements of a dtype chosen at run time (B200_F32 / BF16 / F16), base + idx aligned to V elements.
// V consecutive elements as raw bits: the loads of a row are all issued before the first conversion (rn_cvt)
template <int V>
__device__ __forceinline__ void rn_ld(const void* base, int64_t idx, int dt, uint32_t (&r)[V]) {
    if (dt == B200_F32) {
        const float* p = static_cast<const float*>(base) + idx;
        if constexpr (V == 4) {
            const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
            r[0] = u.x, r[1] = u.y, r[2] = u.z, r[3] = u.w;
        } else if constexpr (V == 2) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p));
            r[0] = u.x, r[1] = u.y;
        } else {
            r[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
        }
    } else {
        const unsigned short* p = static_cast<const unsigned short*>(base) + idx;
        if constexpr (V == 4) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p));
            r[0] = u.x, r[1] = u.y;
        } else if constexpr (V == 2) {
            r[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
        } else {
            r[0] = __ldcs(p);
        }
    }
}

template <int V>
__device__ __forceinline__ void rn_cvt(const uint32_t (&r)[V], int dt, float* v) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
        if (dt == B200_F32) {
            v[j] = __uint_as_float(r[j]);
        } else {
            const uint32_t h = V == 1 ? r[0] & 0xffffu : (r[j >> 1] >> (16 * (j & 1))) & 0xffffu;
            v[j] = dt == B200_BF16 ? __uint_as_float(h << 16) : __half2float(__ushort_as_half((unsigned short)h));
        }
    }
}

template <int V>
__device__ __forceinline__ void rn_st(void* base, int64_t idx, int dt, const float* v) {
    if (dt == B200_F32) {
        float* p = static_cast<float*>(base) + idx;
        if constexpr (V == 4) __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
        else if constexpr (V == 2) __stcs(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
        else __stcs(p, v[0]);
        return;
    }
    uint32_t h[V];
#pragma unroll
    for (int j = 0; j < V; ++j)
        h[j] = dt == B200_BF16 ? __bfloat16_as_ushort(__float2bfloat16_rn(v[j])) : __half_as_ushort(__float2half_rn(v[j]));
    unsigned short* p = static_cast<unsigned short*>(base) + idx;
    if constexpr (V == 4) __stcs(reinterpret_cast<uint2*>(p), make_uint2(h[0] | h[1] << 16, h[2] | h[3] << 16));
    else if constexpr (V == 2) __stcs(reinterpret_cast<unsigned int*>(p), h[0] | h[1] << 16);
    else __stcs(p, (unsigned short)h[0]);
}

// streaming global accesses: activations are touched once per kernel
template <typename T> __device__ __forceinline__ float ldg_stream(const T* p) { return to_f32<T>(__ldcs(p)); }
template <> __device__ __forceinline__ float ldg_stream<__nv_bfloat16>(const __nv_bfloat16* p) {
    unsigned short r = __ldcs(reinterpret_cast<const unsigned short*>(p));
    return __bfloat162float(__ushort_as_bfloat16(r));
}
template <> __device__ __forceinline__ float ldg_stream<__half>(const __half* p) {
    unsigned short r = __ldcs(reinterpret_cast<const unsigned short*>(p));
    return __half2float(__ushort_as_half(r));
}
template <typename T> __device__ __forceinline__ void stg_stream(T* p, float v) { __stcs(p, from_f32<T>(v)); }
template <> __device__ __forceinline__ void stg_stream<__nv_bfloat16>(__nv_bfloat16* p, float v) {
    __stcs(reinterpret_cast<unsigned short*>(p), __bfloat16_as_ushort(__float2bfloat16_rn(v)));
}
template <> __device__ __forceinline__ void stg_stream<__half>(__half* p, float v) {
    __stcs(reinterpret_cast<unsigned short*>(p), __half_as_ushort(__float2half_rn(v)));
}

}  // namespace b200

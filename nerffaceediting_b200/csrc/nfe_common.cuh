// Shared device/host helpers for libnfe_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/nfe_b200.h"

#define NFE_EXPORT extern "C" __attribute__((visibility("default")))

namespace nfe {

// thread-local error text behind nfe_last_error()
void set_error(const char* fmt, ...);
void count_launch();

// Optional per-stage timing (nfe_timing_enable): CUDA events recorded on the launching stream.
enum Stage { STAGE_FIELD_COARSE = 0, STAGE_RESAMPLE = 1, STAGE_FIELD_FINE = 2, STAGE_MARCH_FINAL = 3, STAGE_RUN_MODEL = 4,
             STAGE_COUNT = 5 };
int stage_begin(int stage, cudaStream_t stream);   // returns a token (< 0 when timing is off)
void stage_end(int token, cudaStream_t stream);
struct StageScope {
    int token; cudaStream_t stream;
    StageScope(int stage, cudaStream_t s) : token(stage_begin(stage, s)), stream(s) {}
    ~StageScope() { stage_end(token, stream); }
};

inline int check_launch(const char* what)
{
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}

#define NFE_REQUIRE(cond, ...)                  \
    do {                                        \
        if (!(cond)) {                          \
            nfe::set_error(__VA_ARGS__);        \
            return 1;                           \
        }                                       \
    } while (0)

#define NFE_LAUNCH_CHECK(what)                  \
    do {                                        \
        int _rc = nfe::check_launch(what);      \
        if (_rc) return _rc;                    \
    } while (0)

inline cudaStream_t as_stream(nfe_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

inline int sm_count()
{
    static int cached = 0;
    if (!cached) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        if (cached <= 0) cached = 148;
    }
    return cached;
}

// ---------------------------------------------------------------------------------------------
// Device arithmetic shared by the stage kernels and the fused kernel.  The sampling stage
// (coordinates, bins, CDF) uses explicit round-to-nearest intrinsics so that nvcc never fuses a
// multiply-add the oracle does not have; the MLP / compositing sums may use FMAs.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_ref(float x)
{
    // torch.nn.Softplus(beta=1, threshold=20): x > 20 ? x : log1p(exp(x))
    return x > 20.0f ? x : log1pf(expf(x));
}

__device__ __forceinline__ float sigmoid_ref(float x) { return 1.0f / (1.0f + expf(-x)); }

// o + t*d without contraction (renderer.py:105,122,326,344: separate mul and add kernels)
__device__ __forceinline__ float ray_point(float o, float t, float d) { return __fadd_rn(o, __fmul_rn(t, d)); }

// Bilinear tap set of one plane for grid coordinate (gx, gy): top-left texel and 4 weights,
// grid_sample(bilinear, zeros, align_corners=False) semantics (renderer.py:64).
struct Taps {
    int x0, y0;
    float w[4];  // (x0,y0) (x1,y0) (x0,y1) (x1,y1)
};

__device__ __forceinline__ Taps plane_taps(float gx, float gy, int H, int W)
{
    Taps t;
    const float ix = __fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gx, 1.0f), (float)W), 1.0f), 2.0f);
    const float iy = __fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(gy, 1.0f), (float)H), 1.0f), 2.0f);
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const float fx1 = fx0 + 1.0f, fy1 = fy0 + 1.0f;
    const float wx0 = __fsub_rn(fx1, ix), wx1 = __fsub_rn(ix, fx0);
    const float wy0 = __fsub_rn(fy1, iy), wy1 = __fsub_rn(iy, fy0);
    t.w[0] = __fmul_rn(wx0, wy0);
    t.w[1] = __fmul_rn(wx1, wy0);
    t.w[2] = __fmul_rn(wx0, wy1);
    t.w[3] = __fmul_rn(wx1, wy1);
    // clamp before the int conversion; NaN compares false everywhere and lands on -2 (all taps out)
    const float cx = (fx0 >= -2.0f) ? fminf(fx0, (float)W) : -2.0f;
    const float cy = (fy0 >= -2.0f) ? fminf(fy0, (float)H) : -2.0f;
    t.x0 = (int)cx;
    t.y0 = (int)cy;
    return t;
}

// plane p of the EG3D tri-plane (renderer.py:29-53): 0 -> (x,y), 1 -> (x,z), 2 -> (z,x)
__device__ __forceinline__ void project(float qx, float qy, float qz, int p, float& gx, float& gy)
{
    gx = (p == 2) ? qz : qx;
    gy = (p == 0) ? qy : ((p == 1) ? qz : qx);
}

// Philox4x32-10, counter-based: (seed, subsequence=index, offset) -> 4 uniform uint32.
__device__ __forceinline__ uint4 philox4x32(uint64_t seed, uint64_t index, uint64_t offset)
{
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)offset, c1 = (uint32_t)(offset >> 32), c2 = (uint32_t)index, c3 = (uint32_t)(index >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// U[0,1) with 24 random bits, as torch.rand produces for float32
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// N(0,1) pair by Box-Muller
__device__ __forceinline__ float2 normal2(uint32_t a, uint32_t b)
{
    const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);  // (0,1]
    const float u2 = u01(b);
    const float r = sqrtf(-2.0f * logf(u1));
    float s, c;
    sincospif(2.0f * u2, &s, &c);
    return make_float2(r * c, r * s);
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_min(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// float atomic min/max through the ordered-int trick (valid for any non-NaN floats)
__device__ __forceinline__ void atomic_min_float(float* addr, float v)
{
    if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* addr, float v)
{
    if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// ---- packed fp32 pairs (Blackwell FFMA2 / FADD2 / FMUL2): one issue slot for two lanes of arithmetic; each half
//      rounds exactly like the scalar instruction
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c)
{
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d)
        : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)), "l"(*reinterpret_cast<unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)
{
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b)
{
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}

}  // namespace nfe

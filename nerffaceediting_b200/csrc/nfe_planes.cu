// Plane statistics, (de)normalisation and the channel-last staging of the tri-planes.
// Replaces TriPlaneGenerator.compute_mean_var / normalize_plane / denormalize_plane
// (training/triplane.py:56-68) — three full passes plus broadcast temporaries in the reference.
// All four kernels are pure HBM streams: bytes = read 1x (+ write 1x) of the plane tensor.
#include "nfe_common.cuh"

namespace nfe {

// One CTA per (batch, channel) slab.  Single pass, sum and sum of squares in double: with fp32
// inputs the double accumulators make the one-pass variance formula safe, and the result is
// order-independent to ~1e-16, i.e. deterministic after rounding to fp32.
__global__ void __launch_bounds__(512) plane_stats_kernel(const float* __restrict__ planes, int64_t hw,
                                                          float* __restrict__ mean, float* __restrict__ std_out)
{
    const float* x = planes + (int64_t)blockIdx.x * hw;
    double s = 0.0, ss = 0.0;
    const bool vec = (hw % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (vec) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        const int64_t n4 = hw / 4;
        for (int64_t i = threadIdx.x; i < n4; i += blockDim.x) {
            const float4 v = __ldg(x4 + i);
            // pairwise in fp32 is not exact; keep every add in double
            s += (double)v.x; s += (double)v.y; s += (double)v.z; s += (double)v.w;
            ss += (double)v.x * (double)v.x; ss += (double)v.y * (double)v.y;
            ss += (double)v.z * (double)v.z; ss += (double)v.w * (double)v.w;
        }
    } else {
        for (int64_t i = threadIdx.x; i < hw; i += blockDim.x) {
            const double v = (double)x[i];
            s += v; ss += v * v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    __shared__ double sh_s[16], sh_ss[16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh_s[warp] = s; sh_ss[warp] = ss; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        s = lane < nw ? sh_s[lane] : 0.0;
        ss = lane < nw ? sh_ss[lane] : 0.0;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
        }
        if (lane == 0) {
            const double n = (double)hw;
            const double m = s / n;
            double var = (ss - s * m) / (n - 1.0);
            if (var < 0.0) var = 0.0;
            mean[blockIdx.x] = (float)m;
            std_out[blockIdx.x] = sqrtf((float)var);
        }
    }
}

// (x - mean) / (std + 1e-8), IEEE division to stay bit-comparable with the reference.
__global__ void __launch_bounds__(256) plane_normalize_kernel(const float* __restrict__ planes, const float* __restrict__ mean,
                                                              const float* __restrict__ std_in, int64_t hw, int chunks_per_slab,
                                                              float* __restrict__ out)
{
    const int64_t slab = blockIdx.x / chunks_per_slab;
    const int chunk = blockIdx.x % chunks_per_slab;
    const float m = mean[slab];
    const float d = __fadd_rn(std_in[slab], 1e-8f);
    const int64_t per = (hw + chunks_per_slab - 1) / chunks_per_slab;
    const int64_t lo = chunk * per, hi = min(hw, lo + per);
    const float* x = planes + slab * hw;
    float* y = out + slab * hw;
    const bool vec = (hw % 4 == 0) && (per % 4 == 0) && (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0);
    if (vec) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (int64_t i = lo / 4 + threadIdx.x; i < hi / 4; i += blockDim.x) {
            float4 v = __ldg(x4 + i);
            v.x = __fdiv_rn(__fsub_rn(v.x, m), d); v.y = __fdiv_rn(__fsub_rn(v.y, m), d);
            v.z = __fdiv_rn(__fsub_rn(v.z, m), d); v.w = __fdiv_rn(__fsub_rn(v.w, m), d);
            y4[i] = v;
        }
    } else {
        for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) y[i] = __fdiv_rn(__fsub_rn(x[i], m), d);
    }
}

// x * std' + mean' (mul then add, unfused, as the reference's two ATen kernels)
__global__ void __launch_bounds__(256) plane_denormalize_kernel(const float* __restrict__ norm, const float* __restrict__ mean,
                                                                const float* __restrict__ std_in, int64_t stat_slabs, int64_t hw,
                                                                int chunks_per_slab, float* __restrict__ out)
{
    const int64_t slab = blockIdx.x / chunks_per_slab;
    const int chunk = blockIdx.x % chunks_per_slab;
    const float m = mean[slab % stat_slabs];
    const float d = std_in[slab % stat_slabs];
    const int64_t per = (hw + chunks_per_slab - 1) / chunks_per_slab;
    const int64_t lo = chunk * per, hi = min(hw, lo + per);
    const float* x = norm + slab * hw;
    float* y = out + slab * hw;
    const bool vec = (hw % 4 == 0) && (per % 4 == 0) && (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0);
    if (vec) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (int64_t i = lo / 4 + threadIdx.x; i < hi / 4; i += blockDim.x) {
            float4 v = __ldg(x4 + i);
            v.x = __fadd_rn(__fmul_rn(v.x, d), m); v.y = __fadd_rn(__fmul_rn(v.y, d), m);
            v.z = __fadd_rn(__fmul_rn(v.z, d), m); v.w = __fadd_rn(__fmul_rn(v.w, d), m);
            y4[i] = v;
        }
    } else {
        for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) y[i] = __fadd_rn(__fmul_rn(x[i], d), m);
    }
}

// [n_img, C, hw] -> [n_img, hw, C] through a padded shared tile.  A CTA moves C x 64 pixels:
// reads are 256-byte runs per channel, writes are one contiguous 64*C*4-byte span.
constexpr int CL_PIX = 64;
__global__ void __launch_bounds__(256) to_channel_last_kernel(const float* __restrict__ planes, int channels, int64_t hw,
                                                              int64_t tiles_per_img, float* __restrict__ out)
{
    extern __shared__ float tile[];  // [channels][CL_PIX + 1]
    const int64_t img = blockIdx.x / tiles_per_img;
    const int64_t px0 = (blockIdx.x % tiles_per_img) * CL_PIX;
    const float* src = planes + img * channels * hw;
    float* dst = out + img * hw * channels;
    const int npx = (int)min((int64_t)CL_PIX, hw - px0);
    for (int i = threadIdx.x; i < channels * CL_PIX; i += blockDim.x) {
        const int c = i / CL_PIX, p = i % CL_PIX;
        if (p < npx) tile[c * (CL_PIX + 1) + p] = __ldg(src + (int64_t)c * hw + px0 + p);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < npx * channels; i += blockDim.x) {
        const int p = i / channels, c = i % channels;
        dst[(px0 + p) * channels + c] = tile[c * (CL_PIX + 1) + p];
    }
}

// 32-channel fast path of the staging, optionally fused with the normalisation.
// A warp owns 32 consecutive pixels of one image: lane = pixel.  It reads the 32 channel rows (32
// independent, fully coalesced 128-byte loads per lane), and each lane then holds its pixel's whole
// channel vector, i.e. one 128-byte channel-last texel, written as 8 float4 stores.  With NORMALIZE
// the same registers also produce (x-mean)/(std+1e-8): the NCHW result (coalesced) and its channel-last
// copy, so normalize_plane + both stagings cost one read of the planes instead of three.
constexpr int STAGE_MIN_BLOCKS = 4;
template <bool NORMALIZE>
__global__ void __launch_bounds__(256, STAGE_MIN_BLOCKS) stage32_kernel(const float* __restrict__ planes, const float* __restrict__ mean,
                                                      const float* __restrict__ std_in, int64_t hw, int64_t groups_per_img, int64_t n_groups,
                                                      float* __restrict__ out_norm, float* __restrict__ out_norm_cl, float* __restrict__ out_raw_cl)
{
    const int lane = threadIdx.x & 31;
    int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (group >= n_groups) return;
    // normalize_plane runs right after plane_stats_kernel has streamed the same planes in ascending order: walking them in
    // DESCENDING order finds the last ~100 MB still in the 126 MB L2, and leaves item 0's staged copy hot for the field kernel
    // (c2 step 1.140 -> 1.136 ms on B200, profiles/run_r01_stage_ab.sh)
    if constexpr (NORMALIZE) group = n_groups - 1 - group;
    const int64_t img = group / groups_per_img;
    const int64_t px = (group % groups_per_img) * 32 + lane;
    const bool live = px < hw;
    const float* src = planes + img * 32 * hw + px;
    float x[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) x[c] = live ? __ldg(src + (int64_t)c * hw) : 0.0f;
    if (live && out_raw_cl) {
        float4* dst = reinterpret_cast<float4*>(out_raw_cl + (img * hw + px) * 32);
#pragma unroll
        for (int q = 0; q < 8; ++q) dst[q] = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
    }
    if constexpr (NORMALIZE) {
        // lane c carries the statistics of channel c; broadcast by shuffle
        const float m_l = mean[img * 32 + lane];
        const float d_l = __fadd_rn(std_in[img * 32 + lane], 1e-8f);
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const float m = __shfl_sync(0xffffffffu, m_l, c), d = __shfl_sync(0xffffffffu, d_l, c);
            x[c] = __fdiv_rn(__fsub_rn(x[c], m), d);
        }
        if (live) {
            float* dn = out_norm + img * 32 * hw + px;
            // the reference-layout copy is rarely read back: evict first (with the descending walk: c2 step 1.134-1.136 ms)
#pragma unroll
            for (int c = 0; c < 32; ++c) __stcs(dn + (int64_t)c * hw, x[c]);
            float4* dst = reinterpret_cast<float4*>(out_norm_cl + (img * hw + px) * 32);
#pragma unroll
            for (int q = 0; q < 8; ++q) dst[q] = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
        }
    }
}


// ---- backward of normalize_plane (triplane.py:56-65): norm = (x - mean)/(std + 1e-8), mean/std over H,W (std unbiased).
// With d = std + 1e-8, n = H*W and the upstream gradients (g, g_mean, g_std):
//   gx = g/d - mean(g)/d + g_mean/n + norm * (g_std*d - sum(g*norm)) / ((n-1)*std)
// Pass 1: per slab sum(g) and sum(g*norm) (double accumulation, like the forward statistics); pass 2: the elementwise
// combination.  Two streaming passes (reads g, norm twice; writes gx once) replace ~25 ATen kernels.
__global__ void __launch_bounds__(512) plane_normalize_bwd_sums_kernel(const float* __restrict__ g, const float* __restrict__ norm, int64_t hw,
                                                                       double* __restrict__ sums)
{
    const float* gp = g + (int64_t)blockIdx.x * hw;
    const float* np_ = norm + (int64_t)blockIdx.x * hw;
    double s = 0.0, sn = 0.0;
    const bool vec = (hw % 4 == 0) && (((reinterpret_cast<uintptr_t>(gp) | reinterpret_cast<uintptr_t>(np_)) & 15) == 0);
    if (vec) {
        const float4* g4 = reinterpret_cast<const float4*>(gp);
        const float4* n4 = reinterpret_cast<const float4*>(np_);
        for (int64_t i = threadIdx.x; i < hw / 4; i += blockDim.x) {
            const float4 a = __ldg(g4 + i), b = __ldg(n4 + i);
            s += ((double)a.x + (double)a.y) + ((double)a.z + (double)a.w);
            sn += ((double)a.x * (double)b.x + (double)a.y * (double)b.y) + ((double)a.z * (double)b.z + (double)a.w * (double)b.w);
        }
    } else {
        for (int64_t i = threadIdx.x; i < hw; i += blockDim.x) { s += (double)gp[i]; sn += (double)gp[i] * (double)np_[i]; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); sn += __shfl_xor_sync(0xffffffffu, sn, o); }
    __shared__ double sh_s[16], sh_n[16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh_s[warp] = s; sh_n[warp] = sn; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        s = lane < nw ? sh_s[lane] : 0.0;
        sn = lane < nw ? sh_n[lane] : 0.0;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); sn += __shfl_xor_sync(0xffffffffu, sn, o); }
        if (lane == 0) { sums[2 * blockIdx.x] = s; sums[2 * blockIdx.x + 1] = sn; }
    }
}

__global__ void __launch_bounds__(256) plane_normalize_bwd_apply_kernel(const float* __restrict__ g, const float* __restrict__ norm,
                                                                        const float* __restrict__ std_in, const float* __restrict__ g_mean,
                                                                        const float* __restrict__ g_std, const double* __restrict__ sums,
                                                                        int64_t hw, int chunks_per_slab, float* __restrict__ out)
{
    const int64_t slab = blockIdx.x / chunks_per_slab;
    const int chunk = blockIdx.x % chunks_per_slab;
    const double n = (double)hw, sd = (double)std_in[slab], d = sd + 1e-8;
    const double sum_g = g ? sums[2 * slab] : 0.0, sum_gn = g ? sums[2 * slab + 1] : 0.0;
    const float A = (float)(1.0 / d);
    const float B = (float)(-(sum_g / n) / d + (g_mean ? (double)g_mean[slab] / n : 0.0));
    const float C = (float)(((g_std ? (double)g_std[slab] * d : 0.0) - sum_gn) / ((n - 1.0) * sd));
    const int64_t per = (hw + chunks_per_slab - 1) / chunks_per_slab;
    const int64_t lo = chunk * per, hi = min(hw, lo + per);
    const float* gp = g ? g + slab * hw : nullptr;
    const float* np_ = norm + slab * hw;
    float* y = out + slab * hw;
    const bool vec = (hw % 4 == 0) && (per % 4 == 0) &&
                     (((reinterpret_cast<uintptr_t>(gp) | reinterpret_cast<uintptr_t>(np_) | reinterpret_cast<uintptr_t>(y)) & 15) == 0);
    if (vec) {
        const float4* g4 = reinterpret_cast<const float4*>(gp);
        const float4* n4 = reinterpret_cast<const float4*>(np_);
        float4* y4 = reinterpret_cast<float4*>(y);
        for (int64_t i = lo / 4 + threadIdx.x; i < hi / 4; i += blockDim.x) {
            const float4 a = gp ? __ldg(g4 + i) : make_float4(0.f, 0.f, 0.f, 0.f), b = __ldg(n4 + i);
            y4[i] = make_float4(fmaf(C, b.x, fmaf(A, a.x, B)), fmaf(C, b.y, fmaf(A, a.y, B)), fmaf(C, b.z, fmaf(A, a.z, B)), fmaf(C, b.w, fmaf(A, a.w, B)));
        }
    } else {
        for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) y[i] = fmaf(C, np_[i], fmaf(A, gp ? gp[i] : 0.0f, B));
    }
}


// ---- SR pre-resize (SURVEY.md §8f row f1): F.interpolate(x, size, mode='bilinear', align_corners=False, antialias=...)
// of the rendered feature image (superresolution.py:48-52,80-84,282-286).  One thread per output pixel; the separable
// tap weights are recomputed per thread (<= 2*max(scale,1)+2 taps per axis; 2-3 for the shipped 64^2 -> 128^2 case) and
// the horizontal sums are formed first, like ATen's two passes.  The image (4 MB at c2) was just written by the
// compositing kernel and is read from L2.
struct AxisTaps { int first, n; float scale, support, inv, center; };

__device__ __forceinline__ AxisTaps axis_taps(int o, int in, int out, int antialias)
{
    AxisTaps t;
    t.scale = (float)in / (float)out;
    if (!antialias) {
        float src = fmaxf(t.scale * ((float)o + 0.5f) - 0.5f, 0.0f);
        int i0 = min((int)src, in - 1);
        t.first = i0; t.n = i0 < in - 1 ? 2 : 1; t.center = src - (float)i0;      // center holds the fraction
        t.support = t.inv = 0.0f;
        return t;
    }
    t.support = t.scale >= 1.0f ? t.scale : 1.0f;
    t.inv = t.scale >= 1.0f ? __fdiv_rn(1.0f, t.scale) : 1.0f;
    t.center = t.scale * ((float)o + 0.5f);
    t.first = max((int)(t.center - t.support + 0.5f), 0);
    t.n = min((int)(t.center + t.support + 0.5f), in) - t.first;
    return t;
}

__device__ __forceinline__ float axis_weight(const AxisTaps& t, int j, int antialias)
{
    if (!antialias) return t.n == 1 ? 1.0f : (j == 0 ? 1.0f - t.center : t.center);
    const float x = fabsf(((float)(j + t.first) - t.center + 0.5f) * t.inv);
    return x < 1.0f ? 1.0f - x : 0.0f;
}

constexpr int RESIZE_ROWS = 8;      // output rows per block: the per-column tap set is computed once and reused for all of them

__global__ void __launch_bounds__(128) resize_bilinear_kernel(const float* __restrict__ in, int row_groups, int ih, int iw, int oh, int ow,
                                                              int antialias, float* __restrict__ out)
{
    const int img = blockIdx.x / row_groups, oy0 = (blockIdx.x % row_groups) * RESIZE_ROWS;
    const float* src = in + (int64_t)img * ih * iw;
    float* dst = out + (int64_t)img * oh * ow;
    for (int ox = threadIdx.x; ox < ow; ox += blockDim.x) {
        const AxisTaps tx = axis_taps(ox, iw, ow, antialias);
        float sx = 0.0f;
        for (int j = 0; j < tx.n; ++j) sx += axis_weight(tx, j, antialias);
        const float rx = sx != 0.0f ? __fdiv_rn(1.0f, sx) : 0.0f;            // plain bilinear: the two weights already sum to 1
        for (int r = 0; r < RESIZE_ROWS && oy0 + r < oh; ++r) {
            const AxisTaps ty = axis_taps(oy0 + r, ih, oh, antialias);
            float sy = 0.0f;
            for (int j = 0; j < ty.n; ++j) sy += axis_weight(ty, j, antialias);
            const float ry = sy != 0.0f ? __fdiv_rn(1.0f, sy) : 0.0f;
            float acc = 0.0f;
            for (int jy = 0; jy < ty.n; ++jy) {
                const float* row = src + (int64_t)(ty.first + jy) * iw + tx.first;
                float h = 0.0f;
                for (int jx = 0; jx < tx.n; ++jx) h = fmaf(axis_weight(tx, jx, antialias) * rx, __ldg(row + jx), h);
                acc = fmaf(axis_weight(ty, jy, antialias) * ry, h, acc);
            }
            dst[(int64_t)(oy0 + r) * ow + ox] = acc;
        }
    }
}

}  // namespace nfe

using namespace nfe;

static int chunks_for(int64_t n_slabs, int64_t hw)
{
    // enough CTAs to fill the machine several times over, each streaming >= 16 KB
    int64_t c = (int64_t)sm_count() * 16 / (n_slabs > 0 ? n_slabs : 1);
    const int64_t max_c = hw / 4096 > 0 ? hw / 4096 : 1;
    if (c > max_c) c = max_c;
    if (c < 1) c = 1;
    while (c > 1 && ((hw % c) != 0 || ((hw / c) % 4) != 0)) --c;
    return (int)c;
}

NFE_EXPORT int nfe_plane_stats(const float* planes, int64_t n_slabs, int64_t hw, float* mean, float* std_out, nfe_stream_t stream)
{
    if (n_slabs == 0) return 0;
    NFE_REQUIRE(planes && mean && std_out, "nfe_plane_stats: null pointer");
    NFE_REQUIRE(n_slabs >= 0 && n_slabs < (1ll << 31) && hw >= 2, "nfe_plane_stats: bad sizes (n_slabs=%lld hw=%lld)", (long long)n_slabs, (long long)hw);
    if (n_slabs == 0) return 0;
    plane_stats_kernel<<<(unsigned)n_slabs, 512, 0, as_stream(stream)>>>(planes, hw, mean, std_out);
    NFE_LAUNCH_CHECK("plane_stats_kernel");
    return 0;
}

NFE_EXPORT int nfe_plane_normalize(const float* planes, const float* mean, const float* std_in, int64_t n_slabs, int64_t hw,
                                   float* out, nfe_stream_t stream)
{
    if (n_slabs == 0 || hw == 0) return 0;
    NFE_REQUIRE(planes && mean && std_in && out, "nfe_plane_normalize: null pointer");
    NFE_REQUIRE(n_slabs >= 0 && hw >= 1, "nfe_plane_normalize: bad sizes");
    if (n_slabs == 0) return 0;
    const int chunks = chunks_for(n_slabs, hw);
    NFE_REQUIRE(n_slabs * chunks < (1ll << 31), "nfe_plane_normalize: grid too large");
    plane_normalize_kernel<<<(unsigned)(n_slabs * chunks), 256, 0, as_stream(stream)>>>(planes, mean, std_in, hw, chunks, out);
    NFE_LAUNCH_CHECK("plane_normalize_kernel");
    return 0;
}

NFE_EXPORT int nfe_plane_denormalize(const float* norm, const float* mean, const float* std_in, int64_t n_slabs, int64_t stat_slabs,
                                     int64_t hw, float* out, nfe_stream_t stream)
{
    if (n_slabs == 0 || hw == 0) return 0;
    NFE_REQUIRE(norm && mean && std_in && out, "nfe_plane_denormalize: null pointer");
    NFE_REQUIRE(n_slabs >= 0 && hw >= 1 && stat_slabs >= 1, "nfe_plane_denormalize: bad sizes");
    if (n_slabs == 0) return 0;
    const int chunks = chunks_for(n_slabs, hw);
    NFE_REQUIRE(n_slabs * chunks < (1ll << 31), "nfe_plane_denormalize: grid too large");
    plane_denormalize_kernel<<<(unsigned)(n_slabs * chunks), 256, 0, as_stream(stream)>>>(norm, mean, std_in, stat_slabs, hw, chunks, out);
    NFE_LAUNCH_CHECK("plane_denormalize_kernel");
    return 0;
}

NFE_EXPORT int nfe_planes_to_channel_last(const float* planes, int64_t n_img, int channels, int64_t hw, float* out, nfe_stream_t stream)
{
    if (n_img == 0 || hw == 0) return 0;
    NFE_REQUIRE(planes && out, "nfe_planes_to_channel_last: null pointer");
    NFE_REQUIRE(n_img >= 0 && channels >= 1 && channels <= 256 && hw >= 1, "nfe_planes_to_channel_last: bad sizes");
    if (n_img == 0) return 0;
    if (channels == 32 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        const int64_t groups_per_img = (hw + 31) / 32, n_groups = n_img * groups_per_img;
        NFE_REQUIRE((n_groups + 7) / 8 < (1ll << 31), "nfe_planes_to_channel_last: grid too large");
        stage32_kernel<false><<<(unsigned)((n_groups + 7) / 8), 256, 0, as_stream(stream)>>>(planes, nullptr, nullptr, hw, groups_per_img, n_groups,
                                                                                           nullptr, nullptr, out);
        NFE_LAUNCH_CHECK("stage32_kernel");
        return 0;
    }
    const int64_t tiles = (hw + CL_PIX - 1) / CL_PIX;
    NFE_REQUIRE(n_img * tiles < (1ll << 31), "nfe_planes_to_channel_last: grid too large");
    const size_t smem = (size_t)channels * (CL_PIX + 1) * sizeof(float);
    if (smem > 48 * 1024) cudaFuncSetAttribute(to_channel_last_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    to_channel_last_kernel<<<(unsigned)(n_img * tiles), 256, smem, as_stream(stream)>>>(planes, channels, hw, tiles, out);
    NFE_LAUNCH_CHECK("to_channel_last_kernel");
    return 0;
}

NFE_EXPORT int nfe_plane_normalize_staged(const float* planes, const float* mean, const float* std_in, int64_t n_img, int64_t hw, float* out_norm,
                                          float* out_norm_cl, float* out_raw_cl, nfe_stream_t stream)
{
    if (n_img == 0 || hw == 0) return 0;
    NFE_REQUIRE(planes && mean && std_in && out_norm && out_norm_cl, "nfe_plane_normalize_staged: null pointer");
    NFE_REQUIRE(((reinterpret_cast<uintptr_t>(out_norm_cl) | reinterpret_cast<uintptr_t>(out_raw_cl)) & 15) == 0,
                "nfe_plane_normalize_staged: channel-last outputs must be 16-byte aligned");
    const int64_t groups_per_img = (hw + 31) / 32, n_groups = n_img * groups_per_img;
    NFE_REQUIRE((n_groups + 7) / 8 < (1ll << 31), "nfe_plane_normalize_staged: grid too large");
    stage32_kernel<true><<<(unsigned)((n_groups + 7) / 8), 256, 0, as_stream(stream)>>>(planes, mean, std_in, hw, groups_per_img, n_groups, out_norm,
                                                                                      out_norm_cl, out_raw_cl);
    NFE_LAUNCH_CHECK("stage32_kernel");
    return 0;
}

NFE_EXPORT int nfe_plane_normalize_bwd(const float* g_norm, const float* norm, const float* std_in, const float* g_mean, const float* g_std,
                                       int64_t n_slabs, int64_t hw, double* sums_ws, float* g_planes, nfe_stream_t stream)
{
    if (n_slabs == 0 || hw == 0) return 0;
    NFE_REQUIRE(norm && std_in && g_planes, "nfe_plane_normalize_bwd: null pointer");
    NFE_REQUIRE(!g_norm || sums_ws, "nfe_plane_normalize_bwd: the reduction workspace ([n_slabs,2] doubles) is missing");
    NFE_REQUIRE(n_slabs >= 0 && hw >= 2, "nfe_plane_normalize_bwd: bad sizes");
    NFE_REQUIRE(n_slabs < (1ll << 31), "nfe_plane_normalize_bwd: grid too large");
    if (g_norm) {
        plane_normalize_bwd_sums_kernel<<<(unsigned)n_slabs, 512, 0, as_stream(stream)>>>(g_norm, norm, hw, sums_ws);
        NFE_LAUNCH_CHECK("plane_normalize_bwd_sums_kernel");
    }
    const int chunks = chunks_for(n_slabs, hw);
    NFE_REQUIRE(n_slabs * chunks < (1ll << 31), "nfe_plane_normalize_bwd: grid too large");
    plane_normalize_bwd_apply_kernel<<<(unsigned)(n_slabs * chunks), 256, 0, as_stream(stream)>>>(g_norm, norm, std_in, g_mean, g_std, sums_ws, hw,
                                                                                               chunks, g_planes);
    NFE_LAUNCH_CHECK("plane_normalize_bwd_apply_kernel");
    return 0;
}

NFE_EXPORT int nfe_resize_bilinear(const float* in, int64_t n_img, int in_h, int in_w, int out_h, int out_w, int antialias, float* out,
                                   nfe_stream_t stream)
{
    if (n_img == 0) return 0;
    NFE_REQUIRE(in && out, "nfe_resize_bilinear: null pointer");
    NFE_REQUIRE(n_img > 0 && in_h >= 1 && in_w >= 1 && out_h >= 1 && out_w >= 1, "nfe_resize_bilinear: bad sizes");
    const int row_groups = (out_h + RESIZE_ROWS - 1) / RESIZE_ROWS;
    NFE_REQUIRE(n_img * row_groups < (1ll << 31), "nfe_resize_bilinear: grid too large");
    resize_bilinear_kernel<<<(unsigned)(n_img * row_groups), 128, 0, as_stream(stream)>>>(in, row_groups, in_h, in_w, out_h, out_w, antialias, out);
    NFE_LAUNCH_CHECK("resize_bilinear_kernel");
    return 0;
}

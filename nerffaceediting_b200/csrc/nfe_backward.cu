// Backward pass of the render path (BASELINE config 4: training-step forward + backward).
//
// Gradients are needed w.r.t. both plane tensors and the decoder parameters only: sample positions carry
// no gradient (camera labels are data; depths_fine is detached in the reference, renderer.py:198,211).
// The pieces in this file:
//   march_bwd_kernel        compositing backward, one warp per ray: d(loss)/d(per-sample sigma, seg, rgb) from
//                           d(loss)/d(rgb, seg, depth, weight-sum) of the ray (ray_marcher.py:68-101 differentiated)
//   feature_mean_kernel     recompute of the decoder inputs: plane-mean features [M,32] per plane set
//   scatter_features_kernel gather backward: vectorised red.global.add.v4.f32 of w_tap/3 * d(feature) into the
//                           channel-last plane gradients (the reference's grid_sampler_2d_backward, also atomic)
//   from_channel_last32     channel-last gradients back to the reference's [N,3,32,H,W] layout
// The decoder MLP backward itself (four small GEMM pairs) is run by the host on library GEMMs over the recomputed
// features; see nerffaceediting_b200/autograd.py.
#include "nfe_field.cuh"
#include "nfe_march.cuh"

namespace nfe {

// sample positions of one pass: rays + per-sample depths (sample idx = ray*s_per_ray + s), and the plane geometry
struct FieldGeom {
    int plane_batch, H, W;
    float scale;
    const float* origins; const float* dirs; const float* depths;
    int s_per_ray;
    int64_t m, total;
};

struct MarchBwdArgs {
    const float* depths1; const float* sigma1; const float* rec1; int s1;
    const float* depths2; const float* sigma2; const float* rec2; int s2;
    int64_t n_rays;
    int cs, white_back, inputs_sorted;
    const float* g_rgb;    // [T,32]
    const float* g_seg;    // [T,15] or NULL
    const float* g_depth;  // [T] or NULL
    const float* g_wsum;   // [T] or NULL
    const float* minmax;   // forward depth range {min,max}: the clamp passes gradient only inside it
    float* g_rec1;         // [T,s1,48] = d/d{sigma, seg[15], rgb[32]} per sample
    float* g_rec2;         // [T,s2,48]
};

constexpr int BWD_ARRAYS = 9;  // depth sigma w order raw alpha T dot gsm

constexpr int MARCH_BWD_MIN_BLOCKS = 4;   // 64 registers, 4 blocks per SM: 1.43 -> ~1.0 ms at c4
__global__ void __launch_bounds__(256, MARCH_BWD_MIN_BLOCKS) march_bwd_kernel(MarchBwdArgs a)
{
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int S = a.s1 + a.s2, n_int = S - 1;
    float* s_depth = smem + (size_t)warp * BWD_ARRAYS * S;
    float* s_sigma = s_depth + S;
    float* s_w = s_sigma + S;
    int* s_order = reinterpret_cast<int*>(s_w + S);
    float* s_raw = s_w + 2 * S;
    float* s_alpha = s_raw + S;
    float* s_T = s_alpha + S;
    float* s_dot = s_T + S;
    float* s_gsm = s_dot + S;
    const float dmin = a.minmax ? a.minmax[0] : -3.402823466e+38f, dmax = a.minmax ? a.minmax[1] : 3.402823466e+38f;

    for (int64_t ray = (int64_t)blockIdx.x * warps_per_block + warp; ray < a.n_rays; ray += (int64_t)gridDim.x * warps_per_block) {
        // ---- merge, exactly as the forward
        for (int e = lane; e < S; e += 32) {
            const bool first = e < a.s1;
            s_w[e] = first ? a.depths1[ray * a.s1 + e] : a.depths2[ray * a.s2 + (e - a.s1)];
            s_raw[e] = first ? a.sigma1[ray * a.s1 + e] : a.sigma2[ray * a.s2 + (e - a.s1)];
        }
        __syncwarp();
        for (int e = lane; e < S; e += 32) {
            const float d = s_w[e];
            int rank;
            if (a.s2 == 0) rank = e;
            else if (a.inputs_sorted) {
                const bool first = e < a.s1;
                const float* other = first ? s_w + a.s1 : s_w;
                int lo = 0, hi = first ? a.s2 : a.s1;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    const float v = other[mid];
                    if (first ? (v < d) : (v <= d)) lo = mid + 1; else hi = mid;
                }
                rank = (first ? e : e - a.s1) + lo;
            } else {
                rank = 0;
                for (int j = 0; j < S; ++j) { const float dj = s_w[j]; rank += (dj < d) || (dj == d && j < e); }
            }
            s_depth[rank] = d; s_sigma[rank] = s_raw[e]; s_order[rank] = e;
        }
        __syncwarp();
        // ---- forward quantities per interval: alpha, transmittance, weight
        const int chunk = (n_int + 31) / 32;
        const int i0 = min(n_int, lane * chunk), i1 = min(n_int, i0 + chunk);
        float prod = 1.0f;
        for (int i = i0; i < i1; ++i) {
            const float delta = __fsub_rn(s_depth[i + 1], s_depth[i]);
            const float xs = __fsub_rn(__fdiv_rn(__fadd_rn(s_sigma[i], s_sigma[i + 1]), 2.0f), 1.0f);
            const float dens = fmaxf(xs, 0.0f) + __logf(1.0f + __expf(-fabsf(xs)));
            const float alpha = __fsub_rn(1.0f, __expf(-__fmul_rn(dens, delta)));
            s_alpha[i] = alpha;
            prod *= __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
        }
        float incl = prod;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl *= up;
        }
        float T = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) T = 1.0f;
        float wd = 0.0f, wt = 0.0f;
        for (int i = i0; i < i1; ++i) {
            const float alpha = s_alpha[i];
            const float w = alpha * T;
            s_T[i] = T;
            s_w[i] = w;
            T *= __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
            wd = fmaf(w, 0.5f * (s_depth[i] + s_depth[i + 1]), wd);
            wt += w;
        }
        wd = warp_sum(wd);
        wt = warp_sum(wt);
        __syncwarp();

        // ---- per-sample dot products with the output gradients: dot_k = sum_c gvec[c] * rec_k[c],
        //      gvec = {0, g_seg[15], 2*g_rgb[32]} (rgb is scaled by 2 on output, ray_marcher.py:98)
        const int half = lane >> 4, q = lane & 15;
        const bool on = q < 12;
        float4 gv = make_float4(0.f, 0.f, 0.f, 0.f);
        float g_rgb_sum = 0.0f;
        if (on) {
            if (q >= 4) {
                const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.g_rgb + ray * 32) + (q - 4));
                gv = make_float4(2.0f * g4.x, 2.0f * g4.y, 2.0f * g4.z, 2.0f * g4.w);
                if (half == 0) g_rgb_sum = g4.x + g4.y + g4.z + g4.w;
            } else if (a.g_seg && a.cs) {
                const float* gs = a.g_seg + ray * 15;
                gv = make_float4(q > 0 ? __ldg(gs + 4 * q - 1) : 0.0f, __ldg(gs + 4 * q), __ldg(gs + 4 * q + 1), __ldg(gs + 4 * q + 2));
            }
        }
        g_rgb_sum = warp_sum(g_rgb_sum);
        const float4* r1 = reinterpret_cast<const float4*>(a.rec1 + ray * a.s1 * 48) + (on ? q : 0);
        const float4* r2 = a.s2 ? reinterpret_cast<const float4*>(a.rec2 + (ray * a.s2 - a.s1) * 48) + (on ? q : 0) : r1;
        constexpr int UN = 4;                              // 8 record rows in flight per warp (one load per row used to be waited for in turn)
        for (int k0 = 0; k0 < S; k0 += 2 * UN) {
            float4 v[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int k = k0 + 2 * u + half;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < S && on) {
                    const int e = s_order[k];
                    v[u] = __ldg((e < a.s1 ? r1 : r2) + e * 12);
                }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int k = k0 + 2 * u + half;
                float part = gv.x * v[u].x + gv.y * v[u].y + gv.z * v[u].z + gv.w * v[u].w;
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                if (q == 0 && k < S) s_dot[k] = part;
            }
        }
        __syncwarp();

        // ---- dL/dw_i, suffix sums, dL/d(sigma_mid_i)
        const float d_raw = __fdiv_rn(wd, wt);
        const bool depth_live = a.g_depth && (d_raw == d_raw) && d_raw >= dmin && d_raw <= dmax;
        const float gd = depth_live ? a.g_depth[ray] : 0.0f;
        const float c0 = (a.g_wsum ? a.g_wsum[ray] : 0.0f) - (a.white_back ? 2.0f * g_rgb_sum : 0.0f);
        float local = 0.0f;
        for (int i = i0; i < i1; ++i) {
            float G = 0.5f * (s_dot[i] + s_dot[i + 1]) + c0;
            if (depth_live) G += gd * (0.5f * (s_depth[i] + s_depth[i + 1]) - d_raw) / wt;
            s_gsm[i] = G;
            local += G * s_w[i];
        }
        // exclusive suffix sum over lane chunks
        float suffix = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float dn = __shfl_down_sync(0xffffffffu, suffix, o);
            if (lane + o < 32) suffix += dn;
        }
        float after = __shfl_down_sync(0xffffffffu, suffix, 1);   // sum over all later lanes
        if (lane == 31) after = 0.0f;
        for (int i = i1 - 1; i >= i0; --i) {
            const float G = s_gsm[i], alpha = s_alpha[i];
            const float keep = __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
            const float g_alpha = G * s_T[i] - after / keep;
            after += G * s_w[i];
            const float delta = __fsub_rn(s_depth[i + 1], s_depth[i]);
            const float xs = __fsub_rn(__fdiv_rn(__fadd_rn(s_sigma[i], s_sigma[i + 1]), 2.0f), 1.0f);
            const float sg = __fdividef(1.0f, 1.0f + __expf(-xs));        // d softplus / dx
            s_gsm[i] = g_alpha * delta * (1.0f - alpha) * sg;             // d alpha / d dens = delta * exp(-dens*delta)
        }
        __syncwarp();

        // ---- per-sample gradients, written back in the original (coarse | fine) sample order
        float4* o1 = reinterpret_cast<float4*>(a.g_rec1 + ray * a.s1 * 48) + (on ? q : 0);
        float4* o2 = a.s2 ? reinterpret_cast<float4*>(a.g_rec2 + (ray * a.s2 - a.s1) * 48) + (on ? q : 0) : o1;
        for (int k0 = 0; k0 < S; k0 += 2) {
            const int k = k0 + half;
            if (k < S && on) {
                const float om = 0.5f * ((k > 0 ? s_w[k - 1] : 0.0f) + (k < n_int ? s_w[k] : 0.0f));
                float4 g = make_float4(om * gv.x, om * gv.y, om * gv.z, om * gv.w);
                if (q == 0) g.x = 0.5f * ((k > 0 ? s_gsm[k - 1] : 0.0f) + (k < n_int ? s_gsm[k] : 0.0f));
                const int e = s_order[k];
                (e < a.s1 ? o1 : o2)[e * 12] = g;
            }
        }
        __syncwarp();
    }
}

// plane-mean features of one plane set at ray samples: out [total,32]; 8 lanes per sample
__global__ void __launch_bounds__(256) feature_mean_kernel(FieldGeom gm, const float* __restrict__ set, float* __restrict__ out)
{
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const int c4 = threadIdx.x & 7;
    if (gid >= gm.total) return;
    const int64_t ray = gid / gm.s_per_ray;
    const float t = __ldg(gm.depths + gid);
    const float* o = gm.origins + ray * 3;
    const float* d = gm.dirs + ray * 3;
    const float x = ray_point(__ldg(o), t, __ldg(d)), y = ray_point(__ldg(o + 1), t, __ldg(d + 1)), z = ray_point(__ldg(o + 2), t, __ldg(d + 2));
    const TapSet ts = make_tapset(taps3(__fmul_rn(gm.scale, x), __fmul_rn(gm.scale, y), __fmul_rn(gm.scale, z), gm.H, gm.W), gm.H, gm.W);
    const int64_t item = gm.plane_batch == 1 ? 0 : gid / gm.m;
    const float4 f = gather_set(set + item * (int64_t)3 * gm.H * gm.W * FEAT, ts, c4);
    reinterpret_cast<float4*>(out + gid * FEAT)[c4] = f;
}

__device__ __forceinline__ void red_add_v4(float* addr, float4 v)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// gather backward: g_feat [total,32] (gradient of the plane-MEAN features) -> channel-last plane gradients
__global__ void __launch_bounds__(256) scatter_features_kernel(FieldGeom gm, const float* __restrict__ g_feat, float* __restrict__ g_set)
{
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    const int c4 = threadIdx.x & 7;
    if (gid >= gm.total) return;
    const int64_t ray = gid / gm.s_per_ray;
    const float t = __ldg(gm.depths + gid);
    const float* o = gm.origins + ray * 3;
    const float* d = gm.dirs + ray * 3;
    const float x = ray_point(__ldg(o), t, __ldg(d)), y = ray_point(__ldg(o + 1), t, __ldg(d + 1)), z = ray_point(__ldg(o + 2), t, __ldg(d + 2));
    const TapSet ts = make_tapset(taps3(__fmul_rn(gm.scale, x), __fmul_rn(gm.scale, y), __fmul_rn(gm.scale, z), gm.H, gm.W), gm.H, gm.W);
    const int64_t item = gm.plane_batch == 1 ? 0 : gid / gm.m;
    float4 g = __ldg(reinterpret_cast<const float4*>(g_feat + gid * FEAT) + c4);
    constexpr float third = 1.0f / 3.0f;
    g = make_float4(g.x * third, g.y * third, g.z * third, g.w * third);
    float* base = g_set + item * (int64_t)3 * gm.H * gm.W * FEAT + 4 * c4;
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        const float w = ts.w[i];
        if (w != 0.0f) red_add_v4(base + (int64_t)ts.off4[i] * 4, make_float4(g.x * w, g.y * w, g.z * w, g.w * w));
    }
}

// [n_img, hw, 32] -> [n_img, 32, hw]: lane = pixel, reads its 128-byte texel, writes 32 coalesced channel rows
__global__ void __launch_bounds__(256) from_channel_last32_kernel(const float* __restrict__ in, int64_t hw, int64_t groups_per_img, int64_t n_groups,
                                                                  float* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (group >= n_groups) return;
    const int64_t img = group / groups_per_img;
    const int64_t px = (group % groups_per_img) * 32 + lane;
    if (px >= hw) return;
    const float4* src = reinterpret_cast<const float4*>(in + (img * hw + px) * 32);
    float x[32];
#pragma unroll
    for (int q = 0; q < 8; ++q) { const float4 v = __ldg(src + q); x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w; }
    float* dst = out + img * 32 * hw + px;
#pragma unroll
    for (int c = 0; c < 32; ++c) dst[(int64_t)c * hw] = x[c];
}

}  // namespace nfe

using namespace nfe;

NFE_EXPORT int nfe_composite_bwd(const float* depths1, const float* sigma1, const float* rec1, int s1, const float* depths2, const float* sigma2,
                                 const float* rec2, int s2, int64_t n_rays, int seg_dim, int white_back, const float* g_rgb, const float* g_seg,
                                 const float* g_depth, const float* g_wsum, const float* minmax, float* g_rec1, float* g_rec2, nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(depths1 && sigma1 && rec1 && g_rgb && g_rec1, "nfe_composite_bwd: null pointer");
    NFE_REQUIRE(s2 == 0 || (depths2 && sigma2 && rec2 && g_rec2), "nfe_composite_bwd: second sample set missing");
    const int S = s1 + s2;
    NFE_REQUIRE(S >= 2 && S <= MAX_S, "nfe_composite_bwd: %d samples per ray unsupported (2..%d)", S, MAX_S);
    MarchBwdArgs a = {};
    a.depths1 = depths1; a.sigma1 = sigma1; a.rec1 = rec1; a.s1 = s1; a.depths2 = depths2; a.sigma2 = sigma2; a.rec2 = rec2; a.s2 = s2;
    a.n_rays = n_rays; a.cs = seg_dim; a.white_back = white_back; a.inputs_sorted = 1;
    a.g_rgb = g_rgb; a.g_seg = g_seg; a.g_depth = g_depth; a.g_wsum = g_wsum; a.minmax = minmax; a.g_rec1 = g_rec1; a.g_rec2 = g_rec2;
    int warps = 8;
    while (warps > 1 && (size_t)warps * BWD_ARRAYS * 4 * S > 96 * 1024) warps >>= 1;
    const size_t smem = (size_t)warps * BWD_ARRAYS * 4 * S;
    if (smem > 40 * 1024) cudaFuncSetAttribute(march_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t blocks = (n_rays + warps - 1) / warps;
    const int64_t cap = (int64_t)sm_count() * 8;
    march_bwd_kernel<<<(unsigned)(blocks < cap ? blocks : cap), warps * 32, smem, as_stream(stream)>>>(a);
    NFE_LAUNCH_CHECK("march_bwd_kernel");
    return 0;
}

static int make_geom(FieldGeom& gm, int plane_batch, int height, int width, float box_warp, const float* origins, const float* dirs,
                     const float* depths, int n, int64_t n_rays, int s_per_ray, const char* who)
{
    NFE_REQUIRE(origins && dirs && depths, "%s: null pointer", who);
    NFE_REQUIRE(plane_batch == n || plane_batch == 1, "%s: plane batch %d does not match ray batch %d", who, plane_batch, n);
    NFE_REQUIRE((int64_t)plane_batch * height * width * 3 * (FEAT / 4) < (1ll << 31), "%s: planes exceed the 32-bit texel offsets", who);
    gm.plane_batch = plane_batch; gm.H = height; gm.W = width; gm.scale = (float)(2.0 / (double)box_warp);
    gm.origins = origins; gm.dirs = dirs; gm.depths = depths; gm.s_per_ray = s_per_ray;
    gm.m = n_rays * s_per_ray; gm.total = (int64_t)n * n_rays * s_per_ray;
    return 0;
}

NFE_EXPORT int nfe_feature_mean_fwd(const float* planes_cl, int plane_batch, int height, int width, float box_warp, const float* origins,
                                    const float* dirs, const float* depths, int n, int64_t n_rays, int s_per_ray, float* out, nfe_stream_t stream)
{
    if ((int64_t)n * n_rays * s_per_ray == 0) return 0;
    NFE_REQUIRE(planes_cl && out, "nfe_feature_mean_fwd: null pointer");
    FieldGeom gm = {};
    if (int rc = make_geom(gm, plane_batch, height, width, box_warp, origins, dirs, depths, n, n_rays, s_per_ray, "nfe_feature_mean_fwd")) return rc;
    const int64_t blocks = (gm.total * 8 + 255) / 256;
    NFE_REQUIRE(blocks < (1ll << 31), "nfe_feature_mean_fwd: too many samples for one launch");
    feature_mean_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(gm, planes_cl, out);
    NFE_LAUNCH_CHECK("feature_mean_kernel");
    return 0;
}

NFE_EXPORT int nfe_feature_mean_bwd(const float* g_feat, int plane_batch, int height, int width, float box_warp, const float* origins,
                                    const float* dirs, const float* depths, int n, int64_t n_rays, int s_per_ray, float* g_planes_cl,
                                    nfe_stream_t stream)
{
    if ((int64_t)n * n_rays * s_per_ray == 0) return 0;
    NFE_REQUIRE(g_feat && g_planes_cl, "nfe_feature_mean_bwd: null pointer");
    FieldGeom gm = {};
    if (int rc = make_geom(gm, plane_batch, height, width, box_warp, origins, dirs, depths, n, n_rays, s_per_ray, "nfe_feature_mean_bwd")) return rc;
    const int64_t blocks = (gm.total * 8 + 255) / 256;
    NFE_REQUIRE(blocks < (1ll << 31), "nfe_feature_mean_bwd: too many samples for one launch");
    scatter_features_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(gm, g_feat, g_planes_cl);
    NFE_LAUNCH_CHECK("scatter_features_kernel");
    return 0;
}

NFE_EXPORT int nfe_planes_from_channel_last(const float* planes_cl, int64_t n_img, int channels, int64_t hw, float* out, nfe_stream_t stream)
{
    if (n_img == 0 || hw == 0) return 0;
    NFE_REQUIRE(planes_cl && out, "nfe_planes_from_channel_last: null pointer");
    NFE_REQUIRE(channels == 32, "nfe_planes_from_channel_last: only 32-channel planes are built (got %d)", channels);
    const int64_t groups_per_img = (hw + 31) / 32, n_groups = n_img * groups_per_img;
    NFE_REQUIRE((n_groups + 7) / 8 < (1ll << 31), "nfe_planes_from_channel_last: grid too large");
    from_channel_last32_kernel<<<(unsigned)((n_groups + 7) / 8), 256, 0, as_stream(stream)>>>(planes_cl, hw, groups_per_img, n_groups, out);
    NFE_LAUNCH_CHECK("from_channel_last32_kernel");
    return 0;
}

// Per-ray kernels, one warp per ray: alpha compositing (MipRayMarcher2 / SegMipRayMarcher2,
// ray_marcher.py:25-57,68-101), the coarse+fine merge (unify_samples, renderer.py:150-167,288-300)
// and inverse-CDF importance resampling (sample_importance/sample_pdf, renderer.py:194-253).
// Everything a ray needs between samples stays in the warp's shared-memory slice; cross-lane
// work is shuffle scans.
#include "nfe_march.cuh"

namespace nfe {

__device__ __forceinline__ double shfl_up_double(double v, int delta)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_up_sync(0xffffffffu, lo, delta);
    hi = __shfl_up_sync(0xffffffffu, hi, delta);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_xor_double(double v, int mask)
{
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_xor_sync(0xffffffffu, lo, mask);
    hi = __shfl_xor_sync(0xffffffffu, hi, mask);
    return __hiloint2double(hi, lo);
}

// Weights of the S-1 intervals of one ray (ray_marcher.py:37-47,80-90): s_w[i] = alpha_i * prod_{j<i} (1 - alpha_j + 1e-10).
// Each lane owns a contiguous chunk of intervals; transmittance by a multiplicative warp scan of the chunk products.
// wd / wt return this lane's share of sum w_i * mid-depth_i and sum w_i.  Shared by march_kernel and the fused
// coarse-weights + resample kernel, so both see bit-identical weights.
__device__ __forceinline__ void ray_interval_weights(const float* s_depth, const float* s_sigma, float* s_w, int S, int lane, float& wd, float& wt)
{
    const int n_int = S - 1;
    const int chunk = (n_int + 31) / 32;
    const int i0 = lane * chunk, i1 = min(n_int, i0 + chunk);
    float prod = 1.0f;
    for (int i = i0; i < i1; ++i) {
        const float delta = __fsub_rn(s_depth[i + 1], s_depth[i]);
        const float sig = __fdiv_rn(__fadd_rn(s_sigma[i], s_sigma[i + 1]), 2.0f);
        // SFU exp/log (abs. error ~1e-7): the full-precision versions cost ~80 instructions per interval
        const float xs = __fsub_rn(sig, 1.0f);
        const float dens = fmaxf(xs, 0.0f) + __logf(1.0f + __expf(-fabsf(xs)));
        const float alpha = __fsub_rn(1.0f, __expf(-__fmul_rn(dens, delta)));
        s_w[i] = alpha;  // parked; turned into the weight below
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
    for (int i = i0; i < i1; ++i) {
        const float alpha = s_w[i];
        const float w = __fmul_rn(alpha, T);
        T *= __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
        s_w[i] = w;
        wd = fmaf(w, __fdiv_rn(__fadd_rn(s_depth[i], s_depth[i + 1]), 2.0f), wd);
        wt = __fadd_rn(wt, w);
    }
}

__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ------------------------------------------------------------------------------------------
// march_kernel: optional merge-sort of [set1 | set2] by depth, then mid-point compositing.
//   shared slice per warp: depth[S] sigma[S] weight[S] order[S]
// ------------------------------------------------------------------------------------------
// The packed records go through a per-warp cp.async ring (merge+composite on B200 against register-staged loads: c2 0.142 -> 0.128 ms,
// c3 1.89 -> 1.72 ms, c5 28.7 -> 25.9 ms; 4 / 12 / 16 groups: 0.135 / 0.130 / 0.143).
constexpr int MARCH_RING_GROUPS = 4;    // groups (of 2*MARCH_GROUP_PAIRS rows) in a warp's record ring: 16 rows = 3 KB per warp (6 groups: no better)
constexpr int MARCH_MIN_BLOCKS = 4;     // 64 registers: 4 blocks per SM keep more record rows in flight (merge+composite at c2: 0.157 -> 0.142 ms; 5 is slower)
template <bool SORT>
__global__ void __launch_bounds__(256, MARCH_MIN_BLOCKS) march_kernel(MarchArgs a)
{
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int S = a.s1 + a.s2;
    float* s_depth = smem + (size_t)warp * MARCH_SMEM_FLOATS_PER_SAMPLE * S;
    float* s_sigma = s_depth + S;
    float* s_w = s_sigma + S;
    int* s_order = reinterpret_cast<int*>(s_w + S);
    float* s_raw = s_w + 2 * S;  // unsorted sigma while ranking
    float blk_min = __int_as_float(0x7f800000), blk_max = __int_as_float(0xff800000);

    for (int64_t ray_it = (int64_t)blockIdx.x * warps_per_block + warp; ray_it < a.n_rays; ray_it += (int64_t)gridDim.x * warps_per_block) {
        // Descending ray order: the records the field kernel wrote LAST are still in the 126 MB L2 when this kernel starts
        // (merge + composite at c2: 0.160 -> 0.135 ms).  Fetching a ray's records with cp.async.bulk into shared memory
        // was tried and is slower (0.27 ms: one 8-warp block per SM, each ray's load, weights and sums in series); the
        // per-warp cp.async ring below overlaps the record loads with the merge and the scans instead.
        const int64_t ray = a.n_rays - 1 - ray_it;
        // ---- record ring (packed path, MARCH_RING_GROUPS groups): the rows of a ray are summed in MEMORY order (sum_k omega_k c_order[k] ==
        //      sum_e omega'_e c_e with omega' scattered by entry), so their addresses are known before the merge: the first
        //      MARCH_RING_GROUPS groups are requested here with cp.async and land while the merge and the scans run
        const int rg_half = lane >> 4, rg_q = lane & 15;
        const bool rg_on = rg_q < 12;
        const float4* rg_r1 = nullptr;
        const float4* rg_r2 = nullptr;
        uint32_t rg_slot0 = 0;
        if (a.rec1) {
            rg_r1 = reinterpret_cast<const float4*>(a.rec1 + ray * a.s1 * 48) + rg_q;
            rg_r2 = a.s2 ? reinterpret_cast<const float4*>(a.rec2 + (ray * a.s2 - a.s1) * 48) + rg_q : rg_r1;
            char* ring_base = reinterpret_cast<char*>(smem) + (((size_t)warps_per_block * MARCH_SMEM_FLOATS_PER_SAMPLE * S * 4 + 15) & ~(size_t)15)
                              + (size_t)warp * MARCH_RING_GROUPS * MARCH_RING_GROUP_BYTES;
            rg_slot0 = (uint32_t)__cvta_generic_to_shared(ring_base) + (uint32_t)(rg_half * 192 + rg_q * 16);
            for (int g = 0; g < MARCH_RING_GROUPS; ++g) {
#pragma unroll
                for (int j = 0; j < MARCH_GROUP_PAIRS; ++j) {
                    const int e = 2 * (MARCH_GROUP_PAIRS * g + j) + rg_half;
                    if (rg_on && e < S) cp_async16(rg_slot0 + g * MARCH_RING_GROUP_BYTES + j * 384, (e < a.s1 ? rg_r1 : rg_r2) + e * 12);
                }
                cp_async_commit();
            }
        }
        // ---- load (and merge) depths / densities
        if (SORT) {
            // stage the concatenation in s_w (depth) / s_raw (sigma), then rank-sort (stable: ties keep
            // concatenation order, i.e. coarse before fine).  The coarse list is already sorted and, in
            // parity mode, so is the fine list; a rank sort is also right for the stochastic mode's
            // unsorted fine depths (renderer.py:237).
            for (int e = lane; e < S; e += 32) {
                const bool first = e < a.s1;
                s_w[e] = first ? a.depths1[ray * a.s1 + e] : a.depths2[ray * a.s2 + (e - a.s1)];
                s_raw[e] = first ? a.sigma1[ray * a.s1 + e] : a.sigma2[ray * a.s2 + (e - a.s1)];
            }
            __syncwarp();
            if (a.inputs_sorted) {
                // both lists ascending: merge-path ranks by binary search in the other list
                // (coarse: #fine strictly below; fine: #coarse at or below -> ties keep coarse first)
                for (int e = lane; e < S; e += 32) {
                    const float d = s_w[e];
                    const bool first = e < a.s1;
                    const float* other = first ? s_w + a.s1 : s_w;
                    int lo = 0, hi = first ? a.s2 : a.s1;
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        const float v = other[mid];
                        if (first ? (v < d) : (v <= d)) lo = mid + 1; else hi = mid;
                    }
                    const int rank = (first ? e : e - a.s1) + lo;
                    s_depth[rank] = d; s_sigma[rank] = s_raw[e]; s_order[rank] = e;
                }
            } else {
                for (int e = lane; e < S; e += 32) {
                    const float d = s_w[e];
                    int rank = 0;
#pragma unroll 4
                    for (int j = 0; j < S; ++j) {
                        const float dj = s_w[j];
                        rank += (dj < d) || (dj == d && j < e);
                    }
                    s_depth[rank] = d; s_sigma[rank] = s_raw[e]; s_order[rank] = e;
                }
            }
        } else {
            for (int e = lane; e < S; e += 32) {
                s_depth[e] = a.depths1[ray * a.s1 + e];
                s_sigma[e] = a.sigma1[ray * a.s1 + e];
                s_order[e] = e;
            }
        }
        __syncwarp();

        // ---- weights (ray_interval_weights above); the depth range of the ray for the clamp
        const int n_int = S - 1;
        float dmin = __int_as_float(0x7f800000), dmax = __int_as_float(0xff800000);
        for (int e = lane; e < S; e += 32) { dmin = fminf(dmin, s_depth[e]); dmax = fmaxf(dmax, s_depth[e]); }
        float wd = 0.0f, wt = 0.0f;
        ray_interval_weights(s_depth, s_sigma, s_w, S, lane, wd, wt);
        wd = warp_sum(wd);
        wt = warp_sum(wt);
        dmin = warp_min(dmin);
        dmax = warp_max(dmax);
        blk_min = fminf(blk_min, dmin);
        blk_max = fmaxf(blk_max, dmax);
        __syncwarp();

        // ---- channel sums
        if (a.rec1) {
            // Packed records (48 floats = 12 float4 per sample): a half-warp reads one whole 192-byte row per load,
            // lanes 0-11 take the even rows, lanes 16-27 the odd ones; the two halves are added at the end.
            for (int k = lane; k < S; k += 32) s_sigma[k] = 0.5f * ((k > 0 ? s_w[k - 1] : 0.0f) + (k < n_int ? s_w[k] : 0.0f));
            __syncwarp();
            const int half = lane >> 4, q = lane & 15;
            const bool on = q < 12;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            // omega by entry (s_raw is free after the merge), then walk the ring: group g holds 2*MARCH_GROUP_PAIRS consecutive rows in memory order;
            // every lane reads back exactly the 16 bytes it requested itself, so cp.async.wait_group is all the ordering needed
            for (int k = lane; k < S; k += 32) s_raw[s_order[k]] = s_sigma[k];
            __syncwarp();
            const int n_groups = (S + 2 * MARCH_GROUP_PAIRS - 1) / (2 * MARCH_GROUP_PAIRS);
            int slot = 0;
            for (int g = 0; g < n_groups; ++g) {
                cp_async_wait<MARCH_RING_GROUPS - 1>();       // MARCH_RING_GROUPS groups were committed after group g-1: g has landed
#pragma unroll
                for (int j = 0; j < MARCH_GROUP_PAIRS; ++j) {
                    const int e = 2 * (MARCH_GROUP_PAIRS * g + j) + rg_half;
                    if (rg_on && e < S) {
                        float4 v;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                                     : "r"(rg_slot0 + slot * MARCH_RING_GROUP_BYTES + j * 384) : "memory");
                        const float om = s_raw[e];
                        acc.x = fmaf(om, v.x, acc.x); acc.y = fmaf(om, v.y, acc.y); acc.z = fmaf(om, v.z, acc.z); acc.w = fmaf(om, v.w, acc.w);
                    }
                }
#pragma unroll
                for (int j = 0; j < MARCH_GROUP_PAIRS; ++j) {   // refill the slot just consumed
                    const int e2 = 2 * (MARCH_GROUP_PAIRS * (g + MARCH_RING_GROUPS) + j) + rg_half;
                    if (rg_on && e2 < S) cp_async16(rg_slot0 + slot * MARCH_RING_GROUP_BYTES + j * 384, (e2 < a.s1 ? rg_r1 : rg_r2) + e2 * 12);
                }
                cp_async_commit();
                slot = slot + 1 == MARCH_RING_GROUPS ? 0 : slot + 1;
            }
            acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
            acc.z += __shfl_xor_sync(0xffffffffu, acc.z, 16); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, 16);
            if (half == 0 && on) {
                if (q >= 4) {                                   // rgb channels 4(q-4) .. +3
                    if (a.white_back) { const float bg = 1.0f - wt; acc.x += bg; acc.y += bg; acc.z += bg; acc.w += bg; }
                    const float4 o4 = make_float4(acc.x * 2.0f - 1.0f, acc.y * 2.0f - 1.0f, acc.z * 2.0f - 1.0f, acc.w * 2.0f - 1.0f);
                    if (a.image_rays) {
                        // image layout [item, channel, pixel] (triplane.py:122-125 without the permute+contiguous pass)
                        const int64_t item = ray / a.image_rays, px = ray % a.image_rays;
                        float* im = a.rgb + (item * 32 + 4 * (q - 4)) * a.image_rays + px;
                        im[0] = o4.x; im[a.image_rays] = o4.y; im[2 * a.image_rays] = o4.z; im[3 * a.image_rays] = o4.w;
                    } else {
                        reinterpret_cast<float4*>(a.rgb + ray * 32)[q - 4] = o4;
                    }
                } else if (a.cs) {                              // record floats 4q..4q+3 = {sigma|seg[4q-1 .. 4q+2]}
                    const int64_t item = a.image_rays ? ray / a.image_rays : 0, px = a.image_rays ? ray % a.image_rays : 0;
                    float* sg = a.image_rays ? a.seg + item * 15 * a.image_rays + px : a.seg + ray * 15;
                    const int64_t st = a.image_rays ? a.image_rays : 1;
                    if (q > 0) sg[(4 * q - 1) * st] = acc.x;
                    sg[(4 * q) * st] = acc.y; sg[(4 * q + 1) * st] = acc.z; sg[(4 * q + 2) * st] = acc.w;
                }
            }
        } else if (a.cc > 0) {
            // sum_i w_i (c_i + c_{i+1})/2  ==  sum_k omega_k c_k  with omega_k = (w_{k-1} + w_k)/2 (w_{-1} = w_{S-1} = 0):
            // one FMA per sample row and no carried "previous row"; omega overwrites the (now dead) densities
            for (int k = lane; k < S; k += 32) s_sigma[k] = 0.5f * ((k > 0 ? s_w[k - 1] : 0.0f) + (k < n_int ? s_w[k] : 0.0f));
            __syncwarp();
            for (int c0 = 0; c0 < a.cc; c0 += 32) {
                const int c = c0 + lane;
                const bool on = c < a.cc;
                const bool seg_on = (c0 == 0) && lane < a.cs;
                // row e of the concatenation lives at base1 + e*stride (e < s1) or base2 + e*stride
                const float* c1 = a.colors1 + ray * a.s1 * a.cc + (on ? c : 0);
                const float* c2 = a.s2 ? a.colors2 + (ray * a.s2 - a.s1) * a.cc + (on ? c : 0) : c1;
                const float* g1 = a.cs ? a.segs1 + ray * a.s1 * a.cs + (seg_on ? lane : 0) : nullptr;
                const float* g2 = (a.cs && a.s2) ? a.segs2 + (ray * a.s2 - a.s1) * a.cs + (seg_on ? lane : 0) : g1;
                float acc = 0.0f, acc_s = 0.0f;
                constexpr int UN = 8;  // rows fetched together: the loads are independent, only the sums chain
                int k0 = 0;
                for (; k0 + UN <= S; k0 += UN) {
                    float cur[UN], cur_s[UN];
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        const int e = s_order[k0 + u];
                        cur[u] = __ldg((e < a.s1 ? c1 : c2) + (int64_t)e * a.cc);
                        cur_s[u] = a.cs ? __ldg((e < a.s1 ? g1 : g2) + (int64_t)e * a.cs) : 0.0f;
                    }
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        const float om = s_sigma[k0 + u];
                        acc = fmaf(om, cur[u], acc);
                        acc_s = fmaf(om, cur_s[u], acc_s);
                    }
                }
                for (; k0 < S; ++k0) {
                    const int e = s_order[k0];
                    const float om = s_sigma[k0];
                    acc = fmaf(om, __ldg((e < a.s1 ? c1 : c2) + (int64_t)e * a.cc), acc);
                    if (a.cs) acc_s = fmaf(om, __ldg((e < a.s1 ? g1 : g2) + (int64_t)e * a.cs), acc_s);
                }
                if (on) {
                    if (a.white_back) acc = acc + 1.0f - wt;
                    a.rgb[ray * a.cc + c] = acc * 2.0f - 1.0f;
                }
                if (seg_on) a.seg[ray * a.cs + lane] = acc_s;
            }
            // segs wider than 32 channels are not produced by any decoder of the reference
        }
        if (lane == 0) {
            if (a.depth) a.depth[ray] = __fdiv_rn(wd, wt);  // unclamped; NaN when the ray is empty
            if (a.wsum) a.wsum[ray] = wt;
        }
        if (a.weights) {
            for (int i = lane; i < n_int; i += 32) a.weights[ray * n_int + i] = s_w[i];
        }
        __syncwarp();
    }

    // ---- global depth range for the clamp: block reduce, then one atomic pair per block
    if (a.minmax) {
        __shared__ float red_min[8], red_max[8];
        if (lane == 0) { red_min[warp] = blk_min; red_max[warp] = blk_max; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < warps_per_block; ++w) { blk_min = fminf(blk_min, red_min[w]); blk_max = fmaxf(blk_max, red_max[w]); }
            if (blk_min <= blk_max) { atomic_min_float(a.minmax, blk_min); atomic_max_float(a.minmax + 1, blk_max); }
        }
    }
}

__global__ void init_minmax_kernel(float* minmax)
{
    minmax[0] = __int_as_float(0x7f800000);
    minmax[1] = __int_as_float(0xff800000);
}

// depth = clamp(nan_to_num(depth, nan=+inf), min, max)   (ray_marcher.py:49-50,93-94)
__global__ void finish_depth_kernel(float* __restrict__ depth, int64_t n, const float* __restrict__ minmax)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float lo = minmax[0], hi = minmax[1];
    float d = depth[i];
    if (d != d) d = __int_as_float(0x7f800000);
    if (d == __int_as_float(0x7f800000)) d = 3.402823466e+38f;
    if (d == __int_as_float(0xff800000)) d = -3.402823466e+38f;
    d = fminf(fmaxf(d, lo), hi);
    depth[i] = d;
}

// ------------------------------------------------------------------------------------------
// unify_kernel: stand-alone unify_samples / sort_samples — materialises the sorted attributes.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) unify_kernel(MarchArgs a, float* __restrict__ depths_out, float* __restrict__ colors_out,
                                                    float* __restrict__ segs_out, float* __restrict__ sigma_out)
{
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int S = a.s1 + a.s2;
    float* s_d = smem + (size_t)warp * 2 * S;
    int* s_order = reinterpret_cast<int*>(s_d + S);
    for (int64_t ray = (int64_t)blockIdx.x * warps_per_block + warp; ray < a.n_rays; ray += (int64_t)gridDim.x * warps_per_block) {
        for (int e = lane; e < S; e += 32) s_d[e] = e < a.s1 ? a.depths1[ray * a.s1 + e] : a.depths2[ray * a.s2 + (e - a.s1)];
        __syncwarp();
        for (int e = lane; e < S; e += 32) {
            const float d = s_d[e];
            int rank = 0;
            for (int j = 0; j < S; ++j) {
                const float dj = s_d[j];
                rank += (dj < d) || (dj == d && j < e);
            }
            s_order[rank] = e;
        }
        __syncwarp();
        for (int k = lane; k < S; k += 32) {
            const int e = s_order[k];
            depths_out[ray * S + k] = s_d[e];
            sigma_out[ray * S + k] = e < a.s1 ? a.sigma1[ray * a.s1 + e] : a.sigma2[ray * a.s2 + (e - a.s1)];
        }
        for (int k = 0; k < S; ++k) {
            const int e = s_order[k];
            const bool first = e < a.s1;
            const int64_t row = first ? ray * a.s1 + e : ray * a.s2 + (e - a.s1);
            for (int c = lane; c < a.cc; c += 32) colors_out[(ray * S + k) * a.cc + c] = (first ? a.colors1 : a.colors2)[row * a.cc + c];
            for (int c = lane; c < a.cs; c += 32) segs_out[(ray * S + k) * a.cs + c] = (first ? a.segs1 : a.segs2)[row * a.cs + c];
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// resample_kernel: smoothed coarse weights -> pdf -> cdf -> inverse-CDF samples.
// NORMATIVE arithmetic (SURVEY.md §7.5, oracle nfo_resample_ray): the normaliser is the exact
// sum (double; exact for any order because the addends are fp32 of similar magnitude) rounded to
// fp32, the CDF a double running sum rounded per entry.  No fused multiply-adds.
//   shared slice per warp: z[S] a[S] bins[S] cdf[S]
// ------------------------------------------------------------------------------------------
constexpr int RESAMPLE_MIN_BLOCKS = 4;  // with the coarse weights fused in (c2): 3 blocks 0.060 ms, 4 blocks 0.049 ms (16 bytes of spill), 6 blocks 0.053 ms
// SMOOTH = true : sample_importance — inputs are z_vals [S] and raw coarse weights [S-1];
//                 ns = S-3 pdf entries, bins = the S-1 mid-depths.
// SMOOTH = false: sample_pdf stand-alone — inputs are bins [S] and weights [ns] as given.
template <bool SMOOTH>
__global__ void __launch_bounds__(256, RESAMPLE_MIN_BLOCKS) resample_kernel(ResampleArgs a)
{
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int S = a.S, nw = S - 1, ns = SMOOTH ? S - 3 : a.ns;
    const int per_warp = 4 * S + (a.sort_u ? a.s_f : 0);
    float* s_z = smem + (size_t)warp * per_warp;
    float* s_om = s_z + S;     // omega_j = weight_j + eps, j in [0, ns)
    float* s_bins = s_om + S;
    float* s_cdf = s_bins + S;
    float* s_u = s_cdf + S;    // only when sort_u
    for (int64_t ray = (int64_t)blockIdx.x * warps_per_block + warp; ray < a.n_rays; ray += (int64_t)gridDim.x * warps_per_block) {
        if (SMOOTH) {
            for (int e = lane; e < S; e += 32) s_z[e] = a.z_vals[ray * S + e];
            if (a.sigma) {
                // fused coarse pass (renderer.py:118,340): the compositing weights of the coarse samples are formed here from
                // the densities instead of being written by march_kernel<false> and read back (one launch and a round trip less)
                for (int e = lane; e < S; e += 32) s_om[e] = a.sigma[ray * S + e];
                __syncwarp();
                float wd = 0.0f, wt = 0.0f;
                ray_interval_weights(s_z, s_om, s_cdf, S, lane, wd, wt);
                __syncwarp();
                if (a.weights_out) for (int e = lane; e < nw; e += 32) a.weights_out[ray * nw + e] = s_cdf[e];
            } else {
                for (int e = lane; e < nw; e += 32) s_cdf[e] = a.weights[ray * nw + e];  // raw weights parked in s_cdf
            }
            __syncwarp();
            // max_pool1d(k=2,s=1,pad=1) then avg_pool1d(k=2,s=1), + 0.01 (renderer.py:205-207); bins = mid-depths;
            // only smoothed[1:-1] enters the pdf (renderer.py:210)
            for (int i = lane; i < nw; i += 32) {
                const float w0 = s_cdf[i];
                const float m_i = i > 0 ? fmaxf(s_cdf[i - 1], w0) : w0;                // m[i]
                const float m_n = i + 1 < nw ? fmaxf(w0, s_cdf[i + 1]) : w0;           // m[i+1]
                const float sm = __fadd_rn(__fdiv_rn(__fadd_rn(m_i, m_n), 2.0f), 0.01f);
                if (i >= 1 && i <= ns) s_om[i - 1] = __fadd_rn(sm, a.eps);
                s_bins[i] = __fmul_rn(0.5f, __fadd_rn(s_z[i], s_z[i + 1]));
            }
        } else {
            for (int e = lane; e < S; e += 32) s_bins[e] = a.z_vals[ray * S + e];
            for (int e = lane; e < ns; e += 32) s_om[e] = __fadd_rn(a.weights[ray * ns + e], a.eps);
        }
        __syncwarp();
        double tot = 0.0;
        for (int j = lane; j < ns; j += 32) tot += (double)s_om[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += shfl_xor_double(tot, o);
        const float totf = (float)tot;
        // cdf: contiguous chunk per lane, exclusive double scan across lanes
        const int chunk = (ns + 31) / 32;
        const int j0 = lane * chunk, j1 = min(ns, j0 + chunk);
        double local = 0.0;
        for (int j = j0; j < j1; ++j) local += (double)__fdiv_rn(s_om[j], totf);
        double incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double up = shfl_up_double(incl, o);
            if (lane >= o) incl += up;
        }
        double run = incl - local;
        __syncwarp();
        if (lane == 0) s_cdf[0] = 0.0f;
        for (int j = j0; j < j1; ++j) {
            run += (double)__fdiv_rn(s_om[j], totf);
            s_cdf[j + 1] = (float)run;
        }
        __syncwarp();
        // inverse CDF
        const bool sort_u = a.sort_u && !a.u;
        if (sort_u) {
            // stochastic draws, emitted in ascending order (the sample is monotone in u), so that the fused
            // merge can treat the fine list as sorted; the reference sorts everything later anyway
            for (int k = lane; k < a.s_f; k += 32) s_u[k] = u01(philox4x32(a.seed, (uint64_t)(ray * a.s_f + k), a.offset).x);
            __syncwarp();
        }
        for (int k = lane; k < a.s_f; k += 32) {
            float u;
            int dst = k;
            if (a.u) u = a.u_per_ray ? a.u[ray * a.s_f + k] : a.u[k];
            else if (sort_u) {
                u = s_u[k];
                dst = 0;
                for (int j = 0; j < a.s_f; ++j) {
                    const float uj = s_u[j];
                    dst += (uj < u) || (uj == u && j < k);
                }
            } else u = u01(philox4x32(a.seed, (uint64_t)(ray * a.s_f + k), a.offset).x);
            // searchsorted(right=True): number of cdf entries <= u, over cdf[0..ns]
            int lo = 0, hi = ns + 1;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (s_cdf[mid] <= u) lo = mid + 1; else hi = mid;
            }
            const int below = max(lo - 1, 0), above = min(lo, ns);
            float den = __fsub_rn(s_cdf[above], s_cdf[below]);
            if (den < a.eps) den = 1.0f;
            const float frac = __fdiv_rn(__fsub_rn(u, s_cdf[below]), den);
            const float t = __fadd_rn(s_bins[below], __fmul_rn(frac, __fsub_rn(s_bins[above], s_bins[below])));
            a.out[ray * a.s_f + dst] = t;
            if (a.below) a.below[ray * a.s_f + dst] = below;
            if (a.above) a.above[ray * a.s_f + dst] = above;
        }
        __syncwarp();
    }
}

static int warps_for(int S, int floats_per_sample)
{
    // floats_per_sample*4*S bytes of shared memory per warp; keep a block under ~96 KB
    int w = 8;
    while (w > 1 && (size_t)w * floats_per_sample * 4 * S > 96 * 1024) w >>= 1;
    return w;
}

// dynamic shared memory above the default 48 KB (minus the kernels' small static arrays) needs an opt-in
static constexpr size_t SMEM_OPT_IN = 40 * 1024;

int launch_march(const MarchArgs& a, bool sort, cudaStream_t stream)
{
    const int S = a.s1 + a.s2;
    NFE_REQUIRE(S >= 2 && S <= MAX_S, "ray march: %d samples per ray unsupported (2..%d)", S, MAX_S);
    NFE_REQUIRE(a.cs <= 32, "ray march: at most 32 semantic channels (got %d)", a.cs);
    if (a.n_rays <= 0) return 0;
    const int warps = warps_for(S, MARCH_SMEM_FLOATS_PER_SAMPLE);
    size_t smem = (size_t)warps * MARCH_SMEM_FLOATS_PER_SAMPLE * 4 * S;
    // packed records: cp.async ring of MARCH_RING_GROUPS groups per warp behind the scan arrays
    if (a.rec1) smem = ((smem + 15) & ~(size_t)15) + (size_t)warps * MARCH_RING_GROUPS * MARCH_RING_GROUP_BYTES;
    const int64_t blocks = (a.n_rays + warps - 1) / warps;
    const int64_t cap = (int64_t)sm_count() * 8;
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    if (sort) {
        if (smem > SMEM_OPT_IN) cudaFuncSetAttribute(march_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        march_kernel<true><<<grid, warps * 32, smem, stream>>>(a);
    } else {
        if (smem > SMEM_OPT_IN) cudaFuncSetAttribute(march_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        march_kernel<false><<<grid, warps * 32, smem, stream>>>(a);
    }
    return check_launch("march_kernel");
}

int launch_init_minmax(float* minmax, cudaStream_t stream)
{
    init_minmax_kernel<<<1, 1, 0, stream>>>(minmax);
    return check_launch("init_minmax_kernel");
}

int launch_finish_depth(float* depth, int64_t n, const float* minmax, cudaStream_t stream)
{
    if (n <= 0) return 0;
    finish_depth_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(depth, n, minmax);
    return check_launch("finish_depth_kernel");
}

int launch_resample(const ResampleArgs& a, cudaStream_t stream)
{
    NFE_REQUIRE(a.S >= (a.smooth ? 4 : 2) && a.S <= MAX_S, "importance resampling: %d bins unsupported (%d..%d)", a.S, a.smooth ? 4 : 2, MAX_S);
    NFE_REQUIRE(a.smooth || (a.ns >= 1 && a.ns < a.S), "sample_pdf: %d weights need at least %d bins (got %d)", a.ns, a.ns + 1, a.S);
    NFE_REQUIRE(a.s_f >= 1, "importance resampling: need at least one importance sample");
    if (a.n_rays <= 0) return 0;
    const int per_warp = 4 * a.S + (a.sort_u ? a.s_f : 0);
    int warps = 8;
    while (warps > 1 && (size_t)warps * per_warp * 4 > 96 * 1024) warps >>= 1;
    const size_t smem = (size_t)warps * per_warp * 4;
    const int64_t blocks = (a.n_rays + warps - 1) / warps;
    const int64_t cap = (int64_t)sm_count() * 8;
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    if (a.smooth) {
        if (smem > SMEM_OPT_IN) cudaFuncSetAttribute(resample_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        resample_kernel<true><<<grid, warps * 32, smem, stream>>>(a);
    } else {
        if (smem > SMEM_OPT_IN) cudaFuncSetAttribute(resample_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        resample_kernel<false><<<grid, warps * 32, smem, stream>>>(a);
    }
    return check_launch("resample_kernel");
}

}  // namespace nfe

using namespace nfe;

NFE_EXPORT int nfe_composite_fwd(const float* colors, const float* segs, const float* sigma, const float* depths, int64_t n_rays, int S,
                                 int cc, int cs, int white_back, float* rgb, float* seg, float* depth, float* weights, float* wsum,
                                 float* minmax_ws, nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(sigma && depths, "nfe_composite_fwd: null sigma/depths");
    NFE_REQUIRE(cc == 0 || (colors && rgb), "nfe_composite_fwd: colours given without output (or vice versa)");
    NFE_REQUIRE(cs == 0 || (segs && seg), "nfe_composite_fwd: semantics given without output (or vice versa)");
    NFE_REQUIRE(!depth || minmax_ws, "nfe_composite_fwd: depth output needs the 2-float minmax workspace");
    MarchArgs a = {};
    a.depths1 = depths; a.colors1 = colors; a.segs1 = segs; a.sigma1 = sigma; a.s1 = S; a.s2 = 0;
    a.n_rays = n_rays; a.cc = cc; a.cs = cs; a.white_back = white_back;
    a.rgb = rgb; a.seg = seg; a.depth = depth; a.wsum = wsum; a.weights = weights; a.minmax = depth ? minmax_ws : nullptr;
    if (depth) { if (int rc = launch_init_minmax(minmax_ws, as_stream(stream))) return rc; }
    if (int rc = launch_march(a, false, as_stream(stream))) return rc;
    if (depth) return launch_finish_depth(depth, n_rays, minmax_ws, as_stream(stream));
    return 0;
}

NFE_EXPORT int nfe_finish_depth(float* depth, int64_t n_rays, const float* minmax_dev, nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(depth && minmax_dev, "nfe_finish_depth: null pointer");
    return launch_finish_depth(depth, n_rays, minmax_dev, as_stream(stream));
}

NFE_EXPORT int nfe_importance_resample(const float* z_vals, const float* weights, int64_t n_rays, int S, int s_f, const float* u,
                                       int u_per_ray, uint64_t seed, uint64_t offset, float* out, int32_t* below, int32_t* above,
                                       nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(z_vals && weights && out, "nfe_importance_resample: null pointer");
    ResampleArgs a = {};
    a.z_vals = z_vals; a.weights = weights; a.n_rays = n_rays; a.S = S; a.s_f = s_f; a.u = u; a.u_per_ray = u_per_ray;
    a.seed = seed; a.offset = offset; a.out = out; a.below = below; a.above = above;
    a.smooth = 1; a.eps = 1e-5f;
    return launch_resample(a, as_stream(stream));
}

NFE_EXPORT int nfe_sample_pdf(const float* bins, const float* weights, int64_t n_rays, int n_bins, int n_weights, int s_f, const float* u,
                              int u_per_ray, uint64_t seed, uint64_t offset, float eps, float* out, nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(bins && weights && out, "nfe_sample_pdf: null pointer");
    ResampleArgs a = {};
    a.z_vals = bins; a.weights = weights; a.n_rays = n_rays; a.S = n_bins; a.ns = n_weights; a.s_f = s_f; a.u = u; a.u_per_ray = u_per_ray;
    a.seed = seed; a.offset = offset; a.out = out; a.smooth = 0; a.eps = eps;
    return launch_resample(a, as_stream(stream));
}

NFE_EXPORT int nfe_unify_samples(const float* depths1, const float* colors1, const float* segs1, const float* sigma1, const float* depths2,
                                 const float* colors2, const float* segs2, const float* sigma2, int64_t n_rays, int s1, int s2, int cc, int cs,
                                 float* depths, float* colors, float* segs, float* sigma, nfe_stream_t stream)
{
    if (n_rays <= 0) return 0;
    NFE_REQUIRE(depths1 && sigma1 && depths && sigma, "nfe_unify_samples: null pointer");
    NFE_REQUIRE(s2 == 0 || (depths2 && sigma2), "nfe_unify_samples: second sample set missing");
    NFE_REQUIRE(cc == 0 || (colors1 && colors && (s2 == 0 || colors2)), "nfe_unify_samples: colour pointers missing");
    NFE_REQUIRE(cs == 0 || (segs1 && segs && (s2 == 0 || segs2)), "nfe_unify_samples: semantic pointers missing");
    const int S = s1 + s2;
    NFE_REQUIRE(S >= 1 && S <= MAX_S, "nfe_unify_samples: %d samples per ray unsupported (1..%d)", S, MAX_S);
    if (n_rays <= 0) return 0;
    MarchArgs a = {};
    a.depths1 = depths1; a.colors1 = colors1; a.segs1 = segs1; a.sigma1 = sigma1; a.s1 = s1;
    a.depths2 = depths2; a.colors2 = colors2; a.segs2 = segs2; a.sigma2 = sigma2; a.s2 = s2;
    a.n_rays = n_rays; a.cc = cc; a.cs = cs;
    int warps = 8;
    while (warps > 1 && (size_t)warps * 8 * S > SMEM_OPT_IN) warps >>= 1;
    const size_t smem = (size_t)warps * 8 * S;
    const int64_t blocks = (n_rays + warps - 1) / warps;
    const int64_t cap = (int64_t)sm_count() * 8;
    unify_kernel<<<(unsigned)(blocks < cap ? blocks : cap), warps * 32, smem, as_stream(stream)>>>(a, depths, colors, segs, sigma);
    NFE_LAUNCH_CHECK("unify_kernel");
    return 0;
}

// Host-side launch interface of the per-ray kernels (shared by nfe_march.cu and nfe_render.cu).
#pragma once
#include "nfe_common.cuh"

namespace nfe {

constexpr int MARCH_SMEM_FLOATS_PER_SAMPLE = 5;  // depth, sigma, weight, order, unsorted sigma
constexpr int MARCH_GROUP_PAIRS = 2;  // row pairs per ring group (one cp.async per lane and pair); 2 halves the wait/commit/loop overhead per row: same box, 0.138 -> 0.125 ms
constexpr int MARCH_RING_GROUP_BYTES = MARCH_GROUP_PAIRS * 2 * 192;  // one ring group = pairs of 192-byte record rows (one row per half-warp)
constexpr int MAX_S = 768;  // merged samples per ray (reference configs go up to 192+192, SURVEY.md §8a)

struct MarchArgs {
    // sample set 1 (coarse) and optional set 2 (fine); rows are [n_rays, s, *]
    const float* depths1; const float* colors1; const float* segs1; const float* sigma1; int s1;
    const float* depths2; const float* colors2; const float* segs2; const float* sigma2; int s2;
    // packed alternative to colors/segs (the fused render's workspace): rec[row] = {sigma, seg[15], rgb[32]}, 48 floats;
    // implies cc = 32 and cs = 15 or 0
    const float* rec1; const float* rec2;
    int64_t n_rays;
    int cc, cs;        // colour / semantic channels (0: weights only)
    int64_t image_rays; // packed path only: > 0 writes rgb / seg as images [item, channel, image_rays] instead of [ray, channel]
    int inputs_sorted; // both sample sets ascending in depth: merge by binary search instead of a full rank sort
    int white_back;
    float* rgb;        // [n_rays,cc]
    float* seg;        // [n_rays,cs]
    float* depth;      // [n_rays], UNCLAMPED (finish_depth applies the global clamp)
    float* wsum;       // [n_rays]
    float* weights;    // [n_rays, s1+s2-1] or NULL
    float* minmax;     // device {min,max} of all sample depths, accumulated atomically, or NULL
};

struct ResampleArgs {
    const float* z_vals; const float* weights;  // smooth: depths [S] + raw coarse weights [S-1]; else bins [S] + pdf weights [ns]
    const float* sigma; float* weights_out;     // smooth only: densities [S] instead of `weights` (the kernel forms the compositing weights itself,
                                                // ray_marcher.py:37-47) and, optionally, where to export them [S-1]
    int smooth; int ns; float eps;
    int sort_u;        // stochastic draws only: emit the samples in ascending order
    int64_t n_rays; int S, s_f;
    const float* u; int u_per_ray;
    uint64_t seed, offset;
    float* out; int32_t* below; int32_t* above;
};

int launch_march(const MarchArgs& a, bool sort, cudaStream_t stream);
int launch_init_minmax(float* minmax, cudaStream_t stream);
int launch_finish_depth(float* depth, int64_t n, const float* minmax, cudaStream_t stream);
int launch_resample(const ResampleArgs& a, cudaStream_t stream);

}  // namespace nfe

// Tensor-core (tcgen05 + TMEM) path of the stand-alone decoder (nfe_decoder_fwd in the bf16x3 / bf16 precisions) on
// materialised features.  See nfe_mlp_tc.cuh for the GEMM formulation; this file owns the CTA-level choreography:
//
//   all threads   build the 128-row feature tile (bf16 hi/lo parts) in shared memory
//   fence.proxy.async + barrier
//   one thread    tcgen05.mma layer 1 (both nets) -> tcgen05.commit -> mbarrier
//   all threads   wait, tcgen05.ld own TMEM lane, softplus, write the hidden tile (bf16 parts)
//   fence.proxy.async + barrier
//   one thread    tcgen05.mma layer 2 -> commit -> mbarrier
//   all threads   wait, tcgen05.ld, bias + activations, results out
#include "nfe_field_launch.cuh"
#include "nfe_mlp_tc.cuh"

namespace nfe {

using namespace tcmlp;

template <int KIND, bool SPLIT>
__device__ __forceinline__ void tc_setup(Smem<KIND, SPLIT>& s, const nfe_mlp& net_a, const nfe_mlp& net_b)
{
    if (threadIdx.x < 32) tc::tmem_alloc(&s.tmem_base, TMEM_COLS);
    if (threadIdx.x == 32) {
        tc::mbar_init(&s.bar[0], 1);
        tc::mbar_init(&s.bar[1], 1);
        tc::mbar_fence_init();
    }
    load_params(s, net_a, net_b);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
}

template <int KIND, bool SPLIT>
__device__ __forceinline__ void tc_teardown(Smem<KIND, SPLIT>& s)
{
    tc::fence_before_sync();
    __syncthreads();
    if (threadIdx.x < 32) tc::tmem_dealloc(s.tmem_base, TMEM_COLS);
}

// Runs both layers on the feature tile currently in s.a1 and leaves this thread's outputs in
// (sigma, segv, col).  Must be called by all 128 threads; `parity` flips every call.
template <int KIND, bool SPLIT>
__device__ __forceinline__ void tc_decode_tile(Smem<KIND, SPLIT>& s, uint32_t parity, float& sigma, float (&segv)[16], float (&col)[32])
{
    using T = TcTraits<KIND>;
    const int row = threadIdx.x;                       // TMEM lane == tile row == sample
    const uint32_t tmem = s.tmem_base;
    const uint32_t lane_addr = tmem + ((uint32_t)(row & ~31) << 16);   // a warp may only touch its own 32 lanes

    tc::fence_async_smem();                            // feature tile (generic proxy) -> visible to the tensor core
    tc::fence_before_sync();
    __syncthreads();
    if (threadIdx.x == 0) {
        tc::fence_after_sync();
        issue_layer1<KIND, SPLIT>(s, tmem);
        tc::mma_commit(&s.bar[0]);
    }
    tc::mbar_wait(&s.bar[0], parity);
    tc::fence_after_sync();
    hidden_epilogue<SPLIT>(lane_addr + COL_D1A, s.bias1[0], s.a2[0], row);
    if constexpr (T::HAS_B) hidden_epilogue<SPLIT>(lane_addr + COL_D1B, s.bias1[1], s.a2[1], row);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    if (threadIdx.x == 0) {
        tc::fence_after_sync();
        issue_layer2<KIND, SPLIT>(s, tmem);
        tc::mma_commit(&s.bar[1]);
    }
    tc::mbar_wait(&s.bar[1], parity);
    tc::fence_after_sync();
    output_epilogue<KIND, SPLIT>(s, lane_addr, sigma, segv, col);
}

// ------------------------------------------------------------------------------------------
// Stand-alone decoder on materialised [n,3,m,32] features.
// ------------------------------------------------------------------------------------------
template <int KIND, bool SPLIT>
__global__ void __launch_bounds__(TILE_M, 1) decoder_tc_kernel(nfe_mlp net_a, nfe_mlp net_b, const float* __restrict__ feat_norm,
                                                               const float* __restrict__ feat_denorm, int n, int64_t m,
                                                               float* __restrict__ rgb, float* __restrict__ sigma_out, float* __restrict__ seg)
{
    using T = TcTraits<KIND>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<KIND, SPLIT>& s = *reinterpret_cast<Smem<KIND, SPLIT>*>(smem_raw);
    tc_setup(s, net_a, net_b);

    const int64_t total = (int64_t)n * m;
    const int64_t n_tiles = (total + TILE_M - 1) / TILE_M;
    uint32_t parity = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, parity ^= 1) {
        const int row = threadIdx.x;
        const int64_t idx = tile * TILE_M + row;
        const bool live = idx < total;
        const int64_t b = live ? idx / m : 0, i = live ? idx % m : 0;
        const int64_t o0 = ((b * 3 + 0) * m + i) * FEAT, o1 = ((b * 3 + 1) * m + i) * FEAT, o2 = ((b * 3 + 2) * m + i) * FEAT;
#pragma unroll
        for (int set = 0; set < T::SETS; ++set) {
            const float* f = (T::SETS == 2 && set == 0) ? feat_norm : feat_denorm;
#pragma unroll
            for (int c = 0; c < FEAT / 4; ++c) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (live) {
                    const float4 a0 = __ldg(reinterpret_cast<const float4*>(f + o0) + c);
                    const float4 a1 = __ldg(reinterpret_cast<const float4*>(f + o1) + c);
                    const float4 a2 = __ldg(reinterpret_cast<const float4*>(f + o2) + c);
                    v.x = __fdiv_rn(__fadd_rn(__fadd_rn(a0.x, a1.x), a2.x), 3.0f); v.y = __fdiv_rn(__fadd_rn(__fadd_rn(a0.y, a1.y), a2.y), 3.0f);
                    v.z = __fdiv_rn(__fadd_rn(__fadd_rn(a0.z, a1.z), a2.z), 3.0f); v.w = __fdiv_rn(__fadd_rn(__fadd_rn(a0.w, a1.w), a2.w), 3.0f);
                }
                store_features4<SPLIT>(s.a1[set], row, 4 * c, v);
            }
        }
        float sig, segv[16], col[32];
        tc_decode_tile<KIND, SPLIT>(s, parity, sig, segv, col);
        if (live) {
            sigma_out[idx] = sig;
#pragma unroll
            for (int c = 0; c < 8; ++c)
                reinterpret_cast<float4*>(rgb + idx * 32)[c] = make_float4(col[4 * c], col[4 * c + 1], col[4 * c + 2], col[4 * c + 3]);
            if constexpr (T::HAS_B) {
#pragma unroll
                for (int c = 0; c < 15; ++c) seg[idx * 15 + c] = segv[c];
            }
        }
        // the next tile's MMAs overwrite TMEM and the operand tiles: everyone must be done reading
        tc::fence_before_sync();
        __syncthreads();
        tc::fence_after_sync();
    }
    tc_teardown(s);
}

template <int KIND, bool SPLIT>
static int launch_decoder_tc_kind(const nfe_mlp& a, const nfe_mlp& b, const float* fn, const float* fd, int n, int64_t m, float* rgb, float* sigma,
                                  float* seg, cudaStream_t stream)
{
    const size_t smem = sizeof(Smem<KIND, SPLIT>) + 128;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(decoder_tc_kernel<KIND, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("decoder_tc_kernel: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e)); return 2; }
        configured = true;
    }
    const int64_t n_tiles = ((int64_t)n * m + TILE_M - 1) / TILE_M;
    const int64_t cap = sm_count();
    decoder_tc_kernel<KIND, SPLIT><<<(unsigned)(n_tiles < cap ? n_tiles : cap), TILE_M, smem, stream>>>(a, b, fn, fd, n, m, rgb, sigma, seg);
    return check_launch("decoder_tc_kernel");
}

int launch_decoder_tc(int kind, int precision, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* fn, const float* fd, int n, int64_t m,
                      float* rgb, float* sigma, float* seg, cudaStream_t stream)
{
    nfe_mlp none = {};
    const bool split = precision == NFE_PREC_BF16X3;
    switch (kind) {
        case NFE_DEC_OSG:
            return split ? launch_decoder_tc_kind<NFE_DEC_OSG, true>(*net_a, none, fn, fd, n, m, rgb, sigma, seg, stream)
                         : launch_decoder_tc_kind<NFE_DEC_OSG, false>(*net_a, none, fn, fd, n, m, rgb, sigma, seg, stream);
        case NFE_DEC_DISENTANGLED:
            return split ? launch_decoder_tc_kind<NFE_DEC_DISENTANGLED, true>(*net_a, *net_b, fn, fd, n, m, rgb, sigma, seg, stream)
                         : launch_decoder_tc_kind<NFE_DEC_DISENTANGLED, false>(*net_a, *net_b, fn, fd, n, m, rgb, sigma, seg, stream);
        default:
            return split ? launch_decoder_tc_kind<NFE_DEC_SEGMENTATION, true>(*net_a, *net_b, fn, fd, n, m, rgb, sigma, seg, stream)
                         : launch_decoder_tc_kind<NFE_DEC_SEGMENTATION, false>(*net_a, *net_b, fn, fd, n, m, rgb, sigma, seg, stream);
    }
}

}  // namespace nfe

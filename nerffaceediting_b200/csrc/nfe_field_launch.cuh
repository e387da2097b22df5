// Host-side launch interface of the fused gather+decode kernel (shared by nfe_field.cu and
// nfe_render.cu).
#pragma once
#include "nfe_common.cuh"

namespace nfe {

constexpr int FIELD_THREADS = 512;

struct FieldArgs {
    const float* set_norm;    // channel-last [plane_batch,3,H,W,32]; unused unless the decoder is disentangled
    const float* set_denorm;
    // Single-gather identity (disentangled decoder, pipelined kernel): when non-NULL the de-normalised planes are
    // norm*scale + shift per (item, plane-major channel) — [affine_items, 96] floats each, affine_items = n or 1 —
    // and set_denorm is not read at all.
    const float* affine_scale; const float* affine_shift; int affine_items;
    int plane_batch, H, W;
    float scale;              // 2 / box_warp
    // sample positions: explicit points, or rays + per-sample depths (sample idx = ray*s_per_ray + s)
    const float* coords;      // [n,m,3] or NULL
    const float* origins;     // [n*R,3]
    const float* dirs;
    const float* depths;      // [n*R*s_per_ray]
    int s_per_ray;
    int64_t m;                // samples per batch item
    int64_t total;            // n*m
    float* sigma;             // [total]
    float* rgb;               // [total,32]
    float* seg;               // [total,15]
    // Packed per-sample record used between the render passes instead of rgb/seg: rec[idx] = {sigma, seg[15], rgb[32]}
    // (48 floats = 12 float4, one contiguous 192-byte row per sample).  sigma is still written to `sigma` as well.
    float* rec;
    float density_noise;
    uint64_t seed, offset;
    int sigma_only;           // write sigma only (rgb / seg / rec untouched); the pipelined kernel also skips the work behind them
};

int check_decoder_dims(int kind, const nfe_mlp* net_a, const nfe_mlp* net_b, const char* who);
// precision: NFE_PREC_FP32 -> SIMT fp32 kernel (nfe_field.cu); NFE_PREC_BF16X3 / NFE_PREC_BF16 -> the tcgen05 kernel
// (nfe_field_pipe2.cu)
int launch_field(int kind, int precision, const FieldArgs& a, const nfe_mlp* net_a, const nfe_mlp* net_b, cudaStream_t stream);
// warp-specialised pipelined tensor-core kernel: two alternating epilogue groups, dedicated tap producers
int launch_field_pipe2(int kind, int precision, const FieldArgs& a, const nfe_mlp* net_a, const nfe_mlp* net_b, cudaStream_t stream);
int launch_decoder_tc(int kind, int precision, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* feat_norm, const float* feat_denorm,
                      int n, int64_t m, float* rgb, float* sigma, float* seg, cudaStream_t stream);

}  // namespace nfe

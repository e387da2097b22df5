/*
 * nfe_b200.h — C ABI of libnfe_b200.so: the sm_100a kernels behind NeRFFaceEditing's tri-plane
 * volume-rendering hot path.
 *
 * The reference has no FFI for this path (it is a composition of ATen ops); its operator
 * convention is torch_utils/custom_ops.py:61-157 (JIT-built plugin, tensors in, TORCH_CHECK ->
 * RuntimeError, outputs allocated by the caller's framework, work enqueued on the current
 * stream).  This header is what a binding for the path would target instead: plain device
 * pointers and sizes, an explicit stream, no torch types.  Each entry cites the reference
 * code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; nfe_last_error() then holds a
 *     message (thread-local).  Nothing throws, nothing allocates device memory: outputs and
 *     workspaces are passed in by the caller (size them with the *_workspace_bytes queries);
 *   - all pointers are DEVICE pointers on the current device unless named `host_*`;
 *     tensors are contiguous fp32 unless stated; `stream` is a cudaStream_t;
 *   - work is only enqueued: no call synchronises the device;
 *   - re-entrant; the only global state is an atomic launch counter.
 */
#ifndef NFE_B200_H
#define NFE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* nfe_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------------------------- */
int nfe_version(void);
const char* nfe_last_error(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
uint64_t nfe_launch_count(void);
/* Measurement hook: when enabled, nfe_render_fwd / nfe_run_model_fwd bracket each stage with CUDA
 * events on the launching stream.  nfe_timing_read waits for the recorded events and returns the
 * summed milliseconds and launch counts per stage: 0 field(coarse) 1 coarse weights + resample
 * 2 field(fine) 3 merge+composite 4 run_model. */
int nfe_timing_enable(int on);
int nfe_timing_read(double* ms_by_stage, int64_t* count_by_stage, int n_stages, int reset);

/* Measurement aid (no product path calls it): gathers random 128-byte lines of `table` ([n_lines,32] floats; 25 MB = one plane set
 * keeps it L2-resident) the way the field kernel reads texels — LDG.128, 8 lanes per line, 4 lines per warp instruction, `depth`
 * (4, 8 or 12) independent loads in flight per warp, one CTA of warps_per_cta warps per SM.  *host_lines_out = lines gathered by the
 * launch; time it with events on `stream`.  bench.py reports the result as roofline.l2_gbs_measured. */
int nfe_bench_l2_gather(const float* table, int64_t n_lines, int warps_per_cta, int depth, int iters, int64_t* host_lines_out,
                        float* sink, nfe_stream_t stream);

/* ---- plane statistics: TriPlaneGenerator.compute_mean_var / normalize_plane /
 *      denormalize_plane, training/triplane.py:56-68 (twins utils.py:146-158) ---------------
 * planes is [n_slabs, hw] (a slab = one (batch, channel) image).  std is sqrt of the unbiased
 * variance.  normalize: (x-mean)/(std+1e-8).  denormalize: x*std'+mean' with slab s using
 * statistics entry s % stat_slabs (per-item stats, or one item's stats for the whole batch,
 * triplane.py:100-101). */
int nfe_plane_stats(const float* planes, int64_t n_slabs, int64_t hw, float* mean, float* std_out,
                    nfe_stream_t stream);
int nfe_plane_normalize(const float* planes, const float* mean, const float* std_in, int64_t n_slabs,
                        int64_t hw, float* out, nfe_stream_t stream);
int nfe_plane_denormalize(const float* norm, const float* mean, const float* std_in, int64_t n_slabs,
                          int64_t stat_slabs, int64_t hw, float* out, nfe_stream_t stream);
/* Backward of normalize_plane (the autograd of triplane.py:56-65): upstream gradients g_norm [n_slabs,hw] (may be NULL),
 * g_mean / g_std [n_slabs] (may be NULL) -> g_planes [n_slabs,hw]; norm and std_in are the forward's outputs.
 * sums_ws is a [n_slabs,2] DOUBLE scratch (per-slab sum(g), sum(g*norm)). */
int nfe_plane_normalize_bwd(const float* g_norm, const float* norm, const float* std_in, const float* g_mean,
                            const float* g_std, int64_t n_slabs, int64_t hw, double* sums_ws, float* g_planes,
                            nfe_stream_t stream);
/* SR pre-resize of the rendered feature image (SURVEY.md §8f f1): torch.nn.functional.interpolate(x, size=(out_h,out_w),
 * mode='bilinear', align_corners=False, antialias=antialias) as called at training/superresolution.py:48-52,80-84,282-286.
 * in [n_img, in_h, in_w] (n_img = batch*channels) -> out [n_img, out_h, out_w]. */
int nfe_resize_bilinear(const float* in, int64_t n_img, int in_h, int in_w, int out_h, int out_w, int antialias,
                        float* out, nfe_stream_t stream);
/* Layout staging for the gather: [n_img, C, hw] (reference NCHW, triplane.py:114-115) ->
 * channel-last [n_img, hw, C] so that one bilinear tap is one contiguous C*4-byte line. */
int nfe_planes_to_channel_last(const float* planes, int64_t n_img, int channels, int64_t hw, float* out,
                               nfe_stream_t stream);

/* normalize_plane fused with the staging of BOTH plane sets: planes is [n_img, 32, hw] (n_img = batch*3);
 * one read produces out_norm (same layout), its channel-last copy and the channel-last copy of the
 * raw planes — what DisentangledImportanceRenderer.forward needs from triplane.py:95,113-119.
 * out_raw_cl may be NULL (the single-gather identity needs only the normalised staging). */
int nfe_plane_normalize_staged(const float* planes, const float* mean, const float* std_in, int64_t n_img,
                               int64_t hw, float* out_norm, float* out_norm_cl, float* out_raw_cl,
                               nfe_stream_t stream);

/* ---- rays: RaySampler.forward, training/volumetric_rendering/ray_sampler.py:24-63 -------- */
int nfe_generate_rays(const float* cam2world /*[n,4,4]*/, const float* intrinsics /*[n,3,3]*/, int n,
                      int resolution, float* origins /*[n,res*res,3]*/, float* dirs, nfe_stream_t stream);
/* math_utils.get_ray_limits_box, training/volumetric_rendering/math_utils.py:46-98 */
int nfe_ray_limits_box(const float* origins, const float* dirs, int64_t n_rays, float box_side_length,
                       float* tmin, float* tmax, nfe_stream_t stream);

/* ---- coarse depths: ImportanceRenderer.sample_stratified, renderer.py:169-192 ------------
 * mode 0: scalar limits, t = table[s] + u*delta;  mode 1: per-ray limits (math_utils.linspace,
 * math_utils.py:101-118);  mode 2: disparity space.  `table` is torch.linspace evaluated on the
 * host ([s_c] device floats); ray_start/ray_end are the Python doubles of rendering_options.  u comes from `jitter` ([n_rays,s_c]) if non-NULL, else from the
 * in-kernel Philox stream (seed, offset) if stochastic != 0, else u = 0 (parity mode). */
int nfe_sample_stratified(int64_t n_rays, int s_c, int mode, const float* table, double ray_start,
                          double ray_end, const float* start_per_ray, const float* end_per_ray,
                          const float* jitter, int stochastic, uint64_t seed, uint64_t offset,
                          float* depths /*[n_rays,s_c]*/, nfe_stream_t stream);

/* ---- tri-plane gather: sample_from_planes, renderer.py:55-65 (+ generate_planes /
 *      project_onto_planes :23-53) -----------------------------------------------------------
 * planes_cl is channel-last [plane_batch,3,H,W,C] (see nfe_planes_to_channel_last); plane_batch
 * is n or 1 (one plane set shared by the whole ray batch).  out is [n,3,m,C]. */
int nfe_sample_planes_fwd(const float* planes_cl, int plane_batch, int channels, int height, int width,
                          const float* coords /*[n,m,3]*/, int n, int64_t m, float box_warp, float* out,
                          nfe_stream_t stream);

/* ---- decoders: OSGDecoder / SegmentationOSGDecoder / DisentangledOSGDecoder,
 *      training/triplane.py:167-270 over FullyConnectedLayer, networks_stylegan2.py:96-127 ---
 * An nfe_mlp is FC(in->hidden) . Softplus . FC(hidden->out) given by the RAW parameters and
 * the layer gains (w_eff = weight*wgain, b_eff = bias*bgain), read on every call. */
typedef struct {
    const float* w1; const float* b1; /* [hidden,in], [hidden] */
    const float* w2; const float* b2; /* [out,hidden], [out]   */
    int in_dim, hidden, out_dim;
    float wgain1, bgain1, wgain2, bgain2;
} nfe_mlp;

enum { NFE_DEC_OSG = 0, NFE_DEC_DISENTANGLED = 1, NFE_DEC_SEGMENTATION = 2 };

/* Arithmetic of the decoder MLPs (everything else on the path is fp32 in every mode):
 *   NFE_PREC_FP32    fp32 FFMA on the CUDA cores;
 *   NFE_PREC_BF16X3  tcgen05 tensor cores, each product as 3 bf16 MMAs (hi*hi + lo*hi + hi*lo),
 *                    fp32 accumulation in TMEM: fp32-grade results (meets the 1e-4 tolerance);
 *   NFE_PREC_BF16    tcgen05 tensor cores, plain bf16 operands (1e-2 tolerance). */
enum { NFE_PREC_FP32 = 0, NFE_PREC_BF16X3 = 1, NFE_PREC_BF16 = 2 };

/* decoder(sampled_features[n,3,m,C], ray_directions) stand-alone.  feat_norm may be NULL for
 * OSG / Segmentation (which ignore it).  rgb [n,m,color_dim], sigma [n,m], seg [n,m,seg_dim]. */
int nfe_decoder_fwd(int kind, int precision, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* feat_norm,
                    const float* feat_denorm, int n, int64_t m, int channels, float* rgb, float* sigma,
                    float* seg, nfe_stream_t stream);

/* ---- ray marching: MipRayMarcher2 / SegMipRayMarcher2.run_forward, ray_marcher.py:25-57,68-101
 * colors [n_rays,S,cc], segs [n_rays,S,cs] (NULL when cs == 0), sigma/depths [n_rays,S].
 * weights [n_rays,S-1] and wsum [n_rays] may be NULL.  depth is clamped to the min/max of the
 * whole depths tensor; minmax_ws is a 2-float device scratch. */
int nfe_composite_fwd(const float* colors, const float* segs, const float* sigma, const float* depths,
                      int64_t n_rays, int S, int cc, int cs, int white_back, float* rgb, float* seg,
                      float* depth, float* weights, float* wsum, float* minmax_ws, nfe_stream_t stream);

/* ---- importance resampling: sample_importance + sample_pdf, renderer.py:194-253 -----------
 * z_vals [n_rays,S], weights [n_rays,S-1] -> out [n_rays,s_f].  u: explicit ([s_f] if
 * u_per_ray == 0 else [n_rays,s_f]); NULL -> Philox U[0,1) (seed, offset) as the reference's
 * torch.rand (sample_pdf det=False).  below/above (int32, optional) expose the bin indices. */
int nfe_importance_resample(const float* z_vals, const float* weights, int64_t n_rays, int S, int s_f,
                            const float* u, int u_per_ray, uint64_t seed, uint64_t offset, float* out,
                            int32_t* below, int32_t* above, nfe_stream_t stream);

/* sample_pdf alone, renderer.py:214-253: bins [n_rays,n_bins], weights [n_rays,n_weights]
 * (n_weights < n_bins) -> out [n_rays,s_f]; eps is the reference's `eps` argument (1e-5). */
int nfe_sample_pdf(const float* bins, const float* weights, int64_t n_rays, int n_bins, int n_weights, int s_f,
                   const float* u, int u_per_ray, uint64_t seed, uint64_t offset, float eps, float* out,
                   nfe_stream_t stream);

/* ---- merge: unify_samples / sort_samples, renderer.py:150-167,288-300 ---------------------
 * Sorts the concatenation [coarse | fine] of one ray's samples by depth and permutes every
 * attribute.  Inputs [n_rays,s1,*] and [n_rays,s2,*]; outputs [n_rays,s1+s2,*].  s2 may be 0
 * (sort_samples).  segs may be NULL when cs == 0. */
int nfe_unify_samples(const float* depths1, const float* colors1, const float* segs1, const float* sigma1,
                      const float* depths2, const float* colors2, const float* segs2, const float* sigma2,
                      int64_t n_rays, int s1, int s2, int cc, int cs, float* depths, float* colors,
                      float* segs, float* sigma, nfe_stream_t stream);

/* ---- fused forward: ImportanceRenderer.forward / DisentangledImportanceRenderer.forward,
 *      renderer.py:88-148,301-363, and .run_model, :142-148,259-287 -------------------------- */
typedef struct {
    int kind;                /* NFE_DEC_* */
    int channels, height, width;
    int s_c, s_f;            /* depth_resolution, depth_resolution_importance (0: single pass) */
    int color_dim, seg_dim;  /* 32, 15 (0 for OSG) */
    int white_back;
    float box_warp;
    float density_noise;     /* sigma += N(0,1)*density_noise when > 0 (renderer.py:146-147) */
    int stochastic;          /* 0: parity mode (u_fine = linspace table); 1: Philox jitter */
    uint64_t seed, offset;   /* Philox stream for stochastic mode / density noise */
    int precision;           /* NFE_PREC_* : arithmetic of the decoder MLPs */
    /* Single-gather identity (disentangled decoder, tensor-core modes): if affine_scale != NULL the
     * de-normalised planes are norm*scale + shift per (item, channel) — device [affine_items, 96] floats,
     * affine_items = n or 1 (e.g. std+1e-8 / mean of normalize_plane, or swapped statistics,
     * triplane.py:93-107) — and planes_denorm_cl may be NULL: only the normalised planes are gathered. */
    const float* affine_scale;
    const float* affine_shift;
    int affine_items;
    /* nfe_run_model_fwd only: compute and write sigma alone (rgb / seg may be NULL).  Shape extraction
     * (gen_samples.py:184-222), the density regulariser (loss.py:310-331) and cross-sections read nothing
     * else; with the disentangled decoder the appearance net and the de-normalised gather are skipped. */
    int sigma_only;
    /* nfe_render_fwd only: write rgb / seg as images [n, channel, n_rays] (the feature_image / seg_image
     * of triplane.py:122-125, i.e. after permute(0,2,1).reshape(N,C,H,W)) instead of [n, n_rays, channel]. */
    int image_layout;
} nfe_render_cfg;

/* bytes of device workspace nfe_render_fwd needs for n*n_rays rays with this cfg */
int64_t nfe_render_workspace_bytes(const nfe_render_cfg* cfg, int n, int64_t n_rays);

/* planes_*_cl: channel-last [plane_batch,3,H,W,C]; planes_norm_cl NULL for OSG/Segmentation.
 * depths_coarse [n,n_rays,s_c] (from nfe_sample_stratified); u_fine [s_f] table (parity mode)
 * or NULL.  Outputs rgb [n,n_rays,color_dim], seg [n,n_rays,seg_dim] (NULL if seg_dim == 0),
 * depth [n,n_rays], wsum [n,n_rays].  The depth clamp needs the min/max over ALL sample depths
 * (ray_marcher.py:49-50,93-94): they are accumulated into minmax_out (device float[2], optional)
 * and applied when finish_depth != 0.  A ray-sharded render passes finish_depth = 0, all-reduces
 * minmax_out across ranks (MIN / MAX) and then calls nfe_finish_depth.  depths_fine_out /
 * weights_coarse_out are optional stage taps ([n,n_rays,s_f], [n,n_rays,s_c-1]). */
int nfe_render_fwd(const nfe_render_cfg* cfg, const nfe_mlp* net_a, const nfe_mlp* net_b,
                   const float* planes_norm_cl, const float* planes_denorm_cl, int plane_batch,
                   const float* origins, const float* dirs, int n, int64_t n_rays,
                   const float* depths_coarse, const float* u_fine, float* rgb, float* seg, float* depth,
                   float* wsum, float* minmax_out, int finish_depth, float* depths_fine_out,
                   float* weights_coarse_out, void* workspace, int64_t workspace_bytes, nfe_stream_t stream);

/* Byte offsets, inside an nfe_render_fwd workspace, of what the backward pass re-reads:
 * offsets[0..3] = sigma_c [T,s_c], rec_c [T,s_c,48], sigma_f [T,s_f], rec_f [T,s_f,48] (-1 if absent);
 * a record is {sigma, seg[15], rgb[32]}. */
int nfe_render_workspace_layout(const nfe_render_cfg* cfg, int n, int64_t n_rays, int64_t* offsets);

/* ---- backward (BASELINE config 4).  Gradients flow to the plane tensors and the decoder parameters only;
 *      sample positions carry none (depths_fine is detached in the reference, renderer.py:198,211). ----------
 * nfe_composite_bwd: ray_marcher.py:68-101 differentiated over the merged samples of the final pass.  Inputs are
 * the forward's depths / sigma / records of the coarse (1) and fine (2) sets and the gradients of the ray outputs
 * (g_seg, g_depth, g_wsum optional; minmax = the forward depth range for the clamp); outputs are per-sample
 * gradients in record layout {d sigma, d seg[15], d rgb[32]}. */
int nfe_composite_bwd(const float* depths1, const float* sigma1, const float* rec1, int s1, const float* depths2,
                      const float* sigma2, const float* rec2, int s2, int64_t n_rays, int seg_dim, int white_back,
                      const float* g_rgb, const float* g_seg, const float* g_depth, const float* g_wsum,
                      const float* minmax, float* g_rec1, float* g_rec2, nfe_stream_t stream);
/* Decoder inputs recomputed for the backward: plane-MEAN features [n*n_rays*s_per_ray, 32] of one channel-last
 * plane set at ray samples (sample_from_planes + .mean(1), renderer.py:55-65, triplane.py:251-252) ... */
int nfe_feature_mean_fwd(const float* planes_cl, int plane_batch, int height, int width, float box_warp,
                         const float* origins, const float* dirs, const float* depths, int n, int64_t n_rays,
                         int s_per_ray, float* out, nfe_stream_t stream);
/* ... and its backward: scatter-add (red.global.add.v4.f32) of the feature gradients into channel-last plane
 * gradients [plane_batch,3,H,W,32], which the caller zero-initialises. */
int nfe_feature_mean_bwd(const float* g_feat, int plane_batch, int height, int width, float box_warp,
                         const float* origins, const float* dirs, const float* depths, int n, int64_t n_rays,
                         int s_per_ray, float* g_planes_cl, nfe_stream_t stream);
/* Fused backward of gather + decoder (triplane.py:167-270 and renderer.py:55-65 differentiated) for one
 * pass of samples (sample idx = ray*s_per_ray + s at depth depths[idx]), on the tensor cores:
 * recomputes the plane-mean features and hidden activations, back-propagates the per-sample record gradients
 * g_rec [total,48] = d/d{sigma, seg[15], rgb[32]} (rec = the forward's records, for the colour sigmoid), scatter-adds
 * the feature gradients into the two channel-last plane gradients and ACCUMULATES the raw-parameter gradients
 * (shapes of the parameters; FullyConnectedLayer gains applied) — all gradient buffers are zero-initialised /
 * carried by the caller.  kind: NFE_DEC_DISENTANGLED (net_a = geo_net on the normalised planes, net_b = app_net on the raw ones),
 * NFE_DEC_SEGMENTATION (net_a = net, net_b = seg_net, both on the raw planes: planes_norm_cl / g_planes_norm_cl unused) or
 * NFE_DEC_OSG (net_a = net alone: net_b and the g_*_b buffers may be NULL).
 * Single-gather backward: when affine_scale is non-NULL the raw planes are norm*scale + shift per (item, plane-major
 * channel) ([affine_items,96] floats each, affine_items = n or 1; what normalize_plane / denormalize_plane made,
 * triplane.py:61-68).  planes_cl / g_planes_cl are then unused (may be NULL): only the normalised planes are gathered,
 * their gradient carries both branches, and the gradients w.r.t. scale and shift are ACCUMULATED into
 * g_affine_scale / g_affine_shift [affine_items,96] (zero-initialised by the caller). */
int nfe_field_bwd(int kind, const float* planes_norm_cl, const float* planes_cl, int plane_batch, int height, int width,
                  float box_warp, const float* origins, const float* dirs, const float* depths, int n, int64_t n_rays,
                  int s_per_ray, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* rec, const float* g_rec,
                  float* g_planes_norm_cl, float* g_planes_cl, float* g_w1_a, float* g_b1_a, float* g_w2_a, float* g_b2_a,
                  float* g_w1_b, float* g_b1_b, float* g_w2_b, float* g_b2_b, const float* affine_scale,
                  const float* affine_shift, int affine_items, float* g_affine_scale, float* g_affine_shift,
                  nfe_stream_t stream);
/* Backward of run_model (renderer.py:259-287 differentiated; the density regulariser of training/loss.py:310-331 back-propagates
 * through G.sample_mixed -> run_model): nfe_field_bwd at explicit points.  coords [n,m,3]; rec / g_rec [n*m,48] are the forward's
 * outputs and their gradients packed as records {sigma, seg[15], rgb[32]} (only rec's rgb part is read; absent gradients are
 * zeros).  Everything else as nfe_field_bwd.  Sample coordinates carry no gradient. */
int nfe_run_model_bwd(int kind, const float* planes_norm_cl, const float* planes_cl, int plane_batch, int height, int width,
                      float box_warp, const float* coords, int n, int64_t m, const nfe_mlp* net_a, const nfe_mlp* net_b,
                      const float* rec, const float* g_rec, float* g_planes_norm_cl, float* g_planes_cl, float* g_w1_a,
                      float* g_b1_a, float* g_w2_a, float* g_b2_a, float* g_w1_b, float* g_b1_b, float* g_w2_b, float* g_b2_b,
                      const float* affine_scale, const float* affine_shift, int affine_items, float* g_affine_scale,
                      float* g_affine_shift, nfe_stream_t stream);
/* channel-last [n_img, hw, 32] -> reference layout [n_img, 32, hw] (plane gradients back to [N,3,32,H,W]) */
int nfe_planes_from_channel_last(const float* planes_cl, int64_t n_img, int channels, int64_t hw, float* out,
                                 nfe_stream_t stream);

/* ---- training-side consumers of the rendered maps (SURVEY.md §8f row f4), training/loss.py:28-157,276-293 -------------------
 * remap_seg (loss.py:28-53): BiSeNet's 19 face-parsing labels -> the generator's 15; other values pass through. */
int nfe_remap_seg(const int64_t* labels19, int64_t n, int64_t* out, nfe_stream_t stream);
/* torch.nn.CrossEntropyLoss()(logits [n,c,hw], labels [n,hw]) (loss.py:276-277): mean over all pixels of logsumexp - picked logit.
 * loss is a device float[1]; acc_ws a device double[1] scratch.  bwd: g_logits = (softmax - onehot) * g_loss / (n*hw). */
int nfe_seg_cross_entropy_fwd(const float* logits, const int64_t* labels, int n, int c, int64_t hw, float* loss, double* acc_ws,
                              nfe_stream_t stream);
int nfe_seg_cross_entropy_bwd(const float* logits, const int64_t* labels, int n, int c, int64_t hw, const float* g_loss,
                              float* g_logits, nfe_stream_t stream);
/* RGB-uv histogram distances (RGBuvHistBlock h=64 'inverse-quadratic' with intensity scale, compute_hist_dist,
 * compute_seg_hist_dist, compute_whole_hist_dist: loss.py:57-157).  img [b,3,p] in (-1,1); seg [b,c_seg,p] logits whose argmax masks
 * the pixels of each of the n_labels label ids (device int[n_labels]), or NULL with n_labels == 1 for the whole image;
 * lin = torch.linspace(-3,3,64) (device); weights [n_labels] (SEG2WEIGHT, or {1}).  Outputs (device): hist_raw / hist_norm
 * [n_labels,b,3,64,64], totals [n_labels,b], s_ws / dist [n_labels], loss [1] = sum_l weights[l] * Hellinger distance of items
 * 1..b-1 to item 0 / (b-1).  bwd: g_img [b,3,p] (zero-initialised by the caller) += d(g_loss * loss)/d img; item 0 is the detached
 * target and receives none; g_raw_ws is a [n_labels,b,3,64,64] scratch. */
int nfe_hist_dist_fwd(const float* img, const float* seg, const int* label_ids, const float* lin, int b, int c_seg, int n_labels,
                      int64_t p, float sigma, const float* weights, float* hist_raw, float* hist_norm, float* totals, float* s_ws,
                      float* dist, float* loss, nfe_stream_t stream);
int nfe_hist_dist_bwd(const float* img, const float* seg, const int* label_ids, const float* lin, int b, int c_seg, int n_labels,
                      int64_t p, float sigma, const float* hist_raw, const float* hist_norm, const float* totals, const float* s_ws,
                      const float* weights, const float* g_loss, float* g_raw_ws, float* g_img, nfe_stream_t stream);

/* Depth clamp split out for sharded renders: depth = clamp(nan_to_num(depth, +inf), min, max)
 * with {min,max} read from device memory (ray_marcher.py:49-50,93-94). */
int nfe_finish_depth(float* depth, int64_t n_rays, const float* minmax_dev, nfe_stream_t stream);

/* run_model: gather + decode at explicit points.  coords [n,m,3] -> rgb [n,m,color_dim],
 * sigma [n,m], seg [n,m,seg_dim]. */
int nfe_run_model_fwd(const nfe_render_cfg* cfg, const nfe_mlp* net_a, const nfe_mlp* net_b,
                      const float* planes_norm_cl, const float* planes_denorm_cl, int plane_batch,
                      const float* coords, int n, int64_t m, float* rgb, float* sigma, float* seg,
                      void* workspace, int64_t workspace_bytes, nfe_stream_t stream);

/* ---- backbone / super-resolution plugins (SURVEY.md section 8f row f3) ----------------------------------------------------
 * Element types of the activations these ops move (arithmetic is fp32 inside). */
enum { NFE_DTYPE_F32 = 0, NFE_DTYPE_F16 = 1, NFE_DTYPE_BF16 = 2 };

/* bias_act: replaces the reference's bias_act plugin entry `bias_act(x, b, xref, yref, dy, grad, dim, act, alpha, gain, clamp)`
 * (torch_utils/ops/bias_act.cpp:34-99, kernel bias_act.cu:27-151; Python torch_utils/ops/bias_act.py:51-209).
 * x, xref, yref, dy, y: size_x elements of `dtype` in ONE dense memory order (contiguous or channels-last: the caller passes the
 * order it holds, as the reference does).  b: size_b elements or NULL; element i takes b[(i / step_b) % size_b] (step_b = stride of
 * the bias dimension).  act = the reference's cuda_idx (1 linear, 2 relu, 3 lrelu, 4 tanh, 5 sigmoid, 6 elu, 7 selu, 8 softplus,
 * 9 swish).  grad 0: y = clamp(gain * act(x + b)); grad 1: x is dy, y = dx (needs yref, swish needs xref);
 * grad 2: x is the incoming second-order gradient, dy the first-order one.  clamp < 0 disables clamping. */
int nfe_bias_act(const void* x, const void* b, const void* xref, const void* yref, const void* dy, void* y, int64_t size_x,
                 int size_b, int64_t step_b, int dtype, int grad, int act, float alpha, float gain, float clamp, nfe_stream_t stream);

/* upfirdn2d: replaces the reference's plugin entry `upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1, flip, gain)`
 * (torch_utils/ops/upfirdn2d.cpp:20-107, kernels upfirdn2d.cu:33-204; Python torch_utils/ops/upfirdn2d.py:117-214): zero-insert
 * up-sampling, zero padding (negative = crop), FIR filtering with f [fh,fw] (fp32; true convolution unless flip_filter), decimation.
 * x [n,c,in_h,in_w] and y [n,c,out_h,out_w] with explicit element strides {batch, channel, row, column};
 * out = (in*up + pad0 + pad1 - f + down) / down. */
int nfe_upfirdn2d(const void* x, const float* f, void* y, int n, int c, int in_h, int in_w, int out_h, int out_w, int fh, int fw,
                  const int64_t* x_strides, const int64_t* y_strides, int upx, int upy, int downx, int downy, int padx0, int padx1,
                  int pady0, int pady1, int flip_filter, float gain, int dtype, nfe_stream_t stream);

/* modulated_conv2d + the bias_act that follows it, inference forward: replaces `modulated_conv2d(x, weight, styles, noise, up,
 * padding=k//2, resample_filter, demodulate, flip_weight, fused_modconv)` (training/networks_stylegan2.py:34-91) over
 * conv2d_resample's plain and transposed cases (torch_utils/ops/conv2d_resample.py:48-143; the reference executes them as grouped
 * cuDNN convolutions, conv2d_gradfix.py:37-55) and the layer's `bias_act(x, bias, act, gain, clamp)` (networks_stylegan2.py:322-325,
 * 351-352).  Activations are channels-last: x [batch, in_h, in_w, in_ch], y [batch, in_h*up, in_w*up, out_ch], both `dtype`
 * (NFE_DTYPE_F16: fp16 tensor-core operands as the reference's fp16 layers; NFE_DTYPE_F32: bf16 hi/lo split operands, three MMAs per
 * product).  weight [out_ch, in_ch, k, k] and styles [batch, in_ch] are the fp32 master values; the per-sample fold w*s*demod (and the
 * fp16 pre-normalisation, networks_stylegan2.py:55-57) happens inside.  noise: NULL, or fp32 [in_h*up, in_w*up] with
 * noise_batch_stride 0, or per item with the stride in elements; bias: fp32 [out_ch] or NULL; act = bias_act cuda_idx 1 (linear),
 * 2 (relu), 3 (lrelu); clamp < 0 disables.  up = 2 needs the resample filter f [fh, fw] (upfirdn2d.setup_filter). */
typedef struct nfe_modconv_args {
    const void* x;
    const float* weight;
    const float* styles;
    const float* noise;
    int64_t noise_batch_stride;
    const float* bias;
    void* y;
    const float* filter;
    int fh, fw;
    int batch, in_ch, out_ch, in_h, in_w;
    int ksize, up, demodulate, flip_weight;
    int act;
    float alpha, gain, clamp;
    int dtype;
    int64_t weight_batch_stride;   /* 0: one weight for the batch; > 0: per-item weights [batch][out_ch, in_ch, k, k], this many elements
                                      apart — the grouped-convolution form conv2d_resample receives from a fused modulated_conv2d
                                      (networks_stylegan2.py:84-88), whose weights are modulated already: pass styles = NULL, demodulate = 0 */
} nfe_modconv_args;
int64_t nfe_modconv_workspace_bytes(const nfe_modconv_args* args);
int nfe_modulated_conv2d(const nfe_modconv_args* args, void* workspace, int64_t workspace_bytes, nfe_stream_t stream);

/* Layout conversion of an activation tensor between contiguous NCHW [n, c, hw] and channels-last [n, hw, c] (what
 * `x.contiguous(memory_format=torch.channels_last)` / `.contiguous()` do around the reference's fp16_channels_last layers,
 * networks_stylegan2.py:424-433): the convolution kernel reads and writes channels-last, the reference's own code NCHW. */
int nfe_layout_convert(const void* src, void* dst, int64_t n, int c, int64_t hw, int dtype, int to_channels_last, nfe_stream_t stream);

/* Skip-image accumulation of a synthesis block: img [n, c, hw] (fp32, contiguous NCHW) += y [n, hw, c] (channels-last, NFE_DTYPE_F32 or
 * NFE_DTYPE_F16) — replaces `y = y.to(dtype=torch.float32, memory_format=torch.contiguous_format); img = img.add_(y)`
 * (training/networks_stylegan2.py:456-457, training/superresolution.py:249-250) with one pass. */
int nfe_image_accumulate(const void* y_channels_last, float* img, int64_t n, int c, int64_t hw, int dtype, nfe_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NFE_B200_H */

// Forward of ImportanceRenderer / DisentangledImportanceRenderer (renderer.py:88-148,301-363):
// coarse field evaluation -> coarse weights -> importance resampling -> fine field evaluation ->
// merge + composite.  Per-sample decoder outputs live in the caller's workspace between stages;
// the [N,3,M,32] feature tensors of the reference are never materialised.
#include "nfe_field_launch.cuh"
#include "nfe_march.cuh"

using namespace nfe;

namespace {

struct Workspace {
    float* minmax;    // 2 floats (+pad)
    float* sigma_c; float* rec_c;   // densities (compact, for the weights / merge) and packed records {sigma,seg[15],rgb[32]}
                                    // ({sigma,seg[15]} in a geometry-only render, none for its OSG decoder: see record_floats)
    float* w_c;       // [T, s_c-1], not written: resample_kernel forms the coarse weights itself.  Its size stays in
                      // nfe_render_workspace_bytes, which sets how ops.render_fwd chunks a large render (and so each chunk's Philox offset)
    float* depths_f;  // [T, s_f]
    float* sigma_f; float* rec_f;
    int64_t bytes;
};

int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }

// floats per sample record: {sigma, seg[15], rgb[32]}; a geometry-only render keeps {sigma, seg[15]}, and its OSG decoder
// (no semantics) only the densities
int64_t record_floats(const nfe_render_cfg* cfg)
{
    if (!cfg->geometry_only) return 48;
    return cfg->kind == NFE_DEC_OSG ? 0 : 16;
}

Workspace carve(const nfe_render_cfg* cfg, int64_t rays, void* base)
{
    Workspace w = {};
    char* p = static_cast<char*>(base);
    int64_t off = 0;
    auto take = [&](int64_t floats) {
        float* r = reinterpret_cast<float*>(p + off);
        off += align256(floats * (int64_t)sizeof(float));
        return r;
    };
    const int64_t sc = cfg->s_c, sf = cfg->s_f, rec = record_floats(cfg);
    w.minmax = take(64);
    w.sigma_c = take(rays * sc);
    w.rec_c = take(rays * sc * rec);
    if (sf > 0) {
        w.w_c = take(rays * (sc - 1));
        w.depths_f = take(rays * sf);
        w.sigma_f = take(rays * sf);
        w.rec_f = take(rays * sf * rec);
    }
    w.bytes = off;
    return w;
}

}  // namespace

NFE_EXPORT int64_t nfe_render_workspace_bytes(const nfe_render_cfg* cfg, int n, int64_t n_rays)
{
    if (!cfg || n < 0 || n_rays < 0) return -1;
    return carve(cfg, (int64_t)n * n_rays, nullptr).bytes;
}

NFE_EXPORT int nfe_render_workspace_layout(const nfe_render_cfg* cfg, int n, int64_t n_rays, int64_t* offsets)
{
    NFE_REQUIRE(cfg && offsets && n >= 0 && n_rays >= 0, "nfe_render_workspace_layout: bad arguments");
    NFE_REQUIRE(!cfg->geometry_only, "nfe_render_workspace_layout: a geometry_only render has no backward and no workspace layout for it");
    const Workspace w = carve(cfg, (int64_t)n * n_rays, nullptr);
    auto off = [](const float* p) { return p ? (int64_t)(reinterpret_cast<const char*>(p) - static_cast<const char*>(nullptr)) : (int64_t)-1; };
    offsets[0] = off(w.sigma_c); offsets[1] = off(w.rec_c); offsets[2] = cfg->s_f > 0 ? off(w.sigma_f) : -1; offsets[3] = cfg->s_f > 0 ? off(w.rec_f) : -1;
    return 0;
}

NFE_EXPORT int nfe_render_fwd(const nfe_render_cfg* cfg, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* planes_norm_cl,
                              const float* planes_denorm_cl, int plane_batch, const float* origins, const float* dirs, int n, int64_t n_rays,
                              const float* depths_coarse, const float* u_fine, float* rgb, float* seg, float* depth, float* wsum,
                              float* minmax_out, int finish_depth, float* depths_fine_out, float* weights_coarse_out, void* workspace,
                              int64_t workspace_bytes, nfe_stream_t stream_)
{
    NFE_REQUIRE(cfg, "nfe_render_fwd: null cfg");
    NFE_REQUIRE(cfg->s_c >= 2, "nfe_render_fwd: depth_resolution must be >= 2 (got %d)", cfg->s_c);
    NFE_REQUIRE(cfg->s_f >= 0, "nfe_render_fwd: depth_resolution_importance must be >= 0");
    NFE_REQUIRE(cfg->s_f == 0 || cfg->s_c >= 4, "nfe_render_fwd: importance sampling needs depth_resolution >= 4");
    NFE_REQUIRE(cfg->s_c + cfg->s_f <= MAX_S, "nfe_render_fwd: %d+%d samples per ray exceed %d", cfg->s_c, cfg->s_f, MAX_S);
    NFE_REQUIRE(cfg->color_dim == 32, "nfe_render_fwd: decoder_output_dim must be 32 (got %d)", cfg->color_dim);
    if (int rc = check_decoder_dims(cfg->kind, net_a, net_b, "nfe_render_fwd")) return rc;
    const int64_t rays = (int64_t)n * n_rays;
    if (rays == 0) return 0;  // empty tensors carry null pointers
    const int sc = cfg->s_c, sf = cfg->s_f;
    const int64_t pass_samples = n_rays * (sf > 0 && sf < sc ? sf : sc);
    const bool geometry = cfg->geometry_only != 0;
    FieldArgs f = {};
    if (int rc = field_planes(cfg, planes_norm_cl, planes_denorm_cl, plane_batch, n, pass_samples, false, geometry, "nfe_render_fwd", f)) return rc;
    NFE_REQUIRE(origins && dirs && depths_coarse && (rgb || geometry) && depth && wsum, "nfe_render_fwd: null pointer");
    NFE_REQUIRE(cfg->seg_dim == 0 || seg, "nfe_render_fwd: seg output missing");
    NFE_REQUIRE(cfg->s_f == 0 || cfg->stochastic || u_fine, "nfe_render_fwd: parity mode needs the u_fine table");
    NFE_REQUIRE(workspace, "nfe_render_fwd: null workspace");
    const Workspace w = carve(cfg, rays, workspace);
    NFE_REQUIRE(workspace_bytes >= w.bytes, "nfe_render_fwd: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)w.bytes);
    const bool records = record_floats(cfg) > 0;   // the OSG decoder's geometry-only passes write densities alone
    cudaStream_t stream = as_stream(stream_);
    float* minmax = minmax_out ? minmax_out : w.minmax;

    // ---- coarse pass (renderer.py:104-113,325-336)
    f.origins = origins; f.dirs = dirs; f.depths = depths_coarse; f.s_per_ray = sc;
    f.m = n_rays * sc; f.total = rays * sc;
    f.sigma = w.sigma_c; f.rec = records ? w.rec_c : nullptr;
    f.density_noise = cfg->density_noise; f.seed = cfg->seed; f.offset = cfg->offset + 1;
    {
        StageScope t(STAGE_FIELD_COARSE, stream);
        if (int rc = launch_field(cfg->kind, cfg->precision, f, net_a, net_b, stream)) return rc;
    }

    if (int rc = launch_init_minmax(minmax, stream)) return rc;
    MarchArgs m = {};
    m.n_rays = rays; m.white_back = cfg->white_back;
    if (sf > 0) {
        // ---- coarse weights (renderer.py:118,340) and importance resampling (:120,342)
        // One kernel: coarse compositing weights from the densities, then the inverse-CDF draw
        float* df = depths_fine_out ? depths_fine_out : w.depths_f;
        ResampleArgs r = {};
        r.z_vals = depths_coarse; r.n_rays = rays; r.S = sc; r.s_f = sf; r.smooth = 1; r.eps = 1e-5f; r.sort_u = 1;
        r.sigma = w.sigma_c; r.weights_out = weights_coarse_out;
        r.u = cfg->stochastic ? nullptr : u_fine; r.u_per_ray = 0; r.seed = cfg->seed; r.offset = cfg->offset + 2; r.out = df;
        {
            StageScope t(STAGE_RESAMPLE, stream);
            if (int rc = launch_resample(r, stream)) return rc;
        }
        // ---- fine pass (renderer.py:122-129,344-353)
        f.depths = df; f.s_per_ray = sf; f.m = n_rays * sf; f.total = rays * sf;
        f.sigma = w.sigma_f; f.rec = records ? w.rec_f : nullptr; f.offset = cfg->offset + 3;
        {
            StageScope t(STAGE_FIELD_FINE, stream);
            if (int rc = launch_field(cfg->kind, cfg->precision, f, net_a, net_b, stream)) return rc;
        }
        // ---- merge + composite (renderer.py:131-135,355-359)
        m.depths2 = df; m.rec2 = records ? w.rec_f : nullptr; m.sigma2 = w.sigma_f; m.s2 = sf;
        m.inputs_sorted = 1;  // coarse depths ascend by construction; the fine list is emitted sorted (table u, or sort_u)
    }
    m.depths1 = depths_coarse; m.rec1 = records ? w.rec_c : nullptr; m.sigma1 = w.sigma_c; m.s1 = sc;
    // geometry-only: no colour channels (records {sigma, seg[15]}, or for OSG the weights alone: depth and wsum)
    m.cc = geometry ? 0 : 32; m.cs = cfg->seg_dim; m.rgb = geometry ? nullptr : rgb; m.seg = seg; m.depth = depth; m.wsum = wsum; m.weights = nullptr; m.minmax = minmax;
    m.image_rays = cfg->image_layout ? n_rays : 0;
    StageScope t(STAGE_MARCH_FINAL, stream);
    if (int rc = launch_march(m, sf > 0, stream)) return rc;
    if (finish_depth) return launch_finish_depth(depth, rays, minmax, stream);
    return 0;
}

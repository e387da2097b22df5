// Radiance-field evaluation kernels: stand-alone gather (sample_from_planes), stand-alone
// decoders, and the fused gather+decode kernel behind run_model (renderer.py:142-148,259-287)
// that never materialises the [N,3,M,32] feature tensors.
#include "nfe_field.cuh"
#include "nfe_field_launch.cuh"

namespace nfe {

// ------------------------------------------------------------------------------------------
// Stand-alone gather: one thread per (batch, plane, point, channel-quad).
// ------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(256) gather_kernel(const float* __restrict__ planes_cl, int plane_batch, int C, int H, int W,
                                                     const float* __restrict__ coords, int n, int64_t m, float scale,
                                                     float* __restrict__ out)
{
    const int cq_n = C / VEC;
    const int64_t total = (int64_t)n * 3 * m * cq_n;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int cq = (int)(idx % cq_n);
    const int64_t i = (idx / cq_n) % m;
    const int p = (int)((idx / cq_n / m) % 3);
    const int b = (int)(idx / cq_n / m / 3);
    const float* x = coords + ((int64_t)b * m + i) * 3;
    const float qx = __fmul_rn(scale, x[0]), qy = __fmul_rn(scale, x[1]), qz = __fmul_rn(scale, x[2]);
    float gx, gy;
    project(qx, qy, qz, p, gx, gy);
    const Taps t = plane_taps(gx, gy, H, W);
    const int pb = plane_batch == 1 ? 0 : b;
    const float* plane = planes_cl + ((int64_t)pb * 3 + p) * H * W * C + cq * VEC;
    float acc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[v] = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int xx = t.x0 + (k & 1), yy = t.y0 + (k >> 1);
        if (xx >= 0 && xx < W && yy >= 0 && yy < H) {
            const float* src = plane + ((int64_t)yy * W + xx) * C;
            if constexpr (VEC == 4) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(src));
                acc[0] = __fadd_rn(acc[0], __fmul_rn(v.x, t.w[k])); acc[1] = __fadd_rn(acc[1], __fmul_rn(v.y, t.w[k]));
                acc[2] = __fadd_rn(acc[2], __fmul_rn(v.z, t.w[k])); acc[3] = __fadd_rn(acc[3], __fmul_rn(v.w, t.w[k]));
            } else {
                acc[0] = __fadd_rn(acc[0], __fmul_rn(__ldg(src), t.w[k]));
            }
        }
    }
    float* dst = out + (((int64_t)b * 3 + p) * m + i) * C + cq * VEC;
    if constexpr (VEC == 4) *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    else dst[0] = acc[0];
}

// ------------------------------------------------------------------------------------------
// Stand-alone decoders on materialised [n,3,m,32] features: one sample per lane.
// ------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(256, 1) decoder_kernel(nfe_mlp net_a, nfe_mlp net_b, const float* __restrict__ feat_norm,
                                                         const float* __restrict__ feat_denorm, int n, int64_t m,
                                                         float* __restrict__ rgb, float* __restrict__ sigma, float* __restrict__ seg)
{
    using T = DecoderTraits<KIND>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MlpParams<T::OUT_A>& pa = *reinterpret_cast<MlpParams<T::OUT_A>*>(smem_raw);
    MlpParams<T::OUT_B>& pb = *reinterpret_cast<MlpParams<T::OUT_B>*>(smem_raw + sizeof(MlpParams<T::OUT_A>));
    load_mlp(pa, net_a);
    if (T::HAS_B) load_mlp(pb, net_b);
    __syncthreads();
    const int64_t total = (int64_t)n * m;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = idx / m, i = idx % m;
        const int64_t o0 = ((b * 3 + 0) * m + i) * FEAT, o1 = ((b * 3 + 1) * m + i) * FEAT, o2 = ((b * 3 + 2) * m + i) * FEAT;
        float x[FEAT];
        float outa[T::OUT_A];
        const float* fa = (KIND == NFE_DEC_DISENTANGLED) ? feat_norm : feat_denorm;
#pragma unroll
        for (int k = 0; k < FEAT; ++k) x[k] = __fdiv_rn(__fadd_rn(__fadd_rn(fa[o0 + k], fa[o1 + k]), fa[o2 + k]), 3.0f);
        mlp_eval(pa, x, outa);
        sigma[idx] = outa[0];
        if constexpr (KIND == NFE_DEC_DISENTANGLED) {
            for (int c = 0; c < 15; ++c) seg[idx * 15 + c] = outa[1 + c];
#pragma unroll
            for (int k = 0; k < FEAT; ++k) x[k] = __fdiv_rn(__fadd_rn(__fadd_rn(feat_denorm[o0 + k], feat_denorm[o1 + k]), feat_denorm[o2 + k]), 3.0f);
            float outb[T::OUT_B];
            mlp_eval(pb, x, outb);
#pragma unroll
            for (int c = 0; c < 32; ++c) rgb[idx * 32 + c] = rgb_activation(outb[c]);
        } else {
#pragma unroll
            for (int c = 0; c < 32; ++c) rgb[idx * 32 + c] = rgb_activation(outa[1 + c]);
            if constexpr (KIND == NFE_DEC_SEGMENTATION) {
                float outb[T::OUT_B];
                mlp_eval(pb, x, outb);
                for (int c = 0; c < 15; ++c) seg[idx * 15 + c] = outb[c];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Fused gather + decode.  A warp owns 32 consecutive samples per step:
//   phase 1  8 passes; in each, the four 8-lane groups gather one sample each (12 taps per plane
//            set, 128-byte texel per group per LDG.128) and park the plane-mean in the warp's
//            swizzled shared tile;
//   phase 2  one sample per lane: both MLPs from registers, parameters broadcast from shared;
//   phase 3  results staged through the same tile and written out coalesced.
// GEO: the geometry-only render pass (FieldArgs::geometry_only) — 16-float records {sigma, seg[15]}, no colours; with the
// disentangled decoder only the normalised planes are gathered and app_net is not run.  Its own instantiation, so the
// full kernels keep their code.
// ------------------------------------------------------------------------------------------
template <int KIND, bool GEO>
__global__ void __launch_bounds__(FIELD_THREADS, 1) field_kernel(FieldArgs a, nfe_mlp net_a, nfe_mlp net_b)
{
    using T = DecoderTraits<KIND>;
    constexpr bool NORM_ONLY = GEO && KIND == NFE_DEC_DISENTANGLED;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MlpParams<T::OUT_A>& pa = *reinterpret_cast<MlpParams<T::OUT_A>*>(smem_raw);
    MlpParams<T::OUT_B>& pb = *reinterpret_cast<MlpParams<T::OUT_B>*>(smem_raw + sizeof(MlpParams<T::OUT_A>));
    float4* tiles = reinterpret_cast<float4*>(smem_raw + sizeof(MlpParams<T::OUT_A>) + sizeof(MlpParams<T::OUT_B>));
    load_mlp(pa, net_a);
    if (T::HAS_B && !NORM_ONLY) load_mlp(pb, net_b);
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    float4* tile = tiles + warp * 512;  // 8 KB: two 32x32 feature tiles, later one 32x49 output tile
    float* tile_f = reinterpret_cast<float*>(tile);
    const int g = lane >> 3, c4 = lane & 7;
    const int64_t set_stride = (int64_t)3 * a.H * a.W * FEAT;
    const int64_t n_steps = (a.total + 31) / 32;

    for (int64_t step = (int64_t)blockIdx.x * warps_per_block + warp; step < n_steps; step += (int64_t)gridDim.x * warps_per_block) {
        const int64_t base = step * 32;
        // ---- phase 1: gather
#pragma unroll 2
        for (int j = 0; j < 8; ++j) {
            const int row = 4 * j + g;
            const int64_t idx = base + row;
            float4 fa = make_float4(0.f, 0.f, 0.f, 0.f), fb = fa;
            if (idx < a.total) {
                float x, y, z;
                if (a.coords) {
                    const float* c = a.coords + idx * 3;
                    x = __ldg(c); y = __ldg(c + 1); z = __ldg(c + 2);
                } else {
                    const int64_t ray = idx / a.s_per_ray;
                    const float t = __ldg(a.depths + idx);
                    const float* o = a.origins + ray * 3;
                    const float* d = a.dirs + ray * 3;
                    x = ray_point(__ldg(o), t, __ldg(d)); y = ray_point(__ldg(o + 1), t, __ldg(d + 1)); z = ray_point(__ldg(o + 2), t, __ldg(d + 2));
                }
                const int64_t pbi = a.plane_batch == 1 ? 0 : idx / a.m;
                const TapSet ts = make_tapset(taps3(__fmul_rn(a.scale, x), __fmul_rn(a.scale, y), __fmul_rn(a.scale, z), a.H, a.W), a.H, a.W);
                float4 va[12], vb[12];
                if (T::SETS == 2) gather_load(a.set_norm + pbi * set_stride, ts, c4, va);
                if (!NORM_ONLY) gather_load(a.set_denorm + pbi * set_stride, ts, c4, vb);
                if (T::SETS == 2) fa = gather_reduce(va, ts);
                if (!NORM_ONLY) fb = gather_reduce(vb, ts);
            }
            if (T::SETS == 2) tile[tile_chunk(row, c4)] = fa;
            if (!NORM_ONLY) tile[256 + tile_chunk(row, c4)] = fb;
        }
        __syncwarp();

        // ---- phase 2: decode, one sample per lane
        float x[FEAT];
        float sig, segv[16], col[32];
        {
            const float4* src = tile + (T::SETS == 2 ? 0 : 256);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 v = src[tile_chunk(lane, c)];
                x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
            }
            float outa[T::OUT_A];
            mlp_eval(pa, x, outa);
            sig = outa[0];
            if constexpr (KIND == NFE_DEC_DISENTANGLED) {
#pragma unroll
                for (int c = 0; c < 15; ++c) segv[c] = outa[1 + c];
            } else if constexpr (!GEO) {
#pragma unroll
                for (int c = 0; c < 32; ++c) col[c] = rgb_activation(outa[1 + c]);
            }
        }
        if constexpr (T::HAS_B && !NORM_ONLY) {
            if constexpr (T::SETS == 2) {
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 v = tile[256 + tile_chunk(lane, c)];
                    x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
                }
            }
            float outb[T::OUT_B];
            mlp_eval(pb, x, outb);
            if constexpr (KIND == NFE_DEC_DISENTANGLED) {
#pragma unroll
                for (int c = 0; c < 32; ++c) col[c] = rgb_activation(outb[c]);
            } else {
#pragma unroll
                for (int c = 0; c < 15; ++c) segv[c] = outb[c];
            }
        }
        if (a.density_noise > 0.0f) {  // renderer.py:146-147,285-286
            const uint4 r = philox4x32(a.seed, (uint64_t)(base + lane), a.offset);
            sig += normal2(r.x, r.y).x * a.density_noise;
        }
        __syncwarp();

        // ---- phase 3: stage and write out coalesced
        float* row = tile_f + lane * OUT_STRIDE;
        row[0] = sig;
        if constexpr (T::HAS_B) {
#pragma unroll
            for (int c = 0; c < 15; ++c) row[1 + c] = segv[c];
        }
        if constexpr (!GEO) {
#pragma unroll
            for (int c = 0; c < 32; ++c) row[17 + c] = col[c];
        }
        __syncwarp();
        const int rows = (int)min((int64_t)32, a.total - base);
        if (lane < rows) a.sigma[base + lane] = row[0];
        if constexpr (GEO) {
            // geometry records {sigma, seg[15]}: 16 floats per sample, the whole step is one contiguous span
            for (int e = lane; e < rows * 16; e += 32) a.rec[base * 16 + e] = tile_f[(e >> 4) * OUT_STRIDE + (e & 15)];
        } else if (a.sigma_only) {
            // density-only query: nothing else is written
        } else if (a.rec) {
            // packed records {sigma, seg[15], rgb[32]}: 48 floats per sample, the whole step is one contiguous span
            for (int e = lane; e < rows * 48; e += 32) {
                const int r = e / 48, c = e % 48;
                a.rec[base * 48 + e] = (c == 0 || c >= 16 || T::HAS_B) ? tile_f[r * OUT_STRIDE + (c < 16 ? c : c + 1)] : 0.0f;
            }
        } else {
            for (int e = lane; e < rows * 32; e += 32) a.rgb[base * 32 + e] = tile_f[(e >> 5) * OUT_STRIDE + 17 + (e & 31)];
            if constexpr (T::HAS_B) {
                for (int e = lane; e < rows * 15; e += 32) a.seg[base * 15 + e] = tile_f[(e / 15) * OUT_STRIDE + 1 + (e % 15)];
            }
        }
        __syncwarp();
    }
}

template <int KIND, bool GEO>
static int launch_field_kind(const FieldArgs& a, const nfe_mlp& net_a, const nfe_mlp& net_b, cudaStream_t stream)
{
    using T = DecoderTraits<KIND>;
    const size_t smem = sizeof(MlpParams<T::OUT_A>) + sizeof(MlpParams<T::OUT_B>) + (size_t)(FIELD_THREADS / 32) * 8192;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(field_kernel<KIND, GEO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("field_kernel: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e)); return 2; }
        configured = true;
    }
    const int64_t n_steps = (a.total + 31) / 32;
    const int64_t blocks_needed = (n_steps + FIELD_THREADS / 32 - 1) / (FIELD_THREADS / 32);
    const unsigned grid = (unsigned)(blocks_needed < sm_count() ? blocks_needed : sm_count());
    field_kernel<KIND, GEO><<<grid, FIELD_THREADS, smem, stream>>>(a, net_a, net_b);
    return check_launch("field_kernel");
}

int check_decoder_dims(int kind, const nfe_mlp* net_a, const nfe_mlp* net_b, const char* who)
{
    NFE_REQUIRE(kind >= 0 && kind <= 2, "%s: unknown decoder kind %d", who, kind);
    NFE_REQUIRE(net_a && net_a->w1 && net_a->b1 && net_a->w2 && net_a->b2, "%s: net_a parameters missing", who);
    NFE_REQUIRE(net_a->in_dim == FEAT && net_a->hidden == HIDDEN, "%s: net_a must be %d->%d->out (got %d->%d)", who, FEAT, HIDDEN, net_a->in_dim, net_a->hidden);
    const int want_a = kind == NFE_DEC_DISENTANGLED ? 16 : 33;
    NFE_REQUIRE(net_a->out_dim == want_a, "%s: net_a out_dim %d unsupported for kind %d (want %d)", who, net_a->out_dim, kind, want_a);
    if (kind != NFE_DEC_OSG) {
        NFE_REQUIRE(net_b && net_b->w1 && net_b->b1 && net_b->w2 && net_b->b2, "%s: net_b parameters missing", who);
        NFE_REQUIRE(net_b->in_dim == FEAT && net_b->hidden == HIDDEN, "%s: net_b must be %d->%d->out", who, FEAT, HIDDEN);
        const int want_b = kind == NFE_DEC_DISENTANGLED ? 32 : 15;
        NFE_REQUIRE(net_b->out_dim == want_b, "%s: net_b out_dim %d unsupported for kind %d (want %d)", who, net_b->out_dim, kind, want_b);
    }
    return 0;
}

int field_planes(const nfe_render_cfg* cfg, const float* planes_norm_cl, const float* planes_denorm_cl, int plane_batch, int n,
                 int64_t pass_samples, bool sigma_only, bool geometry_only, const char* who, FieldArgs& f)
{
    NFE_REQUIRE(cfg->channels == FEAT, "%s: planes must have %d channels (got %d)", who, FEAT, cfg->channels);
    NFE_REQUIRE(cfg->height >= 1 && cfg->width >= 1, "%s: bad plane size", who);
    NFE_REQUIRE(cfg->box_warp != 0.0f, "%s: box_warp must be non-zero", who);
    NFE_REQUIRE(cfg->precision >= NFE_PREC_FP32 && cfg->precision <= NFE_PREC_BF16, "%s: unknown precision mode %d", who, cfg->precision);
    NFE_REQUIRE(cfg->seg_dim == (cfg->kind == NFE_DEC_OSG ? 0 : 15), "%s: seg_dim %d unsupported for decoder kind %d", who, cfg->seg_dim, cfg->kind);
    const bool disentangled_tc = cfg->kind == NFE_DEC_DISENTANGLED && cfg->precision != NFE_PREC_FP32;
    // a geometry-only render with the disentangled decoder needs geo_net on the normalised planes alone (every precision)
    const bool norm_only = geometry_only && cfg->kind == NFE_DEC_DISENTANGLED;
    // single-gather identity (cfg->affine_*): the de-normalised planes are norm*scale + shift and are not read
    const bool affine = cfg->affine_scale && cfg->affine_shift && disentangled_tc && !norm_only;
    // a density-only query with the disentangled decoder on the tensor cores reads the normalised planes only
    const bool geo_only = (sigma_only && disentangled_tc) || norm_only;
    NFE_REQUIRE(!cfg->affine_scale || cfg->affine_items == 1 || cfg->affine_items == n, "%s: affine statistics for %d items, batch is %d", who,
                cfg->affine_items, n);
    // the field kernel keeps the statistics of two batch items per 128-sample tile: an item must span at least one tile in each pass
    NFE_REQUIRE(!affine || pass_samples >= 128, "%s: the single-gather identity needs at least 128 samples per item and pass (%lld)", who,
                (long long)pass_samples);
    NFE_REQUIRE(planes_denorm_cl || affine || geo_only, "%s: null pointer to the de-normalised planes", who);
    NFE_REQUIRE(cfg->kind != NFE_DEC_DISENTANGLED || planes_norm_cl, "%s: the disentangled decoder needs the normalised planes", who);
    NFE_REQUIRE(plane_batch == n || plane_batch == 1, "%s: plane batch %d does not match batch %d", who, plane_batch, n);
    f.set_norm = planes_norm_cl; f.set_denorm = planes_denorm_cl; f.plane_batch = plane_batch; f.H = cfg->height; f.W = cfg->width;
    f.scale = (float)(2.0 / (double)cfg->box_warp);
    if (affine) { f.affine_scale = cfg->affine_scale; f.affine_shift = cfg->affine_shift; f.affine_items = cfg->affine_items; }
    // the OSG decoder has no semantics: its geometry-only pass is a density-only one (no records)
    f.sigma_only = sigma_only || (geometry_only && cfg->kind == NFE_DEC_OSG);
    f.geometry_only = geometry_only && cfg->kind != NFE_DEC_OSG;
    return 0;
}

int launch_field(int kind, int precision, const FieldArgs& a, const nfe_mlp* net_a, const nfe_mlp* net_b, cudaStream_t stream)
{
    if (a.total <= 0) return 0;
    NFE_REQUIRE((int64_t)a.H * a.W * 3 * FEAT < (1ll << 31), "planes of %dx%d exceed the 32-bit texel offsets of the gather", a.H, a.W);
    NFE_REQUIRE((int64_t)a.plane_batch * a.H * a.W * 3 * (FEAT / 4) < (1ll << 31), "%d plane sets of %dx%d exceed the 32-bit texel offsets of the gather",
                a.plane_batch, a.H, a.W);
    if (precision != NFE_PREC_FP32) return launch_field_pipe2(kind, precision, a, net_a, net_b, stream);
    nfe_mlp none = {};
    if (a.geometry_only) {
        NFE_REQUIRE(kind != NFE_DEC_OSG && a.rec, "field kernel: a geometry-only pass needs a decoder with semantics and the records");
        if (kind == NFE_DEC_DISENTANGLED) return launch_field_kind<NFE_DEC_DISENTANGLED, true>(a, *net_a, *net_b, stream);
        return launch_field_kind<NFE_DEC_SEGMENTATION, true>(a, *net_a, *net_b, stream);
    }
    switch (kind) {
        case NFE_DEC_OSG: return launch_field_kind<NFE_DEC_OSG, false>(a, *net_a, none, stream);
        case NFE_DEC_DISENTANGLED: return launch_field_kind<NFE_DEC_DISENTANGLED, false>(a, *net_a, *net_b, stream);
        default: return launch_field_kind<NFE_DEC_SEGMENTATION, false>(a, *net_a, *net_b, stream);
    }
}

}  // namespace nfe

using namespace nfe;

NFE_EXPORT int nfe_sample_planes_fwd(const float* planes_cl, int plane_batch, int channels, int height, int width, const float* coords,
                                     int n, int64_t m, float box_warp, float* out, nfe_stream_t stream)
{
    if ((int64_t)n * m == 0) return 0;  // empty tensors carry null pointers
    NFE_REQUIRE(planes_cl && coords && out, "nfe_sample_planes_fwd: null pointer");
    NFE_REQUIRE(plane_batch == n || plane_batch == 1, "nfe_sample_planes_fwd: plane batch %d does not match coordinate batch %d", plane_batch, n);
    NFE_REQUIRE(channels >= 1 && height >= 1 && width >= 1 && n >= 0 && m >= 0, "nfe_sample_planes_fwd: bad sizes");
    NFE_REQUIRE(box_warp != 0.0f, "nfe_sample_planes_fwd: box_warp must be non-zero");
    const float scale = (float)(2.0 / (double)box_warp);
    const bool vec = channels % 4 == 0 && ((reinterpret_cast<uintptr_t>(planes_cl) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    const int64_t total = (int64_t)n * 3 * m * (vec ? channels / 4 : channels);
    if (total == 0) return 0;
    NFE_REQUIRE((total + 255) / 256 < (1ll << 31), "nfe_sample_planes_fwd: too many points for one launch");
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (vec) gather_kernel<4><<<grid, 256, 0, as_stream(stream)>>>(planes_cl, plane_batch, channels, height, width, coords, n, m, scale, out);
    else gather_kernel<1><<<grid, 256, 0, as_stream(stream)>>>(planes_cl, plane_batch, channels, height, width, coords, n, m, scale, out);
    NFE_LAUNCH_CHECK("gather_kernel");
    return 0;
}

template <int KIND>
static int launch_decoder(const nfe_mlp& a, const nfe_mlp& b, const float* fn, const float* fd, int n, int64_t m, float* rgb, float* sigma,
                          float* seg, cudaStream_t stream)
{
    using T = DecoderTraits<KIND>;
    const size_t smem = sizeof(MlpParams<T::OUT_A>) + sizeof(MlpParams<T::OUT_B>);
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(decoder_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        configured = true;
    }
    const int64_t total = (int64_t)n * m;
    const int64_t blocks = (total + 255) / 256;
    const unsigned grid = (unsigned)(blocks < 2 * sm_count() ? blocks : 2 * sm_count());
    decoder_kernel<KIND><<<grid, 256, smem, stream>>>(a, b, fn, fd, n, m, rgb, sigma, seg);
    return check_launch("decoder_kernel");
}

NFE_EXPORT int nfe_decoder_fwd(int kind, int precision, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* feat_norm, const float* feat_denorm,
                               int n, int64_t m, int channels, float* rgb, float* sigma, float* seg, nfe_stream_t stream)
{
    NFE_REQUIRE(precision >= NFE_PREC_FP32 && precision <= NFE_PREC_BF16, "nfe_decoder_fwd: unknown precision mode %d", precision);
    if (int rc = check_decoder_dims(kind, net_a, net_b, "nfe_decoder_fwd")) return rc;
    NFE_REQUIRE(channels == FEAT, "nfe_decoder_fwd: features must have %d channels (got %d)", FEAT, channels);
    if ((int64_t)n * m == 0) return 0;
    NFE_REQUIRE(feat_denorm && rgb && sigma, "nfe_decoder_fwd: null pointer");
    NFE_REQUIRE(kind != NFE_DEC_DISENTANGLED || feat_norm, "nfe_decoder_fwd: the disentangled decoder needs feat_norm");
    NFE_REQUIRE(kind == NFE_DEC_OSG || seg, "nfe_decoder_fwd: seg output missing");
    if ((int64_t)n * m == 0) return 0;
    if (precision != NFE_PREC_FP32) return launch_decoder_tc(kind, precision, net_a, net_b, feat_norm, feat_denorm, n, m, rgb, sigma, seg, as_stream(stream));
    nfe_mlp none = {};
    switch (kind) {
        case NFE_DEC_OSG: return launch_decoder<NFE_DEC_OSG>(*net_a, none, feat_norm, feat_denorm, n, m, rgb, sigma, seg, as_stream(stream));
        case NFE_DEC_DISENTANGLED: return launch_decoder<NFE_DEC_DISENTANGLED>(*net_a, *net_b, feat_norm, feat_denorm, n, m, rgb, sigma, seg, as_stream(stream));
        default: return launch_decoder<NFE_DEC_SEGMENTATION>(*net_a, *net_b, feat_norm, feat_denorm, n, m, rgb, sigma, seg, as_stream(stream));
    }
}

NFE_EXPORT int nfe_run_model_fwd(const nfe_render_cfg* cfg, const nfe_mlp* net_a, const nfe_mlp* net_b, const float* planes_norm_cl,
                                 const float* planes_denorm_cl, int plane_batch, const float* coords, int n, int64_t m, float* rgb,
                                 float* sigma, float* seg, void* workspace, int64_t workspace_bytes, nfe_stream_t stream)
{
    (void)workspace; (void)workspace_bytes;
    NFE_REQUIRE(cfg, "nfe_run_model_fwd: null cfg");
    if (int rc = check_decoder_dims(cfg->kind, net_a, net_b, "nfe_run_model_fwd")) return rc;
    if ((int64_t)n * m == 0) return 0;
    const bool sigma_only = cfg->sigma_only != 0;
    FieldArgs a = {};
    if (int rc = field_planes(cfg, planes_norm_cl, planes_denorm_cl, plane_batch, n, m, sigma_only, false, "nfe_run_model_fwd", a)) return rc;
    NFE_REQUIRE(coords && sigma && (rgb || sigma_only), "nfe_run_model_fwd: null pointer");
    NFE_REQUIRE(cfg->kind == NFE_DEC_OSG || seg || sigma_only, "nfe_run_model_fwd: seg output missing");
    a.coords = coords; a.m = m; a.total = (int64_t)n * m; a.s_per_ray = 1;
    a.sigma = sigma; a.rgb = rgb; a.seg = seg;
    a.density_noise = cfg->density_noise; a.seed = cfg->seed; a.offset = cfg->offset;
    StageScope t(STAGE_RUN_MODEL, as_stream(stream));
    return launch_field(cfg->kind, cfg->precision, a, net_a, net_b, as_stream(stream));
}

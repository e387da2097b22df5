// Field kernel of the tensor-core precisions (bf16x3, bf16): fused gather + decode, warp-specialised so that every SM
// sub-partition always has independent instruction streams to choose from (VERDICT r01 "next" #2).
//
// What round 1's kernel (4 epilogue warps, tap pre-pass inside the gather warps; since removed) was bound by
// (profiles/ncu_r01_final_field_pipe_and_march.txt, profiles/l2_gather_r02.txt):
//   * ONE epilogue warp per sub-partition ran a ~1500-instruction dependent chain per tile (softplus on the SFU, bf16 hi/lo
//     split, TMEM traffic) at an IPC of 0.2 — 46 % of its stall samples were fixed-latency waits, nothing to overlap them with;
//   * the 8 gather warps spent 30 % of their instructions in the tap pre-pass (position -> 12 offsets + 12 weights), run with
//     half-empty warps and two 64-bit divisions per sample, its dependent global loads at the head of their stall list;
//   * the L2 itself was never the limit: LDG.128 gathers of this shape reach 17-20 TB/s on this part, the kernel pulled 5.4.
//
// One persistent CTA per SM, 20 warps (5 per sub-partition):
//
//   warps  0-3   epilogue group 0: tiles 0, 2, 4, ... of this CTA         thread m owns TMEM lane m = sample m of the tile
//   warps  4-7   epilogue group 1: tiles 1, 3, 5, ...                      (two whole, independent epilogues interleave on every
//                                                                          sub-partition instead of one epilogue split by columns)
//   warp   8     MMA issuer (one elected thread)
//   warps  9-11  tap producers: position -> texel offsets + bilinear weights, one sample per lane; the four 32-sample chunks of a
//                tile are dealt over the three warps, up to two tiles ahead of the gather (3 tap buffers)
//   warps 12-19  gather: 8 lanes per sample, LDG.128 per tap, rolling one-pass-ahead texel pipeline, bf16 hi/lo feature tile
//
// Tensor memory: each epilogue group owns one accumulator set of 192 columns: D1A 64 | D1B 64 | D2 <= 64.  The hidden
// activations are written back IN PLACE over the layer-1 accumulators they were computed from (16 fp32 columns in, 8 columns
// of bf16 hi pairs + 8 of lo pairs out), from where the layer-2 MMAs take them as their A operand — no separate hidden
// region, no shared-memory round trip.  Layer 1 of tile i+2 is issued as soon as layer 2 of tile i has consumed that region
// (its own commit), i.e. while group g is still writing tile i's outputs, so an epilogue group never waits for a layer 1.
#include <type_traits>

#include "nfe_field_launch.cuh"
#include "nfe_mlp_tc.cuh"

namespace nfe {

using namespace tcmlp;

namespace p2 {

constexpr int EPI_GROUPS = 2;
constexpr int MMA_WARP = 8;
constexpr int TAP_WARP0 = 9, TAP_WARPS = 3;                 // warps 9 .. 9 + TAP_WARPS - 1 (at most 3: warp 12 is the first gather warp)
static_assert(TAP_WARPS >= 1 && TAP_WARPS <= 3, "tap warps are warps 9-11");
constexpr int GATHER_WARP0 = 12, GATHER_WARPS = 8;
constexpr int THREADS = (GATHER_WARP0 + GATHER_WARPS) * 32;
constexpr int PASSES_PER_TILE = TILE_M / 4;                 // a pass = 4 samples (8 lanes each)
// consecutive passes of a tile each gather warp owns: the first LONG_WARPS warps take PER_LONG, the others PER_LONG - 1
// (8 warps: 4 each)
constexpr int PER_LONG = (PASSES_PER_TILE + GATHER_WARPS - 1) / GATHER_WARPS;
constexpr int LONG_WARPS = PASSES_PER_TILE - (PER_LONG - 1) * GATHER_WARPS;
static_assert(LONG_WARPS >= 1 && LONG_WARPS <= GATHER_WARPS && PER_LONG >= 2, "bad gather split");
constexpr int TAP_BUFS = 3;                                 // tap buffers: the tap warps run up to TAP_BUFS - 1 tiles ahead of the gather
constexpr int GROUP_COLS = 192;                             // D1A 64 | D1B 64 | D2A | D2B (<= 64 together)
constexpr int P2_TMEM_COLS = 512;
constexpr int COL_D2 = 128;
constexpr int REC_STAGE_STRIDE = 208;                       // bytes per staged record row: conflict-free 16-byte stores

// Register re-deal (setmaxnreg works on groups of four warps).  At launch every thread has what 640 threads allow (96).
// Only registers a warp group RELEASES can be claimed by another (asking for more blocks forever), hence the static_asserts.
// Measured at c2 (ms per launch, profiles/pipe2_variants_r02.txt): uniform 96: 0.355; epilogue/gather/misc = 104/104/64: 0.331
// (the default); 96/112/56: 0.347; 104/112/48 and 112/104/48: 0.340-0.342 (at 48 the MMA-issuing thread spills and paces
// everything); 12 gather warps at 80-88 registers: 0.445-0.57 (spills in the gather loop).
constexpr int REGS_LAUNCH = 65536 / THREADS / 8 * 8;        // 96
constexpr int REGS_EPI = 104, REGS_MISC = 64, REGS_GATHER = 104;
static_assert(REGS_EPI > REGS_LAUNCH && REGS_GATHER > REGS_LAUNCH && REGS_MISC < REGS_LAUNCH,
              "the epilogue and gather groups only grow, the MMA / tap group only shrinks");
static_assert(8 * (REGS_EPI - REGS_LAUNCH) + GATHER_WARPS * (REGS_GATHER - REGS_LAUNCH) <= 4 * (REGS_LAUNCH - REGS_MISC),
              "setmaxnreg.inc would wait forever");
static_assert((2 * REGS_EPI + REGS_MISC + (GATHER_WARPS / 4) * REGS_GATHER) * 32 <= 16384, "register file of a sub-partition");

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

template <int KIND, bool SPLIT>
struct Smem {
    using T = TcTraits<KIND>;
    static constexpr int PARTS = SPLIT ? 2 : 1;
    static constexpr int NETS = T::HAS_B ? 2 : 1;
    alignas(128) unsigned char a1[2][T::SETS][PARTS][A1_BYTES];          // feature ring: slot = tile parity = epilogue group
    alignas(128) unsigned char b1[NETS][PARTS][B1_BYTES];
    alignas(128) unsigned char b2a[PARTS][(T::N_A / 8) * B2_SBO];
    alignas(128) unsigned char b2b[PARTS][(T::N_B / 8) * B2_SBO];
    // per sample: 12 texel offsets (float4 units), 12 weights, batch item
    alignas(16) uint4 taps[TAP_BUFS][TILE_M][7];
    // single-gather identity: scale / shift rows (96 floats each) of the batch item the tile starts in and of the next one,
    // copied per tile by the tap warp; the gather reads them with LDS instead of 6 global loads per pass whose lines the texel
    // stream keeps evicting from the (24 KB) L1 — they were 40 % of the gather warps' stall samples
    alignas(16) float aff[TAP_BUFS][2][2][96];          // [buffer][item - first item][scale | shift][channel]
    int aff_item[TAP_BUFS];
    alignas(16) unsigned char recbuf[EPI_GROUPS][TILE_M][REC_STAGE_STRIDE];   // record staging (each warp owns its 32 rows)
    // layer-1 bias, pre-multiplied by log2(e).  Adding it through the tensor core instead (one more K step against a block of ones)
    // measured neutral (profiles/pipe2_variants_r02.txt `bm*`): the gather warps pace the kernel, not the epilogue.
    float bias1[NETS][HIDDEN];
    float bias2a[T::N_A];
    float bias2b[T::N_B];
    alignas(8) uint64_t full[2], empty[2];                                // feature ring
    uint64_t taps_full[TAP_BUFS], taps_empty[TAP_BUFS];
    uint64_t d1_full[2], a2a_full[2], a2b_full[2], d2a_full[2], d2b_full[2], d2_free[2];   // per epilogue group
    uint32_t tmem_base;
};

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
                 :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}

template <int KIND, bool SPLIT>
__device__ void load_params(Smem<KIND, SPLIT>& s, const nfe_mlp& net_a, const nfe_mlp& net_b)
{
    using T = TcTraits<KIND>;
    constexpr int PARTS = SPLIT ? 2 : 1;
    load_weights<PARTS>(s.b1[0][0], B1_BYTES, net_a.w1, net_a.wgain1, HIDDEN, HIDDEN, FEAT, B1_LBO, B1_SBO);
    // softplus runs in base 2 (see hidden_in_place): ln 2 goes into the layer-2 weights, log2(e) into the layer-1 bias
    load_weights<PARTS>(s.b2a[0], sizeof(s.b2a[0]), net_a.w2, net_a.wgain2 * LN2, T::OUT_A, T::N_A, HIDDEN, B2_LBO, B2_SBO);
    for (int i = threadIdx.x; i < HIDDEN; i += blockDim.x) s.bias1[0][i] = folded_bias(net_a.b1, net_a.bgain1, i) * LOG2E;
    for (int i = threadIdx.x; i < T::N_A; i += blockDim.x) s.bias2a[i] = i < T::OUT_A ? folded_bias(net_a.b2, net_a.bgain2, i) : 0.0f;
    if constexpr (T::HAS_B) {
        load_weights<PARTS>(s.b1[1][0], B1_BYTES, net_b.w1, net_b.wgain1, HIDDEN, HIDDEN, FEAT, B1_LBO, B1_SBO);
        load_weights<PARTS>(s.b2b[0], sizeof(s.b2b[0]), net_b.w2, net_b.wgain2 * LN2, T::OUT_B, T::N_B, HIDDEN, B2_LBO, B2_SBO);
        for (int i = threadIdx.x; i < HIDDEN; i += blockDim.x) s.bias1[1][i] = folded_bias(net_b.b1, net_b.bgain1, i) * LOG2E;
        for (int i = threadIdx.x; i < T::N_B; i += blockDim.x) s.bias2b[i] = i < T::OUT_B ? folded_bias(net_b.b2, net_b.bgain2, i) : 0.0f;
    }
}

// sigmoid(x) * 1.002 - 0.001 (triplane.py:188,219,269) for two colours at once
__device__ __forceinline__ float2 rgb_activation2(float2 x)
{
    const float2 n = fmul2(x, make_float2(-LOG2E, -LOG2E));
    float e0, e1, r0, r1;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(n.x));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(n.y));
    const float2 d = fadd2(make_float2(e0, e1), make_float2(1.0f, 1.0f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(d.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(d.y));
    return ffma2(make_float2(r0, r1), make_float2(1.002f, 1.002f), make_float2(-0.001f, -0.001f));
}

// hidden = softplus(D1 + b1) for this thread's row, written back over the accumulator columns it came from: the 16 fp32
// columns [16q, 16q+16) become 8 columns of packed bf16 hi parts at 16q and 8 columns of lo parts at 16q+8.
// Softplus in base-2 units: with t = x*log2(e), softplus(x) = ln2 * (max(t,0) + log2(1 + 2^-|t|)).
template <bool SPLIT>
__device__ __forceinline__ void hidden_in_place(uint32_t taddr, const float* bias1_log2)
{
    const float2 k2 = make_float2(LOG2E, LOG2E), one2 = make_float2(1.0f, 1.0f), neg2 = make_float2(-1.0f, -1.0f);
    // one copy of the 16-column body: smallest code, and the kernel is instruction-cache sensitive
#pragma unroll 1
    for (int q = 0; q < HIDDEN / 16; ++q) {
        float v[16];
        tc::tmem_ld16(taddr + q * 16, v);
        tc::tmem_ld_wait();
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias1_log2 + q * 16 + 4 * i);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float2 t = ffma2(make_float2(v[4 * i + 2 * j], v[4 * i + 2 * j + 1]), k2, j ? make_float2(b4.z, b4.w) : make_float2(b4.x, b4.y));
                float e0, e1, l0, l1;
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-fabsf(t.x)));
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-fabsf(t.y)));
                const float2 s1 = fadd2(make_float2(e0, e1), one2);
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(s1.x));
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(s1.y));
                const float2 hh = fadd2(make_float2(fmaxf(t.x, 0.0f), fmaxf(t.y, 0.0f)), make_float2(l0, l1));
                const __nv_bfloat162 p = __floats2bfloat162_rn(hh.x, hh.y);
                hi[2 * i + j] = *reinterpret_cast<const uint32_t*>(&p);
                if (SPLIT) {
                    const float2 d = ffma2(__bfloat1622float2(p), neg2, hh);      // h - bf16(h), exact
                    const __nv_bfloat162 r = __floats2bfloat162_rn(d.x, d.y);
                    lo[2 * i + j] = *reinterpret_cast<const uint32_t*>(&r);
                }
            }
        }
        tmem_st8(taddr + q * 16, hi);
        if (SPLIT) tmem_st8(taddr + q * 16 + 8, lo);
    }
    tc::tmem_st_wait();
}

// D (+)= H * W2^T with H taken from tensor memory in the in-place layout of hidden_in_place; every lane of the MMA warp calls it, the
// elected one issues
template <bool SPLIT>
__device__ __forceinline__ void issue_layer2(bool leader, uint32_t tmem_d, uint32_t tmem_h, const unsigned char* b_hi, const unsigned char* b_lo, uint32_t idesc)
{
    uint32_t acc = 0;
    const uint64_t db0 = tc::make_desc(0, B2_LBO, B2_SBO);
    const uint32_t bh = tc::smem_u32(b_hi) >> 4, bl = tc::smem_u32(b_lo) >> 4;
    constexpr int TERMS = SPLIT ? 3 : 1;
#pragma unroll
    for (int t = 0; t < TERMS; ++t) {
        const uint32_t part = (t == 1) ? 8u : 0u;                        // hi*hi, lo*hi, hi*lo
        const uint32_t b = (t == 2) ? bl : bh;
#pragma unroll
        for (int ks = 0; ks < HIDDEN / 16; ++ks) {
            if (leader) tc::mma_bf16_ts(tmem_d, tmem_h + ks * 16 + part, db0 + (b + ks * ((2 * B2_LBO) >> 4)), idesc, acc);
            acc = 1;
        }
    }
}

struct SampleRef { int64_t idx; int item; int64_t ray; };

// Tile row -> sample: sample L is index L, in batch item L / m, on ray L / s_per_ray
__device__ __forceinline__ SampleRef sample_of(const FieldArgs& a, int64_t L, bool small)
{
    SampleRef r;
    r.idx = L;
    if (small) {                    // everything fits 31 bits: 32-bit divisions (the 64-bit ones are subroutine calls)
        r.item = (int)((uint32_t)L / (uint32_t)a.m);
        r.ray = (int64_t)((uint32_t)L / (uint32_t)a.s_per_ray);
    } else {
        r.item = (int)(L / a.m);
        r.ray = L / a.s_per_ray;
    }
    return r;
}

// texel load at lane_base + 16*off4 (one IMAD.WIDE + LDG); `streaming` taps (planes 1 and 2: no reuse between the samples a
// warp walks) bypass L1 allocation, plane 0 keeps the read-only path where consecutive samples of a ray share texels
__device__ __forceinline__ float4 ldg_tap(const float4* lane_base, uint32_t off4, bool streaming)
{
    uint64_t addr;
    asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(addr) : "r"(off4), "l"(lane_base));
    if (streaming) return __ldcg(reinterpret_cast<const float4*>(addr));
    return __ldg(reinterpret_cast<const float4*>(addr));
}

#ifdef NFE_PIPE_PROFILE
// Debug build only: cycles each role spends blocked on each barrier (slot k) and in total (slot 15), summed over warps and CTAs.
__device__ unsigned long long g_p2_prof[4][16];
#define P2_WAIT(slot, bar, par) do { const long long t0_ = clock64(); tc::mbar_wait(bar, par); prof_[slot] += clock64() - t0_; } while (0)
#else
#define P2_WAIT(slot, bar, par) tc::mbar_wait(bar, par)
#endif

template <int REGS>
__device__ __forceinline__ void regs_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(REGS)); }
template <int REGS>
__device__ __forceinline__ void regs_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" :: "n"(REGS)); }

// GEO: the geometry-only render pass (FieldArgs::geometry_only): 16-float records {sigma, seg[15]} and no colour work — the
// disentangled decoder runs geo_net on the normalised planes alone (the skip_b path of sigma_only, logits kept), the
// segmentation decoder keeps net's sigma column and seg_net.  A separate instantiation: the full kernels keep their code.
template <int KIND, bool SPLIT, bool GEO>
__global__ void __launch_bounds__(THREADS, 1) field_pipe2_kernel(FieldArgs a, nfe_mlp net_a, nfe_mlp net_b)
{
    using T = TcTraits<KIND>;
    constexpr int P = SPLIT ? 1 : 0;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // (no integer round-up of the base here: it would strip the shared address space and turn every LDS/STS below into a generic
    // LD/ST; the dynamic window starts 1024-byte aligned because the kernel has no static shared memory)
    Smem<KIND, SPLIT>& s = *reinterpret_cast<Smem<KIND, SPLIT>*>(smem_raw);
    // the shuffle tells the compiler the role index is warp-uniform (uniform branches / registers inside the roles)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    // ---- setup
    if (warp == MMA_WARP) tc::tmem_alloc(&s.tmem_base, P2_TMEM_COLS);
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            tc::mbar_init(&s.full[i], GATHER_WARPS);
            tc::mbar_init(&s.empty[i], 1);
            tc::mbar_init(&s.d1_full[i], 1);
            tc::mbar_init(&s.a2a_full[i], 4);
            tc::mbar_init(&s.a2b_full[i], 4);
            tc::mbar_init(&s.d2a_full[i], 1);
            tc::mbar_init(&s.d2b_full[i], 1);
            tc::mbar_init(&s.d2_free[i], 4);
        }
        for (int i = 0; i < TAP_BUFS; ++i) {
            tc::mbar_init(&s.taps_full[i], TAP_WARPS);
            tc::mbar_init(&s.taps_empty[i], GATHER_WARPS);
        }
        tc::mbar_fence_init();
    }
    load_params(s, net_a, net_b);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = s.tmem_base;
    const int64_t n_tiles = (a.total + TILE_M - 1) / TILE_M;
    const int64_t G = gridDim.x;
    // tiles of this CTA: blockIdx.x + it*G, it = 0 .. n_my-1; epilogue group it & 1, feature-ring slot it & 1, tap buffer it % 3
    const int n_my = (int)((n_tiles - blockIdx.x + G - 1) / G);
    // sigma_only with the disentangled decoder: sigma is output 0 of geo_net on the normalised planes, so the
    // de-normalised gather and the whole appearance net are skipped
    const bool skip_b = (GEO || a.sigma_only) && KIND == NFE_DEC_DISENTANGLED;
    const bool has_b = T::HAS_B && !skip_b;
#ifdef NFE_PIPE_PROFILE
    long long prof_[16] = {};
    const long long prof_t0_ = clock64();
#endif

    if (warp >= GATHER_WARP0) {
        // ================================================================ gather warps (producers of the feature tile)
        const int gw = warp - GATHER_WARP0;
        const int g = lane >> 3, c4 = lane & 7;
        const float4* set_a = reinterpret_cast<const float4*>(a.set_norm) + c4;
        const float4* set_b = reinterpret_cast<const float4*>(a.set_denorm) + c4;
        // one plane set is read per pass in the single-gather, density-only and one-set decoders: those run the
        // rolling pipeline below; the two-set gather (24 texels per sample) has no registers left for it
        const bool affine = T::SETS == 2 && a.affine_scale != nullptr;
        const bool rolling = T::SETS == 1 || affine || skip_b;
        const float4* set_r = T::SETS == 2 ? set_a : set_b;
        const int n_pass = gw < LONG_WARPS ? PER_LONG : PER_LONG - 1;
        const int pass0 = gw < LONG_WARPS ? gw * PER_LONG : LONG_WARPS * PER_LONG + (gw - LONG_WARPS) * (PER_LONG - 1);
        const int row0 = 4 * pass0 + g;                     // this lane group's row in its first pass of a tile; pass p: + 4p
        regs_inc<REGS_GATHER>();

        float4 va[12];                    // rolling pipeline: the texels of the NEXT pass, in flight while this one is blended
        if (n_my > 0) {
            P2_WAIT(0, &s.taps_full[0], 0);
            if (rolling) {
                const uint4* src = s.taps[0][row0];
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const uint4 o4 = src[q];
                    va[4 * q] = ldg_tap(set_r, o4.x, q != 0); va[4 * q + 1] = ldg_tap(set_r, o4.y, q != 0);
                    va[4 * q + 2] = ldg_tap(set_r, o4.z, q != 0); va[4 * q + 3] = ldg_tap(set_r, o4.w, q != 0);
                }
            }
        }
        int tb = 0, tb_next = 1;          // tap buffer of this tile / the next one
        for (int it = 0; it < n_my; ++it) {
            const int st = it & 1;
            const bool has_next = it + 1 < n_my;
            P2_WAIT(1, &s.empty[st], ((it >> 1) & 1) ^ 1);      // slot released by the layer-1 commit two tiles ago
            if (rolling) {
                // the body is instantiated for the two pass counts a warp can own; the pass loop stays rolled: unrolling it
                // trades loop bookkeeping for instruction-cache misses, which measured slower
                auto tile_body = [&](auto np_tag) {
                    constexpr int NP = decltype(np_tag)::value;
                    const uint4* tap_row = s.taps[tb][row0];
#pragma unroll 1
                    for (int p = 0; p < NP; ++p) {
                        const int row = row0 + 4 * p;
                        const uint4* cur = tap_row + 4 * p * 7;
                        const bool more = p + 1 < NP;
                        const bool fetch = more || has_next;
                        if (!more && has_next) P2_WAIT(0, &s.taps_full[tb_next], ((it + 1) / TAP_BUFS) & 1);
                        const uint4* nxt = more ? cur + 4 * 7 : s.taps[tb_next][row0];
                        float2 f01[3], f23[3];
#pragma unroll
                        for (int pl = 0; pl < 3; ++pl) {
                            const float4 w4 = *reinterpret_cast<const float4*>(&cur[3 + pl]);
                            const float2 w0 = make_float2(w4.x, w4.x), w1 = make_float2(w4.y, w4.y), w2 = make_float2(w4.z, w4.z), w3 = make_float2(w4.w, w4.w);
                            float2 a01 = fmul2(make_float2(va[4 * pl].x, va[4 * pl].y), w0), a23 = fmul2(make_float2(va[4 * pl].z, va[4 * pl].w), w0);
                            a01 = ffma2(make_float2(va[4 * pl + 1].x, va[4 * pl + 1].y), w1, a01); a23 = ffma2(make_float2(va[4 * pl + 1].z, va[4 * pl + 1].w), w1, a23);
                            a01 = ffma2(make_float2(va[4 * pl + 2].x, va[4 * pl + 2].y), w2, a01); a23 = ffma2(make_float2(va[4 * pl + 2].z, va[4 * pl + 2].w), w2, a23);
                            a01 = ffma2(make_float2(va[4 * pl + 3].x, va[4 * pl + 3].y), w3, a01); a23 = ffma2(make_float2(va[4 * pl + 3].z, va[4 * pl + 3].w), w3, a23);
                            f01[pl] = a01; f23[pl] = a23;
                            if (fetch) {             // refill the four registers just consumed with the next pass's texels
                                const uint4 o4 = nxt[pl];
                                va[4 * pl] = ldg_tap(set_r, o4.x, pl != 0); va[4 * pl + 1] = ldg_tap(set_r, o4.y, pl != 0);
                                va[4 * pl + 2] = ldg_tap(set_r, o4.z, pl != 0); va[4 * pl + 3] = ldg_tap(set_r, o4.w, pl != 0);
                            }
                        }
                        const float2 third2 = make_float2(1.0f / 3.0f, 1.0f / 3.0f);
                        const float2 fa01 = fmul2(fadd2(fadd2(f01[0], f01[1]), f01[2]), third2), fa23 = fmul2(fadd2(fadd2(f23[0], f23[1]), f23[2]), third2);
                        store_features4<SPLIT>(s.a1[st][0], row, 4 * c4, make_float4(fa01.x, fa01.y, fa23.x, fa23.y));
                        if (affine && !skip_b) {
                            // single-gather identity: only the normalised planes are read; the de-normalised features are
                            // s*f_p + m*w_in per plane, statistics from the tile's table in shared memory (the launcher only
                            // enables the identity when an item has at least TILE_M samples, so a tile touches at most two items)
                            const uint4 meta = cur[6];                       // item, w_in of the three planes
                            const float wi[3] = {__uint_as_float(meta.y), __uint_as_float(meta.z), __uint_as_float(meta.w)};
                            const uint32_t rel = a.affine_items == 1 ? 0u : ((uint32_t)((int)meta.x - s.aff_item[tb]) & 1u);
                            const float4* ssc = reinterpret_cast<const float4*>(s.aff[tb][rel][0]) + c4;
                            const float4* ssh = reinterpret_cast<const float4*>(s.aff[tb][rel][1]) + c4;
                            float2 d01[3], d23[3];
#pragma unroll
                            for (int pl = 0; pl < 3; ++pl) {
                                const float4 scl = ssc[pl * 8], shf = ssh[pl * 8];
                                const float2 w2_ = make_float2(wi[pl], wi[pl]);
                                d01[pl] = ffma2(make_float2(scl.x, scl.y), f01[pl], fmul2(make_float2(shf.x, shf.y), w2_));
                                d23[pl] = ffma2(make_float2(scl.z, scl.w), f23[pl], fmul2(make_float2(shf.z, shf.w), w2_));
                            }
                            const float2 fb01 = fmul2(fadd2(fadd2(d01[0], d01[1]), d01[2]), third2), fb23 = fmul2(fadd2(fadd2(d23[0], d23[1]), d23[2]), third2);
                            store_features4<SPLIT>(s.a1[st][T::SETS - 1], row, 4 * c4, make_float4(fb01.x, fb01.y, fb23.x, fb23.y));
                        }
                    }
                };
                if (n_pass == PER_LONG) tile_body(std::integral_constant<int, PER_LONG>{});
                else tile_body(std::integral_constant<int, PER_LONG - 1>{});
            } else {
                if (it > 0) P2_WAIT(0, &s.taps_full[tb], (it / TAP_BUFS) & 1);
#pragma unroll 1
                for (int p = 0; p < n_pass; ++p) {
                    const int row = row0 + 4 * p;
                    TapSet ts;
                    const uint4* src = s.taps[tb][row];
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const uint4 o4 = src[q];
                        ts.off4[4 * q] = (int)o4.x; ts.off4[4 * q + 1] = (int)o4.y; ts.off4[4 * q + 2] = (int)o4.z; ts.off4[4 * q + 3] = (int)o4.w;
                        const uint4 w4 = src[3 + q];
                        ts.w[4 * q] = __uint_as_float(w4.x); ts.w[4 * q + 1] = __uint_as_float(w4.y);
                        ts.w[4 * q + 2] = __uint_as_float(w4.z); ts.w[4 * q + 3] = __uint_as_float(w4.w);
                    }
                    // all 24 texel loads of the sample (two plane sets) are issued before the first blend
                    float4 vb[12];
#pragma unroll
                    for (int i = 0; i < 12; ++i) va[i] = ldg_tap(set_a, (uint32_t)ts.off4[i], false);
#pragma unroll
                    for (int i = 0; i < 12; ++i) vb[i] = ldg_tap(set_b, (uint32_t)ts.off4[i], false);
                    store_features4<SPLIT>(s.a1[st][0], row, 4 * c4, gather_reduce(va, ts));
                    store_features4<SPLIT>(s.a1[st][T::SETS - 1], row, 4 * c4, gather_reduce(vb, ts));
                }
            }
            tc::fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                tc::mbar_arrive(&s.full[st]);
                tc::mbar_arrive(&s.taps_empty[tb]);
            }
            tb = tb_next;
            tb_next = tb_next + 1 == TAP_BUFS ? 0 : tb_next + 1;
        }
    } else if (warp >= TAP_WARP0 && warp < TAP_WARP0 + TAP_WARPS) {
        // ================================================================ tap producers
        // ONE lane per sample turns its position into 12 clamped texel offsets + 12 weights (zero for taps that fall
        // outside: padding_mode='zeros') and parks them in shared memory for the 8 gather lanes of that sample.
        const int tw = warp - TAP_WARP0;
        regs_dec<REGS_MISC>();
        const int64_t set_stride4 = (int64_t)3 * a.H * a.W * (FEAT / 4);     // float4 units
        const bool small = a.total < (1ll << 31);
        // row-wise deal: every tap warp works on every tile — the four 32-sample chunks of a tile go to warps 0 .. TAP_WARPS-1, the
        // remaining ones rotate with the tile — so a tile's taps are ready after at most two rounds, not four (the gather asks for
        // them two tiles after it released the buffer: what counts is the latency of one tile's taps, not only the throughput)
        // The inputs of a chunk (depth + ray, or the point) are fetched one chunk ahead: the loads of the warp's NEXT chunk — which
        // may belong to the next tile; they touch no tap buffer, so they need no barrier — are in flight while this chunk's taps
        // are computed, instead of heading a dependent chain of ~1000 cycles per chunk.
        struct Raw { float t, o[3], d[3]; int item; bool live; };
        auto owner_of = [&](int it, int h) { return h < TAP_WARPS ? h : (it + h) % TAP_WARPS; };
        auto advance = [&](int& it, int& h) {                      // next chunk this warp owns (it == n_my: none left)
            for (;;) {
                if (++h == TILE_M / 32) { h = 0; if (++it >= n_my) return; }
                if (owner_of(it, h) == tw) return;
            }
        };
        auto fetch = [&](int it, int h) {
            Raw r;
            r.t = 0.0f; r.item = 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) r.o[k] = r.d[k] = 0.0f;
            const int64_t L = ((int64_t)blockIdx.x + (int64_t)it * G) * TILE_M + h * 32 + lane;
            r.live = it < n_my && L < a.total;
            if (r.live) {
                const SampleRef sr = sample_of(a, L, small);
                r.item = sr.item;
                if (a.coords) {
                    const float* c = a.coords + sr.idx * 3;
                    r.o[0] = __ldg(c); r.o[1] = __ldg(c + 1); r.o[2] = __ldg(c + 2);
                } else {
                    r.t = __ldg(a.depths + sr.idx);
                    const float* o = a.origins + sr.ray * 3;
                    const float* d = a.dirs + sr.ray * 3;
#pragma unroll
                    for (int k = 0; k < 3; ++k) { r.o[k] = __ldg(o + k); r.d[k] = __ldg(d + k); }
                }
            }
            return r;
        };
        // one loop body, run once more than there are chunks: iteration k fetches chunk k and turns chunk k-1 into taps
        int it = 0, h = -1;
        if (n_my > 0) advance(it, h);
        Raw cur;
        cur.live = false;
        int cit = -1, ch = 0;
#pragma unroll 1
        for (;;) {
            const Raw nxt = fetch(it, h);                          // it == n_my: nothing to fetch, live = false
            if (cit < 0) {
                if (it >= n_my) break;
                cur = nxt; cit = it; ch = h;
                advance(it, h);
                continue;
            }
            const int tb = cit % TAP_BUFS;
            const bool first = ch == tw;                               // chunk h = tw is the first one a warp owns in every tile
            if (first) {
                if (cit >= TAP_BUFS) P2_WAIT(2, &s.taps_empty[tb], ((cit / TAP_BUFS) - 1) & 1);
                if (tw == 0 && T::SETS == 2 && a.affine_scale != nullptr) {
                    const int64_t base = ((int64_t)blockIdx.x + (int64_t)cit * G) * TILE_M;
                    const int item0 = a.affine_items == 1 ? 0 : (int)(small ? (uint32_t)base / (uint32_t)a.m : base / a.m);
                    if (lane == 0) s.aff_item[tb] = item0;
                    for (int i = lane; i < 2 * 2 * 24; i += 32) {           // 2 items x {scale, shift} x 24 float4
                        const int rel = i / 48, which = (i / 24) & 1, c = i % 24;
                        const int item = min(item0 + rel, a.affine_items - 1);
                        const float* src = (which ? a.affine_shift : a.affine_scale) + (int64_t)item * 96;
                        reinterpret_cast<float4*>(s.aff[tb][rel][which])[c] = __ldg(reinterpret_cast<const float4*>(src) + c);
                    }
                }
            }
            {
                const int row = ch * 32 + lane;
                TapSet ts;
#pragma unroll
                for (int i = 0; i < 12; ++i) { ts.off4[i] = 0; ts.w[i] = 0.0f; }
                if (cur.live) {
                    float x, y, z;
                    if (a.coords) { x = cur.o[0]; y = cur.o[1]; z = cur.o[2]; }
                    else { x = ray_point(cur.o[0], cur.t, cur.d[0]); y = ray_point(cur.o[1], cur.t, cur.d[1]); z = ray_point(cur.o[2], cur.t, cur.d[2]); }
                    ts = make_tapset(taps3(__fmul_rn(a.scale, x), __fmul_rn(a.scale, y), __fmul_rn(a.scale, z), a.H, a.W), a.H, a.W);
                    const int item_off = a.plane_batch == 1 ? 0 : (int)(cur.item * set_stride4);
#pragma unroll
                    for (int i = 0; i < 12; ++i) ts.off4[i] += item_off;
                }
                uint4* dst = s.taps[tb][row];
                // batch item and, per plane, the sum of the in-bounds tap weights (what the single-gather identity multiplies the
                // shift by; summed in the order the gather warps used to, so results are bit-identical)
                dst[6] = make_uint4((uint32_t)cur.item, __float_as_uint(((ts.w[0] + ts.w[1]) + ts.w[2]) + ts.w[3]),
                                    __float_as_uint(((ts.w[4] + ts.w[5]) + ts.w[6]) + ts.w[7]), __float_as_uint(((ts.w[8] + ts.w[9]) + ts.w[10]) + ts.w[11]));
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    dst[q] = make_uint4((uint32_t)ts.off4[4 * q], (uint32_t)ts.off4[4 * q + 1], (uint32_t)ts.off4[4 * q + 2], (uint32_t)ts.off4[4 * q + 3]);
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    dst[3 + q] = make_uint4(__float_as_uint(ts.w[4 * q]), __float_as_uint(ts.w[4 * q + 1]), __float_as_uint(ts.w[4 * q + 2]), __float_as_uint(ts.w[4 * q + 3]));
            }
            if (it != cit) {                                       // that was the warp's last chunk of tile cit
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&s.taps_full[tb]);
            }
            if (it >= n_my) break;
            cur = nxt; cit = it; ch = h;
            advance(it, h);
        }
    } else if (warp == MMA_WARP) {
        // ================================================================ MMA issuer: every lane runs the (warp-uniform) loop, one
        // elected lane issues — see tc::elect_one
        regs_dec<REGS_MISC>();
        {
            const bool leader = tc::elect_one();
            constexpr uint32_t idesc1 = tc::make_idesc_bf16(TILE_M, HIDDEN);
            // geometry: net A's layer 2 only for its first 16 columns (sigma and, for the disentangled decoder, the logits; the
            // segmentation decoder's 32 colour columns are not computed)
            constexpr uint32_t idesc2a = tc::make_idesc_bf16(TILE_M, GEO ? 16 : T::N_A);
            constexpr uint32_t idesc2b = tc::make_idesc_bf16(TILE_M, T::N_B);
            // layer 1 of tile `it` into the accumulator set of its group (= ring slot = it & 1)
            auto layer1 = [&](int it) {
                const int st = it & 1;
                const uint32_t tb = tmem + st * GROUP_COLS;
                P2_WAIT(3, &s.full[st], (it >> 1) & 1);          // features landed
                tc::fence_after_sync();
                issue_gemm<SPLIT>(leader, tb + COL_D1A, s.a1[st][0][0], s.a1[st][0][P], A1_LBO, A1_SBO, s.b1[0][0], s.b1[0][P], B1_LBO, B1_SBO, FEAT, idesc1);
                if (has_b)
                    issue_gemm<SPLIT>(leader, tb + COL_D1B, s.a1[st][T::SETS - 1][0], s.a1[st][T::SETS - 1][P], A1_LBO, A1_SBO, s.b1[T::HAS_B ? 1 : 0][0],
                                      s.b1[T::HAS_B ? 1 : 0][P], B1_LBO, B1_SBO, FEAT, idesc1);
                if (leader) {
                    tc::mma_commit(&s.empty[st]);                   // ring slot reusable once these MMAs have read it
                    tc::mma_commit(&s.d1_full[st]);
                }
            };
            if (n_my > 0) layer1(0);
            if (n_my > 1) layer1(1);
            for (int it = 0; it < n_my; ++it) {
                const int gi = it & 1;
                const uint32_t ph = (it >> 1) & 1;
                const uint32_t tb = tmem + gi * GROUP_COLS;
                // layer 2, net A: hidden tile written in place, D2 region released by the group's previous tile
                P2_WAIT(4, &s.a2a_full[gi], ph);
                if (it >= 2) P2_WAIT(5, &s.d2_free[gi], ph ^ 1);
                tc::fence_after_sync();
                issue_layer2<SPLIT>(leader, tb + COL_D2, tb + COL_D1A, s.b2a[0], s.b2a[P], idesc2a);
                if (leader) tc::mma_commit(&s.d2a_full[gi]);
                if (has_b) {
                    P2_WAIT(6, &s.a2b_full[gi], ph);
                    tc::fence_after_sync();
                    issue_layer2<SPLIT>(leader, tb + COL_D2 + T::N_A, tb + COL_D1B, s.b2b[0], s.b2b[P], idesc2b);
                    if (leader) tc::mma_commit(&s.d2b_full[gi]);
                }
                // layer 1 of the group's NEXT tile goes in as soon as layer 2 has consumed the hidden tile (our own commit),
                // i.e. while the group is still writing this tile's outputs
                if (it + 2 < n_my) {
                    P2_WAIT(7, has_b ? &s.d2b_full[gi] : &s.d2a_full[gi], ph);
                    layer1(it + 2);
                }
            }
        }
        __syncwarp();
    } else if (warp < MMA_WARP) {
        // ================================================================ epilogue groups (TMEM lanes 32*(warp&3) ..)
        const int gi = warp >> 2, wq = warp & 3;
        regs_inc<REGS_EPI>();
        const int row = wq * 32 + lane;
        const uint32_t lane_addr = tmem + gi * GROUP_COLS + ((uint32_t)(wq * 32) << 16);
        uint32_t ph = 0;
        for (int it = gi; it < n_my; it += 2, ph ^= 1) {
            const int64_t tile = (int64_t)blockIdx.x + (int64_t)it * G;
            P2_WAIT(8, &s.d1_full[gi], ph);
            tc::fence_after_sync();
            // one copy of the hidden stage serves both nets (net B's overlaps the net-A layer-2 MMA)
#pragma unroll 1
            for (int net = 0; net < (has_b ? 2 : 1); ++net) {
                hidden_in_place<SPLIT>(lane_addr + (net ? COL_D1B : COL_D1A), s.bias1[T::HAS_B ? net : 0]);
                tc::fence_before_sync();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(net ? &s.a2b_full[gi] : &s.a2a_full[gi]);
            }
            P2_WAIT(9, &s.d2a_full[gi], ph);
            tc::fence_after_sync();
            // ---- outputs
            const int64_t L = tile * TILE_M + row;                   // plain order: tile row = sample index
            const bool live = L < a.total;
            const int64_t idx = live ? L : 0;
            // Every output row is assembled in record layout [sigma, seg 15 | rgb 32] in this thread's shared-memory staging row
            // (STS only, never a generic store), then the warp copies its 32 rows out in coalesced 16-byte chunks — to the
            // records, or to the rgb / seg outputs when the caller asked for those.
            float4* rec = reinterpret_cast<float4*>(s.recbuf[gi][row]);
            bool done = false;
            if constexpr (KIND == NFE_DEC_DISENTANGLED) {
                // the production decoder keeps ONE copy of each 16-column step (rolled loops): with four roles sharing every
                // sub-partition's instruction cache, code size is time (profiles/pipe2_variants_r02.txt)
                {
                    float v[16];
                    tc::tmem_ld16(lane_addr + COL_D2, v);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 b4 = *reinterpret_cast<const float4*>(&s.bias2a[4 * c]);
                        const float2 lo2 = fadd2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(b4.x, b4.y));
                        const float2 hi2 = fadd2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(b4.z, b4.w));
                        float4 o = make_float4(lo2.x, lo2.y, hi2.x, hi2.y);
                        if (c == 0) {
                            if (a.density_noise > 0.0f && live) {
                                const uint4 r = philox4x32(a.seed, (uint64_t)idx, a.offset);
                                o.x += normal2(r.x, r.y).x * a.density_noise;
                            }
                            if (live) a.sigma[idx] = o.x;
                        }
                        rec[c] = o;
                    }
                }
                done = a.sigma_only;
                if (!done && !GEO) {
                    P2_WAIT(10, &s.d2b_full[gi], ph);
                    tc::fence_after_sync();
#pragma unroll 1
                    for (int q = 0; q < T::N_B / 16; ++q) {
                        float v[16];
                        tc::tmem_ld16(lane_addr + COL_D2 + T::N_A + q * 16, v);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float4 b4 = *reinterpret_cast<const float4*>(&s.bias2b[q * 16 + 4 * c]);
                            const float2 lo2 = rgb_activation2(fadd2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(b4.x, b4.y)));
                            const float2 hi2 = rgb_activation2(fadd2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(b4.z, b4.w)));
                            rec[4 + 4 * q + c] = make_float4(lo2.x, lo2.y, hi2.x, hi2.y);
                        }
                    }
                }
            } else {
                // OSG / segmentation decoders (sigma shares net A's output row with the colours): straight-line code
                float outa[T::N_A];
#pragma unroll
                for (int q = 0; q < (GEO ? 1 : T::N_A / 16); ++q) {       // geometry: sigma is in the first 16 columns
                    float v[16];
                    tc::tmem_ld16(lane_addr + COL_D2 + q * 16, v);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float2 o2 = fadd2(make_float2(v[2 * i], v[2 * i + 1]), *reinterpret_cast<const float2*>(&s.bias2a[q * 16 + 2 * i]));
                        outa[q * 16 + 2 * i] = o2.x; outa[q * 16 + 2 * i + 1] = o2.y;
                    }
                }
                float sig = outa[0];
                if (a.density_noise > 0.0f && live) {
                    const uint4 r = philox4x32(a.seed, (uint64_t)idx, a.offset);
                    sig += normal2(r.x, r.y).x * a.density_noise;
                }
                if (live) a.sigma[idx] = sig;
                done = a.sigma_only;
                if (!done) {
                    if (!T::HAS_B) {
                        rec[0] = make_float4(sig, 0.f, 0.f, 0.f);
                        rec[1] = rec[2] = rec[3] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    if constexpr (!GEO) {
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                            rec[4 + c] = make_float4(rgb_activation(outa[1 + 4 * c]), rgb_activation(outa[2 + 4 * c]),
                                                     rgb_activation(outa[3 + 4 * c]), rgb_activation(outa[4 + 4 * c]));
                    }
                    if constexpr (T::HAS_B) {
                        P2_WAIT(10, &s.d2b_full[gi], ph);
                        tc::fence_after_sync();
                        float outb[T::N_B];
#pragma unroll
                        for (int q = 0; q < T::N_B / 16; ++q) {
                            float v[16];
                            tc::tmem_ld16(lane_addr + COL_D2 + T::N_A + q * 16, v);
                            tc::tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float2 o2 = fadd2(make_float2(v[2 * i], v[2 * i + 1]), *reinterpret_cast<const float2*>(&s.bias2b[q * 16 + 2 * i]));
                                outb[q * 16 + 2 * i] = o2.x; outb[q * 16 + 2 * i + 1] = o2.y;
                            }
                        }
                        rec[0] = make_float4(sig, outb[0], outb[1], outb[2]);
#pragma unroll
                        for (int c = 1; c < 4; ++c) rec[c] = make_float4(outb[4 * c - 1], outb[4 * c], outb[4 * c + 1], outb[4 * c + 2]);
                    }
                }
            }
            tc::fence_before_sync();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&s.d2_free[gi]);
            if (!done) {
                // rows of this warp: tile rows wq*32 .. +31 = samples L0 .. L0+31, one contiguous run of every output
                const int64_t L0 = tile * TILE_M + wq * 32;
                const int n_rows = (int)min((int64_t)32, a.total - L0);
                const unsigned char* rows = s.recbuf[gi][wq * 32];
                if constexpr (GEO) {
                    float4* gdst = reinterpret_cast<float4*>(a.rec + L0 * 16);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {                      // chunk k*32 + lane = row 8k + lane/4, 16-byte chunk lane%4
                        const int r = 8 * k + (lane >> 2);
                        const float4 v = *reinterpret_cast<const float4*>(rows + r * REC_STAGE_STRIDE + (lane & 3) * 16);
                        if (r < n_rows) gdst[k * 32 + lane] = v;
                    }
                } else if (a.rec) {
                    float4* gdst = reinterpret_cast<float4*>(a.rec + L0 * 48);
                    int r = lane / 12, c = lane % 12;                  // chunk k*32 + lane = row r, 16-byte chunk c of the record
#pragma unroll 4
                    for (int k = 0; k < 12; ++k) {
                        const float4 v = *reinterpret_cast<const float4*>(rows + r * REC_STAGE_STRIDE + c * 16);
                        if (r < n_rows) gdst[k * 32 + lane] = v;
                        r += 2; c += 8;
                        if (c >= 12) { c -= 12; r += 1; }
                    }
                } else {
                    float4* gdst = reinterpret_cast<float4*>(a.rgb + L0 * 32);
#pragma unroll 4
                    for (int k = 0; k < 8; ++k) {                      // colours: 8 chunks per row
                        const int r = 4 * k + (lane >> 3);
                        const float4 v = *reinterpret_cast<const float4*>(rows + r * REC_STAGE_STRIDE + (4 + (lane & 7)) * 16);
                        if (r < n_rows) gdst[k * 32 + lane] = v;
                    }
                    if constexpr (KIND != NFE_DEC_OSG) {
                        float* sdst = a.seg + L0 * 15;
                        int r = lane / 15, c = lane % 15;              // labels: float k*32 + lane = row r, logit c
#pragma unroll 5
                        for (int k = 0; k < 15; ++k) {
                            const float v = *reinterpret_cast<const float*>(rows + r * REC_STAGE_STRIDE + (1 + c) * 4);
                            if (r < n_rows) sdst[k * 32 + lane] = v;
                            r += 2; c += 2;
                            if (c >= 15) { c -= 15; r += 1; }
                        }
                    }
                }
                __syncwarp();          // the rows are rewritten by the group's next tile
            }
        }
    } else {
        regs_dec<REGS_MISC>();            // idle warps of the MMA / tap warp group: setmaxnreg is a warp-group-wide instruction
    }
#ifdef NFE_PIPE_PROFILE
    if (lane == 0 && !(warp > TAP_WARP0 + TAP_WARPS - 1 && warp < GATHER_WARP0)) {
        const int role = warp >= GATHER_WARP0 ? 0 : (warp >= TAP_WARP0 ? 1 : (warp == MMA_WARP ? 2 : 3));
        prof_[15] = clock64() - prof_t0_;
        for (int i = 0; i < 16; ++i) atomicAdd(&g_p2_prof[role][i], (unsigned long long)prof_[i]);
    }
#endif
    // ---- teardown
    tc::fence_before_sync();
    __syncthreads();
    if (warp == MMA_WARP) tc::tmem_dealloc(tmem, P2_TMEM_COLS);
}

template <int KIND, bool SPLIT, bool GEO>
static int launch_kind(const FieldArgs& a, const nfe_mlp& net_a, const nfe_mlp& net_b, cudaStream_t stream)
{
    const size_t smem = sizeof(Smem<KIND, SPLIT>) + 128;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(field_pipe2_kernel<KIND, SPLIT, GEO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("field_pipe2_kernel: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e)); return 2; }
        configured = true;
    }
    const int64_t n_tiles = (a.total + TILE_M - 1) / TILE_M;
    const int64_t cap = sm_count();   // persistent: one CTA per SM (it owns all 512 TMEM columns)
    field_pipe2_kernel<KIND, SPLIT, GEO><<<(unsigned)(n_tiles < cap ? n_tiles : cap), THREADS, smem, stream>>>(a, net_a, net_b);
    return check_launch("field_pipe2_kernel");
}

}  // namespace p2

int launch_field_pipe2(int kind, int precision, const FieldArgs& a, const nfe_mlp* net_a, const nfe_mlp* net_b, cudaStream_t stream)
{
    if (a.total <= 0) return 0;
    nfe_mlp none = {};
    const bool split = precision == NFE_PREC_BF16X3;
    if (a.geometry_only) {
        NFE_REQUIRE(kind != NFE_DEC_OSG && a.rec, "field_pipe2_kernel: a geometry-only pass needs a decoder with semantics and the records");
        if (kind == NFE_DEC_DISENTANGLED)
            return split ? p2::launch_kind<NFE_DEC_DISENTANGLED, true, true>(a, *net_a, *net_b, stream)
                         : p2::launch_kind<NFE_DEC_DISENTANGLED, false, true>(a, *net_a, *net_b, stream);
        return split ? p2::launch_kind<NFE_DEC_SEGMENTATION, true, true>(a, *net_a, *net_b, stream)
                     : p2::launch_kind<NFE_DEC_SEGMENTATION, false, true>(a, *net_a, *net_b, stream);
    }
    switch (kind) {
        case NFE_DEC_OSG:
            return split ? p2::launch_kind<NFE_DEC_OSG, true, false>(a, *net_a, none, stream)
                         : p2::launch_kind<NFE_DEC_OSG, false, false>(a, *net_a, none, stream);
        case NFE_DEC_DISENTANGLED:
            return split ? p2::launch_kind<NFE_DEC_DISENTANGLED, true, false>(a, *net_a, *net_b, stream)
                         : p2::launch_kind<NFE_DEC_DISENTANGLED, false, false>(a, *net_a, *net_b, stream);
        default:
            return split ? p2::launch_kind<NFE_DEC_SEGMENTATION, true, false>(a, *net_a, *net_b, stream)
                         : p2::launch_kind<NFE_DEC_SEGMENTATION, false, false>(a, *net_a, *net_b, stream);
    }
}

}  // namespace nfe

#ifdef NFE_PIPE_PROFILE
NFE_EXPORT int nfe_debug_pipe2_profile(unsigned long long* out64, int reset)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out64, nfe::p2::g_p2_prof, sizeof(unsigned long long) * 64);
    if (reset) { unsigned long long z[64] = {}; cudaMemcpyToSymbol(nfe::p2::g_p2_prof, z, sizeof(z)); }
    return 0;
}
#endif

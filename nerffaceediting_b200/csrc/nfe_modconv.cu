// Modulated convolution of the StyleGAN2 backbone / super-resolution stack (SURVEY.md §8f row f3) as a tcgen05 implicit GEMM.
//
// Replaces, for inference:  modulated_conv2d (training/networks_stylegan2.py:34-91) + conv2d_resample's 3x3 / 1x1 and
// transposed (up = 2) cases (torch_utils/ops/conv2d_resample.py:48-143) + the bias_act that follows every layer
// (networks_stylegan2.py:322-325, 351-352).  The reference runs it as a grouped cuDNN convolution over per-sample weights.
//
// Formulation.  Activations are channels-last ([N,H,W,C]; the reference's own fp16_channels_last layout), so one pixel's channels
// are one contiguous run.  out[pixel, o] = sum_{tap, i} x[pixel + shift(tap), i] * Wm[n][o, i, tap] with the per-sample weights
// Wm = W * style * demodulation folded ONCE per call by the packing kernel (the reference folds them too, fused_modconv=True, and
// rounds them to fp16 exactly there).  GEMM view per CTA: M = 128 * MA pixels (a 16*MA x 8 window of the image), N = up to 256
// output channels, K = taps x input channels, accumulated in tensor memory.
//
//  * A operand (activations): ONE halo window (16*MA+2) x 10 pixels x 64 channels per K chunk is brought into shared memory by
//    cp.async with zero fill (that is the convolution's zero padding) in the layout [channel group of 8][halo pixel][8 channels];
//    8 consecutive pixels of a window row x 8 channels are then exactly one 8x16-byte core matrix of the K-major SWIZZLE_NONE
//    operand layout, the next window row is the next row group (SBO = 160 B), the next channel group the next K core matrix
//    (LBO = the halo size).  Every one of the 9 taps of a 3x3 convolution is the SAME buffer read through a descriptor whose start
//    address is shifted by (dy * 10 + dx) * 16 bytes: no im2col copy exists anywhere, and the activations cross the L2 -> SM link
//    once per 9 taps.
//  * B operand (weights): packed by the packing kernel in exactly the shared-memory operand order, one contiguous block per
//    (K chunk, tap), streamed by ONE thread with cp.async.bulk (the TMA unit's bulk copy, completion on an mbarrier with
//    complete_tx) through a ring of up to 6 slots (a slot holds the widest block of the plan).
//  * roles: warps 0-3 load A during the main loop, warp 4 issues the MMAs (one elected thread, tcgen05.mma kind::f16, fp32
//    accumulate), warp 5 streams B, tcgen05.commit releases the stages; all eight warps run the epilogue (thread = TMEM lane =
//    pixel; warps w and w + 4 share a lane quarter and split the columns).
//  * epilogue, fused: + noise, + bias, activation (linear / relu / lrelu), gain, clamp, conversion; rows staged in shared memory in
//    64-column segments and copied out by their warp in coalesced 16-byte stores (channels-last).
//  * up = 2 (conv2d_resample.py:117-134): the transposed stride-2 convolution is four phase convolutions (even/odd output rows x
//    columns: 4 + 2 + 2 + 1 taps, i.e. the 9 taps once — no multiplication by an inserted zero).  ONE CTA computes all four phases of
//    its window: the halo is loaded once, every tap's MMAs go to the accumulator of the tap's phase (4 accumulators x up to 128
//    columns of tensor memory) — two taps of the same input offset, whose phases sit in adjacent accumulators, as ONE weight block
//    and ONE MMA of twice the width (TapPlan) — and the epilogue writes them interleaved and raw into the (2H+1) x (2W+1)
//    intermediate; ONE pass then applies the low-pass filter, noise, bias, activation and clamp (upfir_finish_tiled_kernel; the
//    reference makes four passes of it: upfirdn2d, add_, bias_act).
//  * ToRGB to <= 4 channels without demodulation (the super-resolution blocks' 256 / 128 -> 3) is a streaming reduction, not a GEMM:
//    torgb_small_kernel.
//
// Arithmetic: fp16 activations -> fp16 operands, one MMA per product (what the reference's fp16 layers do in cuDNN);
// fp32 activations -> bf16 hi/lo split of both operands, three MMAs per product, fp32 accumulate (~16 significand bits per operand,
// the decoder's bf16x3 mode; the reference's fp32 layers run with TF32 disabled, training_loop.py:128-129).
#include <algorithm>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "nfe_common.cuh"
#include "nfe_tc.cuh"

namespace nfe {
namespace mc {

constexpr int HALO_W = 10;
constexpr int TILE_W = 8, MAX_TAPS = 9, THREADS = 256, MAX_SA = 4, MAX_SB = 6;
constexpr int SEG_Q16 = 4;                                // epilogue segment: 4 groups of 16 fp16 columns = 128 bytes of a staged row

constexpr int TABLE_BYTES = 256 + 1024 + 1024 + 128;      // mbarriers + TMEM slot | bias of the N tile | output scale of the N tile | tap tables
constexpr int SMEM_BUDGET = 227 * 1024 - TABLE_BYTES;

constexpr int MAX_ACC = 4;

// Taps and accumulators of one launch.  Plain convolution: every tap feeds every accumulator, accumulator m = window rows
// 16 m .. 16 m + 15.  up = 2: accumulator = output phase (row parity, column parity), each tap feeds the one phase it belongs to.
struct TapPlan {
    int taps, n_acc;
    int dy[MAX_TAPS], dx[MAX_TAPS];       // input pixel of tap t = window pixel + (dy, dx)
    int ky[MAX_TAPS], kx[MAX_TAPS];       // weight element of tap t
    unsigned acc_mask[MAX_TAPS];          // accumulators tap t feeds
    // Weight blocks = what one weight stage holds and one group of MMAs consumes.  Normally a block is a tap.  Two taps that read the SAME
    // shifted window and feed ADJACENT accumulators (up = 2: the taps of one input offset belong to neighbouring output phases) are
    // packed as ONE block of 2 * n_tile rows and issued as ONE MMA of N = 2 * n_tile: an M = 128 MMA costs ~125 cycles whatever N is,
    // so nine N = 128 MMAs per K step become three of N = 256 and three of N = 128.
    int n_blk;
    int blk_tap[MAX_TAPS];                // first tap of block u (its dy / dx / acc_mask)
    int blk_width[MAX_TAPS];              // 1 or 2 taps
    int blk_unit[MAX_TAPS];               // offset of block u in the chunk's packed run, in units of one tap's block
    int tap_blk[MAX_TAPS], tap_half[MAX_TAPS];      // where tap t is packed
    int row_off[MAX_ACC];                 // first window row of the accumulator's 128 pixels
    int gh[MAX_ACC], gw[MAX_ACC];         // output grid of the accumulator
    int oy_off[MAX_ACC], ox_off[MAX_ACC]; // grid pixel (gy, gx) is written to (gy * o_mul + oy_off, gx * o_mul + ox_off)
    int o_mul;
};

struct GemmArgs {
    const void* x;                        // [batch, in_h, in_w, in_ch]
    const unsigned char* packed;
    long long packed_item_stride;
    void* y;
    long long ys_n, ys_h, ys_w;           // element strides of y; the channel stride is 1
    const float* noise;                   // noise[n * noise_n + oy * noise_w + ox] or NULL
    long long noise_n;
    int noise_w;
    const float* bias;
    // shared-weight form (split operands): the packed weights are the same for every item; the style multiplies the ACTIVATIONS in the
    // halo loader and the demodulation coefficient the accumulator in the epilogue — y = d[n,o] * sum W[o,i,k] (s[n,i] x[i]), the
    // reference's own non-fused formulation (networks_stylegan2.py:69-79).  NULL: weights are per item, modulated when packed.
    const float* in_scale;                // [batch, in_ch]
    const float* out_scale;               // [batch, out_ch]
    int batch, in_h, in_w, in_ch, out_ch;
    int n_tile, n_tiles, chunks, kc, sb, b_stage, b_slot, halo, stage_ok;     // b_stage: bytes of one tap's block; b_slot: bytes of a ring slot (the widest block)
    int tiles_x, tiles_y;
    int act;                              // bias_act cuda_idx: 1 linear, 2 relu, 3 lrelu
    float alpha, gain, clamp;
    TapPlan tp;
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int src_bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(tc::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
// bulk copy global -> shared by the TMA unit, completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(tc::smem_u32(dst)), "l"(src), "r"(bytes), "r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" :: "r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 u;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));      // (ordered by the callers' __syncwarp)
    return u;
}
__device__ __forceinline__ float fmax3(float a, float b, float c)
{
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));      // FMNMX3 (sm_100)
    return r;
}

// one lane of the (converged) warp; the callers keep their control flow warp-uniform so that descriptors and barrier addresses
// live in uniform registers: a divergent `if (lane == 0)` loop makes the compiler wrap every tcgen05.mma in an ELECT / R2UR
// waterfall (~24 dependent instructions, ~180 cycles per MMA measured against the 128 the tensor core needs)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
// kind::f16 instruction descriptor: fp32 accumulate, both operands K-major; FMT 0 = fp16, 1 = bf16
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int fmt)
{
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

#ifdef NFE_MC_PROFILE
__device__ unsigned long long g_mc_prof[16];
#define MC_WAIT(slot, bar, par) do { const long long t0_ = clock64(); tc::mbar_wait(bar, par); prof_[slot] += clock64() - t0_; } while (0)
#define MC_FLUSH(slot) atomicAdd(&g_mc_prof[slot], (unsigned long long)prof_[slot])
#define MC_CLK(name) const long long name = clock64()
#else
#define MC_WAIT(slot, bar, par) tc::mbar_wait(bar, par)
#define MC_CLK(name)
#endif

template <class T> __device__ __forceinline__ float act_apply(float v, int act, float alpha)
{
    if (act == 2) return fmaxf(v, 0.0f);
    if (act == 3) return v > 0.0f ? v : v * alpha;
    return v;
}

template <int PARTS> struct Elem { using type = __half; };
template <> struct Elem<2> { using type = float; };

// PARTS = 1: fp16 activations / fp16 operands.  PARTS = 2: fp32 activations / bf16 hi + lo operands, three terms per product.
// MA = window height in units of 16 rows (the window is 16 MA x 8 pixels).
// SA = halo stages (up = 2 has little MMA work per K chunk, its loads must run several chunks ahead: four).
// KG = channel groups of 8 a halo stage holds (8 = chunks of 64 channels; 4 = chunks of 32, the split-operand wide tile).
// PS = persistent: one CTA per SM walks its windows (item = blockIdx.x, + gridDim.x, ...) with dedicated roles — warps 0-3 halo loaders,
// 4-11 epilogue, 12 MMA issue, 13 weight stream — so that the loaders and the weight stream run into the NEXT window's first stages while
// the epilogue of the current one drains tensor memory (all 512 columns are one window's accumulators: the MMAs themselves cannot overlap
// it).  What that removes per window: barrier / table / tensor-memory set-up and the latency of the first halo and weight stages.
constexpr int PS_THREADS = 448;
template <int PARTS, int MA, int SA, int KG, bool PS = false>
__global__ void __launch_bounds__(PS ? PS_THREADS : THREADS, (!PS && MA == 1 && SA == 2 && (PARTS == 1 || KG == 4)) ? 2 : 1) conv_gemm_kernel(const GemmArgs a)
{
    using T = typename Elem<PARTS>::type;
    constexpr int NTHREADS = PS ? PS_THREADS : THREADS;
    constexpr int MMA_WARP = PS ? 12 : 4, B_WARP = PS ? 13 : 5, EPI_WARP0 = PS ? 4 : 0;
    constexpr int HALO_H = 16 * MA + 2;
    constexpr int A_LBO = HALO_H * HALO_W * 16;          // bytes between channel groups of 8 (K core matrices)
    constexpr int A_SBO = HALO_W * 16;                    // bytes between window rows (row groups of 8 pixels)
    constexpr int A_PART = KG * A_LBO, A_STAGE = PARTS * A_PART;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* const sA = smem;
    unsigned char* const sB = smem + SA * A_STAGE;
    uint64_t* const bars = reinterpret_cast<uint64_t*>(sB + a.sb * a.b_slot);
    uint64_t* const a_full = bars, * const a_empty = bars + MAX_SA, * const b_full = bars + 2 * MAX_SA, * const b_empty = b_full + MAX_SB;
    uint64_t* const acc_full = b_empty + MAX_SB;                               // [2]: one per accumulator set
    uint64_t* const acc_empty = acc_full + 2;                                  // [2] PS: the epilogue warps have drained the set
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    float* const s_bias = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bars) + 256);       // this N tile's bias, zero where there is none
    float* const s_oscale = s_bias + 256;                                       // this (item, N tile)'s output scale (demodulation coefficients), 1 where there is none
    uint32_t* const s_tap16 = reinterpret_cast<uint32_t*>(s_oscale + 256);      // per weight block: descriptor offset of its shifted window (16-byte units)
    uint32_t* const s_tmask = s_tap16 + MAX_TAPS;                              // per weight block: accumulators it feeds (bit 8: a block of two taps)
    uint32_t* const s_row16 = s_tmask + MAX_TAPS;                              // per accumulator: descriptor offset of its first window row

#ifdef NFE_MC_PROFILE
    long long prof_[16] = {};
    const long long t_cta0 = clock64();
#endif
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const TapPlan& tp = a.tp;
    // windows of this CTA: one (grid = windows x N tiles x batch) or, persistent, every gridDim.x-th item of the flat list
    const int tiles = a.tiles_x * a.tiles_y;
    const int n_win = PS ? (tiles * a.n_tiles * a.batch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 1;
    auto window = [&](int k, int& x0, int& y0, int& n, int& nt) {
        int tile;
        if constexpr (PS) {
            const int item = (int)blockIdx.x + k * (int)gridDim.x, r = item / tiles;
            tile = item - r * tiles; nt = r % a.n_tiles; n = r / a.n_tiles;
        } else {
            tile = blockIdx.x; nt = blockIdx.y; n = blockIdx.z;
        }
        x0 = (tile % a.tiles_x) * TILE_W; y0 = (tile / a.tiles_x) * (16 * MA);
    };
    const int n_blk = tp.n_blk, n_acc = tp.n_acc;
    // persistent CTA: when a window's accumulators take at most half of tensor memory there are TWO sets, and the MMAs of window k + 1
    // run while the epilogue reads window k out
    const int set_cols = n_acc * a.n_tile, n_sets = (PS && 2 * set_cols <= 512) ? 2 : 1;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < n_sets * set_cols) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int i = 0; i < MAX_SA; ++i) { tc::mbar_init(&a_full[i], 128); tc::mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < MAX_SB; ++i) { tc::mbar_init(&b_full[i], 1); tc::mbar_init(&b_empty[i], 1); }
        tc::mbar_init(&acc_full[0], 1); tc::mbar_init(&acc_full[1], 1);
        tc::mbar_init(&acc_empty[0], 8); tc::mbar_init(&acc_empty[1], 8);
        tc::mbar_fence_init();
    }
    if (warp == MMA_WARP) tc::tmem_alloc(tmem_slot, tmem_cols);
    if (threadIdx.x < MAX_TAPS) {
        s_tap16[threadIdx.x] = (uint32_t)((1 + tp.dy[tp.blk_tap[threadIdx.x]]) * HALO_W + 1 + tp.dx[tp.blk_tap[threadIdx.x]]);
        s_tmask[threadIdx.x] = tp.acc_mask[tp.blk_tap[threadIdx.x]] | (tp.blk_width[threadIdx.x] == 2 ? 0x100u : 0u);      // per BLOCK; bit 8: two taps wide
    }
    if (threadIdx.x < MAX_ACC) s_row16[threadIdx.x] = (uint32_t)(tp.row_off[threadIdx.x] * (HALO_W * 16)) >> 4;
    {
        int x0_, y0_, n0, nt0;
        window(0, x0_, y0_, n0, nt0);
        for (int i = threadIdx.x; i < a.n_tile; i += NTHREADS) {
            const int o = nt0 * a.n_tile + i;
            s_bias[i] = (a.bias && o < a.out_ch) ? __ldg(a.bias + o) : 0.0f;
            s_oscale[i] = (a.out_scale && o < a.out_ch) ? __ldg(a.out_scale + (long long)n0 * a.out_ch + o) : 1.0f;
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
#ifdef NFE_MC_PROFILE
    const long long t_role0 = clock64();
    if (threadIdx.x == 0) { prof_[10] = t_role0 - t_cta0; MC_FLUSH(10); atomicAdd(&g_mc_prof[9], (unsigned long long)n_win); }      // per WINDOW figures
#endif

    if (warp < 4) {
        // ------------------------------------------------------------------ A loader: one halo window per K chunk
        const int kcores = a.kc >> 3;
        const T* xin = static_cast<const T*>(a.x);
        // the chunks of all windows of this CTA form one stream: chunk g = window k, chunk c of it; ring stage g % SA
        for (int k = 0, g = 0; k < n_win; ++k) {
        int x0, y0, n, nt;
        window(k, x0, y0, n, nt);
        for (int c = 0; c < a.chunks; ++c, ++g) {
            const int s = g % SA, r = g / SA;
            if constexpr (PARTS == 1) {
                // up to SA - 1 chunks stay in flight: chunk g - (SA - 1) is handed to the MMA thread before this one is requested
                if (g >= SA - 1) { cp_async_wait_group<SA - 2>(); tc::fence_async_smem(); tc::mbar_arrive(&a_full[(g - (SA - 1)) % SA]); }
            }
            if (r > 0) MC_WAIT(3, &a_empty[s], (r - 1) & 1);
            unsigned char* const dst0 = sA + s * A_STAGE;
            // thread = (channel group k8, pixel slot): 16 halo pixels x 8 channel groups per pass, the pixel index advanced
            // incrementally (no divisions); 8 consecutive threads read one pixel's 64 channels, i.e. one contiguous run.  The fp32
            // path (loads through registers: split into bf16 hi + lo) requests FOUR pixels' loads before it converts and stores any
            // of them: one pixel at a time it ran at one DRAM latency per pixel (27 k cycles per chunk measured).
            const int k8 = threadIdx.x & 7;
            int hy = (threadIdx.x >> 3) / HALO_W, hx = (threadIdx.x >> 3) % HALO_W;
            float4 sc0 = make_float4(1.f, 1.f, 1.f, 1.f), sc1 = sc0;          // styles of this thread's 8 channels (shared-weight form)
            if constexpr (PARTS == 2) {
                if (a.in_scale && k8 < kcores) {
                    const float4* sp = reinterpret_cast<const float4*>(a.in_scale + (long long)n * a.in_ch + c * a.kc + k8 * 8);
                    sc0 = __ldg(sp); sc1 = __ldg(sp + 1);
                }
            }
            if (k8 < kcores) {
                constexpr int BATCH = PARTS == 1 ? 1 : 4;
                for (int hp0 = threadIdx.x >> 3; hp0 < HALO_H * HALO_W; hp0 += 16 * BATCH) {
                    float4 v0[BATCH], v1[BATCH];
                    unsigned char* dsts[BATCH];
                    bool live[BATCH];
#pragma unroll
                    for (int b = 0; b < BATCH; ++b) {
                        const int hp = hp0 + 16 * b;
                        const int gy = y0 - 1 + hy, gx = x0 - 1 + hx;
                        const bool ring = hy == 0 || hy == HALO_H - 1 || hx == 0 || hx == HALO_W - 1;
                        const bool ok = (unsigned)gy < (unsigned)a.in_h && (unsigned)gx < (unsigned)a.in_w;
                        dsts[b] = dst0 + k8 * A_LBO + hp * 16;
                        live[b] = hp < HALO_H * HALO_W && !(!a.halo && ring);       // 1x1: the ring is never read
                        hx += 6; hy += 1;                            // + 16 pixels = one window row and 6 columns
                        if (hx >= HALO_W) { hx -= HALO_W; hy += 1; }
                        const T* src = xin + (((long long)(n * a.in_h + (ok ? gy : 0)) * a.in_w + (ok ? gx : 0)) * a.in_ch + c * a.kc + k8 * 8);
                        if constexpr (PARTS == 1) {
                            if (live[b]) cp_async16(dsts[b], src, ok ? 16 : 0);
                        } else {
                            v0[b] = v1[b] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (live[b] && ok) { v0[b] = __ldg(reinterpret_cast<const float4*>(src)); v1[b] = __ldg(reinterpret_cast<const float4*>(src) + 1); }
                        }
                    }
                    if constexpr (PARTS == 2) {
#pragma unroll
                        for (int b = 0; b < BATCH; ++b) {
                            if (!live[b]) continue;
                            const float v[8] = {v0[b].x * sc0.x, v0[b].y * sc0.y, v0[b].z * sc0.z, v0[b].w * sc0.w,
                                                v1[b].x * sc1.x, v1[b].y * sc1.y, v1[b].z * sc1.z, v1[b].w * sc1.w};
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                __nv_bfloat16 h0, l0, h1, l1;
                                tc::split_bf16(v[2 * q], h0, l0); tc::split_bf16(v[2 * q + 1], h1, l1);
                                hi[q] = tc::pack_bf16(h0, h1); lo[q] = tc::pack_bf16(l0, l1);
                            }
                            *reinterpret_cast<uint4*>(dsts[b]) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            *reinterpret_cast<uint4*>(dsts[b] + A_PART) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                }
            }
            if constexpr (PARTS == 1) {
                cp_async_commit();
            } else {
                tc::fence_async_smem();
                tc::mbar_arrive(&a_full[s]);
            }
        }
        }
        if constexpr (PARTS == 1) {
            const int total = n_win * a.chunks;
            cp_async_wait_group<0>();
            tc::fence_async_smem();
            for (int g = total > SA - 1 ? total - (SA - 1) : 0; g < total; ++g) tc::mbar_arrive(&a_full[g % SA]);
        }
#ifdef NFE_MC_PROFILE
        if (threadIdx.x == 0) { prof_[4] = clock64() - t_role0 - prof_[3]; MC_FLUSH(3); MC_FLUSH(4); }
#endif
    } else if (warp == MMA_WARP) {
        // ------------------------------------------------------------------ MMA issue (one thread).  The descriptors differ only in
        // their 14-bit address field (bytes >> 4), so each one is the constant part plus an add: the issuing thread stays far below
        // the tensor core's 64-128 cycles per instruction.  Every lane runs the loop; one elected lane issues.
        {
            const bool leader = elect_one();
            const uint32_t idesc = make_idesc(128, a.n_tile, PARTS == 1 ? 0 : 1);
            const uint32_t b_lbo = a.n_tile * 16, b_part16 = (a.n_tile * a.kc * 2) >> 4, a_part16 = A_PART >> 4;
            const uint64_t da0 = tc::make_desc(0, A_LBO, A_SBO), db0 = tc::make_desc(0, b_lbo, 128);
            const uint32_t a_k16 = (2 * A_LBO) >> 4, b_k16 = (2 * b_lbo) >> 4;
            // a block of two taps: 2 * n_tile rows per K core matrix column, one MMA of N = 2 * n_tile over two adjacent accumulators
            const uint32_t idesc_w = make_idesc(128, 2 * a.n_tile, PARTS == 1 ? 0 : 1);
            const uint64_t db0_w = tc::make_desc(0, 2 * b_lbo, 128);
            const int ksteps = a.kc >> 4;
            // The loop nest stays ROLLED (tap and accumulator tables in shared memory, filled at start-up): unrolled over taps x
            // accumulators x terms it was 16 k instructions in the split-operand build and ran out of the instruction cache — ~500
            // cycles per MMA measured there against the 143 of the (already 7 k instruction) fp16 build.
            int sb = 0;
            uint32_t sb_par = 0;
            constexpr int TERMS = PARTS == 2 ? 3 : 1;
#pragma unroll 1
            for (int k = 0, g = 0; k < n_win; ++k) {
            uint32_t started = 0;                    // accumulators that hold a partial sum already
            const int set = k % n_sets, use = k / n_sets;
            const uint32_t tmem_set = tmem + set * set_cols;
            if (PS && use > 0) {                     // the set's previous window has been read out
                MC_WAIT(0, &acc_empty[set], (use - 1) & 1);
                tc::fence_after_sync();
            }
#pragma unroll 1
            for (int c = 0; c < a.chunks; ++c, ++g) {
                const int s = g % SA;
                MC_WAIT(0, &a_full[s], (g / SA) & 1);
                tc::fence_after_sync();
                const uint32_t a_base16 = tc::smem_u32(sA + s * A_STAGE) >> 4;
#pragma unroll 1
                for (int t = 0; t < n_blk; ++t) {
                    MC_WAIT(1, &b_full[sb], sb_par);
                    tc::fence_after_sync();
                    const uint32_t b16 = tc::smem_u32(sB + sb * a.b_slot) >> 4, a16 = a_base16 + s_tap16[t], mask = s_tmask[t];
                    const uint32_t wide = (mask >> 8) & 1u;                  // warp-uniform
                    const uint32_t idesc_t = wide ? idesc_w : idesc, bp16 = b_part16 << wide, bk16 = b_k16 << wide;
                    const uint64_t db0_t = wide ? db0_w : db0;
#pragma unroll 1
                    for (int m = 0; m < n_acc; ++m) {
                        if (!((mask >> m) & 1u)) continue;
                        uint32_t accf = (started >> m) & 1u;
                        const uint32_t d_tmem = tmem_set + m * a.n_tile, am = a16 + s_row16[m];
#pragma unroll
                        for (int term = 0; term < TERMS; ++term) {          // hi*hi, lo*hi, hi*lo
                            uint64_t da = da0 + (am + (term == 1 ? a_part16 : 0)), db = db0_t + (b16 + (term == 2 ? bp16 : 0));
#pragma unroll 1
                            for (int j = 0; j < ksteps; ++j) {
                                if (leader) tc::mma_bf16_ss(d_tmem, da, db, idesc_t, accf);
                                accf = 1u; da += a_k16; db += bk16;
                            }
                        }
                        started |= (1u | (wide << 1)) << m;
                    }
                    if (leader) tc::mma_commit(&b_empty[sb]);          // the weight stage is free once these MMAs have read it
                    if (++sb == a.sb) { sb = 0; sb_par ^= 1u; }
                }
                if (leader) tc::mma_commit(&a_empty[s]);
            }
            if (leader) tc::mma_commit(&acc_full[set]);
            }
#ifdef NFE_MC_PROFILE
            if (lane == 0) { prof_[2] = clock64() - t_role0; MC_FLUSH(0); MC_FLUSH(1); MC_FLUSH(2); }
#endif
        }
        __syncwarp();
    } else if (warp == B_WARP) {
        // ------------------------------------------------------------------ B stream (one thread): packed weights, one block per (chunk, tap)
        if (lane == 0) {
            const int per_win = a.chunks * n_blk;
            int sb = 0, u = 0;
            uint32_t sb_par = 1;                    // parity of the PREVIOUS use of the stage
            for (int k = 0, it = 0; k < n_win; ++k) {
            int x0, y0, n, nt;
            window(k, x0, y0, n, nt);
            const unsigned char* src = a.packed + n * a.packed_item_stride + (long long)nt * a.chunks * tp.taps * a.b_stage;
            for (int j = 0; j < per_win; ++j, ++it) {
                if (it >= a.sb) MC_WAIT(7, &b_empty[sb], sb_par);
                const uint32_t bytes = (uint32_t)(a.b_stage * tp.blk_width[u]);         // the blocks of a chunk follow each other in issue order
                mbar_expect_tx(&b_full[sb], bytes);
                bulk_copy(sB + sb * a.b_slot, src, bytes, &b_full[sb]);
                src += bytes;
                if (++u == n_blk) u = 0;
                if (++sb == a.sb) { sb = 0; sb_par ^= 1u; }
            }
            }
#ifdef NFE_MC_PROFILE
            MC_FLUSH(7);
#endif
        }
        __syncwarp();
    }
    if (!PS || (warp >= EPI_WARP0 && warp < EPI_WARP0 + 8)) {
        // ------------------------------------------------------------------ epilogue, eight warps (all of them, or the dedicated ones of the
        // persistent CTA): thread = TMEM lane = pixel of the window; warps w and w + 4 share a lane quarter and take alternate accumulators
        const int ew = warp - EPI_WARP0;
        int nt_bias, n_scale;
        { int x0_, y0_; window(0, x0_, y0_, n_scale, nt_bias); }
#pragma unroll 1
        for (int k = 0; k < n_win; ++k) {
        int x0, y0, n, nt;
        window(k, x0, y0, n, nt);
#ifdef NFE_MC_PROFILE
        const long long t_e0 = clock64();
#endif
        const int set = k % n_sets;
        MC_WAIT(5, &acc_full[set], (k / n_sets) & 1);
        tc::fence_after_sync();
#ifdef NFE_MC_PROFILE
        const long long t_e1 = clock64();
#endif
        if (PS && (nt != nt_bias || (a.out_scale && n != n_scale))) {      // the bias / output-scale tables follow the window's tile and item
            asm volatile("bar.sync 1, 256;" ::: "memory");
            for (int i = threadIdx.x - EPI_WARP0 * 32; i < a.n_tile; i += 256) {
                const int o = nt * a.n_tile + i;
                s_bias[i] = (a.bias && o < a.out_ch) ? __ldg(a.bias + o) : 0.0f;
                s_oscale[i] = (a.out_scale && o < a.out_ch) ? __ldg(a.out_scale + (long long)n * a.out_ch + o) : 1.0f;
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            nt_bias = nt; n_scale = n;
        }
        const int row = (ew & 3) * 32 + lane, py = row >> 3, px = row & 7, grp = ew >> 2;
        T* yout = static_cast<T*>(a.y);
        const float neg_slope = a.act == 1 ? 1.0f : (a.act == 2 ? 0.0f : a.alpha);
        const float gain_pos = a.gain, gain_neg = a.gain * neg_slope, clampv = a.clamp >= 0.0f ? a.clamp : __int_as_float(0x7f800000);
        // the up = 2 intermediate leaves as it is (noise, bias, activation, gain and clamp belong to the filter pass): convert and store
        const bool raw = !a.noise && !a.bias && !a.out_scale && a.act == 1 && a.gain == 1.0f && a.clamp < 0.0f;
        constexpr int VEC = 16 / (int)sizeof(T);
        const bool vec_ok = a.out_ch % VEC == 0 && (reinterpret_cast<uintptr_t>(a.y) & 15) == 0 && a.ys_n % VEC == 0 && a.ys_h % VEC == 0 && a.ys_w % VEC == 0;
        const int nq = a.n_tile / 16;
        const uint32_t t_lane = tmem + set * set_cols + ((uint32_t)((ew & 3) * 32) << 16);
        // Stores: a thread holds 16 channels of ONE pixel at a time, so direct store instructions touch 32 different lines with 16
        // bytes each (measured: the epilogue then runs at the speed of its 8192 partial-sector stores).  Instead every thread builds
        // its pixel's row of n_tile channels, in segments of at most 512 bytes (256 halves / 128 floats), in the (now idle) operand
        // rings — at a pitch of 16 bytes more than the segment, which spreads the lanes over the banks — and the WARP then copies its
        // 32 finished rows out with coalesced 16-byte stores (16 or 32 lanes per row): warp-local, no block-wide synchronisation.
        // (Round 2 first handed each row to the TMA unit as a bulk store; a per-thread cp.async.bulk compiles to a 32-trip waterfall
        // around a uniform-datapath UBLKCP.  Both variants take the same time — the SM's store path is the limit —; the copy-out needs
        // no async-proxy fences and no wait before a row is reused.  The bulk variant was measured and removed:
        // profiles/modconv_tuning_r02.txt #13.)
        // Segments are short (SEG_Q16 fp16 groups = 64 columns): the stage then needs 144-272 bytes per row instead of 528 and fits
        // beside every CTA shape.  (Measured: an SM's stores leave at ~28 bytes per clock — 16 KB per warp in ~4.8 k cycles with 8 warps
        // storing — and segment length does not change the epilogue's length: the stores hold the warp, a segment does not drain
        // behind the next one's arithmetic.  profiles/modconv_tuning_r02.txt #13.)
        constexpr int SEG_Q = SEG_Q16 * 2 / (int)sizeof(T);                          // 16-column groups per segment: 128 bytes of a row
        const int PITCH = min(a.n_tile, SEG_Q * 16) * (int)sizeof(T) + 16;           // row pitch in the stage
        const bool staged = vec_ok && a.stage_ok && (nt + 1) * a.n_tile <= a.out_ch;
        // (the persistent CTA's rings are busy with the next window: its stage is a region of its own behind the tables)
        const uint32_t stage0 = tc::smem_u32(smem) + (PS ? (uint32_t)(SA * A_STAGE + a.sb * a.b_slot + TABLE_BYTES) : 0u);
        const uint32_t warp_rows = stage0 + (uint32_t)((grp * 128 + (ew & 3) * 32) * PITCH);    // this warp's 32 staged rows
        const uint32_t my_row = warp_rows + (uint32_t)(lane * PITCH);
        // The epilogue is bound by its instruction count (8 warps x n_tile / 16 groups of 16 columns; ncu: 60 % of the kernel's executed
        // instructions at 256 x 256 channels).  Per value: (v + noise) + bias as packed f32x2 adds, the slope pair as max(t g+, t g-) —
        // equal to t * (t > 0 ? g+ : g-) for gain > 0 and 0 <= slope <= 1 — folded with the lower clamp into one three-input max,
        // then the upper clamp: 4 instructions instead of 7.  The 16-column groups alternate between two register arrays (the next
        // tcgen05.ld is in flight while this group is processed, without register copies).
        const bool fast_act = a.gain > 0.0f && neg_slope >= 0.0f && neg_slope <= 1.0f;
        const float2 gp2 = make_float2(gain_pos, gain_pos), gn2 = make_float2(gain_neg, gain_neg);
        // two warp groups: with several accumulators they take alternate ones, with a single one they take the two halves of its
        // columns (cut at a segment boundary): warps 4-7 would otherwise idle through the epilogue of every N <= 128 tile
        // (epilogue 6.0 k -> 4.5 k cycles at 128 -> 128 channels)
        const int q_cut = n_acc == 1 ? min(nq, (nq / 2 + SEG_Q - 1) / SEG_Q * SEG_Q) : 0;
        const int q0 = n_acc == 1 && grp == 1 ? q_cut : 0, q1 = n_acc == 1 && grp == 0 ? q_cut : nq;
        for (int m = n_acc == 1 ? 0 : grp; m < n_acc; m += 2) {
            const int gy = y0 + tp.row_off[m] + py, gx = x0 + px;
            const bool valid = gy < tp.gh[m] && gx < tp.gw[m];
            const int oy = gy * tp.o_mul + tp.oy_off[m], ox = gx * tp.o_mul + tp.ox_off[m];
            T* dst = yout + n * a.ys_n + oy * a.ys_h + ox * a.ys_w + nt * a.n_tile;
            const unsigned long long dst_bits = valid ? reinterpret_cast<unsigned long long>(dst) : 0ull;     // what the copy-out of other lanes asks for
            const float nz = (a.noise && valid) ? __ldg(a.noise + n * a.noise_n + (long long)oy * a.noise_w + ox) : 0.0f;
            const float2 nz2 = make_float2(nz, nz);
            // the segment just completed in the warp's staged rows goes out: (qs + 1) * 16 columns = `pieces` 16-byte pieces per row;
            // lane i takes piece i % pieces of row i / pieces, then 32 further on, ...: a store instruction covers whole rows
            auto copy_out = [&](const int q, const int qs) {
                // (`slots` = pieces rounded up to a power of two: lanes whose slot is past the row's pieces sit a trip out — only a tile
                //  of 48, 112, ... channels has such a segment)
                const int pieces = (qs + 1) * (int)sizeof(T), shift = 32 - __clz(pieces - 1), slots = 1 << shift;       // pieces 2 .. 16
                const long long seg_off = (long long)(q - qs) * 16 * (int)sizeof(T);
                __syncwarp();
                // four pieces per trip: the shared-memory reads are issued together, then the stores
#pragma unroll 1
                for (int i0 = lane; i0 < 32 * slots; i0 += 128) {
                    uint4 u[4];
                    unsigned long long d[4];
                    int pcs[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int i = i0 + 32 * k, r = (i >> shift) & 31;
                        pcs[k] = i & (slots - 1);
                        d[k] = __shfl_sync(0xffffffffu, dst_bits, r);
                        if (i >= 32 * slots || pcs[k] >= pieces) d[k] = 0ull;
                        u[k] = lds128(warp_rows + (uint32_t)(r * PITCH + min(pcs[k], pieces - 1) * 16));
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (d[k]) *reinterpret_cast<uint4*>(d[k] + seg_off + pcs[k] * 16) = u[k];
                }
                __syncwarp();                          // the rows are rewritten by the next segment
            };
            auto stage = [&](const int qs, const float (&v)[16]) {
                // (rows outside the image are staged too and skipped by the copy-out: the warp stays converged)
                const uint32_t out = my_row + (uint32_t)(qs * 16 * (int)sizeof(T));
                if constexpr (PARTS == 1) {
                    uint32_t w[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) { const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]); w[i] = *reinterpret_cast<const uint32_t*>(&h); }
                    sts128(out, w[0], w[1], w[2], w[3]); sts128(out + 16, w[4], w[5], w[6], w[7]);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        sts128(out + 16 * i, __float_as_uint(v[4 * i]), __float_as_uint(v[4 * i + 1]), __float_as_uint(v[4 * i + 2]), __float_as_uint(v[4 * i + 3]));
                }
            };
            const uint32_t t_acc = t_lane + m * a.n_tile;
            if (staged && (raw || fast_act)) {
                // ---- the production path: staged rows, packed math, two register arrays
                auto group = [&](const int q, float (&v)[16]) {
                    const int qs = q % SEG_Q;
                    if (!raw) {
#pragma unroll
                        for (int i4 = 0; i4 < 4; ++i4) {
                            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + q * 16 + 4 * i4);      // same address in every lane: broadcast
                            const float4 d4 = *reinterpret_cast<const float4*>(s_oscale + q * 16 + 4 * i4);    // 1 unless the weights are shared
                            const float2 t0 = fadd2(ffma2(make_float2(v[4 * i4], v[4 * i4 + 1]), make_float2(d4.x, d4.y), nz2), make_float2(b4.x, b4.y));
                            const float2 t1 = fadd2(ffma2(make_float2(v[4 * i4 + 2], v[4 * i4 + 3]), make_float2(d4.z, d4.w), nz2), make_float2(b4.z, b4.w));
                            const float2 p0 = fmul2(t0, gp2), n0 = fmul2(t0, gn2), p1 = fmul2(t1, gp2), n1 = fmul2(t1, gn2);
                            v[4 * i4] = fminf(fmax3(p0.x, n0.x, -clampv), clampv); v[4 * i4 + 1] = fminf(fmax3(p0.y, n0.y, -clampv), clampv);
                            v[4 * i4 + 2] = fminf(fmax3(p1.x, n1.x, -clampv), clampv); v[4 * i4 + 3] = fminf(fmax3(p1.y, n1.y, -clampv), clampv);
                        }
                    }
                    stage(qs, v);
                };
                float ra[16], rb[16];
                if (q0 < q1) tc::tmem_ld16(t_acc + q0 * 16, ra);
#pragma unroll 1
                for (int q = q0; q < q1; q += 2) {
                    MC_CLK(t_p0);
                    tc::tmem_ld_wait();
                    if (q + 1 < q1) tc::tmem_ld16(t_acc + (q + 1) * 16, rb);
                    MC_CLK(t_p1);
                    group(q, ra);
                    MC_CLK(t_p2);
                    if (q + 1 < q1) {
                        tc::tmem_ld_wait();
                        if (q + 2 < q1) tc::tmem_ld16(t_acc + (q + 2) * 16, ra);
                        group(q + 1, rb);
                    }
                    MC_CLK(t_p3);
                    // segments hold an even number of groups: one ends with the pair's second group, or with the range
                    const int ql = min(q + 1, q1 - 1), qls = ql % SEG_Q;
                    if (qls == SEG_Q - 1 || ql == q1 - 1) copy_out(ql, qls);
#ifdef NFE_MC_PROFILE
                    { const long long t_p4 = clock64(); prof_[15] += t_p1 - t_p0; prof_[14] += t_p2 - t_p1; prof_[13] += t_p3 - t_p2; prof_[11] += t_p4 - t_p3; }
#endif
                }
            } else {
                // ---- everything else (channel counts or strides that rule out 16-byte stores, tiles past out_ch, unusual slopes): rare, so
                //      compact rather than fast — rolled loops over a group held in local memory, direct stores
                float v[16];
#pragma unroll 1
                for (int q = q0; q < q1; ++q) {
                    tc::tmem_ld16(t_acc + q * 16, v);
                    tc::tmem_ld_wait();
                    const int o0 = nt * a.n_tile + q * 16;
#pragma unroll 1
                    for (int i = 0; i < (valid ? 16 : 0); ++i) {
                        float t = v[i];
                        if (!raw) {
                            t = fmaf(t, s_oscale[q * 16 + i], nz) + s_bias[q * 16 + i];
                            t *= t > 0.0f ? gain_pos : gain_neg;      // linear / relu / lrelu as one slope pair (bias_act.cu:66-75), then the gain
                            t = fminf(fmaxf(t, -clampv), clampv);
                        }
                        if (o0 + i < a.out_ch) {
                            if constexpr (PARTS == 1) dst[q * 16 + i] = __float2half_rn(t); else dst[q * 16 + i] = t;
                        }
                    }
                }
            }
        }
        tc::fence_before_sync();
        if constexpr (PS) {                                // tensor memory is free for the next window's MMAs
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&acc_empty[set]);
        }
#ifdef NFE_MC_PROFILE
        prof_[6] += clock64() - t_e1;
        (void)t_e0;
        if (k == n_win - 1 && threadIdx.x == EPI_WARP0 * 32) { MC_FLUSH(5); MC_FLUSH(6); MC_FLUSH(11); MC_FLUSH(13); MC_FLUSH(14); MC_FLUSH(15); }
#endif
        }
    }
    __syncthreads();
    if (warp == MMA_WARP) {
        tc::fence_after_sync();
        tc::tmem_dealloc(tmem, tmem_cols);
    }
#ifdef NFE_MC_PROFILE
    if (threadIdx.x == 0) atomicAdd(&g_mc_prof[8], (unsigned long long)(clock64() - t_cta0));
#endif
}

// ---------------------------------------------------------------------------------------------- weight folding and packing
struct PackArgs {
    const float* weight;                  // [O, I, k, k]
    const float* styles;                  // [N, I]
    float* dcoef;                         // [N, O] workspace
    float* wmul;                          // [O] workspace (fp16 pre-normalisation, networks_stylegan2.py:55-57)
    float* smax;                          // [N]
    unsigned char* packed;
    long long packed_item_stride;
    long long weight_batch_stride;        // elements between the items' weights (0: shared)
    int batch, out_ch, in_ch, ksize, demodulate, prenorm, parts;
    int shared;                           // pack W alone, once for the batch (the style and the demodulation travel with the GEMM)
    int n_tile, n_tiles, chunks, kc, b_stage;
    TapPlan tp;
};

// one block per output channel: demodulation coefficients rsqrt(sum_{i,k} (w * s)^2 + 1e-8) of every batch item
// (networks_stylegan2.py:59-66).  sum_{i,k} (w s)^2 = sum_i s_i^2 q_i with q_i = sum_k w_ik^2: the weight row is read ONCE, folded over the
// taps into shared memory, and contracted with each item's squared styles (a block per (o, item) re-read it for every item).
__global__ void __launch_bounds__(128) modconv_coef_kernel(const PackArgs a)
{
    extern __shared__ float q_sm[];                 // [in_ch]
    __shared__ float red[4];
    const int o = blockIdx.x, kk = a.ksize * a.ksize, per_o = a.in_ch * kk;
    const float* w = a.weight + (long long)o * per_o;
    auto block_reduce = [&](float v, bool is_max) {
        v = is_max ? warp_max(v) : warp_sum(v);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
        __syncthreads();
        return is_max ? fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3])) : (red[0] + red[1]) + (red[2] + red[3]);
    };
    float wm = 1.0f;
    if (a.prenorm) {                                // networks_stylegan2.py:55-57
        float mw = 0.0f;
        for (int i = threadIdx.x; i < per_o; i += 128) mw = fmaxf(mw, fabsf(__ldg(w + i)));
        mw = block_reduce(mw, true);
        wm = (float)(1.0 / sqrt((double)per_o)) / mw;
    }
    if (threadIdx.x == 0) a.wmul[o] = wm;
    for (int n = 0; n < a.batch; ++n) {
        if (n == 0 || a.weight_batch_stride) {                  // per-item weights: fold this item's row (the pre-normalisation above used item 0's:
            __syncthreads();                                    // it only applies with demodulation, which per-item weights come without)
            const float* wn = w + n * a.weight_batch_stride;
            for (int i = threadIdx.x; i < a.in_ch; i += 128) {
                float q = 0.0f;
                for (int t = 0; t < kk; ++t) { const float v = __ldg(wn + i * kk + t) * wm; q = fmaf(v, v, q); }
                q_sm[i] = q;
            }
            __syncthreads();
        }
        const float* s = a.styles ? a.styles + (long long)n * a.in_ch : nullptr;
        float sm = 1.0f;
        if (a.prenorm) {
            float ms = 0.0f;
            for (int i = threadIdx.x; i < a.in_ch; i += 128) ms = fmaxf(ms, s ? fabsf(__ldg(s + i)) : 1.0f);
            sm = block_reduce(ms, true);
        }
        float acc = 0.0f;
        if (a.demodulate)
            for (int i = threadIdx.x; i < a.in_ch; i += 128) {
                const float s0 = s ? __ldg(s + i) : 1.0f, sv = a.prenorm ? s0 / sm : s0;
                acc = fmaf(sv * sv, q_sm[i], acc);
            }
        acc = block_reduce(acc, false);
        if (threadIdx.x == 0) {
            a.dcoef[(long long)n * a.out_ch + o] = a.demodulate ? 1.0f / sqrtf(acc + 1e-8f) : 1.0f;
            if (o == 0) a.smax[n] = sm;
        }
    }
}

// one thread per (output channel, group of 8 input channels): w * s * d for every tap, rounded to the operand type, stored as one
// 16-byte operand slot per tap in the order [N tile][K chunk][tap][part][channel group][row group][row][8 channels].  The thread's
// 8 x k x k weights are one contiguous run (288 bytes for 3x3), read once from L2 and again from L1 for the other taps; a thread per
// (slot, tap) re-fetched every 32-byte sector eight times and made the packing cost more than the small layers' convolutions.
__global__ void __launch_bounds__(256) modconv_pack_kernel(const PackArgs a)
{
    const int n = blockIdx.y, kk = a.ksize * a.ksize;
    const int kcores = a.kc >> 3, rows = a.n_tile;
    const TapPlan& ph = a.tp;
    // three adjacent lanes share a slot and take every third tap (more threads in flight: the kernel is latency-bound; their reads
    // fall into the same sectors)
    const int tg_n = ph.taps % 3 == 0 ? 3 : 1;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long slot = tid / tg_n;
    const int tg = (int)(tid % tg_n);
    const long long slots = (long long)a.n_tiles * a.chunks * kcores * rows;
    if (slot >= slots) return;
    const int row = (int)(slot % rows); long long r = slot / rows;
    const int k8 = (int)(r % kcores); r /= kcores;
    const int c = (int)(r % a.chunks); const int nt = (int)(r / a.chunks);
    const int o = nt * a.n_tile + row, i0 = c * a.kc + k8 * 8;
    const bool real = o < a.out_ch;
    float sd[8];                                   // style (pre-normalised) of the 8 input channels; the demodulation factor follows
    float wm = 1.0f, d = 0.0f;
    const float* w = a.weight + n * a.weight_batch_stride + ((long long)(real ? o : 0) * a.in_ch + i0) * kk;
    if (real) {
        const float sm = a.prenorm ? a.smax[n] : 1.0f;
        wm = a.prenorm ? a.wmul[o] : 1.0f;
        d = a.shared ? 1.0f : a.dcoef[(long long)n * a.out_ch + o];
        const float* s = (a.styles && !a.shared) ? a.styles + (long long)n * a.in_ch + i0 : nullptr;
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float s0 = s ? __ldg(s + j) : 1.0f; sd[j] = a.prenorm ? s0 / sm : s0; }
    }
    unsigned char* const chunk0 = a.packed + n * a.packed_item_stride + (((long long)nt * a.chunks + c) * ph.taps) * a.b_stage;
#pragma unroll 1
    for (int t = tg; t < ph.taps; t += tg_n) {
        float v[8];
        const int wt = ph.ky[t] * a.ksize + ph.kx[t];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = real ? ((__ldg(w + j * kk + wt) * wm) * sd[j]) * d : 0.0f;
        // block of this tap: `width` taps side by side, [part][K core matrix column][width * rows / 8 row groups][8 rows][16 bytes]
        const int width = ph.blk_width[ph.tap_blk[t]], rowb = ph.tap_half[t] * rows + row, rows_b = width * rows;
        unsigned char* dst = chunk0 + (long long)ph.blk_unit[ph.tap_blk[t]] * a.b_stage + ((long long)k8 * (rows_b / 8) + rowb / 8) * 128 + (rowb & 7) * 16;
        if (a.parts == 1) {
            uint32_t w4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { const __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]); w4[j] = *reinterpret_cast<const uint32_t*>(&h); }
            *reinterpret_cast<uint4*>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
        } else {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                __nv_bfloat16 h0, l0, h1, l1;
                tc::split_bf16(v[2 * j], h0, l0); tc::split_bf16(v[2 * j + 1], h1, l1);
                hi[j] = tc::pack_bf16(h0, h1); lo[j] = tc::pack_bf16(l0, l1);
            }
            *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(dst + width * (a.b_stage / 2)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
    }
}

// ---------------------------------------------------------------------------------------------- up = 2: filter + noise + bias + act
struct FinishArgs {
    const void* t;                        // [batch, th, tw, c] channels-last: the transposed convolution's output
    void* y;                              // [batch, oh, ow, c]
    const float* f;                       // [fh, fw]
    const float* noise; long long noise_n;
    const float* bias;
    int batch, th, tw, oh, ow, c, fh, fw, pad_y0, pad_x0, flip;
    float fgain;
    int act; float alpha, gain, clamp;
};

// y[oy, ox, :] = bias_act(sum_{ky,kx} F[ky,kx] * t[oy + ky - pad, ox + kx - pad, :] * fgain + noise[oy, ox]); 8 channels per thread
// (upfirdn2d.py:169-214 with up = down = 1 on the already up-sampled image; conv2d_resample.py:131, networks_stylegan2.py:84-85,322-325)
template <class T>
__global__ void __launch_bounds__(256) upfir_finish_kernel(const FinishArgs a)
{
    constexpr int V = 16 / (int)sizeof(T) >= 8 ? 8 : 4;     // channels per thread: 8 halves or 4 floats (16 bytes)
    __shared__ float filt[64];
    if ((int)threadIdx.x < a.fh * a.fw) {
        const int ky = threadIdx.x / a.fw, kx = threadIdx.x % a.fw;
        filt[threadIdx.x] = __ldg(a.f + (a.flip ? ky : a.fh - 1 - ky) * a.fw + (a.flip ? kx : a.fw - 1 - kx)) * a.fgain;
    }
    __syncthreads();
    const int cv = a.c / V;
    const long long total = (long long)a.batch * a.oh * a.ow * cv;
    const T* tin = static_cast<const T*>(a.t);
    T* yout = static_cast<T*>(a.y);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c0 = (int)(i % cv) * V; long long r = i / cv;
        const int ox = (int)(r % a.ow); r /= a.ow;
        const int oy = (int)(r % a.oh); const int n = (int)(r / a.oh);
        float acc[V];
#pragma unroll
        for (int j = 0; j < V; ++j) acc[j] = 0.0f;
        for (int ky = 0; ky < a.fh; ++ky) {
            const int iy = oy + ky - a.pad_y0;
            if (iy < 0 || iy >= a.th) continue;
            for (int kx = 0; kx < a.fw; ++kx) {
                const int ix = ox + kx - a.pad_x0;
                if (ix < 0 || ix >= a.tw) continue;
                const float w = filt[ky * a.fw + kx];
                const T* src = tin + (((long long)n * a.th + iy) * a.tw + ix) * a.c + c0;
                if constexpr (sizeof(T) == 2) {
                    const uint4 u = __ldg(reinterpret_cast<const uint4*>(src));
                    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const float2 f2 = __half22float2(h[j]); acc[2 * j] = fmaf(f2.x, w, acc[2 * j]); acc[2 * j + 1] = fmaf(f2.y, w, acc[2 * j + 1]); }
                } else {
                    const float4 u = __ldg(reinterpret_cast<const float4*>(src));
                    acc[0] = fmaf(u.x, w, acc[0]); acc[1] = fmaf(u.y, w, acc[1]); acc[2] = fmaf(u.z, w, acc[2]); acc[3] = fmaf(u.w, w, acc[3]);
                }
            }
        }
        const float nz = a.noise ? __ldg(a.noise + n * a.noise_n + (long long)oy * a.ow + ox) : 0.0f;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            float t = acc[j];
            if constexpr (sizeof(T) == 2) t = __half2float(__float2half_rn(t));      // the reference stores the filtered image in fp16
            t += nz;
            if (a.bias) t += __ldg(a.bias + c0 + j);
            t = act_apply<T>(t, a.act, a.alpha) * a.gain;
            if (a.clamp >= 0.0f) t = fminf(fmaxf(t, -a.clamp), a.clamp);
            acc[j] = t;
        }
        T* dst = yout + (((long long)n * a.oh + oy) * a.ow + ox) * a.c + c0;
        if constexpr (sizeof(T) == 2) {
            uint32_t w4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { const __half2 h = __floats2half2_rn(acc[2 * j], acc[2 * j + 1]); w4[j] = *reinterpret_cast<const uint32_t*>(&h); }
            *reinterpret_cast<uint4*>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
        } else {
            *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        }
    }
}

// Tiled form for filters of at most 4 x 4 (the reference's [1,3,3,1]): a block owns 16 x 16 output pixels x one 128-byte channel
// slice (64 halves / 32 floats), stages the (16 + f - 1)^2 input pixels of that slice in shared memory once (the generic kernel
// above re-reads every input pixel 16 times through L1 / L2: measured 3x the time the bytes need) and then every thread computes
// 16 bytes of channels per output pixel from 16-byte shared-memory reads.
constexpr int FT = 16, FT_IN = FT + 3;
constexpr int FIN_MIN_BLOCKS = 4;

template <class T>
__global__ void __launch_bounds__(256, FIN_MIN_BLOCKS) upfir_finish_tiled_kernel(const FinishArgs a, int tiles_x, int tiles_y, int slices)
{
    constexpr int V = 16 / (int)sizeof(T);                   // channels per 16 bytes
    __shared__ __align__(16) unsigned char tile[FT_IN * FT_IN * 128];
    __shared__ float filt[16], f_row[4], f_col[4];
    __shared__ float s_bias[64];
    // the filter as a zero-padded 4 x 4 table (flipped unless flip_filter, gain folded in) and, when it is an outer product — the
    // reference's [1,3,3,1] is —, its two factors: 4 + 4 taps per output instead of 16
    if (threadIdx.x < 16) {
        const int ky = threadIdx.x >> 2, kx = threadIdx.x & 3;
        filt[threadIdx.x] = (ky < a.fh && kx < a.fw) ? __ldg(a.f + (a.flip ? ky : a.fh - 1 - ky) * a.fw + (a.flip ? kx : a.fw - 1 - kx)) * a.fgain : 0.0f;
    }
    const int bx = blockIdx.x % tiles_x, by = blockIdx.x / tiles_x, sl = blockIdx.y % slices, n = blockIdx.y / slices;
    const int ox0 = bx * FT, oy0 = by * FT, c_base = sl * 8 * V;
    const int groups = min(8, (a.c - c_base) / V);          // 16-byte channel groups of this slice
    if (threadIdx.x < 8 * V) s_bias[threadIdx.x] = (a.bias && c_base + (int)threadIdx.x < a.c) ? __ldg(a.bias + c_base + threadIdx.x) : 0.0f;
    const T* tin = static_cast<const T*>(a.t);
    T* yout = static_cast<T*>(a.y);
    const int g = threadIdx.x & 7;
    // the whole input tile is requested at once with cp.async (zero fill outside the image): ~11 independent 16-byte copies per thread
    // in flight and no staging registers, where dependent load -> store pairs left the block waiting on one latency after another
    if (g < groups)
        for (int p = threadIdx.x >> 3; p < FT_IN * FT_IN; p += 32) {
            const int iy = oy0 + p / FT_IN - a.pad_y0, ix = ox0 + p % FT_IN - a.pad_x0;
            const bool ok = iy >= 0 && iy < a.th && ix >= 0 && ix < a.tw;
            cp_async16(tile + p * 128 + g * 16, tin + (((long long)n * a.th + (ok ? iy : 0)) * a.tw + (ok ? ix : 0)) * a.c + c_base + g * V, ok ? 16 : 0);
        }
    cp_async_commit();
    cp_async_wait_group<0>();
    __syncthreads();
    bool entry_ok = true;
    if (threadIdx.x < 16) {
        float total = 0.0f, r = 0.0f, c = 0.0f;
        const int ky = threadIdx.x >> 2, kx = threadIdx.x & 3;
        for (int i = 0; i < 16; ++i) total += filt[i];
        for (int i = 0; i < 4; ++i) { r += filt[ky * 4 + i]; c += filt[i * 4 + kx]; }
        entry_ok = total != 0.0f && fabsf(filt[threadIdx.x] - r * c / total) <= 1e-6f * fabsf(total);
        if (kx == 0) f_row[ky] = r;                                   // F = f_row (x) f_col with f_col = column sums / total
        if (ky == 0) f_col[kx] = total != 0.0f ? c / total : 0.0f;
    }
    const bool separable = __syncthreads_and(entry_ok);
    if (g >= groups) return;
    const int px = (threadIdx.x >> 3) & 15, half = threadIdx.x >> 7;     // this thread: column px, output rows 8 half .. 8 half + 7
    const int ox = ox0 + px;
    if (ox >= a.ow) return;
    auto load8 = [&](int row, int col, float (&v)[V]) {
        const uint4 u = *reinterpret_cast<const uint4*>(tile + (row * FT_IN + col) * 128 + g * 16);
        if constexpr (sizeof(T) == 2) {
            const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
            for (int j = 0; j < 4; ++j) { const float2 f2 = __half22float2(h[j]); v[2 * j] = f2.x; v[2 * j + 1] = f2.y; }
        } else {
            v[0] = __uint_as_float(u.x); v[1] = __uint_as_float(u.y); v[2] = __uint_as_float(u.z); v[3] = __uint_as_float(u.w);
        }
    };
    // per-thread constants of the epilogue: this thread's V biases, the activation as one slope pair, the clamp (infinite when off)
    float bias_r[V];
#pragma unroll
    for (int j = 0; j < V; ++j) bias_r[j] = s_bias[g * V + j];
    const float neg_slope = a.act == 1 ? 1.0f : (a.act == 2 ? 0.0f : a.alpha);
    const float gain_pos = a.gain, gain_neg = a.gain * neg_slope, clampv = a.clamp >= 0.0f ? a.clamp : __int_as_float(0x7f800000);
    auto finish = [&](int py, float (&acc)[V]) {
        const int oy = oy0 + py;
        if (oy >= a.oh) return;
        const float nz = a.noise ? __ldg(a.noise + n * a.noise_n + (long long)oy * a.ow + ox) : 0.0f;
        const float2 nz2 = make_float2(nz, nz);
        uint32_t w4[V / 2];
#pragma unroll
        for (int j = 0; j < V / 2; ++j) {
            float2 t = make_float2(acc[2 * j], acc[2 * j + 1]);
            if constexpr (sizeof(T) == 2) t = __half22float2(__floats2half2_rn(t.x, t.y));      // the reference stores the filtered image in fp16
            t = fadd2(fadd2(t, nz2), make_float2(bias_r[2 * j], bias_r[2 * j + 1]));
            t.x *= t.x > 0.0f ? gain_pos : gain_neg;                                              // linear / relu / lrelu, then the gain
            t.y *= t.y > 0.0f ? gain_pos : gain_neg;
            t.x = fminf(fmaxf(t.x, -clampv), clampv); t.y = fminf(fmaxf(t.y, -clampv), clampv);
            if constexpr (sizeof(T) == 2) { const __half2 h = __floats2half2_rn(t.x, t.y); w4[j] = *reinterpret_cast<const uint32_t*>(&h); }
            else { acc[2 * j] = t.x; acc[2 * j + 1] = t.y; }
        }
        T* dst = yout + (((long long)n * a.oh + oy) * a.ow + ox) * a.c + c_base + g * V;
        if constexpr (sizeof(T) == 2) *reinterpret_cast<uint4*>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
        else *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    };
    if (separable) {
        const float fx[4] = {f_col[0], f_col[1], f_col[2], f_col[3]}, fy[4] = {f_row[0], f_row[1], f_row[2], f_row[3]};
        // channel pairs as packed f32x2 (one FFMA2 per pair and tap)
        auto load2 = [&](int row, int col, float2 (&v)[V / 2]) {
            const uint4 u = *reinterpret_cast<const uint4*>(tile + (row * FT_IN + col) * 128 + g * 16);
            if constexpr (sizeof(T) == 2) {
                const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = __half22float2(h[j]);
            } else {
                v[0] = make_float2(__uint_as_float(u.x), __uint_as_float(u.y)); v[1] = make_float2(__uint_as_float(u.z), __uint_as_float(u.w));
            }
        };
        float2 hs[4][V / 2];                         // horizontal sums of the last four input rows (static indices: the loop is unrolled)
#pragma unroll
        for (int r = 0; r < 8 + 3; ++r) {
            float2 h[V / 2];
#pragma unroll
            for (int kx = 0; kx < 4; ++kx) {
                float2 v[V / 2];
                load2(8 * half + r, px + kx, v);
                const float2 f2 = make_float2(fx[kx], fx[kx]);
#pragma unroll
                for (int j = 0; j < V / 2; ++j) h[j] = kx == 0 ? ffma2(v[j], f2, make_float2(0.0f, 0.0f)) : ffma2(v[j], f2, h[j]);
            }
#pragma unroll
            for (int j = 0; j < V / 2; ++j) hs[r & 3][j] = h[j];
            if (r >= 3) {
                float acc[V];
#pragma unroll
                for (int j = 0; j < V / 2; ++j) {
                    float2 t = make_float2(0.0f, 0.0f);
#pragma unroll
                    for (int ky = 0; ky < 4; ++ky) t = ffma2(hs[(r - 3 + ky) & 3][j], make_float2(fy[ky], fy[ky]), t);
                    acc[2 * j] = t.x; acc[2 * j + 1] = t.y;
                }
                finish(8 * half + r - 3, acc);
            }
        }
    } else {
#pragma unroll 1
        for (int py = 8 * half; py < 8 * half + 8; ++py) {
            float acc[V];
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = 0.0f;
            for (int ky = 0; ky < 4; ++ky)
                for (int kx = 0; kx < 4; ++kx) {
                    const float w = filt[ky * 4 + kx];
                    float v[V];
                    load8(py + ky, px + kx, v);
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] = fmaf(v[j], w, acc[j]);
                }
            finish(py, acc);
        }
    }
}

// ---------------------------------------------------------------------------------------------- ToRGB to a handful of channels
// 1x1 modulated convolution to at most 4 output channels (ToRGBLayer of the super-resolution blocks: 256 / 128 -> 3), without
// demodulation: 6 FLOP per input byte — a streaming reduction, not a GEMM (through conv_gemm_kernel its windows cost more in fixed
// overhead than in work: 0.2 ms per call against the 0.09 ms the bytes need).  One thread per pixel walks the pixel's channels in
// 16-byte pieces; the per-sample weights w * s sit in shared memory (every lane reads the same address: broadcast).
struct RgbArgs {
    const void* x; const float* weight; const float* styles; const float* bias; void* y;
    long long weight_batch_stride;
    int batch, in_ch, out_ch; long long pixels;
    float neg_slope_gain, gain, clamp;
};

// shared-memory stride (floats) of one 16-byte piece's weights: >= V * O, a multiple of 4 whose quarter is odd, so that the 8 lanes
// of a pixel (8 consecutive pieces) read 8 distinct 16-byte bank groups
__host__ __device__ constexpr int rgb_piece_stride(int v, int o) { int s = (v * o + 3) / 4; return (s | 1) * 4; }

template <class T, int O>
__global__ void __launch_bounds__(256) torgb_small_kernel(const RgbArgs a)
{
    extern __shared__ __align__(16) float wm[];              // [piece][O][channel in piece], pieces rgb_piece_stride apart
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int PS = rgb_piece_stride(V, O);
    static_assert((V * O) % 4 == 0, "piece weights are read as float4");
    const int n = blockIdx.y;
    for (int i = threadIdx.x; i < a.in_ch * O; i += 256) {
        const int c = i / O, o = i % O;
        const float w = o < a.out_ch ? __ldg(a.weight + n * a.weight_batch_stride + (long long)o * a.in_ch + c) : 0.0f;
        float ws = w * (a.styles ? __ldg(a.styles + (long long)n * a.in_ch + c) : 1.0f);
        if constexpr (sizeof(T) == 2) ws = __half2float(__float2half_rn(ws));      // the reference hands cuDNN w.to(x.dtype), networks_stylegan2.py:87
        wm[(c / V) * PS + o * V + (c % V)] = ws;
    }
    __syncthreads();
    const T* xin = static_cast<const T*>(a.x) + (long long)n * a.pixels * a.in_ch;
    T* yout = static_cast<T*>(a.y) + (long long)n * a.pixels * a.out_ch;
    const float clampv = a.clamp >= 0.0f ? a.clamp : __int_as_float(0x7f800000);
    // 8 lanes per pixel: a warp's load instruction covers 4 pixels x 128 contiguous bytes (4 lines, where a lane per pixel would
    // touch 32); the lanes' partial sums meet in three shuffle steps
    const int sub = threadIdx.x & 7;
    const int pieces = a.in_ch / V;
    constexpr int PIX = 2;                                   // pixels per lane group and turn: twice the loads in flight
    const long long turn = (long long)gridDim.x * 32 * PIX;
    for (long long base = ((long long)blockIdx.x * 8 + (threadIdx.x >> 5)) * 4 * PIX; base < a.pixels; base += turn) {
        long long px[PIX];
        const uint4* src[PIX];
        float2 acc2[PIX][O];                                 // even / odd channels of the piece: packed f32x2 FMAs
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            px[i] = base + 4 * i + (threadIdx.x >> 3 & 3);
            src[i] = reinterpret_cast<const uint4*>(xin + (px[i] < a.pixels ? px[i] : 0) * a.in_ch);
#pragma unroll
            for (int o = 0; o < O; ++o) acc2[i][o] = make_float2(0.0f, 0.0f);
        }
#pragma unroll 2
        for (int k = sub; k < pieces; k += 8) {
            uint4 u[PIX];
#pragma unroll
            for (int i = 0; i < PIX; ++i) u[i] = __ldg(src[i] + k);
            float4 w4[O][V / 4];
#pragma unroll
            for (int o = 0; o < O; ++o)
#pragma unroll
                for (int j = 0; j < V / 4; ++j) w4[o][j] = *reinterpret_cast<const float4*>(wm + k * PS + o * V + 4 * j);
#pragma unroll
            for (int i = 0; i < PIX; ++i) {
                float2 v[V / 2];
                if constexpr (sizeof(T) == 2) {
                    const __half2* h = reinterpret_cast<const __half2*>(&u[i]);
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = __half22float2(h[j]);
                } else {
                    v[0] = make_float2(__uint_as_float(u[i].x), __uint_as_float(u[i].y)); v[1] = make_float2(__uint_as_float(u[i].z), __uint_as_float(u[i].w));
                }
#pragma unroll
                for (int o = 0; o < O; ++o) {
#pragma unroll
                    for (int j = 0; j < V / 4; ++j) {
                        acc2[i][o] = ffma2(v[2 * j], make_float2(w4[o][j].x, w4[o][j].y), acc2[i][o]);
                        acc2[i][o] = ffma2(v[2 * j + 1], make_float2(w4[o][j].z, w4[o][j].w), acc2[i][o]);
                    }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
            float acc[O];
#pragma unroll
            for (int o = 0; o < O; ++o) {
                acc[o] = acc2[i][o].x + acc2[i][o].y;
                acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 1);
                acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 2);
                acc[o] += __shfl_xor_sync(0xffffffffu, acc[o], 4);
            }
            // lane `sub` finishes output channel `sub`
            float mine = acc[0];
#pragma unroll
            for (int o = 1; o < O; ++o) mine = sub == o ? acc[o] : mine;
            if (px[i] < a.pixels && sub < a.out_ch) {
                float t = mine + (a.bias ? __ldg(a.bias + sub) : 0.0f);
                t *= t > 0.0f ? a.gain : a.neg_slope_gain;
                t = fminf(fmaxf(t, -clampv), clampv);
                if constexpr (sizeof(T) == 2) yout[px[i] * a.out_ch + sub] = __float2half_rn(t); else yout[px[i] * a.out_ch + sub] = t;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------- host side
struct Plan {
    int parts, ma, sa, kg, n_tile, n_tiles, kc, chunks, b_stage, b_slot, sb, halo, persist, stage_bytes;
    long long packed_item_bytes, coef_bytes, packed_bytes, trans_bytes, total_bytes;
    int th, tw;                            // transposed-convolution intermediate (up = 2)
    int grid_h, grid_w;                    // pixel grid the windows tile
    TapPlan tp;
};

static int make_plan(const nfe_modconv_args& q, Plan& pl)
{
    NFE_REQUIRE(q.dtype == NFE_DTYPE_F32 || q.dtype == NFE_DTYPE_F16, "nfe_modulated_conv2d: dtype must be NFE_DTYPE_F32 or NFE_DTYPE_F16, got %d", q.dtype);
    NFE_REQUIRE(q.batch > 0 && q.in_ch > 0 && q.out_ch > 0 && q.in_h > 0 && q.in_w > 0, "nfe_modulated_conv2d: bad shape");
    NFE_REQUIRE(q.batch <= 65535, "nfe_modulated_conv2d: batch above 65535");
    NFE_REQUIRE(q.ksize == 1 || q.ksize == 3, "nfe_modulated_conv2d: kernel size must be 1 or 3 (the reference's layers), got %d", q.ksize);
    NFE_REQUIRE(q.up == 1 || (q.up == 2 && q.ksize == 3), "nfe_modulated_conv2d: up must be 1, or 2 with a 3x3 kernel, got up=%d k=%d", q.up, q.ksize);
    NFE_REQUIRE(q.in_ch % 16 == 0, "nfe_modulated_conv2d: in_channels must be a multiple of 16, got %d", q.in_ch);
    pl.parts = q.dtype == NFE_DTYPE_F16 ? 1 : 2;
    // plain: two 128-pixel accumulators x 256 columns (fp16) or one x 128 (fp32 split: the operand rings are twice as wide);
    // up = 2: a 128-pixel window, four phase accumulators x 128 columns.  512 columns of tensor memory either way.
    // N tile: 256 output channels wherever 512 columns of tensor memory allow it (an M = 128 MMA costs the same ~134+ cycles at N = 128
    // as at N = 256, see below); up = 2 needs four phase accumulators and stays at 128
    const int n_max = q.up == 1 ? 256 : 128;
    const int o16 = (q.out_ch + 15) / 16 * 16;
    if (o16 <= n_max) { pl.n_tile = o16; pl.n_tiles = 1; }
    else {
        NFE_REQUIRE(q.out_ch % 128 == 0, "nfe_modulated_conv2d: out_channels above %d must be a multiple of 128, got %d", n_max, q.out_ch);
        pl.n_tile = q.out_ch % n_max == 0 ? n_max : 128; pl.n_tiles = q.out_ch / pl.n_tile;
    }
    // CTA shape.  An MMA with M = 128 costs the tensor core at least ~125 cycles (its A-operand fetch) whatever N is, so
    //  * a tile of N <= 128 runs at half rate at best and the epilogue weighs twice as much: `twin` makes the CTA small enough (one
    //    128-pixel window, <= 113 KB of shared memory, <= 256 columns of tensor memory) for TWO CTAs per SM, whose main loops and
    //    epilogues overlap;
    //  * otherwise two 128-pixel windows share every weight stage (`pair`: two accumulators), which halves the weight stream per MMA;
    //  * a 1x1 convolution (ToRGB) has so little work per window that the per-CTA fixed cost dominates: two windows in fp16, never twin
    //    (in fp32 the register-path halo loader is its bottleneck and 64-channel chunks with one window measured fastest);
    //  * a layer whose 256-pixel windows would not even give every SM one CTA (the backbone's 4^2 .. 32^2 blocks) takes one window.
    // The split (fp32) operands need chunks of 32 channels for a wide tile, for twin CTAs and for window pairs: their hi + lo halo and
    // weight stages would not fit otherwise.
    const bool one_by_one = q.ksize == 1;
    const bool can32 = q.in_ch % 32 == 0;
    const long long ctas_256 = (long long)((q.in_h + 31) / 32) * ((q.in_w + TILE_W - 1) / TILE_W) * pl.n_tiles * q.batch;
    //  * a LARGE fp16 layer of N <= 128 does better still as persistent window pairs (below): two 128-column accumulators are half of
    //    tensor memory, so a persistent CTA has TWO sets and issues window k + 1 while the epilogue reads window k out — the overlap the
    //    twin CTAs give, plus shared weight stages and no per-window start-up (128->128 at 512^2: 0.77 -> 0.64 ms; with split operands
    //    the same change measured slower, fp32 SR head 5.64 -> 5.85 ms, so fp32 keeps the twins).
    const bool twin0 = q.up == 1 && pl.n_tile <= 128 && !one_by_one && (pl.parts == 1 || can32);
    const bool twin = twin0 && !(pl.parts == 1 && ctas_256 >= 3ll * sm_count());
    const bool pair = q.up == 1 && !twin && ((pl.parts == 1 && (ctas_256 >= sm_count() || one_by_one)) ||
                                             (pl.parts == 2 && can32 && !one_by_one && ctas_256 >= sm_count()));
    // (up = 2 with split operands: blocks of two taps are 64 KB at 64-channel chunks and the ring holds two; 32-channel chunks — five
    //  slots — measured slower: fp32 SR head 6.13 vs 5.82 ms, profiles/modconv_tuning_r02.txt #14)
    const bool split32 = pl.parts == 2 && can32 && (pl.n_tile > 128 || twin || pair);
    pl.kc = split32 ? 32 : (q.in_ch % 64 == 0 ? 64 : (can32 ? 32 : 16));
    if (pl.parts == 2 && pl.n_tile > 128 && !split32) {        // a wide split tile without 32-channel chunks: fall back to 128 columns
        NFE_REQUIRE(q.out_ch % 128 == 0 || o16 <= 128, "nfe_modulated_conv2d: fp32 needs in_channels to be a multiple of 32 for this out_channels");
        pl.n_tile = o16 <= 128 ? o16 : 128; pl.n_tiles = o16 <= 128 ? 1 : q.out_ch / 128;
    }
    pl.chunks = q.in_ch / pl.kc;
    pl.b_stage = pl.parts * pl.n_tile * pl.kc * 2;
    pl.ma = pair ? 2 : 1;
    pl.sa = (pl.parts == 1 && q.up == 2) ? 4 : 2;
    pl.kg = split32 ? 4 : 8;
    const int halo_h = 16 * pl.ma + 2, a_bytes = pl.sa * pl.parts * pl.kg * halo_h * HALO_W * 16;
    const int budget = twin ? (SMEM_BUDGET + TABLE_BYTES) / 2 - TABLE_BYTES - 1024 : SMEM_BUDGET;       // per-CTA reservation of 1 KB when two share an SM
    pl.halo = q.ksize == 3;
    TapPlan& p = pl.tp;
    p = TapPlan{};
    if (q.up == 1) {
        // conv2d_resample.py:137-139: correlation with the weight as stored (flip_weight) or flipped (conv2d_resample.py:36-37)
        p.taps = q.ksize * q.ksize;
        p.n_acc = pl.ma;
        for (int ky = 0, t = 0; ky < q.ksize; ++ky)
            for (int kx = 0; kx < q.ksize; ++kx, ++t) {
                p.dy[t] = ky - q.ksize / 2; p.dx[t] = kx - q.ksize / 2;
                p.ky[t] = q.flip_weight ? ky : q.ksize - 1 - ky; p.kx[t] = q.flip_weight ? kx : q.ksize - 1 - kx;
                p.acc_mask[t] = (1u << pl.ma) - 1u;
            }
        for (int m = 0; m < pl.ma; ++m) { p.row_off[m] = 16 * m; p.gh[m] = q.in_h; p.gw[m] = q.in_w; p.oy_off[m] = p.ox_off[m] = 0; }
        p.o_mul = 1;
        pl.grid_h = q.in_h; pl.grid_w = q.in_w;
        pl.th = pl.tw = 0;
    } else {
        // conv2d_resample.py:117-134: conv_transpose2d(stride 2): T[2 y + ky, 2 x + kx] += x[y, x] * w[ky, kx], so output rows of
        // parity py take ky = py (from y) and, for py = 0, also ky = 2 (from y - 1); the even phases have one more row / column
        pl.th = 2 * q.in_h + 1; pl.tw = 2 * q.in_w + 1;
        p.n_acc = 4;
        p.taps = 0;
        for (int ky = 0; ky < 3; ++ky)
            for (int kx = 0; kx < 3; ++kx) {
                const int t = p.taps++, py = ky & 1, px = kx & 1;
                p.dy[t] = -(ky / 2); p.dx[t] = -(kx / 2);
                // modulated_conv2d passes flip_weight on; conv2d_resample flips once more for the transposed op (:128)
                p.ky[t] = q.flip_weight ? 2 - ky : ky; p.kx[t] = q.flip_weight ? 2 - kx : kx;
                p.acc_mask[t] = 1u << (py * 2 + px);
            }
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px) {
                const int m = py * 2 + px;
                p.row_off[m] = 0; p.gh[m] = py == 0 ? q.in_h + 1 : q.in_h; p.gw[m] = px == 0 ? q.in_w + 1 : q.in_w; p.oy_off[m] = py; p.ox_off[m] = px;
            }
        p.o_mul = 2;
        pl.grid_h = q.in_h + 1; pl.grid_w = q.in_w + 1;
    }
    // weight blocks: taps in order; a tap takes along a later one that reads the same shifted window, feeds the next accumulator (same
    // window rows) and finds it in the same state (both fresh or both started) — see TapPlan.
    {
        auto single = [](unsigned m) { return m && !(m & (m - 1)); };
        auto bit = [](unsigned m) { int b = 0; while (!((m >> b) & 1u)) ++b; return b; };
        bool used[MAX_TAPS] = {};
        unsigned started = 0;
        int unit = 0;
        p.n_blk = 0;
        for (int t = 0; t < p.taps; ++t) {
            if (used[t]) continue;
            const int u = p.n_blk++;
            p.blk_tap[u] = t; p.blk_width[u] = 1; p.blk_unit[u] = unit; p.tap_blk[t] = u; p.tap_half[t] = 0;
            used[t] = true;
            // (split operands: a two-tap block is 64 KB at 64-channel chunks, the ring then holds two and the CTA cannot be persistent;
            //  merging still measured faster — fp32 SR head 5.52 vs 5.58 ms, 32->256 up=2 0.49 vs 0.55 ms)
            if (q.up == 2 && 2 * pl.n_tile <= 256 && single(p.acc_mask[t])) {
                const int m = bit(p.acc_mask[t]);
                for (int t2 = t + 1; t2 < p.taps && m + 1 < p.n_acc; ++t2) {
                    if (used[t2] || p.dy[t2] != p.dy[t] || p.dx[t2] != p.dx[t] || p.acc_mask[t2] != (1u << (m + 1))) continue;
                    if (p.row_off[m + 1] != p.row_off[m] || ((started >> m) & 1u) != ((started >> (m + 1)) & 1u)) continue;
                    // the pending narrower blocks between t and t2 must not touch accumulator m + 1 first: they are issued later
                    p.blk_width[u] = 2; p.tap_blk[t2] = u; p.tap_half[t2] = 1; used[t2] = true;
                    started |= 1u << (m + 1);
                    break;
                }
            }
            started |= p.acc_mask[t];
            unit += p.blk_width[u];
        }
    }
    {
        int widest = 1;
        for (int u = 0; u < p.n_blk; ++u) widest = std::max(widest, p.blk_width[u]);
        pl.b_slot = widest * pl.b_stage;
        pl.sb = std::min(MAX_SB, (budget - a_bytes) / pl.b_slot);
        NFE_REQUIRE(pl.sb >= 2, "nfe_modulated_conv2d: internal: weight ring does not fit");
        // epilogue stage: two warp groups x 128 rows of one 128-byte segment (+ 16 bytes of pitch)
        pl.stage_bytes = 2 * 128 * (std::min(pl.n_tile * (pl.parts == 1 ? 2 : 4), SEG_Q16 * 32) + 16);
        // Persistent CTAs (conv_gemm_kernel<..., PS = true>) where one CTA fills the SM anyway (twin CTAs overlap each other already),
        // every SM gets several windows, and the weight ring keeps three slots beside the stage region.
        const long long items = (long long)((q.up == 2 ? q.in_h + 1 : q.in_h) + 16 * pl.ma - 1) / (16 * pl.ma) *
                                (((q.up == 2 ? q.in_w + 1 : q.in_w) + TILE_W - 1) / TILE_W) * pl.n_tiles * q.batch;
        const int sb_ps = std::min(MAX_SB, (budget - a_bytes - pl.stage_bytes) / pl.b_slot);
        pl.persist = !twin && items >= 3ll * sm_count() && items < (1ll << 30) && sb_ps >= 3;
        if (pl.persist) pl.sb = sb_ps;
    }
    pl.packed_item_bytes = (long long)pl.n_tiles * pl.chunks * p.taps * pl.b_stage;
    auto up256 = [](long long v) { return (v + 255) / 256 * 256; };
    pl.coef_bytes = up256((long long)(q.batch * q.out_ch + q.out_ch + q.batch) * 4);
    pl.packed_bytes = up256(pl.packed_item_bytes * q.batch);
    pl.trans_bytes = q.up == 2 ? up256((long long)q.batch * pl.th * pl.tw * q.out_ch * (q.dtype == NFE_DTYPE_F16 ? 2 : 4)) : 0;
    pl.total_bytes = pl.coef_bytes + pl.packed_bytes + pl.trans_bytes;
    return 0;
}

template <int PARTS, int MA, int SA, int KG, bool PS = false>
static int launch_gemm(const GemmArgs& g, const Plan& pl, cudaStream_t stream)
{
    const int halo_h = 16 * MA + 2;
    // A ring | B ring | 22 mbarriers + the TMEM slot (256 bytes reserved) | bias table | tap tables | persistent: the epilogue's stage
    const size_t smem = (size_t)SA * PARTS * KG * halo_h * HALO_W * 16 + (size_t)pl.sb * pl.b_slot + TABLE_BYTES + (PS ? pl.stage_bytes : 0);
    static unsigned long long attr_done_mask = 0;         // per device: function attributes belong to the device's context
    int dev = 0;
    cudaGetDevice(&dev);
    const bool attr_done = dev < 64 && ((attr_done_mask >> dev) & 1ull);
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(conv_gemm_kernel<PARTS, MA, SA, KG, PS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_gemm_kernel<PARTS, MA, SA, KG, PS>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) { set_error("conv_gemm_kernel: shared memory opt-in: %s", cudaGetErrorString(e)); return 2; }
        if (dev < 64) attr_done_mask |= 1ull << dev;
    }
    if constexpr (PS) {
        const long long items = (long long)g.tiles_x * g.tiles_y * pl.n_tiles * g.batch;
        conv_gemm_kernel<PARTS, MA, SA, KG, true><<<(unsigned)std::min<long long>(items, sm_count()), PS_THREADS, smem, stream>>>(g);
    } else {
        const dim3 grid((unsigned)(g.tiles_x * g.tiles_y), (unsigned)pl.n_tiles, (unsigned)g.batch);
        conv_gemm_kernel<PARTS, MA, SA, KG><<<grid, THREADS, smem, stream>>>(g);
    }
    return check_launch("conv_gemm_kernel");
}

}  // namespace mc
}  // namespace nfe

using namespace nfe;

NFE_EXPORT int64_t nfe_modconv_workspace_bytes(const nfe_modconv_args* q)
{
    mc::Plan pl;
    if (!q || mc::make_plan(*q, pl)) return -1;
    return pl.total_bytes;
}

// Test hook (host only, no GPU needed): the CTA plan make_plan() derives for a layer, as integers —
// [0] parts [1] ma [2] sa [3] kg [4] n_tile [5] n_tiles [6] kc [7] chunks [8] sb [9] b_stage [10] b_slot [11] persist [12] stage_bytes
// [13] n_blk [14] taps [15] dynamic shared memory of the launch [16] CTAs per SM the kernel is built for [17 ..] width of each weight block
NFE_EXPORT int nfe_debug_modconv_plan(const nfe_modconv_args* q, int* out, int n_out)
{
    mc::Plan pl;
    if (!q || !out || n_out < 17 + mc::MAX_TAPS) return 1;
    if (int rc = mc::make_plan(*q, pl)) return rc;
    const int twin_shape = (!pl.persist && pl.ma == 1 && pl.sa == 2 && (pl.parts == 1 || pl.kg == 4)) ? 2 : 1;      // conv_gemm_kernel's __launch_bounds__
    const int v[17] = {pl.parts, pl.ma, pl.sa, pl.kg, pl.n_tile, pl.n_tiles, pl.kc, pl.chunks, pl.sb, pl.b_stage, pl.b_slot, pl.persist, pl.stage_bytes,
                       pl.tp.n_blk, pl.tp.taps,
                       pl.sa * pl.parts * pl.kg * (16 * pl.ma + 2) * mc::HALO_W * 16 + pl.sb * pl.b_slot + mc::TABLE_BYTES + (pl.persist ? pl.stage_bytes : 0), twin_shape};
    for (int i = 0; i < 17; ++i) out[i] = v[i];
    for (int u = 0; u < mc::MAX_TAPS; ++u) out[17 + u] = u < pl.tp.n_blk ? pl.tp.blk_width[u] : 0;
    return 0;
}

NFE_EXPORT int nfe_modulated_conv2d(const nfe_modconv_args* q, void* workspace, int64_t workspace_bytes, nfe_stream_t stream_)
{
    NFE_REQUIRE(q && q->x && q->weight && q->y, "nfe_modulated_conv2d: null pointer");
    NFE_REQUIRE(q->weight_batch_stride >= 0, "nfe_modulated_conv2d: negative weight_batch_stride");
    mc::Plan pl;
    if (int rc = mc::make_plan(*q, pl)) return rc;
    NFE_REQUIRE(workspace && workspace_bytes >= pl.total_bytes, "nfe_modulated_conv2d: workspace of %lld bytes needed, %lld given",
                (long long)pl.total_bytes, (long long)workspace_bytes);
    NFE_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0 && (reinterpret_cast<uintptr_t>(q->x) & 15) == 0, "nfe_modulated_conv2d: workspace must be 256-byte and x 16-byte aligned");
    NFE_REQUIRE(q->act >= 1 && q->act <= 3, "nfe_modulated_conv2d: the fused epilogue knows linear (1), relu (2) and lrelu (3), got act=%d", q->act);
    NFE_REQUIRE(q->up == 1 || (q->filter && q->fh >= 1 && q->fw >= 1 && q->fh * q->fw <= 64 && q->fh == q->fw), "nfe_modulated_conv2d: up = 2 needs a square resample filter of at most 8 x 8");
    const int vec = q->dtype == NFE_DTYPE_F16 ? 8 : 4;
    NFE_REQUIRE(q->up == 1 || q->out_ch % vec == 0, "nfe_modulated_conv2d: up = 2 needs out_channels to be a multiple of %d", vec);
    cudaStream_t stream = as_stream(stream_);
    if (q->ksize == 1 && q->up == 1 && q->out_ch <= 4 && !q->demodulate && !q->noise && q->in_ch <= 1024) {
        // ToRGB to a few channels: the streaming kernel (in_ch % 16 == 0 is checked by the plan above, so rows are whole 16-byte pieces)
        mc::RgbArgs r;
        r.x = q->x; r.weight = q->weight; r.styles = q->styles; r.bias = q->bias; r.y = q->y; r.weight_batch_stride = q->weight_batch_stride;
        r.batch = q->batch; r.in_ch = q->in_ch; r.out_ch = q->out_ch; r.pixels = (long long)q->in_h * q->in_w;
        const float neg_slope = q->act == 1 ? 1.0f : (q->act == 2 ? 0.0f : q->alpha);
        r.gain = q->gain; r.neg_slope_gain = q->gain * neg_slope; r.clamp = q->clamp;
        const int v = q->dtype == NFE_DTYPE_F16 ? 8 : 4;
        const int o = q->out_ch <= 3 ? 3 : 4;
        const size_t smem = (size_t)(q->in_ch / v) * mc::rgb_piece_stride(v, o) * sizeof(float);     // <= 20 KB at in_ch <= 1024
        const dim3 grid((unsigned)std::min<long long>((r.pixels + 63) / 64, (long long)sm_count() * 8 / std::max(1, std::min(q->batch, 8)) + 1), q->batch);
        if (q->dtype == NFE_DTYPE_F16) {
            if (o == 3) mc::torgb_small_kernel<__half, 3><<<grid, 256, smem, stream>>>(r); else mc::torgb_small_kernel<__half, 4><<<grid, 256, smem, stream>>>(r);
        } else {
            if (o == 3) mc::torgb_small_kernel<float, 3><<<grid, 256, smem, stream>>>(r); else mc::torgb_small_kernel<float, 4><<<grid, 256, smem, stream>>>(r);
        }
        NFE_LAUNCH_CHECK("torgb_small_kernel");
        return 0;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* coef = reinterpret_cast<float*>(ws);
    unsigned char* packed = ws + pl.coef_bytes;
    void* trans = ws + pl.coef_bytes + pl.packed_bytes;

    mc::PackArgs pa;
    pa.weight = q->weight; pa.weight_batch_stride = q->weight_batch_stride; pa.styles = q->styles; pa.dcoef = coef; pa.wmul = coef + (long long)q->batch * q->out_ch; pa.smax = pa.wmul + q->out_ch;
    pa.packed = packed; pa.packed_item_stride = pl.packed_item_bytes;
    pa.batch = q->batch; pa.out_ch = q->out_ch; pa.in_ch = q->in_ch; pa.ksize = q->ksize; pa.demodulate = q->demodulate;
    pa.prenorm = (q->dtype == NFE_DTYPE_F16 && q->demodulate) ? 1 : 0;                     // networks_stylegan2.py:55-57
    pa.parts = pl.parts; pa.n_tile = pl.n_tile; pa.n_tiles = pl.n_tiles; pa.chunks = pl.chunks; pa.kc = pl.kc; pa.b_stage = pl.b_stage;
    pa.tp = pl.tp;
    // Split operands (fp32) with one weight for the batch: pack W ONCE and let the GEMM carry the style (on the activations, in the halo
    // loader) and the demodulation coefficient (on the accumulator, in the epilogue) — the reference's non-fused formulation,
    // networks_stylegan2.py:69-79, equal to the fused one up to fp32 rounding order.  The per-item pack wrote batch x the weight tensor
    // (hi + lo) per layer call: 0.47 ms of a 5.2 ms fp32 backbone pass.
    const bool shared = pl.parts == 2 && q->weight_batch_stride == 0 && q->batch > 1 && (reinterpret_cast<uintptr_t>(q->styles) & 15) == 0;
    pa.shared = shared ? 1 : 0;
    NFE_REQUIRE(q->in_ch <= 8192, "nfe_modulated_conv2d: in_channels above 8192");
    mc::modconv_coef_kernel<<<q->out_ch, 128, (size_t)q->in_ch * sizeof(float), stream>>>(pa);
    NFE_LAUNCH_CHECK("modconv_coef_kernel");
    const long long slots = (long long)pl.n_tiles * pl.chunks * (pl.kc / 8) * pl.n_tile * (pl.tp.taps % 3 == 0 ? 3 : 1);
    mc::modconv_pack_kernel<<<dim3((unsigned)((slots + 255) / 256), shared ? 1 : q->batch), 256, 0, stream>>>(pa);
    NFE_LAUNCH_CHECK("modconv_pack_kernel");

    mc::GemmArgs g;
    g.x = q->x; g.packed = packed; g.packed_item_stride = shared ? 0 : pl.packed_item_bytes;
    g.in_scale = shared ? q->styles : nullptr; g.out_scale = (shared && q->demodulate) ? coef : nullptr;
    g.batch = q->batch; g.in_h = q->in_h; g.in_w = q->in_w; g.in_ch = q->in_ch; g.out_ch = q->out_ch;
    g.n_tile = pl.n_tile; g.n_tiles = pl.n_tiles; g.chunks = pl.chunks; g.kc = pl.kc; g.sb = pl.sb; g.b_stage = pl.b_stage; g.b_slot = pl.b_slot; g.halo = pl.halo;
    {   // the epilogue stages two 128-pixel tiles in the operand rings when they fit
        const long long rings = (long long)pl.sa * pl.parts * pl.kg * (16 * pl.ma + 2) * mc::HALO_W * 16 + (long long)pl.sb * pl.b_slot;
        // rows are staged in segments of SEG_Q16 16-column fp16 groups (128 bytes), one 128-row buffer per epilogue warp group that has an accumulator
        g.stage_ok = (pl.persist || pl.stage_bytes <= rings) ? 1 : 0;
    }
    g.tp = pl.tp;
    g.tiles_x = (pl.grid_w + mc::TILE_W - 1) / mc::TILE_W; g.tiles_y = (pl.grid_h + 16 * pl.ma - 1) / (16 * pl.ma);
    if (q->up == 1) {
        g.y = q->y; g.ys_w = q->out_ch; g.ys_h = (long long)q->in_w * q->out_ch; g.ys_n = (long long)q->in_h * g.ys_h;
        g.noise = q->noise; g.noise_n = q->noise_batch_stride; g.noise_w = q->in_w; g.bias = q->bias;
        g.act = q->act; g.alpha = q->alpha; g.gain = q->gain; g.clamp = q->clamp;
    } else {
        g.y = trans; g.ys_w = q->out_ch; g.ys_h = (long long)pl.tw * q->out_ch; g.ys_n = (long long)pl.th * g.ys_h;
        g.noise = nullptr; g.noise_n = 0; g.noise_w = 0; g.bias = nullptr; g.act = 1; g.alpha = 0.0f; g.gain = 1.0f; g.clamp = -1.0f;
    }
    int rc;
    if (pl.persist)
        rc = pl.parts == 2 ? (pl.kg == 4 ? (pl.ma == 2 ? mc::launch_gemm<2, 2, 2, 4, true>(g, pl, stream) : mc::launch_gemm<2, 1, 2, 4, true>(g, pl, stream))
                                         : mc::launch_gemm<2, 1, 2, 8, true>(g, pl, stream))
             : (pl.ma == 2 ? mc::launch_gemm<1, 2, 2, 8, true>(g, pl, stream)
                           : (pl.sa == 4 ? mc::launch_gemm<1, 1, 4, 8, true>(g, pl, stream) : mc::launch_gemm<1, 1, 2, 8, true>(g, pl, stream)));
    else
        rc = pl.parts == 2 ? (pl.kg == 4 ? (pl.ma == 2 ? mc::launch_gemm<2, 2, 2, 4>(g, pl, stream) : mc::launch_gemm<2, 1, 2, 4>(g, pl, stream))
                                         : mc::launch_gemm<2, 1, 2, 8>(g, pl, stream))
             : (pl.ma == 2 ? mc::launch_gemm<1, 2, 2, 8>(g, pl, stream)
                           : (pl.sa == 4 ? mc::launch_gemm<1, 1, 4, 8>(g, pl, stream) : mc::launch_gemm<1, 1, 2, 8>(g, pl, stream)));
    if (rc) return rc;
    if (q->up == 2) {
        // conv2d_resample.py:97-101,124-131 with padding = k/2 as the layers pass it: the filter pass pads the (2H+1) image by
        // p0 = k/2 + (f+1)/2 - (k-1) before and p1 = k/2 + (f-2)/2 - (k-2) after, gain up^2, and yields 2H x 2W
        mc::FinishArgs f;
        f.t = trans; f.y = q->y; f.f = q->filter; f.noise = q->noise; f.noise_n = q->noise_batch_stride; f.bias = q->bias;
        f.batch = q->batch; f.th = pl.th; f.tw = pl.tw; f.oh = 2 * q->in_h; f.ow = 2 * q->in_w; f.c = q->out_ch; f.fh = q->fh; f.fw = q->fw;
        const int pad0 = q->ksize / 2 + (q->fw + 1) / 2 - (q->ksize - 1), pad1 = q->ksize / 2 + (q->fw - 2) / 2 - (q->ksize - 2);
        NFE_REQUIRE(pl.th + pad0 + pad1 - q->fh + 1 == f.oh, "nfe_modulated_conv2d: a %d-tap resample filter does not yield a 2x image", q->fw);
        f.pad_y0 = f.pad_x0 = pad0; f.flip = 0; f.fgain = 4.0f;
        f.act = q->act; f.alpha = q->alpha; f.gain = q->gain; f.clamp = q->clamp;
        const int slices = (q->out_ch + 8 * vec - 1) / (8 * vec);
        if (q->fh <= 4 && q->fw <= 4 && (long long)q->batch * slices <= 65535) {
            const int tiles_x = (f.ow + mc::FT - 1) / mc::FT, tiles_y = (f.oh + mc::FT - 1) / mc::FT;
            const dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)(q->batch * slices));
            if (q->dtype == NFE_DTYPE_F16) mc::upfir_finish_tiled_kernel<__half><<<grid, 256, 0, stream>>>(f, tiles_x, tiles_y, slices);
            else mc::upfir_finish_tiled_kernel<float><<<grid, 256, 0, stream>>>(f, tiles_x, tiles_y, slices);
            NFE_LAUNCH_CHECK("upfir_finish_tiled_kernel");
        } else {
            const long long work = (long long)q->batch * f.oh * f.ow * (q->out_ch / vec);
            const int blocks = (int)std::min<long long>((work + 255) / 256, (long long)sm_count() * 16);
            if (q->dtype == NFE_DTYPE_F16) mc::upfir_finish_kernel<__half><<<blocks, 256, 0, stream>>>(f);
            else mc::upfir_finish_kernel<float><<<blocks, 256, 0, stream>>>(f);
            NFE_LAUNCH_CHECK("upfir_finish_kernel");
        }
    }
    return 0;
}

#ifdef NFE_MC_PROFILE
// debug builds only: where the roles of conv_gemm_kernel wait (profiles/modconv_role_profile.py)
NFE_EXPORT int nfe_debug_modconv_profile(unsigned long long* out16, int reset)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out16, mc::g_mc_prof, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {}; cudaMemcpyToSymbol(mc::g_mc_prof, z, sizeof(z)); }
    return 0;
}
#endif

// Bilinear sampler (tf.contrib.resampler semantics, SURVEY.md 8(a) S0-S2) for sm_100a.
//
//   forward / grad_warp : one CTA per 1024-pixel OUTPUT tile.  The CTA loads its flow
//     vectors (coalesced float2), forms warp = flow + grid in registers, reduces the
//     bounding box of the taps it needs, stages that SOURCE window into shared memory, then
//     gathers the four taps from shared memory.  When the window does not fit (arbitrary
//     warps) it gathers straight from global (L1/L2).  The arithmetic uses non-contracted
//     fp32 ops in the reference's summation order, so the forward values and grad_warp are
//     bit-equal to the NumPy oracle.  Two forms:
//       sampler_tma_kernel  (C in {1,3,4}, 16-byte aligned rows -- the training path): window,
//         grad_out / target tiles and the output tile move by TMA; MODE 2 fuses forward, the
//         reconstruction loss and grad_warp into one pass (dmv_sampler_loss_fused);
//       sampler_tile_kernel (any C <= 16, any alignment, 1-D sample lists): cp.async staging,
//         predicated taps.
//     Both forms also serve the shared-source entry points (dmv_sampler_fwd_shared_src, dmv_sampler_grad_flow_shared_src,
//     dmv_sampler_loss_fused_shared_src), where output sample b reads source image b / group (one source, many
//     viewpoints): a tile still reads exactly one source image.
//   grad_data : owner-computes scatter.  One CTA owns a 32x16 SOURCE tile; it visits every
//     32-pixel warp chunk of the output whose tap box intersects it (two-level box table from a
//     pre-pass), and each warp accumulates into a warp-private shared-memory copy of the tile.
//     Lanes whose samples share a floor cell are serialised by lane rank (one __match_any_sync
//     per sample), warps are summed in warp order, and every grad_data element is written
//     exactly once: no atomics, no memset, same inputs -> same bits.
//
// HBM-bound: algorithmic bytes per output pixel are 8 + 8C (fwd), 16 + 8C (grad_warp only),
// 8 + 8C (grad_data pass).
#include "tc_common.cuh"

namespace {

using namespace dmv;

// tuning knobs (tools/sampler_variants.sh sweeps them; the defaults are the measured best)
#ifndef SAMPLER_MINBLOCKS
#define SAMPLER_MINBLOCKS 5
#endif
#ifndef SAMPLER_CPASYNC
#define SAMPLER_CPASYNC 16     // 0: ld.global + st.shared, 4: cp.async 4-byte, 16: cp.async 16-byte on an aligned window
#endif
#ifndef SAMPLER_PREREDUCE
#define SAMPLER_PREREDUCE 1   // reduce the tap box over a thread's pixels before the warp reduction
#endif
#ifndef SAMPLER_STAGE_KB
#define SAMPLER_STAGE_KB 40
#endif
#ifndef SAMPLER_TMA
#define SAMPLER_TMA 1          // route image-shaped C in {1,3,4} calls to sampler_tma_kernel
#endif
#ifndef SAMPLER_TMA_MINBLOCKS
#define SAMPLER_TMA_MINBLOCKS 5
#endif
#ifndef SAMPLER_TMA_MINBLOCKS_FWD3
#define SAMPLER_TMA_MINBLOCKS_FWD3 6   // the RGB forward kernel fits 42 registers: a sixth CTA per SM
#endif
// Source window boxes of the TMA kernel, pixels per side.  The row pitch of the staged window is box * C floats, and the
// bank of a tap is (pitch * row + C * col + c) mod 32: with 48 pixels of RGB the pitch is 144 = 16 mod 32, so rows two
// apart collide, and the lanes of a warp read 32 different rows under the reference's (Y,X) grid.  44 pixels (pitch 132 =
// 4 mod 32) spread eight consecutive rows over the banks, and fetch 16 % fewer bytes per tile
// (profiles/r02_sampler_window_variants.txt: 33.1 -> 31.2 us forward, 35.4 -> 33.0 us grad_flow under +-3 pixel jitter).
#ifndef SAMPLER_BOX
#define SAMPLER_BOX 36         // first box: clipped edge tiles, small displacements
#endif
#ifndef SAMPLER_BOX_L
#define SAMPLER_BOX_L 44       // second, larger box tried when the tap box does not fit the first
#endif
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kTilePix = 1024;
constexpr int kPPT = kTilePix / kThreads;  // pixels per thread
constexpr int kStageFloats = SAMPLER_STAGE_KB * 256;   // source window in floats
constexpr int kSrcTileW = 32, kSrcTileH = 16;

struct Geom {
    int B, H, W, C, Ho, Wo;   // B: output samples
    int group;     // output sample b reads source image b / group (the *_shared_src entry points); 1 elsewhere
    int tw_shift;  // output tile is (1024 >> tw_shift) rows x (1 << tw_shift) cols
    int tiles_x, tiles_y;
    unsigned flags;
};

struct Sample {
    float x, y;
    bool valid;
};

// warp = flow + grid (tf_utils.py:35-52, fused) and the resampler's validity rule for one sample
__device__ __forceinline__ Sample make_sample(float2 f, const Geom& g, int i, int j) {
    Sample s;
    s.x = f.x;
    s.y = f.y;
    if (g.flags & DMV_SAMPLER_ADD_GRID) {
        if (g.flags & DMV_SAMPLER_GRID_XY) {
            s.x = __fadd_rn(f.x, (float)j);
            s.y = __fadd_rn(f.y, (float)i);
        } else {  // reference (Y,X) order: channel 0 += row index, channel 1 += column index
            s.x = __fadd_rn(f.x, (float)i);
            s.y = __fadd_rn(f.y, (float)j);
        }
    }
    s.valid = (s.x > -1.0f) && (s.y > -1.0f) && (s.x < (float)g.W) && (s.y < (float)g.H);
    return s;
}

__device__ __forceinline__ Sample load_sample(const float* __restrict__ wf, const Geom& g, int b, int i, int j) {
    return make_sample(__ldg(reinterpret_cast<const float2*>(wf) + ((long long)b * g.Ho + i) * g.Wo + j), g, i, j);
}

__device__ __forceinline__ void tile_origin(const Geom& g, int tile, int& b, int& i0, int& j0) {
    const int per_img = g.tiles_x * g.tiles_y;
    b = tile / per_img;
    const int t = tile - b * per_img;
    const int ty = t / g.tiles_x;
    const int tx = t - ty * g.tiles_x;
    i0 = ty * (kTilePix >> g.tw_shift);
    j0 = tx << g.tw_shift;
}

// Reduce the tap bounding box of a tile into s_box = {xmin, xmax, ymin, ymax} (clipped to the image).
[[maybe_unused]] __device__ __forceinline__ void reduce_box(int* s_box, bool valid, int fx, int fy, int W, int H) {
    int xlo = 0x7fffffff, xhi = -0x7fffffff, ylo = 0x7fffffff, yhi = -0x7fffffff;
    if (valid) {
        xlo = max(fx, 0);
        xhi = min(fx + 1, W - 1);
        ylo = max(fy, 0);
        yhi = min(fy + 1, H - 1);
    }
    xlo = __reduce_min_sync(0xffffffffu, xlo);
    xhi = __reduce_max_sync(0xffffffffu, xhi);
    ylo = __reduce_min_sync(0xffffffffu, ylo);
    yhi = __reduce_max_sync(0xffffffffu, yhi);
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&s_box[0], xlo);
        atomicMax(&s_box[1], xhi);
        atomicMin(&s_box[2], ylo);
        atomicMax(&s_box[3], yhi);
    }
}

// MODE 0: forward.  MODE 1: grad wrt warp/flow.
__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int CT, int MODE>
__global__ void __launch_bounds__(kThreads, SAMPLER_MINBLOCKS) sampler_tile_kernel(
    const float* __restrict__ data, const float* __restrict__ wf, const float* __restrict__ grad_out,
    float* __restrict__ out, int32_t* __restrict__ dbg_idx, uint8_t* __restrict__ dbg_mask, Geom g) {
    extern __shared__ float s_win[];
    __shared__ int s_box[4];
    __shared__ int s_row0;
    const int C = CT ? CT : g.C;
    const int tid = threadIdx.x;
    int b, i0, j0;
    tile_origin(g, blockIdx.x, b, i0, j0);
    if (tid < 4) s_box[tid] = (tid & 1) ? -0x7fffffff : 0x7fffffff;
    // first source row of the tile's image: b / group (group = 1 unless the source is shared).  Kept in shared memory and
    // read where it is used: one more live register costs this kernel spills at its 48-register bound.
    if (tid == 0) s_row0 = (b / g.group) * g.H;
    __syncthreads();

    Sample smp[kPPT];
    int pi[kPPT], pj[kPPT];
    bool inb[kPPT];
    const int tw_mask = (1 << g.tw_shift) - 1;
#if SAMPLER_PREREDUCE
    int bxlo = 0x7fffffff, bxhi = -0x7fffffff, bylo = 0x7fffffff, byhi = -0x7fffffff;
#endif
#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        const int p = k * kThreads + tid;
        pi[k] = i0 + (p >> g.tw_shift);
        pj[k] = j0 + (p & tw_mask);
        inb[k] = (pi[k] < g.Ho) && (pj[k] < g.Wo);
        smp[k].valid = false;
        smp[k].x = smp[k].y = 0.f;
        if (inb[k]) smp[k] = load_sample(wf, g, b, pi[k], pj[k]);
        const int fx = smp[k].valid ? (int)floorf(smp[k].x) : 0;
        const int fy = smp[k].valid ? (int)floorf(smp[k].y) : 0;
#if SAMPLER_PREREDUCE
        if (smp[k].valid) {
            bxlo = min(bxlo, max(fx, 0)); bxhi = max(bxhi, min(fx + 1, g.W - 1));
            bylo = min(bylo, max(fy, 0)); byhi = max(byhi, min(fy + 1, g.H - 1));
        }
#else
        reduce_box(s_box, smp[k].valid, fx, fy, g.W, g.H);
#endif
    }
#if SAMPLER_PREREDUCE
    bxlo = __reduce_min_sync(0xffffffffu, bxlo); bxhi = __reduce_max_sync(0xffffffffu, bxhi);
    bylo = __reduce_min_sync(0xffffffffu, bylo); byhi = __reduce_max_sync(0xffffffffu, byhi);
    if ((tid & 31) == 0) {
        atomicMin(&s_box[0], bxlo); atomicMax(&s_box[1], bxhi);
        atomicMin(&s_box[2], bylo); atomicMax(&s_box[3], byhi);
    }
#endif
    __syncthreads();
    const int xmin = s_box[0], xmax = s_box[1], ymin = s_box[2], ymax = s_box[3];
    const bool any_valid = xmin <= xmax;
    const int nx = xmax - xmin + 1, ny = ymax - ymin + 1;
#if SAMPLER_CPASYNC == 16
    // window start rounded down to 16 bytes (rows are 16-byte aligned when W*C % 4 == 0); pitch = 4 mod 8 floats
    const bool vec16 = (((g.W * C) & 3) == 0) && ((reinterpret_cast<uintptr_t>(data) & 15) == 0);
    const int a0 = vec16 ? ((xmin * C) & ~3) : xmin * C;
    const int seg = vec16 ? ((((xmax + 1) * C - a0) + 3) & ~3) : (nx * C);
    const int pitch = vec16 ? (seg | 4) : (seg | 1);
#else
    const int a0 = xmin * C;
    const int seg = nx * C;
    const int pitch = seg | 1;  // odd pitch: a column read by 32 lanes hits 32 banks
#endif
    const bool staged = any_valid && ((long long)ny * pitch <= kStageFloats);
    if (staged) {
        const int warp = tid >> 5, lane = tid & 31;
        const int row0 = s_row0;
        for (int r = warp; r < ny; r += kWarps) {
            const float* src = data + ((long long)row0 + ymin + r) * g.W * C + a0;
            float* dst = s_win + r * pitch;
#if SAMPLER_CPASYNC == 16
            if (vec16) { for (int e = lane * 4; e < seg; e += 128) cp_async16(dst + e, src + e); }
            else { for (int e = lane; e < seg; e += 32) cp_async4(dst + e, src + e); }
#elif SAMPLER_CPASYNC == 4
            for (int e = lane; e < seg; e += 32) cp_async4(dst + e, src + e);
#else
            for (int e = lane; e < seg; e += 32) dst[e] = __ldg(src + e);
#endif
        }
#if SAMPLER_CPASYNC
        cp_async_wait_all();
#endif
    }
    __syncthreads();

#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        if (!inb[k]) continue;
        const long long opix = ((long long)b * g.Ho + pi[k]) * g.Wo + pj[k];
        const Sample s = smp[k];
        int fx = 0, fy = 0, cx = 0, cy = 0;
        unsigned mask = 0;
        float dx = 0.f, dy = 0.f;
        if (s.valid) {
            fx = (int)floorf(s.x);
            fy = (int)floorf(s.y);
            cx = fx + 1;
            cy = fy + 1;
            dx = __fsub_rn((float)cx, s.x);
            dy = __fsub_rn((float)cy, s.y);
            const bool fxi = fx >= 0, cxi = cx <= g.W - 1, fyi = fy >= 0, cyi = cy <= g.H - 1;
            mask = 1u | ((fxi && fyi) ? 2u : 0u) | ((cxi && cyi) ? 4u : 0u) | ((fxi && cyi) ? 8u : 0u) |
                   ((cxi && fyi) ? 16u : 0u);
        }
        if (MODE == 0) {
            if (dbg_idx) reinterpret_cast<int4*>(dbg_idx)[opix] = make_int4(fx, fy, cx, cy);
            if (dbg_mask) dbg_mask[opix] = (uint8_t)mask;
        }
        const float omdx = __fsub_rn(1.0f, dx), omdy = __fsub_rn(1.0f, dy);
        const float w_ff = __fmul_rn(dx, dy), w_cc = __fmul_rn(omdx, omdy), w_fc = __fmul_rn(dx, omdy),
                    w_cf = __fmul_rn(omdx, dy);
        // base offsets of the four taps (shared window or global)
        long long o_ff, o_cc, o_fc, o_cf;
        const float* base;
        if (staged) {
            base = s_win;
            o_ff = (long long)(fy - ymin) * pitch + (fx * C - a0);
            o_cf = o_ff + C;
            o_fc = o_ff + pitch;
            o_cc = o_fc + C;
        } else {
            base = data;
            o_ff = (((long long)s_row0 + fy) * g.W + fx) * C;
            o_cf = o_ff + C;
            o_fc = o_ff + (long long)g.W * C;
            o_cc = o_fc + C;
        }
        float gw0 = 0.f, gw1 = 0.f;
#pragma unroll
        for (int c = 0; c < (CT ? CT : 16); ++c) {
            if (!CT && c >= C) break;
            float p_ff = 0.f, p_cc = 0.f, p_fc = 0.f, p_cf = 0.f;
            if (mask & 2u) p_ff = base[o_ff + c];
            if (mask & 4u) p_cc = base[o_cc + c];
            if (mask & 8u) p_fc = base[o_fc + c];
            if (mask & 16u) p_cf = base[o_cf + c];
            if (MODE == 0) {
                float v = __fmul_rn(w_ff, p_ff);
                v = __fadd_rn(v, __fmul_rn(w_cc, p_cc));
                v = __fadd_rn(v, __fmul_rn(w_fc, p_fc));
                v = __fadd_rn(v, __fmul_rn(w_cf, p_cf));
                out[opix * C + c] = s.valid ? v : 0.f;
            } else {
                const float gc = s.valid ? __ldg(grad_out + opix * C + c) : 0.f;
                const float a0 = __fadd_rn(__fmul_rn(omdy, __fsub_rn(p_cc, p_fc)), __fmul_rn(dy, __fsub_rn(p_cf, p_ff)));
                const float a1 = __fadd_rn(__fmul_rn(omdx, __fsub_rn(p_cc, p_cf)), __fmul_rn(dx, __fsub_rn(p_fc, p_ff)));
                gw0 = __fadd_rn(gw0, __fmul_rn(gc, a0));
                gw1 = __fadd_rn(gw1, __fmul_rn(gc, a1));
            }
        }
        if (MODE == 1) reinterpret_cast<float2*>(out)[opix] = s.valid ? make_float2(gw0, gw1) : make_float2(0.f, 0.f);
    }
}

// ---------------------------------------------------------------------------------------------
// TMA kernel: the training-path form of forward / grad_warp for image-shaped outputs with C in
// {1,3,4} and 16-byte aligned rows.  Same arithmetic (same bits) as sampler_tile_kernel, but all bulk
// movement is done by the TMA engine so the LSU pipe only carries the flow loads and the tap gathers:
//   * the SOURCE WINDOW of the tile (tap bounding box, reduced from the flow) is one
//     cp.async.bulk.tensor box load in EXTENDED coordinates: the box may start at x = -1 / y = -1
//     and run past W / H, and TMA's out-of-bounds zero fill is exactly the resampler's one-pixel zero
//     border -- taps need no in-range predicates (w * 0 = +0 leaves the sum's bits unchanged);
//   * MODE 0 writes its results to a shared tile that one bulk tensor STORE sends to global (ragged
//     edges are clipped by the tensor map); MODE 1 receives grad_out the same way (bulk load);
//   * lanes own consecutive pixels of a row: scalar LDS/STS at stride C are bank-conflict-free for
//     smooth flows, flow loads / grad_flow stores are coalesced 8-byte accesses.
// floats reserved for the source window: the tiles behind it are bulk-tensor destinations / sources (128-byte aligned)
__host__ __device__ constexpr int win_floats(int C) { return (SAMPLER_BOX_L * SAMPLER_BOX_L * C + 31) & ~31; }
constexpr int kBoxS = SAMPLER_BOX, kBoxL = SAMPLER_BOX_L;   // source window box (pixels); tap boxes beyond the larger one fall back to global gathers

// MODE 2 (training step): forward + reconstruction loss + grad wrt flow in ONE pass -- the warped tile never leaves
// the SM between the three: gen is stored for the caller, d = gen - target feeds the loss partial and, through
// dL/dgen = inv_count * w_c * (2 d | sign d), the flow gradient from the taps that are still in shared memory.
// Per-CTA loss partials (double) are summed in index order by the last CTA (all its threads, fixed tree).
struct FuseArgs {
    float w[4];
    float inv_count;
    int mode;
    double* partials;
    unsigned* counter;
    float* loss_out;
    float* grad_wf;
};

template <int C, int MODE>
__global__ void __launch_bounds__(kThreads, (C == 3 && MODE == 0) ? SAMPLER_TMA_MINBLOCKS_FWD3 : SAMPLER_TMA_MINBLOCKS) sampler_tma_kernel(
    const __grid_constant__ CUtensorMap map_src, const __grid_constant__ CUtensorMap map_src_l,
    const __grid_constant__ CUtensorMap map_io, const __grid_constant__ CUtensorMap map_tgt, const float* __restrict__ data,
    const float* __restrict__ wf, float* __restrict__ out, int32_t* __restrict__ dbg_idx, uint8_t* __restrict__ dbg_mask, Geom g,
    const FuseArgs fa) {
    extern __shared__ __align__(128) float s_dyn[];
    float* s_win = s_dyn;                              // [box][box * C], box = kBoxS or kBoxL
    float* s_io = s_dyn + win_floats(C);               // [32][32 * C]: MODE 0/2 results, MODE 1 grad_out
    float* s_tgt = s_io + 32 * 32 * C;                 // MODE 2: target tile
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ int s_box[4];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int b, i0, j0;
    tile_origin(g, blockIdx.x, b, i0, j0);
    const int bs = b / g.group;    // source image of the tile
    if (tid < 4) s_box[tid] = (tid & 1) ? -0x7fffffff : 0x7fffffff;
    if (tid == 0) {
        tc::mbar_init(&s_bar[0], 1);
        tc::mbar_init(&s_bar[1], 1);
        tc::fence_barrier_init();
        tc::fence_proxy_async();
        if (MODE == 1) {
            tc::mbar_expect_tx(&s_bar[1], 32 * 32 * C * 4);
            tc::tma_load_3d(s_io, &map_io, &s_bar[1], j0 * C, i0, b);
        }
        if (MODE == 2) {
            tc::mbar_expect_tx(&s_bar[1], 32 * 32 * C * 4);
            tc::tma_load_3d(s_tgt, &map_tgt, &s_bar[1], j0 * C, i0, b);
        }
    }
    __syncthreads();

    const int j = j0 + lane;
    float loss_acc = 0.f;
    float sx[kPPT], sy[kPPT];
    bool valid[kPPT];
    int fx[kPPT], fy[kPPT];
    int bxlo = 0x7fffffff, bxhi = -0x7fffffff, bylo = 0x7fffffff, byhi = -0x7fffffff;
    const float fW = (float)g.W, fH = (float)g.H;
    const long long img_pix = (long long)b * g.Ho * g.Wo;
#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        const int i = i0 + warp + k * kWarps;
        const bool inb = (i < g.Ho) && (j < g.Wo);
        float2 f = make_float2(0.f, 0.f);
        if (inb) f = __ldg(reinterpret_cast<const float2*>(wf) + img_pix + (long long)i * g.Wo + j);
        sx[k] = f.x; sy[k] = f.y;
        if (g.flags & DMV_SAMPLER_ADD_GRID) {
            if (g.flags & DMV_SAMPLER_GRID_XY) {
                sx[k] = __fadd_rn(f.x, (float)j);
                sy[k] = __fadd_rn(f.y, (float)i);
            } else {
                sx[k] = __fadd_rn(f.x, (float)i);
                sy[k] = __fadd_rn(f.y, (float)j);
            }
        }
        valid[k] = inb && (sx[k] > -1.0f) && (sy[k] > -1.0f) && (sx[k] < fW) && (sy[k] < fH);
        fx[k] = valid[k] ? __float2int_rd(sx[k]) : 0;
        fy[k] = valid[k] ? __float2int_rd(sy[k]) : 0;
        if (valid[k]) {
            bxlo = min(bxlo, fx[k]); bxhi = max(bxhi, fx[k] + 1);
            bylo = min(bylo, fy[k]); byhi = max(byhi, fy[k] + 1);
        }
    }
    bxlo = __reduce_min_sync(0xffffffffu, bxlo); bxhi = __reduce_max_sync(0xffffffffu, bxhi);
    bylo = __reduce_min_sync(0xffffffffu, bylo); byhi = __reduce_max_sync(0xffffffffu, byhi);
    if (lane == 0) {
        atomicMin(&s_box[0], bxlo); atomicMax(&s_box[1], bxhi);
        atomicMin(&s_box[2], bylo); atomicMax(&s_box[3], byhi);
    }
    __syncthreads();
    // tap box in EXTENDED coordinates (-1 .. W, -1 .. H)
    const int xlo = s_box[0], xhi = s_box[1], ylo = s_box[2], yhi = s_box[3];
    const bool any_valid = xlo <= xhi;
    // the box must start on a 16-byte boundary of the row: x origin floored to 4 pixels unless C == 4 (-1 -> -4)
    const int xa = (C == 4) ? xlo : (xlo & ~3);
    const int span = max(xhi - xa, yhi - ylo);
    const bool staged = any_valid && (span < kBoxL);
    const int box = (span < kBoxS) ? kBoxS : kBoxL;   // smallest box that holds the taps
    const int kPitch = box * C;
    if (staged) {
        if (tid == 0) {
            tc::mbar_expect_tx(&s_bar[0], box * box * C * 4);
            tc::tma_load_3d(s_win, span < kBoxS ? &map_src : &map_src_l, &s_bar[0], xa * C, ylo, bs);
        }
        tc::mbar_wait(&s_bar[0], 0);
    }
    if (MODE >= 1) tc::mbar_wait(&s_bar[1], 0);

#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        const int r = warp + k * kWarps;              // row of the tile
        const int i = i0 + r;
        const bool inb = (i < g.Ho) && (j < g.Wo);
        const int cx = fx[k] + 1, cy = fy[k] + 1;
        const float dx = valid[k] ? __fsub_rn((float)cx, sx[k]) : 0.f;
        const float dy = valid[k] ? __fsub_rn((float)cy, sy[k]) : 0.f;
        if (MODE == 0 && (dbg_idx || dbg_mask) && inb) {
            const long long opix = img_pix + (long long)i * g.Wo + j;
            unsigned mask = 0;
            if (valid[k]) {
                const bool fxi = fx[k] >= 0, cxi = cx <= g.W - 1, fyi = fy[k] >= 0, cyi = cy <= g.H - 1;
                mask = 1u | ((fxi && fyi) ? 2u : 0u) | ((cxi && cyi) ? 4u : 0u) | ((fxi && cyi) ? 8u : 0u) |
                       ((cxi && fyi) ? 16u : 0u);
            }
            if (dbg_idx) reinterpret_cast<int4*>(dbg_idx)[opix] = valid[k] ? make_int4(fx[k], fy[k], cx, cy) : make_int4(0, 0, 0, 0);
            if (dbg_mask) dbg_mask[opix] = (uint8_t)mask;
        }
        const float omdx = __fsub_rn(1.0f, dx), omdy = __fsub_rn(1.0f, dy);
        float p_ff[C], p_cc[C], p_fc[C], p_cf[C];
        if (staged) {
            const float* t = s_win + (valid[k] ? (fy[k] - ylo) * kPitch + (fx[k] - xa) * C : 0);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                p_ff[c] = t[c]; p_cf[c] = t[C + c]; p_fc[c] = t[kPitch + c]; p_cc[c] = t[kPitch + C + c];
            }
        } else {  // tap box larger than the window: predicated gathers from global (L1/L2)
            const bool fxi = fx[k] >= 0, cxi = cx <= g.W - 1, fyi = fy[k] >= 0, cyi = cy <= g.H - 1;
            const float* base = data + (((long long)bs * g.H + fy[k]) * g.W + fx[k]) * C;
            const int rowf = g.W * C;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                p_ff[c] = (valid[k] && fxi && fyi) ? __ldg(base + c) : 0.f;
                p_cf[c] = (valid[k] && cxi && fyi) ? __ldg(base + C + c) : 0.f;
                p_fc[c] = (valid[k] && fxi && cyi) ? __ldg(base + rowf + c) : 0.f;
                p_cc[c] = (valid[k] && cxi && cyi) ? __ldg(base + rowf + C + c) : 0.f;
            }
        }
        float* io = s_io + (r * 32 + lane) * C;
        if (MODE == 0) {
            const float w_ff = __fmul_rn(dx, dy), w_cc = __fmul_rn(omdx, omdy), w_fc = __fmul_rn(dx, omdy),
                        w_cf = __fmul_rn(omdx, dy);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float v = __fmul_rn(w_ff, p_ff[c]);
                v = __fadd_rn(v, __fmul_rn(w_cc, p_cc[c]));
                v = __fadd_rn(v, __fmul_rn(w_fc, p_fc[c]));
                v = __fadd_rn(v, __fmul_rn(w_cf, p_cf[c]));
                io[c] = valid[k] ? v : 0.f;
            }
        } else if (MODE == 2) {
            const float w_ff = __fmul_rn(dx, dy), w_cc = __fmul_rn(omdx, omdy), w_fc = __fmul_rn(dx, omdy),
                        w_cf = __fmul_rn(omdx, dy);
            const float* tg = s_tgt + (r * 32 + lane) * C;
            float g0 = 0.f, g1 = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float v = __fmul_rn(w_ff, p_ff[c]);
                v = __fadd_rn(v, __fmul_rn(w_cc, p_cc[c]));
                v = __fadd_rn(v, __fmul_rn(w_fc, p_fc[c]));
                v = __fadd_rn(v, __fmul_rn(w_cf, p_cf[c]));
                v = valid[k] ? v : 0.f;
                io[c] = v;
                // loss and dL/dgen exactly as loss_flat_kernel (loss.cu): out-of-image pixels have gen = target = 0
                const float d = __fsub_rn(v, tg[c]);
                float gq;
                if (fa.mode == DMV_LOSS_L2) {
                    loss_acc = __fadd_rn(loss_acc, __fmul_rn(__fmul_rn(fa.w[c], d), d));
                    gq = __fmul_rn(2.0f, d);
                } else {
                    loss_acc = __fadd_rn(loss_acc, __fmul_rn(fa.w[c], fabsf(d)));
                    gq = (d > 0.f) ? 1.0f : (d < 0.f ? -1.0f : 0.0f);
                }
                const float gc = __fmul_rn(__fmul_rn(gq, fa.w[c]), fa.inv_count);
                const float a0 = __fadd_rn(__fmul_rn(omdy, __fsub_rn(p_cc[c], p_fc[c])), __fmul_rn(dy, __fsub_rn(p_cf[c], p_ff[c])));
                const float a1 = __fadd_rn(__fmul_rn(omdx, __fsub_rn(p_cc[c], p_cf[c])), __fmul_rn(dx, __fsub_rn(p_fc[c], p_ff[c])));
                g0 = __fadd_rn(g0, __fmul_rn(gc, a0));
                g1 = __fadd_rn(g1, __fmul_rn(gc, a1));
            }
            if (inb) reinterpret_cast<float2*>(fa.grad_wf)[img_pix + (long long)i * g.Wo + j] = valid[k] ? make_float2(g0, g1) : make_float2(0.f, 0.f);
        } else {
            float g0 = 0.f, g1 = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float gc = io[c];
                const float a0 = __fadd_rn(__fmul_rn(omdy, __fsub_rn(p_cc[c], p_fc[c])), __fmul_rn(dy, __fsub_rn(p_cf[c], p_ff[c])));
                const float a1 = __fadd_rn(__fmul_rn(omdx, __fsub_rn(p_cc[c], p_cf[c])), __fmul_rn(dx, __fsub_rn(p_fc[c], p_ff[c])));
                g0 = __fadd_rn(g0, __fmul_rn(gc, a0));
                g1 = __fadd_rn(g1, __fmul_rn(gc, a1));
            }
            if (inb) reinterpret_cast<float2*>(out)[img_pix + (long long)i * g.Wo + j] = valid[k] ? make_float2(g0, g1) : make_float2(0.f, 0.f);
        }
    }
    if (MODE == 0 || MODE == 2) {
        tc::fence_proxy_async();          // generic-proxy writes of s_io -> visible to the bulk store
        __syncthreads();
        if (tid == 0) tc::tma_store_3d(&map_io, s_io, j0 * C, i0, b);
    }
    if (MODE == 2) {
        // deterministic loss: fixed tree inside the CTA, per-CTA partials, ordered sum by the last CTA to finish
        __shared__ double s_red[kWarps];
        __shared__ bool s_last;
        double local = (double)loss_acc;
        for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
        if (lane == 0) s_red[warp] = local;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < kWarps; ++w) t += s_red[w];
            fa.partials[blockIdx.x] = t;
            __threadfence();
            s_last = (atomicAdd(fa.counter, 1u) == gridDim.x - 1);
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            double t = 0.0;
            for (unsigned q = tid; q < gridDim.x; q += kThreads) t += __ldcg(fa.partials + q);   // thread-strided, fixed order
            for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
            __syncthreads();
            if (lane == 0) s_red[warp] = t;
            __syncthreads();
            if (tid == 0) {
                double tot = 0.0;
                for (int w = 0; w < kWarps; ++w) tot += s_red[w];
                *fa.loss_out = (float)(tot * (double)fa.inv_count);
                *fa.counter = 0;          // ready for the next launch (stream-ordered)
            }
        }
    }
    if ((MODE == 0 || MODE == 2) && tid == 0) tc::bulk_commit_wait_read();   // the tile stays in shared memory until the store has read it
}

int encode_f32_map(CUtensorMap* map, const float* base, int inner, int rows, int batch, int box_inner, int box_rows) {
    tc::EncodeTiledFn enc = tc::get_encode();
    if (!enc) return fail(DMV_E_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
    tc::bind_context();
    cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)batch};
    cuuint64_t strides[2] = {(cuuint64_t)inner * 4, (cuuint64_t)inner * 4 * (cuuint64_t)rows};
    cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1u};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("sampler: cuTensorMapEncodeTiled failed (%d) dims %d %d %d box %d %d", (int)r, inner, rows, batch, box_inner, box_rows);
        return DMV_E_CUDA;
    }
    return DMV_OK;
}

// Pre-pass of grad_data: tap box of every output tile and of each of its 32 warp chunks (32 pixels of the tile: an
// 8 x 4 patch of an image, 32 consecutive samples of a 1-D list; chunk_pixel below).  Layout: boxes[tile * kBoxesPerTile] = tile box,
// boxes[tile * kBoxesPerTile + 1 + q] = box of chunk q; an empty box has xmin > xmax.
constexpr int kChunks = kTilePix / 32;
constexpr int kBoxesPerTile = 1 + kChunks;

// Pixel (di, dj) of a tile that lane `lane` of chunk q owns.  Image tiles (32 x 32) are cut into 8-wide x 4-tall patches:
// a compact patch has a compact tap box whatever the orientation of the grid (a 32 x 1 row segment has a 40 x 8 box that
// reaches 2-3 source tiles along its long side).  1-D sample lists (1 x 1024 tiles) are cut into runs of 32 samples.
__device__ __forceinline__ void chunk_pixel(const Geom& g, int q, int lane, int& di, int& dj) {
    if (g.tw_shift == 5) {
        di = (q >> 2) * 4 + (lane >> 3);
        dj = (q & 3) * 8 + (lane & 7);
    } else {
        const int p = q * 32 + lane;
        di = p >> g.tw_shift;
        dj = p & ((1 << g.tw_shift) - 1);
    }
}

__global__ void __launch_bounds__(kThreads) sampler_box_kernel(const float* __restrict__ wf, int4* __restrict__ boxes, Geom g) {
    __shared__ int s_box[4];
    const int tid = threadIdx.x;
    int b, i0, j0;
    tile_origin(g, blockIdx.x, b, i0, j0);
    if (tid < 4) s_box[tid] = (tid & 1) ? -0x7fffffff : 0x7fffffff;
    __syncthreads();
    int4* tile_boxes = boxes + (long long)blockIdx.x * kBoxesPerTile;
#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        const int q = k * kWarps + (tid >> 5);                  // this warp's chunk
        int di, dj;
        chunk_pixel(g, q, tid & 31, di, dj);
        const int i = i0 + di, j = j0 + dj;
        Sample s;
        s.valid = false;
        s.x = s.y = 0.f;
        if (i < g.Ho && j < g.Wo) s = load_sample(wf, g, b, i, j);
        int xlo = 0x7fffffff, xhi = -0x7fffffff, ylo = 0x7fffffff, yhi = -0x7fffffff;
        if (s.valid) {
            const int fx = (int)floorf(s.x), fy = (int)floorf(s.y);
            xlo = max(fx, 0);
            xhi = min(fx + 1, g.W - 1);
            ylo = max(fy, 0);
            yhi = min(fy + 1, g.H - 1);
        }
        xlo = __reduce_min_sync(0xffffffffu, xlo);
        xhi = __reduce_max_sync(0xffffffffu, xhi);
        ylo = __reduce_min_sync(0xffffffffu, ylo);
        yhi = __reduce_max_sync(0xffffffffu, yhi);
        if ((tid & 31) == 0) {
            tile_boxes[1 + q] = make_int4(xlo, xhi, ylo, yhi);
            atomicMin(&s_box[0], xlo);
            atomicMax(&s_box[1], xhi);
            atomicMin(&s_box[2], ylo);
            atomicMax(&s_box[3], yhi);
        }
    }
    __syncthreads();
    if (tid == 0) tile_boxes[0] = make_int4(s_box[0], s_box[1], s_box[2], s_box[3]);
}

// grad wrt the source.  One CTA owns a 32x16 SOURCE tile and visits the warp chunks whose tap box intersects it.  The
// candidates are found in parallel, not by a serial scan (a dependent box load per output tile made the first version of
// this kernel latency-bound: 49 L2 round trips per CTA): (A) every thread tests one output tile's box and the hits are
// compacted, in tile order, into a shared list; (B) for eight listed tiles at a time, warp w tests the 32 chunk boxes of
// tile w with one coalesced load and publishes the hit mask; (C) the hits, enumerated in (tile, chunk) order, are dealt
// round-robin to the warps -- a fixed assignment for given inputs -- and each warp brings in the flow vectors and output
// gradients of up to G chunks at once before it accumulates them.  Under a few pixels of displacement a chunk's box is
// ~15 x 11 source pixels, so an output pixel is visited by ~2.5 source tiles.
// Each warp accumulates into a warp-private copy of the source tile with plain shared-memory read-modify-writes.  Two lanes
// can hit the same cell in the same tap pass only if their samples share the floor cell (a tap pass maps floor cells to
// tap cells one to one), so ONE __match_any_sync on the floor cell ranks the lanes for all four taps; ranks take turns,
// warps are summed in warp order, every grad_data element is written exactly once: same inputs -> same bits.
__host__ __device__ constexpr int grad_data_pitch(int C) { return kSrcTileW * C + 1; }

template <int CT>
__global__ void __launch_bounds__(kThreads) sampler_grad_data_kernel(
    const float* __restrict__ wf, const float* __restrict__ grad_out, const int4* __restrict__ boxes,
    float* __restrict__ grad_data, Geom g, int src_tiles_x, int src_tiles_y) {
    constexpr int CC = CT ? CT : 8;
    constexpr int G = CT ? 4 : 2;
    extern __shared__ float s_acc[];  // [kWarps][kSrcTileH][kSrcTileW*C + 1]
    __shared__ int s_tiles[kThreads];
    __shared__ int s_wcount[kWarps];
    __shared__ unsigned s_mask[kWarps];
    const int C = CT ? CT : g.C;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int per_img = src_tiles_x * src_tiles_y;
    const int b = blockIdx.x / per_img;
    const int st = blockIdx.x - b * per_img;
    const int sty = st / src_tiles_x, stx = st - sty * src_tiles_x;
    const int sx0 = stx * kSrcTileW, sy0 = sty * kSrcTileH;
    const int sx1 = min(sx0 + kSrcTileW, g.W) - 1, sy1 = min(sy0 + kSrcTileH, g.H) - 1;
    // Row pitch of the private tiles: 32 C + 1 floats.  With a multiple of 32 the bank of a cell would depend on its column
    // only, and under the reference's (Y,X) grid the 32 lanes of a chunk hit a handful of columns on 32 different rows
    // (7-way bank conflicts on every read-modify-write: the kernel was bound by the shared-memory pipe); with the odd pitch
    // the row index walks the banks.
    const int pitch = grad_data_pitch(C);
    const int tile_floats = kSrcTileH * pitch;
    for (int e = tid; e < kWarps * tile_floats; e += kThreads) s_acc[e] = 0.f;
    float* acc = s_acc + warp * tile_floats;

    const int out_tiles = g.tiles_x * g.tiles_y;
    const unsigned lt = (1u << lane) - 1u;
    const int4* img_boxes = boxes + (long long)b * out_tiles * kBoxesPerTile;
    auto misses = [&](const int4& bx) { return bx.x > sx1 || bx.y < sx0 || bx.z > sy1 || bx.w < sy0; };

    for (int tbase = 0; tbase < out_tiles; tbase += kThreads) {
        // (A) output tiles whose tap box intersects this source tile, compacted in tile order
        const int t = tbase + tid;
        bool hit = false;
        if (t < out_tiles) hit = !misses(__ldg(img_boxes + (long long)t * kBoxesPerTile));
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        __syncthreads();                         // the previous round's lists are no longer read (and s_acc is zeroed)
        if (lane == 0) s_wcount[warp] = __popc(bal);
        __syncthreads();
        int off = 0, nt = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const int c = s_wcount[w];
            if (w < warp) off += c;
            nt += c;
        }
        if (hit) s_tiles[off + __popc(bal & lt)] = t;
        __syncthreads();
        for (int cb = 0; cb < nt; cb += kWarps) {
            // (B) chunk boxes of tiles cb .. cb+7: one tile per warp, one chunk per lane
            unsigned m = 0;
            if (cb + warp < nt) m = __ballot_sync(0xffffffffu, !misses(__ldg(img_boxes + (long long)s_tiles[cb + warp] * kBoxesPerTile + 1 + lane)));
            if (lane == 0) s_mask[warp] = m;
            __syncthreads();
            int total = 0;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) total += __popc(s_mask[w]);
            // (C) entry e of the (tile, chunk)-ordered hit list goes to warp e % kWarps
            for (int e0 = warp; e0 < total; e0 += kWarps * G) {
                int pi[G], pj[G];
                bool inb[G];
                float2 fl[G];
                float gv[G][CC];
#pragma unroll
                for (int u = 0; u < G; ++u) {
                    const int e = e0 + u * kWarps;
                    inb[u] = false;
                    pi[u] = pj[u] = 0;
                    fl[u] = make_float2(0.f, 0.f);
#pragma unroll
                    for (int c = 0; c < CC; ++c) gv[u][c] = 0.f;
                    if (e < total) {                          // warp-uniform
                        int k = 0, base = 0;
                        for (;;) {
                            const int n = __popc(s_mask[k]);
                            if (e < base + n) break;
                            base += n;
                            ++k;
                        }
                        const int q = (int)__fns(s_mask[k], 0, e - base + 1);
                        const int tl = s_tiles[cb + k];
                        const int ty = tl / g.tiles_x, tx = tl - ty * g.tiles_x;
                        int di, dj;
                        chunk_pixel(g, q, lane, di, dj);
                        pi[u] = ty * (kTilePix >> g.tw_shift) + di;
                        pj[u] = (tx << g.tw_shift) + dj;
                        inb[u] = pi[u] < g.Ho && pj[u] < g.Wo;
                        if (inb[u]) {
                            const long long px = ((long long)b * g.Ho + pi[u]) * g.Wo + pj[u];
                            fl[u] = __ldg(reinterpret_cast<const float2*>(wf) + px);
#pragma unroll
                            for (int c = 0; c < CC; ++c)
                                if (CT || c < C) gv[u][c] = __ldg(grad_out + px * C + c);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < G; ++u) {
                    if (e0 + u * kWarps >= total) break;      // warp-uniform
                    Sample s;
                    s.valid = false;
                    s.x = s.y = 0.f;
                    if (inb[u]) s = make_sample(fl[u], g, pi[u], pj[u]);
                    int key[4] = {-1, -1, -1, -1};     // float offset of the tap's cell in the private tile
                    float wgt[4] = {0.f, 0.f, 0.f, 0.f};
                    int cell = -1 - lane;        // floor cell of the sample; lanes with nothing to add get distinct dummies
                    if (s.valid) {
                        const int fx = (int)floorf(s.x), fy = (int)floorf(s.y);
                        const int cx = fx + 1, cy = fy + 1;
                        const float dx = (float)cx - s.x, dy = (float)cy - s.y;
                        const bool fxo = fx >= sx0 && fx <= sx1, cxo = cx >= sx0 && cx <= sx1;
                        const bool fyo = fy >= sy0 && fy <= sy1, cyo = cy >= sy0 && cy <= sy1;
                        if (fxo && fyo) { key[0] = (fy - sy0) * pitch + (fx - sx0) * C; wgt[0] = dx * dy; }
                        if (cxo && cyo) { key[1] = (cy - sy0) * pitch + (cx - sx0) * C; wgt[1] = (1.f - dx) * (1.f - dy); }
                        if (fxo && cyo) { key[2] = (cy - sy0) * pitch + (fx - sx0) * C; wgt[2] = dx * (1.f - dy); }
                        if (cxo && fyo) { key[3] = (fy - sy0) * pitch + (cx - sx0) * C; wgt[3] = (1.f - dx) * dy; }
                        // fx, fy >= -1 for a valid sample; both lie within one pixel of the source tile when a key is set
                        if ((fxo || cxo) && (fyo || cyo)) cell = (fy - sy0 + 1) * (kSrcTileW + 2) + (fx - sx0 + 1);
                    }
                    const bool mine = cell >= 0;
                    if (!__any_sync(0xffffffffu, mine)) continue;
                    const unsigned peers = __match_any_sync(0xffffffffu, cell);
                    const int rank = __popc(peers & lt);
                    const int rounds = __reduce_max_sync(0xffffffffu, mine ? __popc(peers) : 0);
                    for (int r = 0; r < rounds; ++r) {
                        const bool on = mine && rank == r;
#pragma unroll
                        for (int tap = 0; tap < 4; ++tap) {
                            if (on && key[tap] >= 0) {
                                float* cellp = acc + key[tap];
#pragma unroll
                                for (int c = 0; c < CC; ++c) {
                                    if (!CT && c >= C) break;
                                    cellp[c] += gv[u][c] * wgt[tap];
                                }
                            }
                            __syncwarp();     // the next tap pass may touch a cell another lane wrote in this one
                        }
                    }
                }
            }
            __syncthreads();                     // s_mask is rewritten by the next batch
        }
    }
    __syncthreads();
    // fixed-order sum of the warp-private tiles; each grad_data element is written once
    const int seg = (sx1 - sx0 + 1) * C;
    for (int r = warp; r <= sy1 - sy0; r += kWarps) {
        float* dst = grad_data + (((long long)b * g.H + sy0 + r) * g.W + sx0) * C;
        for (int e = lane; e < seg; e += 32) {
            float sum = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) sum += s_acc[w * tile_floats + r * pitch + e];
            dst[e] = sum;
        }
    }
}

int make_geom(Geom& g, int B, int H, int W, int C, int Ho, int Wo, unsigned flags) {
    DMV_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && Ho > 0 && Wo > 0, DMV_E_INVALID_ARG, "sampler: non-positive dimension");
    DMV_REQUIRE(C <= 16, DMV_E_UNSUPPORTED_SHAPE, "sampler: C > 16 unsupported");
    DMV_REQUIRE((flags & ~3u) == 0, DMV_E_INVALID_ARG, "sampler: unknown flag");
    g.B = B; g.H = H; g.W = W; g.C = C; g.Ho = Ho; g.Wo = Wo; g.flags = flags;
    g.group = 1;
    g.tw_shift = (Ho == 1) ? 10 : 5;  // 1-D sample lists use 1x1024 tiles, images 32x32
    g.tiles_x = ceil_div(Wo, 1 << g.tw_shift);
    g.tiles_y = ceil_div(Ho, kTilePix >> g.tw_shift);
    DMV_REQUIRE((long long)B * g.tiles_x * g.tiles_y < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "sampler: too many tiles");
    return DMV_OK;
}

template <int MODE>
int launch_tile(const float* data, const float* wf, const float* go, float* out, int32_t* di, uint8_t* dm,
                const Geom& g, cudaStream_t st) {
    const int grid = g.B * g.tiles_x * g.tiles_y;
    const bool aligned = (((uintptr_t)data | (uintptr_t)wf | (uintptr_t)go | (uintptr_t)out) & 15) == 0;
    if (SAMPLER_TMA && g.tw_shift == 5 && (g.C == 1 || g.C == 3 || g.C == 4) && ((g.W * g.C) & 3) == 0 && ((g.Wo * g.C) & 3) == 0 &&
        aligned && (!di || ((uintptr_t)di & 15) == 0)) {
        CUtensorMap map_src, map_src_l, map_io;
        const int src_images = g.B / g.group;
        int rc = encode_f32_map(&map_src, data, g.W * g.C, g.H, src_images, kBoxS * g.C, kBoxS);
        if (rc) return rc;
        rc = encode_f32_map(&map_src_l, data, g.W * g.C, g.H, src_images, kBoxL * g.C, kBoxL);
        if (rc) return rc;
        rc = encode_f32_map(&map_io, MODE == 0 ? out : go, g.Wo * g.C, g.Ho, g.B, 32 * g.C, 32);
        if (rc) return rc;
        const size_t wsm = (size_t)(win_floats(g.C) + 32 * 32 * g.C) * sizeof(float);
#define DMV_LAUNCH_TMA(CT)                                                                               \
    do {                                                                                                 \
        static bool attr_done = false;                                                                   \
        if (!attr_done) {                                                                                \
            cudaFuncSetAttribute(sampler_tma_kernel<CT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm); \
            attr_done = true;                                                                            \
        }                                                                                                \
        sampler_tma_kernel<CT, MODE><<<grid, kThreads, wsm, st>>>(map_src, map_src_l, map_io, map_io, data, wf, out, di, dm, g, FuseArgs()); \
    } while (0)
        if (g.C == 1) DMV_LAUNCH_TMA(1);
        else if (g.C == 3) DMV_LAUNCH_TMA(3);
        else DMV_LAUNCH_TMA(4);
#undef DMV_LAUNCH_TMA
        return check_launch(MODE == 0 ? "sampler_fwd(tma)" : "sampler_grad_warp(tma)");
    }
    const size_t smem = kStageFloats * sizeof(float);
#define DMV_LAUNCH_TILE(CT)                                                                              \
    do {                                                                                                 \
        static bool attr_done = false;                                                                   \
        if (!attr_done) {                                                                                \
            cudaFuncSetAttribute(sampler_tile_kernel<CT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            attr_done = true;                                                                            \
        }                                                                                                \
        sampler_tile_kernel<CT, MODE><<<grid, kThreads, smem, st>>>(data, wf, go, out, di, dm, g);       \
    } while (0)
    switch (g.C) {
        case 1: DMV_LAUNCH_TILE(1); break;
        case 3: DMV_LAUNCH_TILE(3); break;
        case 4: DMV_LAUNCH_TILE(4); break;
        default: DMV_LAUNCH_TILE(0); break;
    }
#undef DMV_LAUNCH_TILE
    return check_launch(MODE == 0 ? "sampler_fwd" : "sampler_grad_warp");
}

}  // namespace

extern "C" {

int dmv_sampler_fwd(const float* data, const float* wf, float* out, int32_t* dbg_idx, uint8_t* dbg_mask, int B,
                    int H, int W, int C, int Hout, int Wout, unsigned flags, void* stream) {
    DMV_REQUIRE(data && wf && out, DMV_E_INVALID_ARG, "sampler_fwd: null pointer");
    DMV_REQUIRE(((uintptr_t)wf & 7) == 0, DMV_E_ALIGN, "sampler_fwd: warp/flow must be 8-byte aligned");
    DMV_REQUIRE(!dbg_idx || ((uintptr_t)dbg_idx & 15) == 0, DMV_E_ALIGN, "sampler_fwd: dbg_idx must be 16-byte aligned");
    Geom g;
    int rc = make_geom(g, B, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    return launch_tile<0>(data, wf, nullptr, out, dbg_idx, dbg_mask, g, (cudaStream_t)stream);
}

int dmv_sampler_fwd_shared_src(const float* data, int B_src, int group, const float* wf, float* out, int H, int W, int C,
                               int Hout, int Wout, unsigned flags, void* stream) {
    DMV_REQUIRE(data && wf && out, DMV_E_INVALID_ARG, "sampler_fwd_shared_src: null pointer");
    DMV_REQUIRE(((uintptr_t)wf & 7) == 0, DMV_E_ALIGN, "sampler_fwd_shared_src: warp/flow must be 8-byte aligned");
    DMV_REQUIRE(B_src > 0 && group > 0, DMV_E_INVALID_ARG, "sampler_fwd_shared_src: non-positive B_src or group");
    DMV_REQUIRE((long long)B_src * group < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "sampler_fwd_shared_src: too many samples");
    Geom g;
    int rc = make_geom(g, B_src * group, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    g.group = group;
    return launch_tile<0>(data, wf, nullptr, out, nullptr, nullptr, g, (cudaStream_t)stream);
}

size_t dmv_sampler_bwd_workspace_size(int B, int H, int W, int C, int Hout, int Wout) {
    (void)H; (void)W; (void)C;
    if (B <= 0 || Hout <= 0 || Wout <= 0) return 0;
    const int tw_shift = (Hout == 1) ? 10 : 5;
    const long long tiles = (long long)B * ceil_div(Wout, 1 << tw_shift) * ceil_div(Hout, kTilePix >> tw_shift);
    return (size_t)tiles * kBoxesPerTile * sizeof(int4);
}

int dmv_sampler_bwd(const float* data, const float* wf, const float* grad_out, float* grad_data, float* grad_wf,
                    int B, int H, int W, int C, int Hout, int Wout, unsigned flags, void* workspace,
                    size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(data && wf && grad_out, DMV_E_INVALID_ARG, "sampler_bwd: null pointer");
    DMV_REQUIRE(grad_data || grad_wf, DMV_E_INVALID_ARG, "sampler_bwd: nothing to compute");
    DMV_REQUIRE(((uintptr_t)wf & 7) == 0 && ((uintptr_t)grad_wf & 7) == 0, DMV_E_ALIGN, "sampler_bwd: warp buffers must be 8-byte aligned");
    Geom g;
    int rc = make_geom(g, B, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_wf) {
        rc = launch_tile<1>(data, wf, grad_out, grad_wf, nullptr, nullptr, g, st);
        if (rc) return rc;
    }
    if (grad_data) {
        DMV_REQUIRE(C <= 8, DMV_E_UNSUPPORTED_SHAPE, "sampler_bwd: grad_data supports C <= 8");
        const size_t need = dmv_sampler_bwd_workspace_size(B, H, W, C, Hout, Wout);
        DMV_REQUIRE(workspace && workspace_bytes >= need, DMV_E_WORKSPACE, "sampler_bwd: workspace too small");
        DMV_REQUIRE(((uintptr_t)workspace & 15) == 0, DMV_E_ALIGN, "sampler_bwd: workspace must be 16-byte aligned");
        int4* boxes = reinterpret_cast<int4*>(workspace);
        const int out_tiles = g.B * g.tiles_x * g.tiles_y;
        sampler_box_kernel<<<out_tiles, kThreads, 0, st>>>(wf, boxes, g);
        rc = check_launch("sampler_box");
        if (rc) return rc;
        const int stx = ceil_div(W, kSrcTileW), sty = ceil_div(H, kSrcTileH);
        const int grid = B * stx * sty;
        const size_t smem = (size_t)kWarps * kSrcTileH * grad_data_pitch(C) * sizeof(float);
#define DMV_LAUNCH_GD(CT)                                                                                         \
    do {                                                                                                          \
        cudaFuncSetAttribute(sampler_grad_data_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        sampler_grad_data_kernel<CT><<<grid, kThreads, smem, st>>>(wf, grad_out, boxes, grad_data, g, stx, sty);   \
    } while (0)
        switch (C) {
            case 1: DMV_LAUNCH_GD(1); break;
            case 3: DMV_LAUNCH_GD(3); break;
            case 4: DMV_LAUNCH_GD(4); break;
            default: DMV_LAUNCH_GD(0); break;
        }
#undef DMV_LAUNCH_GD
        rc = check_launch("sampler_grad_data");
        if (rc) return rc;
    }
    return DMV_OK;
}

int dmv_sampler_grad_flow_shared_src(const float* data, int B_src, int group, const float* wf, const float* grad_out, float* grad_wf,
                                     int H, int W, int C, int Hout, int Wout, unsigned flags, void* stream) {
    DMV_REQUIRE(data && wf && grad_out && grad_wf, DMV_E_INVALID_ARG, "sampler_grad_flow_shared_src: null pointer");
    DMV_REQUIRE(((uintptr_t)wf & 7) == 0 && ((uintptr_t)grad_wf & 7) == 0, DMV_E_ALIGN,
                "sampler_grad_flow_shared_src: warp buffers must be 8-byte aligned");
    DMV_REQUIRE(B_src > 0 && group > 0, DMV_E_INVALID_ARG, "sampler_grad_flow_shared_src: non-positive B_src or group");
    DMV_REQUIRE((long long)B_src * group < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "sampler_grad_flow_shared_src: too many samples");
    Geom g;
    int rc = make_geom(g, B_src * group, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    g.group = group;
    return launch_tile<1>(data, wf, grad_out, grad_wf, nullptr, nullptr, g, (cudaStream_t)stream);
}

size_t dmv_sampler_loss_workspace_size(int B, int Hout, int Wout) {
    if (B <= 0 || Hout <= 0 || Wout <= 0) return 0;
    return (size_t)B * ceil_div(Wout, 32) * ceil_div(Hout, 32) * sizeof(double) + 16;
}

}  // extern "C"

namespace {

// dmv_sampler_loss_fused over B_src source images, output sample n warping source n / group (group = 1: the plain call)
int sampler_loss_fused(const float* data, int B_src, int group, const float* wf, const float* target, const float* chan_weight, int mode,
                       float inv_count, float* gen_out, float* grad_wf, float* loss_out, int H, int W, int C, int Hout, int Wout,
                       unsigned flags, void* workspace, size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(data && wf && target && chan_weight && gen_out && grad_wf && loss_out, DMV_E_INVALID_ARG, "sampler_loss_fused: null pointer");
    DMV_REQUIRE(mode == DMV_LOSS_L2 || mode == DMV_LOSS_L1, DMV_E_INVALID_ARG, "sampler_loss_fused: unknown loss mode");
    DMV_REQUIRE(B_src > 0 && group > 0, DMV_E_INVALID_ARG, "sampler_loss_fused: non-positive B_src or group");
    DMV_REQUIRE((long long)B_src * group < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "sampler_loss_fused: too many samples");
    const int B = B_src * group;
    Geom g;
    int rc = make_geom(g, B, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    g.group = group;
    const bool aligned = (((uintptr_t)data | (uintptr_t)wf | (uintptr_t)target | (uintptr_t)gen_out | (uintptr_t)grad_wf) & 15) == 0;
    if (!(g.tw_shift == 5 && (C == 1 || C == 3 || C == 4) && ((W * C) & 3) == 0 && ((Wout * C) & 3) == 0 && aligned))
        return fail(DMV_E_UNSUPPORTED_SHAPE, "sampler_loss_fused: needs C in {1,3,4}, 16-byte aligned rows and buffers, image-shaped output");
    const int grid = g.B * g.tiles_x * g.tiles_y;
    DMV_REQUIRE(workspace && workspace_bytes >= dmv_sampler_loss_workspace_size(B, Hout, Wout) && ((uintptr_t)workspace & 7) == 0, DMV_E_WORKSPACE,
                "sampler_loss_fused: workspace too small or unaligned (it must be zeroed once and not shared)");
    CUtensorMap map_src, map_src_l, map_io, map_tgt;
    rc = encode_f32_map(&map_src, data, W * C, H, B_src, kBoxS * C, kBoxS);
    if (!rc) rc = encode_f32_map(&map_src_l, data, W * C, H, B_src, kBoxL * C, kBoxL);
    if (!rc) rc = encode_f32_map(&map_io, gen_out, Wout * C, Hout, B, 32 * C, 32);
    if (!rc) rc = encode_f32_map(&map_tgt, target, Wout * C, Hout, B, 32 * C, 32);
    if (rc) return rc;
    FuseArgs fa;
    for (int c = 0; c < 4; ++c) fa.w[c] = c < C ? chan_weight[c] : 0.f;
    fa.inv_count = inv_count; fa.mode = mode;
    fa.counter = reinterpret_cast<unsigned*>(workspace);                 // fixed place: survives calls with other grid sizes
    fa.partials = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 16);
    fa.loss_out = loss_out; fa.grad_wf = grad_wf;
    const size_t wsm = (size_t)(win_floats(C) + 2 * 32 * 32 * C) * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
#define DMV_LAUNCH_FUSED(CT)                                                                                  \
    do {                                                                                                      \
        static bool attr_done = false;                                                                        \
        if (!attr_done) {                                                                                     \
            cudaFuncSetAttribute(sampler_tma_kernel<CT, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm); \
            attr_done = true;                                                                                 \
        }                                                                                                     \
        sampler_tma_kernel<CT, 2><<<grid, kThreads, wsm, st>>>(map_src, map_src_l, map_io, map_tgt, data, wf, gen_out, nullptr, nullptr, g, fa); \
    } while (0)
    if (C == 1) DMV_LAUNCH_FUSED(1);
    else if (C == 3) DMV_LAUNCH_FUSED(3);
    else DMV_LAUNCH_FUSED(4);
#undef DMV_LAUNCH_FUSED
    return check_launch("sampler_loss_fused");
}

// ---------------------------------------------------------------------------------------------
// Several source views per target (dmv_sampler_fuse_views_loss): one CTA per 32x32 TARGET tile.  The head of view v is
// [Hout, Wout, 3] (flow in channels 0-1, confidence logit in channel 2) and is read in place.  Arithmetic is that of the
// composition it replaces -- sampler_tma_kernel MODE 0 per view, loss_kernel (loss.cu) with V = views, MODE 1 on its
// grad_gen -- op for op, including the FMAs nvcc forms in loss_kernel under -fmad=true (the fusion sum and the logit
// gradient), so fused_out and grad_head have the composition's bits.
//   pass 0: softmax statistics (max, sum of __expf in view order, one reciprocal) per pixel, kept in registers;
//   pass 1: per view, reduce the tap box, stage that view's window (36^2 / 44^2 box, or global gathers), accumulate the
//           fused tile in shared memory; then the loss and dL/dfused (stored over the target tile);
//   pass 2: per view, in reverse order, restage the window (L2-resident: the first pass just read it) and form the flow
//           and logit gradients.  Keeping every view's window resident instead would take up to 8 x 31 KB of shared
//           memory (C = 4), one CTA per SM; the reverse order reuses the last window of pass 1, so one view stages once.
constexpr int kMaxViews = 8;

struct ViewsArgs {
    const float* head;
    float* grad_head;
    float w[4];
    float inv_count;
    int mode, views;
    bool store_fused;
    double* partials;
    unsigned* counter;
    float* loss_out;
};

// sample of head pixel hp (flow in channels 0-1), grid added as in sampler_tma_kernel
__device__ __forceinline__ void head_sample(const float* __restrict__ head, long long hp, bool inb, int i, int j, const Geom& g,
                                            float& sx, float& sy, bool& valid, int& fx, int& fy) {
    float f0 = 0.f, f1 = 0.f;
    if (inb) { f0 = __ldg(head + hp * 3); f1 = __ldg(head + hp * 3 + 1); }
    sx = f0; sy = f1;
    if (g.flags & DMV_SAMPLER_ADD_GRID) {
        if (g.flags & DMV_SAMPLER_GRID_XY) {
            sx = __fadd_rn(f0, (float)j);
            sy = __fadd_rn(f1, (float)i);
        } else {
            sx = __fadd_rn(f0, (float)i);
            sy = __fadd_rn(f1, (float)j);
        }
    }
    valid = inb && (sx > -1.0f) && (sy > -1.0f) && (sx < (float)g.W) && (sy < (float)g.H);
    fx = valid ? __float2int_rd(sx) : 0;
    fy = valid ? __float2int_rd(sy) : 0;
}

// the staged window of one view: the smallest box that holds its tap box, or none (global gathers)
struct Window {
    bool staged;
    int xa, ylo, pitch;
};

__device__ __forceinline__ Window view_window(const int* box, int C) {
    Window w;
    const int xlo = box[0], xhi = box[1], ylo = box[2], yhi = box[3];
    w.xa = (C == 4) ? xlo : (xlo & ~3);
    w.ylo = ylo;
    const int span = max(xhi - w.xa, yhi - ylo);
    w.staged = (xlo <= xhi) && (span < kBoxL);
    w.pitch = ((span < kBoxS) ? kBoxS : kBoxL) * C;
    return w;
}

template <int C>
__device__ __forceinline__ void stage_window(const Window& w, float* s_win, const CUtensorMap* map_s, const CUtensorMap* map_l,
                                             uint64_t* bar, unsigned& phase, int img) {
    if (!w.staged) return;
    if (threadIdx.x == 0) {
        const int box = w.pitch / C;
        tc::mbar_expect_tx(bar, box * box * C * 4);
        tc::tma_load_3d(s_win, box == kBoxS ? map_s : map_l, bar, w.xa * C, w.ylo, img);
    }
    tc::mbar_wait(bar, phase);
    phase ^= 1u;
}

// the four taps of a sample (sampler_tma_kernel's two window paths) and the bilinear value (MODE 0's op order)
template <int C>
__device__ __forceinline__ void view_taps(const Window& w, const float* s_win, const float* __restrict__ data, int img, const Geom& g,
                                          bool valid, int fx, int fy, float (&p_ff)[C], float (&p_cf)[C], float (&p_fc)[C],
                                          float (&p_cc)[C]) {
    if (w.staged) {
        const float* t = s_win + (valid ? (fy - w.ylo) * w.pitch + (fx - w.xa) * C : 0);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            p_ff[c] = t[c]; p_cf[c] = t[C + c]; p_fc[c] = t[w.pitch + c]; p_cc[c] = t[w.pitch + C + c];
        }
    } else {
        const int cx = fx + 1, cy = fy + 1;
        const bool fxi = fx >= 0, cxi = cx <= g.W - 1, fyi = fy >= 0, cyi = cy <= g.H - 1;
        const float* base = data + (((long long)img * g.H + fy) * g.W + fx) * C;
        const int rowf = g.W * C;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            p_ff[c] = (valid && fxi && fyi) ? __ldg(base + c) : 0.f;
            p_cf[c] = (valid && cxi && fyi) ? __ldg(base + C + c) : 0.f;
            p_fc[c] = (valid && fxi && cyi) ? __ldg(base + rowf + c) : 0.f;
            p_cc[c] = (valid && cxi && cyi) ? __ldg(base + rowf + C + c) : 0.f;
        }
    }
}

template <int C, bool TRAIN>
__global__ void __launch_bounds__(kThreads, 3) sampler_views_kernel(
    const __grid_constant__ CUtensorMap map_src, const __grid_constant__ CUtensorMap map_src_l,
    const __grid_constant__ CUtensorMap map_fused, const __grid_constant__ CUtensorMap map_tgt, const float* __restrict__ data,
    Geom g, const ViewsArgs va) {
    extern __shared__ __align__(128) float s_dyn[];
    float* s_win = s_dyn;                              // one view's source window
    float* s_fused = s_dyn + win_floats(C);            // [32][32 * C] fused tile
    float* s_tgt = s_fused + 32 * 32 * C;              // TRAIN: target tile, then dL/dfused
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ int s_box[kMaxViews][4];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int V = va.views;
    int b, i0, j0;
    tile_origin(g, blockIdx.x, b, i0, j0);
    if (tid < kMaxViews * 4) s_box[tid >> 2][tid & 3] = (tid & 1) ? -0x7fffffff : 0x7fffffff;
    if (tid == 0) {
        tc::mbar_init(&s_bar[0], 1);
        tc::mbar_init(&s_bar[1], 1);
        tc::fence_barrier_init();
        tc::fence_proxy_async();
        if (TRAIN) {
            tc::mbar_expect_tx(&s_bar[1], 32 * 32 * C * 4);
            tc::tma_load_3d(s_tgt, &map_tgt, &s_bar[1], j0 * C, i0, b);
        }
    }
    __syncthreads();
    const int j = j0 + lane;
    const long long plane = (long long)g.B * g.Ho * g.Wo;              // head pixels per view
    const long long pix0 = (long long)b * g.Ho * g.Wo;
    // pass 0: softmax statistics, loss_kernel's order
    float mx[kPPT], inv[kPPT];
#pragma unroll
    for (int k = 0; k < kPPT; ++k) {
        const int i = i0 + warp + k * kWarps;
        mx[k] = -INFINITY;
        inv[k] = 1.0f;
        if (V == 1 || i >= g.Ho || j >= g.Wo) continue;
        const float* lp = va.head + (pix0 + (long long)i * g.Wo + j) * 3 + 2;
        for (int v = 0; v < V; ++v) mx[k] = fmaxf(mx[k], __ldg(lp + v * plane * 3));
        float den = 0.f;
        for (int v = 0; v < V; ++v) den = __fadd_rn(den, __expf(__fsub_rn(__ldg(lp + v * plane * 3), mx[k])));
        inv[k] = 1.0f / den;
    }

    // pass 1: the fused tile
    unsigned phase = 0;
    for (int v = 0; v < V; ++v) {
        const int img = v * g.B + b;
        float sx[kPPT], sy[kPPT];
        bool valid[kPPT];
        int fx[kPPT], fy[kPPT];
        int bxlo = 0x7fffffff, bxhi = -0x7fffffff, bylo = 0x7fffffff, byhi = -0x7fffffff;
#pragma unroll
        for (int k = 0; k < kPPT; ++k) {
            const int i = i0 + warp + k * kWarps;
            head_sample(va.head, (long long)img * g.Ho * g.Wo + (long long)i * g.Wo + j, (i < g.Ho) && (j < g.Wo), i, j, g, sx[k], sy[k],
                        valid[k], fx[k], fy[k]);
            if (valid[k]) {
                bxlo = min(bxlo, fx[k]); bxhi = max(bxhi, fx[k] + 1);
                bylo = min(bylo, fy[k]); byhi = max(byhi, fy[k] + 1);
            }
        }
        bxlo = __reduce_min_sync(0xffffffffu, bxlo); bxhi = __reduce_max_sync(0xffffffffu, bxhi);
        bylo = __reduce_min_sync(0xffffffffu, bylo); byhi = __reduce_max_sync(0xffffffffu, byhi);
        if (lane == 0) {
            atomicMin(&s_box[v][0], bxlo); atomicMax(&s_box[v][1], bxhi);
            atomicMin(&s_box[v][2], bylo); atomicMax(&s_box[v][3], byhi);
        }
        __syncthreads();              // the box is complete and every thread is done with the previous view's window
        const Window w = view_window(s_box[v], C);
        stage_window<C>(w, s_win, &map_src, &map_src_l, &s_bar[0], phase, img);
#pragma unroll
        for (int k = 0; k < kPPT; ++k) {
            const int r = warp + k * kWarps, i = i0 + r;
            if (i >= g.Ho || j >= g.Wo) continue;
            float p_ff[C], p_cf[C], p_fc[C], p_cc[C];
            view_taps<C>(w, s_win, data, img, g, valid[k], fx[k], fy[k], p_ff, p_cf, p_fc, p_cc);
            const float dx = valid[k] ? __fsub_rn((float)(fx[k] + 1), sx[k]) : 0.f;
            const float dy = valid[k] ? __fsub_rn((float)(fy[k] + 1), sy[k]) : 0.f;
            const float omdx = __fsub_rn(1.0f, dx), omdy = __fsub_rn(1.0f, dy);
            const float w_ff = __fmul_rn(dx, dy), w_cc = __fmul_rn(omdx, omdy), w_fc = __fmul_rn(dx, omdy), w_cf = __fmul_rn(omdx, dy);
            float sm = 1.0f;
            if (V > 1)
                sm = __fmul_rn(__expf(__fsub_rn(__ldg(va.head + ((long long)img * g.Ho * g.Wo + (long long)i * g.Wo + j) * 3 + 2), mx[k])), inv[k]);
            float* fu = s_fused + (r * 32 + lane) * C;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float gv = __fmul_rn(w_ff, p_ff[c]);
                gv = __fadd_rn(gv, __fmul_rn(w_cc, p_cc[c]));
                gv = __fadd_rn(gv, __fmul_rn(w_fc, p_fc[c]));
                gv = __fadd_rn(gv, __fmul_rn(w_cf, p_cf[c]));
                gv = valid[k] ? gv : 0.f;
                fu[c] = (V == 1) ? gv : __fmaf_rn(sm, gv, v == 0 ? 0.f : fu[c]);
            }
        }
    }
    if (va.store_fused) {
        tc::fence_proxy_async();          // generic-proxy writes of s_fused -> visible to the bulk store
        __syncthreads();
        if (tid == 0) tc::tma_store_3d(&map_fused, s_fused, j0 * C, i0, b);
    }
    if (TRAIN) {
        // loss and dL/dfused per pixel as dmv_loss_fused_fwd_bwd (mask = 1); dL/dfused replaces the target in shared memory
        tc::mbar_wait(&s_bar[1], 0);
        double local = 0.0;
#pragma unroll
        for (int k = 0; k < kPPT; ++k) {
            const int r = warp + k * kWarps;
            if (i0 + r >= g.Ho || j >= g.Wo) continue;
            const float* fu = s_fused + (r * 32 + lane) * C;
            float* tg = s_tgt + (r * 32 + lane) * C;
            float acc = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float d = __fsub_rn(fu[c], tg[c]);
                float gq;
                if (va.mode == DMV_LOSS_L2) {
                    acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(va.w[c], d), d));
                    gq = __fadd_rn(d, d);
                } else {
                    acc = __fadd_rn(acc, __fmul_rn(va.w[c], fabsf(d)));
                    gq = (d > 0.f) ? 1.0f : (d < 0.f ? -1.0f : 0.0f);
                }
                // one view: loss_flat_kernel's (g * w) * inv_count; several: loss_kernel's g * (w * mask * inv_count)
                tg[c] = (V == 1) ? __fmul_rn(__fmul_rn(gq, va.w[c]), va.inv_count) : __fmul_rn(gq, __fmul_rn(va.w[c], va.inv_count));
            }
            local += (double)acc;
        }

        // pass 2: flow and logit gradients, views in reverse order (the last window of pass 1 is still staged)
        if (va.grad_head) {
            for (int v = V - 1; v >= 0; --v) {
                const int img = v * g.B + b;
                const Window w = view_window(s_box[v], C);
                if (v != V - 1) {
                    __syncthreads();          // every thread is done with the previous view's window
                    stage_window<C>(w, s_win, &map_src, &map_src_l, &s_bar[0], phase, img);
                }
#pragma unroll
                for (int k = 0; k < kPPT; ++k) {
                    const int r = warp + k * kWarps, i = i0 + r;
                    if (i >= g.Ho || j >= g.Wo) continue;
                    const long long hp = (long long)img * g.Ho * g.Wo + (long long)i * g.Wo + j;
                    float sx, sy;
                    bool valid;
                    int fx, fy;
                    head_sample(va.head, hp, true, i, j, g, sx, sy, valid, fx, fy);
                    float p_ff[C], p_cf[C], p_fc[C], p_cc[C];
                    view_taps<C>(w, s_win, data, img, g, valid, fx, fy, p_ff, p_cf, p_fc, p_cc);
                    const float dx = valid ? __fsub_rn((float)(fx + 1), sx) : 0.f;
                    const float dy = valid ? __fsub_rn((float)(fy + 1), sy) : 0.f;
                    const float omdx = __fsub_rn(1.0f, dx), omdy = __fsub_rn(1.0f, dy);
                    const float w_ff = __fmul_rn(dx, dy), w_cc = __fmul_rn(omdx, omdy), w_fc = __fmul_rn(dx, omdy), w_cf = __fmul_rn(omdx, dy);
                    float sm = 1.0f;
                    if (V > 1) sm = __fmul_rn(__expf(__fsub_rn(__ldg(va.head + hp * 3 + 2), mx[k])), inv[k]);
                    const float* fu = s_fused + (r * 32 + lane) * C;
                    const float* gf = s_tgt + (r * 32 + lane) * C;
                    float g0 = 0.f, g1 = 0.f, gl = 0.f;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        // grad_gen = softmax * dL/dfused, and the logit term, as loss_kernel
                        const float gc = (V == 1) ? gf[c] : __fmul_rn(sm, gf[c]);
                        if (V > 1) {
                            float gv = __fmul_rn(w_ff, p_ff[c]);
                            gv = __fadd_rn(gv, __fmul_rn(w_cc, p_cc[c]));
                            gv = __fadd_rn(gv, __fmul_rn(w_fc, p_fc[c]));
                            gv = __fadd_rn(gv, __fmul_rn(w_cf, p_cf[c]));
                            gv = valid ? gv : 0.f;
                            gl = __fmaf_rn(gf[c], __fsub_rn(gv, fu[c]), gl);
                        }
                        // grad wrt the flow through that grad_gen, as MODE 1
                        const float a0 = __fadd_rn(__fmul_rn(omdy, __fsub_rn(p_cc[c], p_fc[c])), __fmul_rn(dy, __fsub_rn(p_cf[c], p_ff[c])));
                        const float a1 = __fadd_rn(__fmul_rn(omdx, __fsub_rn(p_cc[c], p_cf[c])), __fmul_rn(dx, __fsub_rn(p_fc[c], p_ff[c])));
                        g0 = __fadd_rn(g0, __fmul_rn(gc, a0));
                        g1 = __fadd_rn(g1, __fmul_rn(gc, a1));
                    }
                    float* gh = va.grad_head + hp * 3;
                    gh[0] = valid ? g0 : 0.f;
                    gh[1] = valid ? g1 : 0.f;
                    gh[2] = (V > 1) ? __fmul_rn(sm, gl) : 0.f;     // one view: the softmax is constant
                }
            }
        }

        // deterministic loss, as MODE 2: fixed tree in the CTA, per-CTA partials, ordered sum by the last CTA
        __shared__ double s_red[kWarps];
        __shared__ bool s_last;
        for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
        if (lane == 0) s_red[warp] = local;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int q = 0; q < kWarps; ++q) t += s_red[q];
            va.partials[blockIdx.x] = t;
            __threadfence();
            s_last = (atomicAdd(va.counter, 1u) == gridDim.x - 1);
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            double t = 0.0;
            for (unsigned q = tid; q < gridDim.x; q += kThreads) t += __ldcg(va.partials + q);
            for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
            __syncthreads();
            if (lane == 0) s_red[warp] = t;
            __syncthreads();
            if (tid == 0) {
                double tot = 0.0;
                for (int q = 0; q < kWarps; ++q) tot += s_red[q];
                *va.loss_out = (float)(tot * (double)va.inv_count);
                *va.counter = 0;
            }
        }
    }
    if (va.store_fused && tid == 0) tc::bulk_commit_wait_read();   // the tile stays in shared memory until the store has read it
}

}  // namespace

extern "C" {

int dmv_sampler_loss_fused(const float* data, const float* wf, const float* target, const float* chan_weight, int mode, float inv_count,
                           float* gen_out, float* grad_wf, float* loss_out, int B, int H, int W, int C, int Hout, int Wout,
                           unsigned flags, void* workspace, size_t workspace_bytes, void* stream) {
    return sampler_loss_fused(data, B, 1, wf, target, chan_weight, mode, inv_count, gen_out, grad_wf, loss_out, H, W, C, Hout, Wout, flags,
                              workspace, workspace_bytes, stream);
}

int dmv_sampler_loss_fused_shared_src(const float* data, int B_src, int group, const float* wf, const float* target,
                                      const float* chan_weight, int mode, float inv_count, float* gen_out, float* grad_wf,
                                      float* loss_out, int H, int W, int C, int Hout, int Wout, unsigned flags, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    return sampler_loss_fused(data, B_src, group, wf, target, chan_weight, mode, inv_count, gen_out, grad_wf, loss_out, H, W, C, Hout, Wout,
                              flags, workspace, workspace_bytes, stream);
}

int dmv_sampler_fuse_views_loss(const float* data, int views, const float* head, const float* target, const float* chan_weight, int mode,
                                float inv_count, float* fused_out, float* grad_head, float* loss_out, int B, int H, int W, int C, int Hout,
                                int Wout, unsigned flags, void* workspace, size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(data && head, DMV_E_INVALID_ARG, "sampler_fuse_views_loss: null pointer");
    const bool train = target != nullptr;
    if (train) {
        DMV_REQUIRE(chan_weight && loss_out, DMV_E_INVALID_ARG, "sampler_fuse_views_loss: training needs chan_weight and loss_out");
        DMV_REQUIRE(mode == DMV_LOSS_L2 || mode == DMV_LOSS_L1, DMV_E_INVALID_ARG, "sampler_fuse_views_loss: unknown loss mode");
    } else {
        DMV_REQUIRE(fused_out && !grad_head && !loss_out, DMV_E_INVALID_ARG,
                    "sampler_fuse_views_loss: forward only (target NULL) writes fused_out alone: grad_head and loss_out must be NULL");
    }
    DMV_REQUIRE(views >= 1 && views <= kMaxViews, DMV_E_UNSUPPORTED_SHAPE, "sampler_fuse_views_loss: need 1 <= views <= 8");
    DMV_REQUIRE(C == 1 || C == 3 || C == 4, DMV_E_UNSUPPORTED_SHAPE, "sampler_fuse_views_loss: need C in {1,3,4}");
    DMV_REQUIRE((long long)views * B < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "sampler_fuse_views_loss: views * B beyond int");
    Geom g;
    int rc = make_geom(g, B, H, W, C, Hout, Wout, flags);
    if (rc) return rc;
    DMV_REQUIRE(g.tw_shift == 5 && ((W * C) & 3) == 0 && ((Wout * C) & 3) == 0, DMV_E_UNSUPPORTED_SHAPE,
                "sampler_fuse_views_loss: needs image-shaped output (Hout > 1) and W*C, Wout*C multiples of 4");
    DMV_REQUIRE((((uintptr_t)data | (uintptr_t)head | (uintptr_t)target | (uintptr_t)fused_out | (uintptr_t)grad_head) & 15) == 0, DMV_E_ALIGN,
                "sampler_fuse_views_loss: buffers must be 16-byte aligned");
    const int grid = g.B * g.tiles_x * g.tiles_y;
    if (train)
        DMV_REQUIRE(workspace && workspace_bytes >= dmv_sampler_loss_workspace_size(B, Hout, Wout) && ((uintptr_t)workspace & 7) == 0,
                    DMV_E_WORKSPACE, "sampler_fuse_views_loss: workspace too small or unaligned (it must be zeroed once and not shared)");
    CUtensorMap map_src, map_src_l, map_fused, map_tgt;
    rc = encode_f32_map(&map_src, data, W * C, H, views * B, kBoxS * C, kBoxS);
    if (!rc) rc = encode_f32_map(&map_src_l, data, W * C, H, views * B, kBoxL * C, kBoxL);
    if (!rc && fused_out) rc = encode_f32_map(&map_fused, fused_out, Wout * C, Hout, B, 32 * C, 32);
    if (!rc && train) rc = encode_f32_map(&map_tgt, target, Wout * C, Hout, B, 32 * C, 32);
    if (rc) return rc;
    if (!fused_out) map_fused = map_src;              // not read: only a valid map to pass
    if (!train) map_tgt = map_src;
    ViewsArgs va;
    va.head = head; va.grad_head = grad_head;
    for (int c = 0; c < 4; ++c) va.w[c] = (train && c < C) ? chan_weight[c] : 0.f;
    va.inv_count = inv_count; va.mode = mode; va.views = views; va.store_fused = fused_out != nullptr;
    va.counter = train ? reinterpret_cast<unsigned*>(workspace) : nullptr;
    va.partials = train ? reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 16) : nullptr;
    va.loss_out = loss_out;
    const size_t wsm = (size_t)(win_floats(C) + (train ? 2 : 1) * 32 * 32 * C) * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
#define DMV_LAUNCH_VIEWS(CT, TR)                                                                                   \
    do {                                                                                                          \
        static bool attr_done = false;                                                                            \
        if (!attr_done) {                                                                                         \
            cudaFuncSetAttribute(sampler_views_kernel<CT, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm); \
            attr_done = true;                                                                                     \
        }                                                                                                         \
        sampler_views_kernel<CT, TR><<<grid, kThreads, wsm, st>>>(map_src, map_src_l, map_fused, map_tgt, data, g, va); \
    } while (0)
    if (train) {
        if (C == 1) DMV_LAUNCH_VIEWS(1, true);
        else if (C == 3) DMV_LAUNCH_VIEWS(3, true);
        else DMV_LAUNCH_VIEWS(4, true);
    } else {
        if (C == 1) DMV_LAUNCH_VIEWS(1, false);
        else if (C == 3) DMV_LAUNCH_VIEWS(3, false);
        else DMV_LAUNCH_VIEWS(4, false);
    }
#undef DMV_LAUNCH_VIEWS
    return check_launch("sampler_loss_fused");
}

}  // extern "C"

// Fused reconstruction loss, its gradient, and the multi-view confidence-weighted fusion
// (SURVEY.md 8(a) L1-L3, 8(f)-3) in one HBM-bound pass: 12C bytes per pixel for V = 1.
//   fused = sum_v softmax_v(logits)_v * gen_v            (V > 1 only)
//   d_c   = (fused_c - target_c) * mask
//   loss  = inv_count * sum_pixels sum_c w_c * (d_c^2  |  |d_c|)
//   dL/dfused_c = inv_count * w_c * mask * (2 d_c | sign(d_c))
//   dL/dgen_v   = softmax_v * dL/dfused ;  dL/dlogit_v = softmax_v * sum_c dL/dfused_c (gen_v,c - fused_c)
// The scalar is reduced deterministically: per-CTA partials in double, summed in index
// order by the last CTA to finish.
// ssim_loss_kernel: the SSIM + L1 loss (below) over [B, H, W, C] images, one 32x32 tile at a time per CTA.
#include "common.cuh"

namespace {
using namespace dmv;

constexpr int kThreads = 256;
constexpr int kMaxC = 8;
constexpr int kMaxV = 8;

struct LossParams {
    const float* gen;
    const float* logits;
    const float* target;
    const float* mask;
    float* grad_gen;
    float* grad_logits;
    float* fused_out;
    float* loss_out;
    double* partials;
    unsigned* counter;
    long long pixels;
    int C, V, mode;
    float inv_count;
    float w[kMaxC];
};

// Last CTA: ordered sum of the per-CTA partials by all its threads (thread t takes partials t, t + 256, ... in order,
// then a fixed tree) -- deterministic, and not one thread walking a thousand dependent loads.
__device__ __forceinline__ void final_sum(const LossParams& p, double* s_red) {
    __threadfence();
    double t = 0.0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += kThreads) t += __ldcg(p.partials + i);
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) tot += s_red[w];
        *p.loss_out = (float)(tot * (double)p.inv_count);
        *p.counter = 0;  // ready for the next launch (stream-ordered)
    }
}

template <int CT>
__global__ void __launch_bounds__(kThreads) loss_kernel(LossParams p) {
    const int C = CT ? CT : p.C;
    const int V = p.V;
    double local = 0.0;
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long px = (long long)blockIdx.x * kThreads + threadIdx.x; px < p.pixels; px += stride) {
        float sm[kMaxV];
        if (V > 1) {
            float mx = -INFINITY;
            for (int v = 0; v < V; ++v) {
                sm[v] = __ldg(p.logits + v * p.pixels + px);
                mx = fmaxf(mx, sm[v]);
            }
            float den = 0.f;
            for (int v = 0; v < V; ++v) {
                sm[v] = __expf(sm[v] - mx);
                den += sm[v];
            }
            const float inv = 1.0f / den;
            for (int v = 0; v < V; ++v) sm[v] *= inv;
        } else {
            sm[0] = 1.0f;
        }
        const float mk = p.mask ? __ldg(p.mask + px) : 1.0f;
        float gl[kMaxV];
        for (int v = 0; v < V; ++v) gl[v] = 0.f;
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < (CT ? CT : kMaxC); ++c) {
            if (!CT && c >= C) break;
            float gv[kMaxV];
            float fused = 0.f;
            for (int v = 0; v < V; ++v) {
                gv[v] = __ldg(p.gen + ((long long)v * p.pixels + px) * C + c);
                fused += sm[v] * gv[v];
            }
            if (V == 1) fused = gv[0];
            if (p.fused_out) p.fused_out[px * C + c] = fused;
            const float d = (fused - __ldg(p.target + px * C + c)) * mk;
            float g;
            if (p.mode == DMV_LOSS_L2) {
                acc += p.w[c] * d * d;
                g = 2.0f * d;
            } else {
                acc += p.w[c] * fabsf(d);
                g = (d > 0.f) ? 1.0f : (d < 0.f ? -1.0f : 0.0f);
            }
            g *= p.w[c] * mk * p.inv_count;
            for (int v = 0; v < V; ++v) {
                if (p.grad_gen) p.grad_gen[((long long)v * p.pixels + px) * C + c] = sm[v] * g;
                gl[v] += g * (gv[v] - fused);
            }
        }
        if (p.grad_logits && V > 1)
            for (int v = 0; v < V; ++v) p.grad_logits[v * p.pixels + px] = sm[v] * gl[v];
        local += (double)acc;
    }
    // block reduction (fixed tree), then ordered final sum by the last CTA
    __shared__ double s_red[kThreads / 32];
    __shared__ bool s_last;
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
        p.partials[blockIdx.x] = t;
        __threadfence();
        const unsigned done = atomicAdd(p.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last) final_sum(p, s_red);
}

// Plain (single view, unmasked) loss over the flat [pixels*C] arrays: float4 loads/stores, channel = index % C.
__global__ void __launch_bounds__(kThreads) loss_flat_kernel(LossParams p) {
    const long long n4 = (p.pixels * p.C) >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(p.gen);
    const float4* t4 = reinterpret_cast<const float4*>(p.target);
    float4* o4 = reinterpret_cast<float4*>(p.grad_gen);
    double local = 0.0;
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n4; i += stride) {
        const float4 a = __ldg(g4 + i), b = __ldg(t4 + i);
        int c = (int)((i * 4) % p.C);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
        float gv[4], acc = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float w = p.w[c];
            const float d = av[k] - bv[k];
            float g;
            if (p.mode == DMV_LOSS_L2) { acc += w * d * d; g = 2.0f * d; }
            else { acc += w * fabsf(d); g = (d > 0.f) ? 1.0f : (d < 0.f ? -1.0f : 0.0f); }
            gv[k] = g * w * p.inv_count;
            if (++c == p.C) c = 0;
        }
        if (o4) o4[i] = make_float4(gv[0], gv[1], gv[2], gv[3]);
        local += (double)acc;
    }
    __shared__ double s_red[kThreads / 32];
    __shared__ bool s_last;
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
        p.partials[blockIdx.x] = t;
        __threadfence();
        const unsigned done = atomicAdd(p.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last) final_sum(p, s_red);
}

// ---------------------------------------------------------------------------------------------
// SSIM + L1 photometric loss (dmv_ssim_loss_fwd_bwd) of one 32x32 tile and its gradient wrt gen.
//
// Per image n and channel c, x = gen, y = target, both reflection-padded by one pixel (row -1 reads row 1, row H reads
// row H-2).  For the 3x3 window centred on every pixel p (Monodepth2's SSIM without its final clamp):
//   mu = mean, s_xx = mean(x^2) - mu_x^2, s_xy = mean(xy) - mu_x mu_y
//   SSIM_p = (2 mu_x mu_y + C1)(2 s_xy + C2) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),  C1 = 0.01^2, C2 = 0.03^2
//   loss   = inv_count * sum_{n,p,c} w_c * (alpha * (1 - SSIM_p,c) / 2 + (1 - alpha) * |x - y|)
// The gradient of window q wrt one of its nine slots k is (1/9)(dS/dmu_x + 2 dS/ds_xx (x_k - mu_x) + dS/ds_xy (y_k - mu_y)),
// i.e. P_q + Q_q x_k + R_q y_k with per-window coefficients (P, Q, R).  A pixel sums them over every window slot that
// reads it: the 3x3 windows around it and, next to the border, the windows that reach it through the reflection
// (pixel row 1 is also padded row -1, covered by the windows of row 0; row H-2 is also padded row H).
//
// Staged layout: s_x, s_y are [C][36 * 36] planar, local (u, v) <-> image (i0 - 2 + u, j0 - 2 + v) reflected into the
// image: the tile, a one-pixel ring of window centres and the ring those windows read.
namespace ssim {

constexpr int kSide = 36;                 // 32 + 2 * 2
constexpr int kArea = kSide * kSide;
constexpr float kC1 = 0.0001f, kC2 = 0.0009f;

struct Args {
    float w[4];
    float alpha;
    float inv_count;
};

// image row / column of padded index i (one-pixel reflection); indices two or more outside are clamped: only windows
// centred outside the image read them, and those windows are not counted
__device__ __forceinline__ int reflect(int i, int n) {
    i = i < 0 ? -i : i;
    i = i >= n ? 2 * n - 2 - i : i;
    return min(max(i, 0), n - 1);
}

// s[c * kArea + (u * 36 + v)] = img[reflect(i0 - 2 + u), reflect(j0 - 2 + v), c]; img is one [H, W, C] image
template <int C>
__device__ __forceinline__ void stage_reflected(float* s, const float* __restrict__ img, int i0, int j0, int H, int W) {
    for (int e = threadIdx.x; e < kArea * C; e += blockDim.x) {
        const int p = e / C, c = e - p * C;
        const int u = p / kSide, v = p - u * kSide;
        const int gi = reflect(i0 - 2 + u, H), gj = reflect(j0 - 2 + v, W);
        s[c * kArea + p] = __ldg(img + ((long long)gi * W + gj) * C + c);
    }
}

// sum over the 3x3 cells around local (u, v) of the three coefficient planes; EDGE: cells outside [0, 36) skipped
template <bool EDGE>
__device__ __forceinline__ void box3(const float* s_k, int u, int v, float& sp, float& sq, float& sr) {
#pragma unroll
    for (int a = u - 1; a <= u + 1; ++a)
#pragma unroll
        for (int b = v - 1; b <= v + 1; ++b) {
            if (EDGE && (a < 0 || a >= kSide || b < 0 || b >= kSide)) continue;
            const int o = a * kSide + b;
            sp = __fadd_rn(sp, s_k[o]);
            sq = __fadd_rn(sq, s_k[kArea + o]);
            sr = __fadd_rn(sr, s_k[2 * kArea + o]);
        }
}

// Loss and dL/dgen of the tile at (i0, j0) of an H x W image.  Expects s_x / s_y staged and visible to every thread;
// s_k is [3][kArea] scratch.  When want_grad, s_x holds dL/dgen (inv_count and the weights applied) at the tile's
// in-image pixels on return (local rows / columns 2..33); other entries of s_x are left undefined.  Returns this thread's
// share of sum w_c * (alpha (1 - SSIM) / 2 + (1 - alpha) |d|), without inv_count.  Ends with the block synchronised.
template <int C>
__device__ float tile_loss_grad(float* s_x, const float* s_y, float* s_k, int i0, int j0, int H, int W, const Args& a, bool want_grad) {
    const int tid = threadIdx.x;
    const float inv9 = 1.0f / 9.0f;
    const float beta = __fsub_rn(1.0f, a.alpha);
    float acc = 0.f;
#pragma unroll 1
    for (int c = 0; c < C; ++c) {
        const float* x = s_x + c * kArea;
        const float* y = s_y + c * kArea;
        const float k_ssim = __fmul_rn(__fmul_rn(a.alpha, 0.5f), a.w[c]);             // loss of a window: k (1 - S)
        const float gk = -__fmul_rn(__fmul_rn(k_ssim, a.inv_count), inv9);         // dL/dS * (1/9) with inv_count
        // window statistics and coefficients at every local centre; zero where the centre is not an image pixel
        for (int e = tid; e < kArea; e += blockDim.x) {
            const int u = e / kSide, v = e - u * kSide;
            const int gi = i0 - 2 + u, gj = j0 - 2 + v;
            float P = 0.f, Q = 0.f, R = 0.f;
            if (u >= 1 && u < kSide - 1 && v >= 1 && v < kSide - 1 && gi >= 0 && gi < H && gj >= 0 && gj < W) {
                float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;
#pragma unroll
                for (int du = -1; du <= 1; ++du)
#pragma unroll
                    for (int dv = -1; dv <= 1; ++dv) {
                        const float xv = x[e + du * kSide + dv], yv = y[e + du * kSide + dv];
                        sx = __fadd_rn(sx, xv);
                        sy = __fadd_rn(sy, yv);
                        sxx = __fmaf_rn(xv, xv, sxx);
                        syy = __fmaf_rn(yv, yv, syy);
                        sxy = __fmaf_rn(xv, yv, sxy);
                    }
                const float mx = __fmul_rn(sx, inv9), my = __fmul_rn(sy, inv9);
                const float vx = __fmaf_rn(-mx, mx, __fmul_rn(sxx, inv9));
                const float vy = __fmaf_rn(-my, my, __fmul_rn(syy, inv9));
                const float cxy = __fmaf_rn(-mx, my, __fmul_rn(sxy, inv9));
                const float A1 = __fmaf_rn(__fmul_rn(2.0f, mx), my, kC1);
                const float A2 = __fmaf_rn(2.0f, cxy, kC2);
                const float B1 = __fmaf_rn(mx, mx, __fmaf_rn(my, my, kC1));
                const float B2 = __fadd_rn(__fadd_rn(vx, vy), kC2);
                const float rden = __fdiv_rn(1.0f, __fmul_rn(B1, B2));
                const float S = __fmul_rn(__fmul_rn(A1, A2), rden);
                if (u >= 2 && u < kSide - 2 && v >= 2 && v < kSide - 2)          // a tile pixel: its window's loss
                    acc = __fmaf_rn(k_ssim, __fsub_rn(1.0f, S), acc);
                // dS/dmu_x = 2 (mu_y A2 - mu_x S B2) / (B1 B2), dS/ds_xx = -S / B2 = -S B1 / (B1 B2), dS/ds_xy = 2 A1 / (B1 B2)
                const float dmu = __fmul_rn(2.0f, __fmul_rn(__fmaf_rn(my, A2, -__fmul_rn(__fmul_rn(mx, S), B2)), rden));
                const float dvx = -__fmul_rn(__fmul_rn(S, B1), rden);
                const float dcv = __fmul_rn(__fmul_rn(2.0f, A1), rden);
                // slot k: (1/9)(dmu + 2 dvx (x_k - mu_x) + dcv (y_k - mu_y)) = P + Q x_k + R y_k
                P = __fmul_rn(gk, __fsub_rn(__fsub_rn(dmu, __fmul_rn(__fmul_rn(2.0f, dvx), mx)), __fmul_rn(dcv, my)));
                Q = __fmul_rn(gk, __fmul_rn(2.0f, dvx));
                R = __fmul_rn(gk, dcv);
            }
            s_k[e] = P;
            s_k[kArea + e] = Q;
            s_k[2 * kArea + e] = R;
        }
        __syncthreads();
        // per tile pixel: the L1 term, and dL/dgen from every window slot that reads it
        const float kl1 = __fmul_rn(beta, a.w[c]);
        const float gl1 = __fmul_rn(kl1, a.inv_count);
        for (int e = tid; e < 32 * 32; e += blockDim.x) {
            const int r = e >> 5, col = e & 31;
            const int gi = i0 + r, gj = j0 + col;
            if (gi >= H || gj >= W) continue;
            const int u = r + 2, v = col + 2, o = u * kSide + v;
            const float xv = x[o], yv = y[o];
            const float d = __fsub_rn(xv, yv);
            acc = __fmaf_rn(kl1, fabsf(d), acc);
            if (!want_grad) continue;
            float sp = 0.f, sq = 0.f, sr = 0.f;
            box3<false>(s_k, u, v, sp, sq, sr);
            // padded preimages of this pixel other than itself: row -1 (local u - 2) for row 1, row H for row H - 2
            const int ru[2] = {gi == 1 ? u - 2 : -1, gi == H - 2 ? u + 2 : -1};
            const int cv[2] = {gj == 1 ? v - 2 : -1, gj == W - 2 ? v + 2 : -1};
            for (int ia = -1; ia < 2; ++ia) {
                const int uu = ia < 0 ? u : ru[ia];
                if (uu < 0) continue;
                for (int ib = -1; ib < 2; ++ib) {
                    const int vv = ib < 0 ? v : cv[ib];
                    if (vv < 0 || (ia < 0 && ib < 0)) continue;
                    box3<true>(s_k, uu, vv, sp, sq, sr);
                }
            }
            const float sgn = (d > 0.f) ? 1.0f : (d < 0.f ? -1.0f : 0.0f);
            float g = __fadd_rn(sp, __fmul_rn(sq, xv));
            g = __fadd_rn(g, __fmul_rn(sr, yv));
            g = __fadd_rn(g, __fmul_rn(sgn, gl1));
            s_x[c * kArea + o] = g;      // only this thread reads x[o] in this pass
        }
        __syncthreads();                 // s_k is rewritten by the next channel
    }
    return acc;
}

}  // namespace ssim

// SSIM + L1.  Each CTA takes 32x32 tiles blockIdx.x, blockIdx.x + gridDim.x, ... in order: gen and target
// staged with a 2-pixel halo, reflected at the border; the per-CTA sum of its tiles' losses joins the ordered final sum.
struct SsimShape {
    int B, H, W, tiles_x, tiles_y;
    ssim::Args a;
};

template <int C>
__global__ void __launch_bounds__(kThreads, 3) ssim_loss_kernel(LossParams p, SsimShape sh) {
    extern __shared__ float s_ssim[];
    float* s_x = s_ssim;                        // [C][36 * 36] gen, then dL/dgen at the tile pixels
    float* s_y = s_x + C * ssim::kArea;         // [C][36 * 36] target
    float* s_k = s_y + C * ssim::kArea;         // [3][36 * 36] window coefficients
    const int per_img = sh.tiles_x * sh.tiles_y;
    const long long img_floats = (long long)sh.H * sh.W * C;
    double local = 0.0;
    for (int tile = blockIdx.x; tile < sh.B * per_img; tile += gridDim.x) {
        const int b = tile / per_img, t = tile - b * per_img;
        const int i0 = (t / sh.tiles_x) * 32, j0 = (t % sh.tiles_x) * 32;
        __syncthreads();                        // the previous tile's gradient has been written out
        ssim::stage_reflected<C>(s_x, p.gen + b * img_floats, i0, j0, sh.H, sh.W);
        ssim::stage_reflected<C>(s_y, p.target + b * img_floats, i0, j0, sh.H, sh.W);
        __syncthreads();
        local += (double)ssim::tile_loss_grad<C>(s_x, s_y, s_k, i0, j0, sh.H, sh.W, sh.a, p.grad_gen != nullptr);
        if (p.grad_gen) {
            float* dst = p.grad_gen + b * img_floats;
            for (int e = threadIdx.x; e < 32 * 32 * C; e += kThreads) {
                const int q = e / C, c = e - q * C;
                const int r = q >> 5, col = q & 31;
                if (i0 + r < sh.H && j0 + col < sh.W)
                    dst[((long long)(i0 + r) * sh.W + j0 + col) * C + c] = s_x[c * ssim::kArea + (r + 2) * ssim::kSide + col + 2];
            }
        }
    }
    __shared__ double s_red[kThreads / 32];
    __shared__ bool s_last;
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
        p.partials[blockIdx.x] = t;
        __threadfence();
        const unsigned done = atomicAdd(p.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last) final_sum(p, s_red);
}

__global__ void scale_kernel(float* x, const float* s, long long n) {
    const float k = __ldg(s);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] *= k;
}

constexpr int kMaxBlocks = 148 * 8;
}  // namespace

extern "C" {

size_t dmv_loss_workspace_size(long long pixels) {
    (void)pixels;
    return (size_t)kMaxBlocks * sizeof(double) + 16;
}

int dmv_loss_fused_fwd_bwd(const float* gen, const float* logits, int V, const float* target, const float* mask,
                           const float* chan_weight, int mode, float inv_count, float* loss_out, float* grad_gen,
                           float* grad_logits, float* fused_out, long long pixels, int C, void* workspace,
                           size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(gen && target && loss_out && chan_weight, DMV_E_INVALID_ARG, "loss: null pointer");
    DMV_REQUIRE(pixels > 0 && C > 0 && C <= kMaxC, DMV_E_UNSUPPORTED_SHAPE, "loss: need 1 <= C <= 8");
    DMV_REQUIRE(V >= 1 && V <= kMaxV, DMV_E_UNSUPPORTED_SHAPE, "loss: need 1 <= V <= 8");
    DMV_REQUIRE(V == 1 || logits, DMV_E_INVALID_ARG, "loss: V > 1 needs confidence logits");
    DMV_REQUIRE(mode == DMV_LOSS_L2 || mode == DMV_LOSS_L1, DMV_E_INVALID_ARG, "loss: unknown mode");
    DMV_REQUIRE(workspace && workspace_bytes >= dmv_loss_workspace_size(pixels), DMV_E_WORKSPACE, "loss: workspace too small");
    DMV_REQUIRE(((uintptr_t)workspace & 7) == 0, DMV_E_ALIGN, "loss: workspace must be 8-byte aligned");
    LossParams p;
    p.gen = gen; p.logits = logits; p.target = target; p.mask = mask;
    p.grad_gen = grad_gen; p.grad_logits = grad_logits; p.fused_out = fused_out; p.loss_out = loss_out;
    p.partials = reinterpret_cast<double*>(workspace);
    p.counter = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(workspace) + kMaxBlocks * sizeof(double));
    p.pixels = pixels; p.C = C; p.V = V; p.mode = mode; p.inv_count = inv_count;
    for (int c = 0; c < kMaxC; ++c) p.w[c] = c < C ? chan_weight[c] : 0.f;
    long long blocks = dmv::ceil_div_ll(pixels, kThreads);
    if (blocks > kMaxBlocks) blocks = kMaxBlocks;
    cudaStream_t st = (cudaStream_t)stream;
    const bool flat = V == 1 && !mask && !fused_out && ((pixels * C) % 4 == 0) &&
                      ((((uintptr_t)gen | (uintptr_t)target | (uintptr_t)grad_gen) & 15) == 0);
    if (flat) {
        long long fb = dmv::ceil_div_ll(pixels * C / 4, kThreads * 4);
        if (fb > kMaxBlocks) fb = kMaxBlocks;
        if (fb < 1) fb = 1;
        loss_flat_kernel<<<(int)fb, kThreads, 0, st>>>(p);
        return dmv::check_launch("loss_flat");
    }
    switch (C) {
        case 1: loss_kernel<1><<<(int)blocks, kThreads, 0, st>>>(p); break;
        case 3: loss_kernel<3><<<(int)blocks, kThreads, 0, st>>>(p); break;
        case 4: loss_kernel<4><<<(int)blocks, kThreads, 0, st>>>(p); break;
        default: loss_kernel<0><<<(int)blocks, kThreads, 0, st>>>(p); break;
    }
    return dmv::check_launch("loss_fused");
}

int dmv_ssim_loss_fwd_bwd(const float* gen, const float* target, const float* chan_weight, float alpha, float inv_count, float* loss_out,
                          float* grad_gen, int B, int H, int W, int C, void* workspace, size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(gen && target && chan_weight && loss_out, DMV_E_INVALID_ARG, "ssim_loss: null pointer");
    DMV_REQUIRE(alpha >= 0.f && alpha <= 1.f, DMV_E_INVALID_ARG, "ssim_loss: alpha must lie in [0, 1]");
    DMV_REQUIRE(C == 1 || C == 3 || C == 4, DMV_E_UNSUPPORTED_SHAPE, "ssim_loss: need C in {1,3,4}");
    DMV_REQUIRE(B > 0 && H >= 2 && W >= 2, DMV_E_UNSUPPORTED_SHAPE, "ssim_loss: need B >= 1 and H, W >= 2 (the reflection pad)");
    const long long pixels = (long long)B * H * W;
    DMV_REQUIRE(workspace && workspace_bytes >= dmv_loss_workspace_size(pixels), DMV_E_WORKSPACE, "ssim_loss: workspace too small");
    DMV_REQUIRE(((uintptr_t)workspace & 7) == 0, DMV_E_ALIGN, "ssim_loss: workspace must be 8-byte aligned");
    SsimShape sh;
    sh.B = B; sh.H = H; sh.W = W;
    sh.tiles_x = dmv::ceil_div(W, 32);
    sh.tiles_y = dmv::ceil_div(H, 32);
    DMV_REQUIRE((long long)B * sh.tiles_x * sh.tiles_y < (1ll << 31), DMV_E_UNSUPPORTED_SHAPE, "ssim_loss: too many tiles");
    for (int c = 0; c < 4; ++c) sh.a.w[c] = c < C ? chan_weight[c] : 0.f;
    sh.a.alpha = alpha;
    sh.a.inv_count = inv_count;
    LossParams p = {};
    p.gen = gen; p.target = target; p.grad_gen = grad_gen; p.loss_out = loss_out;
    p.partials = reinterpret_cast<double*>(workspace);
    p.counter = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(workspace) + kMaxBlocks * sizeof(double));
    p.pixels = pixels; p.C = C; p.V = 1; p.inv_count = inv_count;
    long long blocks = (long long)B * sh.tiles_x * sh.tiles_y;
    if (blocks > kMaxBlocks) blocks = kMaxBlocks;
    const size_t smem = (size_t)(2 * C + 3) * ssim::kArea * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
#define DMV_LAUNCH_SSIM(CT)                                                                                       \
    do {                                                                                                          \
        static bool attr_done = false;                                                                            \
        if (!attr_done) {                                                                                         \
            cudaFuncSetAttribute(ssim_loss_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
            attr_done = true;                                                                                     \
        }                                                                                                         \
        ssim_loss_kernel<CT><<<(int)blocks, kThreads, smem, st>>>(p, sh);                                         \
    } while (0)
    if (C == 1) DMV_LAUNCH_SSIM(1);
    else if (C == 3) DMV_LAUNCH_SSIM(3);
    else DMV_LAUNCH_SSIM(4);
#undef DMV_LAUNCH_SSIM
    return check_launch("loss_fused");
}

int dmv_scale_by_device_scalar(float* x, const float* scalar, long long n, void* stream) {
    DMV_REQUIRE(x && scalar && n >= 0, DMV_E_INVALID_ARG, "scale: bad argument");
    if (n == 0) return DMV_OK;
    long long blocks = dmv::ceil_div_ll(n, 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    scale_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(x, scalar, n);
    return dmv::check_launch("scale");
}
}

// CUDA-core (SIMT) conv / deconv / linear kernels: the bring-up path and the on-GPU
// cross-check for the tcgen05 implicit-GEMM kernels (DMV_ALGO_SIMT).  bf16 (or fp32 image)
// operands, fp32 accumulation, TF-SAME padding (SURVEY.md 8(a) C1, C2, F1).
//
// Three kernel forms over one geometry cover all nine entry points.  "big" is the side a
// SAME conv reads (H x W x Cin), "small" the side it writes (Ho x Wo x Cout); weights are
// w[r][s][ci][co] with ci on the big side:
//   F  small[n,oh,ow,co] = act( sum_{r,s,ci} big[n,oh*st+r-pt,ow*st+s-pl,ci] w[r,s,ci,co] + b[co] )
//        conv fwd (big = x), deconv dgrad (big = dy)
//   G  big[n,ih,iw,ci]   = act( sum_{r,s,co} small[n,(ih+pt-r)/st,(iw+pl-s)/st,co] w[r,s,ci,co] )
//        conv dgrad (small = dy), deconv fwd (small = x; tf.nn.conv2d_transpose is by
//        definition the input-gradient of a SAME conv)
//   W  dw[r,s,ci,co]     = sum_{n,oh,ow} big[...,ci] * small[n,oh,ow,co]
//        conv wgrad (big = x, small = dy), deconv wgrad (big = dy, small = x)
// W is a deterministic split-K: partial tiles go to the workspace and a second kernel adds
// them in split order.
#include "common.cuh"
#include "conv_impl.h"

namespace {
using namespace dmv;
typedef __nv_bfloat16 bf16;

struct ConvGeom {
    int B, H, W, Cin, Ho, Wo, Cout, kh, kw, st, pt, pl;
};

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 t = __bfloat1622float2(p[k]);
        f[2 * k] = t.x;
        f[2 * k + 1] = t.y;
    }
}

// ---------------------------------------------------------------- form F
template <typename TX, typename TY>
__global__ void __launch_bounds__(128) conv_f_kernel(const TX* __restrict__ X, const bf16* __restrict__ Wt,
                                                      const float* __restrict__ bias, TY* __restrict__ Y, ConvGeom g, int act) {
    const long long total = (long long)g.B * g.Ho * g.Wo;
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int co0 = blockIdx.y * 8;
    if (pix >= total) return;
    const int ow = (int)(pix % g.Wo);
    const int oh = (int)((pix / g.Wo) % g.Ho);
    const int n = (int)(pix / ((long long)g.Wo * g.Ho));
    const bool wvec = (g.Cout % 8 == 0);
    const int nco = min(8, g.Cout - co0);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int r = 0; r < g.kh; ++r) {
        const int ih = oh * g.st + r - g.pt;
        if (ih < 0 || ih >= g.H) continue;
        for (int s = 0; s < g.kw; ++s) {
            const int iw = ow * g.st + s - g.pl;
            if (iw < 0 || iw >= g.W) continue;
            const TX* xp = X + (((long long)n * g.H + ih) * g.W + iw) * g.Cin;
            const bf16* wp = Wt + ((long long)(r * g.kw + s) * g.Cin) * g.Cout + co0;
            for (int ci = 0; ci < g.Cin; ++ci) {
                const float xv = load_as_float(xp + ci);
                if (wvec) {
                    float wf[8];
                    unpack8(__ldg(reinterpret_cast<const uint4*>(wp + (long long)ci * g.Cout)), wf);
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv, wf[j], acc[j]);
                } else {
                    for (int j = 0; j < nco; ++j) acc[j] = fmaf(xv, bf2f(wp[(long long)ci * g.Cout + j]), acc[j]);
                }
            }
        }
    }
    TY* yp = Y + pix * g.Cout + co0;
    for (int j = 0; j < nco; ++j) {
        float v = acc[j] + (bias ? __ldg(bias + co0 + j) : 0.f);
        store_from_float(yp + j, apply_act(v, act));
    }
}

// ---------------------------------------------------------------- form G
template <typename TS, typename TB>
__global__ void __launch_bounds__(128) conv_g_kernel(const TS* __restrict__ S, const bf16* __restrict__ Wt,
                                                      TB* __restrict__ Bg, ConvGeom g, int act) {
    const long long total = (long long)g.B * g.H * g.W;
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int ci0 = blockIdx.y * 8;
    if (pix >= total) return;
    const int iw = (int)(pix % g.W);
    const int ih = (int)((pix / g.W) % g.H);
    const int n = (int)(pix / ((long long)g.W * g.H));
    const int nci = min(8, g.Cin - ci0);
    const bool vec = (g.Cout % 8 == 0) && (sizeof(TS) == 2);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int r = 0; r < g.kh; ++r) {
        const int t = ih + g.pt - r;
        if (t < 0 || (t % g.st) != 0) continue;
        const int oh = t / g.st;
        if (oh >= g.Ho) continue;
        for (int s = 0; s < g.kw; ++s) {
            const int u = iw + g.pl - s;
            if (u < 0 || (u % g.st) != 0) continue;
            const int ow = u / g.st;
            if (ow >= g.Wo) continue;
            const TS* sp = S + (((long long)n * g.Ho + oh) * g.Wo + ow) * g.Cout;
            const bf16* wp = Wt + ((long long)(r * g.kw + s) * g.Cin + ci0) * g.Cout;
            if (vec) {
                for (int co = 0; co < g.Cout; co += 8) {
                    float sv[8];
                    unpack8(*reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(sp) + co), sv);
                    for (int j = 0; j < nci; ++j) {
                        float wf[8];
                        unpack8(__ldg(reinterpret_cast<const uint4*>(wp + (long long)j * g.Cout + co)), wf);
                        float d = 0.f;
#pragma unroll
                        for (int k = 0; k < 8; ++k) d = fmaf(sv[k], wf[k], d);
                        acc[j] += d;
                    }
                }
            } else {
                for (int co = 0; co < g.Cout; ++co) {
                    const float sv = load_as_float(sp + co);
                    for (int j = 0; j < nci; ++j) acc[j] = fmaf(sv, bf2f(wp[(long long)j * g.Cout + co]), acc[j]);
                }
            }
        }
    }
    TB* bp = Bg + pix * g.Cin + ci0;
    for (int j = 0; j < nci; ++j) store_from_float(bp + j, apply_act(acc[j], act));
}

// ---------------------------------------------------------------- form W
constexpr int kWT = 32;  // ci x co tile
template <typename TBig, typename TSm>
__global__ void __launch_bounds__(256) conv_w_kernel(const TBig* __restrict__ Big, const TSm* __restrict__ Sm,
                                                      float* __restrict__ part, ConvGeom g, int ci_tiles, int co_tiles,
                                                      long long chunk) {
    __shared__ float xs[32][kWT + 1];
    __shared__ float ys[32][kWT + 1];
    int t = blockIdx.x;
    const int cot = t % co_tiles; t /= co_tiles;
    const int cit = t % ci_tiles; t /= ci_tiles;
    const int tap = t;
    const int r = tap / g.kw, s = tap - r * g.kw;
    const int ci0 = cit * kWT, co0 = cot * kWT;
    const long long total = (long long)g.B * g.Ho * g.Wo;
    const long long p_begin = (long long)blockIdx.y * chunk;
    const long long p_end = min(total, p_begin + chunk);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // thread computes ci {ty, ty+16} x co {tx, tx+16}
    const int lp = threadIdx.x >> 3, lc = (threadIdx.x & 7) * 4;  // loader: pixel lp, channels lc..lc+3
    float a00 = 0.f, a01 = 0.f, a10 = 0.f, a11 = 0.f;
    for (long long p0 = p_begin; p0 < p_end; p0 += 32) {
        const long long p = p0 + lp;
        float xv[4] = {0.f, 0.f, 0.f, 0.f}, yv[4] = {0.f, 0.f, 0.f, 0.f};
        if (p < p_end) {
            const int ow = (int)(p % g.Wo);
            const int oh = (int)((p / g.Wo) % g.Ho);
            const int n = (int)(p / ((long long)g.Wo * g.Ho));
            const int ih = oh * g.st + r - g.pt, iw = ow * g.st + s - g.pl;
            if (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) {
                const TBig* xp = Big + (((long long)n * g.H + ih) * g.W + iw) * g.Cin + ci0 + lc;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (ci0 + lc + k < g.Cin) xv[k] = load_as_float(xp + k);
            }
            const TSm* yp = Sm + p * g.Cout + co0 + lc;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (co0 + lc + k < g.Cout) yv[k] = load_as_float(yp + k);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            xs[lp][lc + k] = xv[k];
            ys[lp][lc + k] = yv[k];
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const float x0 = xs[q][ty], x1 = xs[q][ty + 16], y0 = ys[q][tx], y1 = ys[q][tx + 16];
            a00 = fmaf(x0, y0, a00);
            a01 = fmaf(x0, y1, a01);
            a10 = fmaf(x1, y0, a10);
            a11 = fmaf(x1, y1, a11);
        }
    }
    float* out = part + (long long)blockIdx.y * g.kh * g.kw * g.Cin * g.Cout + (long long)tap * g.Cin * g.Cout;
    const int ci_a = ci0 + ty, ci_b = ci0 + ty + 16, co_a = co0 + tx, co_b = co0 + tx + 16;
    if (ci_a < g.Cin && co_a < g.Cout) out[(long long)ci_a * g.Cout + co_a] = a00;
    if (ci_a < g.Cin && co_b < g.Cout) out[(long long)ci_a * g.Cout + co_b] = a01;
    if (ci_b < g.Cin && co_a < g.Cout) out[(long long)ci_b * g.Cout + co_a] = a10;
    if (ci_b < g.Cin && co_b < g.Cout) out[(long long)ci_b * g.Cout + co_b] = a11;
}

template <int ZW>
__global__ void __launch_bounds__(32 * ZW) reduce_partials_kernel(const float* __restrict__ part, float* __restrict__ out, long long n,
                                                                   int splits) {
    __shared__ float red[ZW][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long i = (long long)blockIdx.x * 32 + lane;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (i < n) {
        int z = w;
        for (; z + 3 * ZW < splits; z += 4 * ZW) {      // four independent loads in flight, added in z order
            const float a = part[(long long)z * n + i], b = part[(long long)(z + ZW) * n + i];
            const float c = part[(long long)(z + 2 * ZW) * n + i], d = part[(long long)(z + 3 * ZW) * n + i];
            s0 += a; s1 += b; s2 += c; s3 += d;
        }
        for (; z < splits; z += ZW) s0 += part[(long long)z * n + i];
    }
    red[w][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (w == 0 && i < n) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < ZW; ++k) t += red[k][lane];
        out[i] = t;
    }
}

// column sums of a [pixels, C] matrix (bias gradient), deterministic two-stage
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ Y, float* __restrict__ part, long long pixels, int C,
                                                      long long chunk) {
    __shared__ float red[8][33];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int lane_p = threadIdx.x >> 5;
    const long long p_begin = (long long)blockIdx.y * chunk, p_end = min(pixels, p_begin + chunk);
    float s = 0.f;
    if (c < C)
        for (long long p = p_begin + lane_p; p < p_end; p += 8) s += load_as_float(Y + p * C + c);
    red[lane_p][threadIdx.x & 31] = s;
    __syncthreads();
    if (lane_p == 0 && c < C) {
        float t = 0.f;
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x & 31];
        part[(long long)blockIdx.y * C + c] = t;
    }
}

// dpre = dy * act'(y) fused with the bias gradient db[c] = sum_rows dpre[row][c]  (bf16 [rows][C], C % 8 == 0).
// CTA = (CGB column groups of 8 channels) x (256/CGB row lanes) over a contiguous row range; grid.x tiles the
// columns, grid.y the rows.  Four rows are in flight per thread.  CTA partials are summed in grid.y order by
// reduce_partials (deterministic).
// GROUPED (dmv_act_bwd_bias_grouped): row r of dy is the fp32 sum, in t order, of dy rows r * group + t (row pitch ld8
// uint4s); the ungrouped instantiation compiles exactly the plain kernel.
template <bool GROUPED>
__global__ void __launch_bounds__(256) act_bwd_bias_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ y, uint4* __restrict__ dpre,
                                                            float* __restrict__ part, long long rows, int C8, int cgb, long long rows_per_cta,
                                                            int act, int group, long long ld8) {
    __shared__ float red[256][9];
    float sum[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) sum[k] = 0.f;
    const int cl = threadIdx.x % cgb, rl = threadIdx.x / cgb, rstep = 256 / cgb;
    const int cg = blockIdx.x * cgb + cl;
    const long long r0 = (long long)blockIdx.y * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
    auto one = [&](const uint4& a, const uint4& b) {
        uint4 o;
        const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
        __nv_bfloat162* po = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fa = __bfloat1622float2(pa[k]), fb = __bfloat1622float2(pb[k]);
            po[k] = __floats2bfloat162_rn(fa.x * act_grad_from_output(fb.x, act), fa.y * act_grad_from_output(fb.y, act));
            const float2 q = __bfloat1622float2(po[k]);     // the bias gradient sums exactly what wgrad/dgrad will read
            sum[2 * k] += q.x;
            sum[2 * k + 1] += q.y;
        }
        return o;
    };
    long long r = r0 + rl;
    if constexpr (GROUPED) {
        struct F8 { float v[8]; };
        auto gsum = [&](long long row) {          // fp32 sum of the group's dy rows, t = 0 .. group-1 in order
            const uint4* p = dy + row * group * ld8 + cg;
            F8 s;
            uint4 q = __ldg(p);
            const __nv_bfloat162* pq = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = __bfloat1622float2(pq[k]);
                s.v[2 * k] = f.x;
                s.v[2 * k + 1] = f.y;
            }
            for (int t = 1; t < group; ++t) {
                q = __ldg(p + t * ld8);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = __bfloat1622float2(pq[k]);
                    s.v[2 * k] += f.x;
                    s.v[2 * k + 1] += f.y;
                }
            }
            return s;
        };
        auto onef = [&](const F8& a, const uint4& b) {
            uint4 o;
            const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
            __nv_bfloat162* po = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 fb = __bfloat1622float2(pb[k]);
                po[k] = __floats2bfloat162_rn(a.v[2 * k] * act_grad_from_output(fb.x, act), a.v[2 * k + 1] * act_grad_from_output(fb.y, act));
                const float2 q = __bfloat1622float2(po[k]);
                sum[2 * k] += q.x;
                sum[2 * k + 1] += q.y;
            }
            return o;
        };
        for (; r + 3LL * rstep < r1; r += 4LL * rstep) {
            F8 a[4];
            uint4 b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                a[u] = gsum(r + (long long)u * rstep);
                b[u] = __ldg(y + (r + (long long)u * rstep) * C8 + cg);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) dpre[(r + (long long)u * rstep) * C8 + cg] = onef(a[u], b[u]);
        }
        for (; r < r1; r += rstep) {
            const long long i = r * C8 + cg;
            dpre[i] = onef(gsum(r), __ldg(y + i));
        }
    } else {
        for (; r + 3LL * rstep < r1; r += 4LL * rstep) {
            uint4 a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const long long i = (r + (long long)u * rstep) * C8 + cg;
                a[u] = __ldg(dy + i);
                b[u] = __ldg(y + i);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) dpre[(r + (long long)u * rstep) * C8 + cg] = one(a[u], b[u]);
        }
        for (; r < r1; r += rstep) {
            const long long i = r * C8 + cg;
            dpre[i] = one(__ldg(dy + i), __ldg(y + i));
        }
    }
    // reduce over the row lanes: shuffles inside the warp (lanes sharing a column group are cgb apart),
    // then across the 8 warps through shared memory, in a fixed order
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int off = cgb; off < 32; off <<= 1)
#pragma unroll
        for (int k = 0; k < 8; ++k) sum[k] += __shfl_xor_sync(0xffffffffu, sum[k], off);
    const int slots = cgb < 32 ? cgb : 32;
    if (lane < slots)
#pragma unroll
        for (int k = 0; k < 8; ++k) red[warp * 32 + lane][k] = sum[k];
    __syncthreads();
    for (int t = threadIdx.x; t < cgb * 8; t += 256) {
        const int c = t >> 3, k = t & 7;
        float acc = 0.f;
        if (cgb <= 32) {
            for (int w = 0; w < 8; ++w) acc += red[w * 32 + c][k];
        } else {                                  // cgb == 64: even warps hold columns 0..31, odd warps 32..63
            for (int w = (c >> 5); w < 8; w += 2) acc += red[w * 32 + (c & 31)][k];
        }
        part[((long long)blockIdx.y * C8 + blockIdx.x * cgb + c) * 8 + k] = acc;
    }
}

int make_geom(ConvGeom& g, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride) {
    DMV_REQUIRE(B > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && kh > 0 && kw > 0 && stride > 0, DMV_E_INVALID_ARG,
                "conv: non-positive dimension");
    const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
    g.B = B; g.H = H; g.W = W; g.Cin = Cin; g.Ho = ph.out; g.Wo = pw.out; g.Cout = Cout;
    g.kh = kh; g.kw = kw; g.st = stride; g.pt = ph.before; g.pl = pw.before;
    return DMV_OK;
}

struct SplitPlan {
    int ci_tiles, co_tiles, splits;
    long long chunk;
};
SplitPlan plan_split(int taps, int Cin, int Cout, long long pixels) {
    SplitPlan p;
    p.ci_tiles = ceil_div(Cin, kWT);
    p.co_tiles = ceil_div(Cout, kWT);
    const long long tiles = (long long)taps * p.ci_tiles * p.co_tiles;
    long long want = ceil_div_ll(148 * 8, tiles);
    long long max_by_pixels = ceil_div_ll(pixels, 1024);
    long long s = want < max_by_pixels ? want : max_by_pixels;
    if (s < 1) s = 1;
    if (s > 512) s = 512;
    p.chunk = ceil_div_ll(ceil_div_ll(pixels, s), 32) * 32;
    p.splits = (int)ceil_div_ll(pixels, p.chunk);
    return p;
}

template <typename TBig, typename TSm>
int run_wgrad(const TBig* big, const TSm* sm, float* dw, const ConvGeom& g, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int taps = g.kh * g.kw;
    const long long pixels = (long long)g.B * g.Ho * g.Wo;
    const SplitPlan p = plan_split(taps, g.Cin, g.Cout, pixels);
    const long long n = (long long)taps * g.Cin * g.Cout;
    DMV_REQUIRE(ws && ws_bytes >= (size_t)p.splits * n * sizeof(float), DMV_E_WORKSPACE, "wgrad: workspace too small");
    float* part = reinterpret_cast<float*>(ws);
    dim3 grid(taps * p.ci_tiles * p.co_tiles, p.splits);
    conv_w_kernel<TBig, TSm><<<grid, 256, 0, st>>>(big, sm, part, g, p.ci_tiles, p.co_tiles, p.chunk);
    int rc = check_launch("conv_wgrad_simt");
    if (rc) return rc;
    long long blocks = ceil_div_ll(n, 256);
    (void)blocks;
    return reduce_partials(part, dw, n, p.splits, st);
}

template <typename T>
int run_colsum(const T* y, float* db, long long pixels, int C, void* ws, size_t ws_bytes, cudaStream_t st) {
    long long splits = ceil_div_ll(pixels, 2048);
    if (splits > 256) splits = 256;
    const long long chunk = ceil_div_ll(pixels, splits);
    splits = ceil_div_ll(pixels, chunk);
    DMV_REQUIRE(ws && ws_bytes >= (size_t)splits * C * sizeof(float), DMV_E_WORKSPACE, "bias grad: workspace too small");
    float* part = reinterpret_cast<float*>(ws);
    dim3 grid(ceil_div(C, 32), (int)splits);
    colsum_kernel<T><<<grid, 256, 0, st>>>(y, part, pixels, C, chunk);
    int rc = check_launch("colsum");
    if (rc) return rc;
    return reduce_partials(part, db, C, (int)splits, st);
}

template <typename TX, typename TY>
int run_f(const void* x, const void* w, const float* bias, void* y, const ConvGeom& g, int act, cudaStream_t st) {
    const long long pixels = (long long)g.B * g.Ho * g.Wo;
    dim3 grid((unsigned)ceil_div_ll(pixels, 128), ceil_div(g.Cout, 8));
    conv_f_kernel<TX, TY><<<grid, 128, 0, st>>>((const TX*)x, (const bf16*)w, bias, (TY*)y, g, act);
    return check_launch("conv_f_simt");
}
template <typename TS, typename TB>
int run_g(const void* s, const void* w, void* b, const ConvGeom& g, int act, cudaStream_t st) {
    const long long pixels = (long long)g.B * g.H * g.W;
    dim3 grid((unsigned)ceil_div_ll(pixels, 128), ceil_div(g.Cin, 8));
    conv_g_kernel<TS, TB><<<grid, 128, 0, st>>>((const TS*)s, (const bf16*)w, (TB*)b, g, act);
    return check_launch("conv_g_simt");
}

}  // namespace

// ------------------------------------------------------------------ SIMT entry points
// (called by the public dispatchers in conv_api.cu)
namespace dmv {

int reduce_partials(const float* part, float* out, long long n, int splits, cudaStream_t st) {
    const long long blocks = ceil_div_ll(n, 32);
    // few columns: spread z over many warps; many columns: enough CTAs already, keep the chains per thread short anyway
    if (blocks >= 148 * 8 || splits <= 8) reduce_partials_kernel<4><<<(unsigned)blocks, 128, 0, st>>>(part, out, n, splits);
    else if (blocks >= 148 || splits <= 32) reduce_partials_kernel<8><<<(unsigned)blocks, 256, 0, st>>>(part, out, n, splits);
    // few columns, many partials (bias gradients): 16 warps.  (32 warps of 32 registers are half a register file: such a
    // CTA cannot become resident next to a persistent 512-thread kernel and stalled the input-gradient chain behind the
    // fused FC update for up to 190 us, profiles/r02_timeline_final.txt.)
    else reduce_partials_kernel<16><<<(unsigned)blocks, 512, 0, st>>>(part, out, n, splits);
    return check_launch("reduce_partials");
}

size_t act_bwd_bias_workspace(long long rows, int C) {
    (void)rows;
    return (size_t)148 * 6 * C * sizeof(float) + 256;
}

int act_bwd_bias(const void* dy, const void* y, void* dpre, float* db, long long rows, int C, int act, void* ws, size_t ws_bytes,
                 cudaStream_t st, int group, long long ld_dy) {
    if (C % 8 || (((uintptr_t)dy | (uintptr_t)y | (uintptr_t)dpre) & 15)) return fail(DMV_E_UNSUPPORTED_SHAPE, "act_bwd_bias: need C % 8 == 0, 16-byte alignment");
    if (group > 0 && ld_dy % 8) return fail(DMV_E_UNSUPPORTED_SHAPE, "act_bwd_bias_grouped: dy rows must be 16-byte aligned (ld_dy % 8 == 0)");
    const int C8 = C / 8;
    int cgb = 64;
    while (cgb > 1 && (C8 % cgb)) cgb >>= 1;          // largest power of two <= 64 dividing C/8
    const int col_blocks = C8 / cgb;
    const int rstep = 256 / cgb;
    long long row_ctas = ceil_div_ll(148 * 6, col_blocks);
    const long long max_by_rows = ceil_div_ll(rows, (long long)rstep * 4);
    if (row_ctas > max_by_rows) row_ctas = max_by_rows;
    if (row_ctas < 1) row_ctas = 1;
    const long long per = ceil_div_ll(rows, row_ctas);
    row_ctas = ceil_div_ll(rows, per);
    if (!ws || ws_bytes < (size_t)row_ctas * C * sizeof(float)) return fail(DMV_E_WORKSPACE, "act_bwd_bias: workspace too small");
    float* part = reinterpret_cast<float*>(ws);
    dim3 grid(col_blocks, (unsigned)row_ctas);
    if (group > 0)
        act_bwd_bias_kernel<true><<<grid, 256, 0, st>>>((const uint4*)dy, (const uint4*)y, (uint4*)dpre, part, rows, C8, cgb, per, act, group,
                                                        ld_dy / 8);
    else
        act_bwd_bias_kernel<false><<<grid, 256, 0, st>>>((const uint4*)dy, (const uint4*)y, (uint4*)dpre, part, rows, C8, cgb, per, act, 1, C8);
    int rc = check_launch("act_bwd_bias");
    if (rc) return rc;
    return reduce_partials(part, db, C, (int)row_ctas, st);
}

int simt_bias_grad(const void* dy_bf16, float* db, long long pixels, int C, void* ws, size_t ws_bytes, cudaStream_t st) {
    return run_colsum<bf16>((const bf16*)dy_bf16, db, pixels, C, ws, ws_bytes, st);
}

size_t simt_wgrad_workspace(int taps, int Cin, int Cout, long long pixels) {
    const SplitPlan p = plan_split(taps, Cin, Cout, pixels);
    size_t a = (size_t)p.splits * taps * Cin * Cout * sizeof(float);
    size_t b = (size_t)256 * Cout * sizeof(float);
    return (a > b ? a : b) + 256;
}

int simt_conv_fwd(const void* x, int xdt, const void* w, const float* bias, void* y, int ydt, int B, int H, int W, int Cin,
                  int Cout, int kh, int kw, int stride, int act, cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, H, W, Cin, Cout, kh, kw, stride);
    if (rc) return rc;
    if (xdt == DMV_DT_F32 && ydt == DMV_DT_BF16) return run_f<float, bf16>(x, w, bias, y, g, act, st);
    if (xdt == DMV_DT_F32 && ydt == DMV_DT_F32) return run_f<float, float>(x, w, bias, y, g, act, st);
    if (xdt == DMV_DT_BF16 && ydt == DMV_DT_BF16) return run_f<bf16, bf16>(x, w, bias, y, g, act, st);
    if (xdt == DMV_DT_BF16 && ydt == DMV_DT_F32) return run_f<bf16, float>(x, w, bias, y, g, act, st);
    return fail(DMV_E_INVALID_ARG, "conv_fwd: unknown dtype");
}

// big side gradient of a conv whose big side is [B,H,W,Cin]: small = dy (bf16), writes dx (bf16)
int simt_conv_dgrad(const void* dy, const void* w, void* dx, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                    cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, H, W, Cin, Cout, kh, kw, stride);
    if (rc) return rc;
    return run_g<bf16, bf16>(dy, w, dx, g, DMV_ACT_NONE, st);
}

int simt_conv_wgrad(const void* x, int xdt, const void* dy, float* dw, float* db, int B, int H, int W, int Cin, int Cout, int kh,
                    int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, H, W, Cin, Cout, kh, kw, stride);
    if (rc) return rc;
    if (xdt == DMV_DT_F32) rc = run_wgrad<float, bf16>((const float*)x, (const bf16*)dy, dw, g, ws, ws_bytes, st);
    else rc = run_wgrad<bf16, bf16>((const bf16*)x, (const bf16*)dy, dw, g, ws, ws_bytes, st);
    if (rc) return rc;
    if (db) rc = run_colsum<bf16>((const bf16*)dy, db, (long long)g.B * g.Ho * g.Wo, Cout, ws, ws_bytes, st);
    return rc;
}

// deconv: big side is the OUTPUT [B,Hout,Wout,Cout_t]; geometry ci := Cout_t, co := Cin_t
int simt_deconv_fwd(const void* x, const void* w, void* y, int ydt, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                    int stride, int act, cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, Hout, Wout, /*ci=*/Cout, /*co=*/Cin, kh, kw, stride);
    if (rc) return rc;
    if (ydt == DMV_DT_F32) return run_g<bf16, float>(x, w, y, g, act, st);
    return run_g<bf16, bf16>(x, w, y, g, act, st);
}

int simt_deconv_dgrad(const void* dy, int dydt, const void* w, void* dx, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                      int kw, int stride, cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, Hout, Wout, Cout, Cin, kh, kw, stride);
    if (rc) return rc;
    if (dydt == DMV_DT_F32) return run_f<float, bf16>(dy, w, nullptr, dx, g, DMV_ACT_NONE, st);
    return run_f<bf16, bf16>(dy, w, nullptr, dx, g, DMV_ACT_NONE, st);
}

int simt_deconv_wgrad(const void* x, const void* dy, int dydt, float* dw, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                      int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    ConvGeom g;
    int rc = make_geom(g, B, Hout, Wout, Cout, Cin, kh, kw, stride);
    if (rc) return rc;
    if (dydt == DMV_DT_F32) return run_wgrad<float, bf16>((const float*)dy, (const bf16*)x, dw, g, ws, ws_bytes, st);
    return run_wgrad<bf16, bf16>((const bf16*)dy, (const bf16*)x, dw, g, ws, ws_bytes, st);
}

}  // namespace dmv

// tcgen05 / TMEM / TMA implicit-GEMM convolution kernels for sm_100a.
//
// One persistent, warp-specialised kernel covers the "F" and "G" forms of conv_simt.cu
// (conv fwd, conv dgrad, deconv fwd, deconv dgrad) as an implicit GEMM
//     D[pixel, n] = sum_{tap} sum_{c} A_tap[pixel, c] * B[n, (tap, c)]
// with M = a tile of <= 128 output pixels, N = output channels (padded to 16), K = taps x
// channels.  Nothing is im2col'ed in memory:
//   * A: for every (tap, channel chunk) ONE TMA box load of the input window shifted by the
//     tap offset.  The input is described to TMA as a 5-D tensor (C', W', P, H', N); for
//     stride-2 reads it is the parity view [N][H/2][2][W/2][2C] of the same NHWC buffer, so
//     a strided tap is again a plain shifted box.  Out-of-bounds elements are zero-filled
//     by TMA, which is exactly TF-SAME padding (asymmetric pads are just coordinates).
//   * B: weights, K-major: either a packed [n][tap*C + c] copy (F form) or -- for the G
//     form -- the reference HWIO layout itself read as a 3-D tensor (co, ci, tap).
//   * stride-2 G forms (conv dgrad, deconv fwd) are split into the four output-parity
//     classes; each class is a stride-1 problem with its own tap list, and all four are
//     tiles of the same launch.
// Both operands land in 128B/64B-swizzled shared memory, tcgen05.mma (M=128, kind::f16,
// bf16 x bf16 -> fp32) accumulates into double-buffered TMEM, and four epilogue warps read
// TMEM with tcgen05.ld, fuse bias + activation, and store NHWC rows.
// Warp roles: 0 = TMA producer, 1 = MMA issuer (+ TMEM allocator), 2..5 = epilogue.
#include <stdlib.h>

#include "tc_common.cuh"
#include "conv_impl.h"

namespace {
using namespace dmv;
using namespace dmv::tc;

// ----------------------------------------------------------------------------------------------
// kernel
// ----------------------------------------------------------------------------------------------
constexpr int kMaxTaps = 40;
constexpr int kThreads = 192;
// Activation-derivative factor in the input-gradient epilogues (IgemmParams::dact_y).  Compiled OUT by default: measured
// slower than the separate HBM-rate elementwise pass with the present four-epilogue-warp kernels
// (profiles/r02_dact_fusion.txt); the entry points then apply the factor with that pass, same results.  Build with
// -DDMV_DACT_EPILOGUE=1 to get the fused epilogues.
#ifndef DMV_DACT_EPILOGUE
#define DMV_DACT_EPILOGUE 0
#endif
constexpr bool kDactEpilogue = DMV_DACT_EPILOGUE != 0;

struct TapClass {
    int tap_begin, tap_count, k_elem_offset, py, px;
};
struct Tap {
    short dh, dw, ph, pw;   // row/col shift in the (possibly parity-) view, parity plane, channel-plane
    int id;                 // r*kw + s in the reference weight layout
};
struct IgemmParams {
    int num_classes, tiles_per_class, tiles_w, tiles_h, groups;
    int BW, BH, NB, rows;
    int Jh, Jw, Nimg;
    int kc_per_tap, c_plane;      // channel chunks per tap; channels of one parity plane (C of the source)
    int n_real, n_pad;            // total output channels; UMMA N of one N tile (multiple of 16)
    int n_tiles;                  // N tiles (n_pad columns each)
    int out_mul, out_H, out_W;
    int act, out_f32;
    int b_mode;                   // 0: packed K-major [n][K]; 1: reference HWIO read as (co, ci, tap), K-major;
                                  // 2: MN-major [K][n] (linear forward: Matrix[K,N] as stored)
    int stages;
    int k_splits;                 // linear layers: the contraction is cut into k_splits ranges (fp32 partials + finish kernel)
    long long split_stride;       // elements between the partial outputs of consecutive splits
    int halo_pitch, halo_h, min_dh, min_dw;   // halo kernel: window rows x pitch pixels, origin offset of the window
    int planes, plane_bytes;      // halo kernel over a stride-2 source: the two row-parity planes of the parity view are separate
                                  // windows (tap.ph selects one); the column parity is folded into the 2C channels of a row
    int d2s, d2s_c;               // sub-pixel form: column (class, c) of a tile row goes to output pixel (2*jh + py, 2*jw + px), channel c
    TapClass cls[4];
    Tap taps[kMaxTaps];
    const float* bias;
    void* out;
    // input-gradient launches: the bf16 result is multiplied by act'(dact_y[same index]) before it is rounded, i.e. the
    // kernel writes dPre of the layer that produced this launch's input (dX * act'(Y)) instead of dX (NULL: off)
    const bf16* dact_y;
    int dact;
};

// act'(y) of 16 (or 8) consecutive bf16 outputs applied to the fp32 accumulators
__device__ __forceinline__ void apply_dact8(float* f, const bf16* __restrict__ y, int act) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(y));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 v = __bfloat1622float2(h[k]);
        f[2 * k] *= act_grad_from_output(v.x, act);
        f[2 * k + 1] *= act_grad_from_output(v.y, act);
    }
}

// Epilogue of one accumulator tile for one thread (= one output pixel): TMEM -> registers in 16-column
// chunks, + bias (shared memory copy when the layer has a single N tile), activation (uniform switch hoisted
// out of the element loop), NHWC store (bf16 or fp32).
// act'(y) from an already loaded 16-byte group
__device__ __forceinline__ void apply_dact8_reg(float* f, const uint4& q, int act) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 v = __bfloat1622float2(h[k]);
        f[2 * k] *= act_grad_from_output(v.x, act);
        f[2 * k + 1] *= act_grad_from_output(v.y, act);
    }
}

// The epilogue warps know where a tile goes before its MMAs have finished: the first kPreCols columns of the dact factor
// are fetched BEFORE the wait on the accumulator barrier, so their latency hides behind the tensor work.
constexpr int kPreCols = 64;
struct YPre {
    uint4 v[kPreCols / 8];
};
__device__ __forceinline__ void prefetch_dact_row(const IgemmParams& p, bool ok, long long opix, int ncol0, YPre& y) {
    if (!kDactEpilogue || !p.dact_y || p.out_f32 || !ok || (p.n_real & 7)) return;
    const bf16* yq = p.dact_y + opix * p.n_real + ncol0;
#pragma unroll
    for (int j = 0; j < kPreCols / 8; ++j)
        if (ncol0 + j * 8 + 8 <= p.n_real && j * 8 < p.n_pad) y.v[j] = __ldg(reinterpret_cast<const uint4*>(yq + j * 8));
}

template <bool PRE>
__device__ __forceinline__ void epilogue_chunk(const IgemmParams& p, uint32_t taddr, bool ok, long long opix, int ncol0, int ks,
                                               const float* __restrict__ s_bias, int c0, const uint4& y0, const uint4& y1) {
    {
        uint32_t v[16];
        tmem_ld16(taddr + (uint32_t)c0, v);
        tmem_ld_wait();
        if (!ok) return;
        float f[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) f[k] = __uint_as_float(v[k]);
        if (p.bias) {
            if (s_bias) {
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] += s_bias[c0 + k];
            } else {
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (ncol0 + c0 + k < p.n_real) f[k] += __ldg(p.bias + ncol0 + c0 + k);
            }
        }
        switch (p.act) {
            case DMV_ACT_LRELU:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = 0.6f * f[k] + 0.4f * fabsf(f[k]);
                break;
            case DMV_ACT_RELU:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = 0.5f * f[k] + 0.5f * fabsf(f[k]);
                break;
            case DMV_ACT_TANH:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = tanhf(f[k]);
                break;
            default: break;
        }
        if (p.out_f32) {
            float* o = reinterpret_cast<float*>(p.out) + (long long)ks * p.split_stride + opix * p.n_real + ncol0 + c0;
            if (ncol0 + c0 + 16 <= p.n_real && (p.n_real & 3) == 0) {
#pragma unroll
                for (int k = 0; k < 16; k += 4) *reinterpret_cast<float4*>(o + k) = make_float4(f[k], f[k + 1], f[k + 2], f[k + 3]);
            } else {
                for (int k = 0; k < 16 && ncol0 + c0 + k < p.n_real; ++k) o[k] = f[k];
            }
        } else {
            bf16* o = reinterpret_cast<bf16*>(p.out) + opix * p.n_real + ncol0 + c0;
            if (kDactEpilogue && p.dact_y) {
                const bf16* yq = p.dact_y + opix * p.n_real + ncol0 + c0;
                if (ncol0 + c0 + 16 <= p.n_real && (p.n_real & 7) == 0) {
                    if (PRE) {
                        apply_dact8_reg(f, y0, p.dact);
                        apply_dact8_reg(f + 8, y1, p.dact);
                    } else {
                        apply_dact8(f, yq, p.dact);
                        apply_dact8(f + 8, yq + 8, p.dact);
                    }
                } else {
                    for (int k = 0; k < 16 && ncol0 + c0 + k < p.n_real; ++k) f[k] *= act_grad_from_output(__bfloat162float(yq[k]), p.dact);
                }
            }
            if (ncol0 + c0 + 16 <= p.n_real && (p.n_real & 7) == 0) {
                uint4 q0, q1;
                __nv_bfloat162 h;
                h = __floats2bfloat162_rn(f[0], f[1]); q0.x = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[2], f[3]); q0.y = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[4], f[5]); q0.z = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[6], f[7]); q0.w = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[8], f[9]); q1.x = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[10], f[11]); q1.y = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[12], f[13]); q1.z = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[14], f[15]); q1.w = *reinterpret_cast<uint32_t*>(&h);
                reinterpret_cast<uint4*>(o)[0] = q0;
                reinterpret_cast<uint4*>(o)[1] = q1;
            } else {
                for (int k = 0; k < 16 && ncol0 + c0 + k < p.n_real; ++k) o[k] = __float2bfloat16_rn(f[k]);
            }
        }
    }
}

__device__ __forceinline__ void epilogue_row(const IgemmParams& p, uint32_t taddr, bool ok, long long opix, int ncol0, int ks,
                                             const float* __restrict__ s_bias, const YPre& ypre) {
    // the first kPreCols columns use the factors fetched before the accumulator wait (static register indices)
#pragma unroll
    for (int j = 0; j < kPreCols / 16; ++j)
        if (j * 16 < p.n_pad) epilogue_chunk<true>(p, taddr, ok, opix, ncol0, ks, s_bias, j * 16, ypre.v[2 * j], ypre.v[2 * j + 1]);
    for (int c0 = kPreCols; c0 < p.n_pad; c0 += 16) epilogue_chunk<false>(p, taddr, ok, opix, ncol0, ks, s_bias, c0, ypre.v[0], ypre.v[0]);
}

// Sub-pixel epilogue (stride-2 G forms run as ONE stride-1 problem, see launch_subpixel): the accumulator row of
// class-grid pixel (jh, jw) holds 4 x C columns (class-major); class (py, px) goes to output pixel (2jh + py, 2jw + px).
__device__ __forceinline__ void epilogue_row_d2s(const IgemmParams& p, uint32_t taddr, bool row_ok, int n, int jh, int jw) {
    const int C = p.d2s_c;
    for (int c0 = 0; c0 < p.n_pad; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(taddr + (uint32_t)c0, v);
        tmem_ld_wait();
        if (!row_ok || c0 >= 4 * C) continue;
        float f[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) f[k] = __uint_as_float(v[k]);
        switch (p.act) {
            case DMV_ACT_LRELU:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = 0.6f * f[k] + 0.4f * fabsf(f[k]);
                break;
            case DMV_ACT_RELU:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = 0.5f * f[k] + 0.5f * fabsf(f[k]);
                break;
            case DMV_ACT_TANH:
#pragma unroll
                for (int k = 0; k < 16; ++k) f[k] = tanhf(f[k]);
                break;
            default: break;
        }
        if ((C & 15) == 0) {          // the 16 columns belong to one class
            const int cls = c0 / C, cc = c0 - cls * C;
            const int oy = 2 * jh + (cls >> 1), ox = 2 * jw + (cls & 1);
            if (oy >= p.out_H || ox >= p.out_W) continue;
            const long long o = (((long long)n * p.out_H + oy) * p.out_W + ox) * C + cc;
            if (p.out_f32) {
                float* q = reinterpret_cast<float*>(p.out) + o;
#pragma unroll
                for (int k = 0; k < 16; k += 4) *reinterpret_cast<float4*>(q + k) = make_float4(f[k], f[k + 1], f[k + 2], f[k + 3]);
            } else {
                if (kDactEpilogue && p.dact_y) {
                    apply_dact8(f, p.dact_y + o, p.dact);
                    apply_dact8(f + 8, p.dact_y + o + 8, p.dact);
                }
                uint4 q0, q1;
                __nv_bfloat162 h;
                h = __floats2bfloat162_rn(f[0], f[1]); q0.x = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[2], f[3]); q0.y = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[4], f[5]); q0.z = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[6], f[7]); q0.w = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[8], f[9]); q1.x = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[10], f[11]); q1.y = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[12], f[13]); q1.z = *reinterpret_cast<uint32_t*>(&h);
                h = __floats2bfloat162_rn(f[14], f[15]); q1.w = *reinterpret_cast<uint32_t*>(&h);
                uint4* q = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.out) + o);
                q[0] = q0;
                q[1] = q1;
            }
        } else {                      // thin heads (C = 2 flow channels): element-wise
            for (int k = 0; k < 16 && c0 + k < 4 * C; ++k) {
                const int cls = (c0 + k) / C, cc = (c0 + k) - cls * C;
                const int oy = 2 * jh + (cls >> 1), ox = 2 * jw + (cls & 1);
                if (oy >= p.out_H || ox >= p.out_W) continue;
                const long long o = (((long long)n * p.out_H + oy) * p.out_W + ox) * C + cc;
                if (p.out_f32) reinterpret_cast<float*>(p.out)[o] = f[k];
                else reinterpret_cast<bf16*>(p.out)[o] =
                    __float2bfloat16_rn((kDactEpilogue && p.dact_y) ? f[k] * act_grad_from_output(__bfloat162float(p.dact_y[o]), p.dact) : f[k]);
            }
        }
    }
}

// Sub-pixel epilogue for C = 32 (bf16 out): the two column-parity classes of one output row are 128 contiguous bytes
// per tile pixel, and the 8 pixels of a tile row are 1 KB contiguous.  Stored lane by lane that is 32 scattered 16-byte
// pieces per instruction (the kernel was bound by L1 -> L2 write requests); instead each warp stages its 32 x 128 B in an
// XOR-swizzled shared tile and writes it back with four full 128-byte lines per instruction.
__device__ __forceinline__ void epilogue_d2s_c32(const IgemmParams& p, uint32_t taddr, int n, int th, int tw, int quarter, int lane,
                                                 uint4* __restrict__ s_epi, const uint4* __restrict__ ypre) {
    bf16* outp = reinterpret_cast<bf16*>(p.out);
#pragma unroll
    for (int py = 0; py < 2; ++py) {
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
            uint32_t v[16];
            tmem_ld16(taddr + (uint32_t)(py * 64 + q4 * 16), v);
            tmem_ld_wait();
            float f[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) f[k] = __uint_as_float(v[k]);
            switch (p.act) {
                case DMV_ACT_LRELU:
#pragma unroll
                    for (int k = 0; k < 16; ++k) f[k] = 0.6f * f[k] + 0.4f * fabsf(f[k]);
                    break;
                case DMV_ACT_RELU:
#pragma unroll
                    for (int k = 0; k < 16; ++k) f[k] = 0.5f * f[k] + 0.5f * fabsf(f[k]);
                    break;
                case DMV_ACT_TANH:
#pragma unroll
                    for (int k = 0; k < 16; ++k) f[k] = tanhf(f[k]);
                    break;
                default: break;
            }
            if (kDactEpilogue && p.dact_y) {
                // this thread's row is class-grid pixel (jh, jw); columns py*64 + q4*16 .. +15 are channels (q4 & 1) * 16 ..
                // of output pixel (2 jh + py, 2 jw + (q4 >> 1))
                const int m = quarter * 32 + lane;
                const int jh = th * 16 + (m >> 3), jw = tw * 8 + (m & 7);
                const int oy = 2 * jh + py, ox = 2 * jw + (q4 >> 1);
                if (jh < p.Jh && jw < p.Jw && oy < p.out_H && ox < p.out_W) {     // fetched before the accumulator wait
                    apply_dact8_reg(f, ypre[(py * 2 + (q4 >> 1)) * 4 + (q4 & 1) * 2], p.dact);
                    apply_dact8_reg(f + 8, ypre[(py * 2 + (q4 >> 1)) * 4 + (q4 & 1) * 2 + 1], p.dact);
                }
            }
            __nv_bfloat162 h;
            uint4 a, b;
            h = __floats2bfloat162_rn(f[0], f[1]); a.x = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[2], f[3]); a.y = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[4], f[5]); a.z = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[6], f[7]); a.w = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[8], f[9]); b.x = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[10], f[11]); b.y = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[12], f[13]); b.z = *reinterpret_cast<uint32_t*>(&h);
            h = __floats2bfloat162_rn(f[14], f[15]); b.w = *reinterpret_cast<uint32_t*>(&h);
            s_epi[lane * 8 + ((2 * q4) ^ (lane & 7))] = a;
            s_epi[lane * 8 + ((2 * q4 + 1) ^ (lane & 7))] = b;
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int rr = t * 4 + (lane >> 3), cc = lane & 7;
            const int m = quarter * 32 + rr;
            const int jh = th * 16 + (m >> 3), jw = tw * 8 + (m & 7);
            const int oy = 2 * jh + py, ox = 2 * jw + (cc >> 2);
            if (jh < p.Jh && jw < p.Jw && oy < p.out_H && ox < p.out_W) {
                const uint4 q = s_epi[rr * 8 + (cc ^ (rr & 7))];
                *reinterpret_cast<uint4*>(outp + (((long long)n * p.out_H + oy) * p.out_W + 2 * jw) * 32 + cc * 8) = q;
            }
        }
        __syncwarp();
    }
}

template <int KC>
__global__ void __launch_bounds__(kThreads, 1) igemm_kernel(const __grid_constant__ CUtensorMap map_a,
                                                             const __grid_constant__ CUtensorMap map_b,
                                                             const __grid_constant__ IgemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    constexpr int kRowBytes = KC * 2;
    constexpr int kABytes = 128 * kRowBytes;
    const int b_bytes = p.n_pad * kRowBytes;     // mode 2: (n_pad/64) boxes of KC rows x 128 B -- the same size
    const int stage_bytes = kABytes + b_bytes;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* tfull_bar = empty_bar + p.stages;   // [2]
    uint64_t* tempty_bar = tfull_bar + 2;         // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* s_bias = reinterpret_cast<float*>(tmem_slot + 4);     // [n_pad], zero padded (single N tile only)
    if (p.n_tiles == 1)
        for (int i = threadIdx.x; i < p.n_pad; i += kThreads) s_bias[i] = (p.bias && i < p.n_real) ? __ldg(p.bias + i) : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(2 * p.n_pad)) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int total_tiles = p.num_classes * p.tiles_per_class * p.n_tiles * p.k_splits;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t tx = (uint32_t)(p.rows * kRowBytes + b_bytes);
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % p.n_tiles;
                const int ks = (tile / p.n_tiles) % p.k_splits;
                const int sp = tile / (p.n_tiles * p.k_splits);
                const int ci = sp / p.tiles_per_class;
                int t = sp - ci * p.tiles_per_class;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                const int g = t;
                const TapClass& c = p.cls[ci];
                const int per_split = (p.kc_per_tap + p.k_splits - 1) / p.k_splits;      // k_splits > 1 only with one tap
                const int ch0 = p.k_splits > 1 ? ks * per_split : 0;
                const int ch1 = p.k_splits > 1 ? min(p.kc_per_tap, ch0 + per_split) : p.kc_per_tap;
                for (int j = 0; j < c.tap_count; ++j) {
                    const Tap& tp = p.taps[c.tap_begin + j];
                    for (int ch = ch0; ch < ch1; ++ch) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        uint8_t* sa = smem + (size_t)stage * stage_bytes;
                        mbar_expect_tx(&full_bar[stage], tx);
                        tma_load_5d(sa, &map_a, &full_bar[stage], tp.pw * p.c_plane + ch * KC, tw * p.BW + tp.dw, tp.ph,
                                    th * p.BH + tp.dh, g * p.NB);
                        if (p.b_mode == 1) {
                            tma_load_3d(sa + kABytes, &map_b, &full_bar[stage], ch * KC, nt * p.n_pad, tp.id);
                        } else if (p.b_mode == 0) {
                            tma_load_3d(sa + kABytes, &map_b, &full_bar[stage], c.k_elem_offset + (j * p.kc_per_tap + ch) * KC,
                                        nt * p.n_pad, 0);
                        } else {
                            for (int jb = 0; jb < p.n_pad / 64; ++jb)
                                tma_load_3d(sa + kABytes + jb * (KC * 128), &map_b, &full_bar[stage], nt * p.n_pad + jb * 64,
                                            (j * p.kc_per_tap + ch) * KC, 0);
                        }
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            // instruction descriptor: D=f32, A=B=bf16, both K-major, N = n_pad, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (p.b_mode == 2 ? (1u << 16) : 0u) |
                                   ((uint32_t)(p.n_pad >> 3) << 17) | ((128u >> 4) << 24);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const TapClass& c = p.cls[(tile / (p.n_tiles * p.k_splits)) / p.tiles_per_class];
                int kblocks = c.tap_count * p.kc_per_tap;
                if (p.k_splits > 1) {
                    const int ks = (tile / p.n_tiles) % p.k_splits;
                    const int per_split = (p.kc_per_tap + p.k_splits - 1) / p.k_splits;
                    kblocks = min(p.kc_per_tap, (ks + 1) * per_split) - ks * per_split;
                }
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_pad);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint64_t adesc = make_kmajor_desc(sa, kRowBytes);
                    // K-major B: +32 bytes per K=16 step inside the swizzle span; MN-major B: +16 rows of 128 B
                    const uint64_t bdesc = p.b_mode == 2 ? make_mnmajor_desc(sa + kABytes, 128, KC * 128) : make_kmajor_desc(sa + kABytes, kRowBytes);
                    const uint64_t bstep = p.b_mode == 2 ? 128u : 2u;
#pragma unroll
                    for (int k = 0; k < KC / 16; ++k)
                        tc_mma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + bstep * (uint64_t)k, idesc, (kb | k) ? 1u : 0u);
                    tc_commit(&empty_bar[stage]);        // frees the smem slot when these MMAs retire
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                tc_commit(&tfull_bar[acc]);              // accumulator ready for the epilogue
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..5)
        const int quarter = warp & 3;                    // TMEM lanes 32*quarter .. +31
        const int m = quarter * 32 + lane;               // row of the tile = output pixel
        int acc = 0;
        uint32_t acc_phase = 0;
        const int per_img = p.BH * p.BW;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int nt = tile % p.n_tiles;
            const int ks = (tile / p.n_tiles) % p.k_splits;
            const int sp = tile / (p.n_tiles * p.k_splits);
            const int ci = sp / p.tiles_per_class;
            int t = sp - ci * p.tiles_per_class;
            const int tw = t % p.tiles_w; t /= p.tiles_w;
            const int th = t % p.tiles_h; t /= p.tiles_h;
            const int g = t;
            const TapClass& c = p.cls[ci];
            const int ncol0 = nt * p.n_pad;
            const int nb = m / per_img, rem = m - nb * per_img;
            const int bh = rem / p.BW, bw = rem - bh * p.BW;
            const int n = g * p.NB + nb, jh = th * p.BH + bh, jw = tw * p.BW + bw;
            const int oy = p.out_mul * jh + c.py, ox = p.out_mul * jw + c.px;
            const bool ok = (m < p.rows) && (n < p.Nimg) && (jh < p.Jh) && (jw < p.Jw) && (oy < p.out_H) && (ox < p.out_W);
            const long long opix = ((long long)n * p.out_H + oy) * p.out_W + ox;
            YPre ypre;
            prefetch_dact_row(p, ok, opix, ncol0, ypre);
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.n_pad);
            epilogue_row(p, taddr, ok, opix, ncol0, ks, p.n_tiles == 1 ? s_bias : nullptr, ypre);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// ----------------------------------------------------------------------------------------------
// Halo variant for stride-1 layers whose weights fit in shared memory next to the input windows
// (the four largest layers of the graph and their dgrads).  Instead of one TMA box per tap, the CTA
// loads the (16 + kh - 1) x (8 + kw - 1) input window of an 8 x 16 output tile ONCE; the A operand of
// tap (r, s) is the same shared-memory tile addressed through a descriptor that starts (r * pitch + s)
// pixel rows further and strides one window row per 8-row core group.  This works because the
// shared-memory swizzle is a pure function of the address (established with tools/probe), and it cuts
// the L2 -> SM traffic of a 5x5 layer by ~13x.  All kh*kw weight tiles are loaded once per CTA.
template <int KC, int NT, int EPI>      // EPI 1: coalescing sub-pixel epilogue (its own instantiation: it needs more registers)
__global__ void __launch_bounds__(kThreads, EPI ? 1 : 2) halo_kernel(const __grid_constant__ CUtensorMap map_a,
                                                            const __grid_constant__ CUtensorMap map_b,
                                                            const __grid_constant__ IgemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    constexpr int kRowBytes = KC * 2;
    const TapClass& c = p.cls[0];
    const int ntaps = c.tap_count;
    const int wtile_bytes = p.n_pad * kRowBytes;
    const int a_bytes = p.halo_h * p.halo_pitch * kRowBytes;
    const int a_stage = p.planes * p.plane_bytes;          // plane_bytes = a_bytes rounded up to 1024
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* s_w = smem;
    uint8_t* s_a = smem + (size_t)ntaps * wtile_bytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_a + (size_t)p.stages * a_stage);
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* tfull_bar = empty_bar + p.stages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* w_bar = tempty_bar + 2;
    uint64_t* s_bdesc = w_bar + 1;                 // [ntaps] weight-tile descriptors
    uint32_t* s_aoff = reinterpret_cast<uint32_t*>(s_bdesc + kMaxTaps);   // [ntaps] tap offsets (16-byte units)
    uint32_t* tmem_slot = s_aoff + kMaxTaps;
    float* s_bias = reinterpret_cast<float*>(tmem_slot + 4);
    // [4 epilogue warps][32 x 128 B] transpose tiles of the sub-pixel C = 32 epilogue (allocated only then)
    uint4* s_epi_all = reinterpret_cast<uint4*>((reinterpret_cast<uintptr_t>(s_bias + 256) + 127) & ~(uintptr_t)127);
    for (int i = threadIdx.x; i < p.n_pad; i += kThreads) s_bias[i] = (p.bias && i < p.n_real) ? __ldg(p.bias + i) : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(2 * p.n_pad)) tmem_cols <<= 1;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], 4);
        }
        mbar_init(w_bar, 1);
        fence_barrier_init();
    }
    if (threadIdx.x < ntaps) {      // MMA operand descriptors, computed once
        const Tap& tp = p.taps[c.tap_begin + threadIdx.x];
        s_aoff[threadIdx.x] = (uint32_t)(((tp.dh - p.min_dh) * p.halo_pitch + (tp.dw - p.min_dw)) * kRowBytes + tp.ph * p.plane_bytes) >> 4;
        s_bdesc[threadIdx.x] = make_kmajor_desc(smem_u32(s_w) + (uint32_t)(threadIdx.x * wtile_bytes), kRowBytes);
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int total_tiles = p.tiles_per_class;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(w_bar, (uint32_t)(ntaps * wtile_bytes));
            for (int j = 0; j < ntaps; ++j) {
                if (p.b_mode == 1) tma_load_3d(s_w + (size_t)j * wtile_bytes, &map_b, w_bar, 0, 0, p.taps[c.tap_begin + j].id);
                else tma_load_3d(s_w + (size_t)j * wtile_bytes, &map_b, w_bar, c.k_elem_offset + j * KC, 0, 0);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_expect_tx(&full_bar[stage], (uint32_t)(a_bytes * p.planes));
                for (int pl = 0; pl < p.planes; ++pl)
                    tma_load_5d(s_a + (size_t)stage * a_stage + (size_t)pl * p.plane_bytes, &map_a, &full_bar[stage], 0, tw * 8 + p.min_dw, pl,
                                th * 16 + p.min_dh, t);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_pad >> 3) << 17) | ((128u >> 4) << 24);
            // descriptor template for A: SBO = one window row (pitch pixels)
            uint64_t a_tmpl = 0;
            a_tmpl |= (uint64_t)1 << 16;
            a_tmpl |= (uint64_t)((uint32_t)(p.halo_pitch * kRowBytes) >> 4) << 32;
            a_tmpl |= (uint64_t)1 << 46;
            a_tmpl |= (uint64_t)(kRowBytes == 128 ? 2 : 4) << 61;
            mbar_wait(w_bar, 0);
            tc_fence_after();
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            // the issue loop is single-threaded: with a compile-time tap count the descriptors live in registers
            // and every MMA costs one 64-bit add
            uint64_t r_b[NT ? NT : 1];
            uint32_t r_a[NT ? NT : 1];
            if (NT) {
#pragma unroll
                for (int j = 0; j < NT; ++j) { r_b[j] = s_bdesc[j]; r_a[j] = s_aoff[j]; }
            }
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_pad);
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint64_t a_base = a_tmpl | (uint64_t)((smem_u32(s_a + (size_t)stage * a_stage) & 0x3FFFF) >> 4);
                if (NT) {
#pragma unroll
                    for (int j = 0; j < NT; ++j) {
                        const uint64_t adesc = a_base + (uint64_t)r_a[j];
#pragma unroll
                        for (int k = 0; k < KC / 16; ++k)
                            tc_mma_bf16(d_tmem, adesc + (uint64_t)(2 * k), r_b[j] + (uint64_t)(2 * k), idesc, (j | k) ? 1u : 0u);
                    }
                } else {
                    for (int j = 0; j < ntaps; ++j) {
                        const uint64_t adesc = a_base + (uint64_t)s_aoff[j];
                        const uint64_t bdesc = s_bdesc[j];
#pragma unroll
                        for (int k = 0; k < KC / 16; ++k)
                            tc_mma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (j | k) ? 1u : 0u);
                    }
                }
                tc_commit(&empty_bar[stage]);
                tc_commit(&tfull_bar[acc]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        const int bh = m >> 3, bw = m & 7;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int t = tile;
            const int tw = t % p.tiles_w; t /= p.tiles_w;
            const int th = t % p.tiles_h; t /= p.tiles_h;
            const int n = t, oy = th * 16 + bh, ox = tw * 8 + bw;
            const bool ok = (oy < p.out_H) && (ox < p.out_W);
            const long long opix = ((long long)n * p.out_H + oy) * p.out_W + ox;
            YPre ypre;
            uint4 ypre_d2s[EPI == 1 ? 16 : 1];
            if (EPI == 1) {
                if (kDactEpilogue && p.dact_y) {    // class-grid pixel (oy, ox) -> output pixels (2 oy + py, 2 ox + px), 64 bytes each
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int yy = 2 * oy + (q >> 1), xx = 2 * ox + (q & 1);
                        if (oy < p.Jh && ox < p.Jw && yy < p.out_H && xx < p.out_W) {
                            const uint4* yq = reinterpret_cast<const uint4*>(p.dact_y + (((long long)n * p.out_H + yy) * p.out_W + xx) * 32);
#pragma unroll
                            for (int j = 0; j < 4; ++j) ypre_d2s[q * 4 + j] = __ldg(yq + j);
                        }
                    }
                }
            } else if (!p.d2s) {
                prefetch_dact_row(p, ok, opix, 0, ypre);
            }
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * p.n_pad);
            if (EPI == 1) epilogue_d2s_c32(p, taddr, n, th, tw, quarter, lane, s_epi_all + (warp - 2) * 256, ypre_d2s);
            else if (p.d2s) epilogue_row_d2s(p, taddr, (oy < p.Jh) && (ox < p.Jw), n, oy, ox);
            else epilogue_row(p, taddr, ok, opix, 0, 0, s_bias, ypre);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// split-K finish: y[m][n] = act( sum_ks part[ks][m][n] + bias[n] ) in bf16, splits added in order
__global__ void splitk_finish_kernel(const float* __restrict__ part, const float* __restrict__ bias, bf16* __restrict__ y, long long mn, int N,
                                     int splits, int act, const bf16* __restrict__ dact_y, int dact) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < mn; i += stride) {
        float s = 0.f;
        for (int z = 0; z < splits; ++z) s += part[(long long)z * mn + i];
        if (bias) s += __ldg(bias + (int)(i % N));
        s = apply_act(s, act);
        if (kDactEpilogue && dact_y) s *= act_grad_from_output(__bfloat162float(dact_y[i]), dact);
        y[i] = __float2bfloat16_rn(s);
    }
}

// F-form weight packing: w[t][ci][co] (bf16) -> packed[co][t*Cin + ci]
__global__ void pack_f_kernel(const bf16* __restrict__ w, bf16* __restrict__ out, int taps, int Cin, int Cout) {
    const long long n = (long long)taps * Cin * Cout;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int co = (int)(i % Cout);
        const long long r = i / Cout;      // t*Cin + ci
        out[(long long)co * taps * Cin + r] = w[i];
    }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
// Pick the output-tile box (BW x BH x NB <= 128 rows) that wastes the fewest MMA rows.
void choose_tile(int Jh, int Jw, int N, int& BW, int& BH, int& NB) {
    if (Jh * Jw <= 64) {
        BW = Jw; BH = Jh;
        NB = 128 / (Jh * Jw);
        if (NB > N) NB = N;
        if (NB > 256) NB = 256;
        return;
    }
    NB = 1;
    double best = -1.0;
    BW = 1; BH = 1;
    for (int bw = 1; bw <= Jw && bw <= 128; ++bw) {
        int bh = 128 / bw;
        if (bh > Jh) bh = Jh;
        if (bh < 1) continue;
        const long long tiles = (long long)ceil_div(Jw, bw) * ceil_div(Jh, bh);
        const double eff = (double)Jh * Jw / ((double)tiles * 128.0);
        // prefer wider boxes on ties (longer contiguous TMA rows)
        if (eff > best + 1e-9 || (eff > best - 1e-9 && bw > BW)) { best = eff; BW = bw; BH = bh; }
    }
}

struct Problem {
    // source (A) tensor: NHWC bf16 [N][Hs][Ws][Cs], read through a parity view when src_stride == 2
    const void* src; int N, Hs, Ws, Cs, src_stride;
    // weights
    const void* w_hwio; int kh, kw, w_ci, w_co;   // reference layout [kh][kw][w_ci][w_co]
    bool g_form;                                   // contraction over w_co (G) or w_ci (F)
    int k_splits;                                  // > 1: split the contraction (linear layers); needs workspace for partials
    int n_tile;                                    // 0: one N tile covering all output channels
    int b_mode_override;                           // -1: by form; 2: MN-major Matrix[K,N] (linear forward)
    // output
    void* out; int out_f32, out_H, out_W, n_real, out_mul;
    int Jh, Jw;                                    // per-class tiled index space
    const float* bias; int act;
};

// The activation-derivative factor of the NEXT input-gradient launch of this thread (tc_set_dact): taken by launch_igemm
// when it finalises the parameters of a bf16-output launch.
thread_local int tl_pack_mode = 0;     // tc_set_pack_mode: 0, DMV_ALGO_PACK_ONLY or DMV_ALGO_PREPACKED
thread_local const void* tl_dact_y = nullptr;
thread_local int tl_dact = 0;
thread_local bool tl_dact_taken = false;

int launch_igemm(const Problem& q, IgemmParams& p, void* workspace, size_t ws_bytes, cudaStream_t st) {
    const int Cc = q.Cs;                            // contraction channels per tap
    if (p.planes != 2) p.planes = 1;
    const int KC = (p.planes == 2) ? 2 * Cc : ((Cc % 64 == 0) ? 64 : 32);      // planes == 2: a window row holds (pw, c) = 2C channels
    if (p.planes == 2 && (Cc != 32 || q.src_stride != 2)) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: stride-2 halo needs 32 source channels");
    if (Cc % 32 != 0) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: contraction channels must be a multiple of 32");
    if (q.n_tile == 0 && q.n_real > 256) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: more than 256 output channels");
    if (((uintptr_t)q.src & 15) || ((uintptr_t)q.w_hwio & 15) || ((uintptr_t)q.out & 15))
        return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: buffers must be 16-byte aligned");
    p.n_real = q.n_real;
    p.n_pad = q.n_tile ? q.n_tile : ceil_div(q.n_real, 16) * 16;
    p.n_tiles = ceil_div(q.n_real, p.n_pad);
    p.k_splits = 1;
    p.split_stride = 0;
    p.kc_per_tap = (p.planes == 2) ? 1 : Cc / KC;
    p.c_plane = Cc;
    p.Jh = q.Jh; p.Jw = q.Jw; p.Nimg = q.N;
    choose_tile(q.Jh, q.Jw, q.N, p.BW, p.BH, p.NB);
    p.rows = p.BW * p.BH * p.NB;
    p.tiles_w = ceil_div(q.Jw, p.BW);
    p.tiles_h = ceil_div(q.Jh, p.BH);
    p.groups = ceil_div(q.N, p.NB);
    p.tiles_per_class = p.tiles_w * p.tiles_h * p.groups;
    p.out_mul = q.out_mul; p.out_H = q.out_H; p.out_W = q.out_W;
    p.act = q.act; p.out_f32 = q.out_f32; p.bias = q.bias; p.out = q.out;
    p.dact_y = nullptr; p.dact = 0;
    if (kDactEpilogue && tl_dact_y && !q.out_f32) {
        p.dact_y = reinterpret_cast<const bf16*>(tl_dact_y);
        p.dact = tl_dact;
        tl_dact_y = nullptr;
        tl_dact_taken = true;
    }
    const bool prepacked = q.b_mode_override == 3;      // w_hwio already holds the packed [n][K] K-major matrix
    p.b_mode = prepacked ? 0 : (q.b_mode_override >= 0 ? q.b_mode_override : (q.g_form ? 1 : 0));

    const int row_bytes = KC * 2;
    // ---- halo eligibility: stride-1 source, one channel chunk, one tap class, one N tile, weights resident
    bool halo_ok = false;
    int halo_stages = 0, halo_ctas_per_sm = 1;
    size_t halo_smem = 0;
    if ((q.src_stride == 1 || p.planes == 2) && p.num_classes == 1 && p.kc_per_tap == 1 && p.n_tiles == 1 && p.b_mode != 2 && q.out_mul == 1 &&
        q.Jh * q.Jw >= 256 && !getenv("DMV_NO_HALO")) {
        int dh0 = 1 << 20, dh1 = -(1 << 20), dw0 = 1 << 20, dw1 = -(1 << 20);
        for (int j = 0; j < p.cls[0].tap_count; ++j) {
            const Tap& t = p.taps[p.cls[0].tap_begin + j];
            dh0 = t.dh < dh0 ? t.dh : dh0; dh1 = t.dh > dh1 ? t.dh : dh1;
            dw0 = t.dw < dw0 ? t.dw : dw0; dw1 = t.dw > dw1 ? t.dw : dw1;
        }
        p.min_dh = dh0; p.min_dw = dw0;
        p.halo_h = 16 + (dh1 - dh0);
        p.halo_pitch = 8 + (dw1 - dw0);
        const size_t wbytes = (size_t)p.cls[0].tap_count * p.n_pad * row_bytes;
        p.plane_bytes = (int)(((size_t)p.halo_h * p.halo_pitch * row_bytes + 1023) & ~(size_t)1023);
        const size_t a_stage = (size_t)p.planes * p.plane_bytes;
        if (p.halo_pitch <= 256 && p.halo_h <= 256 && wbytes + 2 * a_stage <= 220 * 1024) {
            // two CTAs per SM (the epilogue of one overlaps the MMAs of the other) when the weights leave room
            if (p.n_pad <= 128 && wbytes + 3 * a_stage <= 104 * 1024) {
                halo_ctas_per_sm = 2;
                halo_stages = (int)((104 * 1024 - wbytes) / a_stage);
            } else {
                halo_stages = (int)((220 * 1024 - wbytes) / a_stage);
            }
            if (halo_stages > 6) halo_stages = 6;
            // sub-pixel layers with 32 bf16 output channels: coalescing epilogue through 16 KB of transpose tiles
            size_t epi = 0;
            if (p.d2s && p.d2s_c == 32 && !q.out_f32 && !getenv("DMV_NO_D2S_EPI")) {
                while (halo_stages > 2 && wbytes + (size_t)halo_stages * a_stage + 16 * 1024 + 4096 > (halo_ctas_per_sm == 2 ? 112 : 226) * 1024) --halo_stages;
                if (wbytes + (size_t)halo_stages * a_stage + 16 * 1024 + 4096 <= (halo_ctas_per_sm == 2 ? 112 : 226) * 1024) {
                    p.d2s = 2;
                    epi = 16 * 1024 + 128;
                }
            }
            halo_smem = wbytes + (size_t)halo_stages * a_stage + (2 * halo_stages + 8 + kMaxTaps) * sizeof(uint64_t) + kMaxTaps * 4 + 32 + 256 * sizeof(float) + 1024 + epi;
            halo_ok = true;
            // the halo kernel tiles the image 8 wide x 16 tall, one image per tile
            p.BW = 8; p.BH = 16; p.NB = 1; p.rows = 128;
            p.tiles_w = ceil_div(q.Jw, 8);
            p.tiles_h = ceil_div(q.Jh, 16);
            p.groups = q.N;
            p.tiles_per_class = p.tiles_w * p.tiles_h * p.groups;
        }
    }
    if ((p.d2s || p.planes == 2) && !halo_ok) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: shape not covered by the halo kernel");
    // Deep, spatially small layers (14^2 / 7^2 at 128-256 channels) have fewer M tiles than SMs: cut N into narrower
    // tiles until the launch fills the persistent grid (the A boxes are then re-read per N tile from L2, which is cheap).
    bool n_split = false;
    if (!halo_ok && q.n_tile == 0 && !p.d2s && p.planes != 2 && !getenv("DMV_NO_NSPLIT")) {
        const int m_tiles = p.num_classes * p.tiles_per_class;
        int nt = p.n_pad;
        while (nt > 64 && (nt % 32) == 0 && 2 * m_tiles * ceil_div(q.n_real, nt) <= num_sms() && q.n_real % (nt / 2) == 0) nt /= 2;
        if (nt != p.n_pad) {
            p.n_pad = nt;
            p.n_tiles = ceil_div(q.n_real, nt);
            n_split = true;
        }
    }

    // ---- A map: 5-D (C', W', P, H', N)
    CUtensorMap map_a, map_b;
    {
        const int s = q.src_stride;
        if (s == 2 && ((q.Hs & 1) || (q.Ws & 1))) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: stride-2 source needs even H and W");
        cuuint64_t dims[5] = {(cuuint64_t)(s * q.Cs), (cuuint64_t)(q.Ws / s), (cuuint64_t)s, (cuuint64_t)(q.Hs / s), (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cs * 2;
        cuuint64_t strides[4] = {(cuuint64_t)s * pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)s * q.Ws * pix, (cuuint64_t)q.Hs * q.Ws * pix};
        cuuint32_t box[5] = {(cuuint32_t)KC, (cuuint32_t)p.BW, 1u, (cuuint32_t)p.BH, (cuuint32_t)p.NB};
        int rc = encode_map(&map_a, q.src, 5, dims, strides, box, row_bytes);
        if (rc) return rc;
    }
    // ---- B map: 3-D.  G form reads HWIO directly as (co, ci, tap); F form reads the packed copy as (K, n, 1)
    const int taps_total = q.kh * q.kw;
    if (p.b_mode == 2) {
        // Matrix[K][N] as stored: N contiguous.  Boxes of 64 columns x KC rows, 128-byte swizzle.
        if (p.n_pad % 64) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: MN-major B needs N tiles of 64");
        cuuint64_t dims[3] = {(cuuint64_t)q.w_co, (cuuint64_t)q.w_ci, 1};
        cuuint64_t strides[2] = {(cuuint64_t)q.w_co * 2, (cuuint64_t)q.w_ci * q.w_co * 2};
        cuuint32_t box[3] = {64u, (cuuint32_t)KC, 1u};
        int rc = encode_map(&map_b, q.w_hwio, 3, dims, strides, box, 128);
        if (rc) return rc;
    } else if (q.g_form) {
        cuuint64_t dims[3] = {(cuuint64_t)q.w_co, (cuuint64_t)q.w_ci, (cuuint64_t)taps_total};
        cuuint64_t strides[2] = {(cuuint64_t)q.w_co * 2, (cuuint64_t)q.w_ci * q.w_co * 2};
        cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)p.n_pad, 1u};
        int rc = encode_map(&map_b, q.w_hwio, 3, dims, strides, box, row_bytes);
        if (rc) return rc;
    } else if (prepacked) {
        const cuuint64_t ktot = (cuuint64_t)q.w_ci;
        cuuint64_t dims[3] = {ktot, (cuuint64_t)q.w_co, 1};
        cuuint64_t strides[2] = {ktot * 2, ktot * 2 * (cuuint64_t)q.w_co};
        cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)p.n_pad, 1u};
        int rc = encode_map(&map_b, q.w_hwio, 3, dims, strides, box, row_bytes);
        if (rc) return rc;
    } else {
        const size_t need = (size_t)taps_total * q.w_ci * q.w_co * 2;
        if (!workspace || ws_bytes < need) return fail(DMV_E_WORKSPACE, "tc: workspace too small for packed weights");
        long long blocks = ceil_div_ll((long long)taps_total * q.w_ci * q.w_co, 256);
        if (blocks > 2048) blocks = 2048;
        int rc = DMV_OK;
        if (tl_pack_mode != DMV_ALGO_PREPACKED) {
            pack_f_kernel<<<(int)blocks, 256, 0, st>>>((const bf16*)q.w_hwio, (bf16*)workspace, taps_total, q.w_ci, q.w_co);
            rc = check_launch("tc pack weights");
            if (rc) return rc;
        }
        if (tl_pack_mode == DMV_ALGO_PACK_ONLY) return DMV_OK;
        const cuuint64_t ktot = (cuuint64_t)taps_total * q.w_ci;
        cuuint64_t dims[3] = {ktot, (cuuint64_t)q.w_co, 1};
        cuuint64_t strides[2] = {ktot * 2, ktot * 2 * (cuuint64_t)q.w_co};
        cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)p.n_pad, 1u};
        rc = encode_map(&map_b, workspace, 3, dims, strides, box, row_bytes);
        if (rc) return rc;
    }
    if (tl_pack_mode == DMV_ALGO_PACK_ONLY) return DMV_OK;      // a form that reads the weights in place: nothing to pack
    // ---- halo variant (see halo_kernel)
    if (halo_ok) {
        CUtensorMap map_h;
        const cuuint64_t sp = (cuuint64_t)p.planes;            // 2: parity view [N][H/2][2][W/2][2C] of the same buffer
        cuuint64_t dims[5] = {sp * q.Cs, (cuuint64_t)q.Ws / sp, sp, (cuuint64_t)q.Hs / sp, (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cs * 2;
        cuuint64_t strides[4] = {sp * pix, (cuuint64_t)q.Ws * pix, sp * q.Ws * pix, (cuuint64_t)q.Hs * q.Ws * pix};
        cuuint32_t box[5] = {(cuuint32_t)KC, (cuuint32_t)p.halo_pitch, 1u, (cuuint32_t)p.halo_h, 1u};
        int rc = encode_map(&map_h, q.src, 5, dims, strides, box, row_bytes);
        if (rc) return rc;
        p.stages = halo_stages;
        int grid = num_sms() * halo_ctas_per_sm;
        if (grid > p.tiles_per_class) grid = p.tiles_per_class;
        cudaError_t e = cudaSuccess;
        const int nt = p.cls[0].tap_count;
#define DMV_LAUNCH_HALO(KCV, NTV)                                                                                          \
    do {                                                                                                                   \
        if (p.d2s == 2) {                                                                                                  \
            e = cudaFuncSetAttribute(halo_kernel<KCV, NTV, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)halo_smem); \
            if (e == cudaSuccess) halo_kernel<KCV, NTV, 1><<<grid, kThreads, halo_smem, st>>>(map_h, map_b, p);            \
        } else {                                                                                                           \
            e = cudaFuncSetAttribute(halo_kernel<KCV, NTV, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)halo_smem); \
            if (e == cudaSuccess) halo_kernel<KCV, NTV, 0><<<grid, kThreads, halo_smem, st>>>(map_h, map_b, p);            \
        }                                                                                                                  \
    } while (0)
        if (KC == 64) {
            if (nt == 25) DMV_LAUNCH_HALO(64, 25); else if (nt == 15) DMV_LAUNCH_HALO(64, 15); else if (nt == 9) DMV_LAUNCH_HALO(64, 9); else DMV_LAUNCH_HALO(64, 0);
        } else {
            if (nt == 25) DMV_LAUNCH_HALO(32, 25); else if (nt == 9) DMV_LAUNCH_HALO(32, 9); else DMV_LAUNCH_HALO(32, 0);
        }
#undef DMV_LAUNCH_HALO
        if (e != cudaSuccess) {
            set_error("tc halo: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return DMV_E_CUDA;
        }
        count_tc_launch();
        return check_launch(p.d2s == 2 ? "halo_tc (sub-pixel, coalescing epilogue)"
                            : p.d2s    ? "halo_tc (sub-pixel)"
                            : p.planes == 2 ? "halo_tc (parity planes)"
                                            : "halo_tc");
    }
    // ---- split-K (linear layers): fp32 partials into the workspace, finished by splitk_finish_kernel
    void* final_out = p.out;
    const float* final_bias = p.bias;
    const int final_act = p.act;
    const bf16* final_dact_y = p.dact_y;
    if (q.k_splits > 1) {
        int ks = q.k_splits;
        if (ks > p.kc_per_tap / 4) ks = p.kc_per_tap / 4;
        if (ks < 1) ks = 1;
        ks = ceil_div(p.kc_per_tap, ceil_div(p.kc_per_tap, ks));     // no empty split
        const long long mn = (long long)q.N * q.n_real;
        if (ks > 1 && p.num_classes == 1 && p.cls[0].tap_count == 1 && !q.out_f32 && workspace && ws_bytes >= (size_t)ks * mn * sizeof(float)) {
            p.k_splits = ks;
            p.split_stride = mn;
            p.out = workspace;
            p.out_f32 = 1;
            p.bias = nullptr;
            p.act = DMV_ACT_NONE;
            p.dact_y = nullptr;           // applied by the finish kernel, after the splits are summed
        }
    }
    // ---- shared memory / grid
    const int stage_bytes = 128 * row_bytes + p.n_pad * row_bytes;
    // The pipeline is latency-bound (one TMA box per tap): keep as many bytes in flight per SM as
    // possible.  Narrow layers (N <= 64) run two CTAs per SM, each with half of the shared memory.
    const bool two_per_sm = p.n_pad <= 64;
    // DMV_IGEMM_SMEM2_KB: budget of the two-per-SM form (A/B: a smaller footprint lets a CTA of the chain run next to the
    // persistent fused FC update, fc_adam.cu)
    static int budget2_kb = 0;
    if (!budget2_kb) {
        const char* e = getenv("DMV_IGEMM_SMEM2_KB");
        budget2_kb = e ? atoi(e) : 106;
        if (budget2_kb < 32 || budget2_kb > 106) budget2_kb = 106;
    }
    int stages = ((two_per_sm ? budget2_kb : 200) * 1024) / stage_bytes;
    if (stages > 12) stages = 12;
    if (stages < 2) stages = 2;
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + (2 * stages + 4) * sizeof(uint64_t) + 32 + 256 * sizeof(float) + 1024;
    const int total_tiles = p.num_classes * p.tiles_per_class * p.n_tiles * p.k_splits;
    int grid = num_sms() * (two_per_sm ? 2 : 1);
    if (grid > total_tiles) grid = total_tiles;
    cudaError_t e;
    if (KC == 64) {
        e = cudaFuncSetAttribute(igemm_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) igemm_kernel<64><<<grid, kThreads, smem, st>>>(map_a, map_b, p);
    } else {
        e = cudaFuncSetAttribute(igemm_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) igemm_kernel<32><<<grid, kThreads, smem, st>>>(map_a, map_b, p);
    }
    if (e != cudaSuccess) {
        set_error("tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    count_tc_launch();
    int rc_l = check_launch(p.k_splits > 1 ? "igemm_tc (split-K)" : n_split ? "igemm_tc (N-split)" : "igemm_tc");
    if (rc_l) return rc_l;
    if (p.k_splits > 1) {
        const long long mn = (long long)q.N * q.n_real;
        long long blocks = ceil_div_ll(mn, 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        splitk_finish_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float*>(workspace), final_bias, reinterpret_cast<bf16*>(final_out), mn,
                                                           q.n_real, p.k_splits, final_act, final_dact_y, p.dact);
        return check_launch("splitk_finish");
    }
    return DMV_OK;
}

// ---- sub-pixel form of the stride-2 G problems (deconv fwd, conv dgrad) ---------------------------------
// The four output-parity classes of a stride-2 transposed convolution read the SAME stride-1 source through
// the same few shifts (3 x 3 for a 5 x 5 kernel, 2 x 2 for 3 x 3).  Concatenating the classes along N turns the
// layer into one stride-1 convolution with S shifts and 4 * C output columns whose weight matrix is the
// reference weights scattered by (shift, class) -- zero where a class has no tap at that shift -- followed by a
// depth-to-space store.  One halo load then serves all taps (the per-tap form re-reads the source kh * kw
// times from L2 and is bound by it), and the MMA N grows from C to 4 C.
struct SubpixelTable {
    int S;
    short dh[16], dw[16];
    int tap[4][16];      // reference tap id r * kw + s of (class, shift), -1: none
};

__global__ void pack_subpixel_kernel(const bf16* __restrict__ w, bf16* __restrict__ out, int n_real, int Cs, int n_rows, SubpixelTable t) {
    const long long K = (long long)t.S * Cs, total = (long long)n_rows * K;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int row = (int)(i / K);
        const int kk = (int)(i - (long long)row * K);
        const int j = kk / Cs, k = kk - j * Cs;
        const int cls = row / n_real, n = row - cls * n_real;
        bf16 v = __float2bfloat16_rn(0.f);
        if (cls < 4) {
            const int id = t.tap[cls][j];
            if (id >= 0) v = w[((long long)id * n_real + n) * Cs + k];      // w[tap][n][k]
        }
        out[i] = v;
    }
}

bool subpixel_eligible(int Cs, int n_real, int Jh, int Jw, int kh, int kw) {
    if (getenv("DMV_NO_SUBPIXEL") || getenv("DMV_NO_HALO")) return false;
    if (!(Cs == 32 || Cs == 64) || n_real > 64 || n_real < 1) return false;
    if (n_real >= 16 && (n_real & 15)) return false;
    if (n_real < 16 && (16 % n_real)) return false;
    if (Jh * Jw < 256 || kh > 5 || kw > 5) return false;
    // the halo kernel keeps all S weight tiles resident next to two input windows
    const int S = ((kh + 2) / 2) * ((kw + 2) / 2), dh = (kh + 2) / 2 - 1, dw = (kw + 2) / 2 - 1;
    const size_t wbytes = (size_t)S * ceil_div(4 * n_real, 16) * 16 * Cs * 2;
    const size_t a_stage = ((size_t)(16 + dh) * (8 + dw) * Cs * 2 + 1023) & ~(size_t)1023;
    return wbytes + 2 * a_stage <= 200 * 1024;
}

size_t subpixel_workspace(int Cs, int n_real, int kh, int kw) {
    const int S = ((kh + 2) / 2) * ((kw + 2) / 2);          // upper bound on the number of shifts
    return (size_t)ceil_div(4 * n_real, 16) * 16 * S * Cs * 2 + 256;
}

// taps of the F form (conv-fwd-like): A pixel = out*stride + (r - pt, s - pl)
int build_f(IgemmParams& p, int kh, int kw, int stride, int pt, int pl) {
    if (kh * kw > kMaxTaps) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: too many taps");
    p.num_classes = 1;
    p.cls[0] = TapClass{0, kh * kw, 0, 0, 0};
    for (int r = 0; r < kh; ++r)
        for (int s = 0; s < kw; ++s) {
            Tap& t = p.taps[r * kw + s];
            const int dy = r - pt, dx = s - pl;
            if (stride == 1) {
                t.dh = (short)dy; t.dw = (short)dx; t.ph = 0; t.pw = 0;
            } else {
                t.ph = (short)(((dy % 2) + 2) % 2); t.dh = (short)((dy - t.ph) / 2);
                t.pw = (short)(((dx % 2) + 2) % 2); t.dw = (short)((dx - t.pw) / 2);
            }
            t.id = r * kw + s;
        }
    return DMV_OK;
}

// taps of the G form (conv-dgrad-like): small pixel = (big + pad - tap) / stride, split by output parity
int build_g(IgemmParams& p, int kh, int kw, int stride, int pt, int pl, int w_co) {
    int n = 0;
    p.num_classes = stride * stride;
    if (stride > 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: stride > 2");
    for (int py = 0; py < stride; ++py)
        for (int px = 0; px < stride; ++px) {
            TapClass& c = p.cls[py * stride + px];
            c.tap_begin = n; c.py = py; c.px = px; c.k_elem_offset = 0;
            for (int r = 0; r < kh; ++r) {
                if ((py + pt - r) % stride) continue;
                for (int s = 0; s < kw; ++s) {
                    if ((px + pl - s) % stride) continue;
                    if (n >= kMaxTaps) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: too many taps");
                    Tap& t = p.taps[n++];
                    t.dh = (short)((py + pt - r) / stride); t.dw = (short)((px + pl - s) / stride);
                    t.ph = 0; t.pw = 0; t.id = r * kw + s;
                }
            }
            c.tap_count = n - c.tap_begin;
            if (c.tap_count == 0) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc: empty parity class");
        }
    (void)w_co;
    return DMV_OK;
}

// ---- stride-2 F problems (conv fwd, deconv dgrad) with 32 source channels on the halo kernel ------------------
// In the parity view [N][H/2][2][W/2][2C] a stride-2 tap (r, s) reads row plane ph = (r - pt) mod 2 at window shift
// dh = floor((r - pt) / 2), and column shift dw = floor((s - pl) / 2) with the column parity pw selecting one half of
// the 2C = 64 channels of a window row.  Folding pw into the contraction gives kh x ceil((kw + 1) / 2) taps of K = 64
// (zero weights where s falls outside the kernel), each an ordinary shifted window of one of the TWO planes, which the
// halo kernel loads once per tile instead of once per tap.
static int fdiv2(int a) { return a >= 0 ? a / 2 : -((-a + 1) / 2); }

struct S2Table {
    int n;
    short dh[kMaxTaps], dw[kMaxTaps], ph[kMaxTaps], r[kMaxTaps], s0[kMaxTaps], s1[kMaxTaps];   // s0 / s1: kernel column of pw = 0 / 1, -1: none
};

__global__ void pack_f_s2_kernel(const bf16* __restrict__ w, bf16* __restrict__ out, int kw, int Cin, int Cout, S2Table t) {
    const int K = t.n * 2 * Cin, total = Cout * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int co = i / K, kk = i - co * K;
        const int j = kk / (2 * Cin), rem = kk - j * 2 * Cin;
        const int pw = rem / Cin, c = rem - pw * Cin;
        const int sc = pw ? t.s1[j] : t.s0[j];
        out[i] = sc >= 0 ? w[((long long)(t.r[j] * kw + sc) * Cin + c) * Cout + co] : __float2bfloat16_rn(0.f);
    }
}

bool f_s2_eligible(int Cs, int n_real, int Jh, int Jw, int Hs, int Ws, int kh, int kw, int pt, int pl) {
    if (getenv("DMV_NO_S2HALO") || getenv("DMV_NO_HALO")) return false;
    if (Cs != 32 || (Hs & 1) || (Ws & 1) || Jh * Jw < 256 || n_real > 256 || (n_real & 15)) return false;
    const int ndw = fdiv2(kw - 1 - pl) - fdiv2(-pl) + 1, ndh = fdiv2(kh - 1 - pt) - fdiv2(-pt) + 1;
    const int taps = kh * ndw;
    if (taps > kMaxTaps) return false;
    const size_t wbytes = (size_t)taps * n_real * 128;
    const size_t plane = ((size_t)(16 + ndh - 1) * (8 + ndw - 1) * 128 + 1023) & ~(size_t)1023;
    return wbytes + 2 * 2 * plane <= 220 * 1024;
}

// src [N][Hs][Ws][32] bf16 read with stride 2; w is the reference layout [kh][kw][32][n_real]
int launch_f_s2(const void* src, int N, int Hs, int Ws, const void* w, int kh, int kw, int pt, int pl, const float* bias, int act,
                void* out, int out_f32, int out_H, int out_W, int n_real, void* ws, size_t ws_bytes, cudaStream_t st) {
    S2Table t;
    memset(&t, 0, sizeof(t));
    const int dw_lo = fdiv2(-pl), dw_hi = fdiv2(kw - 1 - pl);
    for (int r = 0; r < kh; ++r)
        for (int dw = dw_lo; dw <= dw_hi; ++dw) {
            const int j = t.n++;
            const int dy = r - pt;
            t.ph[j] = (short)(((dy % 2) + 2) % 2);
            t.dh[j] = (short)((dy - t.ph[j]) / 2);
            t.dw[j] = (short)dw;
            t.r[j] = (short)r;
            const int s0 = 2 * dw + pl, s1 = 2 * dw + 1 + pl;
            t.s0[j] = (short)((s0 >= 0 && s0 < kw) ? s0 : -1);
            t.s1[j] = (short)((s1 >= 0 && s1 < kw) ? s1 : -1);
        }
    const size_t need = (size_t)n_real * t.n * 64 * 2;
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 15)) return fail(DMV_E_WORKSPACE, "tc stride-2 halo: workspace too small");
    int rc = DMV_OK;
    if (tl_pack_mode != DMV_ALGO_PREPACKED) {
        pack_f_s2_kernel<<<ceil_div(n_real * t.n * 64, 256), 256, 0, st>>>((const bf16*)w, (bf16*)ws, kw, 32, n_real, t);
        rc = check_launch("tc pack stride-2");
        if (rc) return rc;
    }
    if (tl_pack_mode == DMV_ALGO_PACK_ONLY) return DMV_OK;
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    p.num_classes = 1;
    p.planes = 2;
    p.cls[0] = TapClass{0, t.n, 0, 0, 0};
    for (int j = 0; j < t.n; ++j) {
        p.taps[j].dh = t.dh[j]; p.taps[j].dw = t.dw[j]; p.taps[j].ph = t.ph[j]; p.taps[j].pw = 0; p.taps[j].id = j;
    }
    Problem q;
    q.src = src; q.N = N; q.Hs = Hs; q.Ws = Ws; q.Cs = 32; q.src_stride = 2;
    q.w_hwio = ws; q.kh = 1; q.kw = t.n; q.w_ci = t.n * 64; q.w_co = n_real; q.g_form = false; q.n_tile = 0; q.b_mode_override = 3; q.k_splits = 1;
    q.out = out; q.out_f32 = out_f32; q.out_H = out_H; q.out_W = out_W; q.n_real = n_real; q.out_mul = 1;
    q.Jh = out_H; q.Jw = out_W; q.bias = bias; q.act = act;
    return launch_igemm(q, p, nullptr, 0, st);
}

// Stride-2 G problem as one stride-1 halo launch (see SubpixelTable).  w is the reference layout read as
// w[tap][n_real][Cs] (conv dgrad: [kh][kw][Cin][Cout]; deconv fwd: [kh][kw][Cout_t][Cin_t]).
int launch_subpixel(const void* src, int N, int Hs, int Ws, int Cs, const void* w, int kh, int kw, int pt, int pl, void* out, int out_f32,
                    int out_H, int out_W, int n_real, int act, void* ws, size_t ws_bytes, cudaStream_t st) {
    IgemmParams g;
    memset(&g, 0, sizeof(g));
    int rc = build_g(g, kh, kw, 2, pt, pl, Cs);
    if (rc) return rc;
    SubpixelTable t;
    memset(&t, 0, sizeof(t));
    for (int c = 0; c < 4; ++c)
        for (int j = 0; j < 16; ++j) t.tap[c][j] = -1;
    for (int c = 0; c < 4; ++c) {
        const TapClass& tc_ = g.cls[c];
        const int cls = tc_.py * 2 + tc_.px;
        for (int j = 0; j < tc_.tap_count; ++j) {
            const Tap& tp = g.taps[tc_.tap_begin + j];
            int sidx = -1;
            for (int z = 0; z < t.S; ++z)
                if (t.dh[z] == tp.dh && t.dw[z] == tp.dw) sidx = z;
            if (sidx < 0) {
                if (t.S >= 16) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc subpixel: too many shifts");
                sidx = t.S++;
                t.dh[sidx] = tp.dh; t.dw[sidx] = tp.dw;
            }
            t.tap[cls][sidx] = tp.id;
        }
    }
    const int n_rows = ceil_div(4 * n_real, 16) * 16;
    const size_t need = (size_t)n_rows * t.S * Cs * 2;
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 15)) return fail(DMV_E_WORKSPACE, "tc subpixel: workspace too small");
    long long blocks = ceil_div_ll((long long)n_rows * t.S * Cs, 256);
    if (blocks > 1184) blocks = 1184;
    if (tl_pack_mode != DMV_ALGO_PREPACKED) {
        pack_subpixel_kernel<<<(int)blocks, 256, 0, st>>>((const bf16*)w, (bf16*)ws, n_real, Cs, n_rows, t);
        rc = check_launch("tc pack subpixel");
        if (rc) return rc;
    }
    if (tl_pack_mode == DMV_ALGO_PACK_ONLY) return DMV_OK;
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    p.num_classes = 1;
    p.cls[0] = TapClass{0, t.S, 0, 0, 0};
    for (int j = 0; j < t.S; ++j) {
        p.taps[j].dh = t.dh[j]; p.taps[j].dw = t.dw[j]; p.taps[j].ph = 0; p.taps[j].pw = 0; p.taps[j].id = j;
    }
    p.d2s = 1; p.d2s_c = n_real;
    Problem q;
    q.src = src; q.N = N; q.Hs = Hs; q.Ws = Ws; q.Cs = Cs; q.src_stride = 1;
    q.w_hwio = ws; q.kh = 1; q.kw = t.S; q.w_ci = t.S * Cs; q.w_co = n_rows; q.g_form = false; q.n_tile = 0; q.b_mode_override = 3; q.k_splits = 1;
    q.out = out; q.out_f32 = out_f32; q.out_H = out_H; q.out_W = out_W; q.n_real = n_rows; q.out_mul = 1;
    q.Jh = ceil_div(out_H, 2); q.Jw = ceil_div(out_W, 2); q.bias = nullptr; q.act = act;
    return launch_igemm(q, p, nullptr, 0, st);
}

}  // namespace

// ----------------------------------------------------------------------------------------------
// entry points used by conv_api.cu
// ----------------------------------------------------------------------------------------------
namespace dmv {
void tc_set_pack_mode(int mode) { tl_pack_mode = mode; }

void tc_set_dact(const void* y_bf16, int act) {
    tl_dact_y = (act != DMV_ACT_NONE) ? y_bf16 : nullptr;
    tl_dact = act;
    tl_dact_taken = false;
}
bool tc_finish_dact() {          // true when a launch applied the factor; clears the request either way
    const bool taken = tl_dact_taken;
    tl_dact_y = nullptr;
    tl_dact_taken = false;
    return taken;
}



size_t tc_pack_workspace(int taps, int Cin, int Cout) {
    // F-form packed copy, or the sub-pixel matrix of a stride-2 G form (4 classes x <= taps shifts, rows padded to 16)
    const size_t big = Cin > Cout ? Cin : Cout, small = Cin > Cout ? Cout : Cin;
    return (size_t)taps * (4 * big + 16) * (small < 32 ? 32 : small) * 2 + 256;
}

// conv fwd: F form, A = x
int tc_conv_fwd(const void* x, int xdt, const void* w, const float* bias, void* y, int ydt, int B, int H, int W, int Cin, int Cout,
                int kh, int kw, int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (xdt != DMV_DT_BF16) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_conv_fwd: bf16 input only");
    if (stride != 1 && stride != 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_conv_fwd: stride");
    const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
    if (stride == 2 && f_s2_eligible(Cin, Cout, ph.out, pw.out, H, W, kh, kw, ph.before, pw.before) && ws_bytes >= (size_t)Cout * kh * ((kw + 2) / 2) * 128)
        return launch_f_s2(x, B, H, W, w, kh, kw, ph.before, pw.before, bias, act, y, ydt == DMV_DT_F32, ph.out, pw.out, Cout, ws, ws_bytes, st);
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_f(p, kh, kw, stride, ph.before, pw.before);
    if (rc) return rc;
    Problem q;
    q.src = x; q.N = B; q.Hs = H; q.Ws = W; q.Cs = Cin; q.src_stride = stride;
    q.w_hwio = w; q.kh = kh; q.kw = kw; q.w_ci = Cin; q.w_co = Cout; q.g_form = false; q.n_tile = 0; q.b_mode_override = -1; q.k_splits = 1;
    q.out = y; q.out_f32 = (ydt == DMV_DT_F32); q.out_H = ph.out; q.out_W = pw.out; q.n_real = Cout; q.out_mul = 1;
    q.Jh = ph.out; q.Jw = pw.out; q.bias = bias; q.act = act;
    return launch_igemm(q, p, ws, ws_bytes, st);
}

// conv dgrad: G form, A = dy (small side), output = dx (big side, Cin channels)
int tc_conv_dgrad(const void* dy, const void* w, void* dx, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                  void* ws, size_t ws_bytes, cudaStream_t st) {
    if (stride != 1 && stride != 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_conv_dgrad: stride");
    const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
    if (stride == 2 && subpixel_eligible(Cout, Cin, ceil_div(H, 2), ceil_div(W, 2), kh, kw) && ws_bytes >= subpixel_workspace(Cout, Cin, kh, kw))
        return launch_subpixel(dy, B, ph.out, pw.out, Cout, w, kh, kw, ph.before, pw.before, dx, 0, H, W, Cin, DMV_ACT_NONE, ws, ws_bytes, st);
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_g(p, kh, kw, stride, ph.before, pw.before, Cout);
    if (rc) return rc;
    Problem q;
    q.src = dy; q.N = B; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cout; q.src_stride = 1;
    q.w_hwio = w; q.kh = kh; q.kw = kw; q.w_ci = Cin; q.w_co = Cout; q.g_form = true; q.n_tile = 0; q.b_mode_override = -1; q.k_splits = 1;
    q.out = dx; q.out_f32 = 0; q.out_H = H; q.out_W = W; q.n_real = Cin; q.out_mul = stride;
    q.Jh = ceil_div(H, stride); q.Jw = ceil_div(W, stride); q.bias = nullptr; q.act = DMV_ACT_NONE;
    return launch_igemm(q, p, ws, ws_bytes, st);
}

// deconv fwd: G form with the deconv's weights w[kh][kw][Cout_t][Cin_t] (ci-role = Cout_t, co-role = Cin_t)
int tc_deconv_fwd(const void* x, const void* w, void* y, int ydt, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                  int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (stride != 1 && stride != 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_deconv_fwd: stride");
    const SamePad ph = same_pad(Hout, kh, stride), pw = same_pad(Wout, kw, stride);
    if (stride == 2 && subpixel_eligible(Cin, Cout, ceil_div(Hout, 2), ceil_div(Wout, 2), kh, kw) &&
        ws_bytes >= subpixel_workspace(Cin, Cout, kh, kw))
        return launch_subpixel(x, B, ph.out, pw.out, Cin, w, kh, kw, ph.before, pw.before, y, ydt == DMV_DT_F32, Hout, Wout, Cout, act, ws,
                               ws_bytes, st);
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_g(p, kh, kw, stride, ph.before, pw.before, Cin);
    if (rc) return rc;
    Problem q;
    q.src = x; q.N = B; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cin; q.src_stride = 1;
    q.w_hwio = w; q.kh = kh; q.kw = kw; q.w_ci = Cout; q.w_co = Cin; q.g_form = true; q.n_tile = 0; q.b_mode_override = -1; q.k_splits = 1;
    q.out = y; q.out_f32 = (ydt == DMV_DT_F32); q.out_H = Hout; q.out_W = Wout; q.n_real = Cout; q.out_mul = stride;
    q.Jh = ceil_div(Hout, stride); q.Jw = ceil_div(Wout, stride); q.bias = nullptr; q.act = act;
    return launch_igemm(q, p, ws, ws_bytes, st);
}

// deconv dgrad: F form over dy (big side, Cout_t channels) with w[kh][kw][Cout_t][Cin_t]
int tc_deconv_dgrad(const void* dy, int dydt, const void* w, void* dx, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                    int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (dydt != DMV_DT_BF16) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_deconv_dgrad: bf16 gradient only");
    if (stride != 1 && stride != 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_deconv_dgrad: stride");
    const SamePad ph = same_pad(Hout, kh, stride), pw = same_pad(Wout, kw, stride);
    if (stride == 2 && f_s2_eligible(Cout, Cin, ph.out, pw.out, Hout, Wout, kh, kw, ph.before, pw.before) && ws_bytes >= (size_t)Cin * kh * ((kw + 2) / 2) * 128)
        return launch_f_s2(dy, B, Hout, Wout, w, kh, kw, ph.before, pw.before, nullptr, DMV_ACT_NONE, dx, 0, ph.out, pw.out, Cin, ws, ws_bytes, st);
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_f(p, kh, kw, stride, ph.before, pw.before);
    if (rc) return rc;
    Problem q;
    q.src = dy; q.N = B; q.Hs = Hout; q.Ws = Wout; q.Cs = Cout; q.src_stride = stride;
    q.w_hwio = w; q.kh = kh; q.kw = kw; q.w_ci = Cout; q.w_co = Cin; q.g_form = false; q.n_tile = 0; q.b_mode_override = -1; q.k_splits = 1;
    q.out = dx; q.out_f32 = 0; q.out_H = ph.out; q.out_W = pw.out; q.n_real = Cin; q.out_mul = 1;
    q.Jh = ph.out; q.Jw = pw.out; q.bias = nullptr; q.act = DMV_ACT_NONE;
    return launch_igemm(q, p, ws, ws_bytes, st);
}


// linear forward: Y[M,N] = X[M,K] Matrix[K,N] + b.  A = X (K-major rows), B = Matrix as stored (MN-major),
// N tiles of 64 columns so that the weight stream (the whole cost at M = 64) is spread over >= 64 CTAs.
static int linear_ntile() {
    const char* e = getenv("DMV_LINEAR_NTILE");
    const int v = e ? atoi(e) : 64;
    return (v == 64 || v == 128 || v == 256) ? v : 64;
}

// Split count of a linear layer's contraction: the launch is n_tiles x ks equal tiles on a persistent grid; pick the
// ks whose tile count fills whole waves of the grid best (a ragged last wave idles most SMs for a whole tile time).
static int linear_splits(int n_tiles, int kblocks, int n_tile) {
    if (kblocks < 1 || n_tiles < 1) return 1;
    const int grid = num_sms() * (n_tile <= 64 ? 2 : 1);
    int kmax = kblocks / 4;
    if (kmax < 1) kmax = 1;
    if (kmax > 32) kmax = 32;
    int best = 1;
    double best_eff = -1.0;
    for (int ks = 1; ks <= kmax; ++ks) {
        const int tiles = n_tiles * ceil_div(kblocks, ceil_div(kblocks, ks));
        const int waves = ceil_div(tiles, grid);
        if (waves > 2) break;
        const double eff = (double)tiles / ((double)waves * grid);
        if (eff > best_eff + 0.02) { best_eff = eff; best = ks; }
    }
    return best;
}

static int linear_ntile_for(long long weights) {
    if (getenv("DMV_LINEAR_NTILE")) return linear_ntile();
    return weights >= (32ll << 20) ? 128 : 64;      // wider weight boxes for the two 51 M-parameter layers
}

size_t tc_linear_workspace(int M, int K, int N) {
    const int nt = linear_ntile_for((long long)K * N);
    const int a = linear_splits(ceil_div(N, nt), K / ((K % 64 == 0) ? 64 : 32), nt), b = linear_splits(ceil_div(K, nt), N / ((N % 64 == 0) ? 64 : 32), nt);
    const size_t fa = (size_t)a * M * N * 4, fb = (size_t)b * M * K * 4;
    return (fa > fb ? fa : fb) + 256;
}

int tc_linear_fwd(const void* x, const void* w, const float* bias, void* y, int M, int K, int N, int act, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
    if (K % 32 || N % 8) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_linear_fwd: need K % 32 == 0 and N % 8 == 0");
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_f(p, 1, 1, 1, 0, 0);
    if (rc) return rc;
    Problem q;
    q.src = x; q.N = M; q.Hs = 1; q.Ws = 1; q.Cs = K; q.src_stride = 1;
    q.w_hwio = w; q.kh = 1; q.kw = 1; q.w_ci = K; q.w_co = N; q.g_form = false; q.n_tile = linear_ntile_for((long long)K * N); q.b_mode_override = 2;
    q.k_splits = (M <= 128) ? linear_splits(ceil_div(N, q.n_tile), K / ((K % 64 == 0) ? 64 : 32), q.n_tile) : 1;
    q.out = y; q.out_f32 = 0; q.out_H = 1; q.out_W = 1; q.n_real = N; q.out_mul = 1;
    q.Jh = 1; q.Jw = 1; q.bias = bias; q.act = act;
    return launch_igemm(q, p, ws, ws_bytes, st);
}

// linear dgrad: dX[M,K] = dY[M,N] Matrix[K,N]^T.  A = dY rows, B = Matrix rows (contraction over N is contiguous:
// K-major), output columns = K in tiles of 64.
int tc_linear_dgrad(const void* dy, const void* w, void* dx, int M, int K, int N, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (N % 32 || K % 8) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_linear_dgrad: need N % 32 == 0 and K % 8 == 0");
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    int rc = build_g(p, 1, 1, 1, 0, 0, N);
    if (rc) return rc;
    Problem q;
    q.src = dy; q.N = M; q.Hs = 1; q.Ws = 1; q.Cs = N; q.src_stride = 1;
    q.w_hwio = w; q.kh = 1; q.kw = 1; q.w_ci = K; q.w_co = N; q.g_form = true; q.n_tile = linear_ntile_for((long long)K * N); q.b_mode_override = -1;
    q.k_splits = (M <= 128) ? linear_splits(ceil_div(K, q.n_tile), N / ((N % 64 == 0) ? 64 : 32), q.n_tile) : 1;
    q.out = dx; q.out_f32 = 0; q.out_H = 1; q.out_W = 1; q.n_real = K; q.out_mul = 1;
    q.Jh = 1; q.Jw = 1; q.bias = nullptr; q.act = DMV_ACT_NONE;
    return launch_igemm(q, p, ws, ws_bytes, st);
}

// ---- thin-channel layers (3-channel image side of e0, 2-channel side of the flow head) -------------------
// The patch matrix P[pixel][Kp] (bf16, k = (tap, ct), zero padded to a multiple of 32) is written once by a gather
// kernel; the layer is then a 1x1 convolution over P on the tensor cores.
static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

size_t tc_thin_workspace(int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw, int stride) {
    const SamePad ph = same_pad(Hb, kh, stride), pw = same_pad(Wb, kw, stride);
    const int Kp = thin_patch_cols(kh * kw, Ct);
    const size_t P = align256((size_t)N * ph.out * pw.out * Kp * 2);
    const size_t packed = align256((size_t)Cw * Kp * 2);
    const size_t dwt = align256((size_t)Kp * Cw * 4);
    const size_t parts = tc_wgrad_workspace(1, Kp, Cw, N, ph.out, pw.out);
    return P + packed + dwt + parts + 1024;
}

int tc_thin_fwd(const void* thin, int thin_dtype, const void* w, const float* bias, void* out, int out_dtype, int N, int Hb, int Wb, int Ct,
                int Cw, int kh, int kw, int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (Cw % 8 || Cw > 256) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_thin_fwd: output channels");
    const SamePad ph = same_pad(Hb, kh, stride), pw = same_pad(Wb, kw, stride);
    if (thin_dtype == DMV_DT_S2D && !thin_s2d_eligible(Hb, Wb, Ct, Cw, kh, kw, stride))
        return fail(DMV_E_INVALID_ARG, "DMV_DT_S2D input for a layer that does not take the space-to-depth path");
    if (thin_s2d_eligible(Hb, Wb, Ct, Cw, kh, kw, stride)) {
        // space-to-depth: stride-1 conv over X2[n][Hb/2][Wb/2][32] with kh2 x kw2 shifts on the halo kernel -- no patch matrix
        const S2dGeom g2 = thin_s2d_geom(Hb, Wb, kh, kw);
        const int S = g2.kh2 * g2.kw2;
        const bool given = thin_dtype == DMV_DT_S2D;          // the caller keeps X2 (dmv_thin_s2d_prep)
        const size_t Xb = given ? 0 : align256((size_t)N * (Hb / 2) * (Wb / 2) * 64), Wp = align256((size_t)Cw * S * 64);
        if (!ws || ws_bytes < Xb + Wp || ((uintptr_t)ws & 255)) return fail(DMV_E_WORKSPACE, "tc_thin_fwd: workspace too small or unaligned");
        uint8_t* base = reinterpret_cast<uint8_t*>(ws);
        const void* x2 = given ? thin : base;
        int rc = given ? DMV_OK : thin_s2d_prep(thin, thin_dtype, base, N, Hb, Wb, Ct, st);
        if (rc) return rc;
        rc = thin_s2d_pack_weights(w, base + Xb, Ct, Cw, kh, kw, ph.before, pw.before, g2, st);
        if (rc) return rc;
        IgemmParams p;
        memset(&p, 0, sizeof(p));
        p.num_classes = 1;
        p.cls[0] = TapClass{0, S, 0, 0, 0};
        for (int j = 0; j < S; ++j) {
            p.taps[j].dh = (short)(g2.dh0 + j / g2.kw2); p.taps[j].dw = (short)(g2.dw0 + j % g2.kw2);
            p.taps[j].ph = 0; p.taps[j].pw = 0; p.taps[j].id = j;
        }
        Problem q;
        q.src = x2; q.N = N; q.Hs = Hb / 2; q.Ws = Wb / 2; q.Cs = 32; q.src_stride = 1;
        q.w_hwio = base + Xb; q.kh = 1; q.kw = S; q.w_ci = S * 32; q.w_co = Cw; q.g_form = false; q.n_tile = 0; q.b_mode_override = 3; q.k_splits = 1;
        q.out = out; q.out_f32 = (out_dtype == DMV_DT_F32); q.out_H = ph.out; q.out_W = pw.out; q.n_real = Cw; q.out_mul = 1;
        q.Jh = ph.out; q.Jw = pw.out; q.bias = bias; q.act = act;
        return launch_igemm(q, p, nullptr, 0, st);
    }
    const int rows = kh * kw * Ct, Kp = thin_patch_cols(kh * kw, Ct);
    const size_t Pb = align256((size_t)N * ph.out * pw.out * Kp * 2), Wb_ = align256((size_t)Cw * Kp * 2);
    if (!ws || ws_bytes < Pb + Wb_ || ((uintptr_t)ws & 255)) return fail(DMV_E_WORKSPACE, "tc_thin_fwd: workspace too small or unaligned");
    uint8_t* base = reinterpret_cast<uint8_t*>(ws);
    int rc = thin_im2col(thin, thin_dtype, base, N, Hb, Wb, Ct, kh, kw, stride, st);
    if (rc) return rc;
    rc = thin_pack_weights(w, base + Pb, rows, Cw, Kp, st);
    if (rc) return rc;
    IgemmParams p;
    memset(&p, 0, sizeof(p));
    rc = build_f(p, 1, 1, 1, 0, 0);
    if (rc) return rc;
    Problem q;
    q.src = base; q.N = N; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Kp; q.src_stride = 1;
    q.w_hwio = base + Pb; q.kh = 1; q.kw = 1; q.w_ci = Kp; q.w_co = Cw; q.g_form = false; q.n_tile = 0; q.b_mode_override = 3; q.k_splits = 1;
    q.out = out; q.out_f32 = (out_dtype == DMV_DT_F32); q.out_H = ph.out; q.out_W = pw.out; q.n_real = Cw; q.out_mul = 1;
    q.Jh = ph.out; q.Jw = pw.out; q.bias = bias; q.act = act;
    return launch_igemm(q, p, nullptr, 0, st);
}

}  // namespace dmv


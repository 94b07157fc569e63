// tcgen05 weight-gradient kernel (conv / deconv / linear wgrad) for sm_100a.
//
//     dW[(tap, ci), co] = sum_{pixels} Big_tap[pixel, ci] * Small[pixel, co]
// is a GEMM whose contraction runs over PIXELS.  Both operands are read straight from the
// NHWC activation tensors as MN-major tcgen05 operands -- no transposed copies:
//   A (M = tap x ci): per (tap, 32/64-channel chunk) one TMA box of the tap-shifted input
//       window [pixels][channels]; boxes are stacked along M until 128 rows are reached
//       (e.g. 4 taps x 32 channels), the LBO of the matrix descriptor being the box size.
//   B (N = co): the matching box of the gradient tensor [pixels][co].
// Stride-2 layers use the same parity-view tensor map as the forward kernel; TMA zero fill
// supplies TF-SAME padding and the ragged image edge.
// One CTA owns a group of M tiles (as many fp32 accumulators as fit the 512 TMEM columns), an
// N tile (<= 256 output channels) and a slice of the pixels; it streams its pixel chunks
// through a TMA/mbarrier pipeline and finally stores its accumulators.  Partial results of
// the pixel slices go to the workspace and are summed in slice order by a second kernel
// (deterministic split-K); a single slice writes dW directly.
// Warp roles: 0 = TMA producer, 1 = MMA issuer (+ TMEM allocator), 2..5 = epilogue.
#include <stdlib.h>

#include "tc_common.cuh"
#include "conv_impl.h"

namespace {
using namespace dmv;
using namespace dmv::tc;

constexpr int kThreads = 192;
constexpr int kMaxBoxes = 200;   // (tap, channel chunk) boxes along M

struct ABox {
    short dh, dw, ph, c_off;   // shift in the parity view, parity plane, channel offset inside the view
    int row0;                  // first dW row of this box: tap_id * Cbig + chunk * CB
};
struct WgradParams {
    int n_boxes, boxes_per_tile, m_tiles, tiles_per_group, groups;   // M decomposition
    int CB, row_bytes_a;            // channels per A box, bytes per smem row of A
    int CBs, row_bytes_b, b_boxes;  // same for B; boxes per N tile
    int n_tile, n_tiles, Cs;        // output channels per N tile (UMMA N), number of N tiles, total
    int BW, BH, NB, rows;           // pixel chunk box; rows = BW*BH*NB (multiple of 16)
    int tiles_w, tiles_h, img_groups, chunks, slices, chunks_per_slice;
    int stages;
    long long out_elems;            // rows_total * Cs (size of one partial)
    float* out;                     // partials (slices > 1) or dW itself
    ABox box[kMaxBoxes];
};

__global__ void __launch_bounds__(kThreads, 1) wgrad_kernel(const __grid_constant__ CUtensorMap map_a,
                                                             const __grid_constant__ CUtensorMap map_b,
                                                             const __grid_constant__ WgradParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int a_box_bytes = p.rows * p.row_bytes_a;
    const int a_bytes = p.boxes_per_tile * a_box_bytes;
    const int b_box_bytes = p.rows * p.row_bytes_b;
    const int b_bytes = p.b_boxes * b_box_bytes;
    const int stage_bytes = a_bytes + b_bytes;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* done_bar = empty_bar + p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
    float* s_tr = reinterpret_cast<float*>(smem + (size_t)p.stages * stage_bytes + 1024);   // [4 warps][32 x 32] epilogue transpose tiles

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // work item of this CTA
    int w = blockIdx.x;
    const int slice = w % p.slices; w /= p.slices;
    const int nt = w % p.n_tiles; w /= p.n_tiles;
    const int grp = w;
    const int mt0 = grp * p.tiles_per_group;
    const int mt1 = min(p.m_tiles, mt0 + p.tiles_per_group);
    const int n_mt = mt1 - mt0;
    const int ch0 = slice * p.chunks_per_slice;
    const int ch1 = min(p.chunks, ch0 + p.chunks_per_slice);

    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(p.tiles_per_group * p.n_tile)) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = ch0; ch < ch1; ++ch) {
                int t = ch;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                const int g = t;
                for (int mt = mt0; mt < mt1; ++mt) {
                    const int b0 = mt * p.boxes_per_tile;
                    const int nb = min(p.boxes_per_tile, p.n_boxes - b0);
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + (size_t)stage * stage_bytes;
                    mbar_expect_tx(&full_bar[stage], (uint32_t)(nb * a_box_bytes + b_bytes));
                    for (int j = 0; j < nb; ++j) {
                        const ABox& bx = p.box[b0 + j];
                        tma_load_5d(sa + j * a_box_bytes, &map_a, &full_bar[stage], bx.c_off, tw * p.BW + bx.dw, bx.ph,
                                    th * p.BH + bx.dh, g * p.NB);
                    }
                    for (int j = 0; j < p.b_boxes; ++j)
                        tma_load_5d(sa + a_bytes + j * b_box_bytes, &map_b, &full_bar[stage], nt * p.n_tile + j * p.CBs, tw * p.BW, 0,
                                    th * p.BH, g * p.NB);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // D = f32, A = B = bf16, both MN-major (bits 15, 16), N = n_tile, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.n_tile >> 3) << 17) |
                                   ((128u >> 4) << 24);
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = ch0; ch < ch1; ++ch) {
                for (int i = 0; i < n_mt; ++i) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint64_t adesc = make_mnmajor_desc(sa, p.row_bytes_a, a_box_bytes);
                    const uint64_t bdesc = make_mnmajor_desc(sa + a_bytes, p.row_bytes_b, b_box_bytes);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(i * p.n_tile);
                    for (int k = 0; k < p.rows / 16; ++k)   // 16 pixels per MMA: advance 16 rows in both operands
                        tc_mma_bf16(d_tmem, adesc + (uint64_t)((k * 16 * p.row_bytes_a) >> 4), bdesc + (uint64_t)((k * 16 * p.row_bytes_b) >> 4),
                                    idesc, (ch > ch0 || k > 0) ? 1u : 0u);
                    tc_commit(&empty_bar[stage]);
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
            tc_commit(done_bar);
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        mbar_wait(done_bar, 0);
        tc_fence_after();
        float* outp = p.out + (long long)slice * p.out_elems;
        const bool have = ch1 > ch0;
        // The accumulator arrives one ROW per lane; stored as is, a warp's 16-byte stores land 32 rows apart and
        // the large linear-layer gradients (205 MB) become request-bound.  Each warp therefore transposes 32 x 32
        // blocks through a private XOR-swizzled shared tile and writes four full 128-byte lines per instruction.
        float* s_t = s_tr + (warp - 2) * 1024;
        for (int i = 0; i < n_mt; ++i) {
            const int bi = (mt0 + i) * p.boxes_per_tile + m / p.CB;       // warp-uniform: 32 | CB
            const bool ok = bi < p.n_boxes;
            const long long row0 = ok ? (long long)p.box[bi].row0 + ((quarter * 32) % p.CB) : 0;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(i * p.n_tile);
            for (int c0 = 0; c0 < p.n_tile; c0 += 32) {
                uint32_t v[32];
                tmem_ld16(taddr + (uint32_t)c0, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
                tmem_ld16(taddr + (uint32_t)(c0 + 16), *reinterpret_cast<uint32_t(*)[16]>(&v[16]));
                tmem_ld_wait();
                if (!ok) continue;
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    *reinterpret_cast<float4*>(s_t + lane * 32 + ((c ^ (lane & 7)) << 2)) =
                        have ? make_float4(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1]), __uint_as_float(v[4 * c + 2]), __uint_as_float(v[4 * c + 3]))
                             : make_float4(0.f, 0.f, 0.f, 0.f);
                __syncwarp();
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const int rr = t * 4 + (lane >> 3), cc = lane & 7;
                    const float4 q = *reinterpret_cast<const float4*>(s_t + rr * 32 + ((cc ^ (rr & 7)) << 2));
                    *reinterpret_cast<float4*>(outp + (row0 + rr) * p.Cs + nt * p.n_tile + c0 + cc * 4) = q;
                }
                __syncwarp();
            }
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
// Halo variant for stride-1 layers with one channel chunk per tap (Cb = 32 or 64) and Cs = 32 or 64:
// the five largest weight gradients of the graph.  Instead of one TMA box per tap and pixel chunk
// (kh*kw re-reads of the input from L2, which bounds the generic kernel), the CTA loads the
// (BH + kh - 1) x (8 + kw - 1) input window of an 8-wide x BH-tall gradient tile ONCE.  The A operand
// of a tap is that window addressed through an MN-major descriptor that starts (r * pitch + s) pixel
// rows further: K group g (8 pixels of tile row 2k + g) sits SBO = one window row apart, and the
// M = 128 rows of one MMA are 128 / CB taps that are neighbours in s (LBO = one pixel) or in r
// (LBO = one window row).  Shared-memory swizzling is a function of the address alone, so shifted
// starts read exactly what TMA wrote.
constexpr int kMaxHTiles = 32;
struct HTile {
    short r0, s0, dir, nvalid;    // first tap, stacking direction (0: along s, 1: along r), taps that exist
};
struct WHaloParams {
    int m_tiles, tiles_per_group, groups;
    int CB, row_bytes_a, row_bytes_b, Cb, Cs;     // Cs = UMMA N (one N tile)
    int BH, pitch, halo_h, kw, pt, pl;
    int tiles_w, tiles_h, chunks, slices, chunks_per_slice, stages;
    int a_stage, b_stage;                          // bytes per stage (1024-aligned)
    long long out_elems;
    float* out;
    HTile tile[kMaxHTiles];
};

__global__ void __launch_bounds__(kThreads, 1) wgrad_halo_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                  const __grid_constant__ CUtensorMap map_b,
                                                                  const __grid_constant__ WHaloParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int stage_bytes = p.a_stage + p.b_stage;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes + 1024);   // 1 KB slack: absent taps of a ragged M tile
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* done_bar = empty_bar + p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int w = blockIdx.x;
    const int slice = w % p.slices; w /= p.slices;
    const int grp = w;
    const int mt0 = grp * p.tiles_per_group;
    const int n_mt = min(p.m_tiles, mt0 + p.tiles_per_group) - mt0;
    const int ch0 = slice * p.chunks_per_slice;
    const int ch1 = min(p.chunks, ch0 + p.chunks_per_slice);
    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(p.tiles_per_group * p.Cs)) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t tx = (uint32_t)(p.halo_h * p.pitch * p.row_bytes_a + p.BH * 8 * p.row_bytes_b);
            for (int ch = ch0; ch < ch1; ++ch) {
                int t = ch;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + (size_t)stage * stage_bytes;
                mbar_expect_tx(&full_bar[stage], tx);
                tma_load_5d(sa, &map_a, &full_bar[stage], 0, tw * 8 - p.pl, 0, th * p.BH - p.pt, t);
                tma_load_5d(sa + p.a_stage, &map_b, &full_bar[stage], 0, tw * 8, 0, th * p.BH, t);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.Cs >> 3) << 17) |
                                   ((128u >> 4) << 24);
            const uint32_t row_step = (uint32_t)(p.pitch * p.row_bytes_a);          // one window row
            // per M tile: descriptor bits that do not depend on the stage
            uint64_t a_hi[kMaxHTiles];
            uint32_t a_off[kMaxHTiles];
            for (int i = 0; i < n_mt; ++i) {
                const HTile& t = p.tile[mt0 + i];
                const uint32_t lbo = t.dir ? row_step : (uint32_t)p.row_bytes_a;
                uint64_t d = 0;
                d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
                d |= (uint64_t)((row_step >> 4) & 0x3FFF) << 32;                     // SBO: next tile row = next 8-pixel K group
                d |= (uint64_t)1 << 46;
                d |= (uint64_t)(p.row_bytes_a == 128 ? 2 : 4) << 61;
                a_hi[i] = d;
                a_off[i] = (uint32_t)((t.r0 * p.pitch + t.s0) * p.row_bytes_a);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = ch0; ch < ch1; ++ch) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                const uint64_t bdesc = make_mnmajor_desc(sa + p.a_stage, p.row_bytes_b, 1024);
                for (int i = 0; i < n_mt; ++i) {
                    const uint32_t d_tmem = tmem_base + (uint32_t)(i * p.Cs);
                    const uint32_t a0 = sa + a_off[i];
                    for (int k = 0; k < p.BH / 2; ++k) {    // 16 pixels per MMA = tile rows 2k, 2k + 1
                        const uint64_t adesc = a_hi[i] | (uint64_t)(((a0 + 2u * k * row_step) & 0x3FFFF) >> 4);
                        tc_mma_bf16(d_tmem, adesc, bdesc + (uint64_t)((k * 16 * p.row_bytes_b) >> 4), idesc, (ch > ch0 || k > 0) ? 1u : 0u);
                    }
                }
                tc_commit(&empty_bar[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            tc_commit(done_bar);
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        mbar_wait(done_bar, 0);
        tc_fence_after();
        float* outp = p.out + (long long)slice * p.out_elems;
        const bool have = ch1 > ch0;
        const int j = m / p.CB, c = m % p.CB;
        for (int i = 0; i < n_mt; ++i) {
            const HTile& t = p.tile[mt0 + i];
            const bool ok = j < t.nvalid;
            const int r = t.r0 + (t.dir ? j : 0), s2 = t.s0 + (t.dir ? 0 : j);
            const long long row = ok ? (long long)(r * p.kw + s2) * p.Cb + c : 0;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(i * p.Cs);
            for (int c0 = 0; c0 < p.Cs; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                if (ok) {
                    float* o = outp + row * p.Cs + c0;
#pragma unroll
                    for (int k = 0; k < 16; k += 4)
                        *reinterpret_cast<float4*>(o + k) =
                            have ? make_float4(__uint_as_float(v[k]), __uint_as_float(v[k + 1]), __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
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
// 2-D stacked halo variant for Cb = Cs = 32: taps are stacked along BOTH MMA dimensions.  With the virtual column
// u = ox + s,   dW[r, s] = sum_{oy, u} x[oy + r - pt, u - pl] * dy[oy, u - s],
// so for a tile of (oy, u) the A operand stacks up to four r (rows of the x window, LBO = one window row) along M and
// the B operand stacks all kw values of s (columns of a dy window with a (kw - 1)-pixel halo on the left, LBO = one
// pixel, in DEcreasing s) along N.  One MMA is M = 128 x N = 32 kw instead of M = 128 x N = 32: 3.5x fewer MMAs for a
// 5 x 5 layer, and the MN-major operand fetch (the bound of the 1-D form) is amortised over kw times the math.
struct WHalo2Params {
    int m_tiles;                  // ceil(kh / 4) accumulators of N = 32 * kw columns
    int kh, kw, pt, pl, BH, pitch_b;
    int tiles_w, tiles_h, chunks, slices, chunks_per_slice, stages;
    int a_stage, b_stage;
    long long out_elems;
    float* out;
};

__global__ void __launch_bounds__(kThreads, 1) wgrad_halo2d_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                    const __grid_constant__ CUtensorMap map_b,
                                                                    const __grid_constant__ WHalo2Params p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int stage_bytes = p.a_stage + p.b_stage;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes + 2048);   // slack: absent r taps of the last M tile
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* done_bar = empty_bar + p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slice = blockIdx.x;
    const int ch0 = slice * p.chunks_per_slice;
    const int ch1 = min(p.chunks, ch0 + p.chunks_per_slice);
    const int N = 32 * p.kw;
    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(p.m_tiles * N)) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t tx = (uint32_t)((p.BH + p.kh - 1) * 8 * 64 + p.BH * p.pitch_b * 64);
            for (int ch = ch0; ch < ch1; ++ch) {
                int t = ch;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + (size_t)stage * stage_bytes;
                mbar_expect_tx(&full_bar[stage], tx);
                tma_load_5d(sa, &map_a, &full_bar[stage], 0, tw * 8 - p.pl, 0, th * p.BH - p.pt, t);
                tma_load_5d(sa + p.a_stage, &map_b, &full_bar[stage], 0, tw * 8 - (p.kw - 1), 0, th * p.BH, t);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
            // A: spans = r (LBO one 8-pixel window row = 512 B), K groups = tile rows (SBO 512 B)
            uint64_t a_hi = 0;
            a_hi |= (uint64_t)(512u >> 4) << 16;
            a_hi |= (uint64_t)(512u >> 4) << 32;
            a_hi |= (uint64_t)1 << 46;
            a_hi |= (uint64_t)4 << 61;
            // B: spans = s descending (LBO one pixel = 64 B), K groups = window rows (SBO pitch_b pixels)
            const uint32_t b_row = (uint32_t)(p.pitch_b * 64);
            uint64_t b_hi = 0;
            b_hi |= (uint64_t)(64u >> 4) << 16;
            b_hi |= (uint64_t)((b_row >> 4) & 0x3FFF) << 32;
            b_hi |= (uint64_t)1 << 46;
            b_hi |= (uint64_t)4 << 61;
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = ch0; ch < ch1; ++ch) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                const uint32_t sb = sa + (uint32_t)p.a_stage;
                for (int i = 0; i < p.m_tiles; ++i) {
                    const uint32_t d_tmem = tmem_base + (uint32_t)(i * N);
                    for (int k = 0; k < p.BH / 2; ++k) {
                        const uint64_t adesc = a_hi | (uint64_t)(((sa + (uint32_t)(4 * i + 2 * k) * 512u) & 0x3FFFF) >> 4);
                        const uint64_t bdesc = b_hi | (uint64_t)(((sb + (uint32_t)(2 * k) * b_row) & 0x3FFFF) >> 4);
                        tc_mma_bf16(d_tmem, adesc, bdesc, idesc, (ch > ch0 || k > 0) ? 1u : 0u);
                    }
                }
                tc_commit(&empty_bar[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            tc_commit(done_bar);
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        mbar_wait(done_bar, 0);
        tc_fence_after();
        float* outp = p.out + (long long)slice * p.out_elems;
        const bool have = ch1 > ch0;
        const int j = m >> 5, ci = m & 31;
        for (int i = 0; i < p.m_tiles; ++i) {
            const int r = 4 * i + j;
            const bool ok = r < p.kh;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(i * N);
            for (int c0 = 0; c0 < N; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                if (ok) {
                    const int s2 = p.kw - 1 - (c0 >> 5);
                    float* o = outp + ((long long)(r * p.kw + s2) * 32 + ci) * 32 + (c0 & 31);
#pragma unroll
                    for (int k = 0; k < 16; k += 4)
                        *reinterpret_cast<float4*>(o + k) =
                            have ? make_float4(__uint_as_float(v[k]), __uint_as_float(v[k + 1]), __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
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
// Stride-2 layers whose shifted tensor has 32 channels (e1, e2, d1, d2): the same 2-D stacking on the PARITY VIEW
// [N][H/2][2][W/2][2C] of the big tensor.  A stride-2 tap (r, s) is plane ph = (r - pt) mod 2 at row shift
// dh = floor((r - pt) / 2), and column shift dw = floor((s - pl) / 2) with the column parity pw choosing one half of
// the 2C = 64 channels of a window row.  With the virtual column u = ox + dw,
//     dW[r, s] = sum_{oy, u} X_ph[oy + dh, u, (pw, ci)] * dy[oy, u - dw],
// so an M tile stacks two dh of one plane (2 x 64 rows, LBO = one window row) and N stacks every dw (columns of a
// dy window with a halo on the left, LBO = one pixel).  Entries whose s = 2 dw + pw + pl falls outside the kernel
// are structural zeros and are not stored.
struct WS2Tile {
    short ph, dh0, nvalid, pad;
};
struct WS2Params {
    int kh, kw, pt, pl, BH, pitch_b, ndw, dw_lo, dw_hi;
    int Cs, row_bytes_b;                     // small tensor channels (32 | 64) = one MMA N span
    int m_tiles, tiles_per_group, groups;
    int dhlo[2], halo_h;                     // first row shift of each plane's window; window height (common)
    int tiles_w, tiles_h, chunks, slices, chunks_per_slice, stages;
    int plane_bytes, b_stage;                // 1024-aligned slot sizes
    long long out_elems;
    float* out;
    WS2Tile tile[8];
};

__global__ void __launch_bounds__(kThreads, 1) wgrad_s2_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                const __grid_constant__ CUtensorMap map_b,
                                                                const __grid_constant__ WS2Params p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int stage_bytes = 2 * p.plane_bytes + p.b_stage;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes + 2048);
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* done_bar = empty_bar + p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slice = blockIdx.x % p.slices, grp = blockIdx.x / p.slices;
    const int mt0 = grp * p.tiles_per_group;
    const int n_mt = min(p.m_tiles, mt0 + p.tiles_per_group) - mt0;
    const int ch0 = slice * p.chunks_per_slice;
    const int ch1 = min(p.chunks, ch0 + p.chunks_per_slice);
    const int N = p.Cs * p.ndw;
    int plane_mask = 0;
    for (int i = 0; i < n_mt; ++i) plane_mask |= 1 << p.tile[mt0 + i].ph;
    uint32_t tmem_cols = 32;
    while (tmem_cols < (uint32_t)(p.tiles_per_group * N)) tmem_cols <<= 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(done_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t a_real = (uint32_t)(p.halo_h * 8 * 128);
            const uint32_t tx = a_real * (uint32_t)__popc(plane_mask) + (uint32_t)(p.BH * p.pitch_b * p.row_bytes_b);
            for (int ch = ch0; ch < ch1; ++ch) {
                int t = ch;
                const int tw = t % p.tiles_w; t /= p.tiles_w;
                const int th = t % p.tiles_h; t /= p.tiles_h;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + (size_t)stage * stage_bytes;
                mbar_expect_tx(&full_bar[stage], tx);
                for (int ph = 0; ph < 2; ++ph)
                    if (plane_mask & (1 << ph))
                        tma_load_5d(sa + ph * p.plane_bytes, &map_a, &full_bar[stage], 0, tw * 8 + p.dw_lo, ph, th * p.BH + p.dhlo[ph], t);
                tma_load_5d(sa + 2 * p.plane_bytes, &map_b, &full_bar[stage], 0, tw * 8 - (p.ndw - 1), 0, th * p.BH, t);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
            // A: 128-byte rows (SWIZZLE_128B); spans = dh (LBO one 8-pixel window row = 1024 B), K groups = tile rows (SBO 1024 B)
            uint64_t a_hi = 0;
            a_hi |= (uint64_t)(1024u >> 4) << 16;
            a_hi |= (uint64_t)(1024u >> 4) << 32;
            a_hi |= (uint64_t)1 << 46;
            a_hi |= (uint64_t)2 << 61;
            // B: spans = dw descending (LBO one pixel), K groups = window rows (SBO pitch_b pixels)
            const uint32_t b_row = (uint32_t)(p.pitch_b * p.row_bytes_b);
            uint64_t b_hi = 0;
            b_hi |= (uint64_t)(((uint32_t)p.row_bytes_b >> 4) & 0x3FFF) << 16;
            b_hi |= (uint64_t)((b_row >> 4) & 0x3FFF) << 32;
            b_hi |= (uint64_t)1 << 46;
            b_hi |= (uint64_t)(p.row_bytes_b == 128 ? 2 : 4) << 61;
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = ch0; ch < ch1; ++ch) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                const uint32_t sb = sa + 2u * (uint32_t)p.plane_bytes;
                for (int i = 0; i < n_mt; ++i) {
                    const WS2Tile& t = p.tile[mt0 + i];
                    const uint32_t d_tmem = tmem_base + (uint32_t)(i * N);
                    const uint32_t a0 = sa + (uint32_t)(t.ph * p.plane_bytes) + (uint32_t)(t.dh0 - p.dhlo[t.ph]) * 1024u;
                    for (int k = 0; k < p.BH / 2; ++k) {
                        const uint64_t adesc = a_hi | (uint64_t)(((a0 + (uint32_t)(2 * k) * 1024u) & 0x3FFFF) >> 4);
                        const uint64_t bdesc = b_hi | (uint64_t)(((sb + (uint32_t)(2 * k) * b_row) & 0x3FFFF) >> 4);
                        tc_mma_bf16(d_tmem, adesc, bdesc, idesc, (ch > ch0 || k > 0) ? 1u : 0u);
                    }
                }
                tc_commit(&empty_bar[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            tc_commit(done_bar);
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;
        mbar_wait(done_bar, 0);
        tc_fence_after();
        float* outp = p.out + (long long)slice * p.out_elems;
        const bool have = ch1 > ch0;
        const int j = m >> 6, pw = (m >> 5) & 1, ci = m & 31;
        for (int i = 0; i < n_mt; ++i) {
            const WS2Tile& t = p.tile[mt0 + i];
            const int r = 2 * (t.dh0 + j) + t.ph + p.pt;
            const bool row_ok = (j < t.nvalid) && r >= 0 && r < p.kh;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(i * N);
            for (int c0 = 0; c0 < N; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                const int jj = c0 / p.Cs, co = c0 - jj * p.Cs;
                const int s2 = 2 * (p.dw_hi - jj) + pw + p.pl;
                if (row_ok && s2 >= 0 && s2 < p.kw) {
                    float* o = outp + ((long long)(r * p.kw + s2) * 32 + ci) * p.Cs + co;
#pragma unroll
                    for (int k = 0; k < 16; k += 4)
                        *reinterpret_cast<float4*>(o + k) =
                            have ? make_float4(__uint_as_float(v[k]), __uint_as_float(v[k + 1]), __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// pixel chunk box: rows = BW*BH*NB a multiple of 16, <= max_rows, maximising the useful fraction
void choose_chunk(int Jh, int Jw, int N, int max_rows, int& BW, int& BH, int& NB) {
    double best = -1.0;
    BW = 16; BH = 1; NB = 1;
    const int wmax = Jw + 15;
    for (int bw = 1; bw <= wmax && bw <= max_rows; ++bw)
        for (int bh = 1; bh <= Jh + 15 && bw * bh <= max_rows; ++bh) {
            int nb = 1;
            if (bw >= Jw && bh >= Jh) nb = max_rows / (bw * bh);
            if (nb > N) nb = N;
            if (nb < 1) nb = 1;
            const int rows = bw * bh * nb;
            if (rows % 16) continue;
            const long long chunks = (long long)ceil_div(Jw, bw) * ceil_div(Jh, bh) * ceil_div(N, nb);
            const double eff = (double)Jh * Jw * N / ((double)chunks * rows);
            // on ties prefer more rows per chunk (fewer pipeline steps), then wider boxes
            if (eff > best + 1e-9 || (eff > best - 1e-9 && (rows > BW * BH * NB || (rows == BW * BH * NB && bw > BW)))) {
                best = eff; BW = bw; BH = bh; NB = nb;
            }
        }
}

struct WProblem {
    const void* big; int N, Hb, Wb, Cb, stride;      // tensor read through tap shifts (conv: x; deconv: dy)
    const void* small; int Hs, Ws, Cs;               // tensor read unshifted (conv: dy; deconv: x)
    int kh, kw, pt, pl;
    float* dw;                                       // [kh*kw][Cb][Cs] fp32
};

size_t plan_wgrad(const WProblem& q, WgradParams& p) {
    memset(&p, 0, sizeof(p));
    p.CB = (q.Cb % 64 == 0) ? 64 : 32;
    p.row_bytes_a = p.CB * 2;
    p.CBs = (q.Cs % 64 == 0) ? 64 : 32;
    p.row_bytes_b = p.CBs * 2;
    p.Cs = q.Cs;
    p.n_tile = q.Cs > 256 ? 256 : q.Cs;
    p.n_tiles = ceil_div(q.Cs, p.n_tile);
    p.b_boxes = p.n_tile / p.CBs;
    const int chunks_c = q.Cb / p.CB;
    p.n_boxes = q.kh * q.kw * chunks_c;
    p.boxes_per_tile = 128 / p.CB;
    p.m_tiles = ceil_div(p.n_boxes, p.boxes_per_tile);
    p.tiles_per_group = 512 / p.n_tile;
    if (p.tiles_per_group > p.m_tiles) p.tiles_per_group = p.m_tiles;
    p.groups = ceil_div(p.m_tiles, p.tiles_per_group);
    const int max_rows = (p.n_tile >= 128) ? 64 : 128;
    choose_chunk(q.Hs, q.Ws, q.N, max_rows, p.BW, p.BH, p.NB);
    p.rows = p.BW * p.BH * p.NB;
    p.tiles_w = ceil_div(q.Ws, p.BW);
    p.tiles_h = ceil_div(q.Hs, p.BH);
    p.img_groups = ceil_div(q.N, p.NB);
    p.chunks = p.tiles_w * p.tiles_h * p.img_groups;
    const int base_ctas = p.groups * p.n_tiles;
    int slices = ceil_div(num_sms(), base_ctas);
    if (slices > p.chunks) slices = p.chunks;
    if (slices < 1) slices = 1;
    p.chunks_per_slice = ceil_div(p.chunks, slices);
    p.slices = ceil_div(p.chunks, p.chunks_per_slice);
    p.out_elems = (long long)q.kh * q.kw * q.Cb * q.Cs;
    return p.slices > 1 ? (size_t)p.slices * p.out_elems * sizeof(float) : 0;
}

bool wgrad_eligible(int Cb, int Cs, int taps) {
    if (Cb % 32 || Cs % 32) return false;
    const int CB = (Cb % 64 == 0) ? 64 : 32;
    if (taps * (Cb / CB) > kMaxBoxes) return false;
    if (Cs > 256 && Cs % 256) return false;
    return true;
}


// ---- halo variant: planning and launch
bool whalo_eligible(const WProblem& q) {
    if (getenv("DMV_NO_WHALO")) return false;
    if (q.stride != 1 || q.kh * q.kw == 1) return false;
    if (!(q.Cb == 32 || q.Cb == 64) || !(q.Cs == 32 || q.Cs == 64)) return false;
    if (q.Hs != q.Hb || q.Ws != q.Wb) return false;          // stride-1 SAME: gradient and input share the resolution
    if (q.Hs * q.Ws < 256 || q.kw > 8 || q.kh > 8) return false;
    return true;
}

int plan_whalo(const WProblem& q, WHaloParams& p) {
    memset(&p, 0, sizeof(p));
    p.CB = q.Cb; p.Cb = q.Cb; p.Cs = q.Cs;
    p.row_bytes_a = q.Cb * 2; p.row_bytes_b = q.Cs * 2;
    p.kw = q.kw; p.pt = q.pt; p.pl = q.pl;
    // tile height: an even number of rows <= 16 that wastes the fewest rows of the image
    int best_bh = 16; double best = -1.0;
    for (int bh = 16; bh >= 8; bh -= 2) {
        const double eff = (double)q.Hs / (ceil_div(q.Hs, bh) * bh);
        if (eff > best + 1e-9) { best = eff; best_bh = bh; }
    }
    p.BH = best_bh;
    p.pitch = 8 + q.kw - 1;
    p.halo_h = p.BH + q.kh - 1;
    p.tiles_w = ceil_div(q.Ws, 8);
    p.tiles_h = ceil_div(q.Hs, p.BH);
    p.chunks = p.tiles_w * p.tiles_h * q.N;
    // M tiles: 128 / CB taps each; rows of taps first (stacked along s), the leftover column stacked along r,
    // any ragged remainder again along s so that absent taps only read a few pixels past the window
    const int spt = 128 / p.CB;
    int n = 0;
    const int full = q.kw / spt, rem = q.kw % spt;
    for (int r = 0; r < q.kh; ++r)
        for (int f = 0; f < full; ++f) p.tile[n++] = HTile{(short)r, (short)(f * spt), 0, (short)spt};
    if (rem) {
        if (rem == 1) {                       // one leftover tap per row: stack rows
            int r = 0;
            for (; r + spt <= q.kh; r += spt) p.tile[n++] = HTile{(short)r, (short)(q.kw - 1), 1, (short)spt};
            for (; r < q.kh; ++r) p.tile[n++] = HTile{(short)r, (short)(q.kw - 1), 0, 1};
        } else {
            for (int r = 0; r < q.kh; ++r) p.tile[n++] = HTile{(short)r, (short)(full * spt), 0, (short)rem};
        }
    }
    if (n > kMaxHTiles) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad halo: too many M tiles");
    p.m_tiles = n;
    p.tiles_per_group = 512 / p.Cs;
    if (p.tiles_per_group > n) p.tiles_per_group = n;
    p.groups = ceil_div(n, p.tiles_per_group);
    p.tiles_per_group = ceil_div(n, p.groups);               // balance the groups
    int slices = ceil_div(num_sms(), p.groups);
    if (slices > p.chunks) slices = p.chunks;
    p.chunks_per_slice = ceil_div(p.chunks, slices);
    p.slices = ceil_div(p.chunks, p.chunks_per_slice);
    p.out_elems = (long long)q.kh * q.kw * q.Cb * q.Cs;
    p.a_stage = (p.halo_h * p.pitch * p.row_bytes_a + 1023) & ~1023;
    p.b_stage = (p.BH * 8 * p.row_bytes_b + 1023) & ~1023;
    return DMV_OK;
}

int run_wgrad_halo(const WProblem& q, void* ws, size_t ws_bytes, cudaStream_t st) {
    WHaloParams p;
    int rc = plan_whalo(q, p);
    if (rc) return rc;
    const size_t need = p.slices > 1 ? (size_t)p.slices * p.out_elems * sizeof(float) : 0;
    if (need > 0 && (!ws || ws_bytes < need)) return fail(DMV_E_WORKSPACE, "tc wgrad halo: workspace too small");
    p.out = p.slices > 1 ? reinterpret_cast<float*>(ws) : q.dw;
    CUtensorMap map_a, map_b;
    {
        cuuint64_t dims[5] = {(cuuint64_t)q.Cb, (cuuint64_t)q.Wb, 1, (cuuint64_t)q.Hb, (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cb * 2;
        cuuint64_t strides[4] = {pix, (cuuint64_t)q.Wb * pix, (cuuint64_t)q.Wb * pix, (cuuint64_t)q.Hb * q.Wb * pix};
        cuuint32_t box[5] = {(cuuint32_t)q.Cb, (cuuint32_t)p.pitch, 1u, (cuuint32_t)p.halo_h, 1u};
        rc = encode_map(&map_a, q.big, 5, dims, strides, box, p.row_bytes_a);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[5] = {(cuuint64_t)q.Cs, (cuuint64_t)q.Ws, 1, (cuuint64_t)q.Hs, (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cs * 2;
        cuuint64_t strides[4] = {pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Hs * q.Ws * pix};
        cuuint32_t box[5] = {(cuuint32_t)q.Cs, 8u, 1u, (cuuint32_t)p.BH, 1u};
        rc = encode_map(&map_b, q.small, 5, dims, strides, box, p.row_bytes_b);
        if (rc) return rc;
    }
    const int stage_bytes = p.a_stage + p.b_stage;
    int stages = (200 * 1024) / stage_bytes;
    if (stages > 8) stages = 8;
    if (stages < 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad halo: stage does not fit shared memory");
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + 1024 + (2 * stages + 1) * sizeof(uint64_t) + 16 + 1024;
    cudaError_t e = cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        set_error("tc wgrad halo: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    wgrad_halo_kernel<<<p.groups * p.slices, kThreads, smem, st>>>(map_a, map_b, p);
    count_tc_launch();
    rc = check_launch("wgrad_halo_tc");
    if (rc) return rc;
    if (p.slices > 1) rc = reduce_partials(reinterpret_cast<const float*>(ws), q.dw, p.out_elems, p.slices, st);
    return rc;
}

// ---- 2-D stacked halo variant (Cb = Cs = 32)
bool whalo2d_eligible(const WProblem& q) {
    if (getenv("DMV_NO_WHALO2D")) return false;
    if (!whalo_eligible(q)) return false;
    if (q.Cb != 32 || q.Cs != 32) return false;
    return ceil_div(q.kh, 4) * 32 * q.kw <= 512 && 32 * q.kw <= 256;
}

int run_wgrad_halo2d(const WProblem& q, void* ws, size_t ws_bytes, cudaStream_t st) {
    WHalo2Params p;
    memset(&p, 0, sizeof(p));
    p.kh = q.kh; p.kw = q.kw; p.pt = q.pt; p.pl = q.pl;
    p.m_tiles = ceil_div(q.kh, 4);
    int best_bh = 16; double best = -1.0;
    for (int bh = 16; bh >= 8; bh -= 2) {
        const double eff = (double)q.Hs / (ceil_div(q.Hs, bh) * bh);
        if (eff > best + 1e-9) { best = eff; best_bh = bh; }
    }
    p.BH = best_bh;
    p.pitch_b = 8 + q.kw - 1;
    p.tiles_w = ceil_div(q.Ws + q.kw - 1, 8);          // virtual columns u = ox + s
    p.tiles_h = ceil_div(q.Hs, p.BH);
    p.chunks = p.tiles_w * p.tiles_h * q.N;
    int slices = num_sms();
    if (slices > p.chunks) slices = p.chunks;
    p.chunks_per_slice = ceil_div(p.chunks, slices);
    p.slices = ceil_div(p.chunks, p.chunks_per_slice);
    p.out_elems = (long long)q.kh * q.kw * 32 * 32;
    p.a_stage = ((p.BH + q.kh - 1) * 8 * 64 + 1023) & ~1023;
    p.b_stage = (p.BH * p.pitch_b * 64 + 1023) & ~1023;
    const size_t need = p.slices > 1 ? (size_t)p.slices * p.out_elems * sizeof(float) : 0;
    if (need > 0 && (!ws || ws_bytes < need)) return fail(DMV_E_WORKSPACE, "tc wgrad halo2d: workspace too small");
    p.out = p.slices > 1 ? reinterpret_cast<float*>(ws) : q.dw;
    CUtensorMap map_a, map_b;
    int rc;
    {
        cuuint64_t dims[5] = {32, (cuuint64_t)q.Wb, 1, (cuuint64_t)q.Hb, (cuuint64_t)q.N};
        cuuint64_t strides[4] = {64, (cuuint64_t)q.Wb * 64, (cuuint64_t)q.Wb * 64, (cuuint64_t)q.Hb * q.Wb * 64};
        cuuint32_t box[5] = {32u, 8u, 1u, (cuuint32_t)(p.BH + q.kh - 1), 1u};
        rc = encode_map(&map_a, q.big, 5, dims, strides, box, 64);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[5] = {32, (cuuint64_t)q.Ws, 1, (cuuint64_t)q.Hs, (cuuint64_t)q.N};
        cuuint64_t strides[4] = {64, (cuuint64_t)q.Ws * 64, (cuuint64_t)q.Ws * 64, (cuuint64_t)q.Hs * q.Ws * 64};
        cuuint32_t box[5] = {32u, (cuuint32_t)p.pitch_b, 1u, (cuuint32_t)p.BH, 1u};
        rc = encode_map(&map_b, q.small, 5, dims, strides, box, 64);
        if (rc) return rc;
    }
    const int stage_bytes = p.a_stage + p.b_stage;
    int stages = (200 * 1024) / stage_bytes;
    if (stages > 8) stages = 8;
    if (stages < 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad halo2d: stage does not fit shared memory");
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + 2048 + (2 * stages + 1) * sizeof(uint64_t) + 16 + 1024;
    cudaError_t e = cudaFuncSetAttribute(wgrad_halo2d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        set_error("tc wgrad halo2d: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    wgrad_halo2d_kernel<<<p.slices, kThreads, smem, st>>>(map_a, map_b, p);
    count_tc_launch();
    rc = check_launch("wgrad_halo2d_tc");
    if (rc) return rc;
    if (p.slices > 1) rc = reduce_partials(reinterpret_cast<const float*>(ws), q.dw, p.out_elems, p.slices, st);
    return rc;
}

// ---- stride-2, 32-channel big tensor: 2-D stacking on the parity view
static int wfdiv2(int a) { return a >= 0 ? a / 2 : -((-a + 1) / 2); }

bool ws2_eligible(const WProblem& q) {
    if (getenv("DMV_NO_WS2")) return false;
    if (q.stride != 2 || q.Cb != 32 || !(q.Cs == 32 || q.Cs == 64)) return false;
    if ((q.Hb & 1) || (q.Wb & 1) || q.Hs * 2 != q.Hb || q.Ws * 2 != q.Wb) return false;
    if (q.Hs * q.Ws < 256 || q.kh > 5 || q.kw > 5) return false;
    const int ndw = wfdiv2(q.kw - 1 - q.pl) - wfdiv2(-q.pl) + 1;
    return q.Cs * ndw <= 256;
}

int run_wgrad_s2(const WProblem& q, void* ws, size_t ws_bytes, cudaStream_t st) {
    WS2Params p;
    memset(&p, 0, sizeof(p));
    p.kh = q.kh; p.kw = q.kw; p.pt = q.pt; p.pl = q.pl;
    p.Cs = q.Cs; p.row_bytes_b = q.Cs * 2;
    p.dw_lo = wfdiv2(-q.pl); p.dw_hi = wfdiv2(q.kw - 1 - q.pl); p.ndw = p.dw_hi - p.dw_lo + 1;
    int span = 0, n = 0;
    for (int ph = 0; ph < 2; ++ph) {
        // dh values of the rows r with (r - pt) mod 2 == ph
        int lo = 1 << 20, hi = -(1 << 20);
        for (int r = 0; r < q.kh; ++r) {
            const int dy = r - q.pt;
            if ((((dy % 2) + 2) % 2) != ph) continue;
            const int dh = (dy - ph) / 2;
            lo = dh < lo ? dh : lo; hi = dh > hi ? dh : hi;
        }
        if (lo > hi) { p.dhlo[ph] = 0; continue; }
        p.dhlo[ph] = lo;
        span = (hi - lo) > span ? (hi - lo) : span;
        for (int dh = lo; dh <= hi; dh += 2) p.tile[n++] = WS2Tile{(short)ph, (short)dh, (short)((dh + 1 <= hi) ? 2 : 1), 0};
    }
    p.m_tiles = n;
    const int N = p.Cs * p.ndw;
    p.tiles_per_group = 512 / N;
    if (p.tiles_per_group > n) p.tiles_per_group = n;
    p.groups = ceil_div(n, p.tiles_per_group);
    int best_bh = 16; double best = -1.0;
    for (int bh = 16; bh >= 8; bh -= 2) {
        const double eff = (double)q.Hs / (ceil_div(q.Hs, bh) * bh);
        if (eff > best + 1e-9) { best = eff; best_bh = bh; }
    }
    p.BH = best_bh;
    p.halo_h = p.BH + span + 1;                      // + 1: the absent second dh of a ragged M tile stays inside the slot
    p.pitch_b = 8 + p.ndw - 1;
    p.tiles_w = ceil_div(q.Ws + p.ndw - 1, 8);
    p.tiles_h = ceil_div(q.Hs, p.BH);
    p.chunks = p.tiles_w * p.tiles_h * q.N;
    int slices = ceil_div(num_sms(), p.groups);
    if (slices > p.chunks) slices = p.chunks;
    p.chunks_per_slice = ceil_div(p.chunks, slices);
    p.slices = ceil_div(p.chunks, p.chunks_per_slice);
    p.out_elems = (long long)q.kh * q.kw * 32 * q.Cs;
    p.plane_bytes = (p.halo_h * 8 * 128 + 1023) & ~1023;
    p.b_stage = (p.BH * p.pitch_b * p.row_bytes_b + 1023) & ~1023;
    const size_t need = p.slices > 1 ? (size_t)p.slices * p.out_elems * sizeof(float) : 0;
    if (need > 0 && (!ws || ws_bytes < need)) return fail(DMV_E_WORKSPACE, "tc wgrad s2: workspace too small");
    p.out = p.slices > 1 ? reinterpret_cast<float*>(ws) : q.dw;
    CUtensorMap map_a, map_b;
    int rc;
    {
        cuuint64_t dims[5] = {64, (cuuint64_t)q.Ws, 2, (cuuint64_t)q.Hs, (cuuint64_t)q.N};
        cuuint64_t strides[4] = {128, (cuuint64_t)q.Wb * 64, (cuuint64_t)q.Wb * 128, (cuuint64_t)q.Hb * q.Wb * 64};
        cuuint32_t box[5] = {64u, 8u, 1u, (cuuint32_t)p.halo_h, 1u};
        rc = encode_map(&map_a, q.big, 5, dims, strides, box, 128);
        if (rc) return rc;
    }
    {
        const cuuint64_t pix = (cuuint64_t)q.Cs * 2;
        cuuint64_t dims[5] = {(cuuint64_t)q.Cs, (cuuint64_t)q.Ws, 1, (cuuint64_t)q.Hs, (cuuint64_t)q.N};
        cuuint64_t strides[4] = {pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Hs * q.Ws * pix};
        cuuint32_t box[5] = {(cuuint32_t)q.Cs, (cuuint32_t)p.pitch_b, 1u, (cuuint32_t)p.BH, 1u};
        rc = encode_map(&map_b, q.small, 5, dims, strides, box, p.row_bytes_b);
        if (rc) return rc;
    }
    const int stage_bytes = 2 * p.plane_bytes + p.b_stage;
    int stages = (200 * 1024) / stage_bytes;
    if (stages > 6) stages = 6;
    if (stages < 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad s2: stage does not fit shared memory");
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + 2048 + (2 * stages + 1) * sizeof(uint64_t) + 16 + 1024;
    cudaError_t e = cudaFuncSetAttribute(wgrad_s2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        set_error("tc wgrad s2: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    wgrad_s2_kernel<<<p.groups * p.slices, kThreads, smem, st>>>(map_a, map_b, p);
    count_tc_launch();
    rc = check_launch("wgrad_s2_tc");
    if (rc) return rc;
    if (p.slices > 1) rc = reduce_partials(reinterpret_cast<const float*>(ws), q.dw, p.out_elems, p.slices, st);
    return rc;
}

int run_wgrad(const WProblem& q, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (ws2_eligible(q)) return run_wgrad_s2(q, ws, ws_bytes, st);
    if (whalo2d_eligible(q)) return run_wgrad_halo2d(q, ws, ws_bytes, st);
    if (whalo_eligible(q)) return run_wgrad_halo(q, ws, ws_bytes, st);
    if (!wgrad_eligible(q.Cb, q.Cs, q.kh * q.kw)) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad: channel counts not covered");
    if (q.stride != 1 && q.stride != 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad: stride");
    if (q.stride == 2 && ((q.Hb & 1) || (q.Wb & 1))) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad: stride-2 source needs even H and W");
    if (((uintptr_t)q.big & 15) || ((uintptr_t)q.small & 15) || ((uintptr_t)q.dw & 15))
        return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad: buffers must be 16-byte aligned");
    WgradParams p;
    const size_t need = plan_wgrad(q, p);
    if (need > 0 && (!ws || ws_bytes < need)) return fail(DMV_E_WORKSPACE, "tc wgrad: workspace too small");
    p.out = p.slices > 1 ? reinterpret_cast<float*>(ws) : q.dw;
    // A boxes: (tap, channel chunk)
    const int chunks_c = q.Cb / p.CB;
    int n = 0;
    for (int r = 0; r < q.kh; ++r)
        for (int s = 0; s < q.kw; ++s)
            for (int c = 0; c < chunks_c; ++c) {
                ABox& b = p.box[n++];
                const int dy = r - q.pt, dx = s - q.pl;
                int ph = 0, pw = 0, dh = dy, dwv = dx;
                if (q.stride == 2) {
                    ph = ((dy % 2) + 2) % 2; dh = (dy - ph) / 2;
                    pw = ((dx % 2) + 2) % 2; dwv = (dx - pw) / 2;
                }
                b.dh = (short)dh; b.dw = (short)dwv; b.ph = (short)ph; b.c_off = (short)(pw * q.Cb + c * p.CB);
                b.row0 = (r * q.kw + s) * q.Cb + c * p.CB;
            }
    CUtensorMap map_a, map_b;
    {
        const int s = q.stride;
        cuuint64_t dims[5] = {(cuuint64_t)(s * q.Cb), (cuuint64_t)(q.Wb / s), (cuuint64_t)s, (cuuint64_t)(q.Hb / s), (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cb * 2;
        cuuint64_t strides[4] = {(cuuint64_t)s * pix, (cuuint64_t)q.Wb * pix, (cuuint64_t)s * q.Wb * pix, (cuuint64_t)q.Hb * q.Wb * pix};
        cuuint32_t box[5] = {(cuuint32_t)p.CB, (cuuint32_t)p.BW, 1u, (cuuint32_t)p.BH, (cuuint32_t)p.NB};
        int rc = encode_map(&map_a, q.big, 5, dims, strides, box, p.row_bytes_a);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[5] = {(cuuint64_t)q.Cs, (cuuint64_t)q.Ws, 1, (cuuint64_t)q.Hs, (cuuint64_t)q.N};
        const cuuint64_t pix = (cuuint64_t)q.Cs * 2;
        cuuint64_t strides[4] = {pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Ws * pix, (cuuint64_t)q.Hs * q.Ws * pix};
        cuuint32_t box[5] = {(cuuint32_t)p.CBs, (cuuint32_t)p.BW, 1u, (cuuint32_t)p.BH, (cuuint32_t)p.NB};
        int rc = encode_map(&map_b, q.small, 5, dims, strides, box, p.row_bytes_b);
        if (rc) return rc;
    }
    const int stage_bytes = p.boxes_per_tile * p.rows * p.row_bytes_a + p.b_boxes * p.rows * p.row_bytes_b;
    int stages = (176 * 1024) / stage_bytes;
    if (stages > 6) stages = 6;
    if (stages < 2) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc wgrad: stage does not fit shared memory");
    p.stages = stages;
    // stages | 1 KB of barriers | 16 KB of epilogue transpose tiles | alignment slack
    const size_t smem = (size_t)stages * stage_bytes + 1024 + 4 * 4096 + 1024;
    cudaError_t e = cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        set_error("tc wgrad: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return DMV_E_CUDA;
    }
    const int grid = p.groups * p.n_tiles * p.slices;
    wgrad_kernel<<<grid, kThreads, smem, st>>>(map_a, map_b, p);
    count_tc_launch();
    int rc = check_launch("wgrad_tc");
    if (rc) return rc;
    if (p.slices > 1) {
        rc = reduce_partials(reinterpret_cast<const float*>(ws), q.dw, p.out_elems, p.slices, st);
    }
    return rc;
}

}  // namespace

namespace dmv {

size_t tc_wgrad_workspace(int taps, int Cin, int Cout, int N, int Hs, int Ws) {
    // one fp32 copy of dW per pixel slice (none when a single slice writes dW directly).  The estimate from the pixel
    // count also covers the halo variants; the generic kernel's own plan is added because its ragged chunk boxes can
    // outnumber pixels / 16 (e.g. a 15 x 17 gradient image).
    if (!wgrad_eligible(Cin, Cout, taps) || N <= 0 || Hs <= 0 || Ws <= 0) return 0;
    const int CB = (Cin % 64 == 0) ? 64 : 32;
    const int n_tile = Cout > 256 ? 256 : Cout;
    const int n_tiles = ceil_div(Cout, n_tile);
    const int m_tiles = ceil_div(taps * (Cin / CB), 128 / CB);
    int tpg = 512 / n_tile;
    if (tpg > m_tiles) tpg = m_tiles;
    const int base = ceil_div(m_tiles, tpg) * n_tiles;
    long long slices = ceil_div(num_sms(), base);
    const long long max_chunks = ceil_div_ll((long long)N * Hs * Ws, 16);
    if (slices > max_chunks) slices = max_chunks;
    size_t need = slices > 1 ? (size_t)slices * (size_t)taps * Cin * Cout * sizeof(float) : 0;
    WProblem q;
    memset(&q, 0, sizeof(q));
    q.N = N; q.Hs = Hs; q.Ws = Ws; q.Cb = Cin; q.Cs = Cout; q.kh = taps; q.kw = 1;
    WgradParams p;
    const size_t plan = plan_wgrad(q, p);
    if (plan > need) need = plan;
    return need ? need + 256 : 0;
}

int tc_conv_wgrad(const void* x, int xdt, const void* dy, float* dw, float* db, int B, int H, int W, int Cin, int Cout, int kh, int kw,
                  int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (xdt != DMV_DT_BF16) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_conv_wgrad: bf16 input only");
    if (db) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_conv_wgrad: bias gradient is taken by the caller");
    const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
    WProblem q;
    q.big = x; q.N = B; q.Hb = H; q.Wb = W; q.Cb = Cin; q.stride = stride;
    q.small = dy; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cout;
    q.kh = kh; q.kw = kw; q.pt = ph.before; q.pl = pw.before; q.dw = dw;
    return run_wgrad(q, ws, ws_bytes, st);
}

int tc_deconv_wgrad(const void* x, const void* dy, int dydt, float* dw, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                    int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (dydt != DMV_DT_BF16) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_deconv_wgrad: bf16 gradient only");
    const SamePad ph = same_pad(Hout, kh, stride), pw = same_pad(Wout, kw, stride);
    WProblem q;
    q.big = dy; q.N = B; q.Hb = Hout; q.Wb = Wout; q.Cb = Cout; q.stride = stride;
    q.small = x; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cin;
    q.kh = kh; q.kw = kw; q.pt = ph.before; q.pl = pw.before; q.dw = dw;
    return run_wgrad(q, ws, ws_bytes, st);
}

int tc_linear_wgrad(const void* x, const void* dy, float* dw, float* db, int M, int K, int N, void* ws, size_t ws_bytes,
                    cudaStream_t st) {
    if (db) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_linear_wgrad: bias gradient is taken by the caller");
    WProblem q;
    q.big = x; q.N = M; q.Hb = 1; q.Wb = 1; q.Cb = K; q.stride = 1;
    q.small = dy; q.Hs = 1; q.Ws = 1; q.Cs = N;
    q.kh = 1; q.kw = 1; q.pt = 0; q.pl = 0; q.dw = dw;
    return run_wgrad(q, ws, ws_bytes, st);
}


int tc_thin_wgrad(const void* thin, int thin_dtype, const void* wide, float* dw, int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw,
                  int stride, void* ws, size_t ws_bytes, cudaStream_t st) {
    const SamePad ph = same_pad(Hb, kh, stride), pw = same_pad(Wb, kw, stride);
    const int rows = kh * kw * Ct, Kp = thin_patch_cols(kh * kw, Ct);
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    if (thin_dtype == DMV_DT_S2D && !thin_s2d_eligible(Hb, Wb, Ct, Cw, kh, kw, stride))
        return fail(DMV_E_INVALID_ARG, "DMV_DT_S2D input for a layer that does not take the space-to-depth path");
    if (thin_s2d_eligible(Hb, Wb, Ct, Cw, kh, kw, stride)) {
        // space-to-depth: stride-1 weight gradient over X2 (halo kernel), then the (shift, block) entries are gathered into dW
        const S2dGeom g2 = thin_s2d_geom(Hb, Wb, kh, kw);
        const int S = g2.kh2 * g2.kw2;
        const bool given = thin_dtype == DMV_DT_S2D;          // the caller keeps X2 (dmv_thin_s2d_prep)
        const size_t Xb = given ? 0 : al((size_t)N * (Hb / 2) * (Wb / 2) * 64), Db = al((size_t)S * 32 * Cw * 4);
        if (!ws || ws_bytes < Xb + Db || ((uintptr_t)ws & 255)) return fail(DMV_E_WORKSPACE, "tc_thin_wgrad: workspace too small or unaligned");
        uint8_t* base = reinterpret_cast<uint8_t*>(ws);
        int rc = given ? DMV_OK : thin_s2d_prep(thin, thin_dtype, base, N, Hb, Wb, Ct, st);
        if (rc) return rc;
        float* dw2 = reinterpret_cast<float*>(base + Xb);
        WProblem q;
        q.big = given ? thin : base; q.N = N; q.Hb = Hb / 2; q.Wb = Wb / 2; q.Cb = 32; q.stride = 1;
        q.small = wide; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cw;
        q.kh = g2.kh2; q.kw = g2.kw2; q.pt = -g2.dh0; q.pl = -g2.dw0; q.dw = dw2;
        rc = run_wgrad(q, base + Xb + Db, ws_bytes - Xb - Db, st);
        if (rc) return rc;
        return thin_s2d_gather_dw(dw2, dw, Ct, Cw, kh, kw, ph.before, pw.before, g2, st);
    }
    if (!wgrad_eligible(Kp, Cw, 1)) return fail(DMV_E_UNSUPPORTED_SHAPE, "tc_thin_wgrad: channel counts not covered");
    const size_t Pb = al((size_t)N * ph.out * pw.out * Kp * 2), Db = al((size_t)Kp * Cw * 4);
    const size_t parts = tc_wgrad_workspace(1, Kp, Cw, N, ph.out, pw.out);
    if (!ws || ws_bytes < Pb + Db + parts || ((uintptr_t)ws & 255)) return fail(DMV_E_WORKSPACE, "tc_thin_wgrad: workspace too small or unaligned");
    uint8_t* base = reinterpret_cast<uint8_t*>(ws);
    int rc = thin_im2col(thin, thin_dtype, base, N, Hb, Wb, Ct, kh, kw, stride, st);
    if (rc) return rc;
    float* dwt = reinterpret_cast<float*>(base + Pb);
    WProblem q;
    q.big = base; q.N = N; q.Hb = ph.out; q.Wb = pw.out; q.Cb = Kp; q.stride = 1;
    q.small = wide; q.Hs = ph.out; q.Ws = pw.out; q.Cs = Cw;
    q.kh = 1; q.kw = 1; q.pt = 0; q.pl = 0; q.dw = dwt;
    rc = run_wgrad(q, base + Pb + Db, ws_bytes - Pb - Db, st);
    if (rc) return rc;
    return copy_f32(dwt, dw, rows * Cw, st);      // drop the zero-padded rows
}

}  // namespace dmv


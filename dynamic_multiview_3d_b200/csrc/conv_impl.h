// Internal interfaces between the public dispatchers (conv_api.cu) and the two kernel
// families.  tc_* return DMV_E_UNSUPPORTED_SHAPE when the tensor-core path does not cover
// a shape; DMV_ALGO_AUTO then falls through to the SIMT kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace dmv {
// out[i] = sum_z part[z * n + i], deterministic: warp w of a CTA sums z = w, w + ZW, ... in order, then the ZW
// warp sums are added in warp order.  The z loop is spread over up to 32 warps so short outputs (bias
// gradients: n = C) are not one long dependent chain.
int reduce_partials(const float* part, float* out, long long n, int splits, cudaStream_t st);
size_t simt_wgrad_workspace(int taps, int Cin, int Cout, long long pixels);
size_t act_bwd_bias_workspace(long long rows, int C);
// group > 0: the grouped form (dmv_act_bwd_bias_grouped), dy row pitch ld_dy elements; group == 0: the plain form
int act_bwd_bias(const void* dy, const void* y, void* dpre, float* db, long long rows, int C, int act, void* ws, size_t ws_bytes,
                 cudaStream_t st, int group = 0, long long ld_dy = 0);
int simt_bias_grad(const void* dy_bf16, float* db, long long pixels, int C, void* ws, size_t ws_bytes, cudaStream_t st);
int simt_conv_fwd(const void* x, int xdt, const void* w, const float* bias, void* y, int ydt, int B, int H, int W, int Cin,
                  int Cout, int kh, int kw, int stride, int act, cudaStream_t st);
int simt_conv_dgrad(const void* dy, const void* w, void* dx, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                    cudaStream_t st);
int simt_conv_wgrad(const void* x, int xdt, const void* dy, float* dw, float* db, int B, int H, int W, int Cin, int Cout, int kh,
                    int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st);
int simt_deconv_fwd(const void* x, const void* w, void* y, int ydt, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                    int stride, int act, cudaStream_t st);
int simt_deconv_dgrad(const void* dy, int dydt, const void* w, void* dx, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                      int kw, int stride, cudaStream_t st);
int simt_deconv_wgrad(const void* x, const void* dy, int dydt, float* dw, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                      int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st);

size_t thin_wgrad_workspace(int taps, int Ct);
int thin_patch_cols(int taps, int Ct);
int thin_im2col(const void* thin, int thin_dtype, void* P, int N, int Hb, int Wb, int Ct, int kh, int kw, int stride, cudaStream_t st);
int thin_pack_weights(const void* w_bf16, void* packed, int rows, int Cw, int Kp, cudaStream_t st);
int copy_f32(const float* src, float* dst, int n, cudaStream_t st);
// thin-channel layers on tensor cores through an explicit patch matrix (conv_tc.cu / wgrad_tc.cu)
size_t tc_thin_workspace(int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw, int stride);
int tc_thin_fwd(const void* thin, int thin_dtype, const void* w_bf16, const float* bias, void* out, int out_dtype, int N, int Hb, int Wb,
                int Ct, int Cw, int kh, int kw, int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_thin_wgrad(const void* thin, int thin_dtype, const void* wide_bf16, float* dw, int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw,
                  int stride, void* ws, size_t ws_bytes, cudaStream_t st);
bool thin_wgrad_eligible(int taps, int Ct, int Cw);
// thin stride-2 layers through space-to-depth (thin_simt.cu / conv_tc.cu / wgrad_tc.cu): X2[n][h/2][w/2][32] holds the
// 2x2 pixel block of the thin tensor as channels (ph, pw, c), zero padded to 32; the layer is then a stride-1 conv
// over X2 with kh2 x kw2 shifts starting at (dh0, dw0)
struct S2dGeom {
    int dh0, kh2, dw0, kw2;
};
bool thin_s2d_eligible(int Hb, int Wb, int Ct, int Cw, int kh, int kw, int stride);
S2dGeom thin_s2d_geom(int Hb, int Wb, int kh, int kw);
int thin_s2d_prep(const void* thin, int thin_dtype, void* X2, int N, int Hb, int Wb, int Ct, cudaStream_t st);
// W2p[cw][(shift, ch')] (bf16, K-major) from w[r][s][ct][cw]
int thin_s2d_pack_weights(const void* w_bf16, void* packed, int Ct, int Cw, int kh, int kw, int pt, int pl, S2dGeom g, cudaStream_t st);
// dW[r][s][ct][cw] (fp32) gathered from dW2[shift][ch'][cw]
int thin_s2d_gather_dw(const float* dw2, float* dw, int Ct, int Cw, int kh, int kw, int pt, int pl, S2dGeom g, cudaStream_t st);
int thin_wgrad(const void* thin, int thin_dtype, const void* wide_bf16, float* dw, int N, int Hb, int Wb, int Ct, int kh, int kw, int stride,
               void* ws, size_t ws_bytes, cudaStream_t st);

// thin stride-2 5x5 layers as single mma.sync bandwidth kernels (thin_mma.cu): no prep pass, no patch matrix
bool thin_mma_eligible(int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw, int stride);
size_t thin_mma_wgrad_workspace(int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw, int stride);
int thin_mma_conv_fwd(const void* thin, int thin_dtype, const void* w_bf16, const float* bias, void* out, int out_dtype, int N, int Hb, int Wb,
                      int Ct, int Cw, int kh, int kw, int stride, int act, cudaStream_t st);
int thin_mma_deconv_fwd(const void* x_bf16, const void* w_bf16, void* y, int y_dtype, int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw,
                        int stride, int act, cudaStream_t st);
int thin_mma_wgrad(const void* thin, int thin_dtype, const void* wide_bf16, float* dw, int N, int Hb, int Wb, int Ct, int Cw, int kh, int kw,
                   int stride, void* ws, size_t ws_bytes, cudaStream_t st);

// Activation-derivative fusion for input-gradient launches: after tc_set_dact(y, act) the next tc_*_dgrad / thin dgrad
// launch of this thread writes dX * act'(y) (y: bf16, same shape as dX); tc_finish_dact() tells whether a launch applied
// it (a path that did not must be followed by an elementwise pass) and clears the request.
void tc_set_dact(const void* y_bf16, int act);
bool tc_finish_dact();
// weight-packing mode of the NEXT tc_* launch of this thread: 0 = pack then run, DMV_ALGO_PACK_ONLY, DMV_ALGO_PREPACKED
void tc_set_pack_mode(int mode);
size_t tc_wgrad_workspace(int taps, int Cin, int Cout, int N, int Hs, int Ws);      // Hs x Ws: the gradient image
size_t tc_pack_workspace(int taps, int Cin, int Cout);
int tc_conv_fwd(const void* x, int xdt, const void* w, const float* bias, void* y, int ydt, int B, int H, int W, int Cin, int Cout,
                int kh, int kw, int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_conv_dgrad(const void* dy, const void* w, void* dx, int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride,
                  void* ws, size_t ws_bytes, cudaStream_t st);
int tc_conv_wgrad(const void* x, int xdt, const void* dy, float* dw, float* db, int B, int H, int W, int Cin, int Cout, int kh,
                  int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_deconv_fwd(const void* x, const void* w, void* y, int ydt, int B, int Hout, int Wout, int Cin, int Cout, int kh, int kw,
                  int stride, int act, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_deconv_dgrad(const void* dy, int dydt, const void* w, void* dx, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                    int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_deconv_wgrad(const void* x, const void* dy, int dydt, float* dw, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                    int kw, int stride, void* ws, size_t ws_bytes, cudaStream_t st);
size_t tc_linear_workspace(int M, int K, int N);
int tc_linear_fwd(const void* x, const void* w, const float* bias, void* y, int M, int K, int N, int act, void* ws, size_t ws_bytes,
                  cudaStream_t st);
int tc_linear_dgrad(const void* dy, const void* w, void* dx, int M, int K, int N, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_linear_wgrad(const void* x, const void* dy, float* dw, float* db, int M, int K, int N, void* ws, size_t ws_bytes,
                    cudaStream_t st);
}  // namespace dmv

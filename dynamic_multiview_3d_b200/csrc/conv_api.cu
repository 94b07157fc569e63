// Public conv / deconv / linear entry points (include/dmv3d.h): argument checks and the
// choice between the tcgen05 implicit-GEMM kernels (conv_tc.cu) and the SIMT kernels
// (conv_simt.cu).  DMV_ALGO_AUTO takes the tensor-core path whenever the shape qualifies.
#include "common.cuh"
#include "conv_impl.h"

using namespace dmv;

#define DMV_CHECK_ALGO(algo) \
    DMV_REQUIRE((algo) == DMV_ALGO_AUTO || (algo) == DMV_ALGO_SIMT || (algo) == DMV_ALGO_TCGEN05, DMV_E_INVALID_ARG, "unknown algo")

// DMV_ALGO_PACK_ONLY / DMV_ALGO_PREPACKED (include/dmv3d.h): split off the flag bits, arm the tensor-core launchers for the
// duration of the call.  ``run`` is the tensor-core attempt of the entry point; under PACK_ONLY nothing else may execute.
struct PackScope {
    int mode;
    explicit PackScope(int& algo) : mode(algo & (DMV_ALGO_PACK_ONLY | DMV_ALGO_PREPACKED)) {
        algo &= ~(DMV_ALGO_PACK_ONLY | DMV_ALGO_PREPACKED);
        tc_set_pack_mode(mode);
    }
    ~PackScope() { tc_set_pack_mode(0); }
    bool pack_only() const { return mode == DMV_ALGO_PACK_ONLY; }
};
static int pack_only_result(int rc) { return (rc == DMV_E_UNSUPPORTED_SHAPE || rc == DMV_E_WORKSPACE) ? DMV_OK : rc; }

// Input gradients with the producer's activation derivative folded in: dx <- dx * act'(y_in).  ``run`` launches the
// input-gradient kernels; the tensor-core paths apply the factor in their epilogue (before the bf16 rounding), any other
// path is followed by one elementwise pass in place.
template <typename F>
static int dgrad_with_dact(const void* y_in, int act_in, void* dx, long long n, cudaStream_t st, F run) {
    if (!y_in || act_in == DMV_ACT_NONE) return run();
    tc_set_dact(y_in, act_in);
    const int rc = run();
    const bool fused = tc_finish_dact();
    if (rc != DMV_OK || fused) return rc;
    return dmv_act_bwd(dx, y_in, dx, DMV_DT_BF16, n, act_in, st);
}

extern "C" {

size_t dmv_act_bwd_bias_workspace_size(long long rows, int C) { return rows > 0 && C > 0 ? act_bwd_bias_workspace(rows, C) : 0; }

int dmv_act_bwd_bias(const void* dy_bf16, const void* y_bf16, void* dpre_bf16, float* db, long long rows, int C, int act, void* workspace,
                     size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(dy_bf16 && y_bf16 && dpre_bf16 && db && rows > 0 && C > 0, DMV_E_INVALID_ARG, "act_bwd_bias: bad argument");
    return act_bwd_bias(dy_bf16, y_bf16, dpre_bf16, db, rows, C, act, workspace, workspace_bytes, (cudaStream_t)stream);
}

int dmv_act_bwd_bias_grouped(const void* dy_bf16, long long ld_dy, int group, const void* y_bf16, void* dpre_bf16, float* db, long long rows,
                             int C, int act, void* workspace, size_t workspace_bytes, void* stream) {
    DMV_REQUIRE(dy_bf16 && y_bf16 && dpre_bf16 && db && rows > 0 && C > 0 && group > 0 && ld_dy >= C, DMV_E_INVALID_ARG,
                "act_bwd_bias_grouped: bad argument");
    DMV_REQUIRE(rows <= (1ll << 62) / group / ld_dy, DMV_E_UNSUPPORTED_SHAPE, "act_bwd_bias_grouped: dy too large");
    return act_bwd_bias(dy_bf16, y_bf16, dpre_bf16, db, rows, C, act, workspace, workspace_bytes, (cudaStream_t)stream, group, ld_dy);
}

size_t dmv_thin_s2d_size(int N, int H, int W, int C_thin, int C_wide, int kh, int kw, int stride) {
    if (N <= 0 || H <= 0 || W <= 0 || C_thin <= 0 || !thin_s2d_eligible(H, W, C_thin, C_wide, kh, kw, stride)) return 0;
    if (thin_mma_eligible(N, H, W, C_thin, C_wide, kh, kw, stride)) return 0;      // single-kernel form: no prep tensor
    return (size_t)N * (H / 2) * (W / 2) * 64;
}

int dmv_thin_s2d_prep(const void* thin, int thin_dtype, void* x2, int N, int H, int W, int C_thin, void* stream) {
    DMV_REQUIRE(thin && x2 && N > 0 && H > 0 && W > 0 && C_thin > 0 && 4 * C_thin <= 32 && !(H & 1) && !(W & 1), DMV_E_INVALID_ARG, "thin_s2d_prep: bad argument");
    DMV_REQUIRE(thin_dtype == DMV_DT_F32 || thin_dtype == DMV_DT_BF16, DMV_E_INVALID_ARG, "thin_s2d_prep: dtype");
    DMV_REQUIRE(((uintptr_t)x2 & 15) == 0, DMV_E_ALIGN, "thin_s2d_prep: x2 must be 16-byte aligned");
    return thin_s2d_prep(thin, thin_dtype, x2, N, H, W, C_thin, (cudaStream_t)stream);
}

// layers with fewer than 8 channels on the image side (e0: 3, flow head: 2) go through a patch matrix
static bool thin_side(int c) { return c < 8; }

size_t dmv_wgrad_workspace_size(int B, int H, int W, int Cbig, int Csmall, int kh, int kw, int stride) {
    if (B <= 0 || H <= 0 || W <= 0 || Cbig <= 0 || Csmall <= 0 || kh <= 0 || kw <= 0 || stride <= 0) return 0;
    const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
    const long long pixels = (long long)B * ph.out * pw.out;
    const int taps = kh * kw;
    size_t a = simt_wgrad_workspace(taps, Cbig, Csmall, pixels);
    size_t b = tc_wgrad_workspace(taps, Cbig, Csmall, B, ph.out, pw.out);
    if (b > a) a = b;
    if (thin_side(Cbig)) {
        size_t c = tc_thin_workspace(B, H, W, Cbig, Csmall, kh, kw, stride);
        if (c > a) a = c;
        c = thin_mma_wgrad_workspace(B, H, W, Cbig, Csmall, kh, kw, stride);
        if (c > a) a = c;
        if (thin_wgrad_eligible(taps, Cbig, Csmall)) {
            c = thin_wgrad_workspace(taps, Cbig);
            if (c > a) a = c;
        }
    }
    return a + 256;
}

size_t dmv_conv_workspace_size(int B, int H, int W, int Cbig, int Csmall, int kh, int kw, int stride) {
    if (B <= 0 || H <= 0 || W <= 0 || Cbig <= 0 || Csmall <= 0 || kh <= 0 || kw <= 0 || stride <= 0) return 0;
    size_t a = tc_pack_workspace(kh * kw, Cbig, Csmall);
    if (H == 1 && W == 1 && kh == 1 && kw == 1) {           // linear layer: split-K partials
        size_t c = tc_linear_workspace(B, Cbig, Csmall);
        if (c > a) a = c;
    }
    if (thin_side(Cbig)) {
        size_t c = tc_thin_workspace(B, H, W, Cbig, Csmall, kh, kw, stride);
        if (c > a) a = c;
    }
    return a + 256;
}

int dmv_conv2d_fwd(const void* x, int x_dtype, const void* w, const float* bias, void* y, int y_dtype, int B, int H, int W,
                   int Cin, int Cout, int kh, int kw, int stride, int act, void* workspace, size_t workspace_bytes, int algo,
                   void* stream) {
    DMV_REQUIRE(x && w && y, DMV_E_INVALID_ARG, "conv2d_fwd: null pointer");
    PackScope pk(algo);
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.pack_only()) {
        if (algo == DMV_ALGO_SIMT || thin_side(Cin) || x_dtype != DMV_DT_BF16) return DMV_OK;
        return pack_only_result(tc_conv_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st));
    }
    if (x_dtype == DMV_DT_S2D) {        // caller-kept space-to-depth tensor: only the tensor-core thin path understands it
        DMV_REQUIRE(algo != DMV_ALGO_SIMT && thin_side(Cin), DMV_E_INVALID_ARG, "conv2d_fwd: DMV_DT_S2D needs the tensor-core thin path");
        return tc_thin_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st);
    }
    if (algo != DMV_ALGO_SIMT && thin_side(Cin)) {
        int rc = thin_mma_conv_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE) return rc;
        rc = tc_thin_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE && rc != DMV_E_WORKSPACE) return rc;
    }
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_conv_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_conv_fwd(x, x_dtype, w, bias, y, y_dtype, B, H, W, Cin, Cout, kh, kw, stride, act, st);
}

int dmv_conv2d_dgrad(const void* dy, const void* w, void* dx, const void* y_in, int act_in, int B, int H, int W, int Cin, int Cout,
                     int kh, int kw, int stride, void* workspace, size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(dy && w && dx, DMV_E_INVALID_ARG, "conv2d_dgrad: null pointer");
    PackScope pk(algo);
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.pack_only()) {
        if (algo == DMV_ALGO_SIMT) return DMV_OK;
        return pack_only_result(tc_conv_dgrad(dy, w, dx, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st));
    }
    return dgrad_with_dact(y_in, act_in, dx, (long long)B * H * W * Cin, st, [&]() -> int {
        if (algo != DMV_ALGO_SIMT) {
            int rc = tc_conv_dgrad(dy, w, dx, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
            if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
        }
        return simt_conv_dgrad(dy, w, dx, B, H, W, Cin, Cout, kh, kw, stride, st);
    });
}

int dmv_conv2d_wgrad(const void* x, int x_dtype, const void* dy, float* dw, float* db, int B, int H, int W, int Cin, int Cout,
                     int kh, int kw, int stride, void* workspace, size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(x && dy && dw, DMV_E_INVALID_ARG, "conv2d_wgrad: null pointer");
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (x_dtype == DMV_DT_S2D) {
        DMV_REQUIRE(algo != DMV_ALGO_SIMT && thin_side(Cin), DMV_E_INVALID_ARG, "conv2d_wgrad: DMV_DT_S2D needs the tensor-core thin path");
        int rc = tc_thin_wgrad(x, x_dtype, dy, dw, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc == DMV_OK && db) {
            const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
            rc = simt_bias_grad(dy, db, (long long)B * ph.out * pw.out, Cout, workspace, workspace_bytes, st);
        }
        return rc;
    }
    if (algo != DMV_ALGO_SIMT && thin_side(Cin)) {   // e0: 3-channel image side
        int rc = thin_mma_wgrad(x, x_dtype, dy, dw, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc == DMV_E_UNSUPPORTED_SHAPE || rc == DMV_E_WORKSPACE)
            rc = tc_thin_wgrad(x, x_dtype, dy, dw, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc == DMV_E_UNSUPPORTED_SHAPE || rc == DMV_E_WORKSPACE) {
            if (!thin_wgrad_eligible(kh * kw, Cin, Cout)) goto generic;
            rc = thin_wgrad(x, x_dtype, dy, dw, B, H, W, Cin, kh, kw, stride, workspace, workspace_bytes, st);
        }
        if (rc == DMV_OK && db) {
            const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
            rc = simt_bias_grad(dy, db, (long long)B * ph.out * pw.out, Cout, workspace, workspace_bytes, st);
        }
        return rc;
    }
generic:
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_conv_wgrad(x, x_dtype, dy, dw, nullptr, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc == DMV_OK && db) {
            const SamePad ph = same_pad(H, kh, stride), pw = same_pad(W, kw, stride);
            rc = simt_bias_grad(dy, db, (long long)B * ph.out * pw.out, Cout, workspace, workspace_bytes, st);
        }
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_conv_wgrad(x, x_dtype, dy, dw, db, B, H, W, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
}

int dmv_deconv2d_fwd(const void* x, const void* w, void* y, int y_dtype, int B, int Hout, int Wout, int Cin, int Cout, int kh,
                     int kw, int stride, int act, void* workspace, size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(x && w && y, DMV_E_INVALID_ARG, "deconv2d_fwd: null pointer");
    PackScope pk(algo);
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.pack_only()) {
        if (algo == DMV_ALGO_SIMT || thin_side(Cout)) return DMV_OK;
        return pack_only_result(tc_deconv_fwd(x, w, y, y_dtype, B, Hout, Wout, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st));
    }
    if (algo != DMV_ALGO_SIMT && thin_side(Cout)) {     // flow head: 2-channel output side
        int rc = thin_mma_deconv_fwd(x, w, y, y_dtype, B, Hout, Wout, Cout, Cin, kh, kw, stride, act, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE) return rc;
    }
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_deconv_fwd(x, w, y, y_dtype, B, Hout, Wout, Cin, Cout, kh, kw, stride, act, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_deconv_fwd(x, w, y, y_dtype, B, Hout, Wout, Cin, Cout, kh, kw, stride, act, st);
}

int dmv_deconv2d_dgrad(const void* dy, int dy_dtype, const void* w, void* dx, const void* y_in, int act_in, int B, int Hout, int Wout,
                       int Cin, int Cout, int kh, int kw, int stride, void* workspace, size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(dy && w && dx, DMV_E_INVALID_ARG, "deconv2d_dgrad: null pointer");
    PackScope pk(algo);
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (pk.pack_only()) {
        if (algo == DMV_ALGO_SIMT || thin_side(Cout) || dy_dtype != DMV_DT_BF16) return DMV_OK;
        return pack_only_result(tc_deconv_dgrad(dy, dy_dtype, w, dx, B, Hout, Wout, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st));
    }
    if (dy_dtype == DMV_DT_S2D)
        DMV_REQUIRE(algo != DMV_ALGO_SIMT && thin_side(Cout), DMV_E_INVALID_ARG, "deconv2d_dgrad: DMV_DT_S2D needs the tensor-core thin path");
    const SamePad ph = same_pad(Hout, kh, stride), pw = same_pad(Wout, kw, stride);
    return dgrad_with_dact(y_in, act_in, dx, (long long)B * ph.out * pw.out * Cin, st, [&]() -> int {
        if (dy_dtype == DMV_DT_S2D)
            return tc_thin_fwd(dy, dy_dtype, w, nullptr, dx, DMV_DT_BF16, B, Hout, Wout, Cout, Cin, kh, kw, stride, DMV_ACT_NONE, workspace,
                               workspace_bytes, st);
        if (algo != DMV_ALGO_SIMT && thin_side(Cout)) {   // flow head: dx = conv of the 2-channel gradient with w[r,s,c,ci]
            int rc = thin_mma_conv_fwd(dy, dy_dtype, w, nullptr, dx, DMV_DT_BF16, B, Hout, Wout, Cout, Cin, kh, kw, stride, DMV_ACT_NONE, st);
            if (rc != DMV_E_UNSUPPORTED_SHAPE) return rc;
            rc = tc_thin_fwd(dy, dy_dtype, w, nullptr, dx, DMV_DT_BF16, B, Hout, Wout, Cout, Cin, kh, kw, stride, DMV_ACT_NONE, workspace,
                                 workspace_bytes, st);
            if (rc != DMV_E_UNSUPPORTED_SHAPE && rc != DMV_E_WORKSPACE) return rc;
        }
        if (algo != DMV_ALGO_SIMT) {
            int rc = tc_deconv_dgrad(dy, dy_dtype, w, dx, B, Hout, Wout, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
            if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
        }
        return simt_deconv_dgrad(dy, dy_dtype, w, dx, B, Hout, Wout, Cin, Cout, kh, kw, stride, st);
    });
}

int dmv_deconv2d_wgrad(const void* x, const void* dy, int dy_dtype, float* dw, int B, int Hout, int Wout, int Cin, int Cout,
                       int kh, int kw, int stride, void* workspace, size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(x && dy && dw, DMV_E_INVALID_ARG, "deconv2d_wgrad: null pointer");
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (dy_dtype == DMV_DT_S2D) {
        DMV_REQUIRE(algo != DMV_ALGO_SIMT && thin_side(Cout), DMV_E_INVALID_ARG, "deconv2d_wgrad: DMV_DT_S2D needs the tensor-core thin path");
        return tc_thin_wgrad(dy, dy_dtype, x, dw, B, Hout, Wout, Cout, Cin, kh, kw, stride, workspace, workspace_bytes, st);
    }
    if (algo != DMV_ALGO_SIMT && thin_side(Cout)) {      // flow head: 2-channel output side
        int rc = thin_mma_wgrad(dy, dy_dtype, x, dw, B, Hout, Wout, Cout, Cin, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE && rc != DMV_E_WORKSPACE) return rc;
        rc = tc_thin_wgrad(dy, dy_dtype, x, dw, B, Hout, Wout, Cout, Cin, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE && rc != DMV_E_WORKSPACE) return rc;
        if (thin_wgrad_eligible(kh * kw, Cout, Cin))
            return thin_wgrad(dy, dy_dtype, x, dw, B, Hout, Wout, Cout, kh, kw, stride, workspace, workspace_bytes, st);
    }
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_deconv_wgrad(x, dy, dy_dtype, dw, B, Hout, Wout, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_deconv_wgrad(x, dy, dy_dtype, dw, B, Hout, Wout, Cin, Cout, kh, kw, stride, workspace, workspace_bytes, st);
}

// linear == 1x1 conv over M "pixels"
int dmv_linear_fwd(const void* x, const void* w, const float* bias, void* y, int M, int K, int N, int act, void* workspace,
                   size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(x && w && y, DMV_E_INVALID_ARG, "linear_fwd: null pointer");
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_linear_fwd(x, w, bias, y, M, K, N, act, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_conv_fwd(x, DMV_DT_BF16, w, bias, y, DMV_DT_BF16, M, 1, 1, K, N, 1, 1, 1, act, st);
}

int dmv_linear_dgrad(const void* dy, const void* w, void* dx, const void* y_in, int act_in, int M, int K, int N, void* workspace,
                     size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(dy && w && dx, DMV_E_INVALID_ARG, "linear_dgrad: null pointer");
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    return dgrad_with_dact(y_in, act_in, dx, (long long)M * K, st, [&]() -> int {
        if (algo != DMV_ALGO_SIMT) {
            int rc = tc_linear_dgrad(dy, w, dx, M, K, N, workspace, workspace_bytes, st);
            if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
        }
        return simt_conv_dgrad(dy, w, dx, M, 1, 1, K, N, 1, 1, 1, st);
    });
}

int dmv_linear_wgrad(const void* x, const void* dy, float* dw, float* db, int M, int K, int N, void* workspace,
                     size_t workspace_bytes, int algo, void* stream) {
    DMV_REQUIRE(x && dy && dw, DMV_E_INVALID_ARG, "linear_wgrad: null pointer");
    DMV_CHECK_ALGO(algo);
    cudaStream_t st = (cudaStream_t)stream;
    if (algo != DMV_ALGO_SIMT) {
        int rc = tc_linear_wgrad(x, dy, dw, nullptr, M, K, N, workspace, workspace_bytes, st);
        if (rc == DMV_OK && db) rc = simt_bias_grad(dy, db, M, N, workspace, workspace_bytes, st);
        if (rc != DMV_E_UNSUPPORTED_SHAPE || algo == DMV_ALGO_TCGEN05) return rc;
    }
    return simt_conv_wgrad(x, DMV_DT_BF16, dy, dw, db, M, 1, 1, K, N, 1, 1, 1, workspace, workspace_bytes, st);
}
}

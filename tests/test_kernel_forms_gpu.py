"""Kernel-form coverage.  Every conv / deconv / linear / elementwise kernel form of csrc/ is reached by at least one case
here, the case proves through the per-label launch counter (dmv_launch_count_named) that the form it names actually
ran, and compares the result with the NumPy oracle evaluated in float64 on bf16-representable inputs.

- FORMS: one row per launch label; a CPU test fails when a label of csrc/ is neither in FORMS nor in EXEMPT.
- GEOMETRY: non-square, odd and eligibility-edge shapes at algo = auto, each with the form it is expected to take.
- the graph's layer shapes under every DMV_NO_* switch that changes their form.
- the update kernels under their once-per-process switches, each setting in a child process."""
import functools
import glob
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle import tf_ops as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dynamic_multiview_3d_b200", "csrc")
gpu = pytest.mark.gpu


def bf16_round(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@functools.lru_cache(maxsize=None)
def launch_labels():
    """Every label passed to check_launch(...) in csrc/*.cu (all string literals of the argument, so a label chosen by a
    conditional expression contributes each of its alternatives)."""
    labels = set()
    for path in sorted(glob.glob(os.path.join(CSRC, "*.cu"))):
        src = open(path).read()
        for m in re.finditer(r"check_launch\((.*?)\);", src, flags=re.S):
            labels.update(re.findall(r'"([^"]+)"', m.group(1)))
    return frozenset(labels)


# --------------------------------------------------------------------------------------------------------------------
# one layer call through the C ABI, checked against the oracle
# --------------------------------------------------------------------------------------------------------------------
F32, BF16 = 1, 0


def _dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda().to(dtype)


def _counts(labels):
    from dynamic_multiview_3d_b200 import _lib
    return {l: _lib.launch_count_named(l) for l in labels}


def run_layer(kind, op, B, H, W, cin, cout, kh, kw, s, y_bf16=False, ws_bytes=None, seed=0):
    """Runs one entry point (kind: conv / deconv; op: fwd / dgrad / wgrad) at algo = auto on seeded bf16-representable
    inputs, checks it against the float64 oracle at the suite's tolerances and returns {label: launches} of the call.
    H, W are the big side (conv input, deconv output).  A thin side (< 8 channels) is fp32, as in the graph.  ws_bytes
    overrides the workspace the library asks for."""
    from dynamic_multiview_3d_b200 import _lib
    L = _lib.load()
    rng = np.random.default_rng(seed * 7919 + B * 1000003 + H * 10007 + W * 1009 + cin * 101 + cout * 11 + kh * 5 + kw * 3 + s)
    st = torch.cuda.current_stream().cuda_stream
    h, w = -(-H // s), -(-W // s)
    labels = launch_labels()
    if kind == "conv":
        thin = cin < 8
        x = bf16_round(rng.random((B, H, W, cin)) if thin else rng.standard_normal((B, H, W, cin)))
        wt = bf16_round(rng.standard_normal((kh, kw, cin, cout)) * T.conv_stddev(kh, kw, cin))
        b = rng.standard_normal(cout).astype(np.float32)
        gy = bf16_round(rng.standard_normal((B, h, w, cout)))
        x64, w64, gy64 = x.astype(np.float64), wt.astype(np.float64), gy.astype(np.float64)
        need = (L.dmv_wgrad_workspace_size if op == "wgrad" else L.dmv_conv_workspace_size)(B, H, W, cin, cout, kh, kw, s)
    else:
        thin = cout < 8
        x = bf16_round(rng.standard_normal((B, h, w, cin)))
        wt = bf16_round(rng.standard_normal((kh, kw, cout, cin)) * T.deconv_stddev(kh, kw, cin, s, s))
        gy = bf16_round(rng.standard_normal((B, H, W, cout)))
        x64, w64, gy64 = x.astype(np.float64), wt.astype(np.float64), gy.astype(np.float64)
        need = (L.dmv_wgrad_workspace_size if op == "wgrad" else L.dmv_conv_workspace_size)(B, H, W, cout, cin, kh, kw, s)
    ws = torch.empty(max(int(need if ws_bytes is None else ws_bytes), 256), dtype=torch.uint8, device="cuda")
    wd = _dev(wt, torch.bfloat16)
    n0 = _counts(labels)
    if kind == "conv":
        xdt = F32 if thin else BF16
        xd = _dev(x, torch.float32 if thin else torch.bfloat16)
        if op == "fwd":
            bd = _dev(b, torch.float32)
            y = torch.empty((B, h, w, cout), dtype=torch.bfloat16 if y_bf16 else torch.float32, device="cuda")
            _lib.call("dmv_conv2d_fwd", xd.data_ptr(), xdt, wd.data_ptr(), bd.data_ptr(), y.data_ptr(), BF16 if y_bf16 else F32, B, H, W, cin, cout,
                      kh, kw, s, 0, ws.data_ptr(), ws.numel(), 0, st)
            outs = [(y, T.conv2d_same(x64, w64, b.astype(np.float64), s, s), 1e-2 if y_bf16 else 1e-4)]
        else:
            gx, gw, gb = T.conv2d_same_grads(x64, w64, gy64, s, s)
            dyd = _dev(gy, torch.bfloat16)
            if op == "dgrad":
                dx = torch.empty((B, H, W, cin), dtype=torch.bfloat16, device="cuda")
                _lib.call("dmv_conv2d_dgrad", dyd.data_ptr(), wd.data_ptr(), dx.data_ptr(), None, 0, B, H, W, cin, cout, kh, kw, s,
                          ws.data_ptr(), ws.numel(), 0, st)
                outs = [(dx, gx, 1e-2)]
            else:
                dw = torch.zeros((kh, kw, cin, cout), device="cuda")
                db = torch.zeros((cout,), device="cuda")
                _lib.call("dmv_conv2d_wgrad", xd.data_ptr(), xdt, dyd.data_ptr(), dw.data_ptr(), db.data_ptr(), B, H, W, cin, cout, kh, kw, s,
                          ws.data_ptr(), ws.numel(), 0, st)
                outs = [(dw, gw, 2e-4), (db, gb, 1e-4)]
    else:
        dydt = F32 if thin else BF16
        xd = _dev(x, torch.bfloat16)
        if op == "fwd":
            y = torch.empty((B, H, W, cout), dtype=torch.bfloat16 if y_bf16 else torch.float32, device="cuda")
            _lib.call("dmv_deconv2d_fwd", xd.data_ptr(), wd.data_ptr(), y.data_ptr(), BF16 if y_bf16 else F32, B, H, W, cin, cout, kh, kw, s, 0,
                      ws.data_ptr(), ws.numel(), 0, st)
            outs = [(y, T.conv2d_transpose_same(x64, w64, (B, H, W, cout), s, s), 1e-2 if y_bf16 else 1e-4)]
        else:
            gx, gw = T.conv2d_transpose_same_grads(x64, w64, gy64, s, s)
            dyd = _dev(gy, torch.float32 if thin else torch.bfloat16)
            if op == "dgrad":
                dx = torch.empty((B, h, w, cin), dtype=torch.bfloat16, device="cuda")
                _lib.call("dmv_deconv2d_dgrad", dyd.data_ptr(), dydt, wd.data_ptr(), dx.data_ptr(), None, 0, B, H, W, cin, cout, kh, kw, s,
                          ws.data_ptr(), ws.numel(), 0, st)
                outs = [(dx, gx, 1e-2)]
            else:
                dw = torch.zeros((kh, kw, cout, cin), device="cuda")
                _lib.call("dmv_deconv2d_wgrad", xd.data_ptr(), dyd.data_ptr(), dydt, dw.data_ptr(), B, H, W, cin, cout, kh, kw, s,
                          ws.data_ptr(), ws.numel(), 0, st)
                outs = [(dw, gw, 2e-4)]
    torch.cuda.synchronize()
    n1 = _counts(labels)
    ran = {l: n1[l] - n0[l] for l in labels if n1[l] != n0[l]}
    for got, ref, tol in outs:
        err = _rel(got.float().cpu().numpy().astype(np.float64), ref)
        assert err < tol, "%s %s %s: relative error %.3g >= %g (forms: %s)" % (kind, op, (B, H, W, cin, cout, kh, kw, s), err, tol, sorted(ran))
    return ran


def run_linear_fwd(M, K, N):
    from dynamic_multiview_3d_b200 import _lib
    L = _lib.load()
    rng = np.random.default_rng(M * 31 + K * 7 + N)
    x = bf16_round(rng.standard_normal((M, K)))
    m = bf16_round(rng.standard_normal((K, N)) * T.linear_stddev(K))
    b = rng.standard_normal(N).astype(np.float32)
    ref = x.astype(np.float64) @ m.astype(np.float64) + b
    y = torch.empty((M, N), dtype=torch.bfloat16, device="cuda")
    ws = torch.empty(max(int(L.dmv_conv_workspace_size(M, 1, 1, K, N, 1, 1, 1)), 256), dtype=torch.uint8, device="cuda")
    labels = launch_labels()
    n0 = _counts(labels)
    xd, md, bd = _dev(x, torch.bfloat16), _dev(m, torch.bfloat16), _dev(b, torch.float32)
    _lib.call("dmv_linear_fwd", xd.data_ptr(), md.data_ptr(), bd.data_ptr(), y.data_ptr(), M, K, N, 0, ws.data_ptr(), ws.numel(), 0,
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    n1 = _counts(labels)
    assert _rel(y.float().cpu().numpy().astype(np.float64), ref) < 1e-2
    return {l: n1[l] - n0[l] for l in labels if n1[l] != n0[l]}


def run_act_bwd_bias(rows, C):
    """dmv_act_bwd_bias with lrelu: dpre = bf16(dy * act'(y)), db = the column sums of exactly that bf16 dpre."""
    from dynamic_multiview_3d_b200 import _lib
    L = _lib.load()
    rng = np.random.default_rng(rows * 13 + C)
    dy = bf16_round(rng.standard_normal((rows, C)))
    y = bf16_round(rng.standard_normal((rows, C)))
    y[0, :8] = 0.0                                               # y == 0: slope 0.6 (TF: f1 + f2 * sign(0))
    slope = np.where(y > 0, 1.0, np.where(y < 0, 0.2, 0.6)).astype(np.float32)
    dpre_ref = bf16_round(dy * slope)
    db_ref = dpre_ref.astype(np.float64).sum(0)
    dyd, yd = _dev(dy, torch.bfloat16), _dev(y, torch.bfloat16)
    dpre = torch.empty((rows, C), dtype=torch.bfloat16, device="cuda")
    db = torch.zeros((C,), device="cuda")
    ws = torch.empty(max(int(L.dmv_act_bwd_bias_workspace_size(rows, C)), 256), dtype=torch.uint8, device="cuda")
    labels = launch_labels()
    n0 = _counts(labels)
    _lib.call("dmv_act_bwd_bias", dyd.data_ptr(), yd.data_ptr(), dpre.data_ptr(), db.data_ptr(), rows, C, 1, ws.data_ptr(), ws.numel(),
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    n1 = _counts(labels)
    assert np.array_equal(dpre.float().cpu().numpy(), dpre_ref)
    assert _rel(db.cpu().numpy().astype(np.float64), db_ref) < 1e-4
    return {l: n1[l] - n0[l] for l in labels if n1[l] != n0[l]}


def _thin_wgrad_small_ws(B, H, W, ct, kh, kw):
    """Workspace that holds the SIMT thin weight gradient's partials (thin_simt.cu run_thin) but not the tensor-core
    patch matrix: the fallback a caller with a tight workspace gets."""
    Ho, Wo = -(-H // 2), -(-W // 2)
    total = B * Ho * Wo
    ctas = min(148 * 4, -(-total // 64))
    per = -(-total // ctas)
    ctas = -(-total // per)
    return ctas * kh * kw * ct * 32 * 4


# --------------------------------------------------------------------------------------------------------------------
# FORMS: one row per launch label.  (labels that must advance, entry, shape, environment)
# shape of a layer row: (kind, op, B, H, W, cin, cout, kh, kw, stride, options); H, W: big side
# --------------------------------------------------------------------------------------------------------------------
NO_THIN = {"DMV_NO_THIN_MMA": "1"}
FORMS = [
    # thin layers (< 8 channels on the image side): single mma.sync kernels, space-to-depth and patch-matrix fallbacks
    (("thin_conv",), ("conv", "fwd", 2, 32, 64, 3, 32, 5, 5, 2, {"y_bf16": True}), {}),
    (("thin_deconv",), ("deconv", "fwd", 2, 32, 64, 32, 2, 5, 5, 2, {}), {}),
    (("thin_wgrad_mma", "thin_wgrad_gather", "reduce_partials"), ("conv", "wgrad", 2, 32, 64, 3, 32, 5, 5, 2, {}), {}),
    (("thin_s2d_prep", "thin_s2d_pack", "halo_tc"), ("conv", "fwd", 2, 32, 64, 3, 32, 5, 5, 2, {"y_bf16": True}), NO_THIN),
    (("thin_s2d_prep", "wgrad_halo2d_tc", "thin_s2d_gather"), ("conv", "wgrad", 2, 32, 64, 3, 32, 5, 5, 2, {}), NO_THIN),
    (("thin_im2col", "thin_pack"), ("deconv", "dgrad", 2, 16, 24, 32, 2, 3, 3, 1, {}), {}),
    (("thin_im2col", "copy_f32"), ("deconv", "wgrad", 2, 16, 24, 32, 2, 3, 3, 1, {}), {}),
    (("thin_wgrad", "thin_wgrad reduce"), ("conv", "wgrad", 1, 128, 128, 3, 32, 5, 5, 2, {"ws": _thin_wgrad_small_ws(1, 128, 128, 3, 5, 5)}),
     {"DMV_NO_THIN_MMA": "1", "DMV_NO_S2D": "1"}),
    # halo kernel, stride-1 source: KC 32 (32 channels) and KC 64 (64 channels) x tap counts 25, 15, 9 and generic (16)
    (("halo_tc", "tc pack weights"), ("conv", "fwd", 2, 16, 24, 32, 32, 5, 5, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 32, 32, 3, 3, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 32, 32, 4, 4, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 64, 32, 5, 5, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 64, 32, 5, 3, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 24, 16, 64, 32, 3, 5, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 64, 64, 3, 3, 1, {}), {}),
    (("halo_tc",), ("conv", "fwd", 2, 16, 24, 64, 32, 4, 4, 1, {}), {}),
    (("halo_tc",), ("conv", "dgrad", 2, 16, 24, 32, 64, 5, 5, 1, {}), {}),
    # halo kernel on two row-parity planes (stride-2 F problems, 32 source channels, KC 64): taps 15, 9 and generic (6)
    (("halo_tc (parity planes)", "tc pack stride-2"), ("conv", "fwd", 2, 32, 40, 32, 32, 5, 5, 2, {}), {}),
    (("halo_tc (parity planes)",), ("conv", "fwd", 2, 32, 40, 32, 32, 3, 5, 2, {}), {}),
    (("halo_tc (parity planes)",), ("conv", "fwd", 2, 32, 40, 32, 64, 3, 3, 2, {}), {}),
    (("halo_tc (parity planes)",), ("deconv", "dgrad", 2, 32, 40, 64, 32, 5, 5, 2, {}), {}),
    # sub-pixel form of the stride-2 G problems: KC 32 / 64 x shifts 9 (k 5) and generic (4, k 3)
    (("halo_tc (sub-pixel)", "tc pack subpixel"), ("deconv", "fwd", 2, 32, 40, 32, 16, 5, 5, 2, {}), {}),
    (("halo_tc (sub-pixel)",), ("deconv", "fwd", 2, 32, 40, 32, 16, 3, 3, 2, {}), {}),
    (("halo_tc (sub-pixel)",), ("deconv", "fwd", 2, 32, 40, 64, 32, 5, 5, 2, {}), {}),
    (("halo_tc (sub-pixel)",), ("deconv", "fwd", 2, 32, 40, 64, 16, 3, 3, 2, {}), {}),
    (("halo_tc (sub-pixel)",), ("conv", "dgrad", 2, 32, 40, 16, 32, 5, 5, 2, {}), {}),
    # ... with the coalescing depth-to-space epilogue (32 bf16 output channels)
    (("halo_tc (sub-pixel, coalescing epilogue)",), ("deconv", "fwd", 2, 32, 40, 32, 32, 5, 5, 2, {"y_bf16": True}), {}),
    (("halo_tc (sub-pixel, coalescing epilogue)",), ("deconv", "fwd", 2, 32, 40, 32, 32, 3, 3, 2, {"y_bf16": True}), {}),
    (("halo_tc (sub-pixel, coalescing epilogue)",), ("deconv", "fwd", 2, 32, 40, 64, 32, 5, 5, 2, {"y_bf16": True}), {}),
    (("halo_tc (sub-pixel, coalescing epilogue)",), ("deconv", "fwd", 2, 32, 40, 64, 32, 3, 3, 2, {"y_bf16": True}), {}),
    (("halo_tc (sub-pixel, coalescing epilogue)",), ("conv", "dgrad", 2, 32, 40, 32, 32, 5, 5, 2, {}), {}),
    # per-tap implicit GEMM
    (("igemm_tc",), ("conv", "fwd", 2, 16, 16, 64, 64, 3, 3, 2, {}), {}),
    (("igemm_tc (N-split)",), ("conv", "fwd", 2, 7, 7, 128, 128, 3, 3, 1, {}), {}),
    (("igemm_tc (split-K)", "splitk_finish"), ("linear", 8, 4096, 256), {}),
    # weight gradients
    (("wgrad_halo2d_tc",), ("conv", "wgrad", 2, 16, 24, 32, 32, 5, 5, 1, {}), {}),
    (("wgrad_halo_tc",), ("conv", "wgrad", 2, 16, 24, 64, 32, 3, 3, 1, {}), {}),
    (("wgrad_s2_tc",), ("conv", "wgrad", 2, 32, 40, 32, 64, 5, 5, 2, {}), {}),
    (("wgrad_tc", "reduce_partials", "colsum"), ("conv", "wgrad", 2, 7, 7, 128, 128, 3, 3, 1, {}), {}),
    # SIMT kernels (channel counts the tensor-core forms do not take)
    (("conv_f_simt",), ("conv", "fwd", 2, 8, 12, 48, 32, 3, 3, 1, {}), {}),
    (("conv_g_simt",), ("conv", "dgrad", 2, 8, 12, 32, 48, 3, 3, 1, {}), {}),
    (("conv_wgrad_simt", "colsum"), ("conv", "wgrad", 2, 8, 12, 48, 32, 3, 3, 1, {}), {}),
    # elementwise
    (("act_bwd_bias",), ("act_bwd_bias", 300, 96), {}),
    # linear forward: igemm on the MN-major weight map, every N tile width
    (("igemm_tc",), ("linear", 130, 256, 512), {"DMV_LINEAR_NTILE": "64"}),
    (("igemm_tc",), ("linear", 130, 256, 512), {"DMV_LINEAR_NTILE": "128"}),
    (("igemm_tc",), ("linear", 130, 256, 512), {"DMV_LINEAR_NTILE": "256"}),
]

# labels checked by other test files (or by the subprocess cases at the end of this file), with where
EXEMPT = {
    "sampler_fwd": "sampler tile kernel: test_sampler_loss_edges_gpu.py (4-byte offset source, C = 16, one-row images)",
    "sampler_fwd(tma)": "sampler TMA kernel, every window path: test_sampler_loss_edges_gpu.py::test_window_paths_match_the_oracle_and_the_tile_kernel",
    "sampler_grad_warp": "sampler tile kernel: test_sampler_loss_edges_gpu.py (4-byte offset source, C = 16, one-row images)",
    "sampler_grad_warp(tma)": "sampler TMA kernel, every window path: test_sampler_loss_edges_gpu.py::test_window_paths_match_the_oracle_and_the_tile_kernel",
    "sampler_box": "sampler grad_data pre-pass: test_sampler_loss_edges_gpu.py::test_sampler_grad_data_generic_channels, test_sampler_gpu.py",
    "sampler_grad_data": "sampler grad_data, C in {5, 7, 8} and one-row images: test_sampler_loss_edges_gpu.py, test_sampler_gpu.py",
    "sampler_loss_fused": "fused warp loss: test_sampler_loss_edges_gpu.py::test_fused_warp_loss_edges and the window-path cases",
    "loss_flat": "reconstruction loss: test_sampler_loss_edges_gpu.py::test_loss_flat_kernel and the block-cap case",
    "loss_fused": "single-view and view-fusion loss: test_sampler_loss_edges_gpu.py::test_loss_kernel_single_view, test_view_fusion_loss",
    "scale": "upstream loss scalar: test_layers_gpu.py::test_fused_loss",
    "u8_to_f32": "input pipeline: test_layers_gpu.py::test_u8_to_f32_matches_reference_division",
    "u8_crop_resize_bicubic": "input pipeline: test_input_pipeline.py",
    "act_fwd": "activations: test_layers_gpu.py::test_activations",
    "act_bwd": "activations: test_layers_gpu.py::test_activations",
    "cast_f32_to_bf16": "dtype casts: test_model_gpu.py (every model step)",
    "cast_bf16_to_f32": "dtype casts: test_model_gpu.py (every model step)",
    "set_flag": "graphed-step flags: test_model_gpu.py::test_train_step_decreases_loss_and_graph_replay_matches_eager",
    "adam_tick": "Adam step scalars to t = 100000: test_update_kernels_gpu.py::test_adam_tick_long_horizon",
    "adam_multi": "Adam value edges, bit-identical across forms: test_update_kernels_gpu.py; switches: test_adam_multi_under_its_switches below",
    "adam_scalar": "Adam scalar kernel (4-byte offset, n % 4 = 3 tail): test_update_kernels_gpu.py::test_adam_edges_bit_identical_across_implementations",
    "linear_wgrad_adam": "fused FC update, generic: test_update_kernels_gpu.py::test_adam_edges_bit_identical_across_implementations; switches below",
    "linear_wgrad_adam (stream)": "fused FC update, streaming: test_update_kernels_gpu.py::test_adam_edges_bit_identical_across_implementations; switches below",
    "dp_exchange_chunk": "data-parallel exchange on emulated ranks at its edges, refusals: test_update_kernels_gpu.py; test_dp_gpu.py",
}


def _row_id(row):
    labels, shape, env = row
    return "%s-%s%s" % (labels[0].replace(" ", "_"), "-".join(str(v) for v in shape if not isinstance(v, dict)),
                        "".join("-%s=%s" % kv for kv in sorted(env.items())))


def _run_row(shape):
    if shape[0] == "linear":
        return run_linear_fwd(*shape[1:])
    if shape[0] == "act_bwd_bias":
        return run_act_bwd_bias(*shape[1:])
    kind, op, B, H, W, cin, cout, kh, kw, s, opt = shape
    return run_layer(kind, op, B, H, W, cin, cout, kh, kw, s, y_bf16=opt.get("y_bf16", False), ws_bytes=opt.get("ws"))


def test_every_launch_label_has_a_form_case():
    """CPU: a kernel form cannot land without a parity case -- every check_launch label of csrc/ is a FORMS row or an
    exemption with its reason; stale rows / exemptions fail too."""
    labels = launch_labels()
    assert len(labels) > 40
    covered = {l for row in FORMS for l in row[0]}
    missing = sorted(labels - covered - set(EXEMPT))
    assert not missing, "launch labels without a FORMS row in tests/test_kernel_forms_gpu.py: %s" % missing
    stale = sorted((covered | set(EXEMPT)) - labels)
    assert not stale, "FORMS / EXEMPT name labels no kernel launches under: %s" % stale
    assert not covered & set(EXEMPT), "labels both covered and exempt: %s" % sorted(covered & set(EXEMPT))


@gpu
@pytest.mark.parametrize("row", FORMS, ids=[_row_id(r) for r in FORMS])
def test_kernel_form(row, monkeypatch):
    labels, shape, env = row
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ran = _run_row(shape)
    for l in labels:
        assert ran.get(l, 0) > 0, "form %r did not run; launches: %s" % (l, ran)


# --------------------------------------------------------------------------------------------------------------------
# GEOMETRY off the training graph, algo = auto: (kind, B, H, W, cin, cout, k, stride, {op: expected form})
# --------------------------------------------------------------------------------------------------------------------
HALO, PLANES, SUB, SUBE = "halo_tc", "halo_tc (parity planes)", "halo_tc (sub-pixel)", "halo_tc (sub-pixel, coalescing epilogue)"
GEOMETRY = [
    # non-square, both orientations, sizes that keep the specialised forms eligible
    ("conv", 2, 16, 40, 32, 32, 5, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo2d_tc"}),
    ("conv", 2, 40, 16, 32, 32, 5, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo2d_tc"}),
    ("conv", 2, 16, 40, 64, 64, 3, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo_tc"}),
    ("conv", 2, 40, 16, 64, 64, 3, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo_tc"}),
    ("conv", 2, 32, 48, 32, 32, 5, 2, {"fwd": PLANES, "dgrad": SUBE, "wgrad": "wgrad_s2_tc"}),
    ("conv", 2, 48, 32, 32, 32, 5, 2, {"fwd": PLANES, "dgrad": SUBE, "wgrad": "wgrad_s2_tc"}),
    ("deconv", 2, 32, 48, 32, 32, 5, 2, {"fwd": SUB, "dgrad": PLANES, "wgrad": "wgrad_s2_tc"}),
    ("deconv", 2, 48, 32, 32, 32, 5, 2, {"fwd": SUB, "dgrad": PLANES, "wgrad": "wgrad_s2_tc"}),
    ("conv", 2, 64, 96, 3, 32, 5, 2, {"fwd": "thin_conv", "wgrad": "thin_wgrad_mma"}),
    ("conv", 2, 96, 64, 3, 32, 5, 2, {"fwd": "thin_conv", "wgrad": "thin_wgrad_mma"}),
    ("deconv", 2, 64, 96, 32, 2, 5, 2, {"fwd": "thin_deconv", "dgrad": "thin_conv", "wgrad": "thin_wgrad_mma"}),
    ("deconv", 2, 96, 64, 32, 2, 5, 2, {"fwd": "thin_deconv", "dgrad": "thin_conv", "wgrad": "thin_wgrad_mma"}),
    # the thin single-kernel rule H/2 % 8 == 0 and W/2 % 16 == 0: passes at 48 x 32, fails at 48 x 40 (space-to-depth)
    ("conv", 1, 48, 32, 3, 32, 5, 2, {"fwd": "thin_conv", "wgrad": "thin_wgrad_mma"}),
    ("conv", 1, 48, 40, 3, 32, 5, 2, {"fwd": "thin_s2d_prep", "wgrad": "thin_s2d_gather"}),
    ("deconv", 1, 48, 40, 32, 2, 5, 2, {"fwd": SUB, "dgrad": "thin_s2d_prep", "wgrad": "thin_s2d_gather"}),
    # odd sizes: stride 2 over odd inputs, deconv to odd outputs, asymmetric SAME padding of k = 4
    ("conv", 2, 15, 16, 32, 32, 5, 2, {"fwd": "conv_f_simt", "dgrad": "igemm_tc", "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 16, 15, 32, 32, 5, 2, {"fwd": "conv_f_simt", "dgrad": "igemm_tc", "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 15, 15, 32, 32, 5, 2, {"fwd": "conv_f_simt", "dgrad": "igemm_tc", "wgrad": "conv_wgrad_simt"}),
    ("conv", 1, 31, 32, 32, 32, 5, 2, {"fwd": "conv_f_simt", "dgrad": SUBE, "wgrad": "conv_wgrad_simt"}),
    ("conv", 1, 32, 31, 16, 64, 3, 2, {"fwd": "conv_f_simt", "dgrad": SUB, "wgrad": "conv_wgrad_simt"}),
    ("deconv", 2, 15, 16, 32, 32, 5, 2, {"fwd": "igemm_tc", "dgrad": "conv_f_simt", "wgrad": "conv_wgrad_simt"}),
    ("deconv", 2, 7, 7, 64, 32, 5, 2, {"fwd": "igemm_tc", "dgrad": "conv_f_simt", "wgrad": "conv_wgrad_simt"}),
    ("deconv", 1, 31, 32, 32, 32, 5, 2, {"fwd": SUB, "dgrad": "conv_f_simt", "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 16, 16, 32, 32, 4, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo2d_tc"}),
    ("conv", 2, 32, 32, 32, 32, 4, 2, {"fwd": PLANES, "dgrad": SUBE, "wgrad": "wgrad_s2_tc"}),
    ("deconv", 2, 32, 32, 32, 32, 4, 2, {"fwd": SUB, "dgrad": PLANES, "wgrad": "wgrad_s2_tc"}),
    ("conv", 2, 16, 16, 64, 64, 4, 2, {"fwd": "igemm_tc", "dgrad": "igemm_tc", "wgrad": "wgrad_tc"}),
    # output area 255 (15 x 17) against 256 (16 x 16): the halo kernels need 256
    ("conv", 2, 15, 17, 32, 32, 3, 1, {"fwd": "igemm_tc", "dgrad": "igemm_tc", "wgrad": "wgrad_tc"}),
    ("conv", 2, 16, 16, 32, 32, 3, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo2d_tc"}),
    # sub-pixel n_real: 8 and 16 divide 16, 24 is not a multiple of 16, 48 is
    ("deconv", 1, 32, 32, 32, 8, 3, 2, {"fwd": SUB}),
    ("deconv", 1, 32, 32, 32, 16, 3, 2, {"fwd": SUB}),
    ("deconv", 1, 32, 32, 32, 24, 3, 2, {"fwd": "igemm_tc"}),
    ("deconv", 1, 32, 32, 32, 48, 3, 2, {"fwd": SUB}),
    # channel counts 16 and 48 (not multiples of 32) and 96 (a multiple of 32, not of 64)
    ("conv", 2, 16, 16, 16, 32, 3, 1, {"fwd": "conv_f_simt", "dgrad": HALO, "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 16, 16, 48, 32, 3, 1, {"fwd": "conv_f_simt", "dgrad": HALO, "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 16, 16, 32, 48, 3, 1, {"fwd": HALO, "dgrad": "conv_g_simt", "wgrad": "conv_wgrad_simt"}),
    ("conv", 2, 16, 16, 96, 32, 3, 1, {"fwd": "igemm_tc", "dgrad": HALO, "wgrad": "wgrad_tc"}),
    ("conv", 2, 16, 16, 32, 96, 3, 1, {"fwd": HALO, "dgrad": "igemm_tc", "wgrad": "wgrad_tc"}),
    # batch 1
    ("conv", 1, 16, 24, 32, 64, 5, 1, {"fwd": HALO, "dgrad": HALO, "wgrad": "wgrad_halo_tc"}),
    ("deconv", 1, 32, 40, 64, 32, 5, 2, {"fwd": SUB, "dgrad": "halo_tc (parity planes)", "wgrad": "wgrad_s2_tc"}),
]
GEOMETRY_CASES = [(g, op) for g in GEOMETRY for op in ("fwd", "dgrad", "wgrad") if op in g[-1]]


@gpu
@pytest.mark.parametrize("g,op", GEOMETRY_CASES, ids=["%s-%s-B%d-%dx%d-%d-%d-k%d-s%d" % ((g[0], op) + g[1:-1]) for g, op in GEOMETRY_CASES])
def test_geometry_off_the_training_graph(g, op):
    kind, B, H, W, cin, cout, k, s, expect = g
    ran = run_layer(kind, op, B, H, W, cin, cout, k, k, s, y_bf16=kind == "conv" and cin < 8)     # e0 writes bf16
    assert ran.get(expect[op], 0) > 0, "expected form %r, launches: %s" % (expect[op], ran)


# --------------------------------------------------------------------------------------------------------------------
# the graph's layer shapes under each fallback switch
# --------------------------------------------------------------------------------------------------------------------
# (kind, k, stride, cin, cout) of REF_LAYERS (test_layers_gpu.py) and SMALL (test_tc_gpu.py), at a reduced, non-square
# spatial size: 16 x 24 at stride 1, 32 x 64 at stride 2 (big side), which keeps the halo and thin forms eligible
GRAPH_LAYERS = [
    ("conv", 5, 2, 3, 32), ("conv", 5, 1, 32, 32), ("conv", 5, 2, 32, 64), ("conv", 5, 1, 64, 64), ("conv", 3, 2, 64, 128),
    ("conv", 3, 1, 128, 128), ("conv", 3, 2, 128, 256), ("conv", 3, 1, 256, 256), ("conv", 5, 1, 32, 64), ("conv", 3, 1, 32, 32),
    ("conv", 3, 1, 64, 64), ("conv", 5, 1, 64, 32), ("conv", 4, 1, 32, 32), ("conv", 3, 2, 32, 32), ("conv", 5, 2, 32, 32),
    ("conv", 3, 2, 32, 64),
    ("deconv", 3, 2, 256, 128), ("deconv", 3, 2, 128, 64), ("deconv", 5, 2, 64, 32), ("deconv", 5, 2, 32, 2), ("deconv", 3, 2, 64, 32),
    ("deconv", 5, 2, 32, 16), ("deconv", 5, 2, 64, 64), ("deconv", 5, 2, 32, 32), ("deconv", 3, 2, 32, 32), ("deconv", 3, 1, 32, 2),
]
SWITCHES = ["DMV_NO_HALO", "DMV_NO_WHALO", "DMV_NO_WHALO2D", "DMV_NO_WS2", "DMV_NO_S2D", "DMV_NO_D2S_EPI", "DMV_NO_NSPLIT",
            "DMV_NO_THIN_MMA", "DMV_NO_SUBPIXEL", "DMV_NO_S2HALO"]
_default_forms = {}


def _graph_layer_call(layer, op):
    kind, k, s, cin, cout = layer
    H, W = (16, 24) if s == 1 else (32, 64)
    thin_e0 = kind == "conv" and cin < 8
    return run_layer(kind, op, 1, H, W, cin, cout, k, k, s, y_bf16=thin_e0)


@gpu
@pytest.mark.parametrize("switch", SWITCHES)
@pytest.mark.parametrize("layer", GRAPH_LAYERS, ids=["%s-k%d-s%d-%d-%d" % l for l in GRAPH_LAYERS])
def test_graph_layer_under_fallback_switch(layer, switch, monkeypatch):
    """Forward, input gradient and weight + bias gradient of the layer with the switch set, against the oracle; a switch
    that leaves all three forms as they are is reported as a skip, not as a pass."""
    changed = []
    for op in ("fwd", "dgrad", "wgrad"):
        if (layer, op) not in _default_forms:
            _default_forms[(layer, op)] = set(_graph_layer_call(layer, op))
        monkeypatch.setenv(switch, "1")
        forms = set(_graph_layer_call(layer, op))          # checked against the oracle inside
        monkeypatch.delenv(switch)
        if forms != _default_forms[(layer, op)]:
            changed.append(op)
    if not changed:
        pytest.skip("%s does not change the form of any pass of this layer" % switch)


# --------------------------------------------------------------------------------------------------------------------
# update kernels under their once-per-process switches: one child process per setting
# --------------------------------------------------------------------------------------------------------------------
def _in_child(fn, env):
    """Runs ``fn`` of this module in a fresh interpreter with ``env`` added (the switches are read once per process) and
    waits for it; the child prints a verdict line when every check passed."""
    code = textwrap.dedent("""
        import sys
        sys.path[:0] = [%r, %r]
        import test_kernel_forms_gpu as t
        t.%s()
        print("form verdict: ok")
    """ % (ROOT, os.path.join(ROOT, "tests"), fn))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "form verdict: ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def child_fc_update():
    """dmv_linear_wgrad_adam under the process's DMV_FC_ADAM_* setting: M = 1, 8, 17, 64, a shape the streaming kernel
    takes (K % 32 == 0, N % 128 == 0, 15 tiles) and a tail shape it does not, grad_scale 0.3, two steps against
    T.adam_tf_step at the tolerances of test_layers_gpu.py::test_linear_wgrad_adam_fused."""
    from dynamic_multiview_3d_b200 import _lib
    stream_variant = os.environ.get("DMV_FC_ADAM_VARIANT", "9") == "9"
    st = torch.cuda.current_stream().cuda_stream
    gs = np.float32(0.3)
    for M in (1, 8, 17, 64):
        for K, N in ((160, 384), (72, 136)):
            rng = np.random.default_rng(M * 7 + K + N)
            theta = (rng.standard_normal((K, N)) * 0.05).astype(np.float32)
            th, m, v = torch.from_numpy(theta).cuda(), torch.zeros(K, N, device="cuda"), torch.zeros(K, N, device="cuda")
            half = torch.zeros(K, N, dtype=torch.bfloat16, device="cuda")
            dw = torch.empty(K, N, device="cuda")
            state = torch.tensor([1.0, 1.0, 0.0, 0.0], device="cuda")
            ref = (theta.copy(), np.zeros((K, N), np.float32), np.zeros((K, N), np.float32))
            label = "linear_wgrad_adam (stream)" if (stream_variant and K % 32 == 0 and N % 128 == 0) else "linear_wgrad_adam"
            for t in (1, 2):
                x = bf16_round(rng.standard_normal((M, K)))
                dy = bf16_round(rng.standard_normal((M, N)) * 10.0 ** rng.integers(-4, 0))
                xt, dyt = _dev(x, torch.bfloat16), _dev(dy, torch.bfloat16)
                n0 = _lib.launch_count_named(label)
                _lib.call("dmv_adam_tick", state.data_ptr(), 1e-3, 0.9, 0.999, st)
                _lib.call("dmv_linear_wgrad_adam", xt.data_ptr(), dyt.data_ptr(), th.data_ptr(), m.data_ptr(), v.data_ptr(), half.data_ptr(),
                          dw.data_ptr(), M, K, N, state.data_ptr(), 0.9, 0.999, 1e-8, float(gs), st)
                torch.cuda.synchronize()
                assert _lib.launch_count_named(label) == n0 + 1, (M, K, N, label)
                g = dw.cpu().numpy()
                gref = (x.astype(np.float64).T @ dy.astype(np.float64)).astype(np.float32)
                assert _rel(g, gref) < 1e-5, (M, K, N)
                ref = T.adam_tf_step(ref[0], (g * gs).astype(np.float32), ref[1], ref[2], t, 1e-3)
                assert _rel(m.cpu().numpy(), ref[1]) < 1e-6, (M, K, N, t)
                assert _rel(v.cpu().numpy(), ref[2]) < 1e-6, (M, K, N, t)
                assert float(np.abs(th.cpu().numpy() - ref[0]).max()) < 1e-6, (M, K, N, t)
                assert torch.equal(half, th.to(torch.bfloat16))


def _adam_call(name, ts, n, state, gs, st, gate=None):
    import ctypes as C
    from dynamic_multiview_3d_b200 import _lib
    arr = lambda key: (C.c_void_p * len(ts))(*[t[key].data_ptr() for t in ts])
    args = [arr("th"), arr("g"), arr("m"), arr("v"), arr("h"), (C.c_longlong * len(n))(*n), len(ts), state.data_ptr(), 0.9, 0.999, 1e-8, gs]
    _lib.call(name, *(args + ([gate.data_ptr()] if gate is not None else []) + [st]))


def child_adam_multi():
    """dmv_adam_multi over 30 tensors (two tables), sizes that are not multiples of 4 (scalar tails) and one tensor at a
    4-byte offset (all scalar), grad_scale 0.5, two steps against T.adam_tf_step; then dmv_adam_multi_gated: gate 0 leaves
    theta, m, v and the bf16 copy bit-unchanged, gate 1 is bit-equal to the ungated call."""
    from dynamic_multiview_3d_b200 import _lib
    rng = np.random.default_rng(5)
    st = torch.cuda.current_stream().cuda_stream
    sizes = [int(rng.integers(1, 3000)) for _ in range(28)] + [4096, 1]
    n0 = {l: _lib.launch_count_named(l) for l in ("adam_multi", "adam_scalar")}

    def make():
        ts = []
        for i, n in enumerate(sizes):
            th = torch.empty(n + 1, device="cuda")
            th = th[1:] if i == 3 else th[:n]                      # tensor 3 starts 4 bytes into its allocation
            th.copy_(torch.from_numpy((rng.standard_normal(n) * 0.1).astype(np.float32)))
            ts.append({"th": th, "g": torch.zeros(n, device="cuda"), "m": torch.zeros(n, device="cuda"), "v": torch.zeros(n, device="cuda"),
                       "h": torch.zeros(n, dtype=torch.bfloat16, device="cuda")})
        return ts

    ts = make()
    state = torch.tensor([1.0, 1.0, 0.0, 0.0], device="cuda")
    ref = [(t["th"].cpu().numpy().copy(), np.zeros(n, np.float32), np.zeros(n, np.float32)) for t, n in zip(ts, sizes)]
    for step in (1, 2):
        gs = [(rng.standard_normal(n) * 10.0 ** rng.integers(-5, 0)).astype(np.float32) for n in sizes]
        for t, g in zip(ts, gs):
            t["g"].copy_(torch.from_numpy(g))
        _lib.call("dmv_adam_tick", state.data_ptr(), 1e-3, 0.9, 0.999, st)
        _adam_call("dmv_adam_multi", ts, sizes, state, 0.5, st)
        torch.cuda.synchronize()
        ref = [T.adam_tf_step(r[0], (g * np.float32(0.5)).astype(np.float32), r[1], r[2], step, 1e-3) for r, g in zip(ref, gs)]
        # moments relative to their scale (the kernels contract m + (g - m)(1 - b1) into one FMA), theta to a thousandth of
        # one step, as test_layers_gpu.py::test_linear_wgrad_adam_fused
        for i, (t, (th, m, v)) in enumerate(zip(ts, ref)):
            assert _rel(t["m"].cpu().numpy(), m) < 1e-6, (i, step)
            assert _rel(t["v"].cpu().numpy(), v) < 1e-6, (i, step)
            assert float(np.abs(t["th"].cpu().numpy() - th).max()) < 1e-6, (i, step)
            assert torch.equal(t["h"], t["th"].to(torch.bfloat16)), (i, step)
    assert _lib.launch_count_named("adam_multi") >= n0["adam_multi"] + 4, "30 tensors must take two tables per step"
    assert _lib.launch_count_named("adam_scalar") > n0["adam_scalar"]
    # gated: a gate of 0 changes nothing, a gate of 1 is the ungated update
    snap = lambda ts: [{k: t[k].clone() for k in ("th", "m", "v", "h")} for t in ts]
    before = snap(ts)
    gate = torch.zeros(1, dtype=torch.int32, device="cuda")
    _adam_call("dmv_adam_multi_gated", ts, sizes, state, 0.5, st, gate)
    torch.cuda.synchronize()
    for t, b in zip(ts, before):
        for k in b:
            assert torch.equal(t[k], b[k]), "gate 0 changed %s" % k
    twin = snap(ts)
    twin = [dict(d, g=t["g"]) for d, t in zip(twin, ts)]
    gate.fill_(1)
    _adam_call("dmv_adam_multi_gated", ts, sizes, state, 0.5, st, gate)
    _adam_call("dmv_adam_multi", twin, sizes, state, 0.5, st)
    torch.cuda.synchronize()
    for t, u in zip(ts, twin):
        for k in ("th", "m", "v", "h"):
            assert torch.equal(t[k], u[k]), "gate 1 differs from the ungated update in %s" % k


def child_igemm_smem2():
    """A narrow deep layer (64 output channels: the two-per-SM igemm form) with its budget forced down to 2 stages."""
    ran = run_layer("conv", "fwd", 2, 7, 7, 256, 64, 3, 3, 1)
    assert ran.get("igemm_tc", 0) > 0, ran


@gpu
@pytest.mark.parametrize("env", [{"DMV_FC_ADAM_VARIANT": "0"}, {"DMV_FC_ADAM_VARIANT": "1"}, {"DMV_FC_ADAM_VARIANT": "4"},
                                 {"DMV_FC_ADAM_VARIANT": "9", "DMV_FC_ADAM_STAGES": "2"}, {"DMV_FC_ADAM_VARIANT": "9", "DMV_FC_ADAM_STAGES": "3"},
                                 {"DMV_FC_ADAM_VARIANT": "9", "DMV_FC_ADAM_CTAS": "1"}, {"DMV_FC_ADAM_VARIANT": "9", "DMV_FC_ADAM_CTAS": "5"}],
                         ids=lambda e: "-".join("%s=%s" % kv for kv in sorted(e.items())))
def test_fc_update_under_its_switches(env):
    _in_child("child_fc_update", env)


@gpu
@pytest.mark.parametrize("env", [{}, {"DMV_ADAM_CTAS": "1"}], ids=["default", "DMV_ADAM_CTAS=1"])
def test_adam_multi_under_its_switches(env):
    _in_child("child_adam_multi", env)


@gpu
def test_igemm_two_per_sm_at_two_stages():
    _in_child("child_igemm_smem2", {"DMV_IGEMM_SMEM2_KB": "32"})

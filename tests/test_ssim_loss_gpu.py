"""The SSIM + L1 photometric loss (include/dmv3d.h, csrc/loss.cu):
  loss = inv_count * sum_{n,p} sum_c w_c * (alpha * (1 - SSIM_p,c) / 2 + (1 - alpha) * |gen - target|)
with a 3x3 SSIM window over images reflection-padded by one pixel.

CPU: a float64 torch restatement of the definition (autograd gives the gradient) pinned by known answers, a float64
restatement of the kernels' per-window coefficient scheme checked against it, the model surface and the refusals.
GPU: the kernel against the oracle, launch counts and refusals, and the models' training step with loss = 'ssim' (the
sampler, this loss and the sampler's flow gradient: the loss has no fused warp form)."""
import ctypes

import numpy as np
import pytest
import torch

from test_sampler_loss_edges_gpu import _Counts

gpu = pytest.mark.gpu
E_INVALID_ARG, E_ALIGN, E_UNSUPPORTED_SHAPE, E_WORKSPACE = -1, -2, -3, -5
C1, C2 = 0.01 ** 2, 0.03 ** 2
CLASSES = ["AppearanceFlowModel", "AppFlowHighDimAngle", "AppFlowLowDimAngle", "AppearanceFlowTinghui"]
WEIGHTS = {1: [0.7], 3: [0.5, 1.0, 1.7], 4: [1.0, 0.3, 0.1, 2.5]}


# ------------------------------------------------------------------------------------------------------- the oracle
def ssim_map(x, y):
    """SSIM per pixel of [N, H, W, C] float64 tensors: 3x3 windows over the reflection-padded images (Monodepth2's SSIM
    module without its clamp)."""
    xp = torch.nn.functional.pad(x.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="reflect")
    yp = torch.nn.functional.pad(y.permute(0, 3, 1, 2), (1, 1, 1, 1), mode="reflect")
    pool = lambda t: torch.nn.functional.avg_pool2d(t, 3, 1)
    mx, my = pool(xp), pool(yp)
    sxx = pool(xp * xp) - mx * mx
    syy = pool(yp * yp) - my * my
    sxy = pool(xp * yp) - mx * my
    s = (2 * mx * my + C1) * (2 * sxy + C2) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
    return s.permute(0, 2, 3, 1)


def oracle(gen, target, alpha, weights, inv_count):
    """(loss, d loss / d gen) in float64; gen, target [..., H, W, C] arrays."""
    shp = gen.shape
    x = torch.tensor(np.asarray(gen, np.float64).reshape((-1,) + shp[-3:]), requires_grad=True)
    y = torch.tensor(np.asarray(target, np.float64).reshape((-1,) + shp[-3:]))
    w = torch.tensor(np.asarray(weights, np.float64))
    per = alpha * (1 - ssim_map(x, y)) / 2 + (1 - alpha) * (x - y).abs()
    loss = (per * w).sum() * inv_count
    loss.backward()
    return float(loss.detach()), x.grad.numpy().reshape(shp)


def coefficient_scheme(gen, target, alpha, weights, inv_count):
    """The kernels' gradient in float64: per window q the coefficients (P, Q, R) with d loss_q / d slot k = P + Q x_k + R y_k,
    summed at each pixel over the 3x3 windows around it and over the windows that reach it through the reflection."""
    N, H, W, C = gen.shape
    x, y = np.asarray(gen, np.float64), np.asarray(target, np.float64)
    pad = lambda a: np.pad(a, ((0, 0), (1, 1), (1, 1), (0, 0)), mode="reflect")
    xp, yp = pad(x), pad(y)
    win = lambda a: sum(a[:, du:du + H, dv:dv + W] for du in range(3) for dv in range(3)) / 9
    mx, my = win(xp), win(yp)
    vx, vy, cxy = win(xp * xp) - mx * mx, win(yp * yp) - my * my, win(xp * yp) - mx * my
    A1, A2, B1, B2 = 2 * mx * my + C1, 2 * cxy + C2, mx * mx + my * my + C1, vx + vy + C2
    S = A1 * A2 / (B1 * B2)
    dmu = 2 * (my * A2 - mx * S * B2) / (B1 * B2)
    dvx, dcv = -S / B2, 2 * A1 / (B1 * B2)
    gk = -alpha / 2 * np.asarray(weights) * inv_count / 9
    P, Q, R = gk * (dmu - 2 * dvx * mx - dcv * my), gk * 2 * dvx, gk * dcv
    # d/d padded slot, then fold the padded ring onto the pixels it reflects
    gp = np.zeros_like(xp)
    for du in range(3):
        for dv in range(3):
            gp[:, du:du + H, dv:dv + W] += P + Q * xp[:, du:du + H, dv:dv + W] + R * yp[:, du:du + H, dv:dv + W]
    g = gp[:, 1:-1, 1:-1].copy()
    rows, cols = np.r_[1, np.arange(H), H - 2], np.r_[1, np.arange(W), W - 2]
    for a in range(H + 2):
        for b in range(W + 2):
            if 1 <= a <= H and 1 <= b <= W:
                continue
            g[:, rows[a], cols[b]] += gp[:, a, b]
    return g + (1 - alpha) * np.asarray(weights) * inv_count * np.sign(x - y)


def _images(rng, N, H, W, C):
    g = rng.random((N, H, W, C))
    t = np.clip(g + 0.2 * rng.standard_normal(g.shape), 0, 1)
    return g.astype(np.float32), t.astype(np.float32)


# ------------------------------------------------------------------------------------------------- CPU: the oracle
def test_identical_images_have_zero_loss():
    g, _ = _images(np.random.default_rng(0), 2, 9, 7, 3)
    loss, grad = oracle(g, g, 0.85, [1, 1, 1], 1.0)
    assert abs(loss) < 1e-12 and np.abs(grad).max() < 1e-9


def test_alpha_zero_is_l1():
    g, t = _images(np.random.default_rng(1), 2, 6, 5, 3)
    w, inv = [0.5, 1.0, 2.0], 1 / 60
    loss, grad = oracle(g, t, 0.0, w, inv)
    d = g.astype(np.float64) - t
    assert np.isclose(loss, (np.abs(d) * w).sum() * inv, rtol=1e-12)
    assert np.allclose(grad, np.sign(d) * w * inv, rtol=1e-12, atol=0)


def test_constant_images_have_the_closed_form():
    a, b, alpha = 0.3, 0.7, 0.85
    g, t = np.full((2, 5, 4, 1), a), np.full((2, 5, 4, 1), b)
    s = (2 * a * b + C1) / (a * a + b * b + C1)              # zero variances: the C2 factors cancel
    loss, _ = oracle(g, t, alpha, [1.0], 1 / 40)
    assert np.isclose(loss, alpha * (1 - s) / 2 + (1 - alpha) * abs(a - b), rtol=1e-12)


@pytest.mark.parametrize("H,W", [(2, 2), (3, 3), (2, 3)])
def test_reflection_at_the_smallest_images_matches_a_hand_padded_computation(H, W):
    rng = np.random.default_rng(H * 10 + W)
    g, t = rng.random((1, H, W, 1)), rng.random((1, H, W, 1))
    ri, rj = [1] + list(range(H)) + [H - 2], [1] + list(range(W)) + [W - 2]
    total = 0.0
    for i in range(H):
        for j in range(W):
            xs = [g[0, ri[i + a], rj[j + b], 0] for a in range(3) for b in range(3)]
            ys = [t[0, ri[i + a], rj[j + b], 0] for a in range(3) for b in range(3)]
            mx, my = np.mean(xs), np.mean(ys)
            sxx = np.mean(np.square(xs)) - mx * mx
            syy = np.mean(np.square(ys)) - my * my
            sxy = np.mean(np.multiply(xs, ys)) - mx * my
            s = (2 * mx * my + C1) * (2 * sxy + C2) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
            total += 0.85 * (1 - s) / 2 + 0.15 * abs(g[0, i, j, 0] - t[0, i, j, 0])
    loss, _ = oracle(g, t, 0.85, [1.0], 1.0)
    assert np.isclose(loss, total, rtol=1e-12)


def test_finite_differences_agree_with_the_gradient():
    rng = np.random.default_rng(5)
    g, t = rng.random((1, 4, 5, 2)), rng.random((1, 4, 5, 2))
    _, grad = oracle(g, t, 0.85, [1.0, 0.5], 1.0)
    h = 1e-6
    for idx in [(0, 0, 0, 0), (0, 1, 2, 1), (0, 3, 4, 0), (0, 2, 0, 1), (0, 0, 3, 1)]:
        gp, gm = g.copy(), g.copy()
        gp[idx] += h
        gm[idx] -= h
        fd = (oracle(gp, t, 0.85, [1.0, 0.5], 1.0)[0] - oracle(gm, t, 0.85, [1.0, 0.5], 1.0)[0]) / (2 * h)
        assert abs(fd - grad[idx]) < 1e-7, (idx, fd, grad[idx])


@pytest.mark.parametrize("H,W", [(2, 2), (3, 3), (2, 5), (7, 4), (11, 9)])
def test_the_kernels_coefficient_scheme_matches_autograd(H, W):
    """The per-window (P, Q, R) coefficients and the reflection fold the kernels use give the oracle's gradient."""
    rng = np.random.default_rng(H * W)
    g, t = rng.random((2, H, W, 3)), rng.random((2, H, W, 3))
    w = WEIGHTS[3]
    _, grad = oracle(g, t, 0.85, w, 0.01)
    assert np.allclose(coefficient_scheme(g, t, 0.85, w, 0.01), grad, rtol=1e-10, atol=1e-14)


# --------------------------------------------------------------------------------------------- CPU: model surface
def _conf(B, H=64, V=19, **kw):
    c = {"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": V, "seed": 3}
    c.update(kw)
    return c


@pytest.mark.parametrize("cls", CLASSES + ["Base_Prediction_Model"])
def test_ssim_changes_neither_the_inputs_nor_the_variables(cls):
    import dynamic_multiview_3d_b200 as pkg
    extra = {"use_color": "", "use_depth": "", "depth_lr_factor": 0.1} if cls == "Base_Prediction_Model" else {}
    M = getattr(pkg, cls)
    for kw in ({}, {"num_targets": 3}):
        ref = M(_conf(2, **extra, **kw), device="meta")
        ssim = M(_conf(2, loss="ssim", ssim_alpha=0.5, **extra, **kw), device="meta")
        assert ssim.input_spec() == ref.input_spec()
        shapes = lambda m: [(k, tuple(v.shape), v.trainable) for k, v in m.store.vars.items()]
        assert shapes(ssim) == shapes(ref)
        assert ssim.ssim_alpha == 0.5 and ref.ssim_alpha == 0.85


@pytest.mark.parametrize("cls", CLASSES)
def test_ssim_with_several_views_is_refused_by_name(cls):
    import dynamic_multiview_3d_b200 as pkg
    with pytest.raises(ValueError, match=cls):
        getattr(pkg, cls)(_conf(2, loss="ssim", num_views=2), device="meta")


def test_multiview_fusion_model_refuses_ssim_by_name():
    import dynamic_multiview_3d_b200 as pkg
    with pytest.raises(ValueError, match="MultiViewFusionAppFlow"):
        pkg.MultiViewFusionAppFlow(_conf(2, loss="ssim"), device="meta")


def test_ssim_l1_loss_refuses_a_mask():
    from dynamic_multiview_3d_b200 import functional as F
    z = torch.zeros((1, 4, 4, 3))
    with pytest.raises(ValueError, match="mask"):
        F.ssim_l1_loss(z, z, mask=torch.ones((1, 4, 4, 1)))
    with pytest.raises(ValueError, match="mask"):
        F.reconstruction_loss(z, z, "ssim", mask=torch.ones((1, 4, 4, 1)))


def test_the_fused_warp_loss_never_applies_to_ssim():
    from dynamic_multiview_3d_b200 import functional as F
    data, flow = torch.zeros((1, 8, 4, 4)), torch.zeros((1, 8, 4, 2))
    assert F.warp_loss_supported(data, flow, mode="l1") and F.warp_loss_supported(data, flow)
    assert not F.warp_loss_supported(data, flow, mode="ssim")


# ------------------------------------------------------------------------------------------------------ GPU helpers
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _loss_ws(pixels):
    return torch.zeros(int(_lib().dmv_loss_workspace_size(pixels)), dtype=torch.uint8, device="cuda")


def ssim_raw(gen, target, weights, alpha, inv, grad=True, grad_buf=None, ws=None):
    """dmv_ssim_loss_fwd_bwd through the C ABI: (rc, loss, grad_gen)."""
    B, H, W, C = gen.shape
    ws = _loss_ws(B * H * W) if ws is None else ws
    loss = torch.empty((), dtype=torch.float32, device="cuda")
    gg = grad_buf if grad_buf is not None else (torch.empty_like(gen) if grad else None)
    w = (ctypes.c_float * C)(*weights)
    rc = _lib().dmv_ssim_loss_fwd_bwd(_ptr(gen), _ptr(target), w, float(alpha), float(inv), _ptr(loss), _ptr(gg), B, H, W, C, _ptr(ws),
                                      ws.numel(), _stream())
    return rc, loss, gg


def _np(t):
    return t.detach().cpu().numpy()


# ----------------------------------------------------------------------------------- GPU: standalone kernel vs oracle
# float32 tolerances.  The loss sums O(1) per-pixel terms into a double per CTA: 1e-5 relative.  The gradient forms
# s_xx = E[x^2] - mu^2 in float32: for a window of values ~1 with a variance ~1e-2 the subtraction loses ~2 decimal
# digits (cancellation of 1 against 1e-2), and dS/ds_xx carries 1 / (s_xx + s_yy + C2), so an element may be off by
# ~1e-7 * 100 relative to the largest gradient: 2e-4 of max |grad| bounds it with a margin.
GRAD_TOL = 2e-4

SHAPES = [(3, 2, 2), (2, 3, 3), (2, 33, 61), (1, 61, 33), (2, 224, 224), (1, 2, 61), (5, 61, 2), (40, 40, 70)]


@gpu
@pytest.mark.parametrize("C", [1, 3, 4])
@pytest.mark.parametrize("alpha", [0.0, 0.85, 1.0])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_standalone_kernel_matches_the_oracle(shape, alpha, C):
    B, H, W = shape
    rng = np.random.default_rng(B * 1000 + H * 10 + W + C)
    g, t = _images(rng, B, H, W, C)
    w, inv = WEIGHTS[C], 1.0 / (B * H * W)
    ref_loss, ref_grad = oracle(g, t, alpha, w, inv)
    gen, tgt = _cuda(g), _cuda(t)
    with _Counts("loss_fused") as n:
        rc, loss, gg = ssim_raw(gen, tgt, w, alpha, inv)
    assert rc == 0 and n.d["loss_fused"] == 1
    assert abs(float(loss) - ref_loss) <= 1e-5 * abs(ref_loss) + 1e-7, (float(loss), ref_loss)
    err = np.abs(_np(gg) - ref_grad).max()
    assert err <= GRAD_TOL * np.abs(ref_grad).max() + 1e-12, (err, np.abs(ref_grad).max())
    # bit-reproducible; the loss-only pass gives the same loss and writes no gradient
    rc2, loss2, gg2 = ssim_raw(gen, tgt, w, alpha, inv)
    assert rc2 == 0 and torch.equal(loss, loss2) and torch.equal(gg, gg2)
    gg.fill_(7.25)                                   # the earlier call's gradient buffer as a sentinel
    rc3, loss3, none = ssim_raw(gen, tgt, w, alpha, inv, grad=False)
    torch.cuda.synchronize()
    assert rc3 == 0 and none is None and torch.equal(loss, loss3) and bool((gg == 7.25).all())


@gpu
def test_standalone_kernel_with_more_tiles_than_ctas():
    """3136 tiles at 64 x 224^2 over at most 1184 CTAs: every CTA walks several tiles."""
    rng = np.random.default_rng(3)
    g, t = _images(rng, 64, 224, 224, 3)
    inv = 1.0 / (64 * 224 * 224)
    ref_loss, ref_grad = oracle(g, t, 0.85, WEIGHTS[3], inv)
    rc, loss, gg = ssim_raw(_cuda(g), _cuda(t), WEIGHTS[3], 0.85, inv)
    assert rc == 0 and abs(float(loss) - ref_loss) <= 1e-5 * ref_loss
    assert np.abs(_np(gg) - ref_grad).max() <= GRAD_TOL * np.abs(ref_grad).max()


@gpu
def test_functional_ssim_l1_loss_op():
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(4)
    g, t = _images(rng, 6, 33, 20, 3)
    gen = _cuda(g).reshape(2, 3, 33, 20, 3).requires_grad_(True)
    loss = F.ssim_l1_loss(gen, _cuda(t).reshape(2, 3, 33, 20, 3), alpha=0.85)
    (2.5 * loss).backward()
    ref_loss, ref_grad = oracle(g, t, 0.85, [1, 1, 1], 1.0 / (6 * 33 * 20))
    assert abs(float(loss.detach()) - ref_loss) <= 1e-5 * ref_loss
    gr = _np(gen.grad).reshape(g.shape)
    assert np.abs(gr - 2.5 * ref_grad).max() <= GRAD_TOL * 2.5 * np.abs(ref_grad).max()
    with torch.no_grad():
        assert torch.equal(F.reconstruction_loss(gen.detach(), _cuda(t).reshape(gen.shape), "ssim", alpha=0.85), loss.detach())


@gpu
def test_standalone_refusals_launch_nothing():
    lib = _lib()
    g = torch.zeros((2, 8, 8, 3), device="cuda")
    ws = torch.zeros(int(lib.dmv_loss_workspace_size(128)) + 16, dtype=torch.uint8, device="cuda")
    loss = torch.empty((), device="cuda")
    w = (ctypes.c_float * 4)(1, 1, 1, 1)
    s = _stream()
    cases = [
        ((None, _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws), ws.numel(), s), E_INVALID_ARG),
        ((_ptr(g), _ptr(g), w, 1.5, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws), ws.numel(), s), E_INVALID_ARG),
        ((_ptr(g), _ptr(g), w, -0.1, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws), ws.numel(), s), E_INVALID_ARG),
        ((_ptr(g), _ptr(g), w, float("nan"), 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws), ws.numel(), s), E_INVALID_ARG),
        ((_ptr(g), _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 2, _ptr(ws), ws.numel(), s), E_UNSUPPORTED_SHAPE),
        ((_ptr(g), _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 1, 8, 3, _ptr(ws), ws.numel(), s), E_UNSUPPORTED_SHAPE),
        ((_ptr(g), _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 8, 1, 3, _ptr(ws), ws.numel(), s), E_UNSUPPORTED_SHAPE),
        ((_ptr(g), _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws), 8, s), E_WORKSPACE),
        ((_ptr(g), _ptr(g), w, 0.85, 1.0, _ptr(loss), _ptr(g), 2, 8, 8, 3, _ptr(ws) + 4, ws.numel() - 8, s), E_ALIGN),
    ]
    torch.cuda.synchronize()
    n0 = lib.dmv_launch_count()
    for args, code in cases:
        assert lib.dmv_ssim_loss_fwd_bwd(*args) == code, args
    torch.cuda.synchronize()
    assert lib.dmv_launch_count() == n0


@gpu
def test_existing_warp_loss_entry_points_still_refuse_ssim_as_a_mode():
    lib = _lib()
    B, H, W, C = 1, 8, 8, 4
    t = torch.zeros((B, H, W, C), device="cuda")
    f = torch.zeros((B, H, W, 2), device="cuda")
    loss = torch.empty((), device="cuda")
    ws = torch.zeros(int(lib.dmv_sampler_loss_workspace_size(B, H, W)), dtype=torch.uint8, device="cuda")
    w = (ctypes.c_float * 4)(1, 1, 1, 1)
    rc = lib.dmv_sampler_loss_fused(_ptr(t), _ptr(f), _ptr(t), w, 2, 1.0, _ptr(t), _ptr(f), _ptr(loss), B, H, W, C, H, W, 1, _ptr(ws),
                                    ws.numel(), _stream())
    assert rc == E_INVALID_ARG


# --------------------------------------------------------------------------------------------------- GPU: models
def _batch(model, B, H, seed=1234, T=1):
    from dynamic_multiview_3d_b200.synthetic import make_batch
    b = make_batch(B, H, "onehot19" if model.viewpoint_dim == 19 else "disp2", seed=seed, depth=True, targets=T)
    return {k: torch.from_numpy(b[k]).cuda() for k in model.INPUT_KEYS}


def _grads(m):
    return {k: v.grad.clone() for k, v in m.store.vars.items() if v.trainable and v.grad is not None}


@gpu
@pytest.mark.parametrize("T", [1, 3])
@pytest.mark.parametrize("cls", CLASSES)
def test_model_step_is_the_explicit_composition(cls, T):
    """loss = 'ssim' trains through the sampler, ssim_l1_loss and the sampler's flow gradient: the step's loss and every
    parameter gradient are those of the explicit calls on a twin model, bit for bit; the loss is the oracle's on the model's
    own gen; the validation pass takes the loss-only mode and gives the same loss."""
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import functional as F
    m = getattr(pkg, cls)(_conf(2, loss="ssim", ssim_alpha=0.8, num_targets=T))
    twin = getattr(pkg, cls)(_conf(2, loss="ssim", ssim_alpha=0.8, num_targets=T))
    batch = _batch(m, 2, 64, T=T)
    with _Counts("sampler_loss_fused", "loss_fused") as n:
        loss = m.step_loss(batch)
        loss.backward()
    assert n.d == {"sampler_loss_fused": 0, "loss_fused": 1}, n.d
    out = twin.forward(batch["image0"], batch["disp"])
    img1 = batch["image1"]
    ref = F.ssim_l1_loss(out["gen"], img1, alpha=0.8, inv_count=1.0 / (img1.numel() // 3), unit_upstream=True)
    ref.backward()
    assert torch.equal(loss.detach(), ref.detach())
    g, gt = _grads(m), _grads(twin)
    assert g.keys() == gt.keys() and len(g) > 10
    for k in g:
        assert torch.equal(g[k], gt[k]), k
    lo, _ = oracle(_np(m.gen), _np(img1), 0.8, [1, 1, 1], 1.0 / (img1.numel() // 3))
    assert abs(float(loss.detach()) - lo) <= 1e-5 * abs(lo)
    with _Counts("loss_fused") as n:
        val = m.eval_loss(batch)
    assert n.d["loss_fused"] == 1 and torch.equal(val, loss.detach())


@gpu
@pytest.mark.parametrize("head", ["tanh", "flow"])
def test_base_prediction_model_loss_is_the_oracle_on_its_outputs(head):
    import dynamic_multiview_3d_b200 as pkg
    m = pkg.Base_Prediction_Model(_conf(2, loss="ssim", ssim_alpha=0.7, use_color="", use_depth="", depth_lr_factor=0.1, head=head))
    batch = _batch(m, 2, 64)
    with torch.no_grad():
        loss = float(m.step_loss(batch))
    n = 2 * 64 * 64
    lc, _ = oracle(_np(m.gen_image1), _np(batch["image1"]), 0.7, [1, 1, 1], 1.0 / n)
    ld, _ = oracle(_np(m.gen_dimage1), _np(batch["depth1"]), 0.7, [0.1], 1.0 / n)
    assert abs(loss - (lc + ld)) <= 1e-5 * abs(lc + ld), (loss, lc + ld)


@gpu
def test_graphed_ssim_step_equals_eager_with_a_deferred_update():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    out = {}
    for graphed in (False, True):
        m = pkg.AppearanceFlowModel(_conf(4, loss="ssim", seed=9))
        red = data_parallel.attach(m, bucket_mb=4.0)
        assert sorted(red.var_wait), "no deferred update"
        batch = _batch(m, 4, 64)
        step = GraphedTrainStep(m, warmup=2) if graphed else m.train_step
        losses = [float(step(batch)) for _ in range(3)]
        val = float(m.eval_loss(batch))
        out[graphed] = (losses, val, m.state_dict())
    assert out[True][0] == out[False][0] and out[True][1] == out[False][1]
    for k, t in out[False][2].items():
        assert torch.equal(t, out[True][2][k]), k


@gpu
def test_ssim_training_lowers_the_loss():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    m = pkg.AppearanceFlowModel(_conf(8, loss="ssim", learning_rate=1e-4, seed=1))
    batch = _batch(m, 8, 64)
    step = GraphedTrainStep(m, warmup=2)
    losses = [float(step(batch)) for _ in range(50)]
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < 0.9 * np.mean(losses[:5]), losses


@gpu
def test_train_main_with_ssim_validates_checkpoints_and_resumes(tmp_path, monkeypatch):
    import json
    from dynamic_multiview_3d_b200 import train
    monkeypatch.setattr(train, "VAL_INTERVAL", 3)
    monkeypatch.setattr(train, "SAVE_INTERVAL", 4)
    monkeypatch.setattr(train, "SUMMARY_INTERVAL", 2)
    conf_py = tmp_path / "conf.py"
    conf_py.write_text(
        "import os\ncurrent_dir = os.path.dirname(os.path.realpath(__file__))\n"
        "from appearance_flow_model import AppearanceFlowModel\n"
        "configuration = {'experiment_name': 'x', 'data_dir': '/nope', 'output_dir': current_dir + '/modeldata',\n"
        " 'current_dir': current_dir, 'num_iterations': 6, 'batch_size': 4, 'learning_rate': 1e-4, 'loss': 'ssim',\n"
        " 'image_size': 64, 'viewpoint_dim': 19, 'train_val_split': 0.95, 'model': AppearanceFlowModel}\n")
    train.main(["--hyper", str(conf_py)])
    out = tmp_path / "modeldata"
    assert (out / "model4").exists() and (out / "model").exists()
    rows = [json.loads(l) for l in open(out / "scalars.jsonl")]
    assert {"training_loss", "val_loss"} <= {r["tag"] for r in rows}
    assert all(np.isfinite(r["value"]) for r in rows)
    (out / "model").unlink()
    train.main(["--hyper", str(conf_py), "--pretrained", str(out / "model4")])
    assert (out / "model").exists()

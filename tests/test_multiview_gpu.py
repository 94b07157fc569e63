"""Several source views per target in the single-view flow models: the fused multi-view warp loss
(dmv_sampler_fuse_views_loss), its operators, the num_views graph of the four appearance-flow classes, and the driver
around it.

- the kernel gives the bits of the composition it replaces (the sampler per view, dmv_loss_fused_fwd_bwd with the
  logits, the sampler's flow gradient on its grad_gen) for fused_out and all three channels of grad_head, on every
  window path, both grid orders and absolute warps, L1 and L2, 1..8 views, C in {1, 3, 4}, logit and flow edges; the
  loss agrees within 1e-6 and repeats bit for bit; a float64 NumPy restatement anchors the semantics;
- one launch under the sampler_loss_fused label, nothing else; refusals launch nothing;
- a model step with num_views = 3 gives the explicit composition's loss and bit-equal parameter gradients; num_views = 1
  is the plain model; the captured step, the loss over training, train.main and the data-parallel step work.
input_spec, the variables, the refusals and the synthetic batches need no GPU."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_sampler_loss_edges_gpu import CATEGORIES, _assert_paths, _Counts, path_warp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ADD_GRID, GRID_XY = 1, 2
E_INVALID_ARG, E_ALIGN, E_UNSUPPORTED_SHAPE, E_WORKSPACE = -1, -2, -3, -5
LOSS = {"l2": 0, "l1": 1}
FLAGS = [0, ADD_GRID, ADD_GRID | GRID_XY]
FLAG_IDS = ["absolute", "ref_yx", "xy"]
CLASSES = ["AppearanceFlowModel", "AppFlowHighDimAngle", "AppFlowLowDimAngle", "AppearanceFlowTinghui"]
WEIGHTS = {1: [0.7], 3: [0.5, 1.0, 1.7], 4: [1.0, 0.3, 0.1, 2.5]}
LABELS = ("sampler_loss_fused", "sampler_fwd(tma)", "sampler_fwd", "loss_fused", "loss_flat", "sampler_grad_warp(tma)",
          "sampler_grad_warp")


def _conf(B, H=64, V=19, **kw):
    c = {"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": V, "seed": 3}
    c.update(kw)
    return c


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("cls", CLASSES)
def test_input_spec_and_variables_with_and_without_num_views(cls):
    import dynamic_multiview_3d_b200 as pkg
    one = getattr(pkg, cls)(_conf(2), device="meta")
    same = getattr(pkg, cls)(_conf(2, num_views=1), device="meta")
    three = getattr(pkg, cls)(_conf(2, num_views=3), device="meta")
    assert one.input_spec() == same.input_spec() == {"image0": (2, 64, 64, 3), "image1": (2, 64, 64, 3), "disp": (2, 19)}
    assert three.input_spec() == {"image0": (3, 2, 64, 64, 3), "image1": (2, 64, 64, 3), "disp": (3, 2, 19)}
    shapes = lambda m: {k: tuple(v.shape) for k, v in m.store.vars.items()}
    assert list(shapes(one)) == list(shapes(three)) and shapes(one) == shapes(same)
    diff = {k for k, s in shapes(one).items() if s != shapes(three)[k]}
    assert diff == {"flow_field/w"}
    w1, w3 = shapes(one)["flow_field/w"], shapes(three)["flow_field/w"]
    assert w1[2] == 2 and w3[2] == 3 and w1[:2] + w1[3:] == w3[:2] + w3[3:]
    assert tuple(three.flow_field.shape) == (3, 2, 64, 64, 2) and tuple(three.confidence.shape) == (3, 2, 64, 64)
    assert tuple(three.gen.shape) == (2, 64, 64, 3)


@pytest.mark.parametrize("cls", CLASSES)
def test_num_views_refusals_name_the_class(cls):
    import dynamic_multiview_3d_b200 as pkg
    M = getattr(pkg, cls)
    with pytest.raises(ValueError, match=cls):
        M(_conf(2, num_views=9), device="meta")
    with pytest.raises(ValueError, match=cls):
        M(_conf(2, num_views=2, num_targets=2), device="meta")
    m = M(_conf(2, num_views=2), device="meta")
    with pytest.raises(NotImplementedError, match=cls):
        m.render({"image0": torch.zeros((2, 64, 64, 3), device="meta")}, torch.zeros((2, 19), device="meta"))
    M(_conf(2, num_views=8), device="meta")


def test_base_prediction_model_refuses_several_views():
    import dynamic_multiview_3d_b200 as pkg
    with pytest.raises(ValueError, match="Base_Prediction_Model"):
        pkg.Base_Prediction_Model(_conf(2, use_color="", num_views=2), device="meta")
    pkg.Base_Prediction_Model(_conf(2, use_color="", num_views=1), device="meta")


def test_tfrecords_refuse_several_views(tmp_path, monkeypatch):
    from dynamic_multiview_3d_b200 import train
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", os.environ.get("CUDA_VISIBLE_DEVICES", "0"))
    conf_py = tmp_path / "conf.py"
    conf_py.write_text("from appearance_flow_model import AppearanceFlowTinghui\n"
                       "configuration = {'data_dir': '/nope', 'output_dir': %r, 'num_iterations': 2, 'batch_size': 2,\n"
                       " 'learning_rate': 1e-4, 'image_size': 64, 'viewpoint_dim': 19, 'num_views': 3,\n"
                       " 'model': AppearanceFlowTinghui}\n" % str(tmp_path))
    with pytest.raises(SystemExit, match="AppearanceFlowTinghui"):
        train.main(["--hyper", str(conf_py), "--tfrecords"])


@pytest.mark.parametrize("viewpoint", ["onehot19", "disp2"])
def test_make_multiview_batch(viewpoint):
    from dynamic_multiview_3d_b200.synthetic import make_multiview_batch
    B, H, Vw = 6, 32, 4
    b = make_multiview_batch(B, H, Vw, viewpoint, seed=5)
    Vd = 19 if viewpoint == "onehot19" else 2
    assert b["image0"].shape == (Vw, B, H, H, 3) and b["image1"].shape == (B, H, H, 3) and b["disp"].shape == (Vw, B, Vd)
    assert b["image0"].dtype == b["image1"].dtype == b["disp"].dtype == np.float32
    assert 0 <= b["image0"].min() and b["image0"].max() <= 1
    bins = b["bins"]
    assert bins.shape == (Vw, B) and bins.min() >= 0 and bins.max() <= 18
    for s in range(B):
        assert len(set(bins[:, s].tolist())) == Vw, bins[:, s]          # distinct bins per target
    if viewpoint == "onehot19":
        assert np.array_equal(b["disp"].argmax(-1), bins) and np.array_equal(b["disp"].sum(-1), np.ones((Vw, B), np.float32))
    else:
        assert np.array_equal(b["disp"][..., 0], np.zeros((Vw, B), np.float32))
        assert np.array_equal(b["disp"][..., 1], np.deg2rad(20.0 * bins).astype(np.float32))
    again = make_multiview_batch(B, H, Vw, viewpoint, seed=5)
    assert all(np.array_equal(b[k], again[k]) for k in b)
    other = make_multiview_batch(B, H, Vw, viewpoint, seed=5, rank=1)
    assert not np.array_equal(b["image1"], other["image1"])
    one = make_multiview_batch(B, H, 1, viewpoint, seed=5)
    assert one["image0"].shape == (1, B, H, H, 3)
    with pytest.raises(ValueError):
        make_multiview_batch(B, H, 20, viewpoint)


def test_synthetic_batch_uses_the_multiview_generator():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.train import synthetic_batch
    m = pkg.AppFlowLowDimAngle(_conf(2, V=2, num_views=3), device="meta")
    b = synthetic_batch(m, seed=4)
    assert set(b) == {"image0", "image1", "disp"}
    assert {k: v.shape for k, v in b.items()} == m.input_spec()


# ------------------------------------------------------------------------------------------------------------- GPU helpers
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


_WS = {}


def _ws(B, Ho, Wo):
    n = int(_lib().load().dmv_sampler_loss_workspace_size(B, Ho, Wo))
    if _WS.get("t") is None or _WS["t"].numel() < n:
        _WS["t"] = torch.zeros(n, dtype=torch.uint8, device="cuda")
    return _WS["t"]


def _views_raw(data, views, head, target, weights, mode, inv, flags, fused=True, grad=True, tail=0, ws=None, ws_bytes=None):
    """One dmv_sampler_fuse_views_loss call; outputs are allocated with ``tail`` sentinel floats past their end."""
    R, H, W, C = data.shape
    B, Ho, Wo = R // views, head.shape[1], head.shape[2]

    def buf(n):
        return torch.full((n + tail,), 7.25, dtype=torch.float32, device="cuda")
    fo = buf(B * Ho * Wo * C) if fused else None
    gh = buf(head.numel()) if grad else None
    loss = buf(1) if target is not None else None
    w = (ctypes.c_float * C)(*weights) if weights is not None else None
    if target is not None and ws is None:
        ws = _ws(B, Ho, Wo)
    rc = _lib().load().dmv_sampler_fuse_views_loss(
        _p(data), views, _p(head), _p(target), w, LOSS[mode], float(inv), _p(fo), _p(gh), _p(loss), B, H, W, C, Ho, Wo, flags,
        _p(ws), ws.numel() if ws_bytes is None and ws is not None else (ws_bytes or 0), _stream())
    return rc, fo, gh, loss


def _composition(data, views, head, target, weights, mode, inv, flags):
    """The calls the kernel replaces: the sampler on every view, the fused loss with the logits (V = views), the sampler's
    flow gradient on its grad_gen -- through the package's operators and autograd."""
    from dynamic_multiview_3d_b200 import functional as F
    R, H, W, C = data.shape
    B = R // views
    flow = head[..., :2].contiguous().requires_grad_(True)
    logit = head[..., 2].contiguous().requires_grad_(True)
    gens = F._Resampler.apply(data, flow, flags)
    Ho, Wo = head.shape[1], head.shape[2]
    out = F.fused_views_loss(gens.reshape(views, B, Ho, Wo, C), logit.reshape(views, B, Ho, Wo), target, mode, weights, inv)
    loss, fused = (out, gens.detach()) if views == 1 else out
    loss.backward()
    gl = logit.grad if views > 1 else torch.zeros_like(logit)
    return loss.detach(), fused.reshape(B, Ho, Wo, C), torch.cat([flow.grad, gl[..., None]], -1)


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int32), b[~nb].view(np.int32))


def _np(t):
    return t.detach().cpu().numpy()


def _inputs(rng, views, B, H, W, Ho, Wo, C, flags, logit_scale=3.0):
    """Sources, a head whose flows reach every window path (path_warp over all views * B rows) and logits, a target."""
    data = rng.random((views * B, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, views * B, H, W, Ho, Wo, C, flags)
    logit = (rng.standard_normal((views * B, Ho, Wo, 1)) * logit_scale).astype(np.float32)
    head = np.concatenate([wf, logit], -1)
    target = rng.random((B, Ho, Wo, C), dtype=np.float32)
    return data, wf, head, target


def _check_against_composition(data, views, head, target, weights, mode, inv, flags, tail=16):
    data_t, head_t, tgt_t = _cuda(data), _cuda(head), _cuda(target)
    keep = [t.clone() for t in (data_t, head_t, tgt_t)]
    with _Counts(*LABELS) as n:
        rc, fo, gh, loss = _views_raw(data_t, views, head_t, tgt_t, weights, mode, inv, flags, tail=tail)
    assert rc == 0, _lib().last_error()
    assert n.d == dict({k: 0 for k in LABELS}, sampler_loss_fused=1), n.d
    assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(keep, (data_t, head_t, tgt_t))), "an input changed"
    B, Ho, Wo, C = target.shape
    nf, ng = B * Ho * Wo * C, head.size
    assert (fo[nf:] == 7.25).all() and (gh[ng:] == 7.25).all() and float(loss[1:].min()) == 7.25, "a sentinel tail was written"
    rloss, rfused, rgrad = _composition(data_t, views, head_t, tgt_t, weights, mode, inv, flags)
    assert _same_bits(_np(fo[:nf]).reshape(target.shape), _np(rfused)), "fused_out differs from the composition"
    g = _np(gh[:ng]).reshape(head.shape)
    r = _np(rgrad)
    for c, what in enumerate(("dL/dflow x", "dL/dflow y", "dL/dlogit")):
        assert _same_bits(g[..., c], r[..., c]), what + " differs from the composition"
    lk, lr = float(loss[0]), float(rloss)
    if np.isnan(lr):
        assert np.isnan(lk)
    else:
        assert lk == pytest.approx(lr, rel=1e-6, abs=1e-30), (lk, lr)
    # bit-reproducible run to run
    _, fo2, gh2, loss2 = _views_raw(data_t, views, head_t, tgt_t, weights, mode, inv, flags)
    assert _same_bits(_np(loss2[:1]), _np(loss[:1])) and torch.equal(gh2.view(torch.int32), gh[:ng].view(torch.int32))
    return fo[:nf].reshape(target.shape), g, lk


# ------------------------------------------------------------------------------------------------------------- GPU: kernel
@gpu
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("mode", ["l2", "l1"])
@pytest.mark.parametrize("views", [1, 2, 4, 8])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_kernel_equals_the_composition_on_every_window_path(C, views, mode, flags):
    """Ragged, non-square output (70 x 100) over a 61 x 76 source: the tiles of every view cycle through the window
    designs (36^2 box, 44^2 box, global gathers, no valid sample) and a few invalid samples."""
    B, H, W, Ho, Wo = 2, 61, 76, 70, 100
    rng = np.random.default_rng(1000 * C + 10 * views + flags + (5 if mode == "l1" else 0))
    data, wf, head, target = _inputs(rng, views, B, H, W, Ho, Wo, C, flags)
    _assert_paths(wf, H, W, C, flags, CATEGORIES)
    _check_against_composition(data, views, head, target, WEIGHTS[C], mode, 1.0 / (B * Ho * Wo), flags)


@gpu
@pytest.mark.parametrize("views", [3, 8])
def test_kernel_over_256_ctas_with_smooth_flows(views):
    """224^2 targets, B = 3 (more than 256 CTAs): small smooth flows, the training regime."""
    B, H, C = 3, 224, 3
    rng = np.random.default_rng(views)
    data = rng.random((views * B, H, H, C), dtype=np.float32)
    head = np.concatenate([rng.uniform(-4, 4, (views * B, H, H, 2)), rng.standard_normal((views * B, H, H, 1))], -1).astype(np.float32)
    target = rng.random((B, H, H, C), dtype=np.float32)
    _check_against_composition(data, views, head, target, WEIGHTS[C], "l2", 1.0 / (B * H * H), ADD_GRID)


LOGIT_EDGES = ["equal", "spread80", "nan", "inf", "minus_inf", "all_minus_inf", "nan_flow"]


@gpu
@pytest.mark.parametrize("edge", LOGIT_EDGES)
@pytest.mark.parametrize("mode", ["l2", "l1"])
def test_logit_and_flow_edges_give_the_composition_bits(edge, mode):
    views, B, H, W, Ho, Wo, C = 4, 2, 40, 44, 64, 96, 3
    rng = np.random.default_rng(LOGIT_EDGES.index(edge))
    data, wf, head, target = _inputs(rng, views, B, H, W, Ho, Wo, C, ADD_GRID)
    logit = head[..., 2]
    pick = rng.random(logit.shape) < 0.05
    if edge == "equal":
        logit[:] = 0.75
    elif edge == "spread80":
        logit[:] = rng.choice(np.array([-80.0, 80.0], np.float32), logit.shape)
    elif edge == "nan":
        logit[pick] = np.nan
    elif edge == "inf":
        logit[pick] = np.inf
    elif edge == "minus_inf":
        logit[pick] = -np.inf
    elif edge == "all_minus_inf":
        logit[:, :8] = -np.inf
    else:
        head[pick, 0] = np.nan
    _check_against_composition(data, views, head, target, WEIGHTS[C], mode, 1.0 / (B * Ho * Wo), ADD_GRID)


@gpu
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
def test_kernel_against_a_float64_oracle(flags):
    """Semantics, independently of the composition: oracle.tf_ops.resampler per view and oracle.graph.fuse_views in
    float64, the loss in float64, the head gradient by central differences of the float64 loss on a few pixels."""
    from oracle import graph as G
    from oracle import tf_ops as T
    views, B, H, W, Ho, Wo, C = 3, 2, 24, 28, 32, 40, 3
    rng = np.random.default_rng(flags)
    data = rng.random((views * B, H, W, C))
    flow = rng.uniform(-3, 3, (views * B, Ho, Wo, 2))
    logit = rng.standard_normal((views * B, Ho, Wo, 1))
    target = rng.random((B, Ho, Wo, C))
    head = np.concatenate([flow, logit], -1).astype(np.float32)
    data32, target32 = data.astype(np.float32), target.astype(np.float32)
    w = WEIGHTS[C]
    inv = 1.0 / (B * Ho * Wo)
    rc, fo, gh, loss = _views_raw(_cuda(data32), views, _cuda(head), _cuda(target32), w, "l2", inv, flags)
    assert rc == 0, _lib().last_error()

    def warp_of(h):
        f = h[..., :2].astype(np.float64)
        if not flags & ADD_GRID:
            return f
        ii, jj = np.meshgrid(np.arange(Ho, dtype=np.float64), np.arange(Wo, dtype=np.float64), indexing="ij")
        gx, gy = (jj, ii) if flags & GRID_XY else (ii, jj)
        return np.stack([f[..., 0] + gx, f[..., 1] + gy], -1)

    def fused64(h):
        gens = T.resampler(data32.astype(np.float64), warp_of(h)).reshape(views, B, Ho, Wo, C)
        return G.fuse_views(G.NumpyOps(), gens, h[..., 2:3].astype(np.float64).reshape(views, B, Ho, Wo, 1))

    def loss64(h):
        d = fused64(h) - target32
        return float((np.asarray(w) * d * d).sum() * inv)

    f64 = fused64(head)
    fo = _np(fo).reshape(f64.shape)
    assert np.allclose(fo, f64, rtol=1e-5, atol=1e-5), np.abs(fo - f64).max()
    assert float(loss[0]) == pytest.approx(loss64(head), rel=1e-5)
    g = _np(gh).reshape(head.shape)
    h64 = head.astype(np.float64)
    for _ in range(12):
        r, i, j, c = rng.integers(views * B), rng.integers(2, Ho - 2), rng.integers(2, Wo - 2), rng.integers(3)
        eps = 1e-4
        hp, hm = h64.copy(), h64.copy()
        hp[r, i, j, c] += eps
        hm[r, i, j, c] -= eps
        num = (loss64(hp) - loss64(hm)) / (2 * eps)
        assert abs(g[r, i, j, c] - num) <= 1e-4 * abs(num) + 1e-8, (r, i, j, c, g[r, i, j, c], num)


@gpu
@pytest.mark.parametrize("C", [1, 3, 4])
def test_forward_only_and_validation_modes(C):
    views, B, H, W, Ho, Wo = 3, 2, 61, 76, 70, 100
    rng = np.random.default_rng(C)
    data, wf, head, target = _inputs(rng, views, B, H, W, Ho, Wo, C, ADD_GRID | GRID_XY)
    data_t, head_t, tgt_t = _cuda(data), _cuda(head), _cuda(target)
    rc, fo, gh, loss = _views_raw(data_t, views, head_t, tgt_t, WEIGHTS[C], "l1", 0.25, ADD_GRID | GRID_XY)
    assert rc == 0
    with _Counts(*LABELS) as n:
        rc, fo1, _, _ = _views_raw(data_t, views, head_t, None, None, "l2", 0.0, ADD_GRID | GRID_XY, grad=False, tail=8)
        assert rc == 0, _lib().last_error()
        rc, fo2, gh2, loss2 = _views_raw(data_t, views, head_t, tgt_t, WEIGHTS[C], "l1", 0.25, ADD_GRID | GRID_XY, fused=False, grad=False)
        assert rc == 0, _lib().last_error()
    assert n.d == dict({k: 0 for k in LABELS}, sampler_loss_fused=2), n.d
    nf = fo.numel()
    assert _same_bits(_np(fo1[:nf]), _np(fo)) and (fo1[nf:] == 7.25).all()
    assert _same_bits(_np(loss2), _np(loss))
    from dynamic_multiview_3d_b200 import functional as F
    assert _same_bits(_np(F.fused_views_warp(data_t, head_t, views, "xy")).ravel(), _np(fo))


@gpu
def test_operators_match_the_abi_and_refuse_a_source_gradient():
    from dynamic_multiview_3d_b200 import functional as F
    views, B, H, C = 2, 2, 64, 3
    rng = np.random.default_rng(9)
    data, wf, head, target = _inputs(rng, views, B, H, H, H, H, C, ADD_GRID)
    data_t, tgt_t = _cuda(data), _cuda(target)
    head_t = _cuda(head).requires_grad_(True)
    rc, fo, gh, loss = _views_raw(data_t, views, head_t.detach(), tgt_t, WEIGHTS[C], "l2", 0.125, ADD_GRID)
    l, fused = F.fused_views_warp_loss(data_t, head_t, tgt_t, views, "l2", WEIGHTS[C], 0.125)
    (3.0 * l).backward()
    assert _same_bits(_np(l).ravel(), _np(loss)) and _same_bits(_np(fused).ravel(), _np(fo))
    assert torch.equal(head_t.grad, (gh * 3.0).reshape(head.shape))
    with torch.no_grad():
        lv, _ = F.fused_views_warp_loss(data_t, head_t, tgt_t, views, "l2", WEIGHTS[C], 0.125)
    assert _same_bits(_np(lv).ravel(), _np(loss))
    with pytest.raises(RuntimeError, match="no gradient wrt the sources"):
        F.fused_views_warp_loss(data_t.clone().requires_grad_(True), head_t, tgt_t, views)
    with pytest.raises(ValueError):
        F.fused_views_warp_loss(data_t, head_t, tgt_t, 3)
    with pytest.raises(ValueError):
        F.fused_views_warp(data_t, head_t.detach()[..., :2], views)


@gpu
def test_refusals_launch_nothing():
    views, B, H, C = 2, 2, 64, 3
    rng = np.random.default_rng(4)
    data, wf, head, target = _inputs(rng, views, B, H, H, H, H, C, ADD_GRID)
    d, h, t = _cuda(data), _cuda(head), _cuda(target)
    L = _lib().load()
    w = (ctypes.c_float * 4)(1, 1, 1, 1)
    fo = torch.empty(target.shape, device="cuda")
    gh = torch.empty(head.shape, device="cuda")
    loss = torch.empty((), device="cuda")
    ws = _ws(B, H, H)
    off = torch.zeros(data.size + 4, device="cuda")[1:1 + data.size].view(data.shape)

    def call(data=d, views=views, head=h, target=t, w=w, mode=0, fused=fo, grad=gh, loss=loss, B=B, C=C, Wd=H, Ho=H, Wo=H,
             ws=ws, ws_bytes=None):
        return L.dmv_sampler_fuse_views_loss(_p(data), views, _p(head), _p(target), w, mode, 0.1, _p(fused), _p(grad), _p(loss), B, H, Wd,
                                             C, Ho, Wo, ADD_GRID, _p(ws), ws.numel() if ws_bytes is None else ws_bytes, _stream())
    cases = [
        (E_INVALID_ARG, dict(data=None)), (E_INVALID_ARG, dict(head=None)), (E_INVALID_ARG, dict(loss=None)),
        (E_INVALID_ARG, dict(w=None)), (E_INVALID_ARG, dict(mode=7)),
        (E_INVALID_ARG, dict(target=None)), (E_INVALID_ARG, dict(target=None, grad=None)),
        (E_INVALID_ARG, dict(target=None, loss=None)), (E_INVALID_ARG, dict(target=None, loss=None, grad=None, fused=None)),
        (E_UNSUPPORTED_SHAPE, dict(views=0)), (E_UNSUPPORTED_SHAPE, dict(views=9)), (E_UNSUPPORTED_SHAPE, dict(C=2)),
        (E_UNSUPPORTED_SHAPE, dict(C=5)), (E_UNSUPPORTED_SHAPE, dict(Ho=1)), (E_UNSUPPORTED_SHAPE, dict(Wo=63)),
        (E_UNSUPPORTED_SHAPE, dict(C=1, Wd=63)), (E_UNSUPPORTED_SHAPE, dict(views=8, B=1 << 28)),
        (E_UNSUPPORTED_SHAPE, dict(B=1 << 22, Ho=4096, Wo=4096)), (E_INVALID_ARG, dict(B=0)),
        (E_ALIGN, dict(data=off)), (E_ALIGN, dict(head=torch.zeros(head.size + 4, device="cuda")[2:2 + head.size])),
        (E_ALIGN, dict(target=torch.zeros(target.size + 4, device="cuda")[1:])),
        (E_WORKSPACE, dict(ws_bytes=16)), (E_WORKSPACE, dict(ws=torch.zeros(0, dtype=torch.uint8, device="cuda"))),
    ]
    torch.cuda.synchronize()
    n0 = _lib().launch_count()
    for code, kw in cases:
        assert call(**kw) == code, (kw, _lib().last_error())
    torch.cuda.synchronize()
    assert _lib().launch_count() == n0
    assert call() == 0


# ------------------------------------------------------------------------------------------------------------- GPU: models
def _views_batch(model, B, Vw, H, seed=1234):
    from dynamic_multiview_3d_b200.synthetic import make_multiview_batch
    b = make_multiview_batch(B, H, Vw, "onehot19" if model.viewpoint_dim == 19 else "disp2", seed=seed)
    return {k: torch.from_numpy(b[k]).cuda() for k in model.INPUT_KEYS}


def _composed_step(m, batch):
    """The same graph as the num_views step, the tail composed of existing operators: flow_resample_layer per view and
    F.fused_views_loss on the head's slices."""
    from dynamic_multiview_3d_b200 import functional as F
    from dynamic_multiview_3d_b200.tf_utils import flow_resample_layer
    from dynamic_multiview_3d_b200.variables import use_store
    Vw, image0, image1 = m.num_views, batch["image0"], batch["image1"]
    B, H = image1.shape[0], image1.shape[1]
    m.store.new_anchor()
    with use_store(m.store):
        head = m._views_head(image0, batch["disp"])
    flat = image0.reshape((Vw * B,) + tuple(image0.shape[2:]))
    gens = [flow_resample_layer(flat[v * B:(v + 1) * B], head[v * B:(v + 1) * B, ..., :2].contiguous(), m.grid_order) for v in range(Vw)]
    logits = head[..., 2].reshape(Vw, B, H, H)
    loss, fused = F.fused_views_loss(torch.stack(gens), logits, image1, m.loss_mode, inv_count=1.0 / (B * H * H))
    return loss, fused


@gpu
@pytest.mark.parametrize("cls", CLASSES)
def test_model_step_equals_the_explicit_composition(cls):
    import dynamic_multiview_3d_b200 as pkg
    B, Vw, H = 2, 3, 64
    a = getattr(pkg, cls)(_conf(B, H, num_views=Vw, loss="l1" if cls == "AppFlowLowDimAngle" else "l2"))
    r = getattr(pkg, cls)(_conf(B, H, num_views=Vw, loss="l1" if cls == "AppFlowLowDimAngle" else "l2"))
    batch = _views_batch(a, B, Vw, H)
    la = a.step_loss(batch)
    la.backward()
    lr, fused = _composed_step(r, batch)
    lr.backward()
    torch.cuda.synchronize()
    la, lr = float(la.detach()), float(lr.detach())
    assert la == pytest.approx(lr, rel=1e-6), (la, lr)
    assert torch.equal(a.gen, fused)
    assert tuple(a.flow_field.shape) == (Vw, B, H, H, 2) and tuple(a.confidence.shape) == (Vw, B, H, H)
    checked = 0
    for k, v in a.store.vars.items():
        if v.trainable:
            assert torch.equal(v.grad, r.store.vars[k].grad), (k, float((v.grad - r.store.vars[k].grad).abs().max()))
            checked += 1
    assert checked > 10
    wp = a.warp_pts
    assert tuple(wp.shape) == (Vw * B, H, H, 2) and torch.isfinite(wp).all()
    assert float(a.eval_loss(batch)) == la


@gpu
def test_num_views_one_is_the_plain_model():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.synthetic import make_batch
    B, H = 2, 64
    a = pkg.AppearanceFlowModel(_conf(B, H))
    b = pkg.AppearanceFlowModel(_conf(B, H, num_views=1))
    assert {k: tuple(v.shape) for k, v in a.store.vars.items()} == {k: tuple(v.shape) for k, v in b.store.vars.items()}
    bt = make_batch(B, H, "onehot19", seed=3)
    batch = {k: torch.from_numpy(bt[k]).cuda() for k in a.INPUT_KEYS}
    la = [float(a.train_step(batch)) for _ in range(2)]
    lb = [float(b.train_step(batch)) for _ in range(2)]
    assert la == lb
    sa, sb = a.state_dict(), b.state_dict()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)


@gpu
def test_graphed_views_step_equals_eager_with_a_deferred_update():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    B, Vw, H = 4, 3, 64
    out = {}
    for graphed in (False, True):
        m = pkg.AppearanceFlowModel(_conf(B, H, num_views=Vw, seed=9))
        red = data_parallel.attach(m, bucket_mb=4.0)
        assert sorted(red.var_wait), "no deferred update"
        batch = _views_batch(m, B, Vw, H)
        step = GraphedTrainStep(m, warmup=2) if graphed else m.train_step
        losses = [float(step(batch)) for _ in range(3)]
        val = float(m.eval_loss(batch))
        sd = m.state_dict()
        out[graphed] = (losses, val, sd)
    assert out[True][0] == out[False][0] and out[True][1] == out[False][1]
    for k, t in out[False][2].items():
        assert torch.equal(t, out[True][2][k]), k


@gpu
def test_views_training_lowers_the_loss():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    B, Vw, H = 4, 3, 64
    m = pkg.AppearanceFlowModel(_conf(B, H, num_views=Vw, learning_rate=1e-4, seed=1))
    batch = _views_batch(m, B, Vw, H)
    step = GraphedTrainStep(m, warmup=2)
    losses = [float(step(batch)) for _ in range(50)]
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < 0.9 * np.mean(losses[:5]), losses


@gpu
def test_visualize_shows_source_frame_zero(tmp_path):
    import dynamic_multiview_3d_b200 as pkg
    B, Vw, H = 2, 3, 64
    m = pkg.AppFlowLowDimAngle(_conf(B, H, V=2, num_views=Vw, output_dir=str(tmp_path)))
    batch = _views_batch(m, B, Vw, H)
    r = m.visualize(batch["image0"], batch["image1"], batch["disp"], iter_num=5)
    assert np.isfinite(r["loss"]) and len(r["correspondences"]) == 6
    for f in ("output_5.png", "tr_gt_5.png", "tr_input_5.png", "flow_5.png", "corr_plot_5.png"):
        assert (tmp_path / f).exists(), f


@gpu
def test_train_main_with_several_views_validates_checkpoints_and_resumes(tmp_path, monkeypatch):
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
        " 'current_dir': current_dir, 'num_iterations': 6, 'batch_size': 4, 'num_views': 3, 'learning_rate': 1e-4,\n"
        " 'image_size': 64, 'viewpoint_dim': 19, 'train_val_split': 0.95, 'model': AppearanceFlowModel}\n")
    train.main(["--hyper", str(conf_py)])
    out = tmp_path / "modeldata"
    assert (out / "model4").exists() and (out / "model").exists()
    rows = [json.loads(l) for l in open(out / "scalars.jsonl")]
    assert {"training_loss", "val_loss"} <= {r["tag"] for r in rows}
    assert all(np.isfinite(r["value"]) for r in rows)
    assert tuple(torch.load(out / "model", map_location="cpu")["flow_field/w"].shape)[2] == 3
    assert float(torch.load(out / "model", map_location="cpu")["__adam_state__"][3]) == 7.0
    (out / "model").unlink()
    train.main(["--hyper", str(conf_py), "--pretrained", str(out / "model4")])
    assert float(torch.load(out / "model", map_location="cpu")["__adam_state__"][3]) == 8.0


_DP_SCRIPT = r"""
import os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
import dynamic_multiview_3d_b200 as pkg
from dynamic_multiview_3d_b200 import data_parallel
from dynamic_multiview_3d_b200.synthetic import make_multiview_batch
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
m = pkg.AppearanceFlowModel({"batch_size": 2, "num_views": 3, "learning_rate": 1e-3, "image_size": 64, "viewpoint_dim": 19, "seed": 0})
data_parallel.attach(m, bucket_mb=4.0)
b = make_multiview_batch(2, 64, 3, "onehot19", seed=7, rank=rank)
batch = {k: torch.from_numpy(b[k]).cuda() for k in m.INPUT_KEYS}
losses = [float(m.train_step(batch)) for _ in range(3)]
m.flush_updates()
half = m.store.flat["half"][:m.store.total].float()
ref = half.clone()
dist.broadcast(ref, src=0)
assert torch.equal(half, ref), "bf16 replicas differ across ranks"
assert all(l == l for l in losses), losses
print("rank %%d ok %%s" %% (rank, losses), flush=True)
torch.cuda.synchronize()
os._exit(0)
"""


@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_views_step_on_two_ranks(tmp_path):
    script = tmp_path / "dp_multiview.py"
    script.write_text(_DP_SCRIPT % {"root": ROOT})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", "2", str(script)],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, CUDA_VISIBLE_DEVICES="0,1"))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert r.stdout.count(" ok ") == 2, r.stdout

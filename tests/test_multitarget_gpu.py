"""Training on several targets of one source: the grouped fused warp loss (dmv_sampler_loss_fused_shared_src), the grouped
flow gradient (dmv_sampler_grad_flow_shared_src), the grouped activation / bias gradient (dmv_act_bwd_bias_grouped), the
grouped step of every single-view model, and the driver around it.

- both sampler forms are bit-equal to the plain calls on the source materialised with repeat_interleave, on every window
  path of the TMA kernel and on the tile kernel; the launch-label counters prove which form ran;
- dmv_act_bwd_bias_grouped is bit-exact against a NumPy restatement (fp32 sum in t order, x act', RNE to bf16);
- a grouped step (B sources x T targets) gives the loss of the T = 1 model fed the repeated batch, the decoder's
  gradients up to fp32 reorder and the encoder's up to one bf16 rounding of the summed feature gradient;
- the captured step, the loss over training and train.main work at T = 4.
input_spec, the refusals, the synthetic batches and the loss count need no GPU."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_sampler_loss_edges_gpu import CATEGORIES, _assert_paths, _at_offset, _Counts, _fused_raw, _fused_ws, _sampler_grad_warp, path_warp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ADD_GRID, GRID_XY = 1, 2
E_INVALID_ARG, E_ALIGN, E_UNSUPPORTED_SHAPE, E_WORKSPACE = -1, -2, -3, -5
LOSS = {"l2": 0, "l1": 1}
ORDERS = [ADD_GRID, ADD_GRID | GRID_XY]
ORDER_IDS = ["ref_yx", "xy"]


def _flow_conf(B, H=64, V=19, **kw):
    c = {"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": V, "seed": 3}
    c.update(kw)
    return c


COLORDEPTH = {"use_color": "", "use_depth": "", "depth_lr_factor": 0.1, "loss": "l1"}
MODELS = {"AppearanceFlowModel": ("AppearanceFlowModel", {}), "AppFlowHighDimAngle": ("AppFlowHighDimAngle", {}),
          "AppFlowLowDimAngle": ("AppFlowLowDimAngle", {}), "AppearanceFlowTinghui": ("AppearanceFlowTinghui", {}),
          "colordepth_tanh": ("Base_Prediction_Model", dict(COLORDEPTH, head="tanh")),
          "colordepth_flow": ("Base_Prediction_Model", dict(COLORDEPTH, head="flow"))}


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("which", list(MODELS))
def test_input_spec_has_the_target_axis_only_when_asked(which):
    import dynamic_multiview_3d_b200 as pkg
    cls, extra = MODELS[which]
    one = getattr(pkg, cls)(_flow_conf(3, **extra), device="meta").input_spec()
    four = getattr(pkg, cls)(_flow_conf(3, num_targets=4, **extra), device="meta").input_spec()
    for k, shp in one.items():
        if k in ("image1", "depth1", "disp"):
            assert four[k] == (3, 4) + shp[1:], (k, four[k])
        else:
            assert four[k] == shp == (3, 64, 64, shp[-1]), (k, four[k])
    assert one["disp"] == (3, 19)


def test_multiobject_classes_refuse_several_targets():
    import dynamic_multiview_3d_b200 as pkg
    base = {"batch_size": 2, "learning_rate": 1e-4, "image_size": 64, "viewpoint_dim": 2, "num_targets": 2}
    with pytest.raises(ValueError, match="MultiObjectAppFlow"):
        pkg.MultiObjectAppFlow(dict(base, use_color="", combination_image=""), device="meta")
    with pytest.raises(ValueError, match="MultiViewFusionAppFlow"):
        pkg.MultiViewFusionAppFlow(dict(base, num_views=4, use_depth=0.1), device="meta")
    pkg.MultiObjectAppFlow(dict(base, num_targets=1, use_color="", combination_image=""), device="meta")


def test_tfrecords_refuse_several_targets(tmp_path, monkeypatch):
    from dynamic_multiview_3d_b200 import train
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", os.environ.get("CUDA_VISIBLE_DEVICES", "0"))
    conf_py = tmp_path / "conf.py"
    conf_py.write_text("from appearance_flow_model import AppearanceFlowModel\n"
                       "configuration = {'data_dir': '/nope', 'output_dir': %r, 'num_iterations': 2, 'batch_size': 2,\n"
                       " 'learning_rate': 1e-4, 'image_size': 64, 'viewpoint_dim': 19, 'num_targets': 4,\n"
                       " 'model': AppearanceFlowModel}\n" % str(tmp_path))
    with pytest.raises(SystemExit, match="num_targets"):
        train.main(["--hyper", str(conf_py), "--tfrecords"])


@pytest.mark.parametrize("viewpoint", ["onehot19", "disp2"])
def test_make_batch_with_targets(viewpoint):
    from dynamic_multiview_3d_b200.synthetic import make_batch
    B, H, T = 5, 32, 4
    one = make_batch(B, H, viewpoint, seed=11, depth=True)
    b = make_batch(B, H, viewpoint, seed=11, depth=True, targets=T)
    Vd = 19 if viewpoint == "onehot19" else 2
    assert b["image0"].shape == (B, H, H, 3) and b["image1"].shape == (B, T, H, H, 3) and b["disp"].shape == (B, T, Vd)
    assert b["depth1"].shape == (B, T, H, H, 1) and b["mask1"].shape == (B, T, H, H, 1) and b["depth0"].shape == (B, H, H, 1)
    # one source image per sample serves all of its targets: it and target 0 are the targets=1 batch of the same seed
    assert np.array_equal(b["image0"], one["image0"]) and np.array_equal(b["depth0"], one["depth0"])
    for k in ("image1", "depth1", "mask1", "disp"):
        assert np.array_equal(b[k][:, 0], one[k]), k
    if viewpoint == "onehot19":
        assert np.array_equal(b["disp"].sum(-1), np.ones((B, T), np.float32))
        bins = b["disp"].argmax(-1)
    else:
        bins = np.rint(np.rad2deg(b["disp"][..., 1]) / 20.0).astype(int)
        assert np.array_equal(b["disp"][..., 0], np.zeros((B, T), np.float32))
    for s in range(B):
        assert len(set(bins[s].tolist())) == T, bins[s]           # distinct azimuth bins per source
    for t in range(1, T):                                          # the targets differ from each other
        assert not np.array_equal(b["image1"][:, t], b["image1"][:, 0])
    assert np.array_equal(make_batch(B, H, viewpoint, seed=11)["image1"], one["image1"])


class _Rec(object):
    """Stands in for the loss entry points: records the inv_count each call receives."""

    def __init__(self):
        self.inv = []

    def warp(self, data, flow, target, mode="l2", weights=None, inv_count=None, grid_order="ref_yx", unit_upstream=False, group=1):
        self.inv.append((inv_count, group))
        return torch.zeros(()), torch.zeros(flow.shape[:-1] + (data.shape[-1],))

    def recon(self, gen, target, mode="l2", weights=None, inv_count=None, mask=None, unit_upstream=False):
        self.inv.append((inv_count, None))
        return torch.zeros(())


def test_loss_count_includes_the_targets(monkeypatch):
    """inv_count = 1 / (B * T * H * W * world): the mean over every target pixel, as the T = 1 model on the repeated batch."""
    from dynamic_multiview_3d_b200 import appearance_flow_model as AFM, functional as F
    B, T, H, world = 3, 4, 32, 2
    m = AFM.AppearanceFlowModel.__new__(AFM.AppearanceFlowModel)
    m.world_size, m.loss_mode, m.grid_order, m.device = world, "l2", "ref_yx", torch.device("cpu")
    m.store = type("S", (), {"new_anchor": lambda self: None})()
    flow = torch.zeros((B * T, H, H, 2))
    monkeypatch.setattr(AFM.AppearanceFlowModel, "_grouped_flow", lambda self, i0, d: (flow, T))
    monkeypatch.setattr(AFM, "use_store", lambda s: __import__("contextlib").nullcontext())
    rec = _Rec()
    monkeypatch.setattr(F, "flow_resample_loss", rec.warp)
    monkeypatch.setattr(F, "reconstruction_loss", rec.recon)
    monkeypatch.setattr(F, "flow_resampler_grouped", lambda d, f, g, o: torch.zeros(f.shape[:-1] + (3,)))
    image0, image1, disp = torch.zeros((B, H, H, 3)), torch.zeros((B, T, H, H, 3)), torch.zeros((B, T, 19))
    m._grouped_forward_and_loss(image0, image1, disp)
    monkeypatch.setenv("DMV_NO_WARP_LOSS", "1")
    m._grouped_forward_and_loss(image0, image1, disp)
    assert rec.inv == [(1.0 / (B * T * H * H * world), T), (1.0 / (B * T * H * H * world), None)]
    assert m.gen.shape == (B, T, H, H, 3) and m.flow_field.shape == (B, T, H, H, 2)
    # the ungrouped count is unchanged: B * H * W * world
    m.gen = torch.zeros((B, H, H, 3))
    m.build_loss(torch.zeros((B, H, H, 3)))
    assert rec.inv[-1] == (1.0 / (B * H * H * world), None)


# ------------------------------------------------------------------------------------------------------ GPU helpers
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _grouped_fused(data, group, wf, target, weights, mode, inv, flags, ws=None, ws_bytes=None):
    B_src, H, W, C = data.shape
    B, Ho, Wo, _ = wf.shape
    ws = _fused_ws(B, Ho, Wo) if ws is None else ws
    gen = torch.empty((B, Ho, Wo, C), dtype=torch.float32, device="cuda")
    gw = torch.empty((B, Ho, Wo, 2), dtype=torch.float32, device="cuda")
    loss = torch.empty((), dtype=torch.float32, device="cuda")
    w = (ctypes.c_float * len(weights))(*weights)
    rc = _lib().load().dmv_sampler_loss_fused_shared_src(_p(data), B_src, group, _p(wf), _p(target), w, mode, float(inv), _p(gen), _p(gw),
                                                         _p(loss), H, W, C, Ho, Wo, flags, _p(ws),
                                                         ws.numel() if ws_bytes is None else ws_bytes, _stream())
    return rc, gen, gw, loss


def _grouped_grad_flow(data, group, wf, go, flags):
    B_src, H, W, C = data.shape
    B, Ho, Wo, _ = wf.shape
    gw = torch.empty((B, Ho, Wo, 2), dtype=torch.float32, device="cuda")
    rc = _lib().load().dmv_sampler_grad_flow_shared_src(_p(data), B_src, group, _p(wf), _p(go), _p(gw), H, W, C, Ho, Wo, flags, _stream())
    assert rc == 0, _lib().last_error()
    return gw


RAGGED = (61, 76, 70, 100)


# ------------------------------------------------------------------------------------------------ grouped warp loss
@gpu
@pytest.mark.parametrize("order", ORDERS, ids=ORDER_IDS)
@pytest.mark.parametrize("B_src,group", [(1, 1), (3, 1), (1, 2), (3, 2), (1, 5), (3, 5)])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_grouped_warp_loss_equals_the_repeated_source(C, B_src, group, order):
    H, W, Ho, Wo = RAGGED
    rng = np.random.default_rng(1000 * C + 100 * B_src + 10 * group + order)
    mode = "l1" if B_src == 3 else "l2"
    data = rng.random((B_src, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, B_src * group, H, W, Ho, Wo, C, order)
    _assert_paths(wf, H, W, C, order, CATEGORIES)
    target = rng.random((B_src * group, Ho, Wo, C), dtype=np.float32)
    weights = [1.0, 0.5, 2.0, 0.1][:C]
    inv = 1.0 / (B_src * group * Ho * Wo)
    d, w, t = (torch.from_numpy(a).cuda() for a in (data, wf, target))
    d0 = d.clone()
    rc, gen_r, gw_r, loss_r = _fused_raw(d.repeat_interleave(group, dim=0).contiguous(), w, t, weights, LOSS[mode], inv, order)
    assert rc == 0, _lib().last_error()
    with _Counts("sampler_loss_fused") as n:
        rc, gen, gw, loss = _grouped_fused(d, group, w, t, weights, LOSS[mode], inv, order)
    assert rc == 0, _lib().last_error()
    assert n.d == {"sampler_loss_fused": 1}, n.d
    assert torch.equal(gen, gen_r) and torch.equal(gw, gw_r) and torch.equal(loss, loss_r)
    assert torch.equal(d, d0)


@gpu
def test_grouped_warp_loss_op_matches_the_abi():
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(5)
    d = torch.from_numpy(rng.random((2, 32, 32, 3), dtype=np.float32)).cuda()
    fl = torch.from_numpy(rng.uniform(-3, 3, (6, 32, 32, 2)).astype(np.float32)).cuda().requires_grad_(True)
    t = torch.from_numpy(rng.random((6, 32, 32, 3), dtype=np.float32)).cuda()
    loss, gen = F.flow_resample_loss(d, fl, t, "l2", group=3)
    loss.backward()
    rc, gen_r, gw_r, loss_r = _fused_raw(d.repeat_interleave(3, 0).contiguous(), fl.detach(), t, [1.0] * 3, 0, 1.0 / (6 * 32 * 32), ADD_GRID)
    assert rc == 0 and torch.equal(loss, loss_r) and torch.equal(gen, gen_r) and torch.equal(fl.grad, gw_r)
    with pytest.raises(ValueError):
        F.flow_resample_loss(d, fl, t, group=4)


@gpu
def test_grouped_warp_loss_refusals_launch_nothing():
    lib = _lib().load()
    d = torch.zeros((2, 32, 32, 3), device="cuda")
    w = torch.zeros((4, 32, 32, 2), device="cuda")
    t = torch.zeros((4, 32, 32, 3), device="cuda")
    t_odd = torch.zeros(t.numel() + 4, device="cuda")[1:1 + t.numel()].view(t.shape)
    d2 = torch.zeros((2, 32, 32, 2), device="cuda")
    ws = _fused_ws(4, 32, 32)
    cases = [(dict(data=None), E_INVALID_ARG), (dict(B_src=0), E_INVALID_ARG), (dict(group=0), E_INVALID_ARG),
             (dict(group=-2), E_INVALID_ARG), (dict(B_src=1 << 16, group=1 << 15), E_UNSUPPORTED_SHAPE),
             (dict(mode=7), E_INVALID_ARG), (dict(target=t_odd), E_UNSUPPORTED_SHAPE), (dict(data=d2, C=2), E_UNSUPPORTED_SHAPE),
             (dict(ws_bytes=16), E_WORKSPACE), (dict(ws=None), E_WORKSPACE)]
    wts = (ctypes.c_float * 3)(1, 1, 1)
    out = [torch.empty((4, 32, 32, 3), device="cuda"), torch.empty((4, 32, 32, 2), device="cuda"), torch.empty((), device="cuda")]
    torch.cuda.synchronize()
    n0 = lib.dmv_launch_count()
    for over, code in cases:
        a = dict(data=d, B_src=2, group=2, target=t, mode=0, C=3, ws=ws, ws_bytes=None)
        a.update(over)
        wsb = a["ws"].numel() if (a["ws_bytes"] is None and a["ws"] is not None) else (a["ws_bytes"] or 0)
        rc = lib.dmv_sampler_loss_fused_shared_src(_p(a["data"]), a["B_src"], a["group"], _p(w), _p(a["target"]), wts, a["mode"], 1.0,
                                                   _p(out[0]), _p(out[1]), _p(out[2]), 32, 32, a["C"], 32, 32, ADD_GRID, _p(a["ws"]), wsb,
                                                   _stream())
        assert rc == code, (over, rc, _lib().last_error())
    torch.cuda.synchronize()
    assert lib.dmv_launch_count() == n0


# ------------------------------------------------------------------------------------------------- grouped flow gradient
@gpu
@pytest.mark.parametrize("order", ORDERS, ids=ORDER_IDS)
@pytest.mark.parametrize("B_src,group", [(1, 2), (3, 1), (3, 5)])
@pytest.mark.parametrize("C,form", [(1, "tma"), (3, "tma"), (4, "tma"), (16, "tile"), (3, "tile_offset")])
def test_grouped_grad_flow_equals_the_repeated_source(C, form, B_src, group, order):
    H, W, Ho, Wo = RAGGED
    rng = np.random.default_rng(31 * C + 100 * B_src + group + order)
    data = rng.random((B_src, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, B_src * group, H, W, Ho, Wo, min(C, 4), order)
    go = rng.standard_normal((B_src * group, Ho, Wo, C)).astype(np.float32)
    offset = form == "tile_offset"
    d = _at_offset(data) if offset else torch.from_numpy(data).cuda()
    rep = _at_offset(np.repeat(data, group, axis=0)) if offset else d.repeat_interleave(group, dim=0).contiguous()
    w, g = torch.from_numpy(wf).cuda(), torch.from_numpy(go).cuda()
    ref = _sampler_grad_warp(rep, w, g, order)
    with _Counts("sampler_grad_warp(tma)", "sampler_grad_warp") as n:
        gw = _grouped_grad_flow(d, group, w, g, order)
    tma = form == "tma"
    assert n.d == {"sampler_grad_warp(tma)": int(tma), "sampler_grad_warp": int(not tma)}, n.d
    assert torch.equal(gw, ref)


@gpu
def test_grouped_resampler_op_gives_the_flow_gradient_and_refuses_a_source_gradient():
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(9)
    d = torch.from_numpy(rng.random((2, 32, 32, 3), dtype=np.float32)).cuda()
    fl = torch.from_numpy(rng.uniform(-3, 3, (8, 32, 32, 2)).astype(np.float32)).cuda()
    go = torch.from_numpy(rng.standard_normal((8, 32, 32, 3)).astype(np.float32)).cuda()
    for order, flags in (("ref_yx", ADD_GRID), ("xy", ADD_GRID | GRID_XY)):
        f = fl.clone().requires_grad_(True)
        out = F.flow_resampler_grouped(d, f, 4, order)
        ref = F.flow_resampler_shared(d, fl, 4, order)
        assert torch.equal(out, ref)
        out.backward(go)
        assert torch.equal(f.grad, _sampler_grad_warp(d.repeat_interleave(4, 0).contiguous(), fl, go, flags))
    with pytest.raises(RuntimeError, match="source"):
        F.flow_resampler_grouped(d.clone().requires_grad_(True), fl, 4)
    with pytest.raises(ValueError):
        F.flow_resampler_grouped(d, fl, 3)


@gpu
def test_grouped_grad_flow_refusals_launch_nothing():
    lib = _lib().load()
    d = torch.zeros((2, 16, 16, 3), device="cuda")
    w = torch.zeros((4, 16, 16, 2), device="cuda")
    g = torch.zeros((4, 16, 16, 3), device="cuda")
    o = torch.zeros((4, 16, 16, 2), device="cuda")
    w_odd = torch.zeros(w.numel() + 2, device="cuda")[1:1 + w.numel()].view(w.shape)
    d17 = torch.zeros((2, 16, 16, 17), device="cuda")
    cases = [(dict(data=None), E_INVALID_ARG), (dict(go=None), E_INVALID_ARG), (dict(out=None), E_INVALID_ARG),
             (dict(B_src=0), E_INVALID_ARG), (dict(group=0), E_INVALID_ARG), (dict(B_src=-1), E_INVALID_ARG),
             (dict(B_src=1 << 16, group=1 << 15), E_UNSUPPORTED_SHAPE), (dict(wf=w_odd), E_ALIGN), (dict(out=w_odd), E_ALIGN),
             (dict(data=d17, C=17), E_UNSUPPORTED_SHAPE), (dict(flags=4), E_INVALID_ARG)]
    torch.cuda.synchronize()
    n0 = lib.dmv_launch_count()
    for over, code in cases:
        a = dict(data=d, B_src=2, group=2, wf=w, go=g, out=o, C=3, flags=ADD_GRID)
        a.update(over)
        rc = lib.dmv_sampler_grad_flow_shared_src(_p(a["data"]), a["B_src"], a["group"], _p(a["wf"]), _p(a["go"]), _p(a["out"]), 16, 16, a["C"],
                                                  16, 16, a["flags"], _stream())
        assert rc == code, (over, rc, _lib().last_error())
    torch.cuda.synchronize()
    assert lib.dmv_launch_count() == n0


# --------------------------------------------------------------------------------------- grouped activation gradient
def _bf16_to_f32(u16):
    return (u16.astype(np.uint32) << 16).view(np.float32)


def _f32_to_bf16(f):
    u = np.ascontiguousarray(f, np.float32).view(np.uint32)
    return ((u + np.uint32(0x7FFF) + ((u >> 16) & np.uint32(1))) >> 16).astype(np.uint16)


def _act_grad(y, act):
    if act == 1:
        return np.where(y > 0, np.float32(1.0), np.where(y < 0, np.float32(0.2), np.float32(0.6))).astype(np.float32)
    return np.where(y > 0, np.float32(1.0), np.float32(0.0)).astype(np.float32)


def _u16(t):
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def _bias_call(name, *args):
    rc = getattr(_lib().load(), name)(*args)
    assert rc == 0, _lib().last_error()


@gpu
@pytest.mark.parametrize("ld_extra", [0, 64], ids=["ld_C", "concat_slice"])
@pytest.mark.parametrize("group", [1, 2, 5])
@pytest.mark.parametrize("rows", [3, 37, 130])
@pytest.mark.parametrize("C", [8, 2048, 4096])
@pytest.mark.parametrize("act", [1, 2], ids=["lrelu", "relu"])
def test_act_bwd_bias_grouped_matches_numpy(act, C, rows, group, ld_extra):
    rng = np.random.default_rng(C + 7 * rows + 11 * group + ld_extra + act)
    ld = C + ld_extra
    full = _f32_to_bf16(rng.standard_normal((rows * group, ld)).astype(np.float32))
    y16 = _f32_to_bf16(rng.standard_normal((rows, C)).astype(np.float32))
    y16[:, :3] = 0                                                  # act' at y == 0
    dyf = torch.from_numpy(full.view(np.int16)).cuda().view(torch.bfloat16)
    dy = dyf[:, :C]                                                 # a column slice of the wider gradient
    y = torch.from_numpy(y16.view(np.int16)).cuda().view(torch.bfloat16)
    dpre = torch.empty((rows, C), dtype=torch.bfloat16, device="cuda")
    db = torch.empty(C, dtype=torch.float32, device="cuda")
    nws = _lib().load().dmv_act_bwd_bias_workspace_size(rows, C)
    ws = torch.empty(int(nws), dtype=torch.uint8, device="cuda")
    with _Counts("act_bwd_bias", "reduce_partials") as n:
        _bias_call("dmv_act_bwd_bias_grouped", dy.data_ptr(), ld, group, y.data_ptr(), dpre.data_ptr(), db.data_ptr(), rows, C, act,
                   ws.data_ptr(), ws.numel(), _stream())
    assert n.d == {"act_bwd_bias": 1, "reduce_partials": 1}, n.d
    f = _bf16_to_f32(full[:, :C]).reshape(rows, group, C)
    s = f[:, 0].copy()
    for t in range(1, group):
        s = (s + f[:, t]).astype(np.float32)
    ref = _f32_to_bf16((s * _act_grad(_bf16_to_f32(y16), act)).astype(np.float32))
    assert np.array_equal(_u16(dpre), ref)
    db_ref = torch.empty_like(db)
    _bias_call("dmv_act_bwd_bias", dpre.data_ptr(), y.data_ptr(), torch.empty_like(dpre).data_ptr(), db_ref.data_ptr(), rows, C, 0,
               ws.data_ptr(), ws.numel(), _stream())
    assert torch.equal(db, db_ref)
    if group == 1 and ld_extra == 0:                                # the plain entry point, bit for bit
        dpre2, db2 = torch.empty_like(dpre), torch.empty_like(db)
        _bias_call("dmv_act_bwd_bias", dy.data_ptr(), y.data_ptr(), dpre2.data_ptr(), db2.data_ptr(), rows, C, act, ws.data_ptr(), ws.numel(),
                   _stream())
        assert torch.equal(dpre.view(torch.int16), dpre2.view(torch.int16)) and torch.equal(db, db2)


@gpu
def test_act_bwd_bias_grouped_refusals_launch_nothing():
    lib = _lib().load()
    rows, C = 4, 16
    dy = torch.zeros((rows * 2, 24), dtype=torch.bfloat16, device="cuda")
    y = torch.zeros((rows, C), dtype=torch.bfloat16, device="cuda")
    dpre = torch.empty_like(y)
    db = torch.empty(C, device="cuda")
    ws = torch.empty(int(lib.dmv_act_bwd_bias_workspace_size(rows, C)), dtype=torch.uint8, device="cuda")
    cases = [(dict(dy=None), E_INVALID_ARG), (dict(ld=8), E_INVALID_ARG), (dict(group=0), E_INVALID_ARG), (dict(rows=0), E_INVALID_ARG),
             (dict(ld=20), E_UNSUPPORTED_SHAPE), (dict(C=12, ld=24), E_UNSUPPORTED_SHAPE), (dict(wsb=4), E_WORKSPACE)]
    torch.cuda.synchronize()
    n0 = lib.dmv_launch_count()
    for over, code in cases:
        a = dict(dy=dy, ld=24, group=2, rows=rows, C=C, wsb=ws.numel())
        a.update(over)
        rc = lib.dmv_act_bwd_bias_grouped(_p(a["dy"]), a["ld"], a["group"], y.data_ptr(), dpre.data_ptr(), db.data_ptr(), a["rows"], a["C"], 1,
                                          ws.data_ptr(), a["wsb"], _stream())
        assert rc == code, (over, rc, _lib().last_error())
    torch.cuda.synchronize()
    assert lib.dmv_launch_count() == n0


# -------------------------------------------------------------------------------------------------- models
def _is_encoder(name):
    return name.split("/")[0] in ("e0", "e0_0", "e1", "e1_0", "e2", "e2_0", "e3", "e3_0", "e4", "e4_0", "fc1", "e_fc0", "e_fc1") \
        or name.startswith(("pre_image0/", "pre_dimage0/"))


def _grouped_batch(model, B, T, H, seed=1234):
    from dynamic_multiview_3d_b200.synthetic import make_batch
    b = make_batch(B, H, "onehot19" if model.viewpoint_dim == 19 else "disp2", seed=seed, depth=True, targets=T)
    return {k: torch.from_numpy(b[k]).cuda() for k in model.INPUT_KEYS}


def _repeated(batch, T):
    """The same supervision as B x T pairs: every source repeated T times, targets and viewpoints flattened."""
    out = {}
    for k, v in batch.items():
        if k in ("image0", "depth0"):
            out[k] = v.repeat_interleave(T, dim=0).contiguous()
        else:
            out[k] = v.reshape((v.shape[0] * T,) + tuple(v.shape[2:])).contiguous()
    return out


def _rel(a, r):
    return float((a - r).norm() / (r.norm() + 1e-30))


@gpu
@pytest.mark.parametrize("which", list(MODELS))
def test_grouped_step_equals_the_repeated_batch_on_cuda_cores(which):
    """algo='simt': every kernel of the path computes each output row on its own, so the forward is batch-invariant and
    the loss is the repeated batch's bit for bit; the decoder sees the same rows in the same order (its gradients agree up
    to the fp32 reorder of the split weight-gradient sums); the encoder's input gradient is one bf16 rounding of the summed
    feature gradient instead of T roundings before the sum (measured within 1e-2 relative L2)."""
    import dynamic_multiview_3d_b200 as pkg
    cls, extra = MODELS[which]
    B, T, H = 3, 4, 64
    g = getattr(pkg, cls)(_flow_conf(B, H, num_targets=T, algo="simt", **extra))
    r = getattr(pkg, cls)(_flow_conf(B * T, H, algo="simt", **extra))
    batch = _grouped_batch(g, B, T, H)
    lg = g.step_loss(batch)
    lg.backward()
    lr = r.step_loss(_repeated(batch, T))
    lr.backward()
    torch.cuda.synchronize()
    assert torch.equal(lg.detach(), lr.detach()), (float(lg), float(lr))
    checked = 0
    for k, v in g.store.vars.items():
        if not v.trainable:
            continue
        gr, rr = v.grad, r.store.vars[k].grad
        assert _rel(gr, rr) < (1e-2 if _is_encoder(k) else 1e-5), (k, _rel(gr, rr))
        checked += 1
    assert checked > 20
    out = g.gen if hasattr(g, "gen") else g.gen_image1
    assert out.shape[:2] == (B, T)


@gpu
def test_grouped_step_on_tensor_cores_matches_the_repeated_batch():
    import dynamic_multiview_3d_b200 as pkg
    B, T, H = 16, 4, 224
    g = pkg.AppearanceFlowModel(_flow_conf(B, H, num_targets=T, loss="l2", seed=0))
    r = pkg.AppearanceFlowModel(_flow_conf(B * T, H, loss="l2", seed=0))
    batch = _grouped_batch(g, B, T, H)
    lg, lr = float(g.eval_loss(batch)), float(r.eval_loss(_repeated(batch, T)))
    assert np.isfinite(lg) and abs(lg - lr) <= 1e-2 * abs(lr), (lg, lr)


@gpu
def test_graphed_grouped_step_equals_eager_with_a_deferred_update():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    B, T, H = 4, 4, 64
    out = {}
    for graphed in (False, True):
        m = pkg.AppearanceFlowModel(_flow_conf(B, H, num_targets=T, seed=9))
        red = data_parallel.attach(m, bucket_mb=4.0)
        assert sorted(red.var_wait), "no deferred update"
        batch = _grouped_batch(m, B, T, H)
        step = GraphedTrainStep(m, warmup=2) if graphed else m.train_step
        losses = [float(step(batch)) for _ in range(3)]
        val = float(m.eval_loss(batch))                       # sees the pending update of the late FC matrices
        sd = m.state_dict()                                   # flushes it
        out[graphed] = (losses, val, sd)
    assert out[True][0] == out[False][0] and out[True][1] == out[False][1]
    for k, t in out[False][2].items():
        assert torch.equal(t, out[True][2][k]), k


@gpu
def test_grouped_training_lowers_the_loss():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    B, T, H = 4, 4, 64
    m = pkg.AppearanceFlowModel(_flow_conf(B, H, num_targets=T, learning_rate=1e-4, seed=1))
    batch = _grouped_batch(m, B, T, H)
    step = GraphedTrainStep(m, warmup=2)
    losses = [float(step(batch)) for _ in range(50)]
    assert all(np.isfinite(losses))
    assert np.mean(losses[-5:]) < 0.9 * np.mean(losses[:5]), losses


@gpu
def test_train_main_with_several_targets_validates_checkpoints_and_resumes(tmp_path, monkeypatch):
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
        " 'current_dir': current_dir, 'num_iterations': 6, 'batch_size': 4, 'num_targets': 4, 'learning_rate': 1e-4,\n"
        " 'image_size': 64, 'viewpoint_dim': 19, 'train_val_split': 0.95, 'model': AppearanceFlowModel}\n")
    train.main(["--hyper", str(conf_py)])
    out = tmp_path / "modeldata"
    assert (out / "model4").exists() and (out / "model").exists()
    rows = [json.loads(l) for l in open(out / "scalars.jsonl")]
    assert {"training_loss", "val_loss"} <= {r["tag"] for r in rows}
    assert all(np.isfinite(r["value"]) for r in rows)
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
from dynamic_multiview_3d_b200.synthetic import make_batch
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
m = pkg.AppearanceFlowModel({"batch_size": 2, "num_targets": 4, "learning_rate": 1e-3, "image_size": 64, "viewpoint_dim": 19, "seed": 0})
data_parallel.attach(m, bucket_mb=4.0)
b = make_batch(2, 64, "onehot19", seed=7, rank=rank, targets=4)
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
def test_data_parallel_grouped_step_on_two_ranks(tmp_path):
    script = tmp_path / "dp_multitarget.py"
    script.write_text(_DP_SCRIPT % {"root": ROOT})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", "2", str(script)],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, CUDA_VISIBLE_DEVICES="0,1"))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert r.stdout.count(" ok ") == 2, r.stdout

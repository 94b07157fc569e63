"""Novel-view rendering: the shared-source sampler form (dmv_sampler_fwd_shared_src), ModelBase.render and its CUDA-graph
form GraphedRender, the state it must leave alone, and the render CLI.

- the shared-source forward is bit-equal to dmv_sampler_fwd on the source materialised with repeat_interleave, on every
  window path of the TMA kernel and on the generic tile kernel; the launch-label counters prove which form ran;
- render is bit-equal to the explicit composition encode -> repeat -> decode -> shared-source warp, and within 1e-2 of
  forward on the repeated batch (fc1 and the joint FCs run at M = B there and M = B * V here: their split-K may differ);
- rendering changes no parameter, moment or optimizer byte, sees a pending deferred update, and does not move the
  workspaces a captured train step holds.
The viewpoint-set builders and the multi-object refusals need no GPU."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_sampler_loss_edges_gpu import CATEGORIES, _assert_paths, _at_offset, _Counts, path_warp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ADD_GRID, GRID_XY = 1, 2
E_INVALID_ARG, E_ALIGN, E_UNSUPPORTED_SHAPE = -1, -2, -3


# ------------------------------------------------------------------------------------------------- viewpoint sets (CPU)
def test_onehot19_is_the_identity():
    from dynamic_multiview_3d_b200 import render as R
    rows = R.viewpoint_set(19, views="onehot19")
    assert rows.dtype == np.float32 and np.array_equal(rows, np.eye(19, dtype=np.float32))


def test_azimuth_sweep_values_and_order():
    """(d_elevation, d_azimuth) in radians, as synthetic.py's disp2 rows: azimuths from START to STOP inclusive, ascending."""
    from dynamic_multiview_3d_b200 import render as R
    rows = R.viewpoint_set(2, azimuths="0:3.0:4", elevation=0.25)
    assert rows.dtype == np.float32 and rows.shape == (4, 2)
    assert np.array_equal(rows[:, 0], np.full(4, 0.25, np.float32))
    assert np.array_equal(rows[:, 1], np.array([0.0, 1.0, 2.0, 3.0], np.float32))
    assert np.array_equal(R.azimuth_sweep("1.5:1.5:1")[0], np.array([0.0, 1.5], np.float32))
    assert np.array_equal(R.azimuth_sweep("2:-2:3")[:, 1], np.array([2.0, 0.0, -2.0], np.float32))


def test_viewpoint_set_of_the_wrong_width_is_refused():
    from dynamic_multiview_3d_b200 import render as R
    with pytest.raises(ValueError, match="viewpoint_dim"):
        R.viewpoint_set(2, views="onehot19")
    with pytest.raises(ValueError, match="viewpoint_dim"):
        R.viewpoint_set(19, azimuths="0:1:5")
    with pytest.raises(ValueError):
        R.viewpoint_set(19, views="onehot19", azimuths="0:1:5")
    with pytest.raises(ValueError):
        R.viewpoint_set(19, views="onehot18")


@pytest.mark.parametrize("spec", ["", "0:1", "0:1:2:3", "a:1:3", "0:1:x", "0:1:2.5", "0:1:0", "0:1:-3", "nan:1:3", "0:inf:3"])
def test_malformed_azimuths_are_refused(spec):
    from dynamic_multiview_3d_b200 import render as R
    with pytest.raises(ValueError):
        R.azimuth_sweep(spec)


def test_cli_refuses_a_source_count_below_one(tmp_path, capsys):
    from dynamic_multiview_3d_b200 import render as R
    with pytest.raises(SystemExit):
        R.main(["--hyper", str(tmp_path / "missing.py"), "--checkpoint", "x", "--out", str(tmp_path), "--num_sources", "0"])
    assert "num_sources" in capsys.readouterr().err


def test_multiobject_classes_refuse_to_render():
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import functional as F
    base = {"batch_size": 2, "learning_rate": 1e-4, "image_size": 64, "viewpoint_dim": 2}
    models = [pkg.MultiObjectAppFlow(dict(base, use_color="", combination_image=""), device="meta"),
              pkg.MultiViewFusionAppFlow(dict(base, num_views=4, use_depth=0.1), device="meta")]
    for m in models:
        src = {"image0": torch.zeros((2, 64, 64, 3), device="meta")}
        with F.meta_mode(), pytest.raises(NotImplementedError, match=type(m).__name__):
            m.render(src, torch.zeros((5, 2), device="meta"))


# ------------------------------------------------------------------------------------------ shared-source sampler (GPU)
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ref_fwd(data, wf, flags):
    """dmv_sampler_fwd on the source materialised per output sample."""
    B, H, W, C = data.shape
    Bo, Ho, Wo, _ = wf.shape
    out = torch.empty((Bo, Ho, Wo, C), dtype=torch.float32, device="cuda")
    rc = _lib().load().dmv_sampler_fwd(data.data_ptr(), wf.data_ptr(), out.data_ptr(), None, None, Bo, H, W, C, Ho, Wo, flags, _stream())
    assert rc == 0, _lib().last_error()
    return out


def _shared_fwd(data, wf, group, flags, pad=64):
    """dmv_sampler_fwd_shared_src into a buffer followed by ``pad`` sentinel floats: (out, sentinel tail)."""
    B_src, H, W, C = data.shape
    Bo, Ho, Wo, _ = wf.shape
    n = Bo * Ho * Wo * C
    buf = torch.full((n + pad,), 1234.5, dtype=torch.float32, device="cuda")
    rc = _lib().load().dmv_sampler_fwd_shared_src(data.data_ptr(), B_src, group, wf.data_ptr(), buf.data_ptr(), H, W, C, Ho, Wo, flags,
                                                  _stream())
    assert rc == 0, _lib().last_error()
    return buf[:n].view(Bo, Ho, Wo, C), buf[n:]


SHAPES = {"ragged": (61, 76, 70, 100), "small_source": (8, 12, 40, 36)}


@gpu
@pytest.mark.parametrize("geom", list(SHAPES))
@pytest.mark.parametrize("flags", [0, ADD_GRID, ADD_GRID | GRID_XY], ids=["absolute", "flow_ref_yx", "flow_xy"])
@pytest.mark.parametrize("B_src,group", [(1, 1), (3, 1), (1, 2), (3, 2), (1, 19), (3, 19)])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_shared_source_tma_form_equals_the_repeated_source(C, B_src, group, flags, geom):
    H, W, Ho, Wo = SHAPES[geom]
    rng = np.random.default_rng(1000 * C + 100 * B_src + 10 * group + flags)
    data = rng.random((B_src, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, B_src * group, H, W, Ho, Wo, C, flags)
    _assert_paths(wf, H, W, C, flags, CATEGORIES if geom == "ragged" else ("none", "box36"))
    d = torch.from_numpy(data).cuda()
    w = torch.from_numpy(wf).cuda()
    d0 = d.clone()
    ref = _ref_fwd(d.repeat_interleave(group, dim=0).contiguous(), w, flags)
    with _Counts("sampler_fwd(tma)", "sampler_fwd") as n:
        out, tail = _shared_fwd(d, w, group, flags)
    assert n.d == {"sampler_fwd(tma)": 1, "sampler_fwd": 0}, n.d
    assert torch.equal(out, ref)
    assert bool((tail == 1234.5).all()) and torch.equal(d, d0)


@gpu
@pytest.mark.parametrize("flags", [0, ADD_GRID, ADD_GRID | GRID_XY], ids=["absolute", "flow_ref_yx", "flow_xy"])
@pytest.mark.parametrize("B_src,group", [(1, 2), (3, 19), (3, 1)])
@pytest.mark.parametrize("C,offset", [(2, False), (5, False), (3, True), (1, True)])
def test_shared_source_tile_form_equals_the_repeated_source(C, offset, B_src, group, flags):
    """The generic tile kernel: C outside {1, 3, 4}, or a source at a 4-byte offset."""
    H, W, Ho, Wo = SHAPES["ragged"]
    rng = np.random.default_rng(7 * C + 100 * B_src + group + flags)
    data = rng.random((B_src, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, B_src * group, H, W, Ho, Wo, min(C, 4), flags)
    d = _at_offset(data) if offset else torch.from_numpy(data).cuda()
    w = torch.from_numpy(wf).cuda()
    d0 = d.clone()
    ref = _ref_fwd(_at_offset(np.repeat(data, group, axis=0)) if offset else d.repeat_interleave(group, dim=0).contiguous(), w, flags)
    with _Counts("sampler_fwd(tma)", "sampler_fwd") as n:
        out, tail = _shared_fwd(d, w, group, flags)
    assert n.d == {"sampler_fwd(tma)": 0, "sampler_fwd": 1}, n.d
    assert torch.equal(out, ref)
    assert bool((tail == 1234.5).all()) and torch.equal(d, d0)


@gpu
def test_shared_source_op_matches_the_abi_and_refuses_gradients():
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(3)
    d = torch.from_numpy(rng.random((2, 32, 32, 3), dtype=np.float32)).cuda()
    fl = torch.from_numpy(rng.uniform(-3, 3, (10, 32, 32, 2)).astype(np.float32)).cuda()
    for order, flags in (("ref_yx", ADD_GRID), ("xy", ADD_GRID | GRID_XY)):
        out = F.flow_resampler_shared(d, fl, 5, order)
        assert out.shape == (10, 32, 32, 3) and torch.equal(out, _ref_fwd(d.repeat_interleave(5, 0).contiguous(), fl, flags))
    with pytest.raises(RuntimeError, match="no backward"):
        F.flow_resampler_shared(d, fl.clone().requires_grad_(True), 5)
    with torch.no_grad():
        F.flow_resampler_shared(d, fl.clone().requires_grad_(True), 5)
    with pytest.raises(ValueError):
        F.flow_resampler_shared(d, fl, 4)


@gpu
def test_shared_source_refusals_launch_nothing():
    L = _lib()
    lib = L.load()
    d = torch.zeros((2, 16, 16, 3), device="cuda")
    w = torch.zeros((4, 16, 16, 2), device="cuda")
    o = torch.zeros((4, 16, 16, 3), device="cuda")
    wf_odd = torch.zeros(4 * 16 * 16 * 2 + 1, device="cuda")[1:]
    p = lambda t: t.data_ptr()
    cases = [
        ((None, 2, 2, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 2, 2, None, p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 2, 2, p(w), None, 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 0, 2, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 2, 0, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), -1, 2, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 2, -4, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 2, 2, p(wf_odd), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_ALIGN),
        ((p(d), 2, 2, p(w), p(o), 16, 16, 17, 16, 16, ADD_GRID), E_UNSUPPORTED_SHAPE),
        ((p(d), 2, 2, p(w), p(o), 16, 16, 3, 16, 16, 4), E_INVALID_ARG),
        ((p(d), 2, 2, p(w), p(o), 16, 16, 3, 0, 16, ADD_GRID), E_INVALID_ARG),
        ((p(d), 1 << 16, 1 << 15, p(w), p(o), 16, 16, 3, 16, 16, ADD_GRID), E_UNSUPPORTED_SHAPE),    # B_src * group = 2^31
        ((p(d), 1 << 16, 1 << 14, p(w), p(o), 16, 16, 3, 64, 64, ADD_GRID), E_UNSUPPORTED_SHAPE),    # 2^30 samples x 4 tiles
    ]
    torch.cuda.synchronize()
    n0 = L.launch_count()
    for args, code in cases:
        rc = lib.dmv_sampler_fwd_shared_src(*args, _stream())
        assert rc == code, (args, rc, L.last_error())
    torch.cuda.synchronize()
    assert L.launch_count() == n0
    assert bool((o == 0).all())


# --------------------------------------------------------------------------------------------------------- models (GPU)
MODELS = {
    "appflow": ("AppearanceFlowModel", {"viewpoint_dim": 19}),
    "highdim": ("AppFlowHighDimAngle", {"viewpoint_dim": 19}),
    "lowdim": ("AppFlowLowDimAngle", {"viewpoint_dim": 19}),
    "tinghui": ("AppearanceFlowTinghui", {"viewpoint_dim": 19}),
    "colordepth_tanh": ("Base_Prediction_Model", {"viewpoint_dim": 2, "use_color": "", "use_depth": "", "depth_lr_factor": 0.1}),
    "colordepth_flow": ("Base_Prediction_Model", {"viewpoint_dim": 2, "use_color": "", "use_depth": "", "depth_lr_factor": 0.1,
                                                  "head": "flow"}),
}


def _model(which, B=3, H=64, seed=5, **extra):
    import dynamic_multiview_3d_b200 as pkg
    cls, conf = MODELS[which]
    return getattr(pkg, cls)(dict({"batch_size": B, "learning_rate": 1e-4, "image_size": H, "seed": seed}, **conf, **extra))


def _sources(m, B, seed=11):
    from dynamic_multiview_3d_b200.synthetic import make_batch
    b = make_batch(B, m.image_shape[0], "onehot19" if m.viewpoint_dim == 19 else "disp2", seed=seed, depth=True)
    return {k: torch.from_numpy(b[k]).cuda() for k in m.render_sources()}


def _views(m):
    from dynamic_multiview_3d_b200 import render as R
    rows = R.viewpoint_set(19, "onehot19") if m.viewpoint_dim == 19 else R.viewpoint_set(2, azimuths="-1.2:1.6:5", elevation=0.1)
    return torch.from_numpy(rows).cuda()


def _composition(m, src, vp):
    """encode -> repeat -> decode -> shared-source warp, spelled out."""
    from dynamic_multiview_3d_b200 import functional as F
    from dynamic_multiview_3d_b200.variables import use_store
    B, V = next(iter(src.values())).shape[0], vp.shape[0]
    code = F.to_bf16(vp.unsqueeze(0).expand(B, V, vp.shape[1]).reshape(B * V, vp.shape[1]))
    with torch.no_grad(), use_store(m.store):
        m.store.new_anchor()
        if "depth0" in m.render_sources():
            feats = m.encode(src["image0"], src["depth0"]).repeat_interleave(V, dim=0)
            out = m.decode(feats, code, lambda key, flow: F.flow_resampler_shared(src[key], flow, V, m.grid_order))
        else:
            flow = m.decode(m.encode(src["image0"]).repeat_interleave(V, dim=0), code)
            out = {"gen": F.flow_resampler_shared(src["image0"], flow, V, m.grid_order), "flow": flow}
    return {k: v.reshape((B, V) + tuple(v.shape[1:])) for k, v in out.items()}


def _forward_repeated(m, src, vp):
    B, V = next(iter(src.values())).shape[0], vp.shape[0]
    disp = vp.unsqueeze(0).expand(B, V, vp.shape[1]).reshape(B * V, vp.shape[1]).contiguous()
    rep = {k: t.repeat_interleave(V, dim=0) for k, t in src.items()}
    with torch.no_grad():
        if "depth0" in m.render_sources():
            out = m.forward(rep["image0"], rep["depth0"], disp)
            out = dict(out, **({"flow_image1": m.flow_image1, "flow_dimage1": m.flow_dimage1} if m.head == "flow" else {}))
        else:
            out = m.forward(rep["image0"], disp)
            out = {"gen": out["gen"], "flow": out["flow_field"]}
    return {k: v.reshape((B, V) + tuple(v.shape[1:])) for k, v in out.items()}


def _expected_keys(which):
    if which.startswith("colordepth"):
        return {"gen_image1", "gen_dimage1"} | ({"flow_image1", "flow_dimage1"} if which.endswith("flow") else set())
    return {"gen", "flow"}


@gpu
@pytest.mark.parametrize("which", list(MODELS))
def test_render_equals_the_composition_and_the_repeated_forward(which):
    m = _model(which)
    src, vp = _sources(m, 3), _views(m)
    V = vp.shape[0]
    out = m.render(src, vp)
    assert set(out) == _expected_keys(which)
    for k, v in out.items():
        assert v.shape[:2] == (3, V) and v.shape[2:4] == (64, 64) and v.dtype == torch.float32, (k, v.shape)
    comp = _composition(m, src, vp)
    assert set(comp) == set(out)
    for k in out:
        assert torch.equal(out[k], comp[k]), k
    # per-source viewpoints [B, V, d] give the same bits as the shared [V, d] rows
    per = m.render(src, vp.unsqueeze(0).expand(3, V, vp.shape[1]).contiguous())
    for k in out:
        assert torch.equal(out[k], per[k]), k
    fwd = _forward_repeated(m, src, vp)
    for k in out:
        a, r = out[k].double(), fwd[k].double()
        assert float((a - r).norm() / r.norm().clamp_min(1e-30)) < 1e-2, (k, float((a - r).norm() / r.norm()))


@gpu
def test_render_at_224_with_64_sources_and_19_views_equals_the_composition():
    m = _model("appflow", B=64, H=224, seed=2)
    src, vp = _sources(m, 64), _views(m)
    out = m.render(src, vp)
    comp = _composition(m, src, vp)
    assert out["gen"].shape == (64, 19, 224, 224, 3)
    for k in out:
        assert torch.equal(out[k], comp[k]), k


@gpu
@pytest.mark.parametrize("which", ["appflow", "colordepth_flow"])
def test_graphed_render_replays_the_eager_render(which):
    from dynamic_multiview_3d_b200.train import GraphedRender
    m = _model(which)
    vp = _views(m)
    g = GraphedRender(m, 3, vp.shape[0])
    for seed in (11, 12):                    # a second set of sources copied into the static buffers
        src = _sources(m, 3, seed=seed)
        got = {k: v.clone() for k, v in g(src, vp).items()}
        ref = m.render(src, vp)
        for k in ref:
            assert torch.equal(got[k], ref[k]), (seed, k)


def _state(m):
    flat = m.store.flat
    return {k: flat[k].clone() for k in ("master", "m", "v", "half")}, m.optimizer.state.clone()


@gpu
def test_rendering_changes_no_training_state():
    from dynamic_multiview_3d_b200.synthetic import make_batch
    from dynamic_multiview_3d_b200.train import GraphedRender
    m = _model("appflow", B=4)
    b = make_batch(4, 64, "onehot19", seed=3)
    m.train_step(*(torch.from_numpy(b[k]).cuda() for k in ("image0", "image1", "disp")))
    m.flush_updates()
    torch.cuda.synchronize()
    before, opt = _state(m)
    m.render(_sources(m, 3), _views(m))
    GraphedRender(m, 2, 19)(_sources(m, 2), _views(m))
    torch.cuda.synchronize()
    after, opt2 = _state(m)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert torch.equal(opt, opt2)


@gpu
def test_render_sees_a_pending_deferred_update(monkeypatch):
    """data_parallel.attach (single process) defers the late FC matrices' update into the next forward pass; a render
    right after train_step must give what it gives after an explicit flush_updates (twin model)."""
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.synthetic import make_batch
    monkeypatch.setenv("DMV_FUSE_FC_ADAM", "0")
    b = make_batch(4, 64, "onehot19", seed=3)
    args = [torch.from_numpy(b[k]).cuda() for k in ("image0", "image1", "disp")]
    outs = []
    for explicit in (False, True):
        m = _model("appflow", B=4, seed=8)
        red = data_parallel.attach(m, bucket_mb=4.0)
        assert "a5/Matrix" in red.var_wait
        for _ in range(2):
            m.train_step(*args)
        assert red.pending_host
        if explicit:
            m.flush_updates()
        outs.append(m.render(_sources(m, 3), _views(m)))
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), k


@gpu
def test_render_leaves_a_captured_train_step_intact():
    """Capture GraphedTrainStep, render 64 sources x 19 views (B x V = 1216 samples against the step's 4), replay the step:
    its loss and parameters equal those of a twin that did not render, and no training workspace or prepack buffer moved."""
    from dynamic_multiview_3d_b200 import functional as F
    from dynamic_multiview_3d_b200.synthetic import make_batch
    from dynamic_multiview_3d_b200.train import GraphedTrainStep
    b = make_batch(4, 64, "onehot19", seed=4)
    args = [torch.from_numpy(b[k]).cuda() for k in ("image0", "image1", "disp")]
    models = [_model("appflow", B=4, seed=6) for _ in range(2)]
    steps = [GraphedTrainStep(m, warmup=2) for m in models]
    losses = [[float(s(*args))] for s in steps]
    ws = {k: v.data_ptr() for k, v in F._workspaces.items()}
    pp = getattr(models[0].store, "prepack", None)
    packs = {k: e[1].data_ptr() for k, e in pp.entries.items()} if pp is not None else {}
    out = models[0].render(_sources(models[0], 64), _views(models[0]))
    assert out["gen"].shape == (64, 19, 64, 64, 3)
    assert {k: F._workspaces[k].data_ptr() for k in ws} == ws
    if pp is not None:
        assert {k: e[1].data_ptr() for k, e in pp.entries.items()} == packs
    del out
    torch.cuda.empty_cache()
    for i, s in enumerate(steps):
        losses[i] += [float(s(*args)) for _ in range(2)]
    assert losses[0] == losses[1]
    for m in models:
        m.flush_updates()
    torch.cuda.synchronize()
    for k in ("master", "m", "v", "half"):
        assert torch.equal(models[0].store.flat[k], models[1].store.flat[k]), k


# ------------------------------------------------------------------------------------------------------------ CLI (GPU)
def _png_size(path):
    with open(path, "rb") as f:
        head = f.read(24)
    assert head[:8] == b"\x89PNG\r\n\x1a\n" and head[12:16] == b"IHDR"
    return struct.unpack(">II", head[16:24])


@gpu
def test_render_cli_writes_strips_and_the_in_process_render(tmp_path):
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import render as R
    from dynamic_multiview_3d_b200.synthetic import make_batch
    from dynamic_multiview_3d_b200.train import load_conf
    conf_py = tmp_path / "conf.py"
    conf_py.write_text(
        "from appearance_flow_model import AppearanceFlowModel\n"
        "configuration = {'experiment_name': 'r', 'data_dir': '/nope', 'output_dir': %r, 'num_iterations': 3,\n"
        " 'batch_size': 4, 'learning_rate': 1e-4, 'image_size': 64, 'viewpoint_dim': 19, 'train_val_split': 0.95,\n"
        " 'model': AppearanceFlowModel}\n" % str(tmp_path))
    conf = load_conf(str(conf_py))
    m = pkg.AppearanceFlowModel(dict(conf, seed=4))
    b = make_batch(4, 64, "onehot19", seed=5)
    for _ in range(3):
        m.train_step(*(torch.from_numpy(b[k]).cuda() for k in ("image0", "image1", "disp")))
    ckpt = tmp_path / "model3"
    torch.save(m.state_dict(), ckpt)
    out_dir = tmp_path / "views"
    r = subprocess.run([sys.executable, "-m", "dynamic_multiview_3d_b200.render", "--hyper", str(conf_py), "--checkpoint", str(ckpt),
                        "--out", str(out_dir), "--num_sources", "3", "--views", "onehot19"],
                       cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    strips = sorted(p for p in os.listdir(out_dir) if p.endswith(".png"))
    assert len(strips) == 3
    for p in strips:
        assert _png_size(out_dir / p) == (64 * 20, 64)
    renders = np.load(out_dir / "renders.npy")
    assert renders.dtype == np.float32 and renders.shape == (3, 19, 64, 64, 3)
    m2 = pkg.AppearanceFlowModel(dict(conf, batch_size=3), build_loss=False)
    m2.load_state_dict(torch.load(ckpt, map_location="cpu"))
    src = R.load_sources(m2, conf, 3)
    ref = m2.render(src, torch.from_numpy(R.onehot19()).cuda())["gen"].cpu().numpy()
    assert np.array_equal(renders, ref)

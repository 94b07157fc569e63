"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol,
the model classes build the reference's variable tables (meta device, no compute), bucket
planning, and the world_size-2 gradient exchange over gloo."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "dmv3d.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(dmv_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from dynamic_multiview_3d_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        subprocess.run(["make", "-C", os.path.join(ROOT, "dynamic_multiview_3d_b200", "csrc"), "-j8"], check=True)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = _declared_symbols()
    assert len(syms) >= 26
    for s in syms:
        assert hasattr(lib, s), "libdmv3d.so does not export %s" % s
    # the ctypes table covers exactly the header
    assert sorted(_lib.SIGNATURES) == syms
    assert _lib.load().dmv_arch() == b"sm_100a"
    assert _lib.load().dmv_version() >= 100


def test_error_reporting_without_gpu():
    from dynamic_multiview_3d_b200 import _lib
    lib = _lib.load()
    rc = lib.dmv_sampler_fwd(None, None, None, None, None, 1, 2, 2, 1, 2, 2, 0, None)
    assert rc == -1 and "null" in _lib.last_error()
    with pytest.raises(_lib.DmvError):
        _lib.check(rc, "dmv_sampler_fwd")
    assert lib.dmv_sampler_bwd_workspace_size(64, 224, 224, 3, 224, 224) == 64 * 49 * 33 * 16      # tile box + 32 chunk boxes
    assert lib.dmv_wgrad_workspace_size(64, 112, 112, 32, 32, 5, 5, 1) > 0
    assert lib.dmv_conv_workspace_size(64, 224, 224, 3, 32, 5, 5, 2) >= 64 * 112 * 112 * 96 * 2


def test_cpu_tensors_are_rejected():
    from dynamic_multiview_3d_b200 import _lib, functional as F
    with pytest.raises(_lib.DmvError):
        F.resampler(torch.zeros(1, 4, 4, 3), torch.zeros(1, 4, 4, 2))


@pytest.mark.parametrize("cls,kind", [("AppearanceFlowModel", "base"), ("AppFlowHighDimAngle", "highdim"),
                                      ("AppFlowLowDimAngle", "lowdim"), ("AppearanceFlowTinghui", "tinghui")])
@pytest.mark.parametrize("H", [128, 224])
def test_variable_tables_match_reference_graph(cls, kind, H):
    import dynamic_multiview_3d_b200 as pkg
    from oracle import graph as G
    m = getattr(pkg, cls)({"batch_size": 2, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19}, device="meta")
    shapes = G.appflow_param_shapes(H, 19, kind)
    assert list(shapes) == list(m.store.vars)
    for k, (_, shp) in shapes.items():
        assert tuple(shp) == m.store.vars[k].shape, k
    assert tuple(m.flow_field.shape) == (2, H, H, 2) and tuple(m.gen.shape) == (2, H, H, 3)
    dead = [v.name for v in m.store.vars.values() if not v.trainable]
    assert dead == (["a0/Matrix", "a0/b", "a1/Matrix", "a1/b"] if kind == "highdim" else [])
    # flat offsets are 64-element aligned and non-overlapping
    # (weights in creation order, then the biases in one tail region that sharded data parallelism keeps replicated)
    offs = sorted((v.offset, v.numel) for v in m.store.vars.values())
    assert all(o % 64 == 0 for o, _ in offs)
    assert all(o2 >= o1 + n1 for (o1, n1), (o2, _) in zip(offs, offs[1:]))
    assert m.store.shard_end % 16384 == 0 and m.store.alloc % 16384 == 0
    assert all((v.offset >= m.store.shard_end) == v.name.endswith("/b") for v in m.store.vars.values())


@pytest.mark.parametrize("head", ["tanh", "flow"])
def test_colordepth_variable_table(head):
    """Base_Prediction_Model (main_model.py) at 224^2: same variables and shapes as the oracle's restatement."""
    import dynamic_multiview_3d_b200 as pkg
    from oracle import graph as G
    conf = {"batch_size": 2, "learning_rate": 1e-4, "image_size": 224, "viewpoint_dim": 2, "use_color": "", "use_depth": "",
            "depth_lr_factor": 0.1, "head": head}
    m = pkg.Base_Prediction_Model(conf, device="meta")
    shapes = G.colordepth_param_shapes(224, 2, conf)
    assert set(shapes) == set(m.store.vars)
    for k, (_, shp) in shapes.items():
        assert tuple(shp) == m.store.vars[k].shape, k
    assert tuple(m.gen_image1.shape) == (2, 224, 224, 3) and tuple(m.gen_dimage1.shape) == (2, 224, 224, 1)
    assert list(m.store.vars)[:2] == ["pre_image0/e0/w", "pre_image0/e0/b"] and m.store.vars["d3_0/w"].shape == (5, 5, 64, 128)


def test_reference_conf_loads_unchanged(tmp_path):
    from dynamic_multiview_3d_b200 import train
    conf_py = tmp_path / "conf.py"
    conf_py.write_text(
        "import os\ncurrent_dir = os.path.dirname(os.path.realpath(__file__))\n"
        "from highdim_angle import AppFlowHighDimAngle\nimport dyn_mult_view\n"
        "configuration = {'experiment_name': 'x', 'data_dir': '/nope', 'output_dir': current_dir + '/modeldata',\n"
        " 'current_dir': current_dir, 'num_iterations': 200000, 'batch_size': 64, 'learning_rate': 1e-4,\n"
        " 'train_val_split': 0.95, 'model': AppFlowHighDimAngle}\n")
    conf = train.load_conf(str(conf_py))
    import dynamic_multiview_3d_b200 as pkg
    assert conf["model"] is pkg.AppFlowHighDimAngle and conf["batch_size"] == 64
    assert train.checkpoint_iteration("/x/y/model120000") == 120000


MO_CONFS = [{"use_color": "", "use_depth": 0.1, "combination_image": "", "gen_sep_images": "", "predict_target_masks": 0.1},
            {"use_color": "", "combination_image": "", "fully_conv": ""}, {"use_depth": 1.0, "gen_sep_images": "", "masked_image_loss": ""}]


@pytest.mark.parametrize("extra", MO_CONFS)
def test_multiobject_variable_table_matches_reference_graph(extra):
    """MultiObjectAppFlow creates the variables of multiobject_appflow.py:123-221 in the reference's order."""
    import dynamic_multiview_3d_b200 as pkg
    from oracle import graph as G
    conf = dict({"batch_size": 2, "learning_rate": 1e-4, "image_size": 64, "viewpoint_dim": 2}, **extra)
    m = pkg.MultiObjectAppFlow(conf, device="meta")
    shapes = G.multiobject_param_shapes(64, 2, conf)
    assert list(shapes) == list(m.store.vars)
    for k, (_, shp) in shapes.items():
        assert tuple(shp) == m.store.vars[k].shape, k
    assert [h[0] for h in G._mo_heads(conf)] == [h[0] for h in m.heads]


def test_multiview_variable_table():
    """Config 5 sits on the multi-object trunk: four pre-encoders, one decoder, one 3-channel flow + confidence head."""
    import dynamic_multiview_3d_b200 as pkg
    from oracle import graph as G
    conf = {"batch_size": 2, "learning_rate": 1e-4, "image_size": 64, "viewpoint_dim": 2, "num_views": 4, "use_depth": 0.1}
    m = pkg.MultiViewFusionAppFlow(conf, device="meta")
    shapes = G.multiview_param_shapes(64, 2, conf)
    assert list(shapes) == list(m.store.vars)
    for k, (_, shp) in shapes.items():
        assert tuple(shp) == m.store.vars[k].shape, k
    assert m.store.vars["dec_image1/d0/w"].shape == (5, 5, 3, 32) and m.store.vars["e2_0/w"].shape == (5, 5, 256, 64)
    assert tuple(m.gens.shape) == (4, 2, 64, 64, 3) and tuple(m.logits.shape) == (4, 2, 64, 64) and tuple(m.flow_field.shape) == (4, 2, 64, 64, 2)
    assert m.INPUT_KEYS == ("image0", "depth0", "image0_mask0", "image0_mask1", "displacement", "image1")


# Experiment confs in the reference's tensorflowdata/<experiment>/conf.py format, one for every way train.py treats a
# conf: each model class imported by the reference's module names, the Base_Prediction_Model fallback, the reference's
# unparsable appflow_multiobject conf, the out-of-scope multiobject_main_model and an MV3D conf.
REF_CONFS = os.path.join(ROOT, "tests", "golden", "confs")


def _reference_confs():
    out = []
    for d, _, files in os.walk(REF_CONFS):
        if "conf.py" in files:
            out.append(os.path.relpath(os.path.join(d, "conf.py"), REF_CONFS))
    return sorted(out)


def test_reference_conf_fixtures_are_present():
    assert len(_reference_confs()) == 9


@pytest.mark.parametrize("rel", _reference_confs())
def test_every_reference_conf_builds_its_model_and_step_plumbing(rel):
    """train.py:40-65 on conf files loaded unchanged (meta device: variable tables and shapes only): the model class
    the conf selects builds, and the driver's plumbing (input_spec / INPUT_KEYS / synthetic batches / checkpoint
    surface) covers it.  Confs of out-of-scope model files fail with a clear import error."""
    from dynamic_multiview_3d_b200 import train
    from dynamic_multiview_3d_b200.model_base import ModelBase
    path = os.path.join(REF_CONFS, rel)
    txt = open(path).read()
    if "multiobject_main_model" in txt:                          # SURVEY 2.1 row 6b: out of scope, no sampler on it
        with pytest.raises(ImportError):
            train.load_conf(path)
        return
    if rel.startswith("appflow_multiobject" + os.sep + "conf.py"):
        with pytest.raises(SyntaxError):                         # the reference file itself is broken (SURVEY section 5)
            train.load_conf(path)
        return
    conf = dict(train.load_conf(path), batch_size=2)
    if "model" not in conf and not ("use_color" in conf or "use_depth" in conf):
        with pytest.raises(ValueError):                          # nobg_nodm confs belong to the MV3D scripts
            train.build_model(conf, device="meta")
        return
    model = train.build_model(conf, device="meta")
    assert isinstance(model, ModelBase)
    spec = model.input_spec()
    assert set(spec) == set(model.INPUT_KEYS)
    b = train.synthetic_batch(model, seed=0)
    assert {k: tuple(v.shape) for k, v in b.items()} == {k: tuple(v) for k, v in spec.items()}
    for name in ("train_step", "eval_loss", "state_dict", "load_state_dict", "step_loss"):
        assert callable(getattr(model, name))
    assert model.image_shape[0] == 128                           # the reference's own size when the conf names none


_CKPT_WORKER = r"""
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, %r)
from dynamic_multiview_3d_b200.data_parallel import ShardedGradientReducer
from dynamic_multiview_3d_b200.model_base import ModelBase
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["MASTER_PORT"], rank=rank, world_size=world)
sizes = [64, 192, 4096, 8192]
alloc = 16384
flat = {k: torch.zeros(alloc) for k in ("grad", "master", "m", "v", "half")}
vars_, off = {}, 0
for i, n in enumerate(sizes):
    sl = slice(off, off + n)
    vars_["v%%d/w" %% i] = types.SimpleNamespace(name="v%%d/w" %% i, offset=off, numel=n, trainable=True, shape=(n,),
                                               master=flat["master"][sl], m=flat["m"][sl], v=flat["v"][sl]); off += n
store = types.SimpleNamespace(vars=vars_, alloc=alloc, flat=flat, trainable_vars=lambda: list(vars_.values()),
                              state_dict=lambda: {k: v.master.clone() for k, v in vars_.items()})
red = ShardedGradientReducer(store, chunk_mb=2048 * 4 / (1 << 20))
# owner-only state: every rank has written only the slices it owns (as ShardedTFAdam does)
for c in range(len(red.chunks)):
    if red.expected[c] == 0: continue
    a, b = red.owned(c)
    idx = torch.arange(a, b, dtype=torch.float32)
    flat["master"][a:b] = idx; flat["m"][a:b] = idx * 2; flat["v"][a:b] = idx * 3


class M(ModelBase):
    pass


m = M(); m.store = store; m._dp = red; m.device = torch.device("cpu")
m.optimizer = types.SimpleNamespace(state=torch.tensor([0.5, 0.25, 0.0, 7.0]))
sd = m.state_dict()                                   # collective: gathers the owners' slices first
for k, v in vars_.items():
    idx = torch.arange(v.offset, v.offset + v.numel, dtype=torch.float32)
    assert torch.equal(sd[k], idx) and torch.equal(sd[k + "/Adam"], idx * 2) and torch.equal(sd[k + "/Adam_1"], idx * 3), k
assert sd["__adam_state__"][3] == 7.0
print("rank", rank, "ok")
dist.destroy_process_group()
"""


def test_sharded_checkpoint_gathers_owner_state_world_size_2_gloo(tmp_path):
    """ModelBase.state_dict under sharded data parallelism (every model class inherits it): masters and Adam moments
    live with their owning rank; the checkpoint holds the complete state on every rank, plus the step state."""
    script = tmp_path / "wc.py"
    script.write_text(_CKPT_WORKER % ROOT)
    port = str(33500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_variable_reuse_within_one_pass_is_refused():
    """The weight-gradient kernels overwrite a variable's gradient slot: a second use of a name in one forward pass
    (TF-style reuse) must raise instead of silently dropping a gradient."""
    from dynamic_multiview_3d_b200.variables import VariableStore
    st = VariableStore(torch.device("meta"))
    st.get("w", [3, 3], "zeros")
    with pytest.raises(RuntimeError):
        st.get("w", [3, 3], "zeros")
    st.new_anchor()
    st.get("w", [3, 3], "zeros")                      # the next pass may use it again


def test_bucket_plan_is_reverse_contiguous():
    from dynamic_multiview_3d_b200.data_parallel import plan_buckets
    table, off = [], 0
    for i, n in enumerate([64, 128, 1 << 20, 64, 3 << 20, 256]):
        table.append(("v%d" % i, off, n))
        off += n
    b = plan_buckets(table, 1 << 20)
    assert b[0][2][0] == "v5"                          # last-created variable first
    assert b[0][1] == off and b[-1][0] == 0            # covers the whole buffer
    assert all(x[0] == y[1] for x, y in zip(b, b[1:]))  # contiguous, descending
    assert sum(len(x[2]) for x in b) == len(table)


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from dynamic_multiview_3d_b200.data_parallel import GradientAllReducer
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["MASTER_PORT"], rank=rank, world_size=world)
sizes = [64, 192, 4096, 64, 8192, 128]
table, off = [], 0
for i, n in enumerate(sizes):
    table.append(("v%%d" %% i, off, n)); off += n
flat = torch.zeros(off)
red = GradientAllReducer(flat, table, bucket_mb=4096 * 4 / (1 << 20), trainable={"v%%d" %% i for i in range(6) if i != 3})
order = []
for i in reversed(range(6)):                      # backward order
    if i == 3: continue                            # a dead variable never reports
    name, o, n = table[i]
    flat[o:o + n] = float(rank + 1) * (i + 1)
    red.on_grad_ready(name)
    order.append(list(red.launched))
red.finish()
exp = torch.cat([torch.full((n,), float(sum(range(1, world + 1))) * (i + 1)) if i != 3 else torch.zeros(n) for i, (_, _, n) in enumerate(table)])
assert torch.equal(flat, exp), (flat[:4], exp[:4])
assert red.pending == red.expected and red.launched == []
assert len(order[-1]) == len(red.buckets)
print("rank", rank, "ok", len(red.buckets), "buckets")
dist.destroy_process_group()
"""


def test_gradient_allreduce_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER % ROOT)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


_SHARD_WORKER = r"""
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, %r)
from dynamic_multiview_3d_b200.data_parallel import ShardedGradientReducer, plan_chunks
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% os.environ["MASTER_PORT"], rank=rank, world_size=world)
sizes = [64, 192, 4096, 64, 8192, 128]
vars_, off = {}, 0
for i, n in enumerate(sizes):
    vars_["v%%d" %% i] = types.SimpleNamespace(name="v%%d" %% i, offset=off, numel=n, trainable=(i != 3)); off += n
alloc = -(-off // 16384) * 16384
store = types.SimpleNamespace(vars=vars_, alloc=alloc, trainable_vars=lambda: [v for v in vars_.values() if v.trainable],
                              flat={k: torch.zeros(alloc) for k in ("grad", "master", "m", "v", "half")})
red = ShardedGradientReducer(store, chunk_mb=2048 * 4 / (1 << 20))        # 2048-element chunks
assert all((e - s) %% (world * 256) == 0 for s, e in red.chunks) and red.chunks[-1][1] == alloc
g = store.flat["grad"]
for i in reversed(range(6)):
    if i == 3: continue
    v = vars_["v%%d" %% i]
    g[v.offset:v.offset + v.numel] = float(rank + 1) * (i + 1)
    red.on_grad_ready(v)
red.finish()
tot = float(sum(range(1, world + 1)))
exp = torch.zeros(alloc)
for i, v in enumerate(vars_.values()):
    if i != 3: exp[v.offset:v.offset + v.numel] = tot * (i + 1)
for c in range(len(red.chunks)):                  # the OWNED slice of every live chunk holds the global sum
    if red.expected[c] == 0: continue
    a, b = red.owned(c)
    assert torch.equal(g[a:b], exp[a:b]), (c, a, b)
# owner-only update, then the all-gather restores identical replicas
for c in range(len(red.chunks)):
    if red.expected[c] == 0: continue
    a, b = red.owned(c)
    store.flat["half"][a:b] = g[a:b] * 0.5
    red.all_gather("half", c)
live = torch.zeros(alloc, dtype=torch.bool)
for c, (s, e) in enumerate(red.chunks):
    if red.expected[c]: live[s:e] = True
assert torch.equal(store.flat["half"][live], (exp * 0.5)[live])
assert red.pending == red.expected and red.launched == []
print("rank", rank, "ok", len(red.chunks), "chunks")
dist.destroy_process_group()
"""


def test_sharded_reduce_scatter_world_size_2_gloo(tmp_path):
    script = tmp_path / "ws.py"
    script.write_text(_SHARD_WORKER % ROOT)
    port = str(31500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_chunk_plan_tiles_the_buffer():
    from dynamic_multiview_3d_b200.data_parallel import plan_chunks
    table, off = [], 0
    for i, n in enumerate([64, 128, 1 << 20, 64, 3 << 20, 256]):
        table.append(("v%d" % i, off, n))
        off += n
    alloc = -(-off // 16384) * 16384
    chunks, v2c, exp = plan_chunks(table, alloc, 1 << 20, 8, {"v%d" % i for i in range(6)})
    assert chunks[0][0] == 0 and chunks[-1][1] == alloc and all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
    assert all((e - s) % (8 * 256) == 0 and e - s <= 1 << 20 for s, e in chunks)
    assert v2c["v0"] == [0] and len(v2c["v4"]) >= 3 and sum(exp) == sum(len(c) for c in v2c.values())
    for name, o, n in table:                       # every variable lies inside the union of its chunks
        cs = v2c[name]
        assert chunks[cs[0]][0] <= o and o + n <= chunks[cs[-1]][1] and cs == list(range(cs[0], cs[-1] + 1))


def test_chunk_groups_begin_at_big_variables():
    """The 224^2 app-flow variable table: the first chunk holds the encoder convolutions only (its exchange cannot start
    before the last weight gradient of the step), every FC matrix starts a chunk group, pieces <= the chunk size."""
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.data_parallel import plan_chunks
    m = pkg.AppearanceFlowModel({"batch_size": 2, "learning_rate": 1e-4, "image_size": 224, "viewpoint_dim": 19}, device="meta")
    st = m.store
    table = [(v.name, v.offset, -(-v.numel // 64) * 64) for v in st.vars.values() if v.offset < st.shard_end]
    live = {v.name for v in st.trainable_vars()}
    for world, elems in ((8, 32 << 20), (2, 32 << 20), (1, 8 << 20)):
        chunks, v2c, exp = plan_chunks(table, st.shard_end, elems, world, live)
        starts = [c[0] for c in chunks]
        assert chunks[0] == (0, st.vars["fc1/Matrix"].offset) and chunks[0][1] - chunks[0][0] < 2 << 20
        assert v2c["e0/w"] == [0] and v2c["e4_0/w"] == [0] and 0 not in v2c["fc1/Matrix"]
        for name in ("fc1/Matrix", "a3/Matrix", "a4/Matrix", "a5/Matrix"):
            assert st.vars[name].offset in starts and st.vars[name].offset % 16384 == 0
        assert chunks[-1][1] == st.shard_end and all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
        assert all((e - s) % (world * 256) == 0 and e - s <= elems for s, e in chunks)
        assert v2c["flow_field/w"] == [len(chunks) - 1] and v2c["a5/Matrix"][-1] == len(chunks) - 1


def test_synthetic_batches_are_deterministic_and_in_range():
    from dynamic_multiview_3d_b200.synthetic import make_batch
    a = make_batch(3, 64, "onehot19", seed=1234, rank=1, depth=True)
    b = make_batch(3, 64, "onehot19", seed=1234, rank=1, depth=True)
    for k in a:
        assert np.array_equal(a[k], b[k])
    assert a["image0"].shape == (3, 64, 64, 3) and a["image0"].dtype == np.float32
    assert 0.0 <= a["image0"].min() and a["image0"].max() <= 1.0
    assert (a["disp"].sum(1) == 1).all() and a["disp"].shape == (3, 19)
    assert a["depth0"].max() == 1.0 and 0.3 <= a["depth0"].min() <= 0.6
    c = make_batch(2, 64, "disp2", views=4)
    assert c["image0"].shape == (2, 4, 64, 64, 3) and c["disp"].shape == (2, 2)


def test_chunk_plan_leaves_out_variables_updated_elsewhere():
    """plan_chunks(skip=...): an FC matrix that Adam updates inside its weight-gradient kernel (optimizer.py) gets chunks of its own
    that nothing reports to and nothing launches; every other variable still lies inside live chunks, and no live chunk touches
    the skipped range."""
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.data_parallel import plan_chunks
    m = pkg.AppearanceFlowModel({"batch_size": 2, "learning_rate": 1e-4, "image_size": 224, "viewpoint_dim": 19}, device="meta")
    st = m.store
    table = [(v.name, v.offset, -(-v.numel // 64) * 64) for v in st.vars.values() if v.offset < st.shard_end]
    live = {v.name for v in st.trainable_vars()}
    skip = {"fc1/Matrix", "a3/Matrix", "a4/Matrix"}
    chunks, v2c, exp = plan_chunks(table, st.shard_end, 8 << 20, 1, live - skip, skip=skip)
    assert chunks[0][0] == 0 and chunks[-1][1] == st.shard_end and all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
    for name in skip:
        v = st.vars[name]
        assert name not in v2c
        inside = [c for c, (s, e) in enumerate(chunks) if s < v.offset + v.numel and e > v.offset]
        assert inside and all(exp[c] == 0 for c in inside), name                 # dead chunks: never launched, never updated
        assert chunks[inside[0]][0] == v.offset and chunks[inside[-1]][1] == v.offset + v.numel
    for name, o, n in table:
        if name in skip or name not in live:
            continue
        cs = v2c[name]
        assert all(exp[c] > 0 for c in cs) and chunks[cs[0]][0] <= o and o + n <= chunks[cs[-1]][1]


def test_fused_update_candidates():
    """optimizer.fusable: big 2-D ``*/Matrix`` variables fed by at most 64 rows; nothing else."""
    import types
    from dynamic_multiview_3d_b200.optimizer import fusable
    def var(name, shape, rows, off=0, trainable=True):
        n = 1
        for d in shape:
            n *= d
        return types.SimpleNamespace(name=name, shape=shape, numel=n, offset=off, trainable=trainable, rows=rows)
    assert fusable(var("fc1/Matrix", (12544, 4096), 64))
    assert fusable(var("a3/Matrix", (4160, 4096), 2, off=16384))
    assert not fusable(var("a3/Matrix", (4160, 4096), 256))          # 4 source frames folded into the batch (config 5)
    assert not fusable(var("a3/Matrix", (4160, 4096), 0))            # never ran forward
    assert not fusable(var("a0/Matrix", (19, 64), 64))               # small
    assert not fusable(var("e3/w", (3, 3, 64, 128), 64))             # not an FC matrix
    assert not fusable(var("fc1/Matrix", (12544, 4096), 64, trainable=False))
    assert not fusable(var("fc1/Matrix", (12544, 4096), 64, off=64))  # not on a chunk-plan boundary


def test_stream_roles_and_tail_lane(monkeypatch):
    """Scheduling knobs of the captured step (functional.py): the chain one priority level above the weight-gradient lanes by
    default, overridable per role; the third weight-gradient lane only in single-process training."""
    from dynamic_multiview_3d_b200 import functional as F
    for k in ("DMV_MAIN_PRIORITY", "DMV_LANE0_PRIORITY", "DMV_LANE1_PRIORITY", "DMV_TAIL_LANE"):
        monkeypatch.delenv(k, raising=False)
    assert (F.stream_priority("main"), F.stream_priority("lane0"), F.stream_priority("lane1"), F.stream_priority("lane2")) == (-1, 0, 0, 0)
    monkeypatch.setenv("DMV_MAIN_PRIORITY", "0")            # historical switch: 0 = the chain at the default priority
    assert F.stream_priority("main") == 0
    monkeypatch.setenv("DMV_MAIN_PRIORITY", "2")
    monkeypatch.setenv("DMV_LANE0_PRIORITY", "1")
    assert (F.stream_priority("main"), F.stream_priority("lane0"), F.stream_priority("lane1")) == (-2, -1, 0)
    before = F.TAIL_LANE
    try:
        F.set_tail_lane(True)
        assert F.TAIL_LANE == 2
        F.set_tail_lane(False)                               # what data_parallel.attach does when gradients are exchanged
        assert F.TAIL_LANE == 0
        monkeypatch.setenv("DMV_TAIL_LANE", "0")
        F.set_tail_lane(True)
        assert F.TAIL_LANE == 0
    finally:
        F.TAIL_LANE = before

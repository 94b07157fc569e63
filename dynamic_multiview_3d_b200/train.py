"""Training driver: restates dyn_mult_view/multi_view_model/train.py (flags :18-22, conf
loading :40-60, loop :117-151, checkpoint cadence :25-31,95-103,134-136) for this build, plus
the CUDA-graph-captured step that the benchmark uses.

    python -m dynamic_multiview_3d_b200.train --hyper path/to/conf.py [--pretrained model123]
"""
import argparse
import importlib.util
import os
import re
import sys
import time
import types

import torch

SUMMARY_INTERVAL = 400   # train.py:25
VAL_INTERVAL = 500       # train.py:28
SAVE_INTERVAL = 10000    # train.py:31


class GraphedTrainStep:
    """model.train_step captured once into a CUDA graph and replayed: removes the per-launch host cost of the ~200
    kernels of a step.  Works for every model class through ModelBase's step interface (``input_spec`` /
    ``train_step(batch)``): a batch is copied into static device buffers (from pinned host memory or device tensors) on
    the same stream before each replay.  Call with a batch dict or with the model's positional tensors (INPUT_KEYS)."""

    def __init__(self, model, warmup=3):
        self.model = model
        dev = model.device
        self.keys = tuple(model.INPUT_KEYS)
        self.static = {k: torch.zeros(shp, dtype=torch.float32, device=dev) for k, shp in model.input_spec().items()}
        self.graph = None
        self.loss = None
        self.warmup = warmup
        self.launches_per_step = 0
        self._stage = None
        self._pending = False
        self._u8 = {}

    # the single-view model's buffers under their historical names
    image0 = property(lambda self: self.static["image0"])
    image1 = property(lambda self: self.static["image1"])
    disp = property(lambda self: self.static["disp"])

    def _batch(self, args):
        if len(args) == 1 and isinstance(args[0], dict):
            return args[0]
        if len(args) != len(self.keys):
            raise TypeError("expected a batch dict or %d tensors %s" % (len(self.keys), self.keys))
        return dict(zip(self.keys, args))

    def capture(self):
        """Warm up (lazy allocations, workspace growth, NCCL channels) and capture.  The warm-up steps are REAL updates,
        so parameters, Adam moments and the step counter are restored afterwards: the reference applies exactly one
        update per iteration (train.py:122), and so does the first call of this object."""
        from . import _lib
        m = self.model
        flat = m.store.flat
        m.flush_updates()               # a deferred optimizer update belongs to the state that is snapshotted
        snap = {k: flat[k].clone() for k in ("master", "m", "v", "half")}
        opt_state = m.optimizer.state.clone()
        # The step's own chain (forward, loss, the dgrad chain of backward) is captured from a HIGH-priority stream; the
        # weight-gradient lanes and the Adam / exchange stream keep the default (lowest) priority.  Kernel nodes inherit
        # the priority of the stream they were captured on, so the block scheduler dispatches the critical chain's CTAs
        # ahead of queued side-stream CTAs instead of behind a 784-CTA weight-gradient or a 2368-CTA Adam grid
        # (profiles/r02_timeline_*.txt: small kernels of the chain waited up to 50 us for SM slots).
        from .functional import stream_priority
        prio = stream_priority("main")
        side = torch.cuda.Stream(device=m.device, priority=prio)
        side.wait_stream(torch.cuda.current_stream(m.device))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                m.train_step(self.static)
        torch.cuda.current_stream(m.device).wait_stream(side)
        torch.cuda.synchronize(m.device)
        self.graph = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(self.graph, stream=side):
            self.loss = m.train_step(self.static)
        self.launches_per_step = _lib.launch_count() - n0
        torch.cuda.synchronize(m.device)
        for k, t in snap.items():
            flat[k].copy_(t)
        m.optimizer.state.copy_(opt_state)
        dp = getattr(m, "_dp", None)
        if dp is not None and hasattr(dp, "reset_deferred"):
            dp.reset_deferred()         # the warm-up steps' pending update is discarded with them
        return self

    def _copy_in(self, batch):
        """Bring a batch into the graph's static fp32 buffers.  uint8 images (the reference's TFRecord pixel format,
        a quarter of the PCIe bytes) are converted on the device: float32(pixel) / 255 (read_tf_records.py:111)."""
        from . import functional as F
        for k, dst in self.static.items():
            src = batch[k]
            if src.dtype == torch.uint8:
                if not src.is_cuda:
                    buf = self._u8.get(k)
                    if buf is None or buf.shape != src.shape:
                        buf = self._u8[k] = torch.empty(src.shape, dtype=torch.uint8, device=dst.device)
                    buf.copy_(src, non_blocking=True)
                    src = buf
                # stored size != model size: central crop + bicubic resize + / 255 in the same kernel (read_tf_records.py:103-111)
                F.prepare_images(src, dst.shape[-2], out=dst)
            else:
                dst.copy_(src, non_blocking=True)

    def replay(self):
        """One more step on the batch that already sits in the static buffers (no copy at all)."""
        self.graph.replay()
        self._after_replay()
        return self.loss

    def _after_replay(self):
        # the replayed step left the late FC matrices' update pending on the device (data_parallel.py: deferred updates);
        # the host-side bookkeeping that an eager train_step does must follow
        dp = getattr(self.model, "_dp", None)
        if dp is not None and getattr(dp, "deferred", None):
            dp.mark_pending()

    def prefetch(self, *args):
        """Start the host->device copy of the NEXT step's batch on a copy stream into staging buffers; it overlaps
        the step that is replayed meanwhile.  The following __call__ with ``staged=True`` consumes it."""
        batch = self._batch(args)
        dev = self.model.device
        if self._stage is None:
            self._stage = {k: torch.empty(self.static[k].shape, dtype=batch[k].dtype, device=dev) for k in self.static}
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._staged_ev = torch.cuda.Event()
            self._consumed_ev = torch.cuda.Event()
            self._consumed_ev.record(torch.cuda.current_stream(dev))
        self._copy_stream.wait_event(self._consumed_ev)          # the previous staged batch has been moved out
        with torch.cuda.stream(self._copy_stream):
            for k, dst in self._stage.items():
                dst.copy_(batch[k], non_blocking=True)
            self._staged_ev.record(self._copy_stream)
        self._pending = True

    def __call__(self, *args, staged=False, prefetch_next=None, async_loss=False):
        """One train step.  ``staged=True``: take the batch handed to prefetch() (a device-side move instead of a PCIe
        copy in front of the step).  ``prefetch_next=batch``: start copying the next step's batch before this step is
        replayed, so the PCIe transfer overlaps it."""
        main = torch.cuda.current_stream(self.model.device)
        if staged:
            main.wait_event(self._staged_ev)
            self._copy_in(self._stage)
            self._consumed_ev.record(main)
            self._pending = False
        else:
            self._copy_in(self._batch(args))
            if self._stage is not None:
                self._consumed_ev.record(main)
        if self.graph is None:
            self.capture()
        if prefetch_next is not None:
            self.prefetch(*(prefetch_next if isinstance(prefetch_next, (tuple, list)) else (prefetch_next,)))
        self.graph.replay()
        self._after_replay()
        if async_loss:
            return self._loss_future(main)
        return self.loss

    def _loss_future(self, main):
        """The step's loss on its way to pinned host memory (4 bytes, D2H behind the step): the caller can enqueue the next
        step before it blocks on ``result()``, so the GPU does not idle between steps while the host reads a scalar.  Two
        slots: read step k's future before calling step k + 2."""
        if not hasattr(self, "_loss_host"):
            self._loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
            self._loss_k = 0
        slot = self._loss_host[self._loss_k & 1]
        self._loss_k += 1
        slot.copy_(self.loss, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(main)
        return LossFuture(slot, ev)


class GraphedRender:
    """model.render for B sources x V viewpoints captured once into a CUDA graph and replayed.  Sources and viewpoints
    are copied into static device buffers (``sources``: dict of [B, H, W, C]; ``viewpoints``: [B, V, viewpoint_dim]) before
    each replay; the result is a dict of static [B, V, H, W, C] tensors that the next replay overwrites.  The graph reads
    the parameters and writes only its own buffers: its workspaces are its own (functional.render_scope), so a captured
    train step and eager renders of other sizes can run in the same process."""

    def __init__(self, model, B, V, warmup=2):
        self.model, self.B, self.V, self.warmup = model, int(B), int(V), warmup
        dev, H = model.device, model.image_shape[0]
        chans = {"image0": 3, "depth0": 1}
        self.sources = {k: torch.zeros((self.B, H, H, chans[k]), dtype=torch.float32, device=dev) for k in model.render_sources()}
        self.viewpoints = torch.zeros((self.B, self.V, model.viewpoint_dim), dtype=torch.float32, device=dev)
        self.role = "graph%d" % id(self)
        self.graph = None
        self.out = None

    def capture(self):
        m = self.model
        m.flush_updates()
        main = torch.cuda.current_stream(m.device)
        side = torch.cuda.Stream(device=m.device)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            for _ in range(self.warmup):          # workspaces grow and modules load outside the capture
                m._render(self.sources, self.viewpoints, role=self.role)
        main.wait_stream(side)
        torch.cuda.synchronize(m.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self.out = m._render(self.sources, self.viewpoints, role=self.role)
        torch.cuda.synchronize(m.device)
        return self

    def __call__(self, sources=None, viewpoints=None):
        """Copy in ``sources`` (fp32, or uint8 pixels prepared on the device) and ``viewpoints`` ([B, V, d] or [V, d]) when
        given, then replay.  Parameters changed by training since the last call are picked up (pending updates flushed)."""
        from . import functional as F
        for k, src in (sources or {}).items():
            dst = self.sources[k]
            if src.dtype == torch.uint8:
                F.prepare_images(src.to(dst.device, non_blocking=True), dst.shape[-2], out=dst)
            else:
                dst.copy_(src, non_blocking=True)
        if viewpoints is not None:
            self.viewpoints.copy_(viewpoints.expand(self.viewpoints.shape) if viewpoints.dim() == 2 else viewpoints, non_blocking=True)
        if self.graph is None:
            self.capture()
        self.model.flush_updates()
        self.graph.replay()
        return self.out


class LossFuture(object):
    def __init__(self, slot, event):
        self.slot, self.event = slot, event

    def result(self):
        self.event.synchronize()
        return float(self.slot)


def install_reference_aliases():
    """Let an unmodified reference conf.py import its model classes by the reference's
    module names (e.g. ``from highdim_angle import AppFlowHighDimAngle``, ``import dyn_mult_view``)."""
    from . import appearance_flow_model as afm
    names = {
        "appearance_flow_model": afm, "highdim_angle": afm, "lowdim_angle": afm, "appearance_flow_tinghui": afm,
    }
    try:
        from . import main_model as mm
        from . import multiobject_appflow as mo
        names["main_model"] = mm
        names["multiobject_appflow"] = mo
    except ImportError:
        pass
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for pkg_name in ("dyn_mult_view", "dyn_mult_view.multi_view_model"):
        if pkg_name not in sys.modules:
            pkg = types.ModuleType(pkg_name)
            pkg.__file__ = os.path.join(here, *pkg_name.split("."), "__init__.py")
            pkg.__path__ = []          # a package without a search path: only the aliases below resolve; anything else
            sys.modules[pkg_name] = pkg  # (e.g. multiobject_main_model, out of scope) raises ModuleNotFoundError
    setattr(sys.modules["dyn_mult_view"], "multi_view_model", sys.modules["dyn_mult_view.multi_view_model"])
    for k, mod in names.items():
        sys.modules.setdefault(k, mod)
        sys.modules.setdefault("dyn_mult_view.multi_view_model." + k, mod)
        setattr(sys.modules["dyn_mult_view.multi_view_model"], k, mod)


def load_conf(path):
    """train.py:40-45: imp.load_source('hyperparams', conf_file).configuration"""
    if not os.path.exists(path):
        sys.exit("Experiment configuration not found")
    install_reference_aliases()
    spec = importlib.util.spec_from_file_location("hyperparams", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.configuration


def checkpoint_iteration(path):
    """train.py:95-103: the iteration number is recovered from the file name ``model<itr>``."""
    m = re.match(r".*model(\d+)", os.path.basename(path) if "/" in path else path)
    return int(m.group(1)) if m else 0


class SummaryWriter:
    """tf.summary.FileWriter(output_dir, flush_secs=10) of train.py:76: TensorBoard event files when the
    ``tensorboard`` package is importable (torch.utils.tensorboard), and always a plain ``scalars.jsonl`` next to them."""

    def __init__(self, out_dir):
        import json
        self._json = json
        self.f = open(os.path.join(out_dir, "scalars.jsonl"), "a")
        self.tb = None
        try:
            from torch.utils.tensorboard import SummaryWriter as TB
            self.tb = TB(log_dir=out_dir, flush_secs=10)
        except Exception:
            self.tb = None

    def add_scalar(self, tag, value, itr):
        self.f.write(self._json.dumps({"tag": tag, "value": float(value), "step": int(itr)}) + "\n")
        if self.tb is not None:
            self.tb.add_scalar(tag, float(value), int(itr))

    def close(self):
        self.f.close()
        if self.tb is not None:
            self.tb.close()


def synthetic_batch(model, seed, rank=0):
    """One synthetic batch (synthetic.py) under the model's INPUT_KEYS -- the stand-in for the TFRecord queue."""
    from . import synthetic as S
    from .multiobject_appflow import MultiObjectAppFlow, MultiViewFusionAppFlow
    H, B = model.image_shape[0], model.batch_size
    vp = "onehot19" if model.viewpoint_dim == 19 else "disp2"
    if isinstance(model, MultiViewFusionAppFlow):
        b = S.make_multiview_multiobject_batch(B, H, model.num_views, seed=seed, rank=rank, viewpoint=vp)
    elif isinstance(model, MultiObjectAppFlow):
        b = S.make_multiobject_batch(B, H, seed=seed, rank=rank)
    else:
        b = S.make_batch(B, H, vp, seed=seed, rank=rank, depth=True)
    return {k: b[k] for k in model.INPUT_KEYS}


def tfrecord_batch(model, fb):
    """Map the reader's feature names (read_tf_records.py:56-63) to the model's input names."""
    alias = {"disp": "displacement", "displacement": "displacement"}
    return {k: fb[alias.get(k, k)] for k in model.INPUT_KEYS}


def build_model(conf, build_loss=True, device=None):
    """train.py:57-65: ``conf['model']`` when given, else Base_Prediction_Model (which needs 'use_color' and/or
    'use_depth'; the reference's nobg_nodm confs set neither and belong to the MV3D scripts, out of scope)."""
    from .main_model import Base_Prediction_Model
    Model = conf["model"] if "model" in conf else Base_Prediction_Model
    return Model(conf, load_tfrec=True, build_loss=build_loss, device=device)


def to_device_f32(batch, device, size=None):
    """Host batch -> device float32 tensors for the un-captured calls; uint8 pixels go through the reader's image
    preparation on the device (crop + bicubic resize to ``size`` + / 255, read_tf_records.py:103-111)."""
    from . import functional as F
    out = {}
    for k, v in batch.items():
        t = v.to(device, non_blocking=True)
        out[k] = F.prepare_images(t, size if size is not None else t.shape[-2]) if t.dtype == torch.uint8 else t
    return out


def main(argv=None):
    """train.py:34-157.  Under ``torchrun`` (WORLD_SIZE > 1) every rank builds the model on its own GPU, the gradient
    exchange of data_parallel.py is attached, each rank reads its own shard of batches, and rank 0 alone logs, writes
    summaries and saves (state_dict is a collective call under sharded data parallelism)."""
    ap = argparse.ArgumentParser()
    ap.add_argument("--hyper", default="conf.py", help="hyperparameters configuration file")
    ap.add_argument("--visualize", default="", help="model within hyperparameter folder to visualise")
    ap.add_argument("--device", default="0", help="the value for CUDA_VISIBLE_DEVICES")
    ap.add_argument("--pretrained", default=None, help="path to model file from which to resume training")
    ap.add_argument("--synthetic", action="store_true", default=True, help="synthetic car-render batches (no TFRecords)")
    ap.add_argument("--tfrecords", action="store_true", help="read conf['data_dir'] TFRecords (read_tf_records.py) instead of synthetic batches")
    ap.add_argument("--num_iterations", type=int, default=None)
    ap.add_argument("--eager", action="store_true", help="do not capture the step into a CUDA graph")
    args = ap.parse_args(argv)
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1:
        os.environ.setdefault("CUDA_VISIBLE_DEVICES", str(args.device))
    conf = load_conf(args.hyper)
    if args.num_iterations is not None:
        conf["num_iterations"] = args.num_iterations
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out_dir = conf.get("output_dir", ".")
    if args.visualize:                        # train.py:47-55
        conf["visualize"] = os.path.join(out_dir, args.visualize)
        conf["batch_size"] = 10
        conf["test_mode"] = ""
    model = build_model(conf, build_loss=not args.visualize)
    os.makedirs(out_dir, exist_ok=True)
    if args.visualize:                        # train.py:86-93: restore <output_dir>/<visualize> and write the figures
        if os.path.exists(conf["visualize"]):
            model.load_state_dict(torch.load(conf["visualize"], map_location="cpu"))
        b = synthetic_batch(model, seed=99)
        info = model.visualize(*(torch.from_numpy(b[k]).to(model.device) for k in model.INPUT_KEYS))
        print("loss", info["loss"])
        if info.get("max_resample_coord") == info.get("max_resample_coord"):      # not NaN: the single-view flow models
            print("max resample coord:", info["max_resample_coord"])
        return
    itr_0 = 0
    if args.pretrained:                       # train.py:95-103: resume AT the checkpoint's iteration
        model.load_state_dict(torch.load(args.pretrained, map_location="cpu"))
        itr_0 = checkpoint_iteration(args.pretrained)
        print("resuming training at iteration: ", itr_0)
    # world > 1: the data-parallel exchange.  world == 1: the same chunk pipeline without an exchange -- Adam chunk by chunk
    # behind its gradients, the last FC matrix's update deferred into the next forward pass (data_parallel.py)
    if world > 1 or os.environ.get("DMV_OVERLAP_ADAM", "1") == "1":
        from . import data_parallel
        data_parallel.attach(model, bucket_mb=float(os.environ.get("DMV_DP_CHUNK_MB", "128" if world > 1 else "32")))
    step = model.train_step if args.eager else GraphedTrainStep(model)
    writer = SummaryWriter(out_dir) if rank == 0 else None
    t_iter = []
    reader = val_reader = None
    if args.tfrecords:                       # train.py:57 load_tfrec=True -> read_tf_records.build_tfrecord_input
        from .read_tf_records import build_tfrecord_input
        rconf = dict(conf, image_size=model.image_shape[0])
        reader = build_tfrecord_input(rconf, training=True)
        val_reader = build_tfrecord_input(rconf, training=False)

    def next_batch(itr, val=False):
        if reader is not None:               # uint8 pixels go over PCIe as stored; /255 happens on the device (_copy_in)
            b = tfrecord_batch(model, (val_reader if val else reader).next_batch())
        else:                                # validation batches come from a disjoint seed range (train_val_split stand-in)
            b = synthetic_batch(model, seed=(10 ** 6 if val else 1234) + itr, rank=rank)
        return {k: torch.from_numpy(v).pin_memory() for k, v in b.items()}

    # the next batch is produced (synthetic generator or TFRecord reader + pinning) by a worker thread while the current step
    # runs, so the loop is not bound by the host-side batch construction
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=1)
    last_itr = conf["num_iterations"]
    ahead = pool.submit(next_batch, itr_0) if itr_0 <= last_itr else None
    for itr in range(itr_0, last_itr + 1):
        t0 = time.time()
        batch = ahead.result()
        ahead = pool.submit(next_batch, itr + 1) if itr < last_itr else None
        loss = step(to_device_f32(batch, model.device, model.image_shape[0])) if args.eager else step(batch)
        if itr % 10 == 0 and rank == 0:
            print("%d %g" % (itr, float(loss)))
        if itr % VAL_INTERVAL == 0 and itr != 0:            # train.py:128-132: one validation batch, no update
            vloss = float(model.eval_loss(to_device_f32(next_batch(itr, val=True), model.device, model.image_shape[0])))
            if writer is not None:
                writer.add_scalar("val_loss", vloss, itr)
        if itr % SAVE_INTERVAL == 0 and itr != 0:           # train.py:134-136 (collective under sharded data parallelism)
            sd = model.state_dict()
            if rank == 0:
                torch.save(sd, os.path.join(out_dir, "model%d" % itr))
        t_iter.append(time.time() - t0)
        if itr % 100 == 1 and rank == 0:
            avg = sum(t_iter) / len(t_iter)
            print("time per iteration: %.4fs; expected for complete training: %.2fh" % (avg, avg / 3600 * conf["num_iterations"]))
        # train.py:150 writes on every iteration NOT divisible by 400 (a bug); the intended cadence is kept (SURVEY App. A)
        if itr % SUMMARY_INTERVAL == 0 and writer is not None:
            writer.add_scalar("training_loss", float(loss), itr)
    pool.shutdown()
    sd = model.state_dict()
    if rank == 0:
        torch.save(sd, os.path.join(out_dir, "model"))
        writer.close()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)          # a process group whose collectives live in a captured graph can block in destroy_process_group


if __name__ == "__main__":
    main()

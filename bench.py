#!/usr/bin/env python
"""Benchmark of the appearance-flow training hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--dump-outputs DIR]

Own arm: one "step" = forward + backward + Adam of the single-view appearance-flow model on a
synthetic 224x224 car-render batch of 64 per GPU (BASELINE configs[1]; data parallel over N
GPUs = weak scaling, configs[2] shape of work per GPU), replayed from a captured CUDA graph.
  value  : samples/s with the batch resident in HBM (CUDA events, max over ranks), K timed steps
  e2e    : samples/s through the public API with pinned-host inputs copied H2D and the loss
           read back D2H inside the timed region, every step; K more timed steps
  roofline / sampler : the dominant kernel of the step and the standalone sampler kernels
           against MEASURED_PEAKS.json
  cpu_baseline : the oracle's torch-CPU port of the same step on the host cores (rank 0, N=1)
Reference arm (--impl reference): that CPU port alone, on a bounded batch-8 sample.
--config selects the BASELINE.json workload (default 2 = configs[1], the one the metric is quoted on; 3 = high-dim
viewpoint variant, 4 = cars_colordepth RGB+depth with per-channel L1, 5 = 4 source frames + confidence fusion on the
multi-object trunk); every one is 64 samples per GPU at 224x224, V=19, captured into one CUDA graph.
--dump-outputs DIR writes what the last timed step computed on rank 0 to DIR/<name>.npy (dump_outputs()).  The inputs
and initial weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, V, BATCH = 224, 19, 64
FWD_GFLOP_PER_SAMPLE = 3.39          # SURVEY 8(a) table
METRIC = "train samples/s @224^2 appflow"


WORKLOADS = {
    2: ("AppearanceFlowModel", {}, "single-view appearance-flow train step (fwd+bwd+Adam), 224x224 synthetic car renders, "
        "one-hot azimuth V=19, batch 64 per GPU (configs[1]; N>1 = batch-sharded data parallel)", "l2 (reference)"),
    3: ("AppFlowHighDimAngle", {}, "appearance flow + offset head with the high-dim viewpoint encoding (highdim_angle.py), 224x224, "
        "one-hot azimuth V=19, batch 64 per GPU = 512 on 8 GPUs (configs[2])", "l2 (reference)"),
    4: ("Base_Prediction_Model", {"use_color": "", "use_depth": "", "depth_lr_factor": 0.1, "loss": "l1"},
        "cars_colordepth: joint RGB+depth decoder (two pre-encoders, split trunk, tanh heads), per-channel L1 with weights "
        "(1,1,1,0.1), 224x224, batch 64 per GPU (configs[3])", "l1 per channel"),
    5: ("MultiViewFusionAppFlow", {"num_views": 4, "use_depth": 0.1},
        "4 source frames per sample of a two-object scene on the multi-object trunk (colour, depth, 2 masks), one 3-channel "
        "flow + confidence head per frame, softmax fusion, 224x224, 64 samples (256 frames) per GPU (configs[4])", "l2"),
}


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        try:
            d = json.load(open(f))
            p.update({k: d[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in d})
            p["src"] = "measured"
        except Exception:
            pass
    return p


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full summary
    (profiles/r01_traffic.json, written by tools/summarise_ncu.py); None when the kernel was not captured."""
    try:
        for name in ("r02_traffic.json", "r01_traffic.json"):
            v = json.load(open(os.path.join(ROOT, "profiles", name))).get(kernel)
            if v is not None:
                return v
        return None
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region: NVML every 10 ms (nvidia-smi fallback)."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.stop_flag, self.smax = index, [], set(), False, None
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].strip().isdigit():
                return int(ids[index])
        return index

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.01 if self.nv else 0.2)

    def sample(self):
        if self.nv:
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in self.REASONS:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            f = [x.strip() for x in out.split(",")]
            self.sm.append(float(f[0]))
            self.smax = float(f[1])
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)
        except Exception:
            pass

    def summary(self):
        self.stop_flag = True
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.smax, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": "nvml" if self.nv else "nvidia-smi"}


def reference_arm(args, rank):
    """The reference path's CPU implementation (oracle torch-CPU port) of the selected config, bounded sample,
    every host thread (oracle/cpu_step.py sets the count itself: torchrun exports OMP_NUM_THREADS=1)."""
    if rank != 0:
        return
    from oracle import cpu_step
    b = 8
    wu = max(1, min(args.warmup, 2))
    sps, ts, cores = cpu_step.time_steps(b, H, V, steps=max(1, min(args.steps, 10)), warmup=wu, config=args.config)
    ms = 1e3 * sorted(ts)[len(ts) // 2]
    what = cpu_step.make_config_step(args.config, 32, V)[2]
    sample = "batch %d of the 224^2 step of config %d (%s), fp32 fwd+bwd+Adam, torch-CPU port of the oracle graph" % (b, args.config, what)
    line = {"impl": "reference", "metric": METRIC, "value": round(sps, 3), "unit": "samples/s", "n_gpus": args.gpus, "steps": len(ts),
            "warmup": wu, "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "CPU reference arm: " + WORKLOADS[args.config][2] + " -- timed at batch %d" % b,
                       "bench_config": args.config, "per_gpu_batch": b, "image": H, "threads": cores},
            "cpu_baseline": {"value": round(sps, 3), "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": round(sps, 3), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def sampler_microbench(torch, pk, iters=20):
    """Standalone sampler kernels at 64 x 224^2 x 3; four rotating input sets (4 x 103 MB > L2)."""
    from dynamic_multiview_3d_b200 import _lib
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev).manual_seed(1)
    sets = []
    for _ in range(4):
        data = torch.rand((BATCH, H, H, 3), device=dev, generator=g)
        flow = (torch.rand((BATCH, H, H, 2), device=dev, generator=g) - 0.5) * 6
        go = torch.randn((BATCH, H, H, 3), device=dev, generator=g)
        sets.append((data, flow, go))
    px = BATCH * H * H
    st = torch.cuda.current_stream().cuda_stream
    out = torch.empty((BATCH, H, H, 3), device=dev)
    gw = torch.empty((BATCH, H, H, 2), device=dev)
    gd = torch.empty((BATCH, H, H, 3), device=dev)
    ws = torch.empty(max(1, _lib.load().dmv_sampler_bwd_workspace_size(BATCH, H, H, 3, H, H)), dtype=torch.uint8, device=dev)

    def fwd(d, f, go):
        _lib.call("dmv_sampler_fwd", d.data_ptr(), f.data_ptr(), out.data_ptr(), None, None, BATCH, H, H, 3, H, H, 1, st)

    def bwd_flow(d, f, go):
        _lib.call("dmv_sampler_bwd", d.data_ptr(), f.data_ptr(), go.data_ptr(), None, gw.data_ptr(), BATCH, H, H, 3, H, H, 1,
                  ws.data_ptr(), ws.numel(), st)

    def bwd_both(d, f, go):
        _lib.call("dmv_sampler_bwd", d.data_ptr(), f.data_ptr(), go.data_ptr(), gd.data_ptr(), gw.data_ptr(), BATCH, H, H, 3, H, H, 1,
                  ws.data_ptr(), ws.numel(), st)

    def timeit(fn, nbytes):
        for i in range(3):
            fn(*sets[i % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(*sets[i % 4])
        e1.record()
        torch.cuda.synchronize()
        us = 1e3 * e0.elapsed_time(e1) / iters
        gbs = nbytes / (us * 1e-6) / 1e9
        return {"us": round(us, 2), "gbs": round(gbs, 1), "frac": round(gbs / pk["hbm_gbs"], 4), "bytes": nbytes}

    res = {"fwd": timeit(fwd, px * (8 + 8 * 3)),                    # SURVEY 8(d): 8 + 8C B/px
           "bwd_grad_flow": timeit(bwd_flow, px * (16 + 8 * 3)),    # 16 + 8C (source is a network input)
           "bwd_both": timeit(bwd_both, px * (16 + 12 * 3)),        # 16 + 12C
           "shape": "64x224x224x3 fp32, flow U(-3,3), reference (Y,X) grid fused", "l2_policy": "4 rotating input sets (412 MB)"}
    # second regime: smooth flows (rotation by 8..11 degrees about the centre), the shape of a trained network's output;
    # U(-3,3) jitter is the worst case for shared-memory bank conflicts in the tap gathers
    import math
    ii, jj = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float32), torch.arange(H, device=dev, dtype=torch.float32), indexing="ij")
    c0 = (H - 1) / 2
    for k in range(4):
        a = math.radians(8.0 + k)
        u = math.cos(a) * (ii - c0) - math.sin(a) * (jj - c0) + c0
        v = math.sin(a) * (ii - c0) + math.cos(a) * (jj - c0) + c0
        sets[k] = (sets[k][0], torch.stack([u - ii, v - jj], -1).unsqueeze(0).repeat(BATCH, 1, 1, 1).contiguous(), sets[k][2])
    res["smooth"] = {"fwd": timeit(fwd, px * (8 + 8 * 3)), "bwd_grad_flow": timeit(bwd_flow, px * (16 + 8 * 3)),
                     "bwd_both": timeit(bwd_both, px * (16 + 12 * 3)),
                     "shape": "same tensors, flow = rotation field of 8..11 degrees"}
    return res


def conv_microbench(torch, pk, iters=20):
    """The heaviest conv layer of the graph (e0_0 / d1_0: 5x5, 32->32 at 112^2, B=64: 41.1 GFLOP) through the C ABI:
    forward, input gradient and weight gradient against the measured BURST bf16 peak -- the figure that applies to a
    kernel timed alone (20 back-to-back launches); the fraction of the sustained peak is reported beside it."""
    from dynamic_multiview_3d_b200 import _lib
    dev = torch.device("cuda", torch.cuda.current_device())
    L = _lib.load()
    B, Hc, C, k = BATCH, 112, 32, 5
    bf = torch.bfloat16
    x = torch.randn((B, Hc, Hc, C), device=dev).to(bf)
    w = (torch.randn((k, k, C, C), device=dev) * 0.05).to(bf)
    b = torch.zeros(C, device=dev)
    y = torch.empty((B, Hc, Hc, C), device=dev, dtype=bf)
    dy = torch.randn((B, Hc, Hc, C), device=dev).to(bf)
    dx = torch.empty_like(x)
    dw = torch.empty((k, k, C, C), device=dev)
    ws = torch.empty(max(L.dmv_conv_workspace_size(B, Hc, Hc, C, C, k, k, 1), L.dmv_wgrad_workspace_size(B, Hc, Hc, C, C, k, k, 1), 256),
                     dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    flop = 2.0 * B * Hc * Hc * k * k * C * C
    calls = {
        "fwd": lambda: _lib.call("dmv_conv2d_fwd", x.data_ptr(), 0, w.data_ptr(), b.data_ptr(), y.data_ptr(), 0, B, Hc, Hc, C, C, k, k, 1, 1,
                                 ws.data_ptr(), ws.numel(), 0, st),
        "dgrad": lambda: _lib.call("dmv_conv2d_dgrad", dy.data_ptr(), w.data_ptr(), dx.data_ptr(), None, 0, B, Hc, Hc, C, C, k, k, 1, ws.data_ptr(),
                                   ws.numel(), 0, st),
        "wgrad": lambda: _lib.call("dmv_conv2d_wgrad", x.data_ptr(), 0, dy.data_ptr(), dw.data_ptr(), None, B, Hc, Hc, C, C, k, k, 1,
                                   ws.data_ptr(), ws.numel(), 0, st),
    }
    out = {"layer": "e0_0 / d1_0: conv 5x5 stride 1, 32->32, 64x112x112 (bf16 in, fp32 accumulate)", "flop_per_launch": flop,
           "peak_tflops": pk["bf16_tflops"], "peak_src": pk["src"] + " (burst)", "peak_tflops_sustained": pk["bf16_tflops_sustained"]}
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = 1e3 * e0.elapsed_time(e1) / iters
        tf = flop / us / 1e6
        out[name] = {"us": round(us, 2), "tflops": round(tf, 1), "frac": round(tf / pk["bf16_tflops"], 4),
                     "frac_of_sustained": round(tf / pk["bf16_tflops_sustained"], 4)}
    return out


def layer_gflop(B):
    """fwd GFLOP per layer at 224^2 (2*M*N*K), SURVEY 8(a) table."""
    t = {}

    def conv(name, hw, k, cin, cout):
        t[name] = 2.0 * B * hw * hw * k * k * cin * cout / 1e9
    conv("e0", 112, 5, 3, 32); conv("e0_0", 112, 5, 32, 32); conv("e1", 56, 5, 32, 32); conv("e1_0", 56, 5, 32, 32)
    conv("e2", 28, 5, 32, 64); conv("e2_0", 28, 5, 64, 64); conv("e3", 14, 3, 64, 128); conv("e3_0", 14, 3, 128, 128)
    conv("e4", 7, 3, 128, 256); conv("e4_0", 7, 3, 256, 256)
    for n, k_, n_ in [("fc1", 12544, 4096), ("a3", 4160, 4096), ("a4", 4096, 4096), ("a5", 4096, 12544), ("a0", V, 64),
                      ("a1", 64, 64), ("a2", 64, 64)]:
        t[n] = 2.0 * B * k_ * n_ / 1e9
    conv("d4", 7, 3, 256, 128); conv("d4_0", 14, 3, 128, 128); conv("d3", 14, 3, 128, 64); conv("d3_0", 28, 5, 64, 64)
    conv("d2", 28, 5, 64, 32); conv("d2_0", 56, 5, 32, 64); conv("d1", 56, 5, 64, 32); conv("d1_0", 112, 5, 32, 32)
    conv("flow_field", 112, 5, 32, 2)
    return t


# the outputs of a step that each benchmarked model class holds after train_step (as configured in WORKLOADS)
DUMP_OUTPUTS = {"AppearanceFlowModel": ("flow_field", "gen"), "AppFlowHighDimAngle": ("flow_field", "gen"),
                "Base_Prediction_Model": ("gen_image1", "gen_dimage1"),
                "MultiViewFusionAppFlow": ("flow_field", "gens", "logits", "fused")}
DUMP_MAX_OUTPUT = 1 << 21        # elements per output array (8 MB in float32)
DUMP_MAX_PARAM = 1 << 18         # elements per parameter (1 MB); the FC matrices are 17M-51M elements
DUMP_MAX_BYTES = 64 << 20


def _dump_sample(t, cap, name):
    """``t`` as a float32 array: whole when it has at most ``cap`` elements; otherwise ``cap`` of its flattened elements
    at indices drawn without replacement from a generator seeded with ``name``, in ascending order -- the same indices
    on every run and build."""
    import numpy as np
    import torch
    x = t.detach()
    if x.numel() > cap:
        idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(x.numel(), cap, replace=False))
        x = x.reshape(-1)[torch.from_numpy(idx).to(x.device)]
    return x.float().cpu().numpy()


def dump_outputs(out_dir, model, loss, world, rank):
    """What the last timed step computed, one ``out_dir/<name>.npy`` per array: ``loss`` (float64 scalar), the model's
    outputs of that step (``gen``, ``flow_field``, ...; rank 0's shard of the batch under data parallelism) and every
    parameter after the step's update (``param.<variable name with '/' -> '.'>``), float32.  Arrays larger than
    DUMP_MAX_OUTPUT / DUMP_MAX_PARAM elements are written as the fixed seeded sample of _dump_sample().  Collective
    under data parallelism: every rank calls it, rank 0 writes."""
    import numpy as np
    import torch
    dp = getattr(model, "_dp", None)
    if world > 1 and hasattr(dp, "gather_full_state"):
        dp.gather_full_state()       # sharded: the fp32 masters live with their owning rank
    else:
        model.flush_updates()        # the late FC matrices' update of the last step may still be pending
    torch.cuda.synchronize()
    if rank != 0:
        return
    arrays = {"loss": np.asarray(loss, dtype=np.float64)}
    for name in DUMP_OUTPUTS[type(model).__name__]:
        t = getattr(model, name, None)
        if not isinstance(t, torch.Tensor):
            raise RuntimeError("%s holds no output %r after its train step" % (type(model).__name__, name))
        arrays[name] = _dump_sample(t, DUMP_MAX_OUTPUT, name)
    for name, v in model.store.vars.items():
        key = "param." + name.replace("/", ".")
        arrays[key] = _dump_sample(v.master, DUMP_MAX_PARAM, key)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json workload (see WORKLOADS)")
    ap.add_argument("--loss", default=None, help="override the workload's loss mode (l1|l2)")
    ap.add_argument("--algo", default=None, help="auto|simt|tcgen05 (default: library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-micro", action="store_true")
    ap.add_argument("--eager", action="store_true", help="do not capture a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, outputs and updated parameters of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl own)")
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly ONE JSON line: everything else a library prints there (e.g. NCCL's version banner)
    # is sent to stderr by pointing fd 1 at fd 2 and keeping the real stdout aside
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        reference_arm(args, rank)
        return 0

    import torch
    import torch.distributed as dist
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import _lib, data_parallel, functional as F
    from dynamic_multiview_3d_b200.train import GraphedTrainStep, synthetic_batch

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product path has no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    W = max(3, args.warmup)
    K = args.steps

    cls_name, extra, workload, loss_name = WORKLOADS[args.config]
    conf = {"batch_size": BATCH, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": V, "loss": "l2", "seed": 0}
    conf.update(extra)
    if args.loss:
        conf["loss"] = args.loss
        loss_name = args.loss
    if args.algo:
        conf["algo"] = args.algo
    Model = getattr(pkg, cls_name)
    model = Model(conf)
    # N > 1: sharded data parallelism.  N == 1: the same chunk pipeline without the exchange -- Adam runs chunk by chunk on a
    # side stream as soon as a chunk's gradients are complete, so the HBM-bound update overlaps the rest of backward.
    exchange = "none"
    if world > 1 or os.environ.get("DMV_OVERLAP_ADAM", "1") == "1":
        red = data_parallel.attach(model, bucket_mb=float(os.environ.get("DMV_DP_CHUNK_MB", "128" if world > 1 else "32")))
        if world > 1:
            exchange = getattr(red, "mode", "allreduce")
            if exchange == "fused":
                exchange += " (one kernel per chunk over peer memory, %s)" % ("multimem in-switch reduction" if red.px.multicast else "fixed-order peer loads")
    b = synthetic_batch(model, seed=1234, rank=rank)
    # The host batch is held in the reference's storage format: uint8 pixels (read_tf_records.py:104-111, images are
    # tf.decode_raw(..., tf.uint8) / 255).  The same quantised images, converted on the device, are the HBM-resident batch.
    u8 = not args.eager and os.environ.get("DMV_BENCH_F32_INPUT", "0") != "1"
    import numpy as np
    host, devb = {}, {}
    for k, v in b.items():
        if u8 and v.ndim >= 4:
            host[k] = torch.from_numpy(np.clip(np.rint(v * 255.0), 0, 255).astype(np.uint8)).pin_memory()
            t8 = host[k].to(dev)
            devb[k] = torch.empty(t8.shape, dtype=torch.float32, device=dev)
            _lib.call("dmv_u8_to_f32", t8.data_ptr(), devb[k].data_ptr(), t8.numel(), 255.0, torch.cuda.current_stream().cuda_stream)
        else:
            host[k] = torch.from_numpy(v).pin_memory()
            devb[k] = host[k].to(dev)
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    if args.eager:
        def step_fn(batch):
            return model.train_step({k: v.to(dev, non_blocking=True) for k, v in batch.items()})
        n0 = _lib.launch_count()
        step_fn(devb)
        launches = _lib.launch_count() - n0
    else:
        step = GraphedTrainStep(model, warmup=2)
        step(devb)
        step_fn = step
        launches = step.launches_per_step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing: the batch sits in the captured step's static input buffers
    resident = (lambda: step.replay()) if not args.eager else (lambda: step_fn(devb))
    for _ in range(W):
        step_fn(devb)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        loss = resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / K
    # ---------------- end-to-end timing (pinned host in, loss out, every step)
    barrier()
    t0 = time.perf_counter()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    last = 0.0
    # every step copies its batch from pinned host memory and reads its loss back.  With the captured step the copy of
    # step k+1 is issued on a copy stream before step k is replayed (GraphedTrainStep.prefetch), so PCIe overlaps compute;
    # step 0's copy is not hidden.  K copies and K loss reads lie inside the timed region.
    pipelined = not args.eager
    hb = host
    if pipelined:
        step.prefetch(hb)
    # The loss of every step is read on the host (4 bytes D2H per step, inside the timed region); with the captured step the
    # read of step k is issued as an async copy behind it and awaited after step k+1 has been enqueued (LossFuture), so the GPU
    # does not idle while the host fetches a scalar.
    fut = None
    for k in range(K):
        if pipelined:
            nxt = step(staged=True, prefetch_next=hb if k + 1 < K else None, async_loss=True)
            if fut is not None:
                last = fut.result()              # D2H read of step k-1's result
            fut = nxt
        else:
            loss = step_fn(hb)
            last = float(loss)                   # D2H read of the step's result
    if fut is not None:
        last = fut.result()
    ee1.record()
    barrier()
    ms_e2e = max(ee0.elapsed_time(ee1), 1e3 * (time.perf_counter() - t0)) / K
    clocks = sampler.summary() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, model, last, world, rank)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    value = world * BATCH / (ms * 1e-3)
    e2e = world * BATCH / (ms_e2e * 1e-3)

    if rank != 0:
        # the remaining work (per-kernel profile, microbenchmarks, CPU baseline) is rank 0's alone.  Wait for it on
        # the rendezvous store -- not on an NCCL barrier -- and leave without tearing the communicator down: a
        # process group whose collectives were captured into a live CUDA graph can block in destroy_process_group.
        finish(world, rank)
        return 0

    # ---------------- per-kernel profile of one eager step -> dominant kernel + roofline
    roof, top = None, []
    if world == 1:
        try:
            # a second, un-pipelined model: every call runs alone on the current stream, so its CUDA-event time is the
            # kernel's own duration (the timed model overlaps Adam chunks with backward on a side stream)
            pmodel = Model(conf)
            for _ in range(2):
                pmodel.train_step(devb)
            with F.profile_calls() as prof:
                pmodel.train_step(devb)
            agg = {}
            for name, tag, t_ms in prof.records:
                agg[(name, tag)] = agg.get((name, tag), 0.0) + t_ms
            total = sum(agg.values())
            ranked = sorted(agg.items(), key=lambda kv: -kv[1])
            top = [{"call": k[0], "var": k[1], "ms": round(v, 4), "share": round(v / total, 4)} for k, v in ranked[:8]]
            gf = layer_gflop(BATCH) if args.config in (2, 3) else {}
            # the dominant kernel the roofline is stated for: the first entry of the ranking that has an algorithmic byte /
            # flop count (other models' lines may be led by a kernel without one, e.g. the multi-frame fusion loss)
            for (dname, dtag), dms in ranked[:6]:
                lname = dtag.split("/")[0]
                if dname == "dmv_linear_wgrad_adam":
                    # the FC matrix's weight gradient + Adam in one pass (csrc/fc_adam.cu): SURVEY 8(d)'s 28 B/param minus the
                    # gradient that is never written or read = 24 B/param (theta, m, v in and out); the bf16 copy (2 B/param)
                    # is moved as well and reported separately.  The bf16 operands (x, dy: < 3 MB) stay in L2.
                    var = pmodel.store.vars[dtag]
                    nbytes = 24.0 * var.numel
                    gbs = nbytes / (dms * 1e-3) / 1e9
                    roof = {"bound": "hbm", "kernel": "dmv_linear_wgrad_adam[%s]" % dtag, "achieved": round(gbs, 1), "peak": pk["hbm_gbs"],
                            "unit": "GB/s", "frac": round(gbs / pk["hbm_gbs"], 4),
                            "traffic": ncu_traffic("fc_wgrad_adam_stream_kernel") if (var.numel == 12544 * 4096 and BATCH <= 64) else None,
                            "peak_src": pk["src"], "bytes_per_launch": nbytes, "bytes_moved_per_launch": 26.0 * var.numel,
                            "ms": round(dms, 4), "share_of_step": round(dms / total, 4)}
                elif lname in gf:
                    tf = gf[lname] / dms          # GFLOP / ms == TFLOP/s
                    peak = pk["bf16_tflops_sustained"]
                    roof = {"bound": "tensor", "kernel": "%s[%s]" % (dname, dtag), "achieved": round(tf, 2), "peak": peak,
                            "unit": "TFLOP/s", "frac": round(tf / peak, 5), "traffic": None, "peak_src": pk["src"] + " (sustained)",
                            "flops_per_launch": gf[lname] * 1e9, "ms": round(dms, 4), "share_of_step": round(dms / total, 4)}
                elif dtag == "adam":
                    # SURVEY 8(d): 28 B/param (read theta, g, m, v; write theta, m, v).  The kernel also writes the bf16 compute
                    # copy (2 B/param), reported separately as bytes_moved_per_launch; `achieved` uses the 8(d) figure.
                    n_adam = pmodel.store.total - sum(v.numel for v in pmodel.store.vars.values() if v.fused_adam)   # fused FC
                    nbytes = 28.0 * n_adam                                                           # matrices are not in this launch
                    gbs = nbytes / (dms * 1e-3) / 1e9
                    roof = {"bound": "hbm", "kernel": "dmv_adam_multi", "achieved": round(gbs, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                            "frac": round(gbs / pk["hbm_gbs"], 4), "traffic": ncu_traffic("adam_multi_kernel[%d]" % n_adam), "peak_src": pk["src"],
                            "bytes_per_launch": nbytes, "bytes_moved_per_launch": 30.0 * n_adam, "params": n_adam,
                            "ms": round(dms, 4), "share_of_step": round(dms / total, 4)}
                if roof is not None:
                    break
        except Exception as ex:      # the profile is explanatory; never lose the bench line over it
            roof = {"error": repr(ex)[:200]}
    micro = None
    if args.config != 2:
        args.no_micro = True          # the standalone sampler / conv microbenchmarks belong to the headline config's line
    if not args.no_micro:
        try:
            micro = sampler_microbench(torch, pk)
        except Exception as ex:
            micro = {"error": repr(ex)[:200]}
    conv = None
    if not args.no_micro:
        try:
            conv = conv_microbench(torch, pk)
        except Exception as ex:
            conv = {"error": repr(ex)[:200]}
    if roof is None and micro and "fwd" in micro:
        roof = {"bound": "hbm", "kernel": "sampler_fwd", "achieved": micro["fwd"]["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": micro["fwd"]["frac"], "traffic": None, "peak_src": pk["src"]}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_step
        sps, ts, cores = cpu_step.time_steps(8, H, V, steps=3, warmup=1, config=args.config)
        cpu = {"value": round(sps, 3), "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "batch 8 of the same 224^2 step (config %d): fp32 fwd+bwd+Adam, torch-CPU port of the oracle graph, 3 timed steps" % args.config}

    step_tflops = 3 * FWD_GFLOP_PER_SAMPLE * BATCH / ms if args.config in (2, 3) else None     # GFLOP/ms = TFLOP/s per GPU
    line = {"metric": METRIC, "value": round(value, 2), "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload, "bench_config": args.config, "model_class": cls_name,
                       "per_gpu_batch": BATCH, "global_batch": BATCH * world, "image": H, "loss": loss_name,
                       "parallelism": "dp%d" % world, "exchange": exchange, "cuda_graph": not args.eager,
                       "host_input": "uint8 pixels (reference TFRecord format), /255 on the device" if u8 else "float32", "algo": args.algo or F.get_default_algo(),
                       "l2_policy": "per-step working set (parameters, Adam state, activations: several GB) >> 126 MB L2"},
            "e2e": {"value": round(e2e, 2), "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": round(ms_e2e, 4)},
            "gpu_launches": int(launches * K), "launches_per_step": int(launches),
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "sampler": micro, "conv": conv, "top_kernels": top,
            "step_tflops_per_gpu": round(step_tflops, 2) if step_tflops else None, "final_loss": last}
    emit(line)
    finish(world, rank)
    return 0


_REAL_STDOUT = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def finish(world, rank):
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        import torch.distributed as dist
        try:
            store = dist.distributed_c10d._get_default_store()
            if rank == 0:
                store.set("dmv_bench_done", "1")
            else:
                store.wait(["dmv_bench_done"])
        except Exception:
            pass
        os._exit(0)


if __name__ == "__main__":
    import signal
    signal.signal(signal.SIGALRM, lambda *a: os._exit(3))    # never sit on a GPU box: hard stop after 20 minutes
    signal.alarm(1200)
    sys.exit(main())

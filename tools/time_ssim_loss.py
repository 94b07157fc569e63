"""SSIM + L1 training objective on the B200: kernel times and the captured train step.

Kernels, at B = 64, 224 x 224, C = 3, under a +-3 pixel jitter flow and a smooth 10-degree rotation flow (reference (Y,X)
grid added in the kernel), with CUDA events, cycling through four input sets (about 670 MB, more than the 126 MB L2):
  composition  dmv_sampler_fwd, dmv_ssim_loss_fwd_bwd, the grad_wf half of dmv_sampler_bwd: the SSIM training tail
  l1_fused     dmv_sampler_loss_fused in L1 mode (warp, loss and flow gradient in one launch), for comparison
  ssim_alone   dmv_ssim_loss_fwd_bwd on a stored gen
Algorithmic bytes per output pixel: 16 + 12C for the two warp-loss arms (source, target, gen out: 4C each; flow in,
flow gradient out: 8 each), 12C for ssim_alone (gen, target, gradient).  Achieved bytes/s is that count over the best
window's time; the share is of the 6548.5 GB/s HBM peak measured on this card model.

Step: config 2's model (AppearanceFlowModel, V = 19) at B = 64, 224 x 224, as a captured train step (GraphedTrainStep with the
chunked Adam pipeline, as bench.py runs it) with loss 'l2', 'l1' and 'ssim'.

Every arm is run in --rounds alternating windows of at least --seconds; the report gives the best window and the spread.
Prints the card and its power limit, and one JSON line.

    python tools/time_ssim_loss.py [--rounds 3] [--seconds 1.0] [--out FILE]
"""
import argparse
import ctypes
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_render import card, timed  # noqa: E402

HBM_PEAK_GBS = 6548.5
B, H, C = 64, 224, 3
ALPHA = 0.85


def _flows(rng, kind):
    if kind == "jitter":
        return rng.uniform(-3, 3, (B, H, H, 2)).astype(np.float32)
    th = math.radians(10.0)
    c = (H - 1) / 2.0
    ii, jj = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(H, dtype=np.float64), indexing="ij")
    x = c + math.cos(th) * (ii - c) - math.sin(th) * (jj - c)
    y = c + math.sin(th) * (ii - c) + math.cos(th) * (jj - c)
    f = np.stack([x - ii, y - jj], -1).astype(np.float32)
    return np.ascontiguousarray(np.broadcast_to(f, (B, H, H, 2)) + rng.uniform(-0.2, 0.2, (B, H, H, 2)).astype(np.float32))


def time_kernels(args, dev):
    from dynamic_multiview_3d_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(0)
    w = (ctypes.c_float * C)(1.0, 1.0, 1.0)
    inv = 1.0 / (B * H * H)
    ws_l1 = torch.zeros(int(lib.dmv_sampler_loss_workspace_size(B, H, H)), dtype=torch.uint8, device=dev)
    ws_loss = torch.zeros(int(lib.dmv_loss_workspace_size(B * H * H)), dtype=torch.uint8, device=dev)
    bbox = torch.empty(0, dtype=torch.uint8, device=dev)
    out = {}
    for kind in ("jitter", "rotation"):
        sets = []
        for _ in range(4):
            sets.append({"src": torch.from_numpy(rng.random((B, H, H, C), dtype=np.float32)).to(dev),
                         "flow": torch.from_numpy(_flows(rng, kind)).to(dev),
                         "target": torch.from_numpy(rng.random((B, H, H, C), dtype=np.float32)).to(dev),
                         "gen": torch.empty((B, H, H, C), device=dev), "gg": torch.empty((B, H, H, C), device=dev),
                         "grad": torch.empty((B, H, H, 2), device=dev), "loss": torch.empty((), device=dev)})
        it = [0]

        def nxt():
            s = sets[it[0] % 4]
            it[0] += 1
            return s

        def composition():
            s = nxt()
            _lib.call("dmv_sampler_fwd", s["src"].data_ptr(), s["flow"].data_ptr(), s["gen"].data_ptr(), None, None, B, H, H, C, H, H, 1, st)
            _lib.call("dmv_ssim_loss_fwd_bwd", s["gen"].data_ptr(), s["target"].data_ptr(), w, ALPHA, inv, s["loss"].data_ptr(),
                      s["gg"].data_ptr(), B, H, H, C, ws_loss.data_ptr(), ws_loss.numel(), st)
            _lib.call("dmv_sampler_bwd", s["src"].data_ptr(), s["flow"].data_ptr(), s["gg"].data_ptr(), None, s["grad"].data_ptr(), B, H, H, C,
                      H, H, 1, bbox.data_ptr(), 0, st)

        def l1_fused():
            s = nxt()
            _lib.call("dmv_sampler_loss_fused", s["src"].data_ptr(), s["flow"].data_ptr(), s["target"].data_ptr(), w, 1, inv,
                      s["gen"].data_ptr(), s["grad"].data_ptr(), s["loss"].data_ptr(), B, H, H, C, H, H, 1, ws_l1.data_ptr(),
                      ws_l1.numel(), st)

        def ssim_alone():
            s = nxt()
            _lib.call("dmv_ssim_loss_fwd_bwd", s["gen"].data_ptr(), s["target"].data_ptr(), w, ALPHA, inv, s["loss"].data_ptr(),
                      s["gg"].data_ptr(), B, H, H, C, ws_loss.data_ptr(), ws_loss.numel(), st)

        arms = {"composition": composition, "l1_fused": l1_fused, "ssim_alone": ssim_alone}
        for fn in arms.values():
            for _ in range(8):
                fn()
        torch.cuda.synchronize()
        res = {k: [] for k in arms}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                n, ms = timed(fn, args.seconds / 2)
                res[name].append(1000.0 * ms / n)
        px = B * H * H
        rep = {}
        for name, v in res.items():
            nbytes = px * (12 * C if name == "ssim_alone" else 16 + 12 * C)
            best = min(v)
            gbs = nbytes / (best * 1e-6) / 1e9
            rep[name] = {"us_per_call": best, "spread_pct": 100.0 * (max(v) - best) / best, "windows_us": v, "algorithmic_bytes": nbytes,
                         "GBps": gbs, "share_of_hbm_peak": gbs / HBM_PEAK_GBS}
        out[kind] = rep
        del sets
        torch.cuda.empty_cache()
    return out


def time_steps(args, dev):
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep, synthetic_batch
    steps = {}
    for loss in ("l2", "l1", "ssim"):
        conf = {"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19, "loss": loss, "seed": 0}
        model = pkg.AppearanceFlowModel(conf)
        if os.environ.get("DMV_OVERLAP_ADAM", "1") == "1":
            data_parallel.attach(model, bucket_mb=float(os.environ.get("DMV_DP_CHUNK_MB", "32")))
        batch = {k: torch.from_numpy(v).to(dev) for k, v in synthetic_batch(model, seed=1234).items()}
        step = GraphedTrainStep(model, warmup=2)
        first = float(step(batch))
        torch.cuda.synchronize()
        steps[loss] = (step, first)
    res = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, (step, _) in steps.items():
            n, ms = timed(step.replay, args.seconds)
            res[k].append(ms / n)
    return {k: {"ms_per_step": min(v), "spread_pct": 100.0 * (max(v) - min(v)) / min(v), "windows_ms": v,
                "samples_per_s": B / (min(v) / 1e3), "first_loss": steps[k][1]} for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if args.rounds < 3:
        sys.exit("--rounds must be at least 3 (the spread needs repeats)")
    if not torch.cuda.is_available():
        sys.exit("time_ssim_loss.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    gpu = card()
    kernels = time_kernels(args, dev)
    steps = time_steps(args, dev)
    report = {"card": gpu, "shape": "B=%d, %dx%d, C=%d, alpha=%g" % (B, H, H, C, ALPHA), "hbm_peak_GBps": HBM_PEAK_GBS,
              "kernels": kernels, "step_model": "AppearanceFlowModel (config 2), 224x224, V=19, captured train step", "steps": steps}
    print("card (name, power limit): %s" % gpu)
    for kind, rep in kernels.items():
        print("%s flow" % kind)
        for k in ("composition", "l1_fused", "ssim_alone"):
            v = rep[k]
            print("  %-12s %8.1f us (spread %.1f %%)  %.0f GB/s = %.2f of the HBM peak" % (k, v["us_per_call"], v["spread_pct"], v["GBps"],
                                                                                          v["share_of_hbm_peak"]))
    for k, v in steps.items():
        print("step loss=%-5s %.3f ms/step (spread %.1f %%): %.0f samples/s" % (k, v["ms_per_step"], v["spread_pct"], v["samples_per_s"]))
    line = json.dumps(report)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

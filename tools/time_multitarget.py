"""Multi-target training throughput: config 2's model (AppearanceFlowModel, 224 x 224, one-hot azimuth V = 19, L2) as a
captured train step (GraphedTrainStep, the chunked Adam pipeline of data_parallel.attach as bench.py runs it) at
(sources B, targets T) = (64, 1), (32, 2), (16, 4) and (64, 4).  B x T targets are supervised per step; the encoder runs on
B sources.

The arms are replayed alternately in windows of at least --seconds each, --rounds times, timed with CUDA events; the report
gives ms/step, supervised targets/s and sources/s per window, the best and the spread.  The (64, 4) arm is captured first:
it needs the largest workspace of every kind, so the later captures reuse the buffers the earlier graphs hold (checked:
the tool stops if a shared workspace moved).

Also times the grouped fused warp loss (dmv_sampler_loss_fused_shared_src, 16 sources x 4 targets) against
dmv_sampler_loss_fused at B = 64 on the source repeated 4 times, with CUDA events, cycling through four input sets (about
550 MB, more than the 126 MB L2).  Prints the card, its power limit and one JSON line.

    python tools/time_multitarget.py [--rounds 3] [--seconds 1.0] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_render import card, timed  # noqa: E402

ARMS = [(64, 4), (64, 1), (32, 2), (16, 4)]        # capture order: largest first (module docstring)


def _workspace_ptrs():
    from dynamic_multiview_3d_b200 import functional as F
    ptrs = {("ws",) + k: v.data_ptr() for k, v in F._workspaces.items()}
    ptrs.update({("loss",) + k: v.data_ptr() for k, v in F._loss_wss.items()})
    return ptrs


def time_steps(args, dev):
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep, synthetic_batch
    H = 224
    steps, held = {}, None
    for B, T in ARMS:
        conf = {"batch_size": B, "num_targets": T, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19, "loss": "l2", "seed": 0}
        model = pkg.AppearanceFlowModel(conf)
        if os.environ.get("DMV_OVERLAP_ADAM", "1") == "1":
            data_parallel.attach(model, bucket_mb=float(os.environ.get("DMV_DP_CHUNK_MB", "32")))
        batch = {k: torch.from_numpy(v).to(dev) for k, v in synthetic_batch(model, seed=1234).items()}
        step = GraphedTrainStep(model, warmup=2)
        loss = float(step(batch))
        torch.cuda.synchronize()
        now = _workspace_ptrs()
        if held is not None:
            moved = [k for k, p in held.items() if now.get(k) != p]
            if moved:
                sys.exit("shared workspaces moved after capturing (%d, %d): %s -- the earlier graphs would read freed memory" % (B, T, moved))
        held = now
        steps[(B, T)] = (step, loss)
    res = {"%dx%d" % a: [] for a in ARMS}
    order = sorted(ARMS, key=lambda a: (a[1], -a[0]))
    for _ in range(args.rounds):
        for B, T in order:
            n, ms = timed(steps[(B, T)][0].replay, args.seconds)
            t = ms / n
            res["%dx%d" % (B, T)].append({"steps": n, "ms_per_step": t, "targets_per_s": B * T / (t / 1e3), "sources_per_s": B / (t / 1e3)})
    summary = {}
    for B, T in ARMS:
        w = res["%dx%d" % (B, T)]
        ms = [x["ms_per_step"] for x in w]
        best = min(ms)
        summary["%dx%d" % (B, T)] = {"sources": B, "targets": T, "first_loss": steps[(B, T)][1], "ms_per_step": best,
                                     "spread_pct": 100.0 * (max(ms) - best) / best,
                                     "targets_per_s": B * T / (best / 1e3), "sources_per_s": B / (best / 1e3)}
    return summary, res


def time_warp_loss(args, dev):
    from dynamic_multiview_3d_b200 import _lib
    lib = _lib.load()
    B_src, G, H, C = 16, 4, 224, 3
    B = B_src * G
    rng = np.random.default_rng(0)
    st = torch.cuda.current_stream().cuda_stream
    src = torch.from_numpy(rng.random((B_src, H, H, C), dtype=np.float32)).to(dev)
    rep = src.repeat_interleave(G, dim=0).contiguous()
    sets = []
    for _ in range(4):
        sets.append({"flow": torch.from_numpy(rng.uniform(-3, 3, (B, H, H, 2)).astype(np.float32)).to(dev),
                     "target": torch.from_numpy(rng.random((B, H, H, C), dtype=np.float32)).to(dev),
                     "gen": torch.empty((B, H, H, C), device=dev), "grad": torch.empty((B, H, H, 2), device=dev),
                     "loss": torch.empty((), device=dev)})
    ws = {k: torch.zeros(int(lib.dmv_sampler_loss_workspace_size(B, H, H)), dtype=torch.uint8, device=dev) for k in ("plain", "grouped")}
    w = (ctypes.c_float * C)(1.0, 1.0, 1.0)
    inv = 1.0 / (B * H * H)
    it = [0]

    def plain():
        s = sets[it[0] % 4]
        it[0] += 1
        _lib.call("dmv_sampler_loss_fused", rep.data_ptr(), s["flow"].data_ptr(), s["target"].data_ptr(), w, 0, inv, s["gen"].data_ptr(),
                  s["grad"].data_ptr(), s["loss"].data_ptr(), B, H, H, C, H, H, 1, ws["plain"].data_ptr(), ws["plain"].numel(), st)

    def grouped():
        s = sets[it[0] % 4]
        it[0] += 1
        _lib.call("dmv_sampler_loss_fused_shared_src", src.data_ptr(), B_src, G, s["flow"].data_ptr(), s["target"].data_ptr(), w, 0, inv,
                  s["gen"].data_ptr(), s["grad"].data_ptr(), s["loss"].data_ptr(), H, H, C, H, H, 1, ws["grouped"].data_ptr(),
                  ws["grouped"].numel(), st)

    for fn in (plain, grouped):
        for _ in range(8):
            fn()
    torch.cuda.synchronize()
    res = {"plain_B64": [], "grouped_16x4": []}
    for _ in range(args.rounds):
        for name, fn in (("plain_B64", plain), ("grouped_16x4", grouped)):
            n, ms = timed(fn, args.seconds / 2)
            res[name].append(1000.0 * ms / n)
    return {k: {"us_per_call": min(v), "spread_pct": 100.0 * (max(v) - min(v)) / min(v), "windows_us": v} for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if args.rounds < 3:
        sys.exit("--rounds must be at least 3 (the spread needs repeats)")
    if not torch.cuda.is_available():
        sys.exit("time_multitarget.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    gpu = card()
    summary, windows = time_steps(args, dev)
    warp = time_warp_loss(args, dev)
    report = {"card": gpu, "model": "AppearanceFlowModel (config 2), 224x224, V=19, l2, captured train step", "steps": summary,
              "step_windows": windows, "warp_loss_224_C3": warp}
    print("card (name, power limit): %s" % gpu)
    for k, v in summary.items():
        print("B x T = %-6s %.3f ms/step (spread %.1f %%): %.0f targets/s, %.0f sources/s"
              % (k, v["ms_per_step"], v["spread_pct"], v["targets_per_s"], v["sources_per_s"]))
    for k, v in warp.items():
        print("warp loss %-13s %.1f us (spread %.1f %%)" % (k, v["us_per_call"], v["spread_pct"]))
    line = json.dumps(report)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

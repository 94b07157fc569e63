"""Several source views per target: the fused multi-view warp loss against the composition it replaces, and the captured
train step of config 2's model with num_views.

1. Kernel against composition at views = 4, B = 16 targets, 224 x 224, C = 3, L2, flows of +-3 pixels: one
   dmv_sampler_fuse_views_loss against the composition -- split the 3-channel head into flow and logit copies,
   dmv_sampler_fwd on every view, dmv_loss_fused_fwd_bwd (V = 4, the logits), dmv_sampler_bwd (flow gradient only) and
   the head gradient reassembled.  Three input sets are cycled (about 900 MB with the composition's buffers, more than
   the 126 MB L2) and the two arms alternate in windows of at least --seconds / 2, timed with CUDA events.  Algorithmic
   bytes per target pixel are counted from shapes (below); GB/s is set against the project's measured HBM rate
   (6548.5 GB/s, DESIGN.md).
2. Captured step: AppearanceFlowModel (config 2: 224 x 224, one-hot azimuth V = 19, L2) as GraphedTrainStep with the
   chunked Adam pipeline of data_parallel.attach, as bench.py runs it, at (targets B, views Vw) = (64, 1), (32, 2),
   (16, 4): 64 encoder and decoder rows each.  ms/step and supervised targets/s per window, the best and the spread.
   The arms with several views are captured first: later captures reuse the workspaces the earlier graphs hold (checked:
   the tool stops if a shared workspace moved).

Prints the card, its power limit and one JSON line.

    python tools/time_multiview.py [--rounds 3] [--seconds 1.0] [--out FILE]
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

HBM_GBS = 6548.5
ARMS = [(16, 4), (32, 2), (64, 1)]        # capture order: the 3-channel head needs the larger workspaces, so first


def kernel_bytes(views, C):
    """Per target pixel: each view reads its head (12 B) and source (4C, one window per tile, counted once) and writes
    its head gradient (12 B); the target is read (4C) and the fused image written (4C)."""
    return views * (24 + 4 * C) + 8 * C


def composition_bytes(views, C):
    """Per target pixel: split (read 12, write 8 + 4), sampler forward (flow 8, source 4C, gen 4C), fused loss (gen 4C,
    logit 4, grad_gen 4C, grad_logit 4; target 4C and fused 4C once), sampler flow gradient (flow 8, source 4C,
    grad_gen 4C, grad_flow 8), reassembly (read 8 + 4, write 12)."""
    per_view = 24 + (8 + 8 * C) + (8 + 8 * C) + (16 + 8 * C) + 24
    return views * per_view + 8 * C


def time_kernel(args, dev):
    from dynamic_multiview_3d_b200 import _lib
    lib = _lib.load()
    views, B, H, C = 4, 16, 224, 3
    R = views * B
    rng = np.random.default_rng(0)
    st = torch.cuda.current_stream().cuda_stream
    w = (ctypes.c_float * C)(1.0, 1.0, 1.0)
    inv = 1.0 / (B * H * H)
    sets = []
    for _ in range(3):
        head = np.concatenate([rng.uniform(-3, 3, (R, H, H, 2)), rng.standard_normal((R, H, H, 1))], -1).astype(np.float32)
        s = {"data": torch.from_numpy(rng.random((R, H, H, C), dtype=np.float32)).to(dev), "head": torch.from_numpy(head).to(dev),
             "target": torch.from_numpy(rng.random((B, H, H, C), dtype=np.float32)).to(dev)}
        s.update(fused=torch.empty((B, H, H, C), device=dev), grad_head=torch.empty((R, H, H, 3), device=dev), loss=torch.empty((), device=dev),
                 flow=torch.empty((R, H, H, 2), device=dev), logit=torch.empty((R, H, H), device=dev), gen=torch.empty((R, H, H, C), device=dev),
                 grad_gen=torch.empty((R, H, H, C), device=dev), grad_logit=torch.empty((R, H, H), device=dev),
                 grad_flow=torch.empty((R, H, H, 2), device=dev), fused_c=torch.empty((B, H, H, C), device=dev),
                 grad_head_c=torch.empty((R, H, H, 3), device=dev), loss_c=torch.empty((), device=dev))
        sets.append(s)
    ws_k = torch.zeros(int(lib.dmv_sampler_loss_workspace_size(B, H, H)), dtype=torch.uint8, device=dev)
    ws_l = torch.zeros(int(lib.dmv_loss_workspace_size(B * H * H)), dtype=torch.uint8, device=dev)
    ws_s = torch.zeros(max(16, int(lib.dmv_sampler_bwd_workspace_size(R, H, H, C, H, H))), dtype=torch.uint8, device=dev)
    it = [0]

    def kernel():
        s = sets[it[0] % 3]
        it[0] += 1
        _lib.call("dmv_sampler_fuse_views_loss", s["data"].data_ptr(), views, s["head"].data_ptr(), s["target"].data_ptr(), w, 0, inv,
                  s["fused"].data_ptr(), s["grad_head"].data_ptr(), s["loss"].data_ptr(), B, H, H, C, H, H, 1, ws_k.data_ptr(), ws_k.numel(), st)

    def composition():
        s = sets[it[0] % 3]
        it[0] += 1
        s["flow"].copy_(s["head"][..., :2])
        s["logit"].copy_(s["head"][..., 2])
        _lib.call("dmv_sampler_fwd", s["data"].data_ptr(), s["flow"].data_ptr(), s["gen"].data_ptr(), None, None, R, H, H, C, H, H, 1, st)
        _lib.call("dmv_loss_fused_fwd_bwd", s["gen"].data_ptr(), s["logit"].data_ptr(), views, s["target"].data_ptr(), None, w, 0, inv,
                  s["loss_c"].data_ptr(), s["grad_gen"].data_ptr(), s["grad_logit"].data_ptr(), s["fused_c"].data_ptr(), B * H * H, C,
                  ws_l.data_ptr(), ws_l.numel(), st)
        _lib.call("dmv_sampler_bwd", s["data"].data_ptr(), s["flow"].data_ptr(), s["grad_gen"].data_ptr(), None, s["grad_flow"].data_ptr(),
                  R, H, H, C, H, H, 1, ws_s.data_ptr(), ws_s.numel(), st)
        s["grad_head_c"][..., :2].copy_(s["grad_flow"])
        s["grad_head_c"][..., 2].copy_(s["grad_logit"])

    for fn in (kernel, composition):
        for _ in range(6):
            fn()
    torch.cuda.synchronize()
    for s in sets:       # the two arms compute the same outputs
        same = torch.equal(s["fused"], s["fused_c"]) and torch.equal(s["grad_head"], s["grad_head_c"])
        if not same:
            sys.exit("the kernel and the composition disagree on the timed inputs")
    res = {"kernel": [], "composition": []}
    for _ in range(args.rounds):
        for name, fn in (("kernel", kernel), ("composition", composition)):
            n, ms = timed(fn, args.seconds / 2)
            res[name].append(1000.0 * ms / n)
    px = B * H * H
    out = {"views": views, "targets": B, "size": H, "C": C, "input_sets": 3,
           "input_set_mb": round(sum(t.numel() * 4 for t in sets[0].values()) / 2 ** 20, 1)}
    for name, nbytes in (("kernel", kernel_bytes(views, C)), ("composition", composition_bytes(views, C))):
        us = min(res[name])
        gbs = nbytes * px / (us * 1e-6) / 1e9
        out[name] = {"us_per_call": us, "spread_pct": 100.0 * (max(res[name]) - us) / us, "windows_us": res[name],
                     "bytes_per_target_pixel": nbytes, "gb_per_s": gbs, "of_measured_hbm": gbs / HBM_GBS}
    out["speedup"] = out["composition"]["us_per_call"] / out["kernel"]["us_per_call"]
    return out


def _workspace_ptrs():
    from dynamic_multiview_3d_b200 import functional as F
    ptrs = {("ws",) + k: v.data_ptr() for k, v in F._workspaces.items()}
    ptrs.update({("loss",) + k: v.data_ptr() for k, v in F._loss_wss.items()})
    return ptrs


def time_steps(args, dev):
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import data_parallel
    from dynamic_multiview_3d_b200.train import GraphedTrainStep, synthetic_batch
    from dynamic_multiview_3d_b200 import _lib, functional as F
    H = 224
    # the fused-loss workspace grows with the number of targets: size it for the largest arm before any capture
    n = int(_lib.load().dmv_sampler_loss_workspace_size(max(B for B, _ in ARMS), H, H))
    F._loss_wss[("warp_loss", dev.type, dev.index)] = torch.zeros(n, dtype=torch.uint8, device=dev)
    steps, held = {}, None
    for B, Vw in ARMS:
        conf = {"batch_size": B, "num_views": Vw, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19, "loss": "l2", "seed": 0}
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
                sys.exit("shared workspaces moved after capturing (%d, %d): %s -- the earlier graphs would read freed memory" % (B, Vw, moved))
        held = now
        steps[(B, Vw)] = (step, loss)
    res = {"%dx%d" % a: [] for a in ARMS}
    for _ in range(args.rounds):
        for B, Vw in ARMS:
            n, ms = timed(steps[(B, Vw)][0].replay, args.seconds)
            t = ms / n
            res["%dx%d" % (B, Vw)].append({"steps": n, "ms_per_step": t, "targets_per_s": B / (t / 1e3)})
    summary = {}
    for B, Vw in ARMS:
        ms = [x["ms_per_step"] for x in res["%dx%d" % (B, Vw)]]
        best = min(ms)
        summary["%dx%d" % (B, Vw)] = {"targets": B, "views": Vw, "encoder_rows": B * Vw, "first_loss": steps[(B, Vw)][1],
                                      "ms_per_step": best, "spread_pct": 100.0 * (max(ms) - best) / best, "targets_per_s": B / (best / 1e3)}
    return summary, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if args.rounds < 3:
        sys.exit("--rounds must be at least 3 (the spread needs repeats)")
    if not torch.cuda.is_available():
        sys.exit("time_multiview.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    gpu = card()
    kern = time_kernel(args, dev)
    summary, windows = time_steps(args, dev)
    report = {"card": gpu, "fuse_views_224_C3": kern,
              "model": "AppearanceFlowModel (config 2), 224x224, V=19, l2, captured train step", "steps": summary, "step_windows": windows}
    print("card (name, power limit): %s" % gpu)
    for k in ("kernel", "composition"):
        v = kern[k]
        print("fuse views %-11s %.1f us (spread %.1f %%), %d B/target px, %.0f GB/s = %.2f of measured HBM"
              % (k, v["us_per_call"], v["spread_pct"], v["bytes_per_target_pixel"], v["gb_per_s"], v["of_measured_hbm"]))
    for k, v in summary.items():
        print("B x Vw = %-6s %.3f ms/step (spread %.1f %%): %.0f targets/s" % (k, v["ms_per_step"], v["spread_pct"], v["targets_per_s"]))
    line = json.dumps(report)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

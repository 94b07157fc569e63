"""Rendering throughput: GraphedRender (each source encoded once, the decoder at B x V) against a captured forward pass on the
source batch repeated V times (the encoder B x V times), config 3's model (AppFlowHighDimAngle, 224 x 224, one-hot
azimuth V = 19), 64 sources x 19 views.

Both are CUDA graphs, replayed alternately in windows of at least --seconds each and timed with CUDA events; the outputs of
the two are compared (they differ in the last bits: fc1 and the joint FCs run at M = 64 in one and M = 1216 in the other).
Prints the card, its power limit and one JSON line.

    python tools/time_render.py [--sources 64] [--views 19] [--rounds 3] [--seconds 1.0] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """Name and power limit of GPU 0 (read-only query)."""
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def timed(fn, seconds):
    """Replays of fn for at least ``seconds`` (calibrated on one replay): (replays, milliseconds)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    n = max(3, int(seconds * 1000.0 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return n, e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sources", type=int, default=64)
    ap.add_argument("--views", type=int, default=19)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_render.py measures on a CUDA device; none is visible")
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.synthetic import make_batch
    from dynamic_multiview_3d_b200.train import GraphedRender
    B, V, H = args.sources, args.views, args.size
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    model = pkg.AppFlowHighDimAngle({"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19}, build_loss=False)
    b = make_batch(B, H, "onehot19", seed=7)
    src = torch.from_numpy(b["image0"]).to(dev)
    vp = torch.eye(19, dtype=torch.float32, device=dev)[:V]

    render = GraphedRender(model, B, V)
    render({"image0": src}, vp)

    # the forward pass on the repeated batch, captured the same way
    rep = src.repeat_interleave(V, dim=0).contiguous()
    disp = vp.unsqueeze(0).expand(B, V, 19).reshape(B * V, 19).contiguous()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):
            model.forward(rep, disp)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    fwd_graph = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(fwd_graph, stream=side):
        fwd_out = model.forward(rep, disp)
    torch.cuda.synchronize()

    render.graph.replay()
    fwd_graph.replay()
    torch.cuda.synchronize()
    g_r, g_f = render.out["gen"].reshape(B * V, H, H, 3).double(), fwd_out["gen"].double()
    f_r, f_f = render.out["flow"].reshape(B * V, H, H, 2).double(), fwd_out["flow_field"].double()
    diff = {"gen_max_abs": float((g_r - g_f).abs().max()), "gen_rel_l2": float((g_r - g_f).norm() / g_f.norm()),
            "flow_max_abs": float((f_r - f_f).abs().max()), "flow_rel_l2": float((f_r - f_f).norm() / f_f.norm())}

    res = {"render": [], "forward": []}
    for _ in range(args.rounds):             # alternating windows: both see the same machine state
        for name, fn in (("render", render.graph.replay), ("forward", fwd_graph.replay)):
            n, ms = timed(fn, args.seconds)
            res[name].append({"replays": n, "ms_per_replay": ms / n, "views_per_s": B * V * n / (ms / 1000.0)})
    best = {k: min(r["ms_per_replay"] for r in v) for k, v in res.items()}
    report = {
        "card": card(), "model": "AppFlowHighDimAngle (config 3)", "image_size": H, "sources": B, "views": V,
        "render_ms": best["render"], "forward_ms": best["forward"],
        "render_views_per_s": B * V / (best["render"] / 1000.0), "forward_views_per_s": B * V / (best["forward"] / 1000.0),
        "speedup": best["forward"] / best["render"], "output_difference": diff, "windows": res,
    }
    line = json.dumps(report)
    print("card (name, power limit): %s" % report["card"])
    print("render %.3f ms (%.0f views/s), forward on the repeated batch %.3f ms (%.0f views/s): %.2fx"
          % (best["render"], report["render_views_per_s"], best["forward"], report["forward_views_per_s"], report["speedup"]))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""Novel views from a trained model: each source image is encoded once and decoded at every viewpoint of a set.

    python -m dynamic_multiview_3d_b200.render --hyper conf.py --checkpoint OUT/model200000 --out DIR \\
           [--tfrecords] [--num_sources N] [--views onehot19 | --azimuths START:STOP:N --elevation E]

Viewpoint sets (rows of the model's viewpoint code, the ``disp`` input):
  onehot19             the 19 one-hot azimuth bins (viewpoint_dim 19), bin k = 20k degrees;
  --azimuths a:b:n     (d_elevation, d_azimuth) rows in radians (viewpoint_dim 2), in the order of synthetic.py /
                       collect_data_node.py:125-131: n azimuths evenly spaced from a to b inclusive, elevation E.
Sources are seeded synthetic batches (synthetic.py) or, with --tfrecords, the conf's TFRecord test split read as the
reference's test_mode reads it (files in order, no shuffling); uint8 pixels are prepared on the device.
Writes one PNG strip per source (the source, then its V renders) and renders.npy, float32 [N, V, H, W, C].
"""
import argparse
import os

import numpy as np
import torch


def onehot19():
    """The 19 one-hot azimuth bins, bin k in row k."""
    return np.eye(19, dtype=np.float32)


def azimuth_sweep(spec, elevation=0.0):
    """'START:STOP:N' -> [N, 2] float32 (d_elevation, d_azimuth) rows in radians, azimuths from START to STOP inclusive."""
    parts = str(spec).split(":")
    if len(parts) != 3:
        raise ValueError("--azimuths takes START:STOP:N, got %r" % (spec,))
    try:
        start, stop, n = float(parts[0]), float(parts[1]), int(parts[2])
    except ValueError:
        raise ValueError("--azimuths takes START:STOP:N with numbers START, STOP and an integer N, got %r" % (spec,))
    if n < 1 or not (np.isfinite(start) and np.isfinite(stop) and np.isfinite(elevation)):
        raise ValueError("--azimuths needs finite bounds and N >= 1, got %r" % (spec,))
    rows = np.empty((n, 2), np.float32)
    rows[:, 0] = elevation
    rows[:, 1] = np.linspace(start, stop, n, dtype=np.float64)
    return rows


def viewpoint_set(viewpoint_dim, views=None, azimuths=None, elevation=0.0):
    """The viewpoint rows the CLI renders: ``views='onehot19'`` or an azimuth sweep; refuses a set whose width is not the
    model's viewpoint_dim."""
    if (views is None) == (azimuths is None):
        raise ValueError("choose one viewpoint set: --views onehot19 or --azimuths START:STOP:N")
    if views is not None:
        if views != "onehot19":
            raise ValueError("unknown viewpoint set %r (known: onehot19)" % (views,))
        rows = onehot19()
    else:
        rows = azimuth_sweep(azimuths, elevation)
    if rows.shape[1] != viewpoint_dim:
        raise ValueError("the viewpoint set has %d columns but the model's viewpoint_dim is %d" % (rows.shape[1], viewpoint_dim))
    return rows


def load_sources(model, conf, n, tfrecords=False, seed=99):
    """n source samples on the model's device, fp32 [n, H, W, C] under the names of model.render_sources()."""
    from . import functional as F
    H = model.image_shape[0]
    keys = model.render_sources()
    if tfrecords:
        from .read_tf_records import build_tfrecord_input
        reader = build_tfrecord_input(dict(conf, image_size=H, batch_size=n, test_mode=""), training=False)
        batch = reader.next_batch()
    else:
        from . import synthetic as S
        batch = S.make_batch(n, H, "onehot19" if model.viewpoint_dim == 19 else "disp2", seed=seed, depth=True)
    out = {}
    for k in keys:
        t = torch.from_numpy(np.ascontiguousarray(batch[k])).to(model.device)
        out[k] = F.prepare_images(t, H) if t.dtype == torch.uint8 else t
    return out


def write_strips(out_dir, sources, renders):
    """One PNG per source: the source image, then its V renders, left to right (visualize.mosaic / write_png)."""
    from .visualize import mosaic, write_png
    paths = []
    N, V = renders.shape[:2]
    for i in range(N):
        row = np.concatenate([sources[i:i + 1], renders[i]], 0)
        img = mosaic(row, (1, V + 1))
        if row.shape[-1] == 3:
            png = np.clip(img * 255.0, 0, 255).astype(np.uint8)
        else:
            png = np.clip(img * 65535.0, 0, 65535).astype(np.uint16)
        path = os.path.join(out_dir, "render_%04d.png" % i)
        write_png(path, png)
        paths.append(path)
    return paths


def main(argv=None):
    ap = argparse.ArgumentParser(description="render novel views of source images from a trained checkpoint")
    ap.add_argument("--hyper", required=True, help="the experiment's conf.py")
    ap.add_argument("--checkpoint", required=True, help="a state_dict saved by train.py (model<itr>)")
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--tfrecords", action="store_true", help="sources from the conf's TFRecord test split instead of synthetic ones")
    ap.add_argument("--num_sources", type=int, default=4)
    ap.add_argument("--views", default=None, help="onehot19: every one-hot azimuth bin")
    ap.add_argument("--azimuths", default=None, help="START:STOP:N azimuths in radians (two-dimensional viewpoints)")
    ap.add_argument("--elevation", type=float, default=0.0, help="elevation difference of the azimuth sweep, radians")
    ap.add_argument("--seed", type=int, default=99, help="seed of the synthetic sources")
    args = ap.parse_args(argv)
    if args.num_sources < 1:
        ap.error("--num_sources must be at least 1")
    if args.views is None and args.azimuths is None:
        args.views = "onehot19"
    from .train import build_model, load_conf
    conf = load_conf(args.hyper)
    conf["batch_size"] = args.num_sources
    model = build_model(conf, build_loss=False)
    try:
        rows = viewpoint_set(model.viewpoint_dim, args.views, args.azimuths, args.elevation)
    except ValueError as e:
        ap.error(str(e))
    model.load_state_dict(torch.load(args.checkpoint, map_location="cpu"))
    sources = load_sources(model, conf, args.num_sources, args.tfrecords, args.seed)
    out = model.render(sources, torch.from_numpy(rows).to(model.device))
    key = "gen" if "gen" in out else ("gen_image1" if "gen_image1" in out else "gen_dimage1")
    src_key = "depth0" if key == "gen_dimage1" else "image0"
    renders = out[key].cpu().numpy()
    os.makedirs(args.out, exist_ok=True)
    np.save(os.path.join(args.out, "renders.npy"), renders.astype(np.float32))
    paths = write_strips(args.out, sources[src_key].cpu().numpy(), renders)
    print("rendered %d sources x %d views -> %s (%d PNG strips, renders.npy %s)" % (renders.shape[0], renders.shape[1], args.out,
                                                                                   len(paths), list(renders.shape)))


if __name__ == "__main__":
    main()

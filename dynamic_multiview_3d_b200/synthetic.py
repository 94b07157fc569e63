"""Deterministic synthetic "car-render-shaped" batches (SURVEY.md 8(d)).

float32 NHWC images in [0,1] on the reference renderer's 0.5-grey background
(multi_view_model/utils/renderer.py:44-47), a filled rotated ellipse as the car blob,
N(0, 0.02) noise; image1 is the same blob rotated by the sampled azimuth difference.
Depth: 1.0 far plane, blob at 0.3-0.6.  Viewpoint: one-hot azimuth (V=19 bins of 20 deg) or
the reference-native (d_elevation, d_azimuth) radians (collect_data_node.py:125-131).
targets=T > 1: T target views per source at distinct azimuth bins, image1 [B, T, H, W, 3], disp [B, T, V] (depth1 /
mask1 likewise).  Target 0 and everything else are the targets=1 batch of the same seed; the other targets are drawn
after it.
make_multiview_batch: several source views of one car per target (the single-view models' num_views).
Host-side NumPy: this is input generation, not part of the measured path.
"""
import numpy as np


def make_batch(batch, size=224, viewpoint="onehot19", seed=1234, rank=0, depth=False, views=1, targets=1):
    rng = np.random.default_rng(seed + rank)
    H = W = size
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    cy, cx = (H - 1) / 2.0, (W - 1) / 2.0

    def blob(yaw, colour, jitter):
        c, s = np.cos(yaw), np.sin(yaw)
        u = ((xx - cx - jitter[0]) * c + (yy - cy - jitter[1]) * s) / (0.275 * W)
        v = (-(xx - cx - jitter[0]) * s + (yy - cy - jitter[1]) * c) / (0.125 * H)
        m = (u * u + v * v) <= 1.0
        img = np.full((H, W, 3), 0.5, np.float32)
        img[m] = colour
        return img, m

    n_src = max(1, views)
    image0 = np.empty((batch, n_src, H, W, 3), np.float32)
    image1 = np.empty((batch, H, W, 3), np.float32)
    depth0 = np.ones((batch, H, W, 1), np.float32)
    depth1 = np.ones((batch, H, W, 1), np.float32)
    mask1 = np.zeros((batch, H, W, 1), np.float32)
    bins = rng.integers(0, 19, size=batch)
    disp = np.zeros((batch, 19 if viewpoint == "onehot19" else 2), np.float32)
    scenes = []
    for b in range(batch):
        colour = rng.uniform(0.1, 0.9, size=3).astype(np.float32)
        jit = rng.uniform(-4, 4, size=2)
        yaw1 = rng.uniform(0, 2 * np.pi)
        daz = np.deg2rad(20.0 * bins[b])
        img1, m1 = blob(yaw1, colour, jit)
        image1[b] = img1
        dval = rng.uniform(0.3, 0.6)
        depth1[b, m1, 0] = dval
        mask1[b, m1, 0] = 1.0
        scenes.append((yaw1 - daz, colour, jit, dval))
        for v in range(n_src):
            yaw0 = yaw1 - daz - np.deg2rad(10.0 * v)
            img0, m0 = blob(yaw0, colour, jit)
            image0[b, v] = img0
            if v == 0:
                depth0[b, m0, 0] = dval
        if viewpoint == "onehot19":
            disp[b, bins[b]] = 1.0
        else:
            disp[b] = (0.0, daz)
    image0 += rng.normal(0, 0.02, image0.shape).astype(np.float32)
    image1 += rng.normal(0, 0.02, image1.shape).astype(np.float32)
    np.clip(image0, 0, 1, out=image0)
    np.clip(image1, 0, 1, out=image1)
    if targets > 1:
        image1, depth1, mask1, disp = _more_targets(rng, blob, scenes, bins, int(targets), viewpoint, image1, depth1, mask1, disp)
    out = {"image0": image0[:, 0] if views <= 1 else image0, "image1": image1, "disp": disp}
    if depth:
        out.update(depth0=depth0, depth1=depth1, mask1=mask1)
    return out


def _more_targets(rng, blob, scenes, bins, T, viewpoint, image1, depth1, mask1, disp):
    """Targets 1 .. T-1 of every source, at azimuth bins (relative to the source) other than target 0's and each other's."""
    if T > 19:
        raise ValueError("at most 19 targets per source (one per azimuth bin)")
    B = len(scenes)
    im = np.empty((B, T) + image1.shape[1:], np.float32)
    dp = np.ones((B, T) + depth1.shape[1:], np.float32)
    mk = np.zeros((B, T) + mask1.shape[1:], np.float32)
    ds = np.zeros((B, T, disp.shape[1]), np.float32)
    im[:, 0], dp[:, 0], mk[:, 0], ds[:, 0] = image1, depth1, mask1, disp
    for b, (yaw0, colour, jit, dval) in enumerate(scenes):
        others = rng.permutation(np.delete(np.arange(19), bins[b]))[:T - 1]
        for t, k in enumerate(others, 1):
            daz = np.deg2rad(20.0 * k)
            img, m = blob(yaw0 + daz, colour, jit)
            im[b, t] = img
            dp[b, t, m, 0] = dval
            mk[b, t, m, 0] = 1.0
            if viewpoint == "onehot19":
                ds[b, t, k] = 1.0
            else:
                ds[b, t] = (0.0, daz)
    im[:, 1:] += rng.normal(0, 0.02, im[:, 1:].shape).astype(np.float32)
    np.clip(im, 0, 1, out=im)
    return im, dp, mk, ds


def make_multiview_batch(batch, size=224, views=2, viewpoint="onehot19", seed=1234, rank=0):
    """Several source views of one car per target (AppearanceFlowModel with num_views): image0 [views, B, H, W, 3],
    disp [views, B, V], image1 [B, H, W, 3].  Source v of sample b shows the car rotated by bins[v, b] * 20 degrees less
    than the target, at an azimuth bin distinct from the sample's other sources; its disp row is that rotation to the
    target: the one-hot bin, or (0, d_azimuth) radians."""
    if not 1 <= views <= 19:
        raise ValueError("views must be 1 .. 19 (one per azimuth bin), got %d" % views)
    rng = np.random.default_rng(seed + rank)
    H = W = size
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    cy, cx = (H - 1) / 2.0, (W - 1) / 2.0

    def blob(yaw, colour, jitter):
        c, s = np.cos(yaw), np.sin(yaw)
        u = ((xx - cx - jitter[0]) * c + (yy - cy - jitter[1]) * s) / (0.275 * W)
        v = (-(xx - cx - jitter[0]) * s + (yy - cy - jitter[1]) * c) / (0.125 * H)
        img = np.full((H, W, 3), 0.5, np.float32)
        img[(u * u + v * v) <= 1.0] = colour
        return img

    image0 = np.empty((views, batch, H, W, 3), np.float32)
    image1 = np.empty((batch, H, W, 3), np.float32)
    disp = np.zeros((views, batch, 19 if viewpoint == "onehot19" else 2), np.float32)
    bins = np.empty((views, batch), np.int64)
    for b in range(batch):
        colour = rng.uniform(0.1, 0.9, size=3).astype(np.float32)
        jit = rng.uniform(-4, 4, size=2)
        yaw1 = rng.uniform(0, 2 * np.pi)
        image1[b] = blob(yaw1, colour, jit)
        bins[:, b] = rng.choice(19, size=views, replace=False)
        for v in range(views):
            daz = np.deg2rad(20.0 * bins[v, b])
            image0[v, b] = blob(yaw1 - daz, colour, jit)
            if viewpoint == "onehot19":
                disp[v, b, bins[v, b]] = 1.0
            else:
                disp[v, b] = (0.0, daz)
    image0 += rng.normal(0, 0.02, image0.shape).astype(np.float32)
    image1 += rng.normal(0, 0.02, image1.shape).astype(np.float32)
    np.clip(image0, 0, 1, out=image0)
    np.clip(image1, 0, 1, out=image1)
    return {"image0": image0, "image1": image1, "disp": disp, "bins": bins}


def make_multiobject_batch(batch, size=128, seed=1234, rank=0):
    """Two-object scenes under the tensor names of read_tf_records_multobj.py:65-80 / multiobject_appflow.py:31-43:
    two blobs (objects 0 and 1) seen from a source and a target viewpoint, their indicator masks, the per-object
    target renders (``*_only0/1``) and depth maps (far plane 1.0, objects at 0.3-0.6)."""
    rng = np.random.default_rng(seed + rank)
    H = W = size
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    names3 = ["image0", "image1", "image1_only0", "image1_only1"]
    names1 = ["image0_mask0", "image0_mask1", "image1_mask0", "image1_mask1", "depth0", "depth1", "depth1_only0", "depth1_only1"]
    out = {k: np.full((batch, H, W, 3), 0.5, np.float32) for k in names3}
    out.update({k: np.zeros((batch, H, W, 1), np.float32) for k in names1 if "mask" in k})
    out.update({k: np.ones((batch, H, W, 1), np.float32) for k in names1 if "depth" in k})
    disp = np.zeros((batch, 2), np.float32)

    def ell(cx, cy, yaw, a, b):
        c, s = np.cos(yaw), np.sin(yaw)
        u = ((xx - cx) * c + (yy - cy) * s) / a
        v = (-(xx - cx) * s + (yy - cy) * c) / b
        return (u * u + v * v) <= 1.0

    for n in range(batch):
        daz = rng.uniform(-0.6, 0.6)
        disp[n] = (0.0, daz)
        for ob in range(2):
            col = rng.uniform(0.1, 0.9, size=3).astype(np.float32)
            cx, cy = rng.uniform(0.3, 0.7) * W, rng.uniform(0.3, 0.7) * H
            yaw, dval = rng.uniform(0, np.pi), rng.uniform(0.3, 0.6)
            m0, m1 = ell(cx, cy, yaw, 0.18 * W, 0.09 * H), ell(cx, cy, yaw + daz, 0.18 * W, 0.09 * H)
            out["image0"][n][m0] = col; out["image0_mask%d" % ob][n][m0] = 1.0; out["depth0"][n][m0] = dval
            out["image1"][n][m1] = col; out["image1_mask%d" % ob][n][m1] = 1.0; out["depth1"][n][m1] = dval
            out["image1_only%d" % ob][n][m1] = col; out["depth1_only%d" % ob][n][m1] = dval
    for k in names3:
        out[k] = np.clip(out[k] + rng.normal(0, 0.02, out[k].shape).astype(np.float32), 0, 1)
    out["displacement"] = disp
    return out


def make_multiview_multiobject_batch(batch, size=224, views=4, seed=1234, rank=0, viewpoint="disp2"):
    """BASELINE config 5 inputs (SURVEY 8(d)): ``views`` source frames of a two-object scene per sample, each with its
    object masks and depth map (tensor names of read_tf_records_multobj.py:65-80, leading axis = source frame), the
    viewpoint change of every frame to the target (``displacement`` [views, B, V]) and the target render ``image1``."""
    rng = np.random.default_rng(seed + rank)
    H = W = size
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    Vd = 19 if viewpoint == "onehot19" else 2
    out = {"image0": np.full((views, batch, H, W, 3), 0.5, np.float32), "depth0": np.ones((views, batch, H, W, 1), np.float32),
           "image0_mask0": np.zeros((views, batch, H, W, 1), np.float32), "image0_mask1": np.zeros((views, batch, H, W, 1), np.float32),
           "displacement": np.zeros((views, batch, Vd), np.float32), "image1": np.full((batch, H, W, 3), 0.5, np.float32)}

    def ell(cx, cy, yaw, a, b):
        c, s = np.cos(yaw), np.sin(yaw)
        u = ((xx - cx) * c + (yy - cy) * s) / a
        v = (-(xx - cx) * s + (yy - cy) * c) / b
        return (u * u + v * v) <= 1.0

    for n in range(batch):
        bins = rng.integers(1, 5, size=views)                     # each frame 20..80 degrees away from the target
        objs = [(rng.uniform(0.1, 0.9, size=3).astype(np.float32), rng.uniform(0.3, 0.7) * W, rng.uniform(0.3, 0.7) * H,
                 rng.uniform(0, np.pi), rng.uniform(0.3, 0.6)) for _ in range(2)]
        for ob, (col, cx, cy, yaw, dval) in enumerate(objs):
            out["image1"][n][ell(cx, cy, yaw, 0.18 * W, 0.09 * H)] = col
        for v in range(views):
            daz = np.deg2rad(20.0 * bins[v]) * (1 if v % 2 == 0 else -1)
            if viewpoint == "onehot19":
                out["displacement"][v, n, (bins[v] * (1 if v % 2 == 0 else -1)) % 19] = 1.0
            else:
                out["displacement"][v, n] = (0.0, daz)
            for ob, (col, cx, cy, yaw, dval) in enumerate(objs):
                m = ell(cx, cy, yaw - daz, 0.18 * W, 0.09 * H)
                out["image0"][v, n][m] = col
                out["image0_mask%d" % ob][v, n][m] = 1.0
                out["depth0"][v, n][m] = dval
    for k in ("image0", "image1"):
        out[k] = np.clip(out[k] + rng.normal(0, 0.02, out[k].shape).astype(np.float32), 0, 1)
    return out

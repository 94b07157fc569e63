"""Evaluation outputs, SURVEY 8(f)-4: the image grids of ``save_images`` (dyn_mult_view/mv3d/utils/tf_utils.py:101-147)
and the ``visualize`` method of the models (appearance_flow_model.py:132-179) without matplotlib / scipy.misc.

``save_images`` lays a batch out exactly like the reference (row-major ``size = [rows, cols]`` mosaic, first
rows*cols images, ``rescale_image`` = (x / 1.5 + 0.5) * 255 for colour and ``rescale_dm`` = (x / 1.5 + 0.5) * 65535 as
16-bit grey for depth maps) and writes PNG through zlib.  matplotlib is not in this image, so the reference's two
FIGURES are rasterised here with a small line drawer: ``quiver_<iter>.png`` (plt.quiver(warp_pts[0,:,:,0],
warp_pts[0,:,:,1]), appearance_flow_model.py:151-154) and ``corr_plot_<iter>.png`` (source | generated image with the
six random correspondence probes joined by lines, :156-179); the flow field is also written as an HSV colour-wheel image.
``visualize_multiobject`` restates multiobject_appflow.py:289-393: every input and output clipped to [0,1] and pickled
to ``imgdata.pkl`` (the reference returns there), plus the per-sample panels of :396-510 as PNG mosaics.
Host-side NumPy on tensors copied back from the device; nothing here is on the measured path.
"""
import math
import os
import re
import struct
import zlib

import numpy as np


def rescale_image(image):
    """tf_utils.py:139-141"""
    return (image / 1.5 + 0.5) * 255


def rescale_dm(image):
    """tf_utils.py:144-146"""
    return (image / 1.5 + 0.5) * 65535


def mosaic(images, size):
    """tf_utils.py:101-119: [N,h,w(,3)] -> [h*rows, w*cols(,3)], image idx at row idx // cols, column idx % cols."""
    images = np.asarray(images)
    h, w = images.shape[1], images.shape[2]
    color = images.ndim == 4 and images.shape[3] == 3
    if images.ndim == 4 and not color:
        images = images[..., 0]
    img = np.zeros((h * size[0], w * size[1], 3) if color else (h * size[0], w * size[1]), np.float64)
    for idx, image in enumerate(images[:size[0] * size[1]]):
        i, j = idx % size[1], int(math.floor(idx / size[1]))
        img[j * h:j * h + h, i * w:i * w + w] = image
    return img


def write_png(path, arr):
    """uint8 [H,W,3] / [H,W] or uint16 [H,W] -> PNG (filter 0 scanlines, one zlib stream)."""
    arr = np.ascontiguousarray(arr)
    if arr.dtype == np.uint16:
        depth, ctype, raw = 16, 0, arr.astype(">u2").tobytes()
        row = arr.shape[1] * 2
    else:
        arr = arr.astype(np.uint8)
        depth, ctype = 8, (2 if arr.ndim == 3 else 0)
        raw, row = arr.tobytes(), arr.shape[1] * (3 if arr.ndim == 3 else 1)
    lines = b"".join(b"\x00" + raw[y * row:(y + 1) * row] for y in range(arr.shape[0]))

    def chunk(tag, data):
        c = struct.pack(">I", len(data)) + tag + data
        return c + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", arr.shape[1], arr.shape[0], depth, ctype, 0, 0, 0)) +
                chunk(b"IDAT", zlib.compress(lines, 6)) + chunk(b"IEND", b""))


def save_images(images, size, image_path, color=True):
    """tf_utils.py:101-123 (scipy.misc.toimage(..., cmin=0, cmax=255|65535) clips to the range)."""
    img = mosaic(images, size)
    if color:
        write_png(image_path, np.clip(rescale_image(img), 0, 255).astype(np.uint8))
    else:
        write_png(image_path, np.clip(rescale_dm(img), 0, 65535).astype(np.uint16))


def flow_to_color(flow):
    """[h,w,2] displacement field -> uint8 RGB: hue = direction, saturation = magnitude / max magnitude."""
    fx, fy = flow[..., 0].astype(np.float64), flow[..., 1].astype(np.float64)
    mag = np.hypot(fx, fy)
    hsv_h = (np.arctan2(fy, fx) / (2 * np.pi)) % 1.0
    s = mag / max(float(mag.max()), 1e-12)
    i = np.floor(hsv_h * 6).astype(int) % 6
    f = hsv_h * 6 - np.floor(hsv_h * 6)
    p, q, t = 1 - s, 1 - s * f, 1 - s * (1 - f)
    one = np.ones_like(s)
    r = np.choose(i, [one, q, p, p, t, one])
    g = np.choose(i, [t, one, one, q, p, p])
    b = np.choose(i, [p, p, t, one, one, q])
    return (np.stack([r, g, b], -1) * 255).astype(np.uint8)


def draw_line(img, x0, y0, x1, y1, color):
    """Rasterise a segment into uint8 [H,W,3] (clipped; DDA)."""
    n = int(max(abs(x1 - x0), abs(y1 - y0), 1))
    xs = np.rint(np.linspace(x0, x1, n + 1)).astype(int)
    ys = np.rint(np.linspace(y0, y1, n + 1)).astype(int)
    ok = (xs >= 0) & (xs < img.shape[1]) & (ys >= 0) & (ys < img.shape[0])
    img[ys[ok], xs[ok]] = color


def draw_arrow(img, x0, y0, x1, y1, color):
    draw_line(img, x0, y0, x1, y1, color)
    dx, dy = x1 - x0, y1 - y0
    ln = math.hypot(dx, dy)
    if ln < 2:
        return
    ux, uy = dx / ln, dy / ln
    h = min(4.0, 0.35 * ln)
    for sgn in (1, -1):                                       # two barbs at +-25 degrees
        c, s_ = math.cos(sgn * 0.44), math.sin(sgn * 0.44)
        draw_line(img, x1, y1, x1 - h * (ux * c - uy * s_), y1 - h * (ux * s_ + uy * c), color)


def quiver_image(warp_pts, cell=12, stride=None):
    """plt.quiver(U, V) of appearance_flow_model.py:153: one arrow per grid node (subsampled so the figure stays
    legible), components (U, V) = the two channels of warp_pts, lengths scaled to the longest arrow, y axis pointing
    up as in matplotlib.  Returns uint8 RGB."""
    U, V = np.asarray(warp_pts[..., 0], np.float64), np.asarray(warp_pts[..., 1], np.float64)
    h, w = U.shape
    stride = stride or max(1, h // 28)
    ii, jj = np.arange(0, h, stride), np.arange(0, w, stride)
    img = np.full((len(ii) * cell + cell, len(jj) * cell + cell, 3), 255, np.uint8)
    mx = max(float(np.hypot(U[np.ix_(ii, jj)], V[np.ix_(ii, jj)]).max()), 1e-12)
    for a, i in enumerate(ii):
        for b, j in enumerate(jj):
            x0, y0 = cell / 2 + b * cell, img.shape[0] - 1 - (cell / 2 + a * cell)          # row 0 at the bottom
            draw_arrow(img, x0, y0, x0 + U[i, j] / mx * cell, y0 - V[i, j] / mx * cell, (30, 30, 160))
    return img


def corr_plot_image(image0, gen, pts_output, sampled):
    """appearance_flow_model.py:156-179: source image (left) and generated image (right); every probe of the generated
    image is joined to the source location it was sampled from (xy = flipped (row, col) pairs, :170-171)."""
    a = np.clip(np.asarray(image0, np.float64), 0, 1)
    b = np.clip(np.asarray(gen, np.float64), 0, 1)
    h, w = a.shape[0], a.shape[1]
    gap = max(8, w // 8)
    img = np.full((h, 2 * w + gap, 3), 255, np.uint8)
    img[:, :w] = (a * 255).astype(np.uint8)
    img[:, w + gap:] = (b * 255).astype(np.uint8)
    cols = [(230, 30, 30), (30, 160, 30), (30, 30, 230), (220, 160, 0), (160, 0, 200), (0, 170, 170)]
    for k, (po, sl) in enumerate(zip(pts_output, sampled)):
        c = cols[k % len(cols)]
        xa, ya = w + gap + int(po[1]), int(po[0])             # xyA = flip(pt_output) on the generated image
        xb, yb = int(sl[1]), int(sl[0])                       # xyB = flip(sampled_location) on the source image
        draw_line(img, xa, ya, xb, yb, c)
        for (x, y) in ((xa, ya), (xb, yb)):
            draw_line(img, x - 2, y, x + 2, y, c)
            draw_line(img, x, y - 2, x, y + 2, c)
    return img


def panel(images, rows, cols):
    """A rows x cols figure of optional [h,w,3] / [h,w,1] float images in [0,1] (None = empty cell), uint8 RGB."""
    ref = next(im for im in images if im is not None)
    h, w = ref.shape[0], ref.shape[1]
    out = np.full((rows * (h + 4) + 4, cols * (w + 4) + 4, 3), 255, np.uint8)
    for k, im in enumerate(images[:rows * cols]):
        if im is None:
            continue
        im = np.clip(np.asarray(im, np.float64), 0, 1)
        if im.ndim == 2 or im.shape[-1] == 1:
            im = np.repeat(im.reshape(h, w, 1), 3, axis=2)
        r, c = divmod(k, cols)
        out[4 + r * (h + 4):4 + r * (h + 4) + h, 4 + c * (w + 4):4 + c * (w + 4) + w] = (im * 255).astype(np.uint8)
    return out


def visualize_multiobject(model, batch, iter_num=None, max_panels=4):
    """multiobject_appflow.py:289-393 (+ the panels of :396-510): forward on ``batch`` without gradients, clip every
    input and every generated output to [0,1], pickle them to <output_dir>/imgdata.pkl (protocol 2, as cPickle wrote it),
    and write img_exp / depth_exp / masks_exp panels for the first ``max_panels`` samples."""
    import pickle
    import torch
    conf = model.conf
    if iter_num is None:
        m = re.match(".*?([0-9]+)$", str(conf.get("visualize", "0")))
        iter_num = m.group(1) if m else "0"
    path = conf.get("output_dir", ".")
    os.makedirs(path, exist_ok=True)
    with torch.no_grad():
        out = model.forward(batch)
        loss = float(model.build_loss(batch).detach())
    d = {k: np.clip(v.detach().float().cpu().numpy(), 0.0, 1.0) for k, v in batch.items() if k != "displacement"}
    d.update({k: np.clip(v.detach().float().cpu().numpy(), 0.0, 1.0) for k, v in out.items() if isinstance(v, torch.Tensor) and v.dim() == 4})
    with open(os.path.join(path, "imgdata.pkl"), "wb") as f:
        pickle.dump(d, f, protocol=2)
    g = lambda k, b: d[k][b] if k in d else None
    for b in range(min(max_panels, d["image0"].shape[0])):
        write_png(os.path.join(path, "img_exp_iter%s_%d.png" % (iter_num, b)), panel(
            [g("image0", b), None, None, g("image1", b), g("image1_only0", b), g("image1_only1", b),
             g("gen_image1", b), g("gen_image1_only0", b), g("gen_image1_only1", b)], 3, 3))
        if "depth0" in d:
            write_png(os.path.join(path, "depth_exp_iter%s_%d.png" % (iter_num, b)), panel(
                [g("depth0", b), None, None, g("depth1", b), g("depth1_only0", b), g("depth1_only1", b),
                 g("gen_depth1", b), g("gen_depth1_only0", b), g("gen_depth1_only1", b)], 3, 3))
        write_png(os.path.join(path, "masks_exp_iter%s_%d.png" % (iter_num, b)), panel(
            [g("image0_mask0", b), g("image0_mask1", b), g("image1_mask0", b), g("image1_mask1", b),
             None, None, g("gen_image1_mask0", b), g("gen_image1_mask1", b)], 2, 4))
    return {"loss": loss, "keys": sorted(d), "max_resample_coord": float("nan")}


def visualize_multiview(model, batch, iter_num=None):
    """Config 5 (not in the reference): the fused prediction, the target and, per source frame, the input, its warp and
    its softmax confidence map as 8x8 grids in the style of appearance_flow_model.py:143-148."""
    import torch
    conf = model.conf
    if iter_num is None:
        m = re.match(".*?([0-9]+)$", str(conf.get("visualize", "0")))
        iter_num = m.group(1) if m else "0"
    path = conf.get("output_dir", ".")
    os.makedirs(path, exist_ok=True)
    with torch.no_grad():
        out = model.forward(batch)
        loss = float(model.build_loss(batch).detach())
    save_images(model.fused.detach().cpu().numpy(), [8, 8], os.path.join(path, "output_%s.png" % iter_num))
    save_images(batch["image1"].detach().cpu().numpy(), [8, 8], os.path.join(path, "tr_gt_%s.png" % iter_num))
    wts = torch.softmax(out["logits"].detach().float(), dim=0).cpu().numpy()
    for v in range(wts.shape[0]):
        save_images(batch["image0"][v].detach().cpu().numpy(), [8, 8], os.path.join(path, "tr_input_v%d_%s.png" % (v, iter_num)))
        save_images(out["gens"][v].detach().cpu().numpy(), [8, 8], os.path.join(path, "warp_v%d_%s.png" % (v, iter_num)))
        write_png(os.path.join(path, "confidence_v%d_%s.png" % (v, iter_num)), (mosaic(wts[v][..., None], [8, 8]) * 255).astype(np.uint8))
    return {"loss": loss, "max_resample_coord": float("nan"), "mean_confidence": [float(w.mean()) for w in wts]}


def visualize(model, image0, image1, disp, iter_num=None, seed=0, source=None):
    """appearance_flow_model.py:132-179 for a model with (image0, disp) -> gen.  Writes output_/tr_gt_/tr_input_<iter>.png
    (8x8 grids), quiver_<iter>.png and corr_plot_<iter>.png (the reference's two figures, rasterised), flow_<iter>.png
    (sample 0 as a colour-wheel image) and returns {'loss', 'max_resample_coord', 'correspondences':
    [(output_pt, sampled_location)] * 6}.  ``source`` [B,H,W,3]: the input the grids and the correspondence plot show when
    it is not image0 itself (source frame 0 of a model with several source views)."""
    import torch
    if iter_num is None:
        m = re.match(".*?([0-9]+)$", str(model.conf.get("visualize", "0")))
        iter_num = m.group(1) if m else "0"
    path = model.conf.get("output_dir", ".")
    os.makedirs(path, exist_ok=True)
    with torch.no_grad():
        out = model.forward(image0, disp)
        loss = float(model.build_loss(image1).detach())
    gen = out["gen"].detach().float().cpu().numpy() if "gen" in out else model.gen.detach().float().cpu().numpy()
    warp_pts = model.warp_pts.cpu().numpy()
    save_images(gen, [8, 8], os.path.join(path, "output_%s.png" % iter_num))
    save_images(image1.detach().cpu().numpy(), [8, 8], os.path.join(path, "tr_gt_%s.png" % iter_num))
    shown = image0 if source is None else source
    save_images(shown.detach().cpu().numpy(), [8, 8], os.path.join(path, "tr_input_%s.png" % iter_num))
    flow = model.flow_field.reshape((-1,) + tuple(model.flow_field.shape[-3:]))
    write_png(os.path.join(path, "flow_%s.png" % iter_num), flow_to_color(flow[0].detach().float().cpu().numpy()))
    H = gen.shape[1]
    rng = np.random.RandomState(seed)
    pts = rng.randint(int(0.3125 * H), int(0.6875 * H), size=(6, 2))           # randint(40, 88) at 128 (:166)
    corr = [(tuple(int(v) for v in p), tuple(int(v) for v in warp_pts[0, p[0], p[1], :].astype("uint32"))) for p in pts]
    write_png(os.path.join(path, "quiver_%s.png" % iter_num), quiver_image(warp_pts[0]))
    write_png(os.path.join(path, "corr_plot_%s.png" % iter_num),
              corr_plot_image(shown[0].detach().cpu().numpy(), gen[0], [c[0] for c in corr], [c[1] for c in corr]))
    return {"loss": loss, "max_resample_coord": float(np.max(warp_pts)), "correspondences": corr}

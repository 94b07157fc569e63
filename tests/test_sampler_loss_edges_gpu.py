"""The training step's tail at its edges: the bilinear sampler's window paths, the fused warp loss and both loss kernels,
each against the oracle (oracle/tf_ops.py and float64 NumPy / torch CPU) at the tolerances of DESIGN §5:
- sampler corner indices and masks bit-exact, outputs and grad_warp bit-equal;
- grad_data within 1e-5 of max |ref| and bit-reproducible;
- loss scalars within 1e-5 relative of float64.
Every case proves which kernel ran with dmv_launch_count_named (the label of its launch check in csrc/).

sampler_tma_kernel picks one of three paths per 32x32 output tile from the tile's tap box: a 36^2 TMA window, a 44^2
window, or predicated global gathers.  `tma_window_plan` restates that choice on the CPU, and every GPU case built to
reach the paths asserts from the plan, before it runs, that each path is present.  The plan's own tests need no GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import tf_ops as T

gpu = pytest.mark.gpu

ADD_GRID, GRID_XY = 1, 2                # DMV_SAMPLER_* of include/dmv3d.h
BOX_S, BOX_L = 36, 44                   # SAMPLER_BOX, SAMPLER_BOX_L of csrc/sampler.cu
CATEGORIES = ("none", "box36", "box44", "gather")
E_INVALID_ARG, E_UNSUPPORTED_SHAPE, E_WORKSPACE = -1, -3, -5
LOSS_MODE = {"l2": 0, "l1": 1}


# ----------------------------------------------------------------------------------------------------------- the plan
def _samples(warp, H, W, flags):
    """(x, y, valid) as the sampler kernels form them: warp = flow + grid in float32 when ADD_GRID is set (channel 0 +=
    row, 1 += column in the reference's (Y,X) order; column, row with GRID_XY), valid = x > -1 && y > -1 && x < W && y < H."""
    B, Ho, Wo, _ = warp.shape
    x, y = warp[..., 0].astype(np.float32), warp[..., 1].astype(np.float32)
    if flags & ADD_GRID:
        ii, jj = np.meshgrid(np.arange(Ho, dtype=np.float32), np.arange(Wo, dtype=np.float32), indexing="ij")
        x, y = (x + jj, y + ii) if flags & GRID_XY else (x + ii, y + jj)
    with np.errstate(invalid="ignore"):
        valid = (x > -1) & (y > -1) & (x < W) & (y < H)
    return x, y, valid


def absolute_warp(warp, flags):
    """The absolute warp the oracle samples at: flow + grid, formed in float32 like the kernel."""
    B, Ho, Wo, _ = warp.shape
    x, y, _ = _samples(warp, 1, 1, flags)
    return np.ascontiguousarray(np.stack([x, y], -1), np.float32)


def tma_window_plan(warp, H, W, C, flags):
    """sampler_tma_kernel's choice for every 32x32 output tile of an image-shaped warp [B, Ho, Wo, 2].

    The tap box of a tile is reduced over its valid samples in extended coordinates (-1 .. W, -1 .. H): xlo = min floor(x),
    xhi = max floor(x) + 1, and the same for y.  The TMA box must start on a 16-byte boundary of a row, so for C in {1, 3}
    its x origin xa is xlo floored to a multiple of 4 (-1 -> -4); for C = 4 it is xlo.  With span = max(xhi - xa, yhi - ylo)
    the tile takes a 36^2 window when span < 36, a 44^2 window when span < 44, and global gathers otherwise; a tile with
    no valid sample ("none") stages nothing.  Returns a dict of [B, tiles_y, tiles_x] arrays: cat (one of CATEGORIES), xa,
    ylo, xhi, yhi, span (meaningless where cat is "none")."""
    B, Ho, Wo, _ = warp.shape
    assert Ho > 1, "Ho = 1 takes the 1 x 1024 sample-list tiling, which the TMA kernel never runs"
    x, y, valid = _samples(warp, H, W, flags)
    fx = np.floor(np.where(valid, x, 0)).astype(np.int64)
    fy = np.floor(np.where(valid, y, 0)).astype(np.int64)
    ty, tx = -(-Ho // 32), -(-Wo // 32)

    def tiles(a, fill):
        return np.pad(a, ((0, 0), (0, ty * 32 - Ho), (0, tx * 32 - Wo)), constant_values=fill).reshape(B, ty, 32, tx, 32)

    v = tiles(valid, False)
    big = 1 << 40
    xlo = np.where(v, tiles(fx, 0), big).min(axis=(2, 4))
    xhi = np.where(v, tiles(fx + 1, 0), -big).max(axis=(2, 4))
    ylo = np.where(v, tiles(fy, 0), big).min(axis=(2, 4))
    yhi = np.where(v, tiles(fy + 1, 0), -big).max(axis=(2, 4))
    any_valid = v.any(axis=(2, 4))
    xa = xlo if C == 4 else (xlo & ~3)
    span = np.where(any_valid, np.maximum(xhi - xa, yhi - ylo), 0)
    cat = np.where(~any_valid, "none", np.where(span < BOX_S, "box36", np.where(span < BOX_L, "box44", "gather")))
    return {"cat": cat, "xa": xa, "ylo": ylo, "xhi": xhi, "yhi": yhi, "span": span}


def _one_tile(x0, x1, y0, y1):
    """A 32x32 absolute warp whose tap box is exactly [x0, x1] x [y0, y1] (x1, y1: the last tap column / row)."""
    w = np.empty((1, 32, 32, 2), np.float32)
    w[..., 0], w[..., 1] = x0 + 0.5, y0 + 0.5
    w[0, 31, 31] = (x1 - 0.5, y1 - 0.5)
    return w


# (C, x0, x1, y0, y1) -> (category, xa, span), worked out by hand from the kernel's rule
HAND_TILES = [
    ((4, 0, 35, 0, 3), ("box36", 0, 35)),          # span 35: the small window
    ((4, 0, 36, 0, 3), ("box44", 0, 36)),          # 36: the large window
    ((4, 0, 43, 0, 3), ("box44", 0, 43)),
    ((4, 0, 44, 0, 3), ("gather", 0, 44)),         # 44: global gathers
    ((4, 5, 9, 10, 45), ("box36", 5, 35)),         # the y extent decides: 35
    ((1, 6, 9, 10, 46), ("box44", 4, 36)),         # y 36; x floored to 4 for C = 1
    ((3, 2, 5, 0, 44), ("gather", 0, 44)),         # y 44
    ((4, -1, 20, 5, 9), ("box36", -1, 21)),        # C = 4: the box starts at x = -1
    ((3, -1, 31, 5, 9), ("box36", -4, 35)),        # C = 3: x origin -1 floored to -4 -> span 35
    ((3, -1, 32, 5, 9), ("box44", -4, 36)),        # ... and 36, where C = 4 would still fit the small box (33)
    ((4, -1, 32, 5, 9), ("box36", -1, 33)),
]


def test_tma_window_plan_hand_computed_tiles():
    for (C, x0, x1, y0, y1), (cat, xa, span) in HAND_TILES:
        p = tma_window_plan(_one_tile(x0, x1, y0, y1), 100, 100, C, 0)
        got = (str(p["cat"][0, 0, 0]), int(p["xa"][0, 0, 0]), int(p["span"][0, 0, 0]))
        assert got == (cat, xa, span), ((C, x0, x1, y0, y1), got)
        assert (p["xhi"][0, 0, 0], p["ylo"][0, 0, 0], p["yhi"][0, 0, 0]) == (x1, y0, y1)
    # x from 9 floored to 8 for C = 1: span 52 - 8 = 44 takes the gathers although x1 - x0 = 43
    p = tma_window_plan(_one_tile(9, 52, -1, 3), 100, 100, 1, 0)
    assert (str(p["cat"][0, 0, 0]), int(p["xa"][0, 0, 0]), int(p["span"][0, 0, 0])) == ("gather", 8, 44)
    p = tma_window_plan(_one_tile(9, 52, -1, 3), 100, 100, 4, 0)
    assert (str(p["cat"][0, 0, 0]), int(p["xa"][0, 0, 0]), int(p["span"][0, 0, 0])) == ("box44", 9, 43)


def test_tma_window_plan_tiles_without_a_valid_sample():
    w = np.full((1, 32, 32, 2), 5.5, np.float32)
    w[..., 0] = -1.0                                       # x = -1 is not > -1
    w[0, 3, 4] = (np.nan, 2.0)
    w[0, 7, 7] = (100.0, 2.0)                              # x = W is not < W
    w[0, 8, 8] = (2.0, -np.inf)
    assert str(tma_window_plan(w, 100, 100, 3, 0)["cat"][0, 0, 0]) == "none"
    w[0, 9, 9] = (99.99, -0.999)                           # one valid sample in the corner: box at (99, -1)
    p = tma_window_plan(w, 100, 100, 3, 0)
    assert (str(p["cat"][0, 0, 0]), int(p["xa"][0, 0, 0]), int(p["xhi"][0, 0, 0]), int(p["ylo"][0, 0, 0]),
            int(p["yhi"][0, 0, 0])) == ("box36", 96, 100, -1, 0)


@pytest.mark.parametrize("flags", [ADD_GRID, ADD_GRID | GRID_XY])
def test_tma_window_plan_forms_the_grid_like_the_kernel(flags):
    """A zero flow on a 64 x 96 output over a 64 x 96 source: tile (0, 1) covers rows 0..31 and columns 32..63.  In the
    reference's (Y,X) order x = row and y = column, so its box is x 0..32, y 32..64 (past H = 64 in extended coordinates);
    in XY order it is x 32..64, y 0..32."""
    p = tma_window_plan(np.zeros((1, 64, 96, 2), np.float32), 64, 96, 4, flags)
    box = tuple(int(p[k][0, 0, 1]) for k in ("xa", "xhi", "ylo", "yhi"))
    assert box == ((32, 64, 0, 32) if flags & GRID_XY else (0, 32, 32, 64))
    assert str(p["cat"][0, 0, 1]) == "box36"
    # reference order, tile (0, 2): y = 64..95 is past H = 64 for every sample -> nothing valid
    assert str(p["cat"][0, 0, 2]) == ("box36" if flags & GRID_XY else "none")


# ----------------------------------------------------------------------------------------------- warps for the paths
def _designs(H, W, C):
    """Tap boxes (x0, x1, y0, y1) in extended coordinates, one per tile, that between them reach every window path and
    both of its boundary spans, boxes that start at -1 and windows that run past W and H.  None: no valid sample."""
    xl = -1 if C == 4 else -4                              # x origin of a box that starts at x = -1
    if min(H, W) < 54:                                     # a source smaller than the 36^2 box: only the small window
        return [(-1, W, -1, H), None, (W - 2, W, H - 2, H), (-1, 2, -1, 2)]
    return [
        (-1, xl + 35, -1, 3),            # span 35, at (-1, -1)
        (8, 44, 10, 14),                 # 36
        (-1, xl + 43, 20, 24),           # 43, at x = -1
        (8, 52, 3, 7),                   # 44 -> gathers
        (2, 6, -1, 34),                  # y span 35, at y = -1
        (2, 6, H - 36, H),               # y 36, the 44^2 window runs past H
        (2, 6, H - 43, H),               # y 43
        (2, 6, 10, 54),                  # y 44 -> gathers
        (W - 5, W, H - 4, H),            # the bottom-right corner: the 36^2 window runs past W and H
        None,
        (-1, W, -1, H),                  # the whole source
        (W - 40, W, 0, 5),               # the 44^2 window past W
    ]


def path_warp(rng, B, H, W, Ho, Wo, C, flags, invalid_frac=0.03):
    """A warp (a flow when ADD_GRID is set) whose tiles take the boxes of _designs in turn.  Samples sit at k/64 past an
    integer, so flow = warp - grid and the kernel's flow + grid are exact in float32.  Each tile's first and last pixel
    pin its box; a few other pixels are made invalid (NaN, +-inf, 1e6, -1, W).  Returns (warp, free) where free marks the
    pixels that may be changed without changing any tile's box."""
    designs = _designs(H, W, C)
    x = np.empty((B, Ho, Wo), np.float32)
    y = np.empty((B, Ho, Wo), np.float32)
    free = np.ones((B, Ho, Wo), bool)
    bad = np.array([np.nan, np.inf, -np.inf, 1e6, -1e6, -1.0], np.float32)
    t = 0
    for b in range(B):
        for i0 in range(0, Ho, 32):
            for j0 in range(0, Wo, 32):
                d = designs[t % len(designs)]
                t += 1
                sl = (b, slice(i0, min(i0 + 32, Ho)), slice(j0, min(j0 + 32, Wo)))
                shape = x[sl].shape
                if d is None:
                    x[sl] = rng.choice(np.append(bad, W), shape)
                    y[sl] = rng.uniform(0, H - 1, shape)
                    continue
                x0, x1, y0, y1 = d
                frac = lambda: rng.integers(1, 64, shape) / np.float32(64)
                x[sl] = rng.integers(x0, x1, shape) + frac()
                y[sl] = rng.integers(y0, y1, shape) + frac()
                x[sl][0, 0], y[sl][0, 0] = x0 + 0.5, y0 + 0.5
                x[sl][-1, -1], y[sl][-1, -1] = x1 - 0.5, y1 - 0.5
                free[sl][0, 0] = free[sl][-1, -1] = False
    drop = free & (rng.random((B, Ho, Wo)) < invalid_frac)
    x[drop] = rng.choice(bad, int(drop.sum()))
    warp = np.stack([x, y], -1)
    if flags & ADD_GRID:
        ii, jj = np.meshgrid(np.arange(Ho, dtype=np.float32), np.arange(Wo, dtype=np.float32), indexing="ij")
        gx, gy = (jj, ii) if flags & GRID_XY else (ii, jj)
        warp = np.stack([x - gx, y - gy], -1)
    return np.ascontiguousarray(warp, np.float32), free


def _assert_paths(warp, H, W, C, flags, expect):
    p = tma_window_plan(warp, H, W, C, flags)
    cats = set(np.unique(p["cat"]).tolist())
    assert cats == set(expect), "the warp generator no longer reaches %s (got %s)" % (sorted(set(expect) - cats), sorted(cats))
    if "gather" in expect:
        spans = set(p["span"][p["cat"] != "none"].tolist())
        assert {35, 36, 43, 44} <= spans, sorted(spans)
        staged = p["cat"] != "none"
        box = np.where(p["span"] < BOX_S, BOX_S, BOX_L)
        assert ((p["xa"] < 0) & staged).any() and ((p["ylo"] < 0) & staged).any()
        assert ((p["xa"] + box > W) & (p["span"] < BOX_L) & staged).any()
        assert ((p["ylo"] + box > H) & (p["span"] < BOX_L) & staged).any()
    return p


# --------------------------------------------------------------------------------------------------------- GPU helpers
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L


def _count(label):
    return _lib().launch_count_named(label)


class _Counts:
    """Launches per label over a with-block."""

    def __init__(self, *labels):
        self.labels = labels

    def __enter__(self):
        torch.cuda.synchronize()
        self.n0 = {k: _count(k) for k in self.labels}
        return self

    def __exit__(self, *a):
        torch.cuda.synchronize()
        self.d = {k: _count(k) - self.n0[k] for k in self.labels}


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _at_offset(a, floats=1):
    """A contiguous CUDA copy of ``a`` that starts ``4 * floats`` bytes past a 16-byte boundary."""
    a = np.ascontiguousarray(a, np.float32)
    buf = torch.zeros(a.size + 4, dtype=torch.float32, device="cuda")
    t = buf[floats:floats + a.size].view(a.shape)
    t.copy_(torch.from_numpy(a))
    assert t.data_ptr() % 16 == 4 * floats and t.is_contiguous()
    return t


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _sampler_fwd(data, wf, flags, Ho, Wo, debug=True):
    B, H, W, C = data.shape
    out = torch.empty((B, Ho, Wo, C), dtype=torch.float32, device="cuda")
    idx = torch.empty((B, Ho, Wo, 4), dtype=torch.int32, device="cuda") if debug else None
    msk = torch.empty((B, Ho, Wo), dtype=torch.uint8, device="cuda") if debug else None
    rc = _lib().load().dmv_sampler_fwd(_ptr(data), _ptr(wf), _ptr(out), _ptr(idx), _ptr(msk), B, H, W, C, Ho, Wo, flags, _stream())
    assert rc == 0, _lib().last_error()
    return out, idx, msk


def _sampler_grad_warp(data, wf, go, flags):
    B, H, W, C = data.shape
    _, Ho, Wo, _ = go.shape
    gw = torch.empty((B, Ho, Wo, 2), dtype=torch.float32, device="cuda")
    rc = _lib().load().dmv_sampler_bwd(_ptr(data), _ptr(wf), _ptr(go), None, _ptr(gw), B, H, W, C, Ho, Wo, flags, None, 0, _stream())
    assert rc == 0, _lib().last_error()
    return gw


def _fused_ws(B, Ho, Wo):
    return torch.zeros(int(_lib().load().dmv_sampler_loss_workspace_size(B, Ho, Wo)), dtype=torch.uint8, device="cuda")


def _fused_raw(data, wf, target, weights, mode, inv, flags, ws=None, Ho=None, Wo=None, ws_bytes=None):
    """dmv_sampler_loss_fused straight through the C ABI: (rc, gen, grad_flow, loss)."""
    B, H, W, C = data.shape
    Ho = wf.shape[1] if Ho is None else Ho
    Wo = wf.shape[2] if Wo is None else Wo
    if ws is None:
        ws = _fused_ws(B, Ho, Wo)
    gen = torch.empty((B, Ho, Wo, C), dtype=torch.float32, device="cuda")
    gw = torch.empty((B, Ho, Wo, 2), dtype=torch.float32, device="cuda")
    loss = torch.empty((), dtype=torch.float32, device="cuda")
    w = (ctypes.c_float * len(weights))(*weights)
    rc = _lib().load().dmv_sampler_loss_fused(_ptr(data), _ptr(wf), _ptr(target), w, mode, float(inv), _ptr(gen), _ptr(gw), _ptr(loss),
                                              B, H, W, C, Ho, Wo, flags, _ptr(ws), ws.numel() if ws_bytes is None else ws_bytes, _stream())
    return rc, gen, gw, loss


def _np(t):
    return t.detach().cpu().numpy()


def _go_of_loss(gen, target, weights, mode, inv):
    """d loss / d gen in float32 in the fused kernel's order: (gq * w_c) * inv_count, gq = 2d or sign(d), d = gen - target."""
    d = (gen - target).astype(np.float32)
    gq = (np.float32(2) * d) if mode == "l2" else np.sign(d).astype(np.float32)
    return ((gq * np.asarray(weights, np.float32)) * np.float32(inv)).astype(np.float32)


def _loss64(gen, target, weights, mode, inv):
    d = gen.astype(np.float64) - target.astype(np.float64)
    e = d * d if mode == "l2" else np.abs(d)
    return float((e * np.asarray(weights, np.float64)).sum() * inv)


# ------------------------------------------------------------------------------------------ 2. window-path parity (GPU)
GEOMS = {"ragged": (2, 61, 76, 70, 100), "small_source": (2, 8, 12, 40, 36)}


@gpu
@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("flags", [0, ADD_GRID, ADD_GRID | GRID_XY], ids=["absolute", "flow_ref_yx", "flow_xy"])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_window_paths_match_the_oracle_and_the_tile_kernel(C, flags, geom):
    """Forward, grad_warp and the fused warp loss on tiles that reach each window path and its boundary spans: bit-equal
    to the oracle, and the same bits from the generic tile kernel (reached with the source at a 4-byte offset)."""
    B, H, W, Ho, Wo = GEOMS[geom]
    rng = np.random.default_rng(C * 100 + flags * 10 + len(geom))
    data = rng.random((B, H, W, C), dtype=np.float32)
    wf, _ = path_warp(rng, B, H, W, Ho, Wo, C, flags)
    _assert_paths(wf, H, W, C, flags, CATEGORIES if geom == "ragged" else ("none", "box36"))
    warp = absolute_warp(wf, flags)
    go = rng.standard_normal((B, Ho, Wo, C)).astype(np.float32)
    target = rng.random((B, Ho, Wo, C), dtype=np.float32)
    weights, mode, inv = [0.5, 1.0, 0.1, 2.0][:C], ("l1" if flags == ADD_GRID else "l2"), 1.0 / (B * Ho * Wo)

    d_al, d_off, w_t, go_t, tg_t = _cuda(data), _at_offset(data), _cuda(wf), _cuda(go), _cuda(target)
    with _Counts("sampler_fwd(tma)", "sampler_grad_warp(tma)", "sampler_loss_fused", "sampler_fwd", "sampler_grad_warp") as n:
        out, idx, msk = _sampler_fwd(d_al, w_t, flags, Ho, Wo)
        gw = _sampler_grad_warp(d_al, w_t, go_t, flags)
        rc, gen, gwf, loss = _fused_raw(d_al, w_t, tg_t, weights, LOSS_MODE[mode], inv, flags)
        assert rc == 0, _lib().last_error()
        out_t, idx_t, msk_t = _sampler_fwd(d_off, w_t, flags, Ho, Wo)
        gw_t = _sampler_grad_warp(d_off, w_t, go_t, flags)
    assert n.d == {"sampler_fwd(tma)": 1, "sampler_grad_warp(tma)": 1, "sampler_loss_fused": 1, "sampler_fwd": 1,
                   "sampler_grad_warp": 1}, n.d

    fx, fy, cx, cy, mask = T.resampler_indices(data.shape, warp)
    ref = T.resampler(data, warp)
    for o, i, m in ((out, idx, msk), (out_t, idx_t, msk_t)):
        assert np.array_equal(_np(i), np.stack([fx, fy, cx, cy], -1)), "corner indices not bit-exact"
        assert np.array_equal(_np(m), mask), "validity masks not bit-exact"
        assert np.array_equal(_np(o), ref), "forward: max |diff| %g" % np.nanmax(np.abs(_np(o) - ref))
    _, gw_ref = T.resampler_grad(data, warp, go)
    assert np.array_equal(_np(gw), gw_ref) and np.array_equal(_np(gw_t), gw_ref)
    # the fused kernel: gen, d loss / d flow through the oracle's grad with the kernel's dL/dgen, loss against float64
    assert np.array_equal(_np(gen), ref)
    go_loss = _go_of_loss(ref, target, weights, mode, inv)
    _, gw_loss = T.resampler_grad(data, warp, go_loss)
    assert np.array_equal(_np(gwf), gw_loss)
    assert float(loss) == pytest.approx(_loss64(ref, target, weights, mode, inv), rel=1e-5)
    # ... and the tile kernel given the same dL/dgen
    assert np.array_equal(_np(_sampler_grad_warp(d_off, w_t, _cuda(go_loss), flags)), _np(gwf))


# --------------------------------------------------------------------------------------- 3. the fused warp loss's edges
def _edge_case(C, order, B=2, H=61, W=76, Ho=70, Wo=100, seed=0):
    """Source, flow and target on the window-path tiles, with NaN, +-inf and +-1e6 flows on free pixels and pixels where
    the target equals the warped source (d = 0: sign(0) = 0 for L1)."""
    flags = ADD_GRID | (GRID_XY if order == "xy" else 0)
    rng = np.random.default_rng(seed)
    data = rng.random((B, H, W, C), dtype=np.float32)
    flow, free = path_warp(rng, B, H, W, Ho, Wo, C, flags)
    spots = free & (rng.random(free.shape) < 0.02)
    flow[spots, rng.integers(0, 2, int(spots.sum()))] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e6, -1e6], np.float32),
                                                                  int(spots.sum()))
    warp = absolute_warp(flow, flags)
    ref = T.resampler(data, warp)
    target = rng.random((B, Ho, Wo, C), dtype=np.float32)
    same = rng.random((B, Ho, Wo)) < 0.1
    target[same] = ref[same]
    return data, flow, target, warp, ref, flags


WEIGHTS = {1: [0.1], 3: [0.0, 0.1, 1.7], 4: [1.0, 0.0, 0.1, 2.5]}


@gpu
@pytest.mark.parametrize("order", ["ref_yx", "xy"])
@pytest.mark.parametrize("mode", ["l2", "l1"])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_fused_warp_loss_edges(C, mode, order):
    """flow_resample_loss with Hout x Wout != H x W, weights 0 and 0.1, invalid and huge flows, d = 0 pixels, an empty tile
    and tiles on every window path: gen bit-equal to the oracle, d loss / d flow bit-equal to the oracle's grad_warp under
    the kernel's dL/dgen and to the three separate calls, the loss within 1e-5 of float64, the same bits twice."""
    from dynamic_multiview_3d_b200 import functional as F
    data, flow, target, warp, ref, flags = _edge_case(C, order, seed=C * 10 + len(mode) + len(order))
    B, Ho, Wo = flow.shape[:3]
    _assert_paths(flow, data.shape[1], data.shape[2], C, flags, CATEGORIES)
    w, inv = WEIGHTS[C], 1.0 / (B * Ho * Wo)
    assert (ref == target).all(-1).any(), "no d = 0 pixel"
    d, t = _cuda(data), _cuda(target)

    rc, gen, gw, loss = _fused_raw(d, _cuda(flow), t, w, LOSS_MODE[mode], inv, flags)
    assert rc == 0, _lib().last_error()
    rc2, gen2, gw2, loss2 = _fused_raw(d, _cuda(flow), t, w, LOSS_MODE[mode], inv, flags)
    assert rc2 == 0 and torch.equal(gen, gen2) and torch.equal(gw, gw2) and _np(loss).tobytes() == _np(loss2).tobytes()
    assert np.array_equal(_np(gen), ref)
    _, gw_ref = T.resampler_grad(data, warp, _go_of_loss(ref, target, w, mode, inv))
    assert np.array_equal(_np(gw), gw_ref)
    assert float(loss) == pytest.approx(_loss64(ref, target, w, mode, inv), rel=1e-5)

    # through autograd, with the upstream scalar chained; k is a power of two, so scaling before the sampler's gradient
    # (the three calls) and after it (the fused kernel) round alike
    k = 0.5
    f = _cuda(flow).requires_grad_(True)
    with _Counts("sampler_loss_fused", "loss_flat") as n:
        l_f, gen_f = F.flow_resample_loss(d, f, t, mode, weights=w, inv_count=inv, grid_order=order)
        (l_f * k).backward()
    assert n.d == {"sampler_loss_fused": 1, "loss_flat": 0}, n.d
    assert torch.equal(gen_f, gen) and float(l_f) == float(loss)
    assert np.array_equal(_np(f.grad), gw_ref * np.float32(k))
    f3 = _cuda(flow).requires_grad_(True)
    with _Counts("sampler_loss_fused", "loss_flat") as n:
        gen3 = F.flow_resampler(d, f3, order)
        l3 = F.reconstruction_loss(gen3, t, mode, weights=w, inv_count=inv)
        (l3 * k).backward()
    assert n.d == {"sampler_loss_fused": 0, "loss_flat": 1}, n.d
    assert torch.equal(gen3.detach(), gen) and torch.equal(f3.grad, f.grad)
    assert float(l3) == pytest.approx(float(loss), rel=1e-5)


@gpu
def test_fused_warp_loss_over_256_ctas_and_grid_size_changes():
    """B = 6 at 224^2 is 294 CTAs: the last CTA's thread-strided sum of the partials takes more than one partial per thread.
    Small, large and small grids in turn on ONE workspace (the counter at its fixed place resets itself) each give the
    right loss; so do the same calls through flow_resample_loss, whose workspace grows on the large call."""
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(17)
    B, H, C = 6, 224, 3
    data = rng.random((B, H, H, C), dtype=np.float32)
    flow = rng.uniform(-3, 3, (B, H, H, 2)).astype(np.float32)
    flow[rng.random((B, H, H)) < 0.01, 0] = np.nan
    flow[5, 192:, 192:] = 1e6                               # the last tile has no valid sample
    target = rng.random((B, H, H, C), dtype=np.float32)
    warp = T.warp_pts_layer(flow)
    ref = T.resampler(data, warp)
    w, inv = [1.0, 0.5, 0.25], 1.0 / (B * H * H)
    d, f, t = _cuda(data), _cuda(flow), _cuda(target)
    assert (B * 7 * 7) > 256
    small = (slice(0, 1), slice(0, 40), slice(0, 36))     # 2 x 2 tiles of image 0 (a 40 x 36 flow over the same source)
    fs, ts = _cuda(flow[small]), _cuda(target[small])
    ref_s = T.resampler(data[:1], T.warp_pts_layer(flow[small]))
    loss64 = {"large": _loss64(ref, target, w, "l2", inv), "small": _loss64(ref_s, target[small], w, "l2", inv)}

    ws = _fused_ws(B, H, H)
    losses = {}
    for which in ("small", "large", "small", "large"):
        args = (d[:1], fs, ts) if which == "small" else (d, f, t)
        rc, gen, gw, loss = _fused_raw(*args, w, 0, inv, ADD_GRID, ws=ws)
        assert rc == 0, _lib().last_error()
        assert float(loss) == pytest.approx(loss64[which], rel=1e-5), which
        assert losses.setdefault(which, float(loss)) == float(loss)
        if which == "large":
            assert np.array_equal(_np(gen), ref)
            _, gw_ref = T.resampler_grad(data, warp, _go_of_loss(ref, target, w, "l2", inv))
            assert np.array_equal(_np(gw), gw_ref)
    F._loss_wss.pop(("warp_loss", "cuda", 0), None)
    for which in ("small", "large", "small"):
        args = (d[:1], fs, ts) if which == "small" else (d, f, t)
        with _Counts("sampler_loss_fused") as n:
            loss, _ = F.flow_resample_loss(*args, "l2", weights=w, inv_count=inv)
        assert n.d == {"sampler_loss_fused": 1} and float(loss) == losses[which], which


# ----------------------------------------------------------------------------------------------- 4. both loss kernels
def _grad_ref(a, b, w, mode, inv, k, kernel, mask=None):
    """dL/dgen in float32 in the kernel's own order, chained by k.  loss_flat: (gq * w_c) * inv.  loss_kernel, with
    d = (gen - target) * mask (mask 1 when absent): gq * ((w_c * mask) * inv), times the softmax weight 1.0 (exact)."""
    w = np.asarray(w, np.float32)
    m = np.ones(a.shape[:-1] + (1,), np.float32) if mask is None else mask
    d = (a - b).astype(np.float32)
    if kernel == "loss_fused":
        d = (d * m).astype(np.float32)
    gq = np.float32(2) * d if mode == "l2" else np.sign(d).astype(np.float32)
    g = (gq * w) * np.float32(inv) if kernel == "loss_flat" else gq * ((w * m) * np.float32(inv))
    return (g.astype(np.float32) * np.float32(k)).astype(np.float32)


def _loss_case(F, a_t, b_t, mode, w, inv, mask_t, k):
    at = a_t.detach().requires_grad_(True)                  # a leaf on the same buffer (and offset) as a_t
    loss = F.reconstruction_loss(at, b_t, mode, weights=w, inv_count=inv, mask=mask_t)
    (loss * k).backward()
    return loss.detach(), at.grad


def _check_loss_kernel(label, a, b, mode, w, a_t, b_t, mask=None, mask_t=None):
    """Two calls of reconstruction_loss, each chained by (loss * k).backward(): both run ``label``, give the same bits,
    the loss within 1e-5 of float64, and d loss / d gen bit-equal to the kernel's float32 order."""
    from dynamic_multiview_3d_b200 import functional as F
    inv, k = 1.0 / (a.size // a.shape[-1]), 0.375
    with _Counts("loss_flat", "loss_fused") as n:
        l1, g1 = _loss_case(F, a_t, b_t, mode, w, inv, mask_t, k)
        l2, g2 = _loss_case(F, a_t, b_t, mode, w, inv, mask_t, k)
    assert n.d == {"loss_flat": 2 * (label == "loss_flat"), "loss_fused": 2 * (label == "loss_fused")}, n.d
    assert _np(l1).tobytes() == _np(l2).tobytes() and torch.equal(g1, g2)
    d = a.astype(np.float64) - b.astype(np.float64)
    if mask is not None:
        d = d * mask
    ref = ((d * d if mode == "l2" else np.abs(d)) * np.asarray(w, np.float64)).sum() * inv
    assert float(l1) == pytest.approx(ref, rel=1e-5)
    assert np.array_equal(_np(g1), _grad_ref(a, b, w, mode, inv, k, label, mask))


def _loss_inputs(rng, shape):
    a = rng.random(shape, dtype=np.float32)
    b = rng.random(shape, dtype=np.float32)
    eq = rng.random(shape[:-1]) < 0.1
    b[eq] = a[eq]                                            # d = 0: sign(0) = 0
    return a, b


LW = {1: [0.1], 2: [0.0, 0.1], 3: [0.1, 0.0, 1.7], 4: [1.0, 0.0, 0.1, 2.5], 5: [0.1, 1.0, 0.0, 3.0, 0.5],
      8: [0.1, 1.0, 0.0, 3.0, 0.5, 0.25, 2.0, 0.7]}


@gpu
@pytest.mark.parametrize("mode", ["l2", "l1"])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_loss_flat_kernel(C, mode):
    """V = 1, no mask, pixels * C a multiple of 4, 16-byte aligned: loss_flat."""
    rng = np.random.default_rng(C + len(mode))
    a, b = _loss_inputs(rng, (5, 33, 16, C))
    _check_loss_kernel("loss_flat", a, b, mode, LW[C], _cuda(a), _cuda(b))


LOSS_ROUTES = [(C, r) for C in (1, 2, 3, 4, 5, 8) for r in ("mask", "offset", "odd") if not (r == "odd" and C % 4 == 0)]


@gpu
@pytest.mark.parametrize("mode", ["l2", "l1"])
@pytest.mark.parametrize("C,route", LOSS_ROUTES)
def test_loss_kernel_single_view(C, route, mode):
    """V = 1 calls that cannot take loss_flat run loss_kernel<C> (loss_kernel<0> for C in {2, 5, 8}): with a mask, with the
    prediction at a 4-byte offset, or with pixels * C not a multiple of 4 (3 x 11 x 7 = 231 pixels)."""
    rng = np.random.default_rng(C * 3 + len(route) + len(mode))
    shape = (3, 11, 7, C) if route == "odd" else (4, 11, 8, C)
    a, b = _loss_inputs(rng, shape)
    if route == "odd":
        assert (a.size % 4) != 0
    mask = rng.choice(np.array([0.0, 0.5, 1.0], np.float32), shape[:-1] + (1,)) if route == "mask" else None
    a_t = _at_offset(a) if route == "offset" else _cuda(a)
    _check_loss_kernel("loss_fused", a, b, mode, LW[C], a_t, _cuda(b), mask, None if mask is None else _cuda(mask))


@gpu
def test_both_loss_kernels_above_the_block_cap():
    """More work than kMaxBlocks = 1184 CTAs cover in one pass: loss_flat at 33 x 224^2 x 3 (1213 blocks wanted) and
    loss_kernel at 7 x 224^2 pixels (> 1184 * 256 = 303,104); both loop grid-stride.  Whole arrays against float64 NumPy."""
    rng = np.random.default_rng(23)
    a, b = _loss_inputs(rng, (33, 224, 224, 3))
    _check_loss_kernel("loss_flat", a, b, "l2", [0.5, 1.0, 0.1], _cuda(a), _cuda(b))
    a, b = a[:7], b[:7]
    mask = (rng.random((7, 224, 224, 1)) < 0.8).astype(np.float32)
    _check_loss_kernel("loss_fused", a, b, "l1", [0.5, 1.0, 0.1], _cuda(a), _cuda(b), mask, _cuda(mask))


def _fusion_inputs(rng, V, B, H, W, C, masked):
    """Logits per pixel: one view at +60 and the rest at -60, all views equal (0 or 60), or standard normal.  The target
    is the float64 fusion moved by 0.05 .. 0.45 either way, so sign(d) cannot differ between the kernel and the float64
    reference; d = 0 comes from mask = 0 (masks take 0, 0.5 and 1)."""
    kind = rng.integers(0, 3, (B, H, W))
    logits = rng.standard_normal((V, B, H, W)).astype(np.float32)
    hot = rng.integers(0, V, (B, H, W))
    one_hot = np.where(np.arange(V)[:, None, None, None] == hot[None], 60.0, -60.0).astype(np.float32)
    logits = np.where(kind[None] == 0, one_hot, logits)
    logits = np.where(kind[None] == 1, np.float32(60.0) * (rng.random((B, H, W)) < 0.5), logits).astype(np.float32)
    gens = rng.random((V, B, H, W, C), dtype=np.float32)
    f64 = (torch.softmax(torch.from_numpy(logits).double(), 0)[..., None] * torch.from_numpy(gens).double()).sum(0).numpy()
    sgn = np.where(rng.random((B, H, W, C)) < 0.5, -1.0, 1.0)
    target = (f64 + sgn * rng.uniform(0.05, 0.45, (B, H, W, C))).astype(np.float32)
    mask = rng.choice(np.array([0.0, 0.5, 1.0], np.float32), (B, H, W, 1)) if masked else None
    return gens, logits, target, mask


@gpu
@pytest.mark.parametrize("masked", [False, True], ids=["unmasked", "masked"])
@pytest.mark.parametrize("mode", ["l2", "l1"])
@pytest.mark.parametrize("C", [1, 3, 4])
@pytest.mark.parametrize("V", [2, 8])
def test_view_fusion_loss(V, C, mode, masked):
    """fused_views_loss (loss_kernel with V views): fused_out, the loss and both gradients against float64 torch autograd,
    chained by (loss * k).backward().  One call asks only for d loss / d gen and one only for d loss / d logits (the other
    pointer is NULL); both give the same fused output and loss bits.

    Tolerances: the softmax uses __expf, whose error is at most 2 + 1.173 |x| ulp.  The logit gaps that give a weight above
    float32's range here are below 8, so each weight is within ~1.2e-6 relative, and fused_out (V weights times values in
    [0, 1), accumulated by FMA) within 4e-6 absolute.  d loss / d gen = softmax * dL/dfused carries the weight's relative
    error: 1e-5 of max |ref|.  d loss / d logit_v = softmax_v * sum_c dL/dfused_c (gen_v,c - fused_c) also carries fused's
    absolute error once per channel: 4e-6 * softmax_v * sum_c |dL/dfused_c| on top of 1e-5 of max |ref|."""
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(V * 100 + C * 10 + len(mode) + masked)
    B, H, W = 2, 9, 13
    gens, logits, target, mask = _fusion_inputs(rng, V, B, H, W, C, masked)
    w, inv, k = [0.5, 1.0, 0.1, 2.0][:C], 1.0 / (B * H * W), 0.625
    tt, mt = _cuda(target), (None if mask is None else _cuda(mask))

    g64 = torch.from_numpy(gens).double().requires_grad_(True)
    l64 = torch.from_numpy(logits).double().requires_grad_(True)
    sm64 = torch.softmax(l64, 0)
    f64 = (sm64[..., None] * g64).sum(0)
    f64.retain_grad()
    d64 = f64 - torch.from_numpy(target).double()
    if mask is not None:
        d64 = d64 * torch.from_numpy(mask).double()
    e64 = d64 * d64 if mode == "l2" else d64.abs()
    ref = (e64 * torch.tensor(w, dtype=torch.float64)).sum() * inv
    (ref * k).backward()
    bound_logits = 4e-6 * sm64.detach().numpy() * f64.grad.abs().sum(-1).numpy()[None]

    outs = []
    for want in ("gen", "logits"):
        gt = _cuda(gens).requires_grad_(want == "gen")
        lt = _cuda(logits).requires_grad_(want == "logits")
        with _Counts("loss_fused", "loss_flat") as n:
            loss, fused = F.fused_views_loss(gt, lt, tt, mode, weights=w, inv_count=inv, mask=mt)
            (loss * k).backward()
        assert n.d == {"loss_fused": 1, "loss_flat": 0}, n.d
        assert (gt.grad is None) == (want != "gen") and (lt.grad is None) == (want != "logits")
        got = _np(gt.grad if want == "gen" else lt.grad)
        exp = (g64 if want == "gen" else l64).grad.numpy()
        err = np.abs(got - exp) - (bound_logits if want == "logits" else 0.0)
        assert err.max() <= 1e-5 * np.abs(exp).max(), (want, err.max() / np.abs(exp).max())
        outs.append((_np(loss).tobytes(), _np(fused)))
    assert outs[0][0] == outs[1][0] and np.array_equal(outs[0][1], outs[1][1])
    assert np.abs(outs[0][1] - f64.detach().numpy()).max() <= 4e-6
    assert float(np.frombuffer(outs[0][0], np.float32)[0]) == pytest.approx(float(ref), rel=1e-5)


# ------------------------------------------------------------------------------------ 5. sampler shapes and refusals
@gpu
def test_sampler_sixteen_channels():
    """C = 16, the tile kernel's largest: forward and grad_warp bit-equal, indices and masks bit-exact."""
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(31)
    B, H, W, C, Ho, Wo = 2, 21, 27, 16, 19, 23
    data = rng.random((B, H, W, C), dtype=np.float32)
    warp = rng.uniform(-2, [W + 1, H + 1], (B, Ho, Wo, 2)).astype(np.float32)
    warp[0, 0, :5, 0] = np.nan
    go = rng.standard_normal((B, Ho, Wo, C)).astype(np.float32)
    wt = _cuda(warp).requires_grad_(True)
    with _Counts("sampler_fwd", "sampler_grad_warp", "sampler_grad_data") as n:
        out, idx, msk = F.resampler_debug(_cuda(data), wt.detach())
        o2 = F.resampler(_cuda(data), wt)
        o2.backward(_cuda(go))
    assert n.d == {"sampler_fwd": 2, "sampler_grad_warp": 1, "sampler_grad_data": 0}, n.d
    fx, fy, cx, cy, mask = T.resampler_indices(data.shape, warp)
    assert np.array_equal(_np(idx), np.stack([fx, fy, cx, cy], -1)) and np.array_equal(_np(msk), mask)
    ref = T.resampler(data, warp)
    assert np.array_equal(_np(out), ref) and np.array_equal(_np(o2), ref)
    assert np.array_equal(_np(wt.grad), T.resampler_grad(data, warp, go)[1])


def _sampler_grads(data, warp, go, flags=0):
    from dynamic_multiview_3d_b200 import functional as F
    d = _cuda(data).requires_grad_(True)
    w = _cuda(warp).requires_grad_(True)
    out = F._Resampler.apply(d, w, flags)
    out.backward(_cuda(go))
    return _np(out), _np(d.grad), _np(w.grad)


@gpu
@pytest.mark.parametrize("C", [5, 7, 8])
def test_sampler_grad_data_generic_channels(C):
    """grad_data at C in {5, 7, 8} runs sampler_grad_data_kernel<0>: within 1e-5 of max |ref| and the same bits twice."""
    rng = np.random.default_rng(C)
    B, H, W, Ho, Wo = 2, 37, 45, 41, 35
    data = rng.random((B, H, W, C), dtype=np.float32)
    flow = rng.uniform(-3, 3, (B, Ho, Wo, 2)).astype(np.float32)
    flow[1, 5:9, 3:30] = rng.uniform(-60, 60, (4, 27, 2))
    go = rng.standard_normal((B, Ho, Wo, C)).astype(np.float32)
    with _Counts("sampler_grad_data", "sampler_box") as n:
        out, gd, gw = _sampler_grads(data, flow, go, ADD_GRID)
        _, gd2, gw2 = _sampler_grads(data, flow, go, ADD_GRID)
    assert n.d == {"sampler_grad_data": 2, "sampler_box": 2}, n.d
    assert np.array_equal(gd, gd2) and np.array_equal(gw, gw2)
    warp = T.warp_pts_layer(flow)
    assert np.array_equal(out, T.resampler(data, warp))
    gd_ref, gw_ref = T.resampler_grad(data, warp, go)
    assert np.array_equal(gw, gw_ref)
    assert np.abs(gd - gd_ref).max() <= 1e-5 * np.abs(gd_ref).max()


@gpu
def test_sampler_one_row_image_wider_than_a_tile():
    """Hout = 1 takes the 1 x 1024 sample-list tiling (and the tile kernel, even for an aligned RGB call); Wout = 2500
    spans three tiles, the last one ragged."""
    rng = np.random.default_rng(37)
    B, H, W, C, Wo = 2, 13, 29, 3, 2500
    data = rng.random((B, H, W, C), dtype=np.float32)
    warp = rng.uniform(-2, [W + 1, H + 1], (B, 1, Wo, 2)).astype(np.float32)
    go = rng.standard_normal((B, 1, Wo, C)).astype(np.float32)
    with _Counts("sampler_fwd", "sampler_fwd(tma)", "sampler_grad_warp", "sampler_grad_data") as n:
        out, gd, gw = _sampler_grads(data, warp, go)
    assert n.d == {"sampler_fwd": 1, "sampler_fwd(tma)": 0, "sampler_grad_warp": 1, "sampler_grad_data": 1}, n.d
    assert np.array_equal(out, T.resampler(data, warp))
    gd_ref, gw_ref = T.resampler_grad(data, warp, go)
    assert np.array_equal(gw, gw_ref)
    assert np.abs(gd - gd_ref).max() <= 1e-5 * np.abs(gd_ref).max()


@gpu
def test_sampler_and_loss_refusals():
    """Calls the library must refuse, with the code include/dmv3d.h gives, before anything is launched."""
    L = _lib().load()
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device="cuda")
    st = _stream()
    torch.cuda.synchronize()
    n0 = _lib().launch_count()
    d17, w = z(1, 8, 8, 17), z(1, 8, 8, 2)
    assert L.dmv_sampler_fwd(_ptr(d17), _ptr(w), _ptr(z(1, 8, 8, 17)), None, None, 1, 8, 8, 17, 8, 8, 0, st) == E_UNSUPPORTED_SHAPE
    d9 = z(1, 8, 8, 9)
    ws = torch.zeros(int(L.dmv_sampler_bwd_workspace_size(1, 8, 8, 9, 8, 8)), dtype=torch.uint8, device="cuda")
    assert L.dmv_sampler_bwd(_ptr(d9), _ptr(w), _ptr(z(1, 8, 8, 9)), _ptr(z(1, 8, 8, 9)), None, 1, 8, 8, 9, 8, 8, 0,
                             _ptr(ws), ws.numel(), st) == E_UNSUPPORTED_SHAPE
    d3 = z(1, 8, 8, 4)
    assert L.dmv_sampler_bwd(_ptr(d3), _ptr(w), _ptr(z(1, 8, 8, 4)), _ptr(z(1, 8, 8, 4)), None, 1, 8, 8, 4, 8, 8, 0,
                             _ptr(ws), 16, st) == E_WORKSPACE
    assert L.dmv_sampler_fwd(_ptr(d3), _ptr(w), _ptr(z(1, 8, 8, 4)), None, None, 1, 8, 8, 4, 8, 8, 4, st) == E_INVALID_ARG
    one = [1.0] * 4
    # fused warp loss: C = 2, Wout * C not a multiple of 4, Hout = 1, short workspace, unknown flag, unknown loss mode
    assert _fused_raw(z(1, 8, 8, 2), z(1, 8, 8, 2), z(1, 8, 8, 2), one[:2], 0, 1.0, ADD_GRID)[0] == E_UNSUPPORTED_SHAPE
    assert _fused_raw(z(1, 8, 8, 3), z(1, 8, 33, 2), z(1, 8, 33, 3), one[:3], 0, 1.0, ADD_GRID)[0] == E_UNSUPPORTED_SHAPE
    assert _fused_raw(z(1, 8, 8, 4), z(1, 1, 8, 2), z(1, 1, 8, 4), one, 0, 1.0, ADD_GRID)[0] == E_UNSUPPORTED_SHAPE
    need = int(L.dmv_sampler_loss_workspace_size(1, 8, 8))
    assert _fused_raw(d3, w, z(1, 8, 8, 4), one, 0, 1.0, ADD_GRID, ws_bytes=need - 1)[0] == E_WORKSPACE
    assert _fused_raw(d3, w, z(1, 8, 8, 4), one, 0, 1.0, 4)[0] == E_INVALID_ARG
    assert _fused_raw(d3, w, z(1, 8, 8, 4), one, 2, 1.0, ADD_GRID)[0] == E_INVALID_ARG
    # reconstruction loss: unknown mode, C = 9
    lws = torch.zeros(int(L.dmv_loss_workspace_size(64)), dtype=torch.uint8, device="cuda")
    cw = (ctypes.c_float * 9)(*([1.0] * 9))
    g, t, lo = z(64, 4), z(64, 4), z(1)
    assert L.dmv_loss_fused_fwd_bwd(_ptr(g), None, 1, _ptr(t), None, cw, 2, 1.0, _ptr(lo), None, None, None, 64, 4,
                                    _ptr(lws), lws.numel(), st) == E_INVALID_ARG
    assert L.dmv_loss_fused_fwd_bwd(_ptr(z(64, 9)), None, 1, _ptr(z(64, 9)), None, cw, 0, 1.0, _ptr(lo), None, None, None, 64, 9,
                                    _ptr(lws), lws.numel(), st) == E_UNSUPPORTED_SHAPE
    torch.cuda.synchronize()
    assert _lib().launch_count() == n0, "a refused call launched a kernel"


# -------------------------------------------------------------------- 6. warp_loss_supported agrees with the C ABI
@gpu
def test_warp_loss_supported_agrees_with_the_abi():
    """For C in 1..5, a few source and output widths, and the source, flow and target at 0 or a small offset:
    warp_loss_supported says yes exactly when dmv_sampler_loss_fused returns 0."""
    from dynamic_multiview_3d_b200 import functional as F
    rng = np.random.default_rng(41)
    seen = set()
    for C in range(1, 6):
        for W, Wo in ((36, 40), (37, 40), (36, 42), (44, 33)):
            B, H, Ho = 1, 34, 33
            data = rng.random((B, H, W, C), dtype=np.float32)
            flow = rng.uniform(-2, 2, (B, Ho, Wo, 2)).astype(np.float32)
            target = rng.random((B, Ho, Wo, C), dtype=np.float32)
            for od, of, ot in ((0, 0, 0), (1, 0, 0), (0, 0, 1), (1, 0, 1), (0, 2, 0)):   # offsets in floats
                d = _at_offset(data, od) if od else _cuda(data)
                f = _at_offset(flow, of) if of else _cuda(flow)
                t = _at_offset(target, ot) if ot else _cuda(target)
                ok = F.warp_loss_supported(d, f, t)
                rc = _fused_raw(d, f, t, [1.0] * C, 0, 1.0 / (Ho * Wo), ADD_GRID)[0]
                assert rc in (0, E_UNSUPPORTED_SHAPE), rc
                assert ok == (rc == 0), (C, W, Wo, od, of, ot, ok, rc)
                seen.add(ok)
    assert seen == {True, False}
    # a non-contiguous source is copied into a fresh (aligned) buffer by flow_resample_loss
    d = _cuda(rng.random((1, 34, 72, 4), dtype=np.float32))[:, :, :36]
    f = _cuda(rng.uniform(-2, 2, (1, 33, 40, 2)).astype(np.float32))
    t = _cuda(rng.random((1, 33, 40, 4), dtype=np.float32))
    assert not d.is_contiguous() and F.warp_loss_supported(d, f, t)
    with _Counts("sampler_loss_fused") as n:
        F.flow_resample_loss(d, f, t)
    assert n.d == {"sampler_loss_fused": 1}


@gpu
def test_model_takes_the_separate_calls_for_offset_inputs():
    """forward_and_loss on a source and a target at a 4-byte offset runs (through the separate sampler and loss calls) and
    gives the loss and flow gradient of aligned inputs.  The flow gradient is bit-equal: with unit channel weights and no
    mask, dL/dgen is gq * inv_count in both loss kernels' order."""
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200 import functional as F
    from dynamic_multiview_3d_b200.synthetic import make_batch
    B, H = 2, 64
    conf = {"batch_size": B, "learning_rate": 1e-4, "image_size": H, "viewpoint_dim": 19, "seed": 3}
    m = pkg.AppearanceFlowModel(conf)
    b = make_batch(B, H, "onehot19")
    img0, img1, disp = b["image0"], b["image1"], _cuda(b["disp"])
    res = {}
    for name, (i0, i1) in {"aligned": (_cuda(img0), _cuda(img1)), "offset": (_at_offset(img0), _at_offset(img1))}.items():
        assert F.warp_loss_supported(i0, torch.empty((B, H, H, 2), device="cuda"), i1) == (name == "aligned")
        with _Counts("sampler_loss_fused", "sampler_fwd", "loss_fused") as n:
            loss = m.forward_and_loss(i0, i1, disp)
            m.flow_field.retain_grad()
            loss.backward()
        res[name] = (float(loss), m.flow_field.detach().clone(), m.flow_field.grad.clone(), n.d)
    assert res["aligned"][3] == {"sampler_loss_fused": 1, "sampler_fwd": 0, "loss_fused": 0}, res["aligned"][3]
    assert res["offset"][3] == {"sampler_loss_fused": 0, "sampler_fwd": 1, "loss_fused": 1}, res["offset"][3]
    assert torch.equal(res["offset"][1], res["aligned"][1]), "the network's flow differs: the comparison below is moot"
    assert res["offset"][0] == pytest.approx(res["aligned"][0], rel=1e-5)
    assert torch.equal(res["offset"][2], res["aligned"][2])

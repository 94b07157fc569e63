"""The update path against a float64 Adam oracle at its edges.

- adam64: TF's float32 ApplyAdam evaluated in float64, with a per-element bound |x - x64| <= k (2^-24 s + 2^-150), s the
  magnitude of the terms that form x, k = 4 for the moments and 5 for theta.  CPU tests show that it accepts the float32 restatement T.adam_tf_step and rejects it
  once its update term is one ulp off.
- Value edges (zero, subnormal, overflowing, infinite and NaN gradients, cancelling moments, four grad scales) through
  every implementation of the update: dmv_adam_multi (float4 and scalar tail), its gated form, dmv_dp_exchange_chunk at
  world 1 (sharded and replicated) and dmv_linear_wgrad_adam (generic and streaming).  They must agree bit for bit.
- dmv_adam_tick over 100000 steps, past the points where the float32 powers b1^t, b2^t turn subnormal and stop moving.
- The exchange kernel on emulated ranks (every rank on one GPU, one stream per rank) at ragged slices, several
  grid-stride passes, non-zero starts, three grid sizes and three grad scales; the refusals of its C ABI.
- The host arguments of the exchange for every model class's variable store (CPU)."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle import tf_ops as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
F32 = np.float32
U24, ETA = 2.0 ** -24, 2.0 ** -150      # unit roundoff of float32; absolute rounding error in its subnormal range
# theta's float32 formula rounds five times (m lr_t, sqrt, + eps, the division, the subtraction), each by at most 2^-24
# of a term <= s: its worst case is 5 units of s, which the float32 restatement reaches on random data (1.08 x 4 units)
THETA_K = 5
LR, B1, B2, EPS = 1e-3, 0.9, 0.999, 1e-8


# --------------------------------------------------------------------------------------------------------------------
# float64 reference and its element-wise bound
# --------------------------------------------------------------------------------------------------------------------
def adam64(theta, g, m, v, lr_t, beta1, beta2, eps, gscale, moments=None):
    """One ApplyAdam step in float64 from float32 inputs.  The gradient ApplyAdam receives is the float32 product
    g * gscale; (1 - beta) are TF's float32 constants (1 - 0.999f = 0.0010000467).  theta's update is evaluated from
    ``moments`` = (m, v) when given (the moments a kernel wrote, already held to their own bounds), else from m64, v64.
    Returns ((theta64, m64, v64), (s_theta, s_m, s_v)): s = magnitude of the terms that form each result."""
    th, m0, v0 = (np.asarray(a, F32).astype(np.float64) for a in (theta, m, v))
    with np.errstate(all="ignore"):
        g = (np.asarray(g, F32) * F32(gscale)).astype(np.float64)
        o1, o2 = float(F32(1.0) - F32(beta1)), float(F32(1.0) - F32(beta2))
        lr_t, eps = float(F32(lr_t)), float(F32(eps))
        m64 = m0 + (g - m0) * o1
        v64 = v0 + (g * g - v0) * o2
        mk, vk = (m64, v64) if moments is None else tuple(np.asarray(a, F32).astype(np.float64) for a in moments)
        upd = mk * lr_t / (np.sqrt(vk) + eps)
        s = (np.abs(th) + np.abs(upd), np.abs(m0) + np.abs(g - m0) * o1, np.abs(v0) + np.abs(g * g - v0) * o2)
        return (th - upd, m64, v64), s


def bound_ratio(x, ref, s, k=4):
    """|x - ref| / (k (2^-24 s + 2^-150)) where the reference is finite (<= 1: inside the bound; a non-finite x there
    counts as infinitely far), 0 elsewhere.  k = 4 for the moments; theta takes k = 5 (THETA_K)."""
    with np.errstate(all="ignore"):
        r = np.abs(np.asarray(x, F32).astype(np.float64) - ref) / (k * (U24 * s + ETA))
    fin = np.isfinite(ref) & np.isfinite(s)
    return np.where(fin, np.nan_to_num(r, nan=np.inf), 0.0)


def check_adam(out, prev, g, t, gscale, lr=LR, what=""):
    """A kernel's step ``out`` = (theta, m, v) from ``prev``: its NaN / +-inf pattern equals T.adam_tf_step's exactly, and
    its finite values lie within the bound of adam64 applied to ``prev``."""
    gs = (np.asarray(g, F32) * F32(gscale)).astype(F32)
    with np.errstate(all="ignore"):
        r32 = T.adam_tf_step(*(np.asarray(a, F32) for a in (prev[0], gs, prev[1], prev[2])), t, lr)
    ref, s = adam64(prev[0], g, prev[1], prev[2], T.adam_lr_t(lr, t), B1, B2, EPS, gscale, moments=(out[1], out[2]))
    for name, a, b, x, sc, k in zip("theta m v".split(), out, r32, ref, s, (THETA_K, 4, 4)):
        # the kernels form g * g - v in one FMA: where g * g alone overflows but g * g - v does not, v stays finite, as its
        # float64 value confirms, while the restatement's is inf.  Such a finite v is held to the bound instead.
        fused = np.isinf(b) & np.isfinite(x) & np.isfinite(a)
        for f in (np.isnan, np.isposinf, np.isneginf):
            assert np.array_equal(f(a)[~fused], f(b)[~fused]), "%s %s: %s pattern differs from T.adam_tf_step" % (what, name, f.__name__)
        # bound: where the restatement is finite, and where the kernel stayed finite past its overflow; an inf that both
        # produce (g * g - v itself overflows) has a finite float64 value and was checked by pattern only
        r =np.where(np.isfinite(b) | fused, bound_ratio(a, x, sc, k), 0.0)
        assert r.max() <= 1.0, "%s %s: %.3g of the bound at %d" % (what, name, r.max(), int(r.argmax()))


def _random_state(rng, n):
    th = (rng.standard_normal(n) * 10.0 ** rng.uniform(-3, 1, n)).astype(F32)
    m = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 2, n)).astype(F32)
    v = (np.abs(rng.standard_normal(n)) * 10.0 ** rng.uniform(-8, 4, n)).astype(F32)
    g = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 3, n)).astype(F32)
    return th, m, v, g


@pytest.mark.parametrize("gscale", [1.0, 0.5, 0.3, 0.125])
def test_bound_accepts_the_float32_restatement(gscale):
    """T.adam_tf_step, the float32 restatement, stays inside the bound over five chained steps of random states whose
    moments span 8 and 12 decades."""
    rng = np.random.default_rng(int(gscale * 1000))
    th, m, v, _ = _random_state(rng, 200000)
    for t in range(1, 6):
        g = _random_state(rng, th.size)[3]
        out = T.adam_tf_step(th, (g * F32(gscale)).astype(F32), m, v, t, LR)
        check_adam(out, (th, m, v), g, t, gscale, what="t=%d" % t)
        th, m, v = out


def test_bound_rejects_one_ulp_in_the_update_term():
    """The same restatement with its update (m lr_t) / (sqrt(v) + eps) moved by one ulp is outside the bound, where
    update and theta are of one size, while the max-normalised check the suite used before (1e-6 of the array's
    maximum) still accepts it."""
    rng = np.random.default_rng(7)
    th, m, v, g = _random_state(rng, 100000)
    th = (rng.standard_normal(th.size) * 1e-3).astype(F32)     # theta of the update's size: s is not dominated by theta
    lr_t = T.adam_lr_t(LR, 3)
    o1, o2 = F32(1.0) - F32(B1), F32(1.0) - F32(B2)
    m1 = (m + (g - m) * o1).astype(F32)
    v1 = (v + (g * g - v) * o2).astype(F32)
    upd = ((m1 * lr_t) / (np.sqrt(v1) + F32(EPS))).astype(F32)
    good = (th - upd).astype(F32)
    bad = (th - np.nextafter(upd, F32(np.inf) * np.sign(upd))).astype(F32)
    ref, s = adam64(th, g, m, v, lr_t, B1, B2, EPS, 1.0, moments=(m1, v1))
    assert bound_ratio(good, ref[0], s[0], THETA_K).max() <= 1.0
    assert bound_ratio(bad, ref[0], s[0], THETA_K).max() > 1.0, "one ulp in the update term must leave the bound"
    assert np.abs(bad - ref[0]).max() <= 1e-6 * np.abs(ref[0]).max(), "the max-normalised check accepts it"


def test_bound_rejects_the_wrong_moment_constant():
    """(1 - beta2) taken as float32(0.001) instead of TF's 1 - 0.999f moves v by 4.7e-5 of its update: outside."""
    rng = np.random.default_rng(8)
    th, m, v, g = _random_state(rng, 10000)
    v = np.zeros_like(v)
    bad = (v + (g * g - v) * F32(0.001)).astype(F32)
    ref, s = adam64(th, g, m, v, 1e-3, B1, B2, EPS, 1.0)
    assert bound_ratio(bad, ref[2], s[2]).max() > 1.0


# --------------------------------------------------------------------------------------------------------------------
# GPU helpers
# --------------------------------------------------------------------------------------------------------------------
def _lib():
    from dynamic_multiview_3d_b200 import _lib as L
    return L


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _adam_multi(name, th, g, m, v, h, state, gscale, stream, gate=None):
    """dmv_adam_multi / _gated over the tensors of the lists th, g, m, v, h."""
    args = [_ptrs(th), _ptrs(g), _ptrs(m), _ptrs(v), _ptrs(h), (C.c_longlong * len(th))(*[t.numel() for t in th]), len(th),
            state.data_ptr(), B1, B2, EPS, gscale]
    _lib().call(name, *(args + ([gate.data_ptr()] if gate is not None else []) + [stream]))


def _exchange_call(grads, halves, sigs, master, m, v, local, start, n, rank, world, slot, rep, state, gscale, ctas, stream):
    return _lib().load().dmv_dp_exchange_chunk(_ptrs(grads), _ptrs(halves), _ptrs(sigs), None, None, master.data_ptr(), m.data_ptr(),
                                               v.data_ptr(), local.data_ptr(), start, n, rank, world, slot, rep, state.data_ptr(),
                                               B1, B2, EPS, gscale, ctas, stream)


def _in_child(fn, *args, timeout=420):
    """Runs ``fn(*args)`` of this module in a fresh interpreter and waits at most ``timeout`` seconds: an exchange that
    could not complete is reported as a failure instead of blocking the suite."""
    code = textwrap.dedent("""
        import sys
        sys.path[:0] = [%r, %r]
        import test_update_kernels_gpu as t
        t.%s(*%r)
        print("update verdict: ok")
    """ % (ROOT, os.path.join(ROOT, "tests"), fn, tuple(args)))
    try:
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired as e:
        pytest.fail("%s%r did not finish in %d s: %s" % (fn, args, timeout, (e.stdout or b"")[-2000:]))
    assert out.returncode == 0 and "update verdict: ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


# --------------------------------------------------------------------------------------------------------------------
# Adam's value edges through every implementation
# --------------------------------------------------------------------------------------------------------------------
def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a, F32)).to(torch.bfloat16)


def _edge_problem(rng, K, N):
    """x (K) and dy (N) of a one-sample linear layer, whose weight gradient x^T dy carries the edge values, and the
    (theta, m, v) table laid over it.  Rows of x: 1 (dy's values themselves: +-inf, NaN, +-1e20 whose square overflows,
    subnormals, 0), 0 (a zero gradient; inf * 0 = NaN), 1e-20 (subnormal products), 2^60 (overflowing products) and
    ordinary scales.  Every third row starts from m = v = 0 (a first step); two rows hold moments that nearly cancel
    the gradient (g - m ~ 0, and m + (g - m)(1 - b1) ~ 0)."""
    xs = [1.0, 0.0, 1e-20, 2.0 ** 60, -3.0, 0.5, 1.0, 1.0]
    x = np.array([xs[k % len(xs)] if k < 16 else rng.standard_normal() * 10.0 ** rng.uniform(-3, 3) for k in range(K)], F32)
    dy = (rng.standard_normal(N) * 10.0 ** rng.uniform(-3, 3, N)).astype(F32)
    dy[:12] = [np.inf, -np.inf, np.nan, 1e20, -1e20, 1e-20, -3e-39, 0.0, 1e-39, 2.0 ** 64, -0.0, 1.0]
    x, dy = _bf16(x).float().numpy(), _bf16(dy).float().numpy()
    with np.errstate(all="ignore"):
        gp = np.outer(x, dy).astype(F32)
    th, m, v, _ = _random_state(rng, K * N)
    th, m, v = th.reshape(K, N), m.reshape(K, N), v.reshape(K, N)
    fresh = np.arange(K) % 3 == 1                      # includes the x = 0 row
    m[fresh], v[fresh] = 0.0, 0.0
    with np.errstate(all="ignore"):
        m[6] = np.where(np.isfinite(gp[6]), gp[6] * F32(1 - 2.0 ** -20), m[6])          # g - m nearly cancels
        m[7] = np.where(np.isfinite(gp[7]), -gp[7] / F32(9.0) * F32(1 + 2.0 ** -18), m[7])  # the new m nearly cancels
    return x, dy, th.astype(F32), m.astype(F32), v.astype(F32)


SUB = 2
SUB_ROW = np.array([1e-40, -1e-40, 1.4e-45, -1.4e-45, 1e-39, -3e-39, 1.17e-38, 0.0, np.inf, -np.inf, np.nan, 1e20, -1e20, 1.0, -1e-3], F32)
FORMS = ("fc", "multi", "scalar", "tail", "gated", "exchange", "exchange-rep")


@gpu
@pytest.mark.parametrize("K,N,fc_label", [(64, 256, "linear_wgrad_adam (stream)"), (40, 136, "linear_wgrad_adam")])
def test_adam_edges_bit_identical_across_implementations(K, N, fc_label):
    """Two steps at each grad scale in {1, 0.5, 0.3, 1/8}.  The linear layer's fused update computes the gradient (its
    dw_out); the same gradient and state then go through dmv_adam_multi on float4 chunks, on the scalar kernel (a tensor
    4 bytes into its allocation), on a float4 body with a scalar tail (n % 4 = 3), its gated form with gate 1 and the
    exchange kernel at world 1, sharded and replicated.  theta, m, v and the bf16 copy are bit-identical across all
    seven; the launch counters prove the form of each; the result matches T.adam_tf_step's NaN / inf pattern and adam64's
    bound; a zero gradient at a first step leaves theta, m and v exactly unchanged."""
    L = _lib()
    L.load()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    n = K * N
    labels = (fc_label, "adam_multi", "adam_scalar", "dp_exchange_chunk")
    for gscale in (1.0, 0.5, 0.3, 0.125):
        rng = np.random.default_rng(int(gscale * 100) + K)
        x, dy, th0, m0, v0 = _edge_problem(rng, K, N)
        bufs = {}
        for f in FORMS:
            off = 1 if f == "scalar" else 0                       # the scalar form's tensors start 4 bytes in
            b = {k: torch.empty(n + 4, device=dev)[off:off + n] for k in ("th", "m", "v", "g")}
            for k, a in (("th", th0), ("m", m0), ("v", v0)):
                b[k].copy_(torch.from_numpy(a.ravel()))
            b["h"] = torch.zeros(n + 8, dtype=torch.bfloat16, device=dev)[2 * off:2 * off + n]
            bufs[f] = b
        ex = {k: torch.zeros(L.load().dmv_dp_signal_words(1), dtype=torch.int32, device=dev) for k in ("sig", "sig-rep")}
        loc = {k: torch.zeros(2, dtype=torch.int32, device=dev) for k in ("exchange", "exchange-rep")}
        gate = torch.ones(1, dtype=torch.int32, device=dev)
        state = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
        prev = prev_fc = (th0.ravel(), m0.ravel(), v0.ravel())
        for t in (1, 2):
            if t == 2:
                x, dy = _edge_problem(rng, K, N)[:2]
            L.call("dmv_adam_tick", state.data_ptr(), LR, B1, B2, st)
            c0 = {l: L.launch_count_named(l) for l in labels}
            b = bufs["fc"]
            xd, dyd = _bf16(x).cuda(), _bf16(dy).cuda()
            L.call("dmv_linear_wgrad_adam", xd.data_ptr(), dyd.data_ptr(), b["th"].data_ptr(), b["m"].data_ptr(), b["v"].data_ptr(),
                   b["h"].data_ptr(), b["g"].data_ptr(), 1, K, N, state.data_ptr(), B1, B2, EPS, gscale, st)
            torch.cuda.synchronize()
            # the others take the linear layer's gradient, but row SUB (x = 1e-20) carries exact subnormals and the edge
            # values whatever the tensor cores make of subnormal products; there the linear layer is checked on its own
            g = b["g"].clone().view(K, N)
            g[SUB] = torch.from_numpy(np.resize(SUB_ROW, N))
            g = g.view(-1)
            ran = {}
            for f in FORMS[1:]:
                b = bufs[f]
                b["g"].copy_(g)
                c = {l: L.launch_count_named(l) for l in labels}
                if f in ("multi", "scalar"):
                    _adam_multi("dmv_adam_multi", [b["th"]], [b["g"]], [b["m"]], [b["v"]], [b["h"]], state, gscale, st)
                elif f == "tail":
                    cut = n - 5                                   # n % 4 = 3: float4 body + 3-element tail, then 5 elements at 12 bytes
                    parts = lambda k: [b[k][:cut], b[k][cut:]]
                    _adam_multi("dmv_adam_multi", parts("th"), parts("g"), parts("m"), parts("v"), parts("h"), state, gscale, st)
                elif f == "gated":
                    _adam_multi("dmv_adam_multi_gated", [b["th"]], [b["g"]], [b["m"]], [b["v"]], [b["h"]], state, gscale, st, gate)
                else:
                    rep = int(f == "exchange-rep")
                    rc = _exchange_call([b["g"]], [b["h"]], [ex["sig-rep" if rep else "sig"]], b["th"], b["m"], b["v"], loc[f], 0, n, 0, 1, 0,
                                        rep, state, gscale, 0, st)
                    assert rc == 0, L.last_error()
                torch.cuda.synchronize()
                ran[f] = {l: L.launch_count_named(l) - c[l] for l in labels}
            assert L.launch_count_named(fc_label) == c0[fc_label] + 1, "the linear update did not take form %r" % fc_label
            want = {"multi": (1, 0, 0), "scalar": (0, 1, 0), "tail": (1, 2, 0), "gated": (1, 0, 0), "exchange": (0, 0, 1),
                    "exchange-rep": (0, 0, 1)}
            for f, (nm, ns, nx) in want.items():
                got = (ran[f]["adam_multi"], ran[f]["adam_scalar"], ran[f]["dp_exchange_chunk"])
                assert got == (nm, ns, nx), (f, got)
            ref = bufs["multi"]
            rows = torch.arange(n, device=dev) // N != SUB
            for f in FORMS:
                for k in ("th", "m", "v", "h"):
                    a, r_ = _bits(bufs[f][k]), _bits(ref[k])
                    if f == "fc":
                        a, r_ = a[rows], r_[rows]
                    assert torch.equal(a, r_), "%s differs from adam_multi in %s (gscale %g, t %d)" % (f, k, gscale, t)
            out = tuple(ref[k].cpu().numpy() for k in ("th", "m", "v"))
            gn = g.cpu().numpy()
            check_adam(out, prev, gn, t, gscale, what="gscale %g t %d" % (gscale, t))
            out_fc = tuple(bufs["fc"][k].cpu().numpy() for k in ("th", "m", "v"))
            check_adam(out_fc, prev_fc, bufs["fc"]["g"].cpu().numpy(), t, gscale, what="linear gscale %g t %d" % (gscale, t))
            prev_fc = out_fc
            assert torch.equal(_bits(ref["h"]), _bits(ref["th"].to(torch.bfloat16)))
            if t == 1:
                # a first step: m = v = +0 (m = -0 becomes -0 + (g - m)(1 - b1) = +0, as in TF)
                z = (gn == 0) & (prev[1].view(np.int32) == 0) & (prev[2].view(np.int32) == 0)
                assert z.sum() >= N // 2
                for a, p in zip(out, prev):
                    assert np.array_equal(a[z].view(np.int32), p[z].view(np.int32)), "a zero first-step gradient changed the state"
                for name, sel in (("subnormal", (gn != 0) & (np.abs(gn) < np.finfo(F32).tiny)), ("overflowing", np.abs(gn) >= 1e20),
                                  ("infinite", np.isinf(gn)), ("NaN", np.isnan(gn))):
                    assert sel.any(), "the gradient holds no %s value" % name
                big = np.isfinite(gn) & (np.abs(gn) * F32(gscale) > 2e19)
                assert np.isposinf(out[2][big]).all() and np.array_equal(out[0][big], prev[0][big]), "g*g overflows: v = inf, theta unchanged"
                assert np.isnan(out[0][np.isinf(gn)]).all()
            prev = out


# --------------------------------------------------------------------------------------------------------------------
# dmv_adam_tick over a long horizon
# --------------------------------------------------------------------------------------------------------------------
TICKS = {(0.9, 0.999): [1, 2, 10, 100, 828, 829, 964, 965, 1000, 20000, 87293, 87294, 96902, 100000],
         (0.5, 0.99): [1, 126, 127, 149, 150, 151, 1000, 8689, 8690, 9876, 9877, 20000]}


def _tick_oracle(lr, b1, b2, ts):
    """{t: (b1^t, b2^t, lr_t, t)} as TF keeps them: float32 running products, lr_t = lr sqrt(1 - b2^t) / (1 - b1^t)."""
    f, out, p1, p2 = F32, {}, F32(1.0), F32(1.0)
    for t in range(1, max(ts) + 1):
        p1, p2 = f(p1 * f(b1)), f(p2 * f(b2))
        if t in ts:
            out[t] = (p1, p2, f(f(lr) * np.sqrt(f(1.0) - p2, dtype=F32) / (f(1.0) - p1)), f(t))
    return out


def test_tick_oracle_reaches_the_power_edges():
    """The checkpoints sit on the float32 powers' edges: first subnormal, then stuck (x * b rounds back to x)."""
    o = _tick_oracle(LR, 0.9, 0.999, TICKS[(0.9, 0.999)])
    tiny = np.finfo(F32).tiny
    assert o[828][0] >= tiny > o[829][0] > o[964][0] and o[965][0] == o[1000][0] == o[100000][0] > 0
    assert F32(o[965][0] * F32(0.9)) == o[965][0] and F32(o[96902][1] * F32(0.999)) == o[96902][1]
    assert o[87293][1] >= tiny > o[87294][1] and o[96902][1] == o[100000][1] > 0
    assert float(o[100000][2]) == float(T.adam_lr_t(LR, 100000))
    o = _tick_oracle(0.01, 0.5, 0.99, TICKS[(0.5, 0.99)])
    assert o[126][0] >= tiny > o[127][0] > 0 and o[150][0] == 0 and o[8689][1] >= tiny > o[8690][1] and o[9876][1] == o[20000][1] > 0


@gpu
def test_adam_tick_long_horizon():
    """The device state {b1^t, b2^t, lr_t, t} after t ticks equals the oracle's float32 running products and
    T.adam_lr_t bit for bit, at beta (0.9, 0.999) up to t = 100000 and (0.5, 0.99), whose b1^t rounds to 0 at t = 150.
    Ticks replay from a captured graph of 1000."""
    L = _lib()
    L.load()
    for (b1, b2), ts in TICKS.items():
        lr = LR if b1 == 0.9 else 0.01
        ref = _tick_oracle(lr, b1, b2, ts)
        state = torch.tensor([1.0, 1.0, 0.0, 0.0], device="cuda")
        s = torch.cuda.Stream()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            cs = torch.cuda.current_stream().cuda_stream
            for _ in range(1000):
                L.call("dmv_adam_tick", state.data_ptr(), lr, b1, b2, cs)
        state.copy_(torch.tensor([1.0, 1.0, 0.0, 0.0]))
        cur = 0
        st = torch.cuda.current_stream().cuda_stream
        for t in ts:
            while t - cur >= 1000:
                graph.replay()
                cur += 1000
            while cur < t:
                L.call("dmv_adam_tick", state.data_ptr(), lr, b1, b2, st)
                cur += 1
            got = state.cpu().numpy()
            want = np.array(ref[t], F32)
            assert np.array_equal(got.view(np.int32), want.view(np.int32)), (b1, b2, t, got, want)
            if t <= 20000:
                assert got[2] == T.adam_lr_t(lr, t, b1, b2), (b1, b2, t)
        del graph


# --------------------------------------------------------------------------------------------------------------------
# the exchange kernel on emulated ranks
# --------------------------------------------------------------------------------------------------------------------
THREADS, SENT32, SENT16 = 256, 0x5EADBEEF, 0x5EAD


def _unroll(world):
    return 1 if world >= 8 else (2 if world >= 4 else 4)


def exchange_grid(n_slice, world, ctas):
    """The grid dmv_dp_exchange_chunk launches (csrc/exchange.cu): at most ``ctas`` (default 4 x 148), at most one CTA
    per four warp-block rounds of the slice, at least 1."""
    want = -(-(n_slice // 4) // (THREADS * _unroll(world) * 4))
    return max(1, min(ctas if ctas > 0 else 4 * 148, want))


def exchange_cases(world):
    """(n_slice, ctas, grad_scale, start): every n_slice with ctas 1, 3 and 0, the grad scale and start rotating.
    The largest slice is ragged and takes 13 grid-stride passes at ctas = 1."""
    sizes = [8, 256, 264, 768, 12288 * _unroll(world) + 264]
    scales = [1.0, 1.0 / world, 0.3]
    cases = []
    for i, n in enumerate(sizes):
        for j, ctas in enumerate((1, 3, 0)):
            cases.append((n, ctas, scales[(i + j) % 3], 36 * ((i + j) % 2)))
    return cases


def test_exchange_cases_reach_the_kernel_edges():
    """The cases include slices that end mid-block (n_slice = 256 mod 512 at world 2, the ragged production chunk),
    slices shorter than a warp block, three or more grid-stride passes, every grad scale and non-zero starts."""
    for world in (1, 2, 4, 8):
        cases = exchange_cases(world)
        blk = 32 * _unroll(world)
        assert any((n // 4) % blk for n, _, _, _ in cases) and any(n // 4 < blk for n, _, _, _ in cases)
        assert any(-(-(n // 4) // (exchange_grid(n, world, c) * 8 * blk)) >= 3 for n, c, _, _ in cases if c == 1)
        assert any(exchange_grid(n, world, c) == 3 for n, c, _, _ in cases if c == 3)
        assert {s for _, _, s, _ in cases} == {1.0, 1.0 / world, 0.3} and {st for *_, st in cases} == {0, 36}
    assert any(n % 512 == 256 for n, *_ in exchange_cases(2))


def _rank_order_sum(gs):
    acc = gs[0].copy()
    for g in gs[1:]:
        acc = (acc + g).astype(F32)
    return acc


def _exchange_case(world, n_slice, ctas, gscale, start, steps, rng, sms):
    """One case on emulated ranks: ``steps`` steps, each with the sharded chunk (slot 0) on every rank's comm stream
    and the replicated tail (slot 1) on its tail stream, all in flight together.  Returns the number of summed
    elements whose rank-order float32 sum differs from the reverse order."""
    L = _lib()
    dev = torch.device("cuda:0")
    tail_n = 264
    chunk = n_slice * world
    tail0 = start + chunk
    end = tail0 + tail_n
    alloc = end + 64                              # sentinels past the last element: >= 64 bytes
    region = end - start
    resident = world * (exchange_grid(n_slice, world, ctas) + exchange_grid(tail_n, world, ctas))
    assert resident <= sms, "every CTA of every rank must be resident at once (%d > %d)" % (resident, sms)
    words = L.load().dmv_dp_signal_words(2)

    def sentinel(dtype):
        return torch.full((alloc,), SENT32 if dtype == torch.int32 else SENT16, dtype=dtype, device=dev)

    ranks = []
    for r in range(world):
        x = {"grad": sentinel(torch.int32).view(torch.float32), "half": sentinel(torch.int16).view(torch.bfloat16)}
        th = (rng.standard_normal(region) * 0.5).astype(F32)
        m = (rng.standard_normal(region) * 1e3).astype(F32)
        v = (np.abs(rng.standard_normal(region)) * 1e12).astype(F32)
        for k, a in (("master", th), ("m", m), ("v", v)):
            x[k] = sentinel(torch.int32).view(torch.float32)
            x[k][start:end].copy_(torch.from_numpy(a))
            x[k + "0"] = x[k].clone()
        x["sig"] = torch.zeros(words, dtype=torch.int32, device=dev)
        x["local"] = torch.zeros(4, dtype=torch.int32, device=dev)
        x["comm"], x["tail"] = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        ranks.append(x)
    # reference: rank q's state over the region, updated by dmv_adam_multi from the rank-order float32 sum
    ref = {k: torch.stack([x[k][start:end] for x in ranks]).contiguous() for k in ("master", "m", "v")}
    ref["half"] = torch.zeros(world, region, dtype=torch.bfloat16, device=dev)
    ref["g"] = torch.empty(world, region, device=dev)
    state = torch.tensor([1.0, 1.0, 0.0, 0.0], device=dev)
    st = torch.cuda.current_stream().cuda_stream
    grads, halves, sigs = [x["grad"] for x in ranks], [x["half"] for x in ranks], [x["sig"] for x in ranks]
    order_diff = 0
    mags = np.array([1e8, 1.0, -1e8, 1e-3], F32)
    for step in range(1, steps + 1):
        gs = [(rng.standard_normal(region) * mags[rng.integers(0, 4, region)]).astype(F32) for _ in range(world)]
        gsum = _rank_order_sum(gs)
        order_diff += int((gsum != _rank_order_sum(gs[::-1])).sum())
        for x, g in zip(ranks, gs):
            x["grad"][start:end].copy_(torch.from_numpy(g))
        grad_before = [x["grad"].clone() for x in ranks]
        ref["g"].copy_(torch.from_numpy(gsum).expand(world, region))
        prev = {k: ref[k].cpu().numpy() for k in ("master", "m", "v")}
        L.call("dmv_adam_tick", state.data_ptr(), LR, B1, B2, st)
        _adam_multi("dmv_adam_multi", list(ref["master"]), list(ref["g"]), list(ref["m"]), list(ref["v"]), list(ref["half"]), state, gscale, st)
        torch.cuda.synchronize()
        c0 = L.launch_count_named("dp_exchange_chunk")
        for r, x in enumerate(ranks):
            for s_, n_, slot, rep in ((x["comm"], n_slice, 0, 0), (x["tail"], tail_n, 1, 1)):
                rc = _exchange_call(grads, halves, sigs, x["master"], x["m"], x["v"], x["local"], start if slot == 0 else tail0, n_, r, world,
                                    slot, rep, state, gscale, ctas, s_.cuda_stream)
                assert rc == 0, L.last_error()
        torch.cuda.synchronize()
        assert L.launch_count_named("dp_exchange_chunk") == c0 + 2 * world
        what = "world %d n_slice %d ctas %d gscale %g start %d step %d" % (world, n_slice, ctas, gscale, start, step)
        for r, x in enumerate(ranks):
            own = slice(start + r * n_slice, start + (r + 1) * n_slice)
            rown = slice(r * n_slice, (r + 1) * n_slice)
            for k in ("master", "m", "v"):
                got, want = _bits(x[k]), _bits(x[k + "0"])
                assert torch.equal(got[own], _bits(ref[k][r][rown])), "%s: rank %d's owned %s" % (what, r, k)
                assert torch.equal(got[tail0:end], _bits(ref[k][r][chunk:])), "%s: rank %d's tail %s" % (what, r, k)
                assert torch.equal(got[:own.start], want[:own.start]) and torch.equal(got[own.stop:tail0], want[own.stop:tail0]), \
                    "%s: rank %d's %s changed outside its slice" % (what, r, k)
                assert torch.equal(got[end:], want[end:]), "%s: rank %d's %s changed past the tail" % (what, r, k)
            assert torch.equal(_bits(x["grad"]), _bits(grad_before[r])), "%s: rank %d's gradient changed" % (what, r)
            h = _bits(x["half"])
            for q in range(world):                    # the owners' bf16 chunk on every rank, the own tail under replicated=1
                assert torch.equal(h[start + q * n_slice:start + (q + 1) * n_slice], _bits(ref["half"][q][q * n_slice:(q + 1) * n_slice])), \
                    "%s: rank %d's bf16 copy of rank %d's slice" % (what, r, q)
            assert torch.equal(h[tail0:end], _bits(ref["half"][r][chunk:])), "%s: rank %d's bf16 tail" % (what, r)
            assert bool((h[:start] == SENT16).all()) and bool((h[end:] == SENT16).all()), "%s: rank %d's bf16 outside the chunk" % (what, r)
            sel = np.r_[rown, chunk:region]
            out = tuple(x[k][start:end].cpu().numpy()[sel] for k in ("master", "m", "v"))
            check_adam(out, tuple(prev[k][r][sel] for k in ("master", "m", "v")), gsum[sel], step, gscale, what="%s rank %d" % (what, r))
        for k in ("master", "m", "v"):
            for x in ranks:
                x[k + "0"] = x[k].clone()
    for x in ranks:
        loc = x["local"].cpu().tolist()
        assert loc == [steps, 0, steps, 0], loc
        sig = x["sig"].cpu().numpy().reshape(2, 2, 8)
        assert (sig[:, :, :world] == steps).all() and (sig[:, :, world:] == 0).all(), sig
    return order_diff


def child_exchange(world):
    torch.cuda.init()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(100 + world)
    diff = 0
    for n, ctas, gscale, start in exchange_cases(world):
        diff += _exchange_case(world, n, ctas, gscale, start, 6, rng, sms)
    if world >= 4:
        assert diff > 0, "the gradients must make the rank-order sum differ from the reverse order"


@gpu
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_exchange_emulated_ranks_at_the_edges(world):
    """Owned theta, m, v bit-equal to dmv_adam_multi on the rank-order float32 sum (and inside adam64's bound), every
    rank's bf16 chunk equal to the owners' results, every byte outside what a rank owns unchanged (sentinels in the
    state and bf16 buffers, the gradients), the slot words at (steps, 0) and the signal words at steps."""
    _in_child("child_exchange", world)


@gpu
def test_exchange_empty_slice_launches_nothing():
    L = _lib()
    t = torch.zeros(64, device="cuda")
    sig = torch.zeros(L.load().dmv_dp_signal_words(1), dtype=torch.int32, device="cuda")
    local = torch.zeros(2, dtype=torch.int32, device="cuda")
    state = torch.tensor([1.0, 1.0, 1e-3, 1.0], device="cuda")
    c0 = L.launch_count_named("dp_exchange_chunk")
    assert _exchange_call([t, t], [t, t], [sig, sig], t, t, t, local, 0, 0, 0, 2, 0, 0, state, 1.0, 0, None) == 0
    torch.cuda.synchronize()
    assert L.launch_count_named("dp_exchange_chunk") == c0 and local.tolist() == [0, 0] and not sig.any()


@gpu
def test_exchange_refusals_launch_nothing():
    """Each refusal returns its documented code (include/dmv3d.h) and launches nothing."""
    L = _lib()
    t = torch.zeros(256, device="cuda")
    h = torch.zeros(256, dtype=torch.bfloat16, device="cuda")
    sig = torch.zeros(L.load().dmv_dp_signal_words(1), dtype=torch.int32, device="cuda")
    local = torch.zeros(2, dtype=torch.int32, device="cuda")
    state = torch.tensor([1.0, 1.0, 1e-3, 1.0], device="cuda")
    INVALID, ALIGN, SHAPE = -1, -2, -3
    base = dict(grads=[t, t], halves=[h, h], sigs=[sig, sig], master=t, m=t, v=t, start=0, n=64, rank=0, world=2, slot=0)
    null = type("Null", (), {"data_ptr": lambda self: 0})()
    cases = [(dict(grads=[t, null]), INVALID), (dict(halves=[null, h]), INVALID), (dict(sigs=[sig, null]), INVALID),
             (dict(grads=[t, t[1:]]), ALIGN), (dict(halves=[h[2:], h]), ALIGN), (dict(master=t[1:]), ALIGN), (dict(m=t[1:]), ALIGN),
             (dict(v=t[1:]), ALIGN), (dict(n=60), ALIGN), (dict(n=12), ALIGN), (dict(start=2), ALIGN), (dict(start=6), ALIGN),
             (dict(world=0), INVALID), (dict(world=3, grads=[t] * 3, halves=[h] * 3, sigs=[sig] * 3), SHAPE),
             (dict(world=5, grads=[t] * 5, halves=[h] * 5, sigs=[sig] * 5), SHAPE),
             (dict(world=9, grads=[t] * 9, halves=[h] * 9, sigs=[sig] * 9), INVALID),
             (dict(rank=2), INVALID), (dict(rank=-1), INVALID), (dict(slot=-1), INVALID)]
    for change, code in cases:
        a = dict(base, **change)
        c0 = L.launch_count_named("dp_exchange_chunk")
        rc = _exchange_call(a["grads"], a["halves"], a["sigs"], a["master"], a["m"], a["v"], local, a["start"], a["n"], a["rank"], a["world"],
                            a["slot"], 0, state, 1.0, 0, None)
        assert rc == code, (change, rc, L.last_error())
        assert L.launch_count_named("dp_exchange_chunk") == c0, change
    torch.cuda.synchronize()
    assert local.tolist() == [0, 0] and not sig.any()


# --------------------------------------------------------------------------------------------------------------------
# host arguments of the exchange (CPU)
# --------------------------------------------------------------------------------------------------------------------
MODELS = [("AppearanceFlowModel", {}), ("AppearanceFlowTinghui", {}), ("AppFlowHighDimAngle", {}), ("AppFlowLowDimAngle", {}),
          ("Base_Prediction_Model", {"viewpoint_dim": 2, "use_color": "", "use_depth": "", "depth_lr_factor": 0.1, "head": "flow"}),
          ("MultiObjectAppFlow", {"image_size": 64, "viewpoint_dim": 2, "use_color": "", "use_depth": 0.1, "combination_image": "",
                                  "gen_sep_images": "", "predict_target_masks": 0.1}),
          ("MultiViewFusionAppFlow", {"image_size": 64, "viewpoint_dim": 2, "num_views": 4, "use_depth": 0.1})]


@pytest.mark.parametrize("cls,extra", MODELS, ids=[m[0] for m in MODELS])
def test_exchange_arguments_tile_every_store(cls, extra):
    """For every model class's variable store at world 2, 4 and 8 and chunk sizes 128, 32 and 4 MB: every
    (start, n_slice, slot, replicated) meets the C ABI's preconditions (start % 4, n_slice % 8, 16-byte aligned slices),
    the owned slices tile [0, shard_end) without overlap, the tail stays inside [shard_end, alloc) and covers it, and
    slots are unique and below the slot count the exchange allocates."""
    import dynamic_multiview_3d_b200 as pkg
    from dynamic_multiview_3d_b200.data_parallel import exchange_args, plan_chunks
    conf = dict({"batch_size": 2, "learning_rate": 1e-4, "image_size": 224, "viewpoint_dim": 19}, **extra)
    st = getattr(pkg, cls)(conf, device="meta").store
    table = [(v.name, v.offset, -(-v.numel // 64) * 64) for v in st.vars.values() if v.offset < st.shard_end]
    live = {v.name for v in st.trainable_vars()}
    ragged = 0
    for world in (2, 4, 8):
        for mb in (128, 32, 4):
            chunks = plan_chunks(table, st.shard_end, int(mb * (1 << 20) / 4), world, live)[0]
            args = [exchange_args(chunks, c, world, st.shard_end, st.alloc) for c in list(range(len(chunks))) + [-1]]
            owned = []
            for start, n, slot, rep in args:
                assert start >= 0 and start % 4 == 0 and n > 0 and n % 8 == 0 and 0 <= slot <= len(chunks), (start, n, slot)
                if rep:
                    assert start == st.shard_end and start + n <= st.alloc and n >= st.alloc - st.shard_end, (start, n)
                else:
                    owned += [(start + r * n, start + (r + 1) * n) for r in range(world)]
                    ragged += world == 2 and n % 512 == 256
            assert len({a[2] for a in args}) == len(args) and args[-1][3] == 1 and sum(a[3] for a in args) == 1
            owned.sort()
            assert owned[0][0] == 0 and owned[-1][1] == st.shard_end and all(a[1] == b[0] for a, b in zip(owned, owned[1:]))
    if cls == "AppearanceFlowModel":
        assert ragged > 0, "the 224^2 store has world-2 chunks that end mid-block (n_slice = 256 mod 512)"

"""torch.autograd glue over the C ABI of libdmv3d.so.

PyTorch owns device memory, streams and the autograd tape; every computation here is one
call into libdmv3d with raw device pointers on the current CUDA stream.  Nothing falls back
to PyTorch or CPU arithmetic: a tensor that is not on a CUDA device raises.

Parameter gradients are NOT routed through autograd: the wgrad kernels write them straight
into the variable's slot of the flat gradient buffer (variables.py) and backward returns
None for parameters.  ``anchor`` is a dummy leaf that keeps the tape alive when the only
differentiable inputs are parameters (first layer on a network input).
"""
import ctypes as C

import torch

from . import _lib
from ._lib import ACT, ALGO, ALGO_PACK_ONLY, ALGO_PREPACKED, DT_BF16, DT_F32, DT_S2D, LOSS, SAMPLER_ADD_GRID, SAMPLER_GRID_XY
from ._lib import call as _real_call

_workspaces = {}
_default_algo = "auto"


def set_default_algo(name):
    """'auto' (tcgen05 where covered, else SIMT), 'simt', or 'tcgen05'."""
    global _default_algo
    if name not in ALGO:
        raise ValueError(name)
    _default_algo = name


def get_default_algo():
    return _default_algo


def _algo(a):
    return ALGO[_default_algo if a is None else a]


def _stream(t):
    if t.is_meta:
        return None
    return torch.cuda.current_stream(t.device).cuda_stream


def call(name, *args):
    """Launch through the C ABI.  Tensors on the ``meta`` device carry shapes only (used by the
    CPU host-logic tests to build a model's variable table without a GPU): their data
    pointers are 0 and nothing is launched -- and nothing is computed either."""
    if _meta_depth[0]:
        return
    if _profile[0] is None:
        _real_call(name, *args)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _real_call(name, *args)
    e1.record()
    _profile[0].append((name, _tag[0], e0, e1))


_profile = [None]
_tag = [""]


class profile_calls:
    """Context: time every C-ABI call with CUDA events on the current stream.
    ``records`` -> [(entry point, variable tag, milliseconds)] after exit."""

    def __enter__(self):
        self._raw = []
        _profile[0] = self._raw
        return self

    def __exit__(self, *a):
        _profile[0] = None
        torch.cuda.synchronize()
        self.records = [(n, t, e0.elapsed_time(e1)) for n, t, e0, e1 in self._raw]


_meta_depth = [0]


class meta_mode:
    """Context: shape inference only (inputs on the meta device)."""

    def __enter__(self):
        _meta_depth[0] += 1

    def __exit__(self, *a):
        _meta_depth[0] -= 1


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda and not t.is_meta:
            raise _lib.DmvError("tensor on %s: the path runs on CUDA only (no CPU fallback)" % t.device)


def _dt(t):
    if t.dtype == torch.bfloat16:
        return DT_BF16
    if t.dtype == torch.float32:
        return DT_F32
    raise TypeError("unsupported dtype %s" % t.dtype)


def _p(t):
    return None if (t is None or t.is_meta) else t.data_ptr()


# --- weight gradients on a side stream -----------------------------------------------------------------------
# dgrad is the critical chain of backward; every wgrad only needs (input, dPre) and can run next to it.  The side
# stream forks behind an event after dPre is ready and is joined before the optimizer (join_side_stream).  It has its
# own scratch buffer, and the tensors it reads are kept alive until the join (the caching allocator does not know that
# another stream still uses them).
_side = {}
_used = set()          # keys of _side whose stream took work in the current pass (only those are joined: a stream that
                       # was not forked inside a graph capture must not be waited on inside it)
_held = []
_join_queued = [False]


def side_stream_enabled():
    import os
    return os.environ.get("DMV_SIDE_WGRAD", "1") == "1" and not _meta_depth[0] and _profile[0] is None


def stream_priority(role):
    """CUDA stream priority of a role in the captured step (lower = dispatched first; kernel nodes of a graph inherit the
    priority of the stream they were captured on).  Default: the step's own chain -- forward, loss, the input-gradient chain
    of backward, the viewpoint branch -- one level above everything else (weight-gradient lanes, Adam / exchange streams).
    ``DMV_MAIN_PRIORITY`` / ``DMV_LANE0_PRIORITY`` / ``DMV_LANE1_PRIORITY`` = n set a role to level -n (0 = default
    priority).  MEASURED (profiles/r02_fc_variant_priority_sweep.txt): three levels (chain -2, convolution weight gradients
    -1, FC lane 0) cost 1 % with the persistent fused FC kernel (2.607 against 2.578 ms/step) -- that kernel occupies the
    shared memory of every SM whatever its priority; they only pay with the one-tile-per-CTA form of the kernel, which is
    slower overall (2.69 ms)."""
    import os
    default = {"main": -1}.get(role, 0)
    env = os.environ.get("DMV_%s_PRIORITY" % role.upper())
    return default if env is None else -abs(int(env))


class side_stream:
    """Context: run the enclosed launches on one of the device's side streams ("lanes"), ordered after everything
    enqueued so far on the current stream.  ``keep`` are tensors the side work reads.  Lane 0 carries the convolution
    weight gradients; lane 1 the weight gradients of the big FC matrices, so that they do not queue behind ~0.4 ms of
    decoder convolution gradients: their chunks are 97 % of the bytes of the data-parallel exchange / of Adam's
    traffic, and the earlier they are written the more of it hides behind the encoder's backward."""

    def __init__(self, device, *keep, lane=0):
        key = (device.type, device.index, lane)
        st = _side.get(key)
        if st is None:
            st = _side[key] = torch.cuda.Stream(device=device, priority=stream_priority("lane%d" % lane))
        self.stream, self.device, self.key = st, device, key
        _held.extend(t for t in keep if t is not None)

    def __enter__(self):
        main = torch.cuda.current_stream(self.device)
        if not _join_queued[0]:
            # join when this backward pass ends (engine callback, as DDP does): after loss.backward() returns, every
            # gradient is ordered on the stream that called it
            _join_queued[0] = True
            dev = self.device
            torch.autograd.Variable._execution_engine.queue_callback(lambda: _auto_join(dev, main))
        ev = torch.cuda.Event()
        ev.record(main)
        self.stream.wait_event(ev)
        _used.add(self.key)
        self.ctx = torch.cuda.stream(self.stream)
        self.ctx.__enter__()
        return self.stream

    def __exit__(self, *a):
        return self.ctx.__exit__(*a)


class branch:
    """Context: run an independent branch of the forward graph on its own stream, forked behind everything enqueued so
    far on the current stream; ``join(t)`` makes the current stream wait for it and hands the result over.

    The viewpoint FCs (three 64-wide linear layers on a [B, V] code) are single-CTA kernels: 26 us of pure latency in the
    forward pass and -- because autograd replays a node on the stream its forward ran on -- ~200 us of the critical chain
    in backward, where they sat between the a3 and fc1 input gradients with the rest of the GPU idle
    (profiles/r02_timeline_immediate.txt).  On a branch stream they run next to the encoder (forward) and next to fc1's
    backward.  The stream is joined with the weight-gradient lanes when backward ends (_auto_join)."""

    def __init__(self, device, *inputs):
        self.device = device
        self.on = side_stream_enabled() and device.type == "cuda"
        if self.on:
            key = (device.type, device.index, "branch")
            st = _side.get(key)
            if st is None:
                # same (high) priority as the captured main chain (train.py): the branch is a handful of tiny kernels, and at
                # the default priority they starved behind the chain's persistent grids until the chain itself blocked on them
                st = _side[key] = torch.cuda.Stream(device=device, priority=stream_priority("main"))
            self.stream, self.key = st, key
            for t in inputs:
                t.record_stream(st)

    def __enter__(self):
        if self.on:
            self.main = torch.cuda.current_stream(self.device)
            ev = torch.cuda.Event()
            ev.record(self.main)
            self.stream.wait_event(ev)
            _used.add(self.key)
            self.ctx = torch.cuda.stream(self.stream)
            self.ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.on:
            self.done = torch.cuda.Event()
            self.done.record(self.stream)
            return self.ctx.__exit__(*a)
        return False

    def join(self, t):
        if self.on:
            self.main.wait_event(self.done)
            t.record_stream(self.main)
        return t


def lane_events(device):
    """One event per side stream that took work in this pass, recorded now.  The weight-gradient lanes are not ordered against
    each other: whoever consumes gradients written on several lanes (a data-parallel chunk whose variables reported from
    different lanes) waits for all of them, not only for the lane that delivered the last one."""
    evs = []
    for key in _used:
        if (key[0], key[1]) == (device.type, device.index):
            ev = torch.cuda.Event()
            ev.record(_side[key])
            evs.append(ev)
    return evs


def reset_side_stream_state():
    """Start of a forward pass: forget a join that a failed backward pass left queued."""
    if _join_queued[0]:
        _join_queued[0] = False
        for key in list(_used):
            torch.cuda.current_stream(torch.device(key[0], key[1])).wait_stream(_side[key])
        del _held[:]
    _used.clear()


def _auto_join(device, main):
    _join_queued[0] = False
    for key in list(_used):
        if (key[0], key[1]) == (device.type, device.index):
            main.wait_stream(_side[key])
            _used.discard(key)
    del _held[:]


def side_workspace(nbytes, device, lane=0):
    key = ("side", device.type, device.index, lane)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


class _main_stream_ctx:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


BIG_LINEAR = 1 << 20      # weights; linear layers this large take side-stream lane 1
# Lane of the step's last weight gradients (e0, the viewpoint FCs): a third lane in single-process training, so that they
# do not queue behind e0_0's on lane 0 at the end of the step, where nothing else is left to overlap with.  Under data
# parallelism (data_parallel.attach) they stay on lane 0: that path was validated on 2 - 8 GPUs with two lanes.
TAIL_LANE = 2 if __import__("os").environ.get("DMV_TAIL_LANE", "1") == "1" else 0


def set_tail_lane(on):
    global TAIL_LANE
    TAIL_LANE = 2 if (on and __import__("os").environ.get("DMV_TAIL_LANE", "1") == "1") else 0


def _wgrad_ctx(device, *keep, lane=0):
    """(context manager, workspace function) for a weight-gradient launch."""
    if side_stream_enabled():
        import os
        if os.environ.get("DMV_FC_LANE", "1") != "1":
            lane = 0
        return side_stream(device, *keep, lane=lane), (lambda n, d, lane=lane: side_workspace(n, d, lane))
    return _main_stream_ctx(), workspace


def workspace(nbytes, device):
    """One growable scratch buffer per device AND stream: launches that share it are ordered on that stream (the
    forward / dgrad chain on the main stream, an independent branch of the graph on its own)."""
    # keyed by the ROLE of the current stream, not by the stream object: capture streams come and go (one per captured
    # graph) and a buffer per stream object would never be released
    br = _side.get((device.type, device.index, "branch")) if device.type == "cuda" else None
    role = "branch" if (br is not None and torch.cuda.current_stream(device) == br) else "main"
    key = (device.type, device.index, role) if _render_role[0] is None else (device.type, device.index, role, _render_role[0])
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


# --- rendering next to training ------------------------------------------------------------------------------------
# A captured train step holds the addresses of the workspaces and prepack buffers it was captured with.  A render at
# B x V samples needs larger workspaces; growing the training ones would free memory the graph still uses.  Inside
# render_scope every workspace is keyed by the scope's role as well, prepacking is off (the layers pack inline) and the
# FC matrices keep the row count of the training pass (optimizer.fusable reads it).
_render_role = [None]


class render_scope:
    """Context: launches of an inference pass that must leave every training buffer alone.  ``role`` names the set of
    workspaces it uses: a captured render graph takes its own so that a later render of another size cannot move them."""

    def __init__(self, role="render"):
        self.role = role

    def __enter__(self):
        self.prev = _render_role[0]
        _render_role[0] = self.role

    def __exit__(self, *a):
        _render_role[0] = self.prev


def rendering():
    return _render_role[0] is not None


# --- weight packing off the critical chain ------------------------------------------------------------------------
# Several tensor-core forms read the bf16 weights in a packed layout written by a small kernel in front of the layer
# (include/dmv3d.h: DMV_ALGO_PACK_ONLY / DMV_ALGO_PREPACKED): ~20 launches of 2-8 us per step that sat on the forward /
# input-gradient chain (profiles/r02_timeline_immediate.txt).  A layer registers its packing call the first time it runs;
# from then on the train step replays all of them on a side stream at its start (the weights are final by then: Adam ran at
# the end of the previous step) into per-layer buffers, and the layer waits for its event and skips the packing kernel.
class Prepack(object):
    def __init__(self, store):
        self.store = store
        self.entries = {}          # key -> [pack_call(ws, flags, stream), buffer, event or None]
        self.live = False
        self.stream = None

    @staticmethod
    def enabled(store):
        import os
        return (store.device.type == "cuda" and os.environ.get("DMV_PREPACK", "1") == "1" and not _meta_depth[0] and _profile[0] is None
                and _render_role[0] is None)

    def register(self, key, nbytes, pack_call):
        if key not in self.entries:
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.store.device)
            self.entries[key] = [pack_call, buf, None]

    def begin(self):
        """Start of a train step: pack every registered layer's weights on the side stream."""
        if not self.entries:
            return
        dev = self.store.device
        if self.stream is None:
            self.stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        ev = torch.cuda.Event()
        ev.record(main)
        self.stream.wait_event(ev)
        with torch.cuda.stream(self.stream):
            for e in self.entries.values():
                e[0](e[1], ALGO_PACK_ONLY, self.stream.cuda_stream)
                e[2] = torch.cuda.Event()
                e[2].record(self.stream)
        self.live = True

    def take(self, key):
        """(buffer, PREPACKED flag) if this step packed ``key`` -- the current stream then waits for it -- else None."""
        if not self.live:
            return None
        e = self.entries.get(key)
        if e is None or e[2] is None:
            return None
        torch.cuda.current_stream(self.store.device).wait_event(e[2])
        return e[1]

    def end(self):
        if self.live:
            self.live = False
            torch.cuda.current_stream(self.store.device).wait_stream(self.stream)
            for e in self.entries.values():
                e[2] = None


def _prepack_of(store):
    pp = getattr(store, "prepack", None)
    if pp is None and Prepack.enabled(store):
        pp = store.prepack = Prepack(store)
    return pp if (pp is not None and Prepack.enabled(store)) else None


def same_out(n, s):
    return -(-n // s)


def _anchor_for(t):
    a = torch.zeros(1, device=t.device, requires_grad=True)
    return a


# --- activation-derivative fusion between consecutive layers ----------------------------------------------------
# Backward of a hidden layer L needs dPre_L = dY_L * act'(Y_L).  dY_L is the input gradient dX of the layer(s) that
# consume Y_L, and Y_L is exactly their saved input -- so the consumer's dgrad kernel applies act'(its own input) in its
# epilogue and hands back dPre_L directly (include/dmv3d.h, y_in / act_in); the producer then skips its elementwise
# pass and only sums the bias gradient (on the weight-gradient side stream).  The hand-shake is a cell attached to the
# producer's output tensor: a consuming layer that will fuse marks it in its forward; the producer reads it in its
# backward.  Tensors that pass through torch ops (cat, chunk, slicing) carry no cell: both sides fall back to the
# separate pass.  ``reshape`` below keeps the cell across a view.  A tagged tensor must not be fed to a fusing layer AND
# used by a torch op directly (no graph of this package does).
# MEASURED (round 2, profiles/r02_dact_fusion.txt): with the present kernels the fusion LOSES -- the tensor-core kernels of
# the wide layers are bound by their four epilogue warps, and the extra 2 B/element read there costs more (e1 dgrad
# 29 -> 83 us, d1 dgrad 40 -> 75 us, flow head 59 -> 86 us; step 2.91 -> 3.22 ms) than the HBM-rate elementwise pass it
# removes (6 B/element at 5.9 TB/s).  It is therefore OFF by default (DMV_FUSE_DACT=1 turns the hand-shake on, and the
# library must be built with -DDMV_DACT_EPILOGUE=1 for the fused epilogues -- otherwise the entry points apply the factor
# with the elementwise pass themselves, same results); the C ABI keeps the capability and its tests.  The remedy is a
# producer-warp TMA load of the Y tile, not more epilogue loads.
class _ActCell(object):
    __slots__ = ("act", "fused")

    def __init__(self, act):
        self.act, self.fused = act, False


def fuse_dact_enabled():
    import os
    return os.environ.get("DMV_FUSE_DACT", "0") == "1" and not _meta_depth[0]


def _out_cell(act, out_dtype):
    return _ActCell(act) if (act in ("lrelu", "relu") and out_dtype == torch.bfloat16 and fuse_dact_enabled()) else None


def _claim_input(x):
    """Consumer side, in forward: returns the producer's cell if this layer's dgrad will apply act'(x)."""
    cell = getattr(x, "_dmv_cell", None)
    if cell is None or not x.requires_grad or not torch.is_grad_enabled() or x.dtype != torch.bfloat16 or not x.is_contiguous():
        return None
    cell.fused = True
    return cell


def reshape(y, shape):
    """y.reshape(shape) that keeps the activation cell when the result is a view of the same storage."""
    r = y.reshape(shape)
    cell = getattr(y, "_dmv_cell", None)
    if cell is not None and r.data_ptr() == y.data_ptr() and r.is_contiguous():
        r._dmv_cell = cell
    return r


# ----------------------------------------------------------------------------- conv / deconv / linear
class _Conv2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, x, wvar, bvar, stride, act, algo, out_dtype, in_cell, out_cell):
        _need_cuda(x)
        x = x.contiguous()
        B, H, W, Cin = x.shape
        kh, kw, wcin, Cout = wvar.shape
        assert wcin == Cin, (wvar.name, wvar.shape, x.shape)
        y = torch.empty((B, same_out(H, stride), same_out(W, stride), Cout), dtype=out_dtype, device=x.device)
        _tag[0] = wvar.name
        need = _lib.load().dmv_conv_workspace_size(B, H, W, Cin, Cout, kh, kw, stride)
        ws = workspace(need, x.device)
        # thin stride-2 layer (e0): build the space-to-depth tensor once and keep it for the weight gradient
        xs, xs_dt = x, _dt(x)
        n2 = _lib.load().dmv_thin_s2d_size(B, H, W, Cin, Cout, kh, kw, stride) if (Cin < 8 and algo != ALGO["simt"] and not _meta_depth[0]) else 0
        if n2:
            xs = torch.empty(n2, dtype=torch.uint8, device=x.device)
            call("dmv_thin_s2d_prep", _p(x), _dt(x), _p(xs), B, H, W, Cin, _stream(x))
            xs_dt = DT_S2D
        pp = _prepack_of(wvar.store) if (Cin >= 8 and xs_dt == DT_BF16) else None
        flags = 0
        if pp is not None:
            key, ydt, a = (wvar.name, "fwd"), _dt(y), ACT[act]
            pre = pp.take(key)
            if pre is not None:
                ws, flags = pre, ALGO_PREPACKED
            else:                  # (pointers are read at packing time: data_parallel.attach may re-home the bf16 buffer)
                pp.register(key, need, lambda buf, fl, s_: call(
                    "dmv_conv2d_fwd", buf.data_ptr(), DT_BF16, wvar.half.data_ptr(), None, buf.data_ptr(), ydt, B, H, W, Cin, Cout, kh, kw, stride, a,
                    buf.data_ptr(), buf.numel(), algo | fl, s_))
        call("dmv_conv2d_fwd", _p(xs), xs_dt, _p(wvar.half), _p(bvar.master) if bvar is not None else None, _p(y), _dt(y),
             B, H, W, Cin, Cout, kh, kw, stride, ACT[act], _p(ws), ws.numel(), algo | flags, _stream(x))
        ctx.save_for_backward(x if ctx.needs_input_grad[1] or not n2 else xs, y, xs)
        ctx.xshape, ctx.xdtype, ctx.xs_dt = tuple(x.shape), x.dtype, xs_dt
        ctx.cfg = (wvar, bvar, stride, act, algo)
        ctx.cells = (in_cell, out_cell)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y, xs = ctx.saved_tensors
        wvar, bvar, stride, act, algo = ctx.cfg
        B, H, W, Cin = ctx.xshape
        kh, kw, _, Cout = wvar.shape
        st = _stream(y)
        _tag[0] = wvar.name
        dy = dy.contiguous()
        bias_done = False
        in_cell, out_cell = ctx.cells
        if out_cell is not None and out_cell.fused and dy.dtype == torch.bfloat16:
            dpre = dy                          # the consumer's dgrad epilogue already applied act'(y)
        elif bvar is not None and ACT[act] and y.dtype == torch.bfloat16 and dy.dtype == torch.bfloat16 and Cout % 8 == 0:
            dpre = torch.empty_like(y)
            rows = y.numel() // Cout
            ws = workspace(_lib.load().dmv_act_bwd_bias_workspace_size(rows, Cout), x.device)
            call("dmv_act_bwd_bias", _p(dy), _p(y), _p(dpre), _p(bvar.grad), rows, Cout, ACT[act], _p(ws), ws.numel(), st)
            bias_done = True
        elif dy.dtype != torch.bfloat16 or ACT[act]:
            dpre = torch.empty(y.shape, dtype=y.dtype, device=y.device)
            call("dmv_act_bwd", _p(dy), _p(y), _p(dpre), _dt(y), y.numel(), ACT[act], st)
            if dpre.dtype != torch.bfloat16:
                h = torch.empty(y.shape, dtype=torch.bfloat16, device=y.device)
                call("dmv_cast_f32_to_bf16", _p(dpre), _p(h), h.numel(), st)
                dpre = h
        else:
            dpre = dy
        dx = None
        if ctx.needs_input_grad[1]:
            dx = torch.empty(ctx.xshape, dtype=torch.bfloat16, device=y.device)
            need = _lib.load().dmv_conv_workspace_size(B, H, W, Cin, Cout, kh, kw, stride)
            ws = workspace(need, y.device)
            pp = _prepack_of(wvar.store) if in_cell is None else None
            flags = 0
            if pp is not None:
                key = (wvar.name, "dgrad")
                pre = pp.take(key)
                if pre is not None:
                    ws, flags = pre, ALGO_PREPACKED
                else:
                    pp.register(key, need, lambda buf, fl, s_: call(
                        "dmv_conv2d_dgrad", buf.data_ptr(), wvar.half.data_ptr(), buf.data_ptr(), None, 0, B, H, W, Cin, Cout, kh, kw, stride,
                        buf.data_ptr(), buf.numel(), algo | fl, s_))
            call("dmv_conv2d_dgrad", _p(dpre), _p(wvar.half), _p(dx), _p(x) if in_cell is not None else None,
                 ACT[in_cell.act] if in_cell is not None else 0, B, H, W, Cin, Cout, kh, kw, stride, _p(ws), ws.numel(), algo | flags, st)
            if ctx.xdtype != torch.bfloat16:
                dxf = torch.empty(ctx.xshape, dtype=ctx.xdtype, device=y.device)
                call("dmv_cast_bf16_to_f32", _p(dx), _p(dxf), dx.numel(), st)
                dx = dxf
        nws = _lib.load().dmv_wgrad_workspace_size(B, H, W, Cin, Cout, kh, kw, stride)
        # the LAST weight gradient of the step (e0: the 3-channel image layer) does not queue behind e0_0's on lane 0: the two
        # run side by side at the end of backward, where nothing else is left to overlap with
        wctx, wsf = _wgrad_ctx(y.device, xs, dpre, lane=TAIL_LANE if Cin <= 4 else 0)
        with wctx:
            ws = wsf(nws, y.device)
            call("dmv_conv2d_wgrad", _p(xs), ctx.xs_dt, _p(dpre), _p(wvar.grad), _p(bvar.grad) if (bvar is not None and not bias_done) else None,
                 B, H, W, Cin, Cout, kh, kw, stride, _p(ws), ws.numel(), algo, _stream(y))
            store = wvar.store
            if bvar is not None:
                store.notify_grad(bvar)
            store.notify_grad(wvar)
        return None, dx, None, None, None, None, None, None, None, None


class _Deconv2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, x, wvar, out_hw, stride, act, algo, out_dtype, in_cell, out_cell):
        _need_cuda(x)
        x = x.contiguous()
        if x.dtype != torch.bfloat16:
            raise TypeError("deconv input must be bf16")
        B, Hin, Win, Cin = x.shape
        kh, kw, Cout, wcin = wvar.shape
        assert wcin == Cin, (wvar.name, wvar.shape, x.shape)
        Ho, Wo = out_hw
        assert same_out(Ho, stride) == Hin and same_out(Wo, stride) == Win, "output_shape inconsistent with input"
        y = torch.empty((B, Ho, Wo, Cout), dtype=out_dtype, device=x.device)
        _tag[0] = wvar.name
        need = _lib.load().dmv_conv_workspace_size(B, Ho, Wo, Cout, Cin, kh, kw, stride)
        ws = workspace(need, x.device)
        pp = _prepack_of(wvar.store) if Cout >= 8 else None
        flags = 0
        if pp is not None:
            key, ydt, a = (wvar.name, "fwd"), _dt(y), ACT[act]
            pre = pp.take(key)
            if pre is not None:
                ws, flags = pre, ALGO_PREPACKED
            else:
                pp.register(key, need, lambda buf, fl, s_: call(
                    "dmv_deconv2d_fwd", buf.data_ptr(), wvar.half.data_ptr(), buf.data_ptr(), ydt, B, Ho, Wo, Cin, Cout, kh, kw, stride, a, buf.data_ptr(),
                    buf.numel(), algo | fl, s_))
        call("dmv_deconv2d_fwd", _p(x), _p(wvar.half), _p(y), _dt(y), B, Ho, Wo, Cin, Cout, kh, kw, stride, ACT[act], _p(ws),
             ws.numel(), algo | flags, _stream(x))
        ctx.save_for_backward(x, y)
        ctx.cfg = (wvar, stride, act, algo)
        ctx.cells = (in_cell, out_cell)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y = ctx.saved_tensors
        wvar, stride, act, algo = ctx.cfg
        B, Ho, Wo, Cout = y.shape
        kh, kw, _, Cin = wvar.shape
        st = _stream(x)
        _tag[0] = wvar.name
        dy = dy.contiguous()
        in_cell, out_cell = ctx.cells
        if out_cell is not None and out_cell.fused and dy.dtype == torch.bfloat16:
            dpre = dy
        elif ACT[act]:
            dpre = torch.empty(y.shape, dtype=y.dtype, device=y.device)
            call("dmv_act_bwd", _p(dy), _p(y), _p(dpre), _dt(y), y.numel(), ACT[act], st)
        else:
            dpre = dy
        dx = None
        # thin stride-2 head (flow field): one space-to-depth pass of the gradient serves dgrad and wgrad
        dps, dps_dt = dpre, _dt(dpre)
        n2 = _lib.load().dmv_thin_s2d_size(B, Ho, Wo, Cout, Cin, kh, kw, stride) if (Cout < 8 and algo != ALGO["simt"] and not _meta_depth[0]) else 0
        if n2:
            dps = torch.empty(n2, dtype=torch.uint8, device=x.device)
            call("dmv_thin_s2d_prep", _p(dpre), _dt(dpre), _p(dps), B, Ho, Wo, Cout, st)
            dps_dt = DT_S2D
        if ctx.needs_input_grad[1]:
            dx = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
            need = _lib.load().dmv_conv_workspace_size(B, Ho, Wo, Cout, Cin, kh, kw, stride)
            ws = workspace(need, x.device)
            pp = _prepack_of(wvar.store) if (in_cell is None and Cout >= 8 and dps_dt == DT_BF16) else None
            flags = 0
            if pp is not None:
                key = (wvar.name, "dgrad")
                pre = pp.take(key)
                if pre is not None:
                    ws, flags = pre, ALGO_PREPACKED
                else:
                    pp.register(key, need, lambda buf, fl, s_: call(
                        "dmv_deconv2d_dgrad", buf.data_ptr(), DT_BF16, wvar.half.data_ptr(), buf.data_ptr(), None, 0, B, Ho, Wo, Cin, Cout, kh, kw, stride,
                        buf.data_ptr(), buf.numel(), algo | fl, s_))
            call("dmv_deconv2d_dgrad", _p(dps), dps_dt, _p(wvar.half), _p(dx), _p(x) if in_cell is not None else None,
                 ACT[in_cell.act] if in_cell is not None else 0, B, Ho, Wo, Cin, Cout, kh, kw, stride, _p(ws), ws.numel(), algo | flags, st)
        nws = _lib.load().dmv_wgrad_workspace_size(B, Ho, Wo, Cout, Cin, kh, kw, stride)
        wctx, wsf = _wgrad_ctx(x.device, x, dps)
        with wctx:
            ws = wsf(nws, x.device)
            call("dmv_deconv2d_wgrad", _p(x), _p(dps), dps_dt, _p(wvar.grad), B, Ho, Wo, Cin, Cout, kh, kw, stride, _p(ws),
                 ws.numel(), algo, _stream(x))
            wvar.store.notify_grad(wvar)
        return None, dx, None, None, None, None, None, None, None, None


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, x, wvar, bvar, act, algo, in_cell, out_cell, group):
        _need_cuda(x)
        x = x.contiguous()
        if x.dtype != torch.bfloat16:
            raise TypeError("linear input must be bf16")
        M, K = x.shape
        wk, N = wvar.shape
        assert wk == K, (wvar.name, wvar.shape, x.shape)
        y = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
        _tag[0] = wvar.name
        if _render_role[0] is None:
            wvar.rows = M
        if wvar.store.pre_use_hook is not None and _render_role[0] is None:   # a render flushes pending updates first
            wvar.store.pre_use_hook(wvar)        # a deferred optimizer update of this matrix must have landed
        ws = workspace(_lib.load().dmv_conv_workspace_size(M, 1, 1, K, N, 1, 1, 1), x.device)
        call("dmv_linear_fwd", _p(x), _p(wvar.half), _p(bvar.master) if bvar is not None else None, _p(y), M, K, N, ACT[act],
             _p(ws), ws.numel(), algo, _stream(x))
        ctx.save_for_backward(x, y)
        ctx.cfg = (wvar, bvar, act, algo)
        ctx.cells = (in_cell, out_cell)
        ctx.group = group
        if group > 1:              # every row consumed ``group`` times: the consumer sees the rows repeated
            return y.repeat_interleave(group, dim=0)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, y = ctx.saved_tensors
        wvar, bvar, act, algo = ctx.cfg
        M, K = x.shape
        N = wvar.shape[1]
        st = _stream(x)
        _tag[0] = wvar.name
        dy = dy.contiguous() if ctx.group == 1 else _row_pitched(dy, N)
        bias_done = False
        in_cell, out_cell = ctx.cells
        if ctx.group > 1:
            # the sum over the ``group`` uses of each row, act' and the bias gradient in one pass; dy may be the slice of a
            # concat's gradient (row pitch > N)
            dpre = torch.empty_like(y)
            ws = workspace(_lib.load().dmv_act_bwd_bias_workspace_size(M, N), x.device)
            call("dmv_act_bwd_bias_grouped", _p(dy), dy.stride(0), ctx.group, _p(y), _p(dpre), _p(bvar.grad), M, N, ACT[act], _p(ws),
                 ws.numel(), st)
            bias_done = True
        elif out_cell is not None and out_cell.fused:
            dpre = dy
        elif bvar is not None and ACT[act] and N % 8 == 0:
            dpre = torch.empty_like(y)
            ws = workspace(_lib.load().dmv_act_bwd_bias_workspace_size(M, N), x.device)
            call("dmv_act_bwd_bias", _p(dy), _p(y), _p(dpre), _p(bvar.grad), M, N, ACT[act], _p(ws), ws.numel(), st)
            bias_done = True
        elif ACT[act]:
            dpre = torch.empty_like(y)
            call("dmv_act_bwd", _p(dy), _p(y), _p(dpre), DT_BF16, y.numel(), ACT[act], st)
        else:
            dpre = dy
        dx = None
        if ctx.needs_input_grad[1]:
            dx = torch.empty_like(x)
            ws = workspace(_lib.load().dmv_conv_workspace_size(M, 1, 1, K, N, 1, 1, 1), x.device)
            call("dmv_linear_dgrad", _p(dpre), _p(wvar.half), _p(dx), _p(x) if in_cell is not None else None,
                 ACT[in_cell.act] if in_cell is not None else 0, M, K, N, _p(ws), ws.numel(), algo, st)
        nws = _lib.load().dmv_wgrad_workspace_size(M, 1, 1, K, N, 1, 1, 1)
        # small matrices (the viewpoint FCs): autograd runs their nodes last, so on lane 0 their few-microsecond kernels would
        # sit behind every convolution weight gradient, at the very end of the step
        wctx, wsf = _wgrad_ctx(x.device, x, dpre, lane=1 if K * N >= BIG_LINEAR else TAIL_LANE)
        live = wvar.store.adam_live if wvar.fused_adam else None
        with wctx:
            ws = wsf(nws, x.device)
            if live is not None:
                # single-process training: Adam consumes the weight-gradient tile in registers (optimizer.py); the gradient
                # of this matrix is never written.  Ordered after the dgrad above, which reads the bf16 weights it rewrites.
                if bvar is not None and not bias_done:        # bias gradient alone: column sums of dPre (act' == 1, in place)
                    bws = wsf(_lib.load().dmv_act_bwd_bias_workspace_size(M, N), x.device)
                    call("dmv_act_bwd_bias", _p(dpre), _p(dpre), _p(dpre), _p(bvar.grad), M, N, 0, _p(bws), bws.numel(), _stream(x))
                call("dmv_linear_wgrad_adam", _p(x), _p(dpre), _p(wvar.master), _p(wvar.m), _p(wvar.v), _p(wvar.half), None, M, K, N,
                     live.state.data_ptr(), live.beta1, live.beta2, live.eps, live.grad_scale, _stream(x))
                if bvar is not None:
                    wvar.store.notify_grad(bvar)
            else:
                call("dmv_linear_wgrad", _p(x), _p(dpre), _p(wvar.grad), _p(bvar.grad) if (bvar is not None and not bias_done) else None, M, K, N,
                     _p(ws), ws.numel(), algo, _stream(x))
                if bvar is not None:
                    wvar.store.notify_grad(bvar)
                wvar.store.notify_grad(wvar)
        return None, dx, None, None, None, None, None, None, None


def _row_pitched(dy, N):
    """dy [R, N] as dmv_act_bwd_bias_grouped reads it: unit column stride, a row pitch >= N that keeps rows 16-byte aligned.
    A column slice of a wider gradient qualifies as it is; anything else is copied."""
    if dy.stride(1) == 1 and dy.stride(0) >= N and dy.stride(0) % 8 == 0 and dy.data_ptr() % 16 == 0:
        return dy
    return dy.contiguous()


def _tagged(y, cell):
    if cell is not None:
        y._dmv_cell = cell
    return y


def conv2d(x, wvar, bvar, stride, act=None, algo=None, out_dtype=torch.bfloat16):
    cell = _out_cell(act, out_dtype)
    return _tagged(_Conv2d.apply(wvar.store.anchor, x, wvar, bvar, int(stride), act, _algo(algo), out_dtype, _claim_input(x), cell), cell)


def deconv2d(x, wvar, out_hw, stride, act=None, algo=None, out_dtype=torch.bfloat16):
    cell = _out_cell(act, out_dtype)
    return _tagged(_Deconv2d.apply(wvar.store.anchor, x, wvar, (int(out_hw[0]), int(out_hw[1])), int(stride), act, _algo(algo), out_dtype,
                                   _claim_input(x), cell), cell)


def linear(x, wvar, bvar, act=None, algo=None, group=1):
    """x @ W + b with ``act``.  group > 1: the layer runs once on x [rows, K] and returns [rows * group, N], each row
    repeated ``group`` times (one source feeding ``group`` targets); backward sums the uses of each row in the bias /
    activation-gradient pass (dmv_act_bwd_bias_grouped) and runs dgrad / wgrad at the layer's own rows."""
    group = int(group)
    if group == 1:
        cell = _out_cell(act, torch.bfloat16)
        return _tagged(_Linear.apply(wvar.store.anchor, x, wvar, bvar, act, _algo(algo), _claim_input(x), cell, 1), cell)
    if group < 1:
        raise ValueError("group must be >= 1, got %d" % group)
    if bvar is None or not ACT[act] or wvar.shape[1] % 8:
        raise ValueError("linear(group=%d) needs a bias, an activation and N %% 8 == 0 (%s: act %s, N %d)"
                         % (group, wvar.name, act, wvar.shape[1]))
    return _Linear.apply(wvar.store.anchor, x, wvar, bvar, act, _algo(algo), None, None, group)


# ----------------------------------------------------------------------------- activations
class _Act(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, act):
        _need_cuda(x)
        x = x.contiguous()
        y = torch.empty_like(x)
        call("dmv_act_fwd", _p(x), _p(y), _dt(x), x.numel(), ACT[act], _stream(x))
        ctx.save_for_backward(y)
        ctx.act = act
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(y)
        call("dmv_act_bwd", _p(dy), _p(y), _p(dx), _dt(y), y.numel(), ACT[ctx.act], _stream(y))
        return dx, None


def activation(x, act):
    return _Act.apply(x, act)


# ----------------------------------------------------------------------------- sampler
class _Resampler(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data, wf, flags):
        _need_cuda(data, wf)
        if data.dtype != torch.float32 or wf.dtype != torch.float32:
            raise TypeError("resampler runs in float32 (reference precision)")
        data = data.contiguous()
        wf = wf.contiguous()
        B, H, W, Cc = data.shape
        assert wf.shape[0] == B and wf.shape[-1] == 2
        out_shape = tuple(wf.shape[:-1]) + (Cc,)
        if wf.dim() == 4:
            Ho, Wo = wf.shape[1], wf.shape[2]
        else:                                   # [B, N, 2] sample lists
            Ho, Wo = 1, int(wf.numel() // (2 * B))
        out = torch.empty(out_shape, dtype=torch.float32, device=data.device)
        _tag[0] = "sampler"
        call("dmv_sampler_fwd", _p(data), _p(wf), _p(out), None, None, B, H, W, Cc, Ho, Wo, flags, _stream(data))
        ctx.save_for_backward(data, wf)
        ctx.geom = (B, H, W, Cc, Ho, Wo, flags)
        return out

    @staticmethod
    def backward(ctx, go):
        data, wf = ctx.saved_tensors
        B, H, W, Cc, Ho, Wo, flags = ctx.geom
        go = go.contiguous()
        need_d, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gd = torch.empty_like(data) if need_d else None
        gw = torch.empty_like(wf) if need_w else None
        if not (need_d or need_w):
            return None, None, None
        nws = _lib.load().dmv_sampler_bwd_workspace_size(B, H, W, Cc, Ho, Wo)
        ws = workspace(nws, data.device)
        _tag[0] = "sampler"
        call("dmv_sampler_bwd", _p(data), _p(wf), _p(go), _p(gd), _p(gw), B, H, W, Cc, Ho, Wo, flags, _p(ws), ws.numel(),
             _stream(data))
        return gd, gw, None


def resampler(data, warp):
    """tf.contrib.resampler.resampler(data[B,H,W,C], warp[B,...,2]); warp[...,0] = x, [...,1] = y."""
    return _Resampler.apply(data, warp, 0)


def flow_resampler(data, flow, grid_order="ref_yx"):
    """resample_layer(src, warp_pts_layer(flow)) with the grid formed inside the kernel."""
    flags = SAMPLER_ADD_GRID | (SAMPLER_GRID_XY if grid_order == "xy" else 0)
    if grid_order not in ("ref_yx", "xy"):
        raise ValueError(grid_order)
    return _Resampler.apply(data, flow, flags)


def flow_resampler_shared(data, flow, group, grid_order="ref_yx"):
    """flow_resampler with each source shared by ``group`` consecutive flows: data [B_src,H,W,C], flow [B_src*group,Ho,Wo,2]
    -> [B_src*group,Ho,Wo,C], output sample n warping data[n // group].  One launch (dmv_sampler_fwd_shared_src), no copy of
    the sources.  Forward only: it raises where autograd would need a gradient through it."""
    if grid_order not in ("ref_yx", "xy"):
        raise ValueError(grid_order)
    _need_cuda(data, flow)
    if torch.is_grad_enabled() and (data.requires_grad or flow.requires_grad):
        raise RuntimeError("flow_resampler_shared has no backward: call it under torch.no_grad() or on tensors that need no gradient")
    if data.dtype != torch.float32 or flow.dtype != torch.float32:
        raise TypeError("resampler runs in float32 (reference precision)")
    if data.dim() != 4 or flow.dim() != 4 or flow.shape[-1] != 2:
        raise ValueError("data [B_src,H,W,C] and flow [B_src*group,Ho,Wo,2] expected, got %s and %s" % (tuple(data.shape), tuple(flow.shape)))
    group = int(group)
    B_src, H, W, Cc = data.shape
    if flow.shape[0] != B_src * group:
        raise ValueError("flow holds %d samples, not B_src * group = %d * %d" % (flow.shape[0], B_src, group))
    data, flow = data.contiguous(), flow.contiguous()
    Ho, Wo = flow.shape[1], flow.shape[2]
    out = torch.empty((flow.shape[0], Ho, Wo, Cc), dtype=torch.float32, device=data.device)
    flags = SAMPLER_ADD_GRID | (SAMPLER_GRID_XY if grid_order == "xy" else 0)
    _tag[0] = "sampler"
    call("dmv_sampler_fwd_shared_src", _p(data), B_src, group, _p(flow), _p(out), H, W, Cc, Ho, Wo, flags, _stream(data))
    return out


class _GroupedResampler(torch.autograd.Function):
    """flow -> warped sources, output sample n reading data[n // group]; the gradient wrt the flow only."""

    @staticmethod
    def forward(ctx, data, flow, group, flags):
        B_src, H, W, Cc = data.shape
        Ho, Wo = flow.shape[1], flow.shape[2]
        out = torch.empty((flow.shape[0], Ho, Wo, Cc), dtype=torch.float32, device=data.device)
        _tag[0] = "sampler"
        call("dmv_sampler_fwd_shared_src", _p(data), B_src, group, _p(flow), _p(out), H, W, Cc, Ho, Wo, flags, _stream(data))
        ctx.save_for_backward(data, flow)
        ctx.geom = (B_src, group, H, W, Cc, Ho, Wo, flags)
        return out

    @staticmethod
    def backward(ctx, go):
        data, flow = ctx.saved_tensors
        B_src, group, H, W, Cc, Ho, Wo, flags = ctx.geom
        go = go.contiguous()
        gw = torch.empty_like(flow)
        _tag[0] = "sampler"
        call("dmv_sampler_grad_flow_shared_src", _p(data), B_src, group, _p(flow), _p(go), _p(gw), H, W, Cc, Ho, Wo, flags, _stream(data))
        return None, gw, None, None


def flow_resampler_grouped(data, flow, group, grid_order="ref_yx"):
    """Differentiable flow_resampler with each source shared by ``group`` consecutive flows (training on several targets of
    one source): data [B_src,H,W,C], flow [B_src*group,Ho,Wo,2] -> [B_src*group,Ho,Wo,C], output sample n warping
    data[n // group].  Backward gives the flow gradient (dmv_sampler_grad_flow_shared_src); the source is a network input
    and gets none: it raises if ``data`` needs a gradient."""
    if grid_order not in ("ref_yx", "xy"):
        raise ValueError(grid_order)
    _need_cuda(data, flow)
    if torch.is_grad_enabled() and data.requires_grad:
        raise RuntimeError("flow_resampler_grouped has no gradient wrt the source: pass a source that needs no gradient")
    if data.dtype != torch.float32 or flow.dtype != torch.float32:
        raise TypeError("resampler runs in float32 (reference precision)")
    if data.dim() != 4 or flow.dim() != 4 or flow.shape[-1] != 2:
        raise ValueError("data [B_src,H,W,C] and flow [B_src*group,Ho,Wo,2] expected, got %s and %s" % (tuple(data.shape), tuple(flow.shape)))
    group = int(group)
    if group < 1 or flow.shape[0] != data.shape[0] * group:
        raise ValueError("flow holds %d samples, not B_src * group = %d * %d" % (flow.shape[0], data.shape[0], group))
    flags = SAMPLER_ADD_GRID | (SAMPLER_GRID_XY if grid_order == "xy" else 0)
    return _GroupedResampler.apply(data.contiguous(), flow.contiguous(), group, flags)


_loss_wss = {}


class _WarpLoss(torch.autograd.Function):
    """flow -> (loss, gen): resample_layer(src, warp_pts_layer(flow)), the reconstruction loss against the target and
    d loss / d flow in one kernel (dmv_sampler_loss_fused).  The source and the target are network inputs."""

    @staticmethod
    def forward(ctx, data, flow, target, flags, weights, mode, inv_count, unit_upstream, group):
        _need_cuda(data, flow, target)
        data, flow, target = data.contiguous(), flow.contiguous(), target.contiguous()
        B_src, H, W, Cc = data.shape
        B = flow.shape[0]
        Ho, Wo = flow.shape[1], flow.shape[2]
        gen = torch.empty((B, Ho, Wo, Cc), dtype=torch.float32, device=data.device)
        gflow = torch.empty_like(flow)
        loss = torch.empty((), dtype=torch.float32, device=data.device)
        w = (C.c_float * Cc)(*[float(x) for x in weights])
        nws = _lib.load().dmv_sampler_loss_workspace_size(B, Ho, Wo)
        key = ("warp_loss", data.device.type, data.device.index)
        ws = _loss_wss.get(key)
        if ws is None or ws.numel() < nws:             # zeroed once: holds a self-resetting counter
            ws = _loss_wss[key] = torch.zeros(int(nws), dtype=torch.uint8, device=data.device)
        _tag[0] = "warp_loss"
        if group == 1:
            call("dmv_sampler_loss_fused", _p(data), _p(flow), _p(target), w, LOSS[mode], float(inv_count), _p(gen), _p(gflow), _p(loss),
                 B, H, W, Cc, Ho, Wo, flags, _p(ws), ws.numel(), _stream(data))
        else:
            call("dmv_sampler_loss_fused_shared_src", _p(data), B_src, group, _p(flow), _p(target), w, LOSS[mode], float(inv_count), _p(gen),
                 _p(gflow), _p(loss), H, W, Cc, Ho, Wo, flags, _p(ws), ws.numel(), _stream(data))
        ctx.gflow, ctx.unit_upstream = gflow, unit_upstream
        ctx.mark_non_differentiable(gen)
        return loss, gen

    @staticmethod
    def backward(ctx, gloss, _ggen):
        gflow = ctx.gflow
        if not ctx.unit_upstream:
            _tag[0] = "warp_loss"
            call("dmv_scale_by_device_scalar", _p(gflow), _p(gloss.contiguous().to(torch.float32)), gflow.numel(), _stream(gflow))
        return None, gflow, None, None, None, None, None, None, None


def _passed_aligned16(t):
    """The buffer a call passes for ``t`` (``t.contiguous()``) starts on a 16-byte boundary: a contiguous tensor is passed
    as it is, possibly at an offset into its storage; any other is copied into a fresh allocation."""
    return not t.is_contiguous() or t.data_ptr() % 16 == 0


def warp_loss_supported(data, flow, target=None, mode="l2"):
    """True exactly when dmv_sampler_loss_fused accepts the call ``flow_resample_loss(data, flow, target, mode)`` makes:
    C in {1,3,4}, W*C and Wout*C multiples of 4, an image-shaped flow (Hout > 1) and 16-byte aligned source, flow and
    target.  Never for mode 'ssim': the SSIM + L1 loss has no fused warp form (a fused kernel measured no faster than the
    sampler, ssim_l1_loss and the sampler's flow gradient as separate calls), so its callers take those calls.
    The C ABI returns DMV_E_UNSUPPORTED_SHAPE otherwise, so a caller with a view at an offset must take the separate calls.
    Without ``target`` only the source and the flow are checked: pass the target wherever it is known."""
    Cc, W, Wo = data.shape[-1], data.shape[2], flow.shape[2]
    return (flow.dim() == 4 and data.numel() > 0 and flow.numel() > 0 and flow.shape[1] > 1 and Cc in (1, 3, 4)
            and (W * Cc) % 4 == 0 and (Wo * Cc) % 4 == 0
            and mode in LOSS
            and all(_passed_aligned16(t) for t in (data, flow, target) if t is not None))


def flow_resample_loss(data, flow, target, mode="l2", weights=None, inv_count=None, grid_order="ref_yx", unit_upstream=False, group=1):
    """(loss, gen) of the training step's tail: warp ``data`` by ``flow`` (grid formed in the kernel), compare with
    ``target``.  One launch instead of sampler forward + loss + sampler backward.  group > 1: ``data`` holds B_src
    sources and flow / target B_src * group samples, sample n warping source n // group
    (dmv_sampler_loss_fused_shared_src)."""
    if grid_order not in ("ref_yx", "xy"):
        raise ValueError(grid_order)
    flags = SAMPLER_ADD_GRID | (SAMPLER_GRID_XY if grid_order == "xy" else 0)
    Cc = data.shape[-1]
    weights = [1.0] * Cc if weights is None else list(weights)
    if inv_count is None:
        inv_count = 1.0 / (target.numel() // Cc)
    group = int(group)
    if group < 1 or flow.shape[0] != data.shape[0] * group:
        raise ValueError("flow holds %d samples, not B_src * group = %d * %d" % (flow.shape[0], data.shape[0], group))
    return _WarpLoss.apply(data, flow, target, flags, tuple(weights), mode, inv_count, unit_upstream, group)


class _ViewsWarpLoss(torch.autograd.Function):
    """head -> (loss, fused): every view's warp by channels 0-1 of its head, the softmax fusion by channel 2, the loss
    and d loss / d head in one kernel (dmv_sampler_fuse_views_loss).  The sources and the target are network inputs."""

    @staticmethod
    def forward(ctx, data, head, target, views, flags, weights, mode, inv_count, unit_upstream, want_grad):
        Cc = data.shape[-1]
        B, Ho, Wo = target.shape[0], target.shape[1], target.shape[2]
        fused = torch.empty((B, Ho, Wo, Cc), dtype=torch.float32, device=data.device)
        grad_head = torch.empty_like(head) if want_grad else None       # a validation pass computes the loss alone
        loss = torch.empty((), dtype=torch.float32, device=data.device)
        w = (C.c_float * Cc)(*[float(x) for x in weights])
        nws = _lib.load().dmv_sampler_loss_workspace_size(B, Ho, Wo)
        key = ("warp_loss", data.device.type, data.device.index)
        ws = _loss_wss.get(key)
        if ws is None or ws.numel() < nws:             # zeroed once: holds a self-resetting counter
            ws = _loss_wss[key] = torch.zeros(int(nws), dtype=torch.uint8, device=data.device)
        _tag[0] = "warp_loss"
        call("dmv_sampler_fuse_views_loss", _p(data), views, _p(head), _p(target), w, LOSS[mode], float(inv_count), _p(fused),
             _p(grad_head), _p(loss), B, data.shape[1], data.shape[2], Cc, Ho, Wo, flags, _p(ws), ws.numel(), _stream(data))
        ctx.grad_head, ctx.unit_upstream = grad_head, unit_upstream
        ctx.mark_non_differentiable(fused)
        return loss, fused

    @staticmethod
    def backward(ctx, gloss, _gfused):
        gh = ctx.grad_head
        if not ctx.unit_upstream:
            _tag[0] = "warp_loss"
            call("dmv_scale_by_device_scalar", _p(gh), _p(gloss.contiguous().to(torch.float32)), gh.numel(), _stream(gh))
        return None, gh, None, None, None, None, None, None, None, None


def _views_args(data, head, views, grid_order, target=None):
    if grid_order not in ("ref_yx", "xy"):
        raise ValueError(grid_order)
    _need_cuda(data, head, *([target] if target is not None else []))
    views = int(views)
    if data.dim() != 4 or head.dim() != 4 or head.shape[-1] != 3:
        raise ValueError("data [views*B,H,W,C] and head [views*B,Hout,Wout,3] expected, got %s and %s"
                         % (tuple(data.shape), tuple(head.shape)))
    if views < 1 or head.shape[0] != data.shape[0] or data.shape[0] % views:
        raise ValueError("data and head hold %d and %d rows, not views * B with views = %d" % (data.shape[0], head.shape[0], views))
    if target is not None and (target.shape[0] * views != data.shape[0] or tuple(target.shape[1:3]) != tuple(head.shape[1:3])
                               or target.shape[-1] != data.shape[-1]):
        raise ValueError("target %s does not match data %s and head %s" % (tuple(target.shape), tuple(data.shape), tuple(head.shape)))
    tensors = [data, head] + ([target] if target is not None else [])
    if any(t.dtype != torch.float32 for t in tensors):
        raise TypeError("the multi-view warp runs in float32 (reference precision)")
    return views, SAMPLER_ADD_GRID | (SAMPLER_GRID_XY if grid_order == "xy" else 0)


def fused_views_warp_loss(data, head, target, views, mode="l2", weights=None, inv_count=None, grid_order="ref_yx", unit_upstream=False):
    """(loss, fused) of several source views per target (Zhou et al.'s multi-view appearance flow), view v of target b in
    row v*B + b: data [views*B,H,W,C], head [views*B,Hout,Wout,3] (flow in channels 0-1, confidence logit in 2), target
    [B,Hout,Wout,C].  fused = sum_v softmax_v(logit) * warp(data_v, flow_v); backward gives d loss / d head, all three
    channels.  One launch (dmv_sampler_fuse_views_loss) in place of the sampler, the fused loss and the sampler's flow
    gradient; the sources get no gradient: it raises if ``data`` needs one."""
    views, flags = _views_args(data, head, views, grid_order, target)
    if torch.is_grad_enabled() and data.requires_grad:
        raise RuntimeError("fused_views_warp_loss has no gradient wrt the sources: pass sources that need no gradient")
    Cc = data.shape[-1]
    weights = [1.0] * Cc if weights is None else list(weights)
    if inv_count is None:
        inv_count = 1.0 / (target.numel() // Cc)
    want_grad = torch.is_grad_enabled() and head.requires_grad
    return _ViewsWarpLoss.apply(data.contiguous(), head.contiguous(), target.contiguous(), views, flags, tuple(weights), mode, inv_count,
                                unit_upstream, want_grad)


def fused_views_warp(data, head, views, grid_order="ref_yx"):
    """Forward only of fused_views_warp_loss: data [views*B,H,W,C], head [views*B,Hout,Wout,3] -> fused [B,Hout,Wout,C]."""
    views, flags = _views_args(data, head, views, grid_order)
    data, head = data.contiguous(), head.contiguous()
    B, Cc = data.shape[0] // views, data.shape[-1]
    Ho, Wo = head.shape[1], head.shape[2]
    fused = torch.empty((B, Ho, Wo, Cc), dtype=torch.float32, device=data.device)
    _tag[0] = "sampler"
    call("dmv_sampler_fuse_views_loss", _p(data), views, _p(head), None, None, 0, 0.0, _p(fused), None, None, B, data.shape[1],
         data.shape[2], Cc, Ho, Wo, flags, None, 0, _stream(data))
    return fused


def resampler_debug(data, wf, flags=0):
    """Forward plus the bit-exact targets: corner indices [.,4] int32 and predicate mask uint8."""
    _need_cuda(data, wf)
    data, wf = data.contiguous(), wf.contiguous()
    B, H, W, Cc = data.shape
    Ho, Wo = (wf.shape[1], wf.shape[2]) if wf.dim() == 4 else (1, int(wf.numel() // (2 * B)))
    out = torch.empty(tuple(wf.shape[:-1]) + (Cc,), dtype=torch.float32, device=data.device)
    idx = torch.empty(tuple(wf.shape[:-1]) + (4,), dtype=torch.int32, device=data.device)
    mask = torch.empty(tuple(wf.shape[:-1]), dtype=torch.uint8, device=data.device)
    call("dmv_sampler_fwd", _p(data), _p(wf), _p(out), _p(idx), _p(mask), B, H, W, Cc, Ho, Wo, flags, _stream(data))
    return out, idx, mask


# ----------------------------------------------------------------------------- losses
class _FusedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gen, logits, target, mask, weights, mode, inv_count, want_fused, unit_upstream=False):
        _need_cuda(gen, target)
        gen = gen.contiguous()
        target = target.contiguous()
        V = 1 if logits is None else gen.shape[0]
        Cc = gen.shape[-1]
        pixels = target.numel() // Cc
        if logits is not None:
            logits = logits.contiguous()
        if mask is not None:
            mask = mask.contiguous()
        w = (C.c_float * Cc)(*[float(x) for x in weights])
        loss = torch.empty((), dtype=torch.float32, device=gen.device)
        need_g = ctx.needs_input_grad[0]
        need_l = logits is not None and ctx.needs_input_grad[1]
        gg = torch.empty_like(gen) if need_g else None
        gl = torch.empty_like(logits) if need_l else None
        fused = torch.empty_like(target) if (want_fused and V > 1) else None
        nws = _lib.load().dmv_loss_workspace_size(pixels)
        ws = _loss_ws(gen.device, nws)
        _tag[0] = "loss"
        call("dmv_loss_fused_fwd_bwd", _p(gen), _p(logits), V, _p(target), _p(mask), w, LOSS[mode], float(inv_count), _p(loss),
             _p(gg), _p(gl), _p(fused), pixels, Cc, _p(ws), ws.numel(), _stream(gen))
        ctx.grads = (gg, gl)
        ctx.unit_upstream = unit_upstream
        ctx.mark_non_differentiable(*([fused] if fused is not None else []))
        if fused is not None:
            return loss, fused
        return loss

    @staticmethod
    def backward(ctx, gloss, *unused):
        gg, gl = ctx.grads
        if ctx.unit_upstream:       # the caller guarantees d(total)/d(this loss) == 1: nothing to chain
            return gg, gl, None, None, None, None, None, None, None
        st = _stream(gloss)
        _tag[0] = "loss"
        gloss = gloss.contiguous().to(torch.float32)
        # chain the upstream scalar on the device (1.0 for a plain loss.backward())
        if gg is not None:
            call("dmv_scale_by_device_scalar", _p(gg), _p(gloss), gg.numel(), st)
        if gl is not None:
            call("dmv_scale_by_device_scalar", _p(gl), _p(gloss), gl.numel(), st)
        return gg, gl, None, None, None, None, None, None, None


def _loss_ws(device, nbytes):
    """The loss workspace holds a self-resetting counter, so it is zero-initialised once and
    never shared with other kernels."""
    key = (device.type, device.index)
    ws = _loss_wss.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(int(nbytes), dtype=torch.uint8, device=device)
        _loss_wss[key] = ws
    return ws


class _SsimLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gen, target, weights, alpha, inv_count, unit_upstream):
        _need_cuda(gen, target)
        gen, target = gen.contiguous(), target.contiguous()
        H, W, Cc = gen.shape[-3], gen.shape[-2], gen.shape[-1]
        B = gen.numel() // (H * W * Cc)
        w = (C.c_float * Cc)(*[float(x) for x in weights])
        loss = torch.empty((), dtype=torch.float32, device=gen.device)
        gg = torch.empty_like(gen) if ctx.needs_input_grad[0] else None
        ws = _loss_ws(gen.device, _lib.load().dmv_loss_workspace_size(B * H * W))
        _tag[0] = "loss"
        call("dmv_ssim_loss_fwd_bwd", _p(gen), _p(target), w, float(alpha), float(inv_count), _p(loss), _p(gg), B, H, W, Cc, _p(ws),
             ws.numel(), _stream(gen))
        ctx.gg, ctx.unit_upstream = gg, unit_upstream
        return loss

    @staticmethod
    def backward(ctx, gloss):
        gg = ctx.gg
        if not ctx.unit_upstream:
            _tag[0] = "loss"
            call("dmv_scale_by_device_scalar", _p(gg), _p(gloss.contiguous().to(torch.float32)), gg.numel(), _stream(gg))
        return gg, None, None, None, None, None


def ssim_l1_loss(gen, target, alpha=0.85, weights=None, inv_count=None, unit_upstream=False, mask=None):
    """inv_count * sum_{images, pixels, c} w_c * (alpha * (1 - SSIM) / 2 + (1 - alpha) * |gen - target|) with a 3x3 SSIM
    window over reflection-padded images (Monodepth2's SSIM without its clamp; include/dmv3d.h states it in full).
    gen and target are [..., H, W, C] with H, W >= 2 and C in {1,3,4}; leading axes are images.  inv_count defaults to
    1 / (images * H * W).  One launch (dmv_ssim_loss_fwd_bwd) with the gradient wrt gen fused in; no mask."""
    if mask is not None:
        raise ValueError("ssim_l1_loss takes no mask: a 3x3 window over masked pixels has no defined SSIM here")
    if gen.shape != target.shape or gen.dim() < 3:
        raise ValueError("gen and target must both be [..., H, W, C], got %s and %s" % (tuple(gen.shape), tuple(target.shape)))
    Cc = gen.shape[-1]
    weights = [1.0] * Cc if weights is None else list(weights)
    if inv_count is None:
        inv_count = 1.0 / (target.numel() // Cc)
    return _SsimLoss.apply(gen, target, tuple(weights), float(alpha), inv_count, unit_upstream)


def reconstruction_loss(gen, target, mode="l2", weights=None, inv_count=None, mask=None, unit_upstream=False, alpha=0.85):
    """mean_{b,h,w} sum_c w_c * (d^2 | |d|), d = (gen - target) * mask; gradient fused in.  mode 'ssim': ssim_l1_loss
    with ``alpha`` (no mask).
    unit_upstream=True: the loss enters the optimised objective with coefficient 1 (fold other coefficients
    into ``weights``), so backward skips the pass that chains the upstream scalar."""
    if mode == "ssim":
        return ssim_l1_loss(gen, target, alpha, weights, inv_count, unit_upstream, mask)
    Cc = gen.shape[-1]
    weights = [1.0] * Cc if weights is None else list(weights)
    if inv_count is None:
        inv_count = 1.0 / (target.numel() // Cc)
    return _FusedLoss.apply(gen, None, target, mask, tuple(weights), mode, inv_count, False, unit_upstream)


def fused_views_loss(gens, logits, target, mode="l2", weights=None, inv_count=None, mask=None, want_fused=True):
    """Confidence-weighted fusion of V warped views + loss (SURVEY 8(f)-3):
    gens [V,B,H,W,C], logits [V,B,H,W] -> (loss, fused [B,H,W,C])."""
    Cc = gens.shape[-1]
    weights = [1.0] * Cc if weights is None else list(weights)
    if inv_count is None:
        inv_count = 1.0 / (target.numel() // Cc)
    return _FusedLoss.apply(gens, logits, target, mask, tuple(weights), mode, inv_count, want_fused)


# ----------------------------------------------------------------------------- input images
def prepare_images(u8, size, out=None):
    """read_tf_records.py:100-111 on the device: uint8 [..., H0, W0, C] as stored -> central crop to min(H0, W0) ->
    tf.image.resize_bicubic to [size, size] -> float32 / 255.  One kernel; with H0 = W0 = size it is the plain
    uint8 -> float32 / 255 conversion."""
    _need_cuda(u8)
    if u8.dtype != torch.uint8:
        raise TypeError("prepare_images takes uint8 pixels")
    u8 = u8.contiguous()
    H0, W0, Cc = u8.shape[-3], u8.shape[-2], u8.shape[-1]
    lead = tuple(u8.shape[:-3])
    n = 1
    for d in lead:
        n *= int(d)
    if out is None:
        out = torch.empty(lead + (size, size, Cc), dtype=torch.float32, device=u8.device)
    _tag[0] = "input"
    if H0 == size and W0 == size and out.numel() % 4 == 0:
        call("dmv_u8_to_f32", _p(u8), _p(out), out.numel(), 255.0, _stream(u8))
    else:
        call("dmv_u8_crop_resize_bicubic", _p(u8), _p(out), n, H0, W0, Cc, size, 255.0, _stream(u8))
    return out


# ----------------------------------------------------------------------------- casts (network inputs)
def to_bf16(x):
    """fp32 -> bf16 for non-differentiable network inputs (viewpoint codes)."""
    _need_cuda(x)
    x = x.contiguous()
    if x.dtype == torch.bfloat16:
        return x
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    call("dmv_cast_f32_to_bf16", _p(x), _p(y), x.numel(), _stream(x))
    return y


def to_f32(x):
    _need_cuda(x)
    x = x.contiguous()
    if x.dtype == torch.float32:
        return x
    y = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    call("dmv_cast_bf16_to_f32", _p(x), _p(y), x.numel(), _stream(x))
    return y

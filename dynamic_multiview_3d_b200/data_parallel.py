"""Batch-sharded data parallelism: one process per GPU, ONE exchange per step over NVLink 5 / NVSwitch.
New work relative to the reference, which is single-GPU (SURVEY.md 8(e)).  Three modes (``attach``):

  fused     (default, CUDA, world > 1)  ZeRO-1 style.  The flat buffers are cut into chunks that begin where the big
            FC matrices begin (``plan_chunks``); when the last gradient of a chunk has been written, ONE hand-written
            kernel (csrc/exchange.cu, include/dmv3d.h: dmv_dp_exchange_chunk) runs on a side stream: the owner of each
            1/world slice sums the gradient straight out of its peers' buffers (symmetric memory; fixed rank order, or
            multimem.ld_reduce through the switch), applies TF-Adam to its fp32 masters and moments, and writes the
            refreshed bf16 compute copy into every rank's buffer.  No NCCL kernels, no gradient write-back.
  sharded   the same pipeline on NCCL collectives: reduce_scatter -> owner Adam -> all_gather of the bf16 copies
            (fallback when peer mapping is unavailable; what the CPU / gloo host-logic tests run).
  allreduce bucketed sum-allreduce in REVERSE creation order (the order backward produces gradients), replicated Adam.

The loss already divides by the GLOBAL pixel count, so the summed gradient is the global-batch gradient and Adam needs
no rescale.  Everything is stream-ordered (events, no host sync), hence capturable in a CUDA graph.  The three modes give
bit-identical parameters (tools/check_dp.py, tests/test_dp_gpu.py).
"""
import torch
import torch.distributed as dist


def _wait_for_gradients(stream, device):
    """``stream`` waits for everything enqueued so far on the current stream AND on every weight-gradient lane: the variables
    of one chunk may have reported from different lanes (conv weights on lane 0, big FC matrices on lane 1), and the lanes are
    not ordered against each other."""
    from . import functional as F
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(device))
    stream.wait_event(ev)
    for e in F.lane_events(device):
        stream.wait_event(e)


def plan_buckets(var_table, bucket_elems):
    """var_table: [(name, offset, padded_numel)] in creation order -> buckets, last variable first.
    Each bucket is (start, end, [names]) with start/end offsets into the flat buffer."""
    buckets, names, start, end = [], [], None, None
    for name, off, n in reversed(var_table):
        if not names:
            end = off + n
        start = off
        names.append(name)
        if end - start >= bucket_elems:
            buckets.append((start, end, names))
            names = []
    if names:
        buckets.append((start, end, names))
    return buckets


class GradientAllReducer:
    def __init__(self, flat_grad, var_table, bucket_mb=32.0, group=None, trainable=None):
        """flat_grad: 1-D fp32 tensor; var_table as in plan_buckets; trainable: names that will
        actually report a gradient each step (others are not waited for)."""
        self.flat = flat_grad
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.buckets = plan_buckets(var_table, int(bucket_mb * (1 << 20) / 4))
        self.var2bucket = {}
        self.expected = []
        for bi, (_, _, names) in enumerate(self.buckets):
            live = [n for n in names if trainable is None or n in trainable]
            self.expected.append(len(live))
            for n in live:
                self.var2bucket[n] = bi
        self.pending = list(self.expected)
        self.cuda = flat_grad.is_cuda
        self.comm_stream = torch.cuda.Stream(device=flat_grad.device) if self.cuda else None
        self.launched = []

    def on_grad_ready(self, var):
        bi = self.var2bucket.get(var.name if hasattr(var, "name") else var)
        if bi is None:
            return
        self.pending[bi] -= 1
        if self.pending[bi] == 0:
            self._launch(bi)

    def _launch(self, bi):
        start, end, _ = self.buckets[bi]
        chunk = self.flat[start:end]
        self.launched.append(bi)
        if self.world == 1:
            return
        if self.cuda:
            _wait_for_gradients(self.comm_stream, self.flat.device)
            with torch.cuda.stream(self.comm_stream):
                dist.all_reduce(chunk, op=dist.ReduceOp.SUM, group=self.group)
        else:
            dist.all_reduce(chunk, op=dist.ReduceOp.SUM, group=self.group)

    def finish(self):
        """Join the side stream; buckets whose variables never reported (should not happen)
        are reduced now so the ranks stay consistent."""
        for bi, p in enumerate(self.pending):
            if p > 0 and self.expected[bi] > 0:
                self._launch(bi)
        if self.cuda and self.world > 1:
            torch.cuda.current_stream(self.flat.device).wait_stream(self.comm_stream)
        self.pending = list(self.expected)
        self.launched = []


def plan_chunks(var_table, alloc, chunk_elems, world, trainable=None, big=1 << 20, skip=()):
    """Chunks of the flat buffer for the sharded mode.  Returns (chunks, var2chunks, expected):
    chunks = [(start, end)] tiling [0, alloc) (every length a multiple of world*256), var2chunks maps a variable name to
    the chunks it overlaps, expected[c] = number of trainable variables overlapping chunk c.

    Backward writes gradients from the END of the buffer towards its start, so a chunk is complete when its LOWEST
    variable has reported.  Chunk groups therefore begin where a big variable (>= ``big`` elements: the FC matrices)
    begins -- the group is that matrix plus the small variables created after it, whose gradients arrive earlier -- and
    each group is cut into pieces of at most ``chunk_elems``.  In particular the first group holds only the encoder's
    convolution weights: the exchange that cannot start before the very last weight gradient of the step is a few MB,
    not a slice of fc1 (a uniform grid from offset 0 put 100+ MB behind e0's gradient)."""
    unit = world * 256
    chunk_elems = max(unit, (chunk_elems // unit) * unit)
    assert alloc % unit == 0, "flat buffers must be allocated to a multiple of world*256 elements"
    cuts = {0, alloc}
    for name, off, n in var_table:
        if n >= big and off % unit == 0 and 0 < off < alloc:
            cuts.add(off)
        if name in skip:            # updated elsewhere (optimizer.py, fused FC update): its range gets chunks of its own,
            cuts.add(off)           # which nothing reports to and nothing launches
            cuts.add(off + n)
    cuts = sorted(cuts)
    chunks = []
    for g0, g1 in zip(cuts, cuts[1:]):
        pieces = -(-(g1 - g0) // chunk_elems)
        per = -(-(g1 - g0) // (pieces * unit)) * unit
        chunks += [(s, min(g1, s + per)) for s in range(g0, g1, per)]
    starts = [c[0] for c in chunks]
    import bisect
    var2chunks, expected = {}, [0] * len(chunks)
    for name, off, n in var_table:
        if (trainable is not None and name not in trainable) or name in skip:
            continue
        cs = list(range(bisect.bisect_right(starts, off) - 1, bisect.bisect_right(starts, off + n - 1)))
        var2chunks[name] = cs
        for c in cs:
            expected[c] += 1
    return chunks, var2chunks, expected


def exchange_args(chunks, c, world, shard_end, alloc):
    """(start, n_slice, slot, replicated) of dmv_dp_exchange_chunk: for chunk ``c`` of ``chunks``, sharded (rank r owns
    [start + r * n_slice, start + (r + 1) * n_slice)), or for c < 0 the replicated bias tail [shard_end, alloc) in the last
    slot, its length rounded up to the kernel's multiple of 8."""
    if c >= 0:
        s, e = chunks[c]
        return s, (e - s) // world, c, 0
    return shard_end, -(-(alloc - shard_end) // 8) * 8, len(chunks), 1


class ShardedGradientReducer:
    """ZeRO-1 style exchange: per chunk a reduce-scatter of the gradients (each rank receives the sum of
    its 1/world slice, in place), Adam on the owned slices only (optimizer state and the fp32 masters are
    updated by their owner), then an all-gather of the refreshed bf16 compute copies.  Against the plain
    allreduce this moves 25 % fewer bytes over NVLink and divides the HBM-bound Adam pass (15 % of a
    single-GPU step) by the world size.  Chunks are launched on a side stream as soon as the last
    gradient overlapping them has been written (backward produces them from the end of the buffer)."""

    def __init__(self, store, chunk_mb=32.0, group=None):
        self.store = store
        self.flat = store.flat
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        # [0, shard_end): weights, sharded; [shard_end, alloc): biases, replicated (their fp32 masters feed the epilogues)
        self.shard_end = getattr(store, "shard_end", store.alloc)
        table = [(v.name, v.offset, -(-v.numel // 64) * 64) for v in store.vars.values() if v.offset < self.shard_end]
        trainable = {v.name for v in store.trainable_vars()}
        # single process: the FC matrices that Adam updates inside their weight-gradient kernel (optimizer.py) take no part
        fused = {v.name for v in store.vars.values() if getattr(v, "fused_adam", False)}
        assert not (fused and self.world > 1), "attach() clears the fused-update marks when gradients are exchanged"
        for v in store.vars.values():
            assert v.name not in fused or (v.offset % (self.world * 256) == 0 and v.numel % (self.world * 256) == 0), v.name
        self.chunks, self.var2chunks, self.expected = plan_chunks(table, self.shard_end, int(chunk_mb * (1 << 20) / 4), self.world, trainable,
                                                                  skip=fused)
        self.pending = list(self.expected)
        self.rep_names = {v.name for v in store.vars.values() if v.offset >= self.shard_end and v.name in trainable}
        self.rep_pending = len(self.rep_names)
        self.cuda = self.flat["grad"].is_cuda
        self.comm_stream = torch.cuda.Stream(device=self.flat["grad"].device) if self.cuda else None
        self.launched = []
        self.native = (not dist.is_initialized()) or dist.get_backend(group) == "nccl"
        self.adam = None        # ShardedTFAdam: when attached, a chunk's update and bf16 all-gather follow its reduce-scatter
        self.started = False
        self._plan_deferred()

    # -- deferred updates (single process) ------------------------------------------------------------------------
    # The late FC matrices (a3, a4, a5: 85 M of the 139 M parameters) finish their weight gradients in the middle of
    # backward, and their HBM-bound Adam pass (2.5 GB) then competes with the HBM-bound FC backward itself: that stretch
    # of the step ran at the memory roofline for ~0.7 ms with the tensor cores idle (profiles/r02_timeline_*.txt).
    # Nothing reads those weights again until the FC layers of the NEXT forward pass, which starts with ~0.35 ms of
    # tensor-bound encoder convolutions -- so their chunks are updated there: apply_deferred() launches them on the side
    # stream at the start of the next train_step, each FC layer's forward waits for its own chunks, and the result is
    # bit-identical to updating at the end of the step (same gradients, same step scalars: the tick of the next step
    # comes after its forward).  The launches are gated on a device flag (dmv_adam_multi_gated) so that a captured CUDA
    # graph can contain them unconditionally: the first replay, with nothing pending, skips them.
    def _plan_deferred(self):
        import os
        self.deferred, self.var_wait, self.chunk_done = [], {}, {}
        self.gate, self.pending_host = None, False
        env = os.environ.get("DMV_DEFER_ADAM", "auto")
        if self.world != 1 or not self.cuda or env == "0":
            return
        big = [v for v in self.store.vars.values() if v.trainable and v.offset < self.shard_end and v.numel >= (1 << 20)
               and v.name.endswith("/Matrix")]
        names = set(env.split(",")) if env not in ("auto", "1") else {v.name for v in big[1:]}    # all but the first-created (fc1):
        for v in big:                                                                              # its gradient comes last
            if v.name not in names or getattr(v, "fused_adam", False):
                continue
            cs = [c for c, (s, e) in enumerate(self.chunks) if v.offset <= s and e <= v.offset + v.numel and self.expected[c] > 0]
            if cs:
                self.deferred += cs
                self.var_wait[v.name] = cs[-1]
        self.deferred.sort()                       # ascending offset = the order the forward pass uses them in
        if self.deferred:
            self.gate = torch.zeros(1, dtype=torch.int32, device=self.flat["grad"].device)
            self.store.pre_use_hook = self.wait_var

    def apply_deferred(self):
        """Start of a train step (and before any other use of the weights): launch the pending updates on the side stream."""
        if not self.deferred or self.adam is None:
            return
        from . import functional as F
        dev = self.flat["grad"].device
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        self.comm_stream.wait_event(ev)
        with torch.cuda.stream(self.comm_stream):
            for c in self.deferred:
                self.adam.update_chunk(c, self.comm_stream.cuda_stream, gate=self.gate)
                done = torch.cuda.Event()
                done.record(self.comm_stream)
                self.chunk_done[c] = done
            F._tag[0] = "adam"
            F.call("dmv_set_flag", self.gate.data_ptr(), 0, self.comm_stream.cuda_stream)
            self.all_done = torch.cuda.Event()
            self.all_done.record(self.comm_stream)
        self.pending_host = False

    def wait_var(self, var):
        """Forward pass, before a layer reads ``var``: its deferred update must have landed."""
        c = self.var_wait.get(var.name)
        if c is None:
            return
        if self.pending_host:                      # a forward pass outside train_step (validation, visualisation)
            self.apply_deferred()
        done = self.chunk_done.get(c)
        if done is not None:
            torch.cuda.current_stream(self.flat["grad"].device).wait_event(done)

    def flush(self):
        """Apply what is pending and join: parameters, moments and bf16 copies are those of the completed steps."""
        if self.deferred and self.adam is not None:
            if self.pending_host:
                self.apply_deferred()
            torch.cuda.current_stream(self.flat["grad"].device).wait_stream(self.comm_stream)

    def reset_deferred(self):
        """Forget pending updates (the parameters were restored from a snapshot)."""
        if self.gate is not None:
            self.gate.zero_()
            self.pending_host = False
            self.chunk_done, self.all_done = {}, None      # events recorded during a graph capture are not waitable outside it

    def mark_pending(self):
        """A captured step was replayed: its deferred update is pending on the device; the events of the capture are void."""
        self.pending_host = True
        self.chunk_done, self.all_done = {}, None

    def owned(self, c):
        s, e = self.chunks[c]
        n = (e - s) // self.world
        return s + self.rank * n, s + (self.rank + 1) * n

    def on_grad_ready(self, var):
        name = var.name if hasattr(var, "name") else var
        if not self.started:
            self.started = True
            if self.adam is not None:
                if self.deferred and getattr(self, "all_done", None) is not None:   # the deferred updates read the step scalars
                    torch.cuda.current_stream(self.flat["grad"].device).wait_event(self.all_done)
                self.adam.tick()            # on the main stream, ahead of every chunk of this step
        if name in self.rep_names:
            self.rep_pending -= 1
            if self.rep_pending == 0:
                self._launch(-1)
            return
        for c in self.var2chunks.get(name, ()):
            self.pending[c] -= 1
            if self.pending[c] == 0:
                self._launch(c)

    def _reduce_scatter(self, c):
        if c < 0:                          # the replicated tail: plain allreduce
            dist.all_reduce(self.flat["grad"][self.shard_end:self.store.alloc], op=dist.ReduceOp.SUM, group=self.group)
            return
        s, e = self.chunks[c]
        a, b = self.owned(c)
        g = self.flat["grad"]
        if self.native:
            dist.reduce_scatter_tensor(g[a:b], g[s:e], op=dist.ReduceOp.SUM, group=self.group)
        else:                              # gloo (CPU host-logic tests): same result on the owned slice
            dist.all_reduce(g[s:e], op=dist.ReduceOp.SUM, group=self.group)

    def _launch(self, c):
        """Chunk pipeline on the side stream: reduce-scatter -> Adam on the owned slice -> all-gather of the bf16
        copies.  Every variable overlapping the chunk has finished its backward (dgrad included), so nothing on the
        main stream reads these weights again in this step and the whole tail overlaps the rest of backward."""
        if c >= 0:
            self.launched.append(c)
            if self.deferred and c in self._deferred_chunks():
                return                     # updated at the start of the next step (apply_deferred)
        if self.cuda:
            _wait_for_gradients(self.comm_stream, self.flat["grad"].device)
            with torch.cuda.stream(self.comm_stream):
                if self.world > 1:
                    self._reduce_scatter(c)
                if self.adam is not None and c >= 0:
                    self.adam.update_chunk(c, self.comm_stream.cuda_stream)
                    self.all_gather("half", c)
        elif self.world > 1:
            self._reduce_scatter(c)

    def finish(self):
        for c, p in enumerate(self.pending):
            if p > 0 and self.expected[c] > 0:
                self._launch(c)
        if self.rep_pending > 0 and self.rep_names:
            self._launch(-1)
        self.rep_pending = len(self.rep_names)
        self.started = False
        if self.cuda:
            torch.cuda.current_stream(self.flat["grad"].device).wait_stream(self.comm_stream)
            if getattr(self, "tail_stream", None) is not None and getattr(self, "tail_done", False):
                torch.cuda.current_stream(self.flat["grad"].device).wait_stream(self.tail_stream)
        if self.deferred and self.adam is not None:
            from . import functional as F
            F._tag[0] = "adam"
            F.call("dmv_set_flag", self.gate.data_ptr(), 1, torch.cuda.current_stream(self.flat["grad"].device).cuda_stream)
            self.pending_host = True
        self.order = list(self.launched)
        self.pending = list(self.expected)
        self.launched = []

    def _deferred_chunks(self):
        ds = getattr(self, "_deferred_set", None)
        if ds is None or len(ds) != len(self.deferred):
            ds = self._deferred_set = set(self.deferred)
        return ds

    def all_gather(self, key, c):
        """In-place all-gather of chunk c of flat[key] from the owners' slices."""
        if self.world == 1:
            return
        s, e = self.chunks[c]
        a, b = self.owned(c)
        t = self.flat[key]
        if self.native:
            dist.all_gather_into_tensor(t[s:e], t[a:b], group=self.group)
        else:
            parts = [torch.empty_like(t[a:b]) for _ in range(self.world)]
            dist.all_gather(parts, t[a:b].clone(), group=self.group)
            t[s:e].copy_(torch.cat(parts))

    def gather_full_state(self):
        """Checkpoint time: every rank gets the complete fp32 masters and Adam moments."""
        self.flush()
        for c in range(len(self.chunks)):
            if self.expected[c] > 0:
                for key in ("master", "m", "v"):
                    self.all_gather(key, c)


class ShardedTFAdam:
    """TFAdam over the slices this rank owns, chunk by chunk; each chunk's bf16 all-gather is enqueued on the
    side stream right behind its update so the exchange overlaps the remaining updates."""

    def __init__(self, base, red):
        import ctypes as C
        self.base, self.red = base, red
        self.state = base.state
        self.lr, self.beta1, self.beta2, self.eps, self.grad_scale = base.lr, base.beta1, base.beta2, base.eps, base.grad_scale
        f = red.flat
        self.args = {}
        for c in range(len(red.chunks)):
            if red.expected[c] == 0:
                continue
            a, b = red.owned(c)
            vp = C.c_void_p * 1
            self.args[c] = (vp(f["master"].data_ptr() + 4 * a), vp(f["grad"].data_ptr() + 4 * a), vp(f["m"].data_ptr() + 4 * a),
                            vp(f["v"].data_ptr() + 4 * a), vp(f["half"].data_ptr() + 2 * a), (C.c_longlong * 1)(b - a))
        a, b = red.shard_end, red.store.alloc     # replicated biases: every rank updates all of them
        self.rep = None
        if b > a and red.rep_names:
            vp = C.c_void_p * 1
            self.rep = (vp(f["master"].data_ptr() + 4 * a), vp(f["grad"].data_ptr() + 4 * a), vp(f["m"].data_ptr() + 4 * a),
                        vp(f["v"].data_ptr() + 4 * a), vp(f["half"].data_ptr() + 2 * a), (C.c_longlong * 1)(b - a))

    def tick(self):
        from . import functional as F
        st = torch.cuda.current_stream(self.red.flat["grad"].device).cuda_stream
        F._tag[0] = "adam"
        F.call("dmv_adam_tick", self.state.data_ptr(), self.lr, self.beta1, self.beta2, st)

    def begin_step(self):
        """Before backward (ModelBase.train_step): advance the step scalars; arm the fused FC update (optimizer.py)."""
        red = self.red
        if red.cuda:
            # the tick goes on the stream train_step runs on, ahead of backward: every chunk's update -- whichever
            # weight-gradient lane triggers it -- is ordered behind it
            if red.deferred and getattr(red, "all_done", None) is not None:   # the deferred updates read the previous scalars
                torch.cuda.current_stream(red.flat["grad"].device).wait_event(red.all_done)
            self.tick()
            red.started = True
        if self.base.fused_vars():
            red.store.adam_live = self

    def end_backward(self):
        self.red.store.adam_live = None

    def update_chunk(self, c, st, gate=None):
        from . import functional as F
        p, g, m, v, h, n = self.args[c]
        F._tag[0] = "adam"
        if gate is not None:
            F.call("dmv_adam_multi_gated", p, g, m, v, h, n, 1, self.state.data_ptr(), self.beta1, self.beta2, self.eps, self.grad_scale,
                   gate.data_ptr(), st)
        else:
            F.call("dmv_adam_multi", p, g, m, v, h, n, 1, self.state.data_ptr(), self.beta1, self.beta2, self.eps, self.grad_scale, st)

    def step(self):
        """Called after ShardedGradientReducer.finish(): the sharded chunks are already updated and gathered (side
        stream, joined); what is left is the replicated bias tail, whose allreduce has completed."""
        from . import functional as F
        if getattr(self.red, "tail_done", False):     # the fused exchange summed and updated the bias tail itself
            self.red.tail_done = False
            return
        if self.rep is not None:
            st = torch.cuda.current_stream(self.red.flat["grad"].device).cuda_stream
            p, g, m, v, h, n = self.rep
            F._tag[0] = "adam"
            F.call("dmv_adam_multi", p, g, m, v, h, n, 1, self.state.data_ptr(), self.beta1, self.beta2, self.eps, self.grad_scale, st)

    @property
    def t(self):
        return int(self.state[3].item())


class PeerExchange:
    """The buffers and pointer tables of dmv_dp_exchange_chunk (include/dmv3d.h): the flat gradient and bf16 buffers of
    every rank mapped into every rank's address space (torch.distributed._symmetric_memory: CUDA VMM handles exchanged
    over the process group; a multicast mapping through the NVSwitch when the driver offers one), the symmetric signal
    words, and this rank's local epoch/ticket words.  Plumbing only -- the exchange itself is one kernel per chunk."""

    def __init__(self, store, slots, group=None, use_multicast=None):
        import ctypes as C
        import os
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.store, self.group = store, group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        dev = store.device
        alloc = store.alloc
        words = _lib.load().dmv_dp_signal_words(slots)
        g = symm.empty(alloc, dtype=torch.float32, device=dev)
        h = symm.empty(alloc, dtype=torch.bfloat16, device=dev)
        sig = symm.empty(words, dtype=torch.int32, device=dev)
        sig.zero_()
        gname = self.group.group_name
        self.hg, self.hh, self.hs = symm.rendezvous(g, gname), symm.rendezvous(h, gname), symm.rendezvous(sig, gname)
        # re-home the gradient and bf16 buffers into the symmetric allocations (the weight-gradient kernels and Adam
        # address them through the variables' views)
        g.copy_(store.flat["grad"])
        h.copy_(store.flat["half"])
        store.flat["grad"], store.flat["half"] = g, h
        for v in store.vars.values():
            sl = slice(v.offset, v.offset + v.numel)
            v.grad, v.half = g[sl].view(v.shape), h[sl].view(v.shape)
        self.sig = sig
        self.local = torch.zeros(2 * slots, dtype=torch.int32, device=dev)
        vp = C.c_void_p * self.world
        self.grad_peers = vp(*[int(p) for p in self.hg.buffer_ptrs])
        self.half_peers = vp(*[int(p) for p in self.hh.buffer_ptrs])
        self.sig_peers = vp(*[int(p) for p in self.hs.buffer_ptrs])
        if use_multicast is None:
            # in-switch reduction (multimem) pays from 4 ranks up: measured 3.33 vs 3.56 ms/step at 8 GPUs, but 1.2 vs 0.75 ms
            # for the raw exchange at 2 (every byte then crosses the switch twice); DMV_DP_MULTICAST = 0 | 1 overrides
            env = os.environ.get("DMV_DP_MULTICAST", "auto")
            use_multicast = (self.world >= 4) if env == "auto" else (env == "1")
        mc_g, mc_h = int(getattr(self.hg, "multicast_ptr", 0) or 0), int(getattr(self.hh, "multicast_ptr", 0) or 0)
        self.multicast = bool(use_multicast and mc_g and mc_h)
        self.grad_mc, self.half_mc = (mc_g, mc_h) if self.multicast else (None, None)
        # Grid of the exchange kernel.  Alone it is fastest with every SM busy, but it runs NEXT TO the backward pass: at 8
        # GPUs 64 CTAs give 2.83 ms/step where 148 give 3.09 and 592 give 3.33 (profiles/r02_bench_8gpu_c2_fused_mc_ctas*.json)
        # -- fewer resident CTAs steal fewer issue slots from the tensor-core kernels' epilogue warps, and the transfer
        # has the whole backward pass to finish in.  At 2 GPUs the kernel also carries half of Adam's HBM traffic and
        # wants more (592: 2.97 ms, 64: 3.26 ms).  DMV_DP_CTAS overrides.
        self.ctas = int(os.environ.get("DMV_DP_CTAS", "0")) or max(32, 512 // self.world)
        torch.cuda.synchronize(dev)
        dist.barrier(group=self.group)            # every rank's signal words are zero before anyone signals


class FusedShardedReducer(ShardedGradientReducer):
    """Sharded data parallelism with the exchange fused into ONE hand-written kernel per chunk over peer memory
    (csrc/exchange.cu): the owner's Adam reads the summed gradient of its slice from its peers (in-switch reduction with
    multimem.ld_reduce when a multicast mapping exists, fixed-order peer loads otherwise), updates theta/m/v and
    broadcasts the bf16 copy (multimem.st / peer stores).  Reduce-scatter + Adam + all-gather become one launch: no
    gradient write-back, no second read, no NCCL kernels.  The bias tail (replicated fp32 masters) is summed by every
    rank from its peers in the same fixed order and updated locally."""

    def __init__(self, store, chunk_mb=32.0, group=None):
        super().__init__(store, chunk_mb, group)
        self.px = PeerExchange(store, len(self.chunks) + 1, group)
        self.flat = store.flat
        self.tail_done = False
        self.tail_stream = torch.cuda.Stream(device=store.flat["grad"].device)

    def _exchange(self, c, st):
        from . import functional as F
        ad, px, f = self.adam, self.px, self.flat
        start, n, slot, rep = exchange_args(self.chunks, c, self.world, self.shard_end, self.store.alloc)
        F._tag[0] = "dp_exchange"
        F.call("dmv_dp_exchange_chunk", px.grad_peers, px.half_peers, px.sig_peers, px.grad_mc, px.half_mc,
               f["master"].data_ptr(), f["m"].data_ptr(), f["v"].data_ptr(), px.local.data_ptr(), start, n, self.rank, self.world,
               slot, rep, ad.state.data_ptr(), ad.beta1, ad.beta2, ad.eps, ad.grad_scale, px.ctas, st)

    def _launch(self, c):
        if c >= 0:
            self.launched.append(c)
        if self.adam is None:
            raise RuntimeError("the fused exchange needs the optimizer attached (build_loss=True)")
        # The bias tail and the first chunk (encoder convolutions) both complete with the very last gradients of the step and
        # are tiny: each is two cross-GPU handshakes of latency (~35 us) whatever its size.  They run side by side, the tail
        # on a stream of its own (profiles/r02_timeline_2gpu.txt: 72 us of serialised tail after backward).
        st = self.tail_stream if c < 0 else self.comm_stream
        _wait_for_gradients(st, self.flat["grad"].device)
        with torch.cuda.stream(st):
            self._exchange(c, st.cuda_stream)
        if c < 0:
            self.tail_done = True


def attach(model, bucket_mb=32.0, group=None, mode=None):
    """Make ``model.train_step`` data-parallel over the default (or given) process group.
    mode "fused" (default on CUDA with world > 1): one hand-written kernel per chunk over peer memory (reduce-scatter +
    owner-only Adam + bf16 all-gather, csrc/exchange.cu); "sharded": the same pipeline on NCCL collectives (also the
    fallback when no peer mapping can be made, and what CPU/gloo runs use); "allreduce": bucketed allreduce, replicated Adam."""
    import os
    store = model.store
    mode = mode or os.environ.get("DMV_DP_MODE", "fused")
    if dist.is_initialized() and dist.get_world_size(group) > 1 and hasattr(model.optimizer, "disable_fusion"):
        model.optimizer.disable_fusion()       # the gradients of the FC matrices must exist in memory to be exchanged
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        from . import functional as F
        F.set_tail_lane(False)                 # the exchange's tail chunk follows the last gradients: keep them on lane 0
    if mode == "fused" and not (dist.is_initialized() and dist.get_world_size(group) > 1 and store.flat["grad"].is_cuda
                                and model.optimizer is not None):
        mode = "sharded"
    if mode in ("sharded", "fused"):
        if mode == "fused":
            if dist.get_world_size(group) > 1:        # replicas must start from identical parameters
                dist.broadcast(store.flat["master"], src=0, group=group)
                store.refresh_half()
            try:
                red = FusedShardedReducer(store, bucket_mb, group)
            except Exception as ex:               # no peer mapping on this box / torch build: the NCCL pipeline still works
                import sys
                print("data_parallel: fused exchange unavailable (%r); using the NCCL reduce-scatter pipeline" % (ex,), file=sys.stderr)
                mode, red = "sharded", ShardedGradientReducer(store, bucket_mb, group)
        else:
            red = ShardedGradientReducer(store, bucket_mb, group)
        red.mode = mode
        store.grad_ready_hook = red.on_grad_ready
        model._dp = red
        model.world_size = red.world
        if red.world > 1 and mode != "fused":
            dist.broadcast(store.flat["master"], src=0, group=group)
            store.refresh_half()
        if model.optimizer is not None:
            model.optimizer = ShardedTFAdam(model.optimizer, red)
            red.adam = model.optimizer
        return red
    table = sorted(((v.name, v.offset, -(-v.numel // 64) * 64) for v in store.vars.values()), key=lambda t: t[1])
    red = GradientAllReducer(store.flat["grad"], table, bucket_mb, group, {v.name for v in store.trainable_vars()})
    store.grad_ready_hook = red.on_grad_ready
    model._dp = red
    model.world_size = red.world
    # replicas must start from identical parameters: broadcast rank 0's masters
    if red.world > 1:
        dist.broadcast(store.flat["master"], src=0, group=group)
        store.refresh_half()
    return red

"""
DenoiserEngine — compiles UNetVideoModel.forward (reference unet.py:428-464 + rpe.py:133-174) into a flat
schedule of libfdm_sm100.so kernel launches over a static HBM arena, one schedule ("plan") per input shape.

Design (B200-first, not a module walk):
  * activations are channels-last [N=B*T][H][W][C]; the residual stream, GroupNorm statistics and softmax
    are fp32; tensors that feed GEMMs ("operands") are bf16 in precision="bf16" and fp32 in "fp32".
  * GroupNorm statistics are produced by the epilogue of the kernel that writes the tensor (atomics into
    [N][C] sum/sumsq), so GN+SiLU(+FiLM) is ONE read + ONE write; th.cat skip connections are never
    materialised in fp32 (the GN kernel reads two sources); the 1x1 skip conv of a ResBlock is a second
    K-segment of its out-conv; permute/reshape copies of FactorizedAttentionBlock disappear (kernels index
    the [B*T][HW][C] layout directly).
  * everything that depends only on (t, frame_indices) — time MLP, all FiLM projections, all RPENet tables —
    is computed once per step up front in 6 launches.
  * the plan owns every intermediate buffer (liveness-packed arena), so a step is replayable as a CUDA graph.
"""
import ctypes as C
import os

import torch as th

from . import _native as N_


class NativeShapeError(RuntimeError):
    pass


class Buf:
    """A region of the plan's arena (or of its statistics arena)."""
    __slots__ = ("name", "nbytes", "offset", "first", "last", "persistent", "arena")

    def __init__(self, name, nbytes, persistent=False, arena="main"):
        self.name, self.nbytes, self.persistent, self.arena = name, (int(nbytes) + 255) // 256 * 256, persistent, arena
        self.offset, self.first, self.last = None, None, None


class ProblemArray:
    """A device array of C structs (`cls`, one per item: a field dict like a launch's) that a launch reads through a pointer
    field.  Items name arena buffers, so Plan.finalize writes the array once offsets are known.  `encode(host array, count)`:
    the bytes to store instead of the structs (the RPE-table blob); `fields(items)`: launch fields that depend on items added
    after the launch was emitted (weight-pack launches)."""
    __slots__ = ("cls", "items", "encode", "fields", "dev")

    def __init__(self, cls, items, encode=None, fields=None):
        self.cls, self.items, self.encode, self.fields, self.dev = cls, items, encode, fields, None

    def __iter__(self):  # unpacks as (device array, struct class, items)
        return iter((self.dev, self.cls, self.items))


class Plan:
    def __init__(self, engine, B, T, H, W):
        self.engine, self.B, self.T, self.H, self.W = engine, B, T, H, W
        self.ops = []        # (entry point name, struct class, {field: python value | Buf | tensor | (Buf, byte offset)})
        self.bops = []       # backward schedule (training plans only), same format
        self.cur = self.ops  # list that op() appends to
        self.train = False
        self.tape = []       # backward emitters, one per forward block, run in reverse after the forward schedule is built
        self.bzero_bytes = 0  # arena zeroed at the start of every backward (atomic accumulators, GroupNorm-backward sums)
        self.pack_problems = []  # (src param, src2, dst tensor, co, ci, k, mode): re-packed by ONE launch per forward
        self.bside = set()       # indices into bops of the launches that run on the backward side stream (weight gradients)
        self.bwd_side_stream = self.ev_bfork = self.ev_bjoin = None
        self.bjoin_before = -1   # index into bops where the main stream first needs side-stream results (conditioning path)
        self.bufs = []
        self.pending = []    # ProblemArray of every launch that takes one, filled by finalize()
        self.keep = []       # tensors that must outlive the plan (timestep tables, packed weights)
        self.calls = None    # [(fn, byref(struct))] after finalize()
        self.stats_bytes = 0
        self.graphs = {}     # CUDA graphs captured over this plan (see gaussian_diffusion._graph_sampler)
        self._warm = set()
        self.debug = os.environ.get("FDM_DEBUG_TAPS", "0") == "1"
        self.taps = {}       # module name -> (Buf, C, H, W) of that layer's fp32 NHWC output (readable when debug)
        self.side_begin = self.side_end = self.join_at = 0  # op index range of the RPE-table branch / its first consumer
        self.side_stream = self.ev_fork = self.ev_join = None
        self.attn_maps = {"spatial": [], "temporal": [], "mixed": []}  # collect_attn plans: (Buf in the zeroed arena, shape)
        self.flops = 0       # algorithmic 2*MAC of every conv / linear / attention matmul of one forward
        self.res_a2 = []     # (Buf, C, H, W) of every ResBlock's second GroupNorm output (conv2's operand; dropout applied), in order
        self.drop_p = 0.0    # training plans: ResBlock dropout probability, with its device {seed, nonce} buffer
        self.drop_philox = None
        self.drop_nonce = 0

    def refresh_dropout(self):
        """New dropout masks for the next training forward: {seed, nonce} written on the current stream (the kernels read the buffer
        at run time, so captured forward / backward graphs pick it up).  The seed is one draw of torch's default generator, so
        torch.manual_seed decides the masks; the nonce counts this plan's forwards."""
        self.drop_nonce += 1
        self.drop_philox[0].fill_(int(th.randint(0, 2 ** 62, ()).item()))
        self.drop_philox[1].fill_(self.drop_nonce)

    # ---- buffers
    def buf(self, name, nbytes, persistent=False):
        # FDM_DEBUG_TAPS=1: no buffer reuse, so every intermediate can be read back after a run (tests/debugging)
        b = Buf(name, nbytes, persistent or self.debug or self.train)
        self.bufs.append(b)
        return b

    def bzero(self, name, nbytes):
        b = Buf(name, nbytes, True, "bzero")
        b.offset = self.bzero_bytes
        self.bzero_bytes += b.nbytes
        return b

    def zeroed(self, name, nbytes):
        """A buffer in the statistics arena: zeroed at the head of every run (GroupNorm statistics and other accumulators written
        with atomics)."""
        b = Buf(name, nbytes, True, "stats")
        b.offset = self.stats_bytes
        self.stats_bytes += b.nbytes
        return b

    def problem_array(self, cls, items, encode=None, fields=None):
        arr = ProblemArray(cls, items, encode, fields)
        self.pending.append(arr)
        return arr

    @staticmethod
    def field_values(fields):
        """The values of a launch's fields, with the values of its problem array's items in place of the array."""
        for v in fields.values():
            if isinstance(v, ProblemArray):
                for it in v.items:
                    yield from it.values()
            else:
                yield v

    def op(self, fn, cls, **fields):
        if self.cur is self.ops:  # liveness of the arena buffers a forward launch reads or writes
            idx = len(self.ops)
            for v in self.field_values(fields):
                b = v[0] if isinstance(v, tuple) else v
                if isinstance(b, Buf) and b.arena == "main":
                    b.first = idx if b.first is None else b.first
                    b.last = idx
        self.cur.append((fn, cls, fields))

    # ---- liveness-based packing (first-fit over a free list), then struct materialisation
    def finalize(self, device):
        free, top = [], 0  # free: [(offset, size)]
        release = {}
        for b in self.bufs:
            if b.first is None:
                b.first = b.last = 0
            if not b.persistent:
                release.setdefault(b.last, []).append(b)
        order = sorted(self.bufs, key=lambda b: (0 if b.persistent else 1, b.first))
        # persistent buffers first, at the bottom of the arena
        for b in order:
            if b.persistent:
                b.offset, top = top, top + b.nbytes
        by_first = {}
        for b in self.bufs:
            if not b.persistent:
                by_first.setdefault(b.first, []).append(b)
        for i in range(len(self.ops)):
            for b in by_first.get(i, []):
                slot = next((k for k, (o, s) in enumerate(free) if s >= b.nbytes), None)
                if slot is None:
                    b.offset, top = top, top + b.nbytes
                else:
                    o, s = free.pop(slot)
                    b.offset = o
                    if s > b.nbytes:
                        free.append((o + b.nbytes, s - b.nbytes))
            for b in release.get(i, []):
                free.append((b.offset, b.nbytes))
                free.sort()
                merged = []
                for o, s in free:  # coalesce neighbours
                    if merged and merged[-1][0] + merged[-1][1] == o:
                        merged[-1] = (merged[-1][0], merged[-1][1] + s)
                    else:
                        merged.append((o, s))
                free = merged
        self.arena = th.empty(max(top, 256), dtype=th.uint8, device=device)
        self.stats_arena = th.zeros(max(self.stats_bytes, 256) // 4, dtype=th.float32, device=device)
        self.bzero_arena = th.zeros(max(self.bzero_bytes, 256) // 4, dtype=th.float32, device=device)
        self.arena_bytes = top
        value = lambda v: self.ptr(v) if isinstance(v, (Buf, tuple, th.Tensor, ProblemArray)) or v is None else v
        for a in self.pending:
            arr = (a.cls * max(len(a.items), 1))()
            for st, it in zip(arr, a.items):
                for k, v in it.items():
                    setattr(st, k, value(v))
            raw = bytes(arr) if a.encode is None else a.encode(arr, len(a.items))
            dev = th.zeros(len(raw) + 128, dtype=th.uint8, device=device)
            a.dev = dev[(-dev.data_ptr()) % 128:][:len(raw)]  # tensor maps need 128-byte alignment
            a.dev.copy_(th.frombuffer(bytearray(raw), dtype=th.uint8))
        lib = N_.lib()
        self.calls, self.bcalls = [], []
        self._structs = []
        for ops, calls in ((self.ops, self.calls), (self.bops, self.bcalls)):
            for fn, cls, fields in ops:
                for v in list(fields.values()):
                    if isinstance(v, ProblemArray) and v.fields is not None:
                        fields.update(v.fields(v.items))
                st = cls()
                for k, v in fields.items():
                    setattr(st, k, value(v))
                self._structs.append(st)
                calls.append((fn, getattr(lib, fn), C.byref(st)))

    def ptr(self, v):
        if v is None:
            return None
        if isinstance(v, th.Tensor):
            return v.data_ptr()
        if isinstance(v, ProblemArray):
            return v.dev.data_ptr()
        off = 0
        if isinstance(v, tuple):
            v, off = v
        base = {"main": self.arena, "stats": self.stats_arena, "bzero": self.bzero_arena}[v.arena]
        return base.data_ptr() + v.offset + off

    def set_t_source(self, table):
        """Timestep embedding input: the float `t` buffer (table=None) or t_table[t_index] looked up on the device."""
        st = self._structs[self.temb_op]
        if table is None:
            st.t, st.t_index, st.t_table = self.ptr(self.t), None, None
        else:
            st.t, st.t_index, st.t_table = None, self.ptr(self.t_index), table.data_ptr()
            if not any(k is table for k in self.keep):
                self.keep.append(table)

    def tap(self, name):
        """fp32 NCHW copy of a layer output (only meaningful with FDM_DEBUG_TAPS=1, after run())."""
        b, Cc, Hh, Ww = self.taps[name]
        return self.view(b, (self.B * self.T, Hh, Ww, Cc), th.float32).permute(0, 3, 1, 2).contiguous()

    def view(self, b, shape, dtype):
        n = 1
        for s in shape:
            n *= s
        esz = th.empty((), dtype=dtype).element_size()
        return self.arena[b.offset:b.offset + n * esz].view(dtype).view(*shape)

    def run_graphed(self, which, device, seg=None):
        """Training: the forward ("fwd") / backward ("bwd") schedule as ONE CUDA graph replay; `seg` = (lo, hi) replays only that
        range of the backward schedule (its own graph: the overlapped gradient exchange interleaves NCCL calls between the
        segments).  The first call of each runs eagerly (lazy module loading, cudaFuncSetAttribute), the second captures;
        FDM_NO_GRAPH=1 keeps everything eager."""
        if which == "fwd":
            body = self.run
        elif seg is None:
            body = self.run_backward
        else:
            body = lambda st: self.run_backward(st, seg[0], seg[1])
        cur = lambda: th.cuda.current_stream(device).cuda_stream
        if os.environ.get("FDM_NO_GRAPH", "0") == "1":
            return body(cur())
        key = ("train", which, seg)
        if key not in self.graphs:
            if key not in self._warm:
                self._warm.add(key)
                return body(cur())
            th.cuda.current_stream(device).synchronize()
            g = th.cuda.CUDAGraph()
            with th.cuda.graph(g, capture_error_mode="thread_local"):
                body(cur())
            self.graphs[key] = g
        self.graphs[key].replay()

    def run_backward(self, stream, lo=0, hi=None):
        """Launch the backward schedule (training plans), or its launches [lo, hi): zero the accumulator arena and the flat
        parameter-gradient buffer (lo == 0 only), then every backward kernel in order on `stream`.  The caller has copied
        d(loss)/d(eps) into `geps_view`.  A partial range ends with the side stream joined, so that everything it launched —
        hence every gradient bucket that is final at `hi` — is ordered before whatever the caller enqueues next."""
        hi = len(self.bcalls) if hi is None else hi
        if lo == 0:
            self.bzero_arena.zero_()
            self.pgrad.zero_()
        s = C.c_void_p(stream)
        side = self.bwd_side_stream
        if side is not None:
            # weight-gradient launches only feed parameter gradients: they run on a side stream (parallel branches of the CUDA
            # graph), each ordered after the main-stream kernel that produced its gradient operand, so the dgrad / GroupNorm /
            # attention chain — the critical path — does not wait for them.  Buffers are never reused in training plans; the
            # split-K workspace is shared only among side-stream launches (serialised there).
            main = th.cuda.current_stream(self.arena.device)
            assert main.cuda_stream == stream, "Plan.run_backward expects torch's current stream"
            ss = C.c_void_p(side.cuda_stream)
        used_side = False
        for i in range(lo, hi):
            name, fn, ref = self.bcalls[i]
            if side is not None and i == self.bjoin_before and used_side:
                self.ev_bjoin.record(side)
                main.wait_event(self.ev_bjoin)
            if side is not None and i in self.bside:
                self.ev_bfork.record(main)
                side.wait_event(self.ev_bfork)
                rc = fn(ref, ss)
                used_side = True
            else:
                rc = fn(ref, s)
            if rc != 0:
                N_.check(rc, name)
        if side is not None and used_side:
            self.ev_bjoin.record(side)
            main.wait_event(self.ev_bjoin)

    def backward_segments(self):
        """[(lo, hi, (first, last+1) of the gradient bucket that is final at hi)]: the backward schedule cut at the completion
        points of the gradient buckets (see DenoiserEngine._grad_buckets)."""
        segs, lo = [], 0
        for b_lo, b_hi, done in self.grad_buckets:
            segs.append((lo, done + 1, (b_lo, b_hi)))
            lo = done + 1
        return segs

    def run(self, stream):
        """Launch the whole schedule on `stream` (the raw cudaStream_t of torch's CURRENT stream).  The caller has filled the
        input buffers.  The RPE-table branch (rpe_hidden + the 21 RPENet output GEMMs: small grids that depend only on
        (t, frame_indices)) is forked onto a side stream and joined before the first temporal attention, so it overlaps the
        stem / first ResBlocks instead of running in front of them; inside a CUDA-graph capture the fork/join become graph
        edges."""
        self.stats_arena.zero_()
        s = C.c_void_p(stream)
        lo, hi, join = self.side_begin, self.side_end, self.join_at
        use_side = hi > lo and self.side_stream is not None
        if use_side:
            main = th.cuda.current_stream(self.arena.device)
            assert main.cuda_stream == stream, "Plan.run expects torch's current stream"
            ss = C.c_void_p(self.side_stream.cuda_stream)
        for i, (name, fn, ref) in enumerate(self.calls):
            if use_side:
                if i == lo:
                    self.ev_fork.record(main)
                    self.side_stream.wait_event(self.ev_fork)
                if i == join:
                    main.wait_event(self.ev_join)
            rc = fn(ref, ss if (use_side and lo <= i < hi) else s)
            if rc != 0:
                N_.check(rc, name)
            if use_side and i == hi - 1:
                self.ev_join.record(self.side_stream)


class _DenoiserFn(th.autograd.Function):
    """UNetVideoModel.forward as ONE autograd node: forward = the plan's kernel schedule, backward = its backward schedule
    (conv dgrad/wgrad, GroupNorm / attention / conditioning-path backward kernels of libfdm_sm100.so); parameter gradients come
    back as views of one flat buffer.  Replaces the ~1500-node autograd graph torch builds for the reference model."""

    @staticmethod
    def forward(ctx, engine, x, x0, timesteps, frame_indices, obs_mask, latent_mask, *params):
        B, T, Cx, H, W = x.shape
        P = engine.plan_for(B, T, H, W, x.device, train=True, drop_p=engine.train_dropout())
        if P.drop_philox is not None:
            P.refresh_dropout()
        engine.load_inputs(P, x, x0, timesteps, frame_indices, obs_mask, latent_mask)
        P.run_graphed("fwd", x.device)
        P.generation = getattr(P, "generation", 0) + 1
        ctx.plan, ctx.generation = P, P.generation
        ctx.route = grad_route(engine.model)
        return P.eps_view.clone()

    @staticmethod
    def backward(ctx, g):
        P = ctx.plan
        if P.generation != ctx.generation:
            raise RuntimeError("the activations of this forward were overwritten by a later forward of the same shape "
                               "(the training plan keeps ONE set of saved activations): call backward before the next forward")
        P.geps_view.copy_(g)
        return (None,) * 7 + ctx.route.hand_over(P, g.device)


class GradRoute:
    """Where the native backward's flat parameter gradient (`Plan.pgrad`) goes: one per model, see `grad_route(model)`.

      sink          the optim.FlatAdamW bound to the model (flat-gradient mode), or None
      reduce        reduce(flat): blocking in-place mean-allreduce (sharding.FlatGradDataParallel), or None
      reduce_async  reduce_async(view) -> finish: starts a bucket's mean-allreduce, finish() makes the current stream wait for it;
                    or None (one allreduce after the whole backward)
      synced        False inside FlatGradDataParallel.no_sync()
      pending       the sink holds gradients accumulated under no_sync() that have not been reduced yet (FlatAdamW.zero_grad
                    clears it)
    """
    __slots__ = ("sink", "reduce", "reduce_async", "synced", "pending")

    def __init__(self):
        self.sink = self.reduce = self.reduce_async = None
        self.synced, self.pending = True, False

    def hand_over(self, P, device):
        """Run the backward schedule of the training plan `P` and deliver its gradient.  Returns the gradients of the parameter
        inputs of _DenoiserFn: per-parameter views without a sink, (None,) for the sink's anchor otherwise.

        | sink | reduce        | state                       | what happens                                                     |
        |------|---------------|-----------------------------|------------------------------------------------------------------|
        | no   | no            | –                           | run bwd; return per-parameter views of P.pgrad.clone()           |
        | no   | yes           | –                           | run bwd; clone; reduce(clone); return views                      |
        | yes  | no            | –                           | run bwd; sink.receive(P.pgrad)                                   |
        | yes  | yes           | not synced                  | run bwd; receive; pending = True                                 |
        | yes  | yes           | synced, pending             | run bwd; receive; reduce(sink.flat_g); pending = False           |
        | yes  | yes + async,  | synced, not pending         | one bwd graph per P.backward_segments() entry, each followed by  |
        |      | > 1 bucket    |                             | reduce_async(P.pgrad[b_lo:b_hi]); then every finish(); receive   |
        | yes  | yes           | synced, not pending, else   | run bwd; reduce(P.pgrad); receive                                |
        """
        sink, reduce = self.sink, self.reduce
        if sink is None:
            P.run_graphed("bwd", device)
            flat = P.pgrad.clone()  # the plan's buffer is reused by the next backward; autograd owns this copy
            if reduce is not None:
                reduce(flat)
            views = th._C._nn.unflatten_dense_tensors(flat, P.unflat)
            return tuple(views[i] for i in P.unflat_pick)
        # flat-gradient mode (optim.FlatAdamW(..., model=model)): the parameters' .grad are persistent views of the optimizer's flat
        # gradient buffer, so the whole hand-over is ONE allreduce (in place, on the plan's buffer) and ONE copy / add — no
        # per-parameter views, AccumulateGrad nodes or zero_grad loops (1.5 ms of host time per step for 390 tensors)
        if reduce is not None and self.synced and not self.pending:
            if self.reduce_async is not None and len(P.grad_buckets) > 1:
                # overlapped gradient exchange (reference: DDP's bucketed allreduce during backward, train_util.py:118-125): the
                # backward schedule runs as one CUDA graph per gradient bucket; as soon as a segment is enqueued, the bucket that is
                # final at its end is all-reduced (NCCL's stream waits for the segment, the next segment does not wait for NCCL)
                finishes = []
                for lo, hi, (b_lo, b_hi) in P.backward_segments():
                    P.run_graphed("bwd", device, seg=(lo, hi))
                    finishes.append(self.reduce_async(P.pgrad[b_lo:b_hi]))
                for finish in finishes:
                    finish()
            else:
                P.run_graphed("bwd", device)
                reduce(P.pgrad)
            sink.receive(P.pgrad)
            return (None,)
        P.run_graphed("bwd", device)
        sink.receive(P.pgrad)
        if reduce is not None:
            if self.synced:  # first synchronised backward after no_sync(): reduce the accumulated total once
                reduce(sink.flat_g)
            self.pending = not self.synced
        return (None,)


def grad_route(model):
    """The GradRoute of `model` (any nn.Module), created on first use."""
    route = getattr(model, "_grad_route", None)
    if route is None:
        route = model._grad_route = GradRoute()
    return route


class DenoiserEngine:
    def __init__(self, model, precision="bf16"):
        if precision not in ("bf16", "fp32"):
            raise ValueError(f"precision must be 'bf16' or 'fp32', got {precision!r}")
        N_.verify_struct_sizes()
        self.model, self.precision = model, precision
        self.op_dtype = N_.BF16 if precision == "bf16" else N_.F32
        self.op_torch = th.bfloat16 if precision == "bf16" else th.float32
        self.op_size = 2 if precision == "bf16" else 4
        self.use_tc = precision == "bf16"
        self.plans = {}
        self._params = self._n_params = None
        self._train_probe = None
        self.train_plans = {}
        self.packed = {}
        self._versions = None
        # use_scale_shift_norm=False (unet.py:204-206: h = GN(h + emb)) is served on the inference path (fdm_gn_apply film_add);
        # the GroupNorm backward kernels implement the scale/shift form only (forward_train raises)
        self.film_cols = 2 if model.use_scale_shift_norm else 1

    def invalidate(self):
        """Drop the packed inference weights, inference plans and their captured sampler graphs.  Needed after parameter
        updates that bypass torch's version counter: writes through `p.data` (p.data.copy_(ema), dist.broadcast(p.data), raw
        pointer kernels).  load_state_dict / optimizer steps / in-place ops on the Parameter are detected automatically."""
        self.packed.clear()
        self.plans.clear()
        self._versions = None

    # ------------------------------------------------------------------ weights
    def param_list(self):
        """The model's parameters in registration order, cached: walking the module tree (nn.Module.parameters -> named_modules)
        costs ~0.7 ms per traversal for the 390 tensors, and the launch-bound cfg2 training step did it twice per step."""
        if self._params is None or len(self._params) != self._n_params_registered():
            self._params = list(self.model.parameters())
        return self._params

    def _n_params_registered(self):
        if self._n_params is None:
            self._n_params = sum(1 for _ in self.model.parameters())
        return self._n_params

    def _param_versions(self):
        return tuple(p._version for p in self.model.parameters()) + (next(self.model.parameters()).data_ptr(),)

    def refresh_weights(self):
        """(Re)pack weights if any parameter changed (optimizer step, load_state_dict, .to())."""
        v = self._param_versions()
        if v != self._versions:
            self.packed.clear()
            self.plans.clear()
            self._versions = v

    # ------------------------------------------------------------------ plan compiler
    def plan_for(self, B, T, H, W, device, train=False, slot=0, collect_attn=False, drop_p=0.0):
        """`slot`: distinct plans (own arena, own streams) of the same shape — sub-batches run concurrently by the sampler.
        `drop_p`: ResBlock dropout of a training plan (part of its key: a plan built without dropout never serves one with it)"""
        if train:
            # training plans survive optimizer steps: their packed weights are refreshed by ONE fdm_pack_weights launch at the
            # head of every forward; they are rebuilt only when a parameter's storage moves (.to(), re-materialisation)
            # parameter storage moves as a whole (.to(), FlatAdamW flattening): three probes decide whether the full signature
            # (390 data_ptr() calls, ~0.2 ms of host time on the launch-bound small model) has to be rebuilt
            pl = self.param_list()
            probe = (B, T, H, W, str(device), drop_p, pl[0].data_ptr(), pl[len(pl) // 2].data_ptr(), pl[-1].data_ptr())
            if self._train_probe is not None and self._train_probe[0] == probe:
                return self._train_probe[1]
            key = (B, T, H, W, str(device), drop_p, tuple(p.data_ptr() for p in pl))
            if key in self.train_plans:
                self._train_probe = (probe, self.train_plans[key])
            if key not in self.train_plans:
                self.train_plans.clear()
                with th.cuda.device(device):
                    self.train_plans[key] = self._compile(B, T, H, W, device, train=True, drop_p=drop_p)
                self._train_probe = (probe, self.train_plans[key])
            return self.train_plans[key]
        self.refresh_weights()
        key = (B, T, H, W, str(device), slot, bool(collect_attn))
        if key not in self.plans:
            with th.cuda.device(device):
                self.plans[key] = self._compile(B, T, H, W, device, collect_attn=collect_attn)
        return self.plans[key]

    def _compile(self, B, T, H, W, device, train=False, collect_attn=False, drop_p=0.0):
        from .plan_compiler import PlanCompiler
        return PlanCompiler(self, B, T, H, W, device, train=train, collect_attn=collect_attn, drop_p=drop_p).compile()

    # ------------------------------------------------------------------ execution
    def load_conditioning(self, P, x0, frame_indices, obs_mask, latent_mask):
        """Copy the per-stage inputs (constant across diffusion steps) into the plan's static buffers."""
        P.x0_view.copy_(x0)
        P.fi_view.copy_(frame_indices)
        P.obs_view.copy_(obs_mask.reshape(P.B, P.T))
        th.clamp(obs_mask.reshape(P.B, P.T) + latent_mask.reshape(P.B, P.T), max=1, out=P.mask_view)

    def load_inputs(self, P, x, x0, timesteps, frame_indices, obs_mask, latent_mask):
        """Copy one denoiser call's inputs into the plan's static buffers, with the float `t` buffer as the timestep source."""
        self.load_conditioning(P, x0, frame_indices, obs_mask, latent_mask)
        P.set_t_source(None)
        P.x_view.copy_(x)
        P.t_view.copy_(timesteps.reshape(P.B).float())

    def train_dropout(self):
        """Dropout probability of the ResBlocks in a training forward (unet.py:167,203-206): the model's `dropout` in train mode,
        0 in eval mode."""
        p = float(getattr(self.model, "dropout", 0) or 0) if self.model.training else 0.0
        if not 0.0 <= p <= 1.0:
            raise ValueError(f"dropout probability has to be between 0 and 1, but got {p}")
        return p

    def forward_train(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask):
        """Differentiable forward (w.r.t. the parameters) through the native forward + backward schedules."""
        if frame_indices is None:
            raise ValueError("frame_indices is required (temporal RPE, rpe.py:146)")
        if not self.model.use_scale_shift_norm:
            raise NotImplementedError("native training implements use_scale_shift_norm=True (the reference default, script_util.py:34); "
                                      "use FDM_TRAIN_ENGINE=autograd for the additive-embedding ResBlocks (unet.py:204-206)")
        p = self.train_dropout()
        if p > 0 and not x.is_cuda:
            # the masks exist only inside the sm_100a GroupNorm kernels: refuse loudly rather than train without them
            raise NotImplementedError(f"native ResBlock dropout (dropout={p}) draws its masks on a CUDA device; for CPU tensors use the "
                                      "PyTorch expression of the network (FDM_ALLOW_TORCH_TRAIN=1), which applies nn.Dropout")
        sink = grad_route(self.model).sink
        if sink is not None:  # flat-gradient mode: ONE anchor tensor stands in for the 390 parameters in the autograd graph
            return _DenoiserFn.apply(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask, sink.anchor)
        return _DenoiserFn.apply(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask, *self.param_list())

    def forward(self, x, x0, timesteps, frame_indices, obs_mask, latent_mask, collect_attn=False):
        """eps, or (eps, attns) with collect_attn: attns = {"spatial": [...], "temporal": [...], "mixed": []}, one head-averaged
        map per attention block in forward order, as UNetVideoModel.forward(return_attn_weights=True) returns them upstream
        (unet.py:454-464; spatial [B*T, HW, HW], temporal [B*HW, T, T])."""
        B, T, Cx, H, W = x.shape
        if frame_indices is None:
            raise ValueError("frame_indices is required (temporal RPE, rpe.py:146)")
        with N_.device_guard(x.device):
            P = self.plan_for(B, T, H, W, x.device, collect_attn=collect_attn)
            self.load_inputs(P, x, x0, timesteps, frame_indices, obs_mask, latent_mask)
            P.run(th.cuda.current_stream(x.device).cuda_stream)
            eps = P.eps_view.clone()
            if not collect_attn:
                return eps
            attns = {"spatial": [], "temporal": [], "mixed": []}
            for key in ("spatial", "temporal"):
                for buf, shape in P.attn_maps[key]:
                    n = shape[0] * shape[1] * shape[2]
                    flat = P.stats_arena.view(th.uint8)[buf.offset:buf.offset + 4 * n].view(th.float32)
                    attns[key].append(flat.view(*shape).clone())
            return eps, attns

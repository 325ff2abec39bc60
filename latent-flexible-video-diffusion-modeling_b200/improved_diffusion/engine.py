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
import torch.nn as nn

from . import _native as N_
from .nn import timestep_freqs


class NativeShapeError(RuntimeError):
    pass


class Buf:
    """A region of the plan's arena (or of its statistics arena)."""
    __slots__ = ("name", "nbytes", "offset", "first", "last", "persistent", "arena")

    def __init__(self, name, nbytes, persistent=False, arena="main"):
        self.name, self.nbytes, self.persistent, self.arena = name, (int(nbytes) + 255) // 256 * 256, persistent, arena
        self.offset, self.first, self.last = None, None, None


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
        self.keep = []       # tensors that must outlive the plan (weights views, problem arrays)
        self.calls = None    # [(fn, byref(struct))] after finalize()
        self.stats_bytes = 0
        self.graphs = {}     # CUDA graphs captured over this plan (see gaussian_diffusion._graph_sampler)
        self._warm = set()
        self.debug = os.environ.get("FDM_DEBUG_TAPS", "0") == "1"
        self.taps = {}       # module name -> (Buf, C, H, W) of that layer's fp32 NHWC output (readable when debug)
        self.side_begin = self.side_end = self.join_at = 0  # op index range of the RPE-table branch / its first consumer
        self.side_stream = self.ev_fork = self.ev_join = None
        self.temporal_attn_maps = []  # (workspace Buf, B, T, HW, C, heads) of every tcgen05 temporal attention (attention weights)
        self.attn_maps = {"spatial": [], "temporal": [], "mixed": []}  # collect_attn plans: (Buf in the zeroed arena, shape)
        self.flops = 0       # algorithmic 2*MAC of every conv / linear / attention matmul of one forward
        self.conv_flops = 0
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

    def stats(self, name, n, c):
        b = Buf(name, n * c * 2 * 8, True, "stats")
        b.offset = self.stats_bytes
        self.stats_bytes += b.nbytes
        return b

    def zeroed(self, name, nbytes):
        """A buffer in the statistics arena: zeroed at the head of every run (accumulators written with atomics)."""
        b = Buf(name, nbytes, True, "stats")
        b.offset = self.stats_bytes
        self.stats_bytes += b.nbytes
        return b

    def op(self, fn, cls, **fields):
        if self.cur is not self.ops:
            self.cur.append((fn, cls, fields))
            return
        idx = len(self.ops)
        for v in fields.values():
            b = v[0] if isinstance(v, tuple) else v
            if isinstance(b, Buf) and b.arena == "main":
                b.first = idx if b.first is None else b.first
                b.last = idx
        self.ops.append((fn, cls, fields))

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
        lib = N_.lib()
        self.calls, self.bcalls = [], []
        self._structs = []
        for ops, calls in ((self.ops, self.calls), (self.bops, self.bcalls)):
            for fn, cls, fields in ops:
                st = cls()
                for k, v in fields.items():
                    setattr(st, k, self.ptr(v) if isinstance(v, (Buf, tuple, th.Tensor)) or v is None else v)
                self._structs.append(st)
                calls.append((fn, getattr(lib, fn), C.byref(st)))

    def ptr(self, v):
        if v is None:
            return None
        if isinstance(v, th.Tensor):
            return v.data_ptr()
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
        engine.load_conditioning(P, x0, frame_indices, obs_mask, latent_mask)
        P.set_t_source(None)
        P.x_view.copy_(x)
        P.t_view.copy_(timesteps.reshape(B).float())
        P.run_graphed("fwd", x.device)
        P.generation = getattr(P, "generation", 0) + 1
        ctx.plan, ctx.generation, ctx.engine = P, P.generation, engine
        ctx.sink = getattr(engine.model, "_fdm_flat_sink", None)
        return P.eps_view.clone()

    @staticmethod
    def backward(ctx, g):
        P = ctx.plan
        if P.generation != ctx.generation:
            raise RuntimeError("the activations of this forward were overwritten by a later forward of the same shape "
                               "(the training plan keeps ONE set of saved activations): call backward before the next forward")
        P.geps_view.copy_(g)
        sink = ctx.sink
        model = ctx.engine.model
        sync = getattr(model, "_fdm_grad_sync", None)
        bucket_sync = getattr(model, "_fdm_grad_sync_bucket", None)
        overlap = (sink is not None and sync is not None and bucket_sync is not None and getattr(model, "_fdm_grad_sync_on", True)
                   and not getattr(sink, "unsynced", False) and len(P.grad_buckets) > 1)
        if overlap:
            # overlapped gradient exchange (reference: DDP's bucketed allreduce during backward, train_util.py:118-125): the backward
            # schedule runs as one CUDA graph per gradient bucket; as soon as a segment is enqueued, the bucket that is final at its
            # end is all-reduced (NCCL's stream waits for the segment, the next segment does not wait for NCCL)
            pending = []
            for lo, hi, (b_lo, b_hi) in P.backward_segments():
                P.run_graphed("bwd", g.device, seg=(lo, hi))
                pending.append(bucket_sync(P.pgrad[b_lo:b_hi]))
            for finish in pending:
                finish()
            sink.receive(P.pgrad)
            return (None,) * 8
        P.run_graphed("bwd", g.device)
        if sink is not None:
            # flat-gradient mode (optim.FlatAdamW(..., model=model)): the parameters' .grad are persistent views of the optimizer's
            # flat gradient buffer, so the whole hand-over is ONE allreduce (in place, on the plan's buffer) and ONE copy / add —
            # no per-parameter views, AccumulateGrad nodes or zero_grad loops (1.5 ms of host time per step for 390 tensors)
            if sync is None:
                sink.receive(P.pgrad)
            elif not getattr(ctx.engine.model, "_fdm_grad_sync_on", True):  # FlatGradDataParallel.no_sync(): accumulate locally
                sink.receive(P.pgrad)
                sink.unsynced = True
            elif getattr(sink, "unsynced", False):  # first synchronised backward after no_sync(): reduce the accumulated total
                sink.receive(P.pgrad)
                sync(sink.flat_g)
                sink.unsynced = False
            else:
                sync(P.pgrad)
                sink.receive(P.pgrad)
            return (None,) * 8
        flat = P.pgrad.clone()  # the plan's buffer is reused by the next backward; autograd owns this copy
        sync = getattr(ctx.engine.model, "_fdm_grad_sync", None)
        if sync is not None:  # sharding.FlatGradDataParallel: ONE allreduce over the whole flat gradient
            sync(flat)
        views = th._C._nn.unflatten_dense_tensors(flat, P.unflat)
        return (None,) * 7 + tuple(views[i] for i in P.unflat_pick)


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

    def _pack_simt(self, w):
        """[co][ci][kh][kw] or [co][ci] -> fp32 [tap][ci][co]"""
        key = ("simt", w.data_ptr())
        if key not in self.packed:
            w4 = w.detach().float()
            if w4.dim() == 2:
                w4 = w4[:, :, None, None]
            co, ci, kh, kw = w4.shape
            self.packed[key] = w4.permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous()
        return self.packed[key]

    def _pack_tc(self, w):
        """[co][ci][kh][kw] or [co][ci] -> bf16 [tap = kw*k + kh][co_pad][ci_pad]  (K-major B operand, filter-column major taps,
        ci_pad % 64 == 0, co_pad % 16 == 0)"""
        key = ("tc", w.data_ptr())
        if key not in self.packed:
            w4 = w.detach().float()
            if w4.dim() == 2:
                w4 = w4[:, :, None, None]
            co, ci, kh, kw = w4.shape
            cip, cop = (ci + 63) // 64 * 64, (co + 15) // 16 * 16
            out = th.zeros(kh * kw, cop, cip, dtype=th.bfloat16, device=w.device)
            out[:, :co, :ci] = w4.permute(3, 2, 0, 1).reshape(kh * kw, co, ci).to(th.bfloat16)
            self.packed[key] = out
        return self.packed[key]

    def _pack_tc_up(self, w):
        """nearest x2 upsample + 3x3 conv (unet.py:85-93) without the upsampled tensor: output pixel (2y+a, 2x+b) sees the input rows
        y + {a-1, a} and columns x + {b-1, b}; the 3x3 weights that land on the same input pixel are summed in fp32.
        [co][ci][3][3] -> bf16 [phase = 2a + b][tap = 2s' + r'][co_pad][ci_pad]  (conv_halo.cu `up` mode, include/fdm_b200.h)"""
        key = ("tcup", w.data_ptr())
        if key not in self.packed:
            w4 = w.detach().float()
            co, ci, _, _ = w4.shape
            cip, cop = (ci + 63) // 64 * 64, (co + 15) // 16 * 16
            sets = {0: ([0], [1, 2]), 1: ([0, 1], [2])}
            out = th.zeros(16, cop, cip, dtype=th.bfloat16, device=w.device)
            for a in (0, 1):
                for b in (0, 1):
                    for sp in (0, 1):
                        for rp in (0, 1):
                            ws = w4[:, :, sets[a][rp], :][:, :, :, sets[b][sp]].sum(dim=(2, 3))
                            out[(2 * a + b) * 4 + 2 * sp + rp, :co, :ci] = ws.to(th.bfloat16)
            self.packed[key] = out
        return self.packed[key]

    def up_tc_ok(self, Cc, H, W):
        """Upsample convs the halo kernel's phase mode takes (H x W = the LOW-resolution input): whole image rows per 128-pixel tile"""
        # (the 32-column tile variant is not instantiated for the phase mode)
        return self.use_tc and self.halo_map_ok(H, W) and Cc % 8 == 0 and Cc >= 64

    def halo_map_ok(self, H, W):
        return W in (16, 32, 64, 128) and H % (128 // W) == 0

    def _f32(self, p):
        key = ("f32", p.data_ptr())
        if key not in self.packed:
            self.packed[key] = p.detach().float().contiguous()
        return self.packed[key]

    def _bias_sum(self, b0, b1):
        key = ("bsum", b0.data_ptr(), b1.data_ptr())
        if key not in self.packed:
            self.packed[key] = (b0.detach().float() + b1.detach().float()).contiguous()
        return self.packed[key]

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

    def _grad_buckets(self, P, params):
        """Partition the flat parameter-gradient buffer into FDM_GRAD_BUCKETS (default 4) ranges of consecutive slots and find, for
        each, the backward launch after which it is final: [(first element, one past the last element, index of that launch)].
        The slots are in gradient-completion order (optim.completion_order), so the `done` indices ascend: bucket k can be
        all-reduced while launches done_k+1 ... run.  Every parameter must have a writer (DDP find_unused_parameters=False)."""
        import bisect
        base, n = P.pgrad.data_ptr(), P.pgrad.numel()
        by_off = sorted((o, i) for i, o in enumerate(P.flat_offs))
        starts = [o for o, _ in by_off]
        last = [-1] * len(params)

        def note(v, j):
            if isinstance(v, th.Tensor) and base <= v.data_ptr() < base + 4 * n:
                i = by_off[bisect.bisect_right(starts, (v.data_ptr() - base) // 4) - 1][1]
                last[i] = max(last[i], j)
        for j, (_, _, f) in enumerate(P.bops):
            for v in f.values():
                note(v, j)
        for k, (_, _, items) in enumerate(P.pending):
            j = P.pending_at.get(k)
            if j is not None:
                for it in items:
                    for v in it.values():
                        note(v, j)
        names = [nm for nm, _ in self.model.named_parameters()]
        missing = [names[i] for i in range(len(params)) if last[i] < 0]
        if missing:
            raise AssertionError(f"backward schedule: no gradient writer for {missing[:5]} (+{max(0, len(missing) - 5)})")
        want = max(1, int(os.environ.get("FDM_GRAD_BUCKETS", "4")))
        order, n_early = P.flat_order, P.n_early
        size = lambda i: (params[i].numel() + 3) // 4 * 4
        early_total = sum(size(i) for i in order[:n_early])
        groups, cur, acc, k = [], [], 0, 1
        for i in order[:n_early]:
            cur.append(i)
            acc += size(i)
            if want > 2 and acc >= k * early_total / (want - 1) and len(groups) < want - 2:
                groups.append(cur)
                cur, k = [], k + 1
        if cur:
            groups.append(cur)
        if order[n_early:]:
            groups.append(list(order[n_early:]))
        buckets, done_so_far = [], -1
        for g in groups:
            lo = min(P.flat_offs[i] for i in g)
            hi = max(P.flat_offs[i] + size(i) for i in g)
            done_so_far = max(done_so_far, max(last[i] for i in g))
            if buckets and buckets[-1][2] == done_so_far:   # nothing runs between the two completion points: one bucket
                buckets[-1] = (buckets[-1][0], hi, done_so_far)
            else:
                buckets.append((lo, hi, done_so_far))
        assert buckets[0][0] == 0 and buckets[-1][1] == n and all(a[1] == b[0] for a, b in zip(buckets, buckets[1:])), buckets
        buckets[-1] = (buckets[-1][0], buckets[-1][1], len(P.bops) - 1)
        return buckets

    def _temporal_ws(self, B, T, Cc, heads, hw):
        """Workspace bytes of the tcgen05 temporal attention for this shape, or None when the CUDA-core kernel serves it.
        hw=None: is the shape family (T, head dim) taken at all (every attention map of the U-Net has HW % 16 == 0)."""
        a = N_.AttnTemporalArgs(B=B, T=T, HW=hw or 256, C=Cc, heads=heads, qkv_dtype=self.op_dtype, out_dtype=self.op_dtype)
        n = int(N_.lib().fdm_attn_temporal_workspace(C.byref(a)))
        return n if n > 0 else None

    def tc_ok(self, C0, C1, Cout, k, stride, upsample, Ho, Wo):
        """Shapes the tcgen05 implicit-GEMM kernel takes (conv_tc.cu); everything else runs on the CUDA-core engine."""
        if not self.use_tc or upsample:
            return False
        if C0 % 8 or (C1 and C1 % 8):
            return False
        # the 128-pixel M tile must be a box in (w, h, frame): whole rows of one frame, or whole frames
        hw = Ho * Wo
        if Wo >= 128:
            return Wo % 128 == 0
        if hw >= 128:
            return 128 % Wo == 0 and hw % 128 == 0
        return 128 % hw == 0 and (hw % 32 == 0 or 32 % hw == 0)

    def _compile(self, B, T, H, W, device, train=False, collect_attn=False, drop_p=0.0):
        m = self.model
        from .unet import ResBlock, FactorizedAttentionBlock, Downsample, Upsample
        P = Plan(self, B, T, H, W)
        P.train = train
        if train and drop_p > 0:
            P.drop_p = drop_p
            P.drop_philox = th.zeros(2, dtype=th.int64, device=device)
        Nf = B * T
        opd, osz = self.op_dtype, self.op_size
        mc, ted = m.model_channels, m.model_channels * 4
        Cin = m.in_channels  # includes indicator channel
        f32 = self._f32
        bias_sum = self._bias_sum
        pack_fwd = lambda w, tc: (self._pack_tc if tc else self._pack_simt)(w)
        if train:
            # ---- training plan: parameters are read in place (fp32) and packed operands live in persistent tensors that ONE
            #      fdm_pack_weights launch refreshes at the head of every forward; parameter gradients go to one flat buffer
            params = list(m.parameters())
            for p_ in params:
                assert p_.dtype == th.float32 and p_.is_contiguous(), "training plans expect contiguous fp32 master weights"
            # densely packed in parameter order: ONE C++ call (unflatten_dense_tensors) turns a clone of it into the per-parameter
            # gradients — 390 Python-side narrow+view pairs per step were ~2 ms of host time on the launch-bound cfg2 step
            # 16-byte aligned slots (vectorised optimizer kernels) in gradient-COMPLETION order (optim.completion_order): the head and
            # the last output blocks first, the conditioning path (time MLP, FiLM projections, RPENets) last — a bucket of consecutive
            # slots is final once the backward schedule passes one point, so its allreduce overlaps the rest of the backward
            from .optim import model_flat_layout
            _, offs_list, total, order, n_early = model_flat_layout(m)
            P.pgrad = th.zeros(total, dtype=th.float32, device=device)
            P.unflat, P.unflat_pick = [], [0] * len(params)  # templates for unflatten_dense_tensors (flat order) + padding stubs
            for i in order:
                p_, n_ = params[i], (params[i].numel() + 3) // 4 * 4
                P.unflat_pick[i] = len(P.unflat)
                P.unflat.append(p_)
                if n_ != p_.numel():
                    P.unflat.append(th.empty(n_ - p_.numel()))
            offs = {id(p_): o_ for p_, o_ in zip(params, offs_list)}
            P.flat_order, P.flat_offs, P.n_early = order, offs_list, n_early
            P.pgrad_views = [P.pgrad[offs[id(p_)]:offs[id(p_)] + p_.numel()].view(p_.shape) for p_ in params]
            pg = lambda p_: P.pgrad[offs[id(p_)]:offs[id(p_)] + p_.numel()]  # gradient slot of a parameter
            f32 = lambda p_: p_.detach()
            packed = {}
            r16, r64 = (lambda v: (v + 15) // 16 * 16), (lambda v: (v + 63) // 64 * 64)

            def pack_w(w, mode):
                key = (mode, id(w))
                if key not in packed:
                    co, ci = w.shape[0], w.shape[1]
                    k = w.shape[2] if w.dim() == 4 else 1
                    shape, dty = {N_.PACK_TC_FWD: ((k * k, r16(co), r64(ci)), th.bfloat16),
                                  N_.PACK_TC_DGRAD: ((k * k, r16(ci), r64(co)), th.bfloat16),
                                  N_.PACK_SIMT_FWD: ((k * k, ci, co), th.float32),
                                  N_.PACK_SIMT_DGRAD: ((k * k, co, ci), th.float32)}[mode]
                    packed[key] = th.zeros(shape, dtype=dty, device=device)
                    P.pack_problems.append((w, None, packed[key], co, ci, k, mode))
                return packed[key]

            def bias_sum(b0, b1):
                key = ("sum2", id(b0))
                if key not in packed:
                    packed[key] = th.zeros(b0.numel(), dtype=th.float32, device=device)
                    P.pack_problems.append((b0, b1, packed[key], b0.numel(), 1, 1, N_.PACK_SUM2))
                return packed[key]

            pack_fwd = lambda w, tc: pack_w(w, N_.PACK_TC_FWD if tc else N_.PACK_SIMT_FWD)
            pack_dgrad = lambda w, tc: pack_w(w, N_.PACK_TC_DGRAD if tc else N_.PACK_SIMT_DGRAD)
            P.keep.append(packed)
            pack_fields = dict(problems=None, count=0, max_elems=0)
            P.op("fdm_pack_weights", N_.PackWeightsArgs, **pack_fields)
            pack_fields = P.ops[-1][2]
            pack_fields_d = None

        # ---------------- persistent inputs / outputs
        P.x = P.buf("x", Nf * (Cin - 1) * H * W * 4, True)
        P.x0 = P.buf("x0", Nf * (Cin - 1) * H * W * 4, True)
        P.obs = P.buf("obs", Nf * 4, True)
        P.mask = P.buf("mask", Nf * 4, True)
        P.fi = P.buf("fi", Nf * 8, True)
        P.t = P.buf("t", B * 4, True)
        P.t_index = P.buf("t_index", B * 8, True)
        P.eps = P.buf("eps", Nf * m.out_channels * H * W * 4, True)
        P.use_t_index = False
        P.t_table = None

        # ---------------- conditioning path
        res_blocks, attn_blocks = [], []
        for blk in list(m.input_blocks) + [m.middle_block] + list(m.output_blocks):
            for layer in blk:
                if isinstance(layer, ResBlock):
                    res_blocks.append(layer)
                elif isinstance(layer, FactorizedAttentionBlock):
                    attn_blocks.append(layer)
        cols = 0
        film_off, te_off = {}, {}
        for rb in res_blocks:
            film_off[id(rb)] = cols
            cols += self.film_cols * rb.out_channels
        for ab in attn_blocks:
            for which in ("rpe_q", "rpe_k", "rpe_v"):
                te_off[(id(ab), which)] = cols
                cols += ab.channels
        cond_cols = cols
        freqs = timestep_freqs(mc).to(device)
        P.keep.append(freqs)
        # (persistent: the conditioning chain runs on the side stream, concurrently with main-stream launches whose buffers must
        # not alias these)
        temb = P.buf("temb", B * mc * 4, True)
        h1 = P.buf("time_h1", B * ted * 4, True)
        emb = P.buf("emb", B * ted * 4, True)
        cond = P.buf("cond", B * cond_cols * 4, True)  # live for the whole forward
        P.temb_op = len(P.ops)
        P.op("fdm_timestep_embedding", N_.TimestepEmbeddingArgs, t=P.t, t_index=None, t_table=None, freqs=freqs, out=temb,
             B=B, dim=mc)

        self._pending_groups = []

        def emit_group(problems):
            # device array is filled in after finalize() (needs resolved pointers); reserve its storage now
            dev = th.zeros(len(problems) * C.sizeof(N_.LinearProblem), dtype=th.uint8, device=device)
            P.keep.append(dev)
            self._pending_groups.append((dev, problems))
            touch = {}
            for i, pr in enumerate(problems):
                for k in ("x", "y"):
                    b = pr[k][0] if isinstance(pr[k], tuple) else pr[k]
                    if isinstance(b, Buf):
                        touch[f"_{k}{i}"] = b
            idx = len(P.ops)
            P.flops += sum(2 * pr["M"] * pr["K"] * pr["Nout"] for pr in problems)
            P.op("fdm_grouped_linear", N_.GroupedLinearArgs, problems=dev, count=len(problems),
                 max_M=max(p["M"] for p in problems), max_Nout=max(p["Nout"] for p in problems),
                 max_K=max(p["K"] for p in problems))
            for b in touch.values():  # liveness of buffers referenced only through the device problem array
                if b.arena == "main":
                    b.first = idx if b.first is None else b.first
                    b.last = idx

        te0, te2 = m.time_embed[0], m.time_embed[2]
        emit_group([dict(x=temb, w=f32(te0.weight), b=f32(te0.bias), y=h1, M=B, K=mc, Nout=ted, ldx=mc, ldy=ted, silu_in=0)])
        emit_group([dict(x=h1, w=f32(te2.weight), b=f32(te2.bias), y=emb, M=B, K=ted, Nout=ted, ldx=ted, ldy=ted, silu_in=1)])
        probs = []
        for rb in res_blocks:
            lin = rb.emb_layers[1]
            probs.append(dict(x=emb, w=f32(lin.weight), b=f32(lin.bias), y=(cond, film_off[id(rb)] * 4), M=B, K=ted,
                              Nout=self.film_cols * rb.out_channels, ldx=ted, ldy=cond_cols, silu_in=1, lin=lin,
                              off=film_off[id(rb)]))
        for ab in attn_blocks:
            for which in ("rpe_q", "rpe_k", "rpe_v"):
                net = getattr(ab.temporal_attention, which).rpe_net
                lin = net.embed_diffusion_time
                probs.append(dict(x=emb, w=f32(lin.weight), b=f32(lin.bias), y=(cond, te_off[(id(ab), which)] * 4), M=B,
                                  K=ted, Nout=ab.channels, ldx=ted, ldy=cond_cols, silu_in=0, lin=lin,
                                  off=te_off[(id(ab), which)]))
        emit_group(probs)
        film_probs = probs
        # RPENet hidden + output tables for every temporal attention.  bf16 mode: the C x C output linear of each net runs on
        # tcgen05 (fdm_conv, 1x1 over the B*T*T rows, bf16 hidden); fp32 mode: one grouped CUDA-core launch.
        R, R_op = {}, {}
        hid = {}
        rh_probs, out_probs, rpe_tc = [], [], []
        hsz = self.op_size if self.use_tc else 4
        # inference plans whose temporal attentions ALL run on tcgen05: ONE fused launch produces every bf16 table (hidden layer
        # generated in shared memory as the GEMM's A operand: rpe_tables_tc.cu) instead of fdm_rpe_hidden + one GEMM per net
        fuse_tables = (self.use_tc and not train and bool(attn_blocks)
                       and max(ab.channels for ab in attn_blocks) <= 512
                       and all(self._temporal_ws(B, T, ab.channels, ab.temporal_attention.num_heads, None) is not None
                               for ab in attn_blocks))
        for ab in attn_blocks:
            Cc = ab.channels
            for which in ("rpe_q", "rpe_k", "rpe_v"):
                net = getattr(ab.temporal_attention, which).rpe_net
                # (side-stream lifetime: never aliased with main-branch buffers)
                hb = None if fuse_tables else P.buf(f"rpe_hidden", B * T * T * Cc * hsz, True)
                # bf16 copies of the tables are the B operands of the tcgen05 temporal attention (attn_temporal_tc.cu); the fp32
                # tables are only kept where something still reads them: the CUDA-core kernel (shapes the tcgen05 engine does not
                # take) and the backward kernels of training plans
                # (training plans keep the CUDA-core forward: its backward kernels re-form P in fp32 from the fp32 tables, and a
                # forward that rounded P / R to bf16 would leave the analytically-zero gradients (RPE output biases: softmax shift
                # invariance) with more noise than torch's own autocast backward — measured 0.148 vs 0.14 allowed)
                tc_here = (self.use_tc and not train
                           and self._temporal_ws(B, T, ab.channels, ab.temporal_attention.num_heads, None) is not None)
                rop = P.buf(f"rpe_R_op", B * T * T * Cc * 2, True) if tc_here else None
                rb_ = P.buf(f"rpe_R", B * T * T * Cc * 4, True) if (train or not tc_here) else None
                hid[(id(ab), which)], R[(id(ab), which)] = hb, rb_
                R_op[(id(ab), which)] = rop
                rh_probs.append(dict(wd=f32(net.embed_distances.weight), bd=f32(net.embed_distances.bias), hidden=hb, C=Cc,
                                     te_off=te_off[(id(ab), which)]))
                if not self.use_tc:
                    out_probs.append(dict(x=hb, w=f32(net.out.weight), b=f32(net.out.bias), y=rb_, M=B * T * T, K=Cc, Nout=Cc,
                                          ldx=Cc, ldy=Cc, silu_in=0))
                rpe_tc.append((hb, Cc, net, rb_, rop))
        self._pending_rpe_tc = []
        self._pending_rt = None
        if fuse_tables:
            assert all(rop is not None and rb_ is None for _, _, _, rb_, rop in rpe_tc)
            nbytes = int(N_.lib().fdm_rpe_tables_blob_bytes(len(rpe_tc)))
            blob = th.zeros(nbytes + 128, dtype=th.uint8, device=device)
            blob = blob[(-blob.data_ptr()) % 128:][:nbytes]  # tensor maps need 128-byte alignment
            P.keep.append(blob)
            self._pending_rt = (blob, [dict(wd=f32(net.embed_distances.weight), bd=f32(net.embed_distances.bias), bo=f32(net.out.bias),
                                            w_packed=self._pack_tc(net.out.weight), out_op=rop, out_f32=None, C=Cc, te_off=q_["te_off"])
                                       for (hb, Cc, net, rb_, rop), q_ in zip(rpe_tc, rh_probs)])
            P.flops += sum(2 * B * T * T * Cc * Cc for _, Cc, _, _, _ in rpe_tc)
            P.rpe_table_channels = [Cc for _, Cc, _, _, _ in rpe_tc]
            idx = len(P.ops)
            P.side_begin = idx
            P.op("fdm_rpe_tables", N_.RpeTablesArgs, te=cond, frame_indices=P.fi, blob=blob, count=len(rpe_tc), B=B, T=T,
                 te_stride=cond_cols, max_C=max(Cc for _, Cc, _, _, _ in rpe_tc))
            for _, _, _, _, rop in rpe_tc:
                rop.first = idx if rop.first is None else rop.first
                rop.last = idx
            P.side_end = len(P.ops)
            rpe_tc = []
            self._pending_rh = None
        elif rh_probs:
            dev = th.zeros(len(rh_probs) * C.sizeof(N_.RpeHiddenProblem), dtype=th.uint8, device=device)
            P.keep.append(dev)
            self._pending_rh = (dev, rh_probs)
            idx = len(P.ops)
            P.side_begin = idx
            P.op("fdm_rpe_hidden", N_.RpeHiddenArgs, te=cond, frame_indices=P.fi, problems=dev, B=B, T=T,
                 te_stride=cond_cols, count=len(rh_probs), max_C=max(p["C"] for p in rh_probs),
                 hidden_dtype=self.op_dtype if self.use_tc else N_.F32)
            for p_ in rh_probs:
                b = p_["hidden"]
                b.first = idx if b.first is None else b.first
                b.last = idx
            if train:
                # the DGRAD weight layouts are only read by the backward schedule: packed on the side stream (this branch),
                # off the forward's dependent chain
                P.op("fdm_pack_weights", N_.PackWeightsArgs, problems=None, count=0, max_elems=0)
                pack_fields_d = P.ops[-1][2]
            if self.use_tc:
                self._pending_rpe_tc = rpe_tc  # emitted right after the conv helper is defined
            else:
                emit_group(out_probs)
            P.side_end = len(P.ops)
        else:
            self._pending_rh = None

        # ---------------- conv helper
        def conv(a0, C0, Hin, Win, w0, Cout, k, stride=1, upsample=0, a1=None, C1=0, w1=None, bias=None, resid=None,
                 y_f32=None, y_op=None, stats=None, out_nchw=0, a_dtype=None, flop_c0=None, n_frames=None,
                 **resid_norm):
            a_dtype = opd if a_dtype is None else a_dtype
            Nf_ = Nf if n_frames is None else n_frames
            Hv, Wv = (Hin * 2, Win * 2) if upsample else (Hin, Win)
            Ho, Wo = (Hv + 2 * (k // 2) - k) // stride + 1, (Wv + 2 * (k // 2) - k) // stride + 1
            tc = a_dtype == N_.BF16 and self.tc_ok(C0, C1, Cout, k, stride, upsample, Ho, Wo) and (out_nchw or Cout % 4 == 0)
            up_tc = bool(upsample) and a_dtype == N_.BF16 and k == 3 and C0 == Cout and not train and self.up_tc_ok(C0, Hin, Win)
            fl = 2 * Nf_ * Ho * Wo * Cout * (k * k * (flop_c0 or C0) + C1)  # algorithmic: padded channels do not count
            P.flops += fl
            P.conv_flops += fl
            pack = lambda w_: pack_fwd(w_, tc)
            if up_tc:
                tc, pack = True, self._pack_tc_up
            P.op("fdm_conv", N_.ConvArgs, a0=a0, w0=pack(w0), a1=a1, w1=pack(w1) if w1 is not None else None, bias=bias,
                 resid=resid, y_f32=y_f32, y_op=y_op, stats=stats, N=Nf_, Hin=Hin, Win=Win, C0=C0, C1=C1, Cout=Cout,
                 ksize=k, stride=stride, upsample=upsample, a_dtype=a_dtype, op_dtype=opd, out_nchw=out_nchw,
                 engine=N_.CONV_TC if tc else N_.CONV_SIMT, **resid_norm)
            return Ho, Wo

        for hb, Cc, net, rb_, rop in self._pending_rpe_tc:
            conv(hb, Cc, 1, 1, net.out.weight, Cc, 1, bias=f32(net.out.bias), y_f32=rb_, y_op=rop, n_frames=B * T * T)
            P.side_end = len(P.ops)
        self._pending_rpe_tc = []

        # ---------------- backward helpers (training plans): every forward block below registers ONE emitter on P.tape;
        # the emitters run in reverse once the forward schedule is complete and append to P.bops
        P.pending = []   # (device byte tensor, struct class, [field dicts]) filled in after finalize()
        P.pending_at = {}  # index into P.pending -> index of the backward launch that consumes that problem array
        gbufs, ginit = {}, set()
        lib = N_.lib()
        F32_, hdt = N_.F32, (opd if self.use_tc else N_.F32)

        def gact(a):
            """fp32 gradient buffer of a residual-stream tensor"""
            if id(a.buf) not in gbufs:
                gbufs[id(a.buf)] = P.buf("g_act", Nf * a.H * a.W * a.C * 4)
            return gbufs[id(a.buf)]

        def acc(a):
            """1 once the gradient buffer of `a` holds a contribution (later writers accumulate, the first one overwrites)"""
            k_, r_ = id(a.buf), 0
            if k_ in ginit:
                r_ = 1
            ginit.add(k_)
            return r_

        def to_op(g, Cc, Hh, Ww, n=None, up=0, biases=()):
            """fp32 gradient -> operand-dtype copy feeding dgrad / wgrad (up = 2: zero insertion for a stride-2 conv).  `biases`:
            bias parameters of the conv whose output gradient this is — their gradient (the column sums) falls out of the same
            read (fp32 atomics into the zeroed flat gradient buffer)."""
            f_ = 2 if up else 1
            o_ = P.buf("g_op", (n or Nf) * Hh * f_ * Ww * f_ * Cc * osz)
            assert not (biases and (up or Cc > 1024))
            P.op("fdm_cast", N_.CastArgs, x=g, out=o_, N=n or Nf, H=Hh, W=Ww, C=Cc, upsample=up, op_dtype=opd,
                 colsum=pg(biases[0]) if biases else None, colsum2=pg(biases[1]) if len(biases) > 1 else None)
            return o_

        preop = {}  # id(activation buffer) -> operand-dtype copy of its FINAL gradient, already written (with the bias sums) by the
        #             GroupNorm backward that was the last contributor to it

        def get_op(act):
            """operand-dtype copy of the complete gradient of `act` + the bias gradient of its producing conv"""
            if id(act.buf) in preop:
                return preop[id(act.buf)]
            return to_op(gact(act), act.C, act.H, act.W, biases=act.biases)

        def dgrad(gy, Cg, Hg, Wg, w, Co, k, out_op=None, out_f32=None, resid=None, n=None):
            """gradient wrt a stride-1 conv's input: fdm_conv over the rotated / channel-swapped weights"""
            tc = self.use_tc and opd == N_.BF16 and self.tc_ok(Cg, 0, Co, k, 1, 0, Hg, Wg) and Co % 4 == 0
            fl = 2 * (n or Nf) * Hg * Wg * Co * k * k * Cg
            P.bflops += fl
            P.op("fdm_conv", N_.ConvArgs, a0=gy, w0=pack_dgrad(w, tc), a1=None, w1=None, bias=None, resid=resid,
                 y_f32=out_f32, y_op=out_op, stats=None, N=n or Nf, Hin=Hg, Win=Wg, C0=Cg, C1=0, Cout=Co, ksize=k, stride=1,
                 upsample=0, a_dtype=opd, op_dtype=opd, out_nchw=0, engine=N_.CONV_TC if tc else N_.CONV_SIMT)

        def wgrad(a, a_dtype, Cs, Cw, Hin, Win, gy, Co, k, stride, w, biases=(), n=None, dw=None):
            """dW (PyTorch layout, into the flat parameter-gradient buffer unless `dw` names a scratch buffer) and the bias
            gradient(s); a is None: bias gradient only"""
            fields = dict(N=n or Nf, Hin=Hin, Win=Win, C=Cs, Cw=Cw, Cout=Co, ksize=k, stride=stride, a_dtype=a_dtype,
                          dy_dtype=opd, engine=N_.CONV_TC if self.use_tc else N_.CONV_SIMT)
            need = int(lib.fdm_conv_wgrad_workspace(C.byref(N_.ConvWgradArgs(**fields))))
            P.wg_ws.nbytes = max(P.wg_ws.nbytes, (need + 255) // 256 * 256)
            pad_ = k // 2
            P.bflops += 2 * (n or Nf) * ((Hin + 2 * pad_ - k) // stride + 1) * ((Win + 2 * pad_ - k) // stride + 1) * Co * k * k * Cw
            P.bside.add(len(P.bops))
            P.op("fdm_conv_wgrad", N_.ConvWgradArgs, a=a, dy=gy, dw=(dw if dw is not None else pg(w)) if a is not None else None,
                 dbias=pg(biases[0]) if biases else None,
                 dbias2=pg(biases[1]) if len(biases) > 1 else None, workspace=P.wg_ws, workspace_bytes=need, **fields)

        def gn_bwd(xa, xb, gn, foff, dy_op, dy_f32, draw, silu, last=False, dpass=None, dropf=None):
            """`last`: this GroupNorm is the LAST contributor (in backward order) to xa's gradient — true for the first forward
            consumer of a tensor — so the launch also emits the operand copy + bias sums its producer needs (checked after the
            schedule is complete: no later launch may write that gradient).  `dropf`: the dropout fields of the forward launch,
            whose mask the backward regenerates."""
            Cc = xa.C + (xb.C if xb else 0)
            ab_ = P.bzero("gn_ab", Nf * Cc * 16)
            gop = None
            if last:
                gop = P.buf("g_op", Nf * xa.H * xa.W * xa.C * osz)
                preop[id(xa.buf)] = gop
                fused_checks.append((len(P.bops), gact(xa)))
            fields = dict(xa=xa.buf, xb=xb.buf if xb else None, stats_a=xa.st,
                          stats_b=xb.st if xb else None, gamma=f32(gn.weight), beta=f32(gn.bias), film=cond if foff is not None else None,
                          dy_op=dy_op, dy_f32=dy_f32, draw_op=draw, gxa=gact(xa), gxb=gact(xb) if xb else None, ab=ab_,
                          dgamma=pg(gn.weight), dbeta=pg(gn.bias), dfilm=dcond if foff is not None else None, N=Nf, HW=xa.H * xa.W,
                          Ca=xa.C, Cb=xb.C if xb else 0, T=T, film_stride=cond_cols if foff is not None else 0,
                          film_off=foff if foff is not None else 0, silu=silu, op_dtype=opd, acc_a=acc(xa),
                          acc_b=acc(xb) if xb else 0, eps=gn.eps, dpass_a=dpass, gop_a=gop,
                          cs_a=pg(xa.biases[0]) if (gop is not None and xa.biases) else None,
                          cs2_a=pg(xa.biases[1]) if (gop is not None and len(xa.biases) > 1) else None, **(dropf or {}))
            # sums + apply on the main chain; the parameter-gradient launch (dgamma, dbeta, FiLM scale/shift gradients) only reads
            # the sums and feeds parameter gradients / the conditioning-path backward at the very end: side stream
            P.op("fdm_gn_bwd", N_.GnBwdArgs, phases=5, **fields)
            P.bside.add(len(P.bops))
            P.op("fdm_gn_bwd", N_.GnBwdArgs, phases=2, **fields)

        fused_checks = []  # (index of the fusing launch in bops, gradient buffer) for the post-compile safety check
        if train:
            P.bflops = 0
            P.wg_ws = P.buf("wgrad_ws", 256)
            dcond = P.buf("dcond", B * cond_cols * 4)
            dRb = {}
            for ab in attn_blocks:
                for which in ("rpe_q", "rpe_k", "rpe_v"):
                    dRb[(id(ab), which)] = P.bzero("dR", B * T * T * ab.channels * 4)

            def cond_bwd():
                P.bjoin_before = len(P.bops)  # consumes dcond (written on the side stream by the GroupNorm parameter launches)
                BTT = B * T * T
                rp = []
                for ab in attn_blocks:
                    Cc = ab.channels
                    for which in ("rpe_q", "rpe_k", "rpe_v"):
                        net, key = getattr(ab.temporal_attention, which).rpe_net, (id(ab), which)
                        g_ = to_op(dRb[key], Cc, 1, 1, n=BTT, biases=(net.out.bias,))
                        dh = P.buf("rpe_dhid", BTT * Cc * osz)
                        dgrad(g_, Cc, 1, 1, net.out.weight, Cc, 1, out_op=dh, n=BTT)
                        wgrad(hid[key], hdt, Cc, Cc, 1, 1, g_, Cc, 1, 1, net.out.weight, n=BTT)
                        rp.append(dict(wd=f32(net.embed_distances.weight), bd=f32(net.embed_distances.bias), dhidden=dh,
                                       dwd=pg(net.embed_distances.weight), dbd=pg(net.embed_distances.bias), C=Cc,
                                       te_off=te_off[key]))
                if rp:
                    dev_ = th.zeros(len(rp) * C.sizeof(N_.RpeHiddenBwdProblem), dtype=th.uint8, device=device)
                    P.pending.append((dev_, N_.RpeHiddenBwdProblem, rp))
                    P.pending_at[len(P.pending) - 1] = len(P.bops)
                    P.op("fdm_rpe_hidden_bwd", N_.RpeHiddenBwdArgs, te=cond, frame_indices=P.fi, problems=dev_, dte=dcond,
                         B=B, T=T, te_stride=cond_cols, count=len(rp), max_C=max(r_["C"] for r_ in rp), dhidden_dtype=opd)

                def lin_bwd(problems):
                    dev_ = th.zeros(len(problems) * C.sizeof(N_.LinearBwdProblem), dtype=th.uint8, device=device)
                    P.pending.append((dev_, N_.LinearBwdProblem, problems))
                    P.pending_at[len(P.pending) - 1] = len(P.bops)
                    P.op("fdm_grouped_linear_bwd", N_.GroupedLinearBwdArgs, problems=dev_, count=len(problems),
                         max_M=max(q_["M"] for q_ in problems), max_Nout=max(q_["Nout"] for q_ in problems),
                         max_K=max(q_["K"] for q_ in problems))
                parts = P.buf("demb_parts", len(film_probs) * B * ted * 4)
                lin_bwd([dict(x=emb, w=f32(q_["lin"].weight), dy=(dcond, q_["off"] * 4), dw=pg(q_["lin"].weight),
                              db=pg(q_["lin"].bias), dx_part=(parts, i_ * B * ted * 4), M=B, K=ted, Nout=q_["Nout"], ldx=ted,
                              ldy=cond_cols, silu_in=q_["silu_in"]) for i_, q_ in enumerate(film_probs)])
                demb = P.buf("demb", B * ted * 4)
                P.op("fdm_sum_parts", N_.SumPartsArgs, parts=parts, out=demb, part_stride=B * ted, n=B * ted,
                     count=len(film_probs), accumulate=0)
                dh1 = P.buf("dtime_h1", B * ted * 4)
                lin_bwd([dict(x=h1, w=f32(te2.weight), dy=demb, dw=pg(te2.weight), db=pg(te2.bias), dx_part=dh1, M=B, K=ted,
                              Nout=ted, ldx=ted, ldy=ted, silu_in=1)])
                lin_bwd([dict(x=temb, w=f32(te0.weight), dy=dh1, dw=pg(te0.weight), db=pg(te0.bias), dx_part=None, M=B, K=mc,
                              Nout=ted, ldx=mc, ldy=ted, silu_in=0)])
            P.tape.append(cond_bwd)

        # ---------------- network body
        # bf16 mode: the stem conv runs on tcgen05 over a bf16 copy of the network input, channels zero-padded to 8
        stem_tc = self.use_tc and self.tc_ok(8, 0, m.model_channels, 3, 1, 0, H, W) and Cin <= 8
        if stem_tc:
            xin = P.buf("xin", Nf * H * W * 8 * 2)
            P.op("fdm_input_prep", N_.InputPrepArgs, x=P.x, x0=P.x0, obs_mask=P.obs, xin=None, xin_bf16=xin, N=Nf, C=Cin - 1,
                 H=H, W=W, Cpad=8)
        else:
            xin = P.buf("xin", Nf * H * W * Cin * 4)
            P.op("fdm_input_prep", N_.InputPrepArgs, x=P.x, x0=P.x0, obs_mask=P.obs, xin=xin, xin_bf16=None, N=Nf, C=Cin - 1,
                 H=H, W=W, Cpad=0)

        class Act:  # residual-stream tensor: fp32 NHWC + its GroupNorm statistics (+ optional bf16 operand copy)
            def __init__(s, buf, st, Cc, Hh, Ww):
                s.buf, s.st, s.C, s.H, s.W, s.op = buf, st, Cc, Hh, Ww, None
                s.biases = ()  # bias parameters of the conv that produces this tensor (their gradient = column sums of its gradient)

        def with_op_copy(act):
            """Ask the producing conv to also store a bf16 copy (a stride-2 Downsample conv reads it directly: no cast pass)."""
            act.op = P.buf("act_op", Nf * act.H * act.W * act.C * osz)
            return act.op

        def new_act(name, Cc, Hh, Ww):
            return Act(P.buf(name, Nf * Hh * Ww * Cc * 4), P.stats(name, Nf, Cc), Cc, Hh, Ww)

        def res_block(rb, xa, xb=None, want_op=False):
            Hh, Ww = xa.H, xa.W
            Ci = xa.C + (xb.C if xb else 0)
            Co = rb.out_channels
            hw = Hh * Ww
            has_skip = not isinstance(rb.skip_connection, nn.Identity)
            a1 = P.buf("res_a1", Nf * hw * Ci * osz)
            raw = P.buf("res_raw", Nf * hw * Ci * osz) if has_skip else None
            gn, c1 = rb.in_layers[0], rb.in_layers[2]
            P.op("fdm_gn_apply", N_.GnApplyArgs, xa=xa.buf, xb=xb.buf if xb else None, stats_a=xa.st,
                 stats_b=xb.st if xb else None, gamma=f32(gn.weight), beta=f32(gn.bias), film=None, out_op=a1, out_f32=None,
                 raw_op=raw, N=Nf, HW=hw, Ca=xa.C, Cb=xb.C if xb else 0, T=T, film_stride=0, film_off=0, silu=1,
                 op_dtype=opd, eps=gn.eps)
            # the first conv's output is read by ONE consumer, the second GroupNorm: inference plans in bf16 mode store it once, in
            # bf16 (statistics still come from the fp32 accumulators in the conv epilogue): 6 instead of 10 bytes per element through
            # conv epilogue + GN-apply.  Training plans keep it in fp32 (the GroupNorm backward re-reads it).
            h1_bf16 = self.use_tc and not train
            if h1_bf16:
                h1_ = Act(P.buf("res_h1_op", Nf * hw * Co * osz), P.stats("res_h1", Nf, Co), Co, Hh, Ww)
                conv(a1, Ci, Hh, Ww, c1.weight, Co, 3, bias=f32(c1.bias), y_op=h1_.buf, stats=h1_.st)
            else:
                h1_ = new_act("res_h1", Co, Hh, Ww)
                conv(a1, Ci, Hh, Ww, c1.weight, Co, 3, bias=f32(c1.bias), y_f32=h1_.buf, stats=h1_.st)
            h1_.biases = (c1.bias,)
            gn2, c2 = rb.out_layers[0], rb.out_layers[3]
            a2 = P.buf("res_a2", Nf * hw * Co * osz)
            P.res_a2.append((a2, Co, Hh, Ww))
            # dropout (train mode, p > 0): one salt per ResBlock; the backward regenerates the mask from the same fields
            dropf = dict(drop_philox=P.drop_philox, drop_p=P.drop_p, drop_salt=len(P.res_a2)) if P.drop_philox is not None else {}
            P.op("fdm_gn_apply", N_.GnApplyArgs, xa=h1_.buf, xb=None, stats_a=h1_.st, stats_b=None, gamma=f32(gn2.weight),
                 beta=f32(gn2.bias), film=cond, out_op=a2, out_f32=None, raw_op=None, N=Nf, HW=hw, Ca=Co, Cb=0, T=T,
                 film_stride=cond_cols, film_off=film_off[id(rb)], silu=1, op_dtype=opd, eps=gn2.eps, xa_bf16=1 if h1_bf16 else 0,
                 film_add=0 if m.use_scale_shift_norm else 1, **dropf)
            out = new_act("res_out", Co, Hh, Ww)
            yop = with_op_copy(out) if want_op else None
            sk = rb.skip_connection
            out.biases = (c2.bias, sk.bias) if has_skip else (c2.bias,)
            if has_skip:
                if sk.kernel_size != (1, 1):
                    raise NotImplementedError("ResBlock(use_conv=True) 3x3 skip is never built by create_model")
                conv(a2, Co, Hh, Ww, c2.weight, Co, 3, a1=raw, C1=Ci, w1=sk.weight, bias=bias_sum(c2.bias, sk.bias),
                     y_f32=out.buf, y_op=yop, stats=out.st)
            else:
                conv(a2, Co, Hh, Ww, c2.weight, Co, 3, bias=f32(c2.bias), resid=xa.buf, y_f32=out.buf, y_op=yop, stats=out.st)

            def bwd():
                g_out = gact(out)
                go = get_op(out)
                da2 = P.buf("d_a2", Nf * hw * Co * osz)
                dgrad(go, Co, Hh, Ww, c2.weight, Co, 3, out_op=da2)
                draw = None
                if has_skip:
                    wgrad(a2, opd, Co, Co, Hh, Ww, go, Co, 3, 1, c2.weight)
                    draw = P.buf("d_raw", Nf * hw * Ci * osz)
                    dgrad(go, Co, Hh, Ww, sk.weight, Ci, 1, out_op=draw)
                    wgrad(raw, opd, Ci, Ci, Hh, Ww, go, Co, 1, 1, sk.weight)
                else:
                    wgrad(a2, opd, Co, Co, Hh, Ww, go, Co, 3, 1, c2.weight)  # identity residual: g_xa += g_out inside the last gn_bwd
                gn_bwd(h1_, None, gn2, film_off[id(rb)], da2, None, None, 1, last=True, dropf=dropf)
                gh = get_op(h1_)
                da1 = P.buf("d_a1", Nf * hw * Ci * osz)
                dgrad(gh, Co, Hh, Ww, c1.weight, Ci, 3, out_op=da1)
                wgrad(a1, opd, Ci, Ci, Hh, Ww, gh, Co, 3, 1, c1.weight)
                gn_bwd(xa, xb, gn, None, da1, None, draw, 1, last=True, dpass=None if has_skip else g_out)
            if train:
                P.tape.append(bwd)
            return out

        def attention(ab, x, want_op=False):
            Cc, Hh, Ww, hw = x.C, x.H, x.W, x.H * x.W
            ta, sa = ab.temporal_attention, ab.spatial_attention
            # Inference plans in bf16 mode: the GroupNorm of each half runs in the operand path of its qkv linear (fdm_norm_linear:
            # the normalised tensor is never written) and the proj_out epilogue recomputes the residual GN(x) from x and the
            # saved statistics (fdm_conv resid_norm) — 2 launches and 24 bytes per element less per attention block.
            def nl_ok(a_mode):
                if not self.use_tc or train:
                    return False
                probe = N_.NormLinearArgs(B=B, T=T, HW=hw, K=Cc, Cout=3 * Cc, a_mode=a_mode)
                return bool(lib.fdm_norm_linear_supported(C.byref(probe)))

            def norm_qkv(src, a_mode, norm, lin, out, stats=None, tstats=None):
                P.op("fdm_norm_linear", N_.NormLinearArgs, x=src, stats=stats, tstats=tstats, gamma=f32(norm.weight),
                     beta=f32(norm.bias), w=pack_fwd(lin.weight, True), bias=f32(lin.bias), y_op=out, B=B, T=T, HW=hw, K=Cc,
                     Cout=3 * Cc, a_mode=a_mode, eps=norm.eps)
                fl = 2 * Nf * hw * 3 * Cc * Cc
                P.flops += fl
                P.conv_flops += fl

            # --- temporal: GN over (C/32 x T) per (b, pixel)
            qkv = P.buf("ta_qkv", Nf * hw * 3 * Cc * osz)
            t_fused = nl_ok(2)
            if t_fused:
                xn = None
                tst = P.buf("ta_tstats", B * hw * 32 * 2 * 4)
                norm_qkv(x.buf, 2, ta.norm, ta.qkv, qkv, tstats=tst)
            else:
                xn = P.buf("ta_xn", Nf * hw * Cc * 4)
                xn_op = P.buf("ta_xn_op", Nf * hw * Cc * osz)
                P.op("fdm_temporal_gn", N_.TemporalGnArgs, x=x.buf, gamma=f32(ta.norm.weight), beta=f32(ta.norm.bias),
                     out_f32=xn, out_op=xn_op, B=B, T=T, HW=hw, C=Cc, op_dtype=opd, eps=ta.norm.eps)
                conv(xn_op, Cc, Hh, Ww, ta.qkv.weight, 3 * Cc, 1, bias=f32(ta.qkv.bias), y_op=qkv)
            o = P.buf("ta_o", Nf * hw * Cc * osz)
            P.flops += 10 * T * T * Cc * B * hw  # QK^T, PV and the three contextual RPE einsums (rpe.py:72-83,144,166)
            ws_bytes = self._temporal_ws(B, T, Cc, ta.num_heads, hw) if (self.use_tc and not train) else None
            ws = P.buf("ta_ws", ws_bytes) if ws_bytes else None
            if ws is None and R[(id(ab), "rpe_q")] is None:
                raise NativeShapeError(f"temporal attention: no kernel takes T={T}, HW={hw}, C={Cc}, heads={ta.num_heads}")
            # return_attn_weights=True plans: the tcgen05 kernels also accumulate the head-averaged attention weights — the maps
            # RPEAttention.forward logs (rpe.py:128-130) — into zero-initialised fp32 buffers
            t_mean = s_mean = None
            if collect_attn:
                if ws is None or not self.use_tc:
                    raise NativeShapeError("attention-map logging is served by the tcgen05 attention kernels (bf16 mode)")
                t_mean = P.zeroed("ta_attn_mean", B * hw * T * T * 4)
                s_mean = P.zeroed("sa_attn_mean", Nf * hw * hw * 4)
                P.attn_maps["temporal"].append((t_mean, (B * hw, T, T)))
                P.attn_maps["spatial"].append((s_mean, (Nf, hw, hw)))
            P.op("fdm_attn_temporal", N_.AttnTemporalArgs, qkv=qkv, Rq=R[(id(ab), "rpe_q")], Rk=R[(id(ab), "rpe_k")],
                 Rv=R[(id(ab), "rpe_v")], mask=P.mask, out=o, B=B, T=T, HW=hw, C=Cc, heads=ta.num_heads,
                 qkv_dtype=opd, out_dtype=opd, Rq_op=R_op.get((id(ab), "rpe_q")) if ws else None,
                 Rk_op=R_op.get((id(ab), "rpe_k")) if ws else None, Rv_op=R_op.get((id(ab), "rpe_v")) if ws else None,
                 workspace=ws, workspace_bytes=ws_bytes or 0, attn_mean=t_mean)
            if ws is not None:
                P.temporal_attn_maps.append((ws, B, T, hw, Cc, ta.num_heads))
            y = new_act("ta_y", Cc, Hh, Ww)
            y.biases = (ta.proj_out.bias,)
            if t_fused:
                conv(o, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, bias=f32(ta.proj_out.bias), resid=x.buf, y_f32=y.buf, stats=y.st,
                     resid_norm=2, rn_T=T, rn_eps=ta.norm.eps, rn_tstats=tst, rn_gamma=f32(ta.norm.weight),
                     rn_beta=f32(ta.norm.bias))
            else:
                conv(o, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, bias=f32(ta.proj_out.bias), resid=xn, y_f32=y.buf, stats=y.st)
            # --- spatial: plain per-frame GroupNorm, attention over the pixels of each frame
            qkv2 = P.buf("sa_qkv", Nf * hw * 3 * Cc * osz)
            s_fused = nl_ok(1)
            if s_fused:
                yn = None
                norm_qkv(y.buf, 1, sa.norm, sa.qkv, qkv2, stats=y.st)
            else:
                yn = P.buf("sa_yn", Nf * hw * Cc * 4)
                yn_op = P.buf("sa_yn_op", Nf * hw * Cc * osz)
                P.op("fdm_gn_apply", N_.GnApplyArgs, xa=y.buf, xb=None, stats_a=y.st, stats_b=None, gamma=f32(sa.norm.weight),
                     beta=f32(sa.norm.bias), film=None, out_op=yn_op, out_f32=yn, raw_op=None, N=Nf, HW=hw, Ca=Cc, Cb=0, T=T,
                     film_stride=0, film_off=0, silu=0, op_dtype=opd, eps=sa.norm.eps)
                conv(yn_op, Cc, Hh, Ww, sa.qkv.weight, 3 * Cc, 1, bias=f32(sa.qkv.bias), y_op=qkv2)
            o2 = P.buf("sa_o", Nf * hw * Cc * osz)
            P.flops += 4 * hw * hw * Cc * Nf
            # training: the tcgen05 forward also saves the log-sum-exp of every score row for the tcgen05 backward kernels
            sa_lse = P.buf("sa_lse", Nf * sa.num_heads * hw * 4) if (train and self.use_tc) else None
            P.op("fdm_attn_spatial", N_.AttnSpatialArgs, qkv=qkv2, out=o2, N=Nf, L=hw, C=Cc, heads=sa.num_heads,
                 qkv_dtype=opd, out_dtype=opd, engine=0 if self.use_tc else 1, lse=sa_lse, attn_mean=s_mean)
            z = new_act("sa_z", Cc, Hh, Ww)
            z.biases = (sa.proj_out.bias,)
            if s_fused:
                conv(o2, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, bias=f32(sa.proj_out.bias), resid=y.buf, y_f32=z.buf,
                     y_op=with_op_copy(z) if want_op else None, stats=z.st, resid_norm=3, rn_eps=sa.norm.eps, rn_stats=y.st,
                     rn_gamma=f32(sa.norm.weight), rn_beta=f32(sa.norm.bias))
            else:
                conv(o2, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, bias=f32(sa.proj_out.bias), resid=yn, y_f32=z.buf,
                     y_op=with_op_copy(z) if want_op else None, stats=z.st)

            def bwd():
                n_tok = Nf * hw
                # spatial half: z = proj(o2) + yn ; o2 = attn(qkv2) ; qkv2 = qkv(yn_op) ; yn = GN(y)
                g_z = gact(z)
                gz = get_op(z)
                do2 = P.buf("d_sa_o", n_tok * Cc * osz)
                dgrad(gz, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, out_op=do2)
                wgrad(o2, opd, Cc, Cc, Hh, Ww, gz, Cc, 1, 1, sa.proj_out.weight)
                dqkv2 = P.buf("d_sa_qkv", n_tok * 3 * Cc * osz)
                P.bflops += 10 * hw * hw * Cc * Nf
                P.op("fdm_attn_spatial_bwd", N_.AttnSpatialBwdArgs, qkv=qkv2, out=o2, dout=do2, dqkv=dqkv2,
                     lse=sa_lse if sa_lse is not None else P.at_lse, dsum=P.at_dsum, N=Nf, L=hw, C=Cc, heads=sa.num_heads,
                     dtype=opd, lse_from_forward=1 if sa_lse is not None else 0)
                P.at_rows = max(P.at_rows, Nf * sa.num_heads * hw)
                dyn = P.buf("d_sa_yn", n_tok * Cc * osz)
                dgrad(dqkv2, 3 * Cc, Hh, Ww, sa.qkv.weight, Cc, 1, out_op=dyn)
                wgrad(yn_op, opd, Cc, Cc, Hh, Ww, dqkv2, 3 * Cc, 1, 1, sa.qkv.weight, (sa.qkv.bias,))
                gn_bwd(y, None, sa.norm, None, dyn, g_z, None, 0, last=True)
                # temporal half: y = proj(o) + xn ; o = attn_rpe(qkv, R) ; qkv = qkv(xn_op) ; xn = temporalGN(x)
                g_y = gact(y)
                gy = get_op(y)
                do = P.buf("d_ta_o", n_tok * Cc * osz)
                dgrad(gy, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, out_op=do)
                wgrad(o, opd, Cc, Cc, Hh, Ww, gy, Cc, 1, 1, ta.proj_out.weight)
                dqkv = P.buf("d_ta_qkv", n_tok * 3 * Cc * osz)
                P.bflops += 25 * T * T * Cc * B * hw
                P.op("fdm_attn_temporal_bwd", N_.AttnTemporalBwdArgs, qkv=qkv, out=o, Rq=R[(id(ab), "rpe_q")],
                     Rk=R[(id(ab), "rpe_k")], Rv=R[(id(ab), "rpe_v")], mask=P.mask, dout=do, dqkv=dqkv,
                     dRq=dRb[(id(ab), "rpe_q")], dRk=dRb[(id(ab), "rpe_k")], dRv=dRb[(id(ab), "rpe_v")], lse=P.at_lse,
                     dsum=P.at_dsum, B=B, T=T, HW=hw, C=Cc, heads=ta.num_heads, dtype=opd)
                P.at_rows = max(P.at_rows, B * ta.num_heads * T * hw)
                dxn = P.buf("d_ta_xn", n_tok * Cc * osz)
                dgrad(dqkv, 3 * Cc, Hh, Ww, ta.qkv.weight, Cc, 1, out_op=dxn)
                wgrad(xn_op, opd, Cc, Cc, Hh, Ww, dqkv, 3 * Cc, 1, 1, ta.qkv.weight, (ta.qkv.bias,))
                P.op("fdm_temporal_gn_bwd", N_.TemporalGnBwdArgs, x=x.buf, gamma=f32(ta.norm.weight), dy_op=dxn, dy_f32=g_y,
                     gx=gact(x), dgamma=pg(ta.norm.weight), dbeta=pg(ta.norm.bias), B=B, T=T, HW=hw, C=Cc, op_dtype=opd,
                     accumulate=acc(x), eps=ta.norm.eps)
            if train:
                P.tape.append(bwd)
            return z

        def resample(layer, x, down, want_op=False):
            cv = layer.op if down else layer.conv
            Ho, Wo = (x.H // 2, x.W // 2) if down else (x.H * 2, x.W * 2)
            out = new_act("down" if down else "up", x.C, Ho, Wo)
            out.biases = (cv.bias,)
            Hc, Wc = (x.H, x.W) if down else (Ho, Wo)  # spatial size of the conv's input
            a = None
            if not down and not train and self.up_tc_ok(x.C, x.H, x.W):
                # inference: four 2x2-tap phase convs over the LOW-resolution operand copy (4/9 of the FLOPs, a 4x smaller cast)
                a = x.op
                if a is None:
                    a = P.buf("resample_a", Nf * x.H * x.W * x.C * osz)
                    P.op("fdm_cast", N_.CastArgs, x=x.buf, out=a, N=Nf, H=x.H, W=x.W, C=x.C, upsample=0, op_dtype=opd, colsum=None,
                         colsum2=None)
                conv(a, x.C, x.H, x.W, cv.weight, x.C, 3, upsample=1, bias=f32(cv.bias), y_f32=out.buf, stats=out.st,
                     y_op=with_op_copy(out) if want_op else None)
            elif (self.use_tc and self.tc_ok(x.C, 0, x.C, 3, 2 if down else 1, 0, Ho, Wo)) or (train and not down):
                if down and x.op is not None:
                    a = x.op  # the producing conv already stored the bf16 operand copy
                else:
                    # bf16 operand copy of the fp32 stream (nearest x2 upsample folded into the cast, unet.py:85), then tcgen05
                    a = P.buf("resample_a", Nf * Hc * Wc * x.C * osz)
                    P.op("fdm_cast", N_.CastArgs, x=x.buf, out=a, N=Nf, H=x.H, W=x.W, C=x.C, upsample=0 if down else 1,
                         op_dtype=opd, colsum=None, colsum2=None)
                conv(a, x.C, Hc, Wc, cv.weight, x.C, 3, stride=2 if down else 1, bias=f32(cv.bias), y_f32=out.buf,
                     stats=out.st, y_op=with_op_copy(out) if (want_op and not train) else None)
            else:
                # the CUDA-core engine gathers straight from the fp32 stream (stride 2 / folded nearest upsample)
                conv(x.buf, x.C, x.H, x.W, cv.weight, x.C, 3, stride=2 if down else 1, upsample=0 if down else 1,
                     bias=f32(cv.bias), y_f32=out.buf, stats=out.st, a_dtype=N_.F32)

            def bwd():
                Cc = x.C
                g_out = gact(out)
                go = get_op(out)
                if down:
                    # dgrad of the stride-2 conv = stride-1 conv over the zero-inserted gradient, accumulated in place into g_x
                    z_ = to_op(g_out, Cc, Ho, Wo, up=2)
                    gx = gact(x)
                    dgrad(z_, Cc, Hc, Wc, cv.weight, Cc, 3, out_f32=gx, resid=gx if acc(x) else None)
                    if self.use_tc and a is not None:
                        # tcgen05 wgrad is stride-1: the zero-inserted gradient against the full-resolution input is the same sum
                        wgrad(a, opd, Cc, Cc, Hc, Wc, z_, Cc, 3, 1, cv.weight)
                    else:
                        wgrad(a if a is not None else x.buf, opd if a is not None else F32_, Cc, Cc, Hc, Wc, go, Cc, 3, 2,
                              cv.weight)
                else:
                    da = P.buf("d_up_a", Nf * Ho * Wo * Cc * osz)
                    dgrad(go, Cc, Ho, Wo, cv.weight, Cc, 3, out_op=da)
                    wgrad(a, opd, Cc, Cc, Ho, Wo, go, Cc, 3, 1, cv.weight)
                    P.op("fdm_accum", N_.AccumArgs, src=da, dst=gact(x), N=Nf, H=x.H, W=x.W, C=Cc, pool=1, src_dtype=opd,
                         accumulate=acc(x))
            if train:
                P.tape.append(bwd)
            return out

        names = {id(mod): name for name, mod in m.named_modules()}

        def run_stage(stage, h, skip=None, feeds_downsample=False):
            layers = list(stage)
            for li, layer in enumerate(layers):
                want_op = feeds_downsample and li == len(layers) - 1 and self.use_tc
                # inference: the phase-mode upsample conv reads the low-resolution bf16 operand — let the producing conv store it
                # (one more epilogue store instead of a cast launch)
                if (not train and h is not None and li + 1 < len(layers) and isinstance(layers[li + 1], Upsample)
                        and isinstance(layer, (ResBlock, FactorizedAttentionBlock))
                        and self.up_tc_ok(getattr(layer, "out_channels", h.C), h.H, h.W)):
                    want_op = True
                if isinstance(layer, nn.Conv2d):  # stem
                    out = new_act("stem", layer.out_channels, H, W)
                    out.biases = (layer.bias,)
                    if stem_tc:
                        conv(xin, 8, H, W, layer.weight, layer.out_channels, 3, bias=f32(layer.bias), y_f32=out.buf,
                             y_op=with_op_copy(out) if want_op else None, stats=out.st, a_dtype=N_.BF16, flop_c0=Cin)
                    else:
                        conv(xin, Cin, H, W, layer.weight, layer.out_channels, 3, bias=f32(layer.bias), y_f32=out.buf,
                             stats=out.st, a_dtype=N_.F32)
                    h = out

                    def bwd(layer=layer, out=out):
                        go = get_op(out)
                        if stem_tc and layer.out_channels % 64 == 0:
                            # tcgen05 wgrad wants >= 64 stored input channels: a zero-padded bf16 copy of the network input
                            # (7/8 of the MMA rows are zeros — still ~20x faster than CUDA cores on the 128-px model)
                            xin64 = P.buf("xin64", Nf * H * W * 64 * 2)
                            P.op("fdm_input_prep", N_.InputPrepArgs, x=P.x, x0=P.x0, obs_mask=P.obs, xin=None, xin_bf16=xin64,
                                 N=Nf, C=Cin - 1, H=H, W=W, Cpad=64)
                            wgrad(xin64, N_.BF16, 64, Cin, H, W, go, layer.out_channels, 3, 1, layer.weight)
                            return
                        wgrad(xin, N_.BF16 if stem_tc else F32_, 8 if stem_tc else Cin, Cin, H, W, go, layer.out_channels, 3, 1,
                              layer.weight)
                    if train:
                        P.tape.append(bwd)
                elif isinstance(layer, ResBlock):
                    h = res_block(layer, h, skip, want_op=want_op)
                    skip = None
                elif isinstance(layer, FactorizedAttentionBlock):
                    h = attention(layer, h, want_op=want_op)
                elif isinstance(layer, Downsample):
                    h = resample(layer, h, True, want_op=want_op)
                elif isinstance(layer, Upsample):
                    h = resample(layer, h, False, want_op=want_op)
                else:
                    raise NotImplementedError(type(layer))
                P.taps[names[id(layer)]] = (h.buf, h.C, h.H, h.W)
            return h

        h, hs = None, []
        in_stages = list(m.input_blocks)
        for si, stage in enumerate(in_stages):
            nxt = in_stages[si + 1] if si + 1 < len(in_stages) else None
            feeds = nxt is not None and len(nxt) == 1 and isinstance(nxt[0], Downsample)
            h = run_stage(stage, h, feeds_downsample=feeds)   # pushed as a U-Net skip
            hs.append(h)
        h = run_stage(m.middle_block, h)
        for stage in m.output_blocks:
            h = run_stage(stage, h, hs.pop())
        gn, cv = m.out[0], m.out[2]
        a = P.buf("head_a", Nf * H * W * h.C * osz)
        P.op("fdm_gn_apply", N_.GnApplyArgs, xa=h.buf, xb=None, stats_a=h.st, stats_b=None, gamma=f32(gn.weight),
             beta=f32(gn.bias), film=None, out_op=a, out_f32=None, raw_op=None, N=Nf, HW=H * W, Ca=h.C, Cb=0, T=T,
             film_stride=0, film_off=0, silu=1, op_dtype=opd, eps=gn.eps)
        conv(a, h.C, H, W, cv.weight, m.out_channels, 3, bias=f32(cv.bias), y_f32=P.eps, out_nchw=1)

        if train:
            h_last, head_a, Co_ = h, a, m.out_channels
            P.geps = P.buf("geps", Nf * Co_ * H * W * 4, True)
            P.at_rows = 1
            P.at_lse, P.at_dsum = P.buf("attn_lse", 256), P.buf("attn_dsum", 256)

            def head_bwd():
                tc_head = self.use_tc and self.tc_ok(8, 0, h_last.C, 3, 1, 0, H, W) and Co_ <= 8
                Cp = 8 if tc_head else Co_
                ge_p = P.buf("geps_op", Nf * H * W * Cp * osz)
                P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge_p, N=Nf, C=Co_, H=H, W=W, Cpad=Cp, op_dtype=opd)
                ge = ge_p
                if Cp != Co_:
                    ge = P.buf("geps_op_true", Nf * H * W * Co_ * osz)
                    P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge, N=Nf, C=Co_, H=H, W=W, Cpad=Co_, op_dtype=opd)
                da = P.buf("d_head_a", Nf * H * W * h_last.C * osz)
                dgrad(ge_p, Cp, H, W, cv.weight, h_last.C, 3, out_op=da)
                if tc_head and h_last.C % 64 == 0:
                    # same trick on the output side: the eps gradient zero-padded to 64 channels feeds the tcgen05 wgrad; the first
                    # Co_ rows of its [64][C][3][3] result are the head's weight gradient
                    ge64 = P.buf("geps_op64", Nf * H * W * 64 * osz)
                    P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge64, N=Nf, C=Co_, H=H, W=W, Cpad=64, op_dtype=opd)
                    dw64 = P.buf("head_dw64", 64 * h_last.C * 9 * 4)
                    wgrad(head_a, opd, h_last.C, h_last.C, H, W, ge64, 64, 3, 1, cv.weight, (), dw=dw64)
                    P.bside.add(len(P.bops))  # consumes the side-stream wgrad's scratch: same stream
                    P.op("fdm_sum_parts", N_.SumPartsArgs, parts=dw64, out=pg(cv.weight), part_stride=0, n=Co_ * h_last.C * 9,
                         count=1, accumulate=0)
                    wgrad(None, opd, h_last.C, h_last.C, H, W, ge, Co_, 3, 1, cv.weight, (cv.bias,))
                else:
                    wgrad(head_a, opd, h_last.C, h_last.C, H, W, ge, Co_, 3, 1, cv.weight, (cv.bias,))
                gn_bwd(h_last, None, gn, None, da, None, None, 1, last=True)
            P.tape.append(head_bwd)
            P.cur = P.bops
            for emit in reversed(P.tape):
                emit()
            P.cur = P.ops
            # a fused operand copy is only valid if nothing writes that gradient afterwards
            grad_out_fields = ("gxa", "gxb", "dst", "y_f32", "gx")
            for idx, gbuf in fused_checks:
                for j in range(idx + 1, len(P.bops)):
                    fn_j, _, f_j = P.bops[j]
                    if fn_j == "fdm_gn_bwd" and f_j.get("phases") == 2:
                        continue  # parameter-gradient launch: does not write activation gradients
                    if any(f_j.get(k) is gbuf for k in grad_out_fields):
                        raise AssertionError(f"backward schedule: {fn_j} (#{j}) writes a gradient after its operand copy was fused (#{idx})")
            P.grad_buckets = self._grad_buckets(P, params)
            P.at_lse.nbytes = P.at_dsum.nbytes = (P.at_rows * 4 + 255) // 256 * 256
            dgrad_modes = (N_.PACK_TC_DGRAD, N_.PACK_SIMT_DGRAD)
            groups = [(pack_fields, [q_ for q_ in P.pack_problems if pack_fields_d is None or q_[6] not in dgrad_modes])]
            if pack_fields_d is not None:
                groups.append((pack_fields_d, [q_ for q_ in P.pack_problems if q_[6] in dgrad_modes]))
            for fields_, probs_ in groups:
                dev_ = th.zeros(max(len(probs_), 1) * C.sizeof(N_.PackProblem), dtype=th.uint8, device=device)
                P.pending.append((dev_, N_.PackProblem, [dict(src=s_, src2=s2_, dst=d_, co=co_, ci=ci_, k=k_, mode=mo_)
                                                        for s_, s2_, d_, co_, ci_, k_, mo_ in probs_]))
                fields_.update(problems=dev_, count=len(probs_),
                               max_elems=max([co_ * ci_ * k_ * k_ for _, _, _, co_, ci_, k_, _ in probs_] or [1]))

        # The whole conditioning chain — timestep embedding, time MLP, FiLM / RPE time projections, RPENet tables: everything that
        # depends only on (t, frame_indices) — runs on a side stream and is joined before its first consumer on the main stream
        # (the first FiLM GroupNorm-apply, or the first temporal attention), so it overlaps input prep, stem and the first convs
        # instead of heading every step.  Inside a CUDA-graph capture the fork / join become graph edges.
        cond_bufs = {id(cond)} | {id(v) for v in R.values() if v is not None} | {id(v) for v in R_op.values() if v is not None}

        def reads_cond(fields):
            for v in fields.values():
                b_ = v[0] if isinstance(v, tuple) else v
                if isinstance(b_, Buf) and id(b_) in cond_bufs:
                    return True
            return False
        if not train and P.side_end > P.side_begin:
            P.side_begin = P.temb_op
        P.join_at = next((i for i, (fn, _, f_) in enumerate(P.ops) if i >= P.side_end and reads_cond(f_)), len(P.ops))
        if th.device(device).type == "cuda" and P.side_end > P.side_begin and P.join_at >= P.side_end:
            P.side_stream = th.cuda.Stream(device)
            P.ev_fork, P.ev_join = th.cuda.Event(), th.cuda.Event()
        # skip-connection activations must stay alive until their consumer: handled by liveness (first/last use)
        P.finalize(device)
        # fill the device-side problem arrays now that pointers are known
        for dev, problems in self._pending_groups:
            arr = (N_.LinearProblem * len(problems))()
            for i, pr in enumerate(problems):
                for k in ("x", "w", "b", "y"):
                    setattr(arr[i], k, P.ptr(pr[k]))
                for k in ("M", "K", "Nout", "ldx", "ldy", "silu_in"):
                    setattr(arr[i], k, pr[k])
            dev.copy_(th.frombuffer(bytearray(bytes(arr)), dtype=th.uint8))
        if self._pending_rh is not None:
            dev, problems = self._pending_rh
            arr = (N_.RpeHiddenProblem * len(problems))()
            for i, pr in enumerate(problems):
                arr[i].wd, arr[i].bd, arr[i].hidden = P.ptr(pr["wd"]), P.ptr(pr["bd"]), P.ptr(pr["hidden"])
                arr[i].C, arr[i].te_off = pr["C"], pr["te_off"]
            dev.copy_(th.frombuffer(bytearray(bytes(arr)), dtype=th.uint8))
        self._pending_groups, self._pending_rh = [], None
        if getattr(self, "_pending_rt", None) is not None:
            blob, items = self._pending_rt
            arr = (N_.RpeTableProblem * len(items))()
            for i, it in enumerate(items):
                for k, v in it.items():
                    setattr(arr[i], k, P.ptr(v) if isinstance(v, (Buf, tuple, th.Tensor)) or v is None else v)
            host = (C.c_uint8 * blob.numel())()
            N_.check(N_.lib().fdm_rpe_tables_prepare(C.byref(arr), len(items), C.byref(host), blob.numel()), "fdm_rpe_tables_prepare")
            blob.copy_(th.frombuffer(bytearray(bytes(host)), dtype=th.uint8))
            self._pending_rt = None
        for dev, cls, items in P.pending:
            arr = (cls * len(items))()
            for i, it in enumerate(items):
                for k, v in it.items():
                    setattr(arr[i], k, P.ptr(v) if isinstance(v, (Buf, tuple, th.Tensor)) or v is None else v)
            dev.copy_(th.frombuffer(bytearray(bytes(arr)), dtype=th.uint8))
            P.keep.append(dev)
        if train:
            P.geps_view = P.view(P.geps, (B, T, m.out_channels, H, W), th.float32)
            P.n_bwd_launches = len(P.bcalls)
            if th.device(device).type == "cuda":
                P.bwd_side_stream = th.cuda.Stream(device)
                P.ev_bfork, P.ev_bjoin = th.cuda.Event(), th.cuda.Event()
        # typed views of the I/O buffers
        Cx = Cin - 1
        P.x_view = P.view(P.x, (B, T, Cx, H, W), th.float32)
        P.x0_view = P.view(P.x0, (B, T, Cx, H, W), th.float32)
        P.obs_view = P.view(P.obs, (B, T), th.float32)
        P.mask_view = P.view(P.mask, (B, T), th.float32)
        P.fi_view = P.view(P.fi, (B, T), th.int64)
        P.t_view = P.view(P.t, (B,), th.float32)
        P.t_index_view = P.view(P.t_index, (B,), th.int64)
        P.eps_view = P.view(P.eps, (B, T, m.out_channels, H, W), th.float32)
        P.n_launches = len(P.calls) + 1  # + the statistics memset
        return P

    # ------------------------------------------------------------------ execution
    def load_conditioning(self, P, x0, frame_indices, obs_mask, latent_mask):
        """Copy the per-stage inputs (constant across diffusion steps) into the plan's static buffers."""
        P.x0_view.copy_(x0)
        P.fi_view.copy_(frame_indices)
        P.obs_view.copy_(obs_mask.reshape(P.B, P.T))
        th.clamp(obs_mask.reshape(P.B, P.T) + latent_mask.reshape(P.B, P.T), max=1, out=P.mask_view)

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
        sink = getattr(self.model, "_fdm_flat_sink", None)
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
            self.load_conditioning(P, x0, frame_indices, obs_mask, latent_mask)
            P.set_t_source(None)
            P.x_view.copy_(x)
            P.t_view.copy_(timesteps.reshape(B).float())
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

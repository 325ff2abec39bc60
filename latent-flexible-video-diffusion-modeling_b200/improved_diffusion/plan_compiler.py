"""
PlanCompiler — compiles UNetVideoModel.forward (and, for training plans, its backward) for one input shape into a Plan: a flat
schedule of libfdm_sm100.so launches over the plan's arenas (engine.py).  One compiler per compile: it holds the plan, the model,
the shape, the weight source and the conditioning layout; the block emitters are its methods, each block's backward emitter next
to its forward.  Backward emitters are appended to P.tape during the forward and run in reverse once the forward is complete.
"""
import bisect
import ctypes as C
import os

import torch as th
import torch.nn as nn

from . import _native as N_
from .engine import Buf, NativeShapeError, Plan
from .nn import timestep_freqs
from .unet import Downsample, FactorizedAttentionBlock, ResBlock, Upsample


class HostWeights:
    """Inference plans: weights converted / packed on the host once, cached in engine.packed (dropped by invalidate() and
    refresh_weights())."""

    def __init__(self, engine):
        self.packed = engine.packed

    def _cached(self, key, make):
        if key not in self.packed:
            self.packed[key] = make()
        return self.packed[key]

    def f32(self, p):
        return self._cached(("f32", p.data_ptr()), lambda: p.detach().float().contiguous())

    def bias_sum(self, b0, b1):
        return self._cached(("bsum", b0.data_ptr(), b1.data_ptr()), lambda: (b0.detach().float() + b1.detach().float()).contiguous())

    def fwd(self, w, tc):
        """[co][ci][kh][kw] or [co][ci] -> tc: bf16 [tap = kw*k + kh][co_pad][ci_pad]  (K-major B operand, filter-column major taps,
        ci_pad % 64 == 0, co_pad % 16 == 0); otherwise fp32 [tap][ci][co]"""
        def make():
            w4 = w.detach().float()
            if w4.dim() == 2:
                w4 = w4[:, :, None, None]
            co, ci, kh, kw = w4.shape
            if not tc:
                return w4.permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous()
            cip, cop = (ci + 63) // 64 * 64, (co + 15) // 16 * 16
            out = th.zeros(kh * kw, cop, cip, dtype=th.bfloat16, device=w.device)
            out[:, :co, :ci] = w4.permute(3, 2, 0, 1).reshape(kh * kw, co, ci).to(th.bfloat16)
            return out
        return self._cached(("tc" if tc else "simt", w.data_ptr()), make)

    def up(self, w):
        """nearest x2 upsample + 3x3 conv (unet.py:85-93) without the upsampled tensor: output pixel (2y+a, 2x+b) sees the input rows
        y + {a-1, a} and columns x + {b-1, b}; the 3x3 weights that land on the same input pixel are summed in fp32.
        [co][ci][3][3] -> bf16 [phase = 2a + b][tap = 2s' + r'][co_pad][ci_pad]  (conv_halo.cu `up` mode, include/fdm_b200.h)"""
        def make():
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
            return out
        return self._cached(("tcup", w.data_ptr()), make)


class TrainWeights:
    """Training plans: parameters are read in place (fp32) and packed operands live in persistent tensors that ONE
    fdm_pack_weights launch refreshes at the head of every forward.  The DGRAD layouts, read only by the backward schedule, get a
    second pack launch on the RPE-table side stream once `dgrad_launch()` has emitted it."""
    DGRAD = (N_.PACK_TC_DGRAD, N_.PACK_SIMT_DGRAD)

    def __init__(self, P, device):
        self.P, self.device, self.packed = P, device, {}
        P.keep.append(self.packed)
        self.fwd_arr, self.dgrad_arr = self._pack_launch(), None

    def _pack_launch(self):
        arr = self.P.problem_array(N_.PackProblem, [], fields=lambda items: dict(
            count=len(items), max_elems=max([it["co"] * it["ci"] * it["k"] * it["k"] for it in items] or [1])))
        self.P.op("fdm_pack_weights", N_.PackWeightsArgs, problems=arr)
        return arr

    def dgrad_launch(self):
        self.dgrad_arr = self._pack_launch()

    def _pack(self, key, w, src2, shape, dtype, co, ci, k, mode):
        if key not in self.packed:
            self.packed[key] = th.zeros(shape, dtype=dtype, device=self.device)
            self.P.pack_problems.append((w, src2, self.packed[key], co, ci, k, mode))
            arr = self.dgrad_arr if (mode in self.DGRAD and self.dgrad_arr is not None) else self.fwd_arr
            arr.items.append(dict(src=w, src2=src2, dst=self.packed[key], co=co, ci=ci, k=k, mode=mode))
        return self.packed[key]

    def _pack_w(self, w, mode):
        co, ci = w.shape[0], w.shape[1]
        k = w.shape[2] if w.dim() == 4 else 1
        r16, r64 = (lambda v: (v + 15) // 16 * 16), (lambda v: (v + 63) // 64 * 64)
        shape, dty = {N_.PACK_TC_FWD: ((k * k, r16(co), r64(ci)), th.bfloat16),
                      N_.PACK_TC_DGRAD: ((k * k, r16(ci), r64(co)), th.bfloat16),
                      N_.PACK_SIMT_FWD: ((k * k, ci, co), th.float32),
                      N_.PACK_SIMT_DGRAD: ((k * k, co, ci), th.float32)}[mode]
        return self._pack((mode, id(w)), w, None, shape, dty, co, ci, k, mode)

    def f32(self, p):
        return p.detach()

    def bias_sum(self, b0, b1):
        return self._pack(("sum2", id(b0)), b0, b1, (b0.numel(),), th.float32, b0.numel(), 1, 1, N_.PACK_SUM2)

    def fwd(self, w, tc):
        return self._pack_w(w, N_.PACK_TC_FWD if tc else N_.PACK_SIMT_FWD)

    def dgrad(self, w, tc):
        return self._pack_w(w, N_.PACK_TC_DGRAD if tc else N_.PACK_SIMT_DGRAD)


class Act:
    """Residual-stream tensor: fp32 NHWC + its GroupNorm statistics (+ optional bf16 operand copy)."""

    def __init__(s, buf, st, Cc, Hh, Ww):
        s.buf, s.st, s.C, s.H, s.W, s.op = buf, st, Cc, Hh, Ww, None
        s.biases = ()  # bias parameters of the conv that produces this tensor (their gradient = column sums of its gradient)


RPE_NETS = ("rpe_q", "rpe_k", "rpe_v")


class PlanCompiler:
    def __init__(self, engine, B, T, H, W, device, train=False, collect_attn=False, drop_p=0.0):
        self.e, self.m = engine, engine.model
        self.B, self.T, self.H, self.W, self.Nf, self.device = B, T, H, W, B * T, device
        self.train, self.collect_attn = train, collect_attn
        self.use_tc, self.opd, self.osz = engine.use_tc, engine.op_dtype, engine.op_size
        self.lib = N_.lib()
        self.P = P = Plan(engine, B, T, H, W)
        P.train = train
        if train and drop_p > 0:
            P.drop_p = drop_p
            P.drop_philox = th.zeros(2, dtype=th.int64, device=device)
        self.res_blocks, self.attn_blocks = [], []
        for blk in list(self.m.input_blocks) + [self.m.middle_block] + list(self.m.output_blocks):
            for layer in blk:
                if isinstance(layer, ResBlock):
                    self.res_blocks.append(layer)
                elif isinstance(layer, FactorizedAttentionBlock):
                    self.attn_blocks.append(layer)
        # conditioning layout: one [B][cond_cols] fp32 buffer holds every FiLM projection and RPENet time embedding
        cols = 0
        self.film_off, self.te_off = {}, {}
        for rb in self.res_blocks:
            self.film_off[id(rb)] = cols
            cols += engine.film_cols * rb.out_channels
        for ab in self.attn_blocks:
            for which in RPE_NETS:
                self.te_off[(id(ab), which)] = cols
                cols += ab.channels
        self.cond_cols = cols
        self.R, self.R_op, self.hid = {}, {}, {}  # RPE output tables (fp32, bf16 operand) and hidden layers per (block, net)
        # backward state: fp32 gradient buffers of residual-stream tensors, which of them already hold a contribution, operand
        # copies of final gradients written by a fusing GroupNorm backward, and (launch, gradient) pairs of those fusions
        self.gbufs, self.ginit, self.preop, self.fused_checks = {}, set(), {}, []
        if train:
            self.params = list(self.m.parameters())
            for p_ in self.params:
                assert p_.dtype == th.float32 and p_.is_contiguous(), "training plans expect contiguous fp32 master weights"
            self.w = TrainWeights(P, device)
            self._flat_grads()
        else:
            self.w = HostWeights(engine)

    def _flat_grads(self):
        # densely packed in parameter order: ONE C++ call (unflatten_dense_tensors) turns a clone of it into the per-parameter
        # gradients — 390 Python-side narrow+view pairs per step were ~2 ms of host time on the launch-bound cfg2 step
        # 16-byte aligned slots (vectorised optimizer kernels) in gradient-COMPLETION order (optim.completion_order): the head and
        # the last output blocks first, the conditioning path (time MLP, FiLM projections, RPENets) last — a bucket of consecutive
        # slots is final once the backward schedule passes one point, so its allreduce overlaps the rest of the backward
        from .optim import model_flat_layout
        P, params = self.P, self.params
        _, offs_list, total, order, n_early = model_flat_layout(self.m)
        P.pgrad = th.zeros(total, dtype=th.float32, device=self.device)
        P.unflat, P.unflat_pick = [], [0] * len(params)  # templates for unflatten_dense_tensors (flat order) + padding stubs
        for i in order:
            p_, n_ = params[i], (params[i].numel() + 3) // 4 * 4
            P.unflat_pick[i] = len(P.unflat)
            P.unflat.append(p_)
            if n_ != p_.numel():
                P.unflat.append(th.empty(n_ - p_.numel()))
        self.offs = {id(p_): o_ for p_, o_ in zip(params, offs_list)}
        P.flat_order, P.flat_offs, P.n_early = order, offs_list, n_early

    def pg(self, p_):
        """gradient slot of a parameter in the flat buffer"""
        o = self.offs[id(p_)]
        return self.P.pgrad[o:o + p_.numel()]

    # ------------------------------------------------------------------ shape rules
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

    def up_tc_ok(self, Cc, H, W):
        """Upsample convs the halo kernel's phase mode takes (H x W = the LOW-resolution input): whole image rows per 128-pixel tile"""
        # (the 32-column tile variant is not instantiated for the phase mode)
        return self.use_tc and W in (16, 32, 64, 128) and H % (128 // W) == 0 and Cc % 8 == 0 and Cc >= 64

    def temporal_ws(self, Cc, heads, hw):
        """Workspace bytes of the tcgen05 temporal attention for this shape, or None when the CUDA-core kernel serves it.
        hw=None: is the shape family (T, head dim) taken at all (every attention map of the U-Net has HW % 16 == 0)."""
        a = N_.AttnTemporalArgs(B=self.B, T=self.T, HW=hw or 256, C=Cc, heads=heads, qkv_dtype=self.opd, out_dtype=self.opd)
        n = int(self.lib.fdm_attn_temporal_workspace(C.byref(a)))
        return n if n > 0 else None

    # ------------------------------------------------------------------ compile
    def compile(self):
        P, m, B, T, H, W, Nf = self.P, self.m, self.B, self.T, self.H, self.W, self.Nf
        Cin = m.in_channels  # includes indicator channel
        # ---------------- persistent inputs / outputs
        P.x = P.buf("x", Nf * (Cin - 1) * H * W * 4, True)
        P.x0 = P.buf("x0", Nf * (Cin - 1) * H * W * 4, True)
        P.obs = P.buf("obs", Nf * 4, True)
        P.mask = P.buf("mask", Nf * 4, True)
        P.fi = P.buf("fi", Nf * 8, True)
        P.t = P.buf("t", B * 4, True)
        P.t_index = P.buf("t_index", B * 8, True)
        P.eps = P.buf("eps", Nf * m.out_channels * H * W * 4, True)
        self.conditioning()
        self.rpe_tables()
        if self.train:
            P.bflops = 0
            P.wg_ws = P.buf("wgrad_ws", 256)
            self.dcond = P.buf("dcond", B * self.cond_cols * 4)
            self.dRb = {(id(ab), which): P.bzero("dR", B * T * T * ab.channels * 4)
                        for ab in self.attn_blocks for which in RPE_NETS}
            P.tape.append(self.conditioning_bwd)
        self.body()
        if self.train:
            self.backward()
        self.streams()
        P.finalize(self.device)
        if self.train:
            P.geps_view = P.view(P.geps, (B, T, m.out_channels, H, W), th.float32)
            P.n_bwd_launches = len(P.bcalls)
            if th.device(self.device).type == "cuda":
                P.bwd_side_stream = th.cuda.Stream(self.device)
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

    # ------------------------------------------------------------------ conditioning path
    def grouped_linear(self, problems):
        self.P.flops += sum(2 * pr["M"] * pr["K"] * pr["Nout"] for pr in problems)
        self.P.op("fdm_grouped_linear", N_.GroupedLinearArgs, problems=self.P.problem_array(N_.LinearProblem, problems),
                  count=len(problems), max_M=max(p["M"] for p in problems), max_Nout=max(p["Nout"] for p in problems),
                  max_K=max(p["K"] for p in problems))

    def conditioning(self):
        P, m, B, w = self.P, self.m, self.B, self.w
        mc, ted = m.model_channels, m.model_channels * 4
        freqs = timestep_freqs(mc).to(self.device)
        P.keep.append(freqs)
        # (persistent: the conditioning chain runs on the side stream, concurrently with main-stream launches whose buffers must
        # not alias these)
        self.temb = P.buf("temb", B * mc * 4, True)
        self.h1 = P.buf("time_h1", B * ted * 4, True)
        self.emb = P.buf("emb", B * ted * 4, True)
        self.cond = P.buf("cond", B * self.cond_cols * 4, True)  # live for the whole forward
        P.temb_op = len(P.ops)
        P.op("fdm_timestep_embedding", N_.TimestepEmbeddingArgs, t=P.t, t_index=None, t_table=None, freqs=freqs, out=self.temb,
             B=B, dim=mc)
        te0, te2 = m.time_embed[0], m.time_embed[2]
        self.grouped_linear([dict(x=self.temb, w=w.f32(te0.weight), b=w.f32(te0.bias), y=self.h1, M=B, K=mc, Nout=ted, ldx=mc,
                                  ldy=ted, silu_in=0)])
        self.grouped_linear([dict(x=self.h1, w=w.f32(te2.weight), b=w.f32(te2.bias), y=self.emb, M=B, K=ted, Nout=ted, ldx=ted,
                                  ldy=ted, silu_in=1)])
        # FiLM projections and RPENet time embeddings: (linear, column offset in cond, width, SiLU on the input)
        self.cond_lins = [(rb.emb_layers[1], self.film_off[id(rb)], self.e.film_cols * rb.out_channels, 1) for rb in self.res_blocks]
        self.cond_lins += [(getattr(ab.temporal_attention, which).rpe_net.embed_diffusion_time, self.te_off[(id(ab), which)],
                            ab.channels, 0) for ab in self.attn_blocks for which in RPE_NETS]
        self.grouped_linear([dict(x=self.emb, w=w.f32(lin.weight), b=w.f32(lin.bias), y=(self.cond, off * 4), M=B, K=ted,
                                  Nout=nout, ldx=ted, ldy=self.cond_cols, silu_in=silu) for lin, off, nout, silu in self.cond_lins])

    def rpe_tables(self):
        """RPENet hidden + output tables for every temporal attention.  bf16 mode: the C x C output linear of each net runs on
        tcgen05 (fdm_conv, 1x1 over the B*T*T rows, bf16 hidden); fp32 mode: one grouped CUDA-core launch."""
        P, B, T, w, train = self.P, self.B, self.T, self.w, self.train
        rh_probs, out_probs, nets = [], [], []
        hsz = self.osz if self.use_tc else 4
        # inference plans whose temporal attentions ALL run on tcgen05: ONE fused launch produces every bf16 table (hidden layer
        # generated in shared memory as the GEMM's A operand: rpe_tables_tc.cu) instead of fdm_rpe_hidden + one GEMM per net
        fuse_tables = (self.use_tc and not train and bool(self.attn_blocks)
                       and max(ab.channels for ab in self.attn_blocks) <= 512
                       and all(self.temporal_ws(ab.channels, ab.temporal_attention.num_heads, None) is not None
                               for ab in self.attn_blocks))
        for ab in self.attn_blocks:
            Cc = ab.channels
            for which in RPE_NETS:
                net, key = getattr(ab.temporal_attention, which).rpe_net, (id(ab), which)
                # (side-stream lifetime: never aliased with main-branch buffers)
                hb = None if fuse_tables else P.buf("rpe_hidden", B * T * T * Cc * hsz, True)
                # bf16 copies of the tables are the B operands of the tcgen05 temporal attention (attn_temporal_tc.cu); the fp32
                # tables are only kept where something still reads them: the CUDA-core kernel (shapes the tcgen05 engine does not
                # take) and the backward kernels of training plans
                # (training plans keep the CUDA-core forward: its backward kernels re-form P in fp32 from the fp32 tables, and a
                # forward that rounded P / R to bf16 would leave the analytically-zero gradients (RPE output biases: softmax shift
                # invariance) with more noise than torch's own autocast backward — measured 0.148 vs 0.14 allowed)
                tc_here = (self.use_tc and not train
                           and self.temporal_ws(ab.channels, ab.temporal_attention.num_heads, None) is not None)
                rop = P.buf("rpe_R_op", B * T * T * Cc * 2, True) if tc_here else None
                rb_ = P.buf("rpe_R", B * T * T * Cc * 4, True) if (train or not tc_here) else None
                self.hid[key], self.R[key], self.R_op[key] = hb, rb_, rop
                rh_probs.append(dict(wd=w.f32(net.embed_distances.weight), bd=w.f32(net.embed_distances.bias), hidden=hb, C=Cc,
                                     te_off=self.te_off[key]))
                if not self.use_tc:
                    out_probs.append(dict(x=hb, w=w.f32(net.out.weight), b=w.f32(net.out.bias), y=rb_, M=B * T * T, K=Cc, Nout=Cc,
                                          ldx=Cc, ldy=Cc, silu_in=0))
                nets.append((hb, Cc, net, rb_, rop))
        if fuse_tables:
            assert all(rop is not None and rb_ is None for _, _, _, rb_, rop in nets)

            def encode(arr, n):  # tensor maps + problems, encoded by the library
                host = (C.c_uint8 * int(self.lib.fdm_rpe_tables_blob_bytes(n)))()
                N_.check(self.lib.fdm_rpe_tables_prepare(C.byref(arr), n, C.byref(host), len(host)), "fdm_rpe_tables_prepare")
                return bytes(host)
            blob = P.problem_array(N_.RpeTableProblem, [
                dict(wd=q_["wd"], bd=q_["bd"], bo=w.f32(net.out.bias), w_packed=w.fwd(net.out.weight, True), out_op=rop,
                     out_f32=None, C=Cc, te_off=q_["te_off"]) for (hb, Cc, net, rb_, rop), q_ in zip(nets, rh_probs)], encode=encode)
            P.flops += sum(2 * B * T * T * Cc * Cc for _, Cc, _, _, _ in nets)
            P.rpe_table_channels = [Cc for _, Cc, _, _, _ in nets]
            P.side_begin = len(P.ops)
            P.op("fdm_rpe_tables", N_.RpeTablesArgs, te=self.cond, frame_indices=P.fi, blob=blob, count=len(nets), B=B, T=T,
                 te_stride=self.cond_cols, max_C=max(Cc for _, Cc, _, _, _ in nets))
            P.side_end = len(P.ops)
        elif rh_probs:
            P.side_begin = len(P.ops)
            P.op("fdm_rpe_hidden", N_.RpeHiddenArgs, te=self.cond, frame_indices=P.fi,
                 problems=P.problem_array(N_.RpeHiddenProblem, rh_probs), B=B, T=T, te_stride=self.cond_cols, count=len(rh_probs),
                 max_C=max(p["C"] for p in rh_probs), hidden_dtype=self.opd if self.use_tc else N_.F32)
            if train:
                # the DGRAD weight layouts are only read by the backward schedule: packed on the side stream (this branch),
                # off the forward's dependent chain
                w.dgrad_launch()
            if self.use_tc:
                for hb, Cc, net, rb_, rop in nets:
                    self.conv(hb, Cc, 1, 1, net.out.weight, Cc, 1, bias=w.f32(net.out.bias), y_f32=rb_, y_op=rop, n_frames=B * T * T)
            else:
                self.grouped_linear(out_probs)
            P.side_end = len(P.ops)

    def conditioning_bwd(self):
        P, m, B, T, w, pg, osz = self.P, self.m, self.B, self.T, self.w, self.pg, self.osz
        mc, ted = m.model_channels, m.model_channels * 4
        te0, te2 = m.time_embed[0], m.time_embed[2]
        P.bjoin_before = len(P.bops)  # consumes dcond (written on the side stream by the GroupNorm parameter launches)
        BTT = B * T * T
        rp = []
        for ab in self.attn_blocks:
            Cc = ab.channels
            for which in RPE_NETS:
                net, key = getattr(ab.temporal_attention, which).rpe_net, (id(ab), which)
                g_ = self.to_op(self.dRb[key], Cc, 1, 1, n=BTT, biases=(net.out.bias,))
                dh = P.buf("rpe_dhid", BTT * Cc * osz)
                self.dgrad(g_, Cc, 1, 1, net.out.weight, Cc, 1, out_op=dh, n=BTT)
                self.wgrad(self.hid[key], self.opd if self.use_tc else N_.F32, Cc, Cc, 1, 1, g_, Cc, 1, 1, net.out.weight, n=BTT)
                rp.append(dict(wd=w.f32(net.embed_distances.weight), bd=w.f32(net.embed_distances.bias), dhidden=dh,
                               dwd=pg(net.embed_distances.weight), dbd=pg(net.embed_distances.bias), C=Cc, te_off=self.te_off[key]))
        if rp:
            P.op("fdm_rpe_hidden_bwd", N_.RpeHiddenBwdArgs, te=self.cond, frame_indices=P.fi,
                 problems=P.problem_array(N_.RpeHiddenBwdProblem, rp), dte=self.dcond, B=B, T=T, te_stride=self.cond_cols,
                 count=len(rp), max_C=max(r_["C"] for r_ in rp), dhidden_dtype=self.opd)

        def lin_bwd(problems):
            P.op("fdm_grouped_linear_bwd", N_.GroupedLinearBwdArgs, problems=P.problem_array(N_.LinearBwdProblem, problems),
                 count=len(problems), max_M=max(q_["M"] for q_ in problems), max_Nout=max(q_["Nout"] for q_ in problems),
                 max_K=max(q_["K"] for q_ in problems))
        lins = self.cond_lins
        parts = P.buf("demb_parts", len(lins) * B * ted * 4)
        lin_bwd([dict(x=self.emb, w=w.f32(lin.weight), dy=(self.dcond, off * 4), dw=pg(lin.weight), db=pg(lin.bias),
                      dx_part=(parts, i_ * B * ted * 4), M=B, K=ted, Nout=nout, ldx=ted, ldy=self.cond_cols, silu_in=silu)
                 for i_, (lin, off, nout, silu) in enumerate(lins)])
        demb = P.buf("demb", B * ted * 4)
        P.op("fdm_sum_parts", N_.SumPartsArgs, parts=parts, out=demb, part_stride=B * ted, n=B * ted, count=len(lins), accumulate=0)
        dh1 = P.buf("dtime_h1", B * ted * 4)
        lin_bwd([dict(x=self.h1, w=w.f32(te2.weight), dy=demb, dw=pg(te2.weight), db=pg(te2.bias), dx_part=dh1, M=B, K=ted,
                      Nout=ted, ldx=ted, ldy=ted, silu_in=1)])
        lin_bwd([dict(x=self.temb, w=w.f32(te0.weight), dy=dh1, dw=pg(te0.weight), db=pg(te0.bias), dx_part=None, M=B, K=mc,
                      Nout=ted, ldx=mc, ldy=ted, silu_in=0)])

    # ------------------------------------------------------------------ convolutions
    def conv(self, a0, C0, Hin, Win, w0, Cout, k, stride=1, upsample=0, a1=None, C1=0, w1=None, bias=None, resid=None,
             y_f32=None, y_op=None, stats=None, out_nchw=0, a_dtype=None, flop_c0=None, n_frames=None, **resid_norm):
        a_dtype = self.opd if a_dtype is None else a_dtype
        Nf_ = self.Nf if n_frames is None else n_frames
        Hv, Wv = (Hin * 2, Win * 2) if upsample else (Hin, Win)
        Ho, Wo = (Hv + 2 * (k // 2) - k) // stride + 1, (Wv + 2 * (k // 2) - k) // stride + 1
        tc = a_dtype == N_.BF16 and self.tc_ok(C0, C1, Cout, k, stride, upsample, Ho, Wo) and (out_nchw or Cout % 4 == 0)
        up_tc = bool(upsample) and a_dtype == N_.BF16 and k == 3 and C0 == Cout and not self.train and self.up_tc_ok(C0, Hin, Win)
        self.P.flops += 2 * Nf_ * Ho * Wo * Cout * (k * k * (flop_c0 or C0) + C1)  # algorithmic: padded channels do not count
        pack = lambda w_: self.w.fwd(w_, tc)
        if up_tc:
            tc, pack = True, self.w.up
        self.P.op("fdm_conv", N_.ConvArgs, a0=a0, w0=pack(w0), a1=a1, w1=pack(w1) if w1 is not None else None, bias=bias,
                  resid=resid, y_f32=y_f32, y_op=y_op, stats=stats, N=Nf_, Hin=Hin, Win=Win, C0=C0, C1=C1, Cout=Cout,
                  ksize=k, stride=stride, upsample=upsample, a_dtype=a_dtype, op_dtype=self.opd, out_nchw=out_nchw,
                  engine=N_.CONV_TC if tc else N_.CONV_SIMT, **resid_norm)
        return Ho, Wo

    def dgrad(self, gy, Cg, Hg, Wg, w, Co, k, out_op=None, out_f32=None, resid=None, n=None):
        """gradient wrt a stride-1 conv's input: fdm_conv over the rotated / channel-swapped weights"""
        opd = self.opd
        tc = self.use_tc and opd == N_.BF16 and self.tc_ok(Cg, 0, Co, k, 1, 0, Hg, Wg) and Co % 4 == 0
        self.P.bflops += 2 * (n or self.Nf) * Hg * Wg * Co * k * k * Cg
        self.P.op("fdm_conv", N_.ConvArgs, a0=gy, w0=self.w.dgrad(w, tc), a1=None, w1=None, bias=None, resid=resid,
                  y_f32=out_f32, y_op=out_op, stats=None, N=n or self.Nf, Hin=Hg, Win=Wg, C0=Cg, C1=0, Cout=Co, ksize=k, stride=1,
                  upsample=0, a_dtype=opd, op_dtype=opd, out_nchw=0, engine=N_.CONV_TC if tc else N_.CONV_SIMT)

    def wgrad(self, a, a_dtype, Cs, Cw, Hin, Win, gy, Co, k, stride, w, biases=(), n=None, dw=None):
        """dW (PyTorch layout, into the flat parameter-gradient buffer unless `dw` names a scratch buffer) and the bias
        gradient(s); a is None: bias gradient only"""
        P, pg = self.P, self.pg
        fields = dict(N=n or self.Nf, Hin=Hin, Win=Win, C=Cs, Cw=Cw, Cout=Co, ksize=k, stride=stride, a_dtype=a_dtype,
                      dy_dtype=self.opd, engine=N_.CONV_TC if self.use_tc else N_.CONV_SIMT)
        need = int(self.lib.fdm_conv_wgrad_workspace(C.byref(N_.ConvWgradArgs(**fields))))
        P.wg_ws.nbytes = max(P.wg_ws.nbytes, (need + 255) // 256 * 256)
        pad_ = k // 2
        P.bflops += 2 * (n or self.Nf) * ((Hin + 2 * pad_ - k) // stride + 1) * ((Win + 2 * pad_ - k) // stride + 1) * Co * k * k * Cw
        P.bside.add(len(P.bops))
        P.op("fdm_conv_wgrad", N_.ConvWgradArgs, a=a, dy=gy, dw=(dw if dw is not None else pg(w)) if a is not None else None,
             dbias=pg(biases[0]) if biases else None,
             dbias2=pg(biases[1]) if len(biases) > 1 else None, workspace=P.wg_ws, workspace_bytes=need, **fields)

    # ------------------------------------------------------------------ activation gradients
    def gact(self, a):
        """fp32 gradient buffer of a residual-stream tensor"""
        if id(a.buf) not in self.gbufs:
            self.gbufs[id(a.buf)] = self.P.buf("g_act", self.Nf * a.H * a.W * a.C * 4)
        return self.gbufs[id(a.buf)]

    def acc(self, a):
        """1 once the gradient buffer of `a` holds a contribution (later writers accumulate, the first one overwrites)"""
        r_ = 1 if id(a.buf) in self.ginit else 0
        self.ginit.add(id(a.buf))
        return r_

    def to_op(self, g, Cc, Hh, Ww, n=None, up=0, biases=()):
        """fp32 gradient -> operand-dtype copy feeding dgrad / wgrad (up = 2: zero insertion for a stride-2 conv).  `biases`:
        bias parameters of the conv whose output gradient this is — their gradient (the column sums) falls out of the same
        read (fp32 atomics into the zeroed flat gradient buffer)."""
        f_ = 2 if up else 1
        o_ = self.P.buf("g_op", (n or self.Nf) * Hh * f_ * Ww * f_ * Cc * self.osz)
        assert not (biases and (up or Cc > 1024))
        self.P.op("fdm_cast", N_.CastArgs, x=g, out=o_, N=n or self.Nf, H=Hh, W=Ww, C=Cc, upsample=up, op_dtype=self.opd,
                  colsum=self.pg(biases[0]) if biases else None, colsum2=self.pg(biases[1]) if len(biases) > 1 else None)
        return o_

    def get_op(self, act):
        """operand-dtype copy of the complete gradient of `act` + the bias gradient of its producing conv (already written, with
        the bias sums, by the GroupNorm backward that was the last contributor to it, if one was)"""
        if id(act.buf) in self.preop:
            return self.preop[id(act.buf)]
        return self.to_op(self.gact(act), act.C, act.H, act.W, biases=act.biases)

    # ------------------------------------------------------------------ GroupNorm
    def gn_apply(self, xa, gn, out_op, xb=None, out_f32=None, raw_op=None, silu=1, film_off=None, **extra):
        """GroupNorm (+ FiLM from the conditioning buffer at `film_off`) (+ SiLU) of xa [‖ xb] into operand / fp32 copies"""
        P = self.P
        P.op("fdm_gn_apply", N_.GnApplyArgs, xa=xa.buf, xb=xb.buf if xb else None, stats_a=xa.st, stats_b=xb.st if xb else None,
             gamma=self.w.f32(gn.weight), beta=self.w.f32(gn.bias), film=self.cond if film_off is not None else None,
             out_op=out_op, out_f32=out_f32, raw_op=raw_op, N=self.Nf, HW=xa.H * xa.W, Ca=xa.C, Cb=xb.C if xb else 0, T=self.T,
             film_stride=self.cond_cols if film_off is not None else 0, film_off=film_off or 0, silu=silu, op_dtype=self.opd,
             eps=gn.eps, **extra)

    def gn_bwd(self, xa, xb, gn, foff, dy_op, dy_f32, draw, silu, last=False, dpass=None, dropf=None):
        """`last`: this GroupNorm is the LAST contributor (in backward order) to xa's gradient — true for the first forward
        consumer of a tensor — so the launch also emits the operand copy + bias sums its producer needs (checked after the
        schedule is complete: no later launch may write that gradient).  `dropf`: the dropout fields of the forward launch,
        whose mask the backward regenerates."""
        P, pg, gact, acc, Nf = self.P, self.pg, self.gact, self.acc, self.Nf
        Cc = xa.C + (xb.C if xb else 0)
        ab_ = P.bzero("gn_ab", Nf * Cc * 16)
        gop = None
        if last:
            gop = P.buf("g_op", Nf * xa.H * xa.W * xa.C * self.osz)
            self.preop[id(xa.buf)] = gop
            self.fused_checks.append((len(P.bops), gact(xa)))
        film = foff is not None
        fields = dict(xa=xa.buf, xb=xb.buf if xb else None, stats_a=xa.st,
                      stats_b=xb.st if xb else None, gamma=self.w.f32(gn.weight), beta=self.w.f32(gn.bias),
                      film=self.cond if film else None, dy_op=dy_op, dy_f32=dy_f32, draw_op=draw, gxa=gact(xa),
                      gxb=gact(xb) if xb else None, ab=ab_, dgamma=pg(gn.weight), dbeta=pg(gn.bias),
                      dfilm=self.dcond if film else None, N=Nf, HW=xa.H * xa.W, Ca=xa.C, Cb=xb.C if xb else 0, T=self.T,
                      film_stride=self.cond_cols if film else 0, film_off=foff if film else 0, silu=silu, op_dtype=self.opd,
                      acc_a=acc(xa), acc_b=acc(xb) if xb else 0, eps=gn.eps, dpass_a=dpass, gop_a=gop,
                      cs_a=pg(xa.biases[0]) if (gop is not None and xa.biases) else None,
                      cs2_a=pg(xa.biases[1]) if (gop is not None and len(xa.biases) > 1) else None, **(dropf or {}))
        # sums + apply on the main chain; the parameter-gradient launch (dgamma, dbeta, FiLM scale/shift gradients) only reads
        # the sums and feeds parameter gradients / the conditioning-path backward at the very end: side stream
        P.op("fdm_gn_bwd", N_.GnBwdArgs, phases=5, **fields)
        P.bside.add(len(P.bops))
        P.op("fdm_gn_bwd", N_.GnBwdArgs, phases=2, **fields)

    # ------------------------------------------------------------------ blocks
    def with_op_copy(self, act):
        """Ask the producing conv to also store a bf16 copy (a stride-2 Downsample conv reads it directly: no cast pass)."""
        act.op = self.P.buf("act_op", self.Nf * act.H * act.W * act.C * self.osz)
        return act.op

    def new_act(self, name, Cc, Hh, Ww):
        return Act(self.P.buf(name, self.Nf * Hh * Ww * Cc * 4), self.P.zeroed(name, self.Nf * Cc * 16), Cc, Hh, Ww)

    def stem(self, layer, want_op):
        P, H, W, Nf, Cin = self.P, self.H, self.W, self.Nf, self.m.in_channels
        stem_tc, xin = self.stem_tc, self.xin
        out = self.new_act("stem", layer.out_channels, H, W)
        out.biases = (layer.bias,)
        if stem_tc:
            self.conv(xin, 8, H, W, layer.weight, layer.out_channels, 3, bias=self.w.f32(layer.bias), y_f32=out.buf,
                      y_op=self.with_op_copy(out) if want_op else None, stats=out.st, a_dtype=N_.BF16, flop_c0=Cin)
        else:
            self.conv(xin, Cin, H, W, layer.weight, layer.out_channels, 3, bias=self.w.f32(layer.bias), y_f32=out.buf,
                      stats=out.st, a_dtype=N_.F32)

        def bwd():
            go = self.get_op(out)
            if stem_tc and layer.out_channels % 64 == 0:
                # tcgen05 wgrad wants >= 64 stored input channels: a zero-padded bf16 copy of the network input
                # (7/8 of the MMA rows are zeros — still ~20x faster than CUDA cores on the 128-px model)
                xin64 = P.buf("xin64", Nf * H * W * 64 * 2)
                P.op("fdm_input_prep", N_.InputPrepArgs, x=P.x, x0=P.x0, obs_mask=P.obs, xin=None, xin_bf16=xin64,
                     N=Nf, C=Cin - 1, H=H, W=W, Cpad=64)
                self.wgrad(xin64, N_.BF16, 64, Cin, H, W, go, layer.out_channels, 3, 1, layer.weight)
                return
            self.wgrad(xin, N_.BF16 if stem_tc else N_.F32, 8 if stem_tc else Cin, Cin, H, W, go, layer.out_channels, 3, 1,
                       layer.weight)
        if self.train:
            P.tape.append(bwd)
        return out

    def res_block(self, rb, xa, xb=None, want_op=False):
        P, Nf, osz, opd, f32 = self.P, self.Nf, self.osz, self.opd, self.w.f32
        Hh, Ww = xa.H, xa.W
        Ci = xa.C + (xb.C if xb else 0)
        Co = rb.out_channels
        hw = Hh * Ww
        has_skip = not isinstance(rb.skip_connection, nn.Identity)
        a1 = P.buf("res_a1", Nf * hw * Ci * osz)
        raw = P.buf("res_raw", Nf * hw * Ci * osz) if has_skip else None
        gn, c1 = rb.in_layers[0], rb.in_layers[2]
        self.gn_apply(xa, gn, a1, xb=xb, raw_op=raw)
        # the first conv's output is read by ONE consumer, the second GroupNorm: inference plans in bf16 mode store it once, in
        # bf16 (statistics still come from the fp32 accumulators in the conv epilogue): 6 instead of 10 bytes per element through
        # conv epilogue + GN-apply.  Training plans keep it in fp32 (the GroupNorm backward re-reads it).
        h1_bf16 = self.use_tc and not self.train
        if h1_bf16:
            h1_ = Act(P.buf("res_h1_op", Nf * hw * Co * osz), P.zeroed("res_h1", Nf * Co * 16), Co, Hh, Ww)
            self.conv(a1, Ci, Hh, Ww, c1.weight, Co, 3, bias=f32(c1.bias), y_op=h1_.buf, stats=h1_.st)
        else:
            h1_ = self.new_act("res_h1", Co, Hh, Ww)
            self.conv(a1, Ci, Hh, Ww, c1.weight, Co, 3, bias=f32(c1.bias), y_f32=h1_.buf, stats=h1_.st)
        h1_.biases = (c1.bias,)
        gn2, c2 = rb.out_layers[0], rb.out_layers[3]
        a2 = P.buf("res_a2", Nf * hw * Co * osz)
        P.res_a2.append((a2, Co, Hh, Ww))
        # dropout (train mode, p > 0): one salt per ResBlock; the backward regenerates the mask from the same fields
        dropf = dict(drop_philox=P.drop_philox, drop_p=P.drop_p, drop_salt=len(P.res_a2)) if P.drop_philox is not None else {}
        self.gn_apply(h1_, gn2, a2, film_off=self.film_off[id(rb)], xa_bf16=1 if h1_bf16 else 0,
                      film_add=0 if self.m.use_scale_shift_norm else 1, **dropf)
        out = self.new_act("res_out", Co, Hh, Ww)
        yop = self.with_op_copy(out) if want_op else None
        sk = rb.skip_connection
        out.biases = (c2.bias, sk.bias) if has_skip else (c2.bias,)
        if has_skip:
            if sk.kernel_size != (1, 1):
                raise NotImplementedError("ResBlock(use_conv=True) 3x3 skip is never built by create_model")
            self.conv(a2, Co, Hh, Ww, c2.weight, Co, 3, a1=raw, C1=Ci, w1=sk.weight, bias=self.w.bias_sum(c2.bias, sk.bias),
                      y_f32=out.buf, y_op=yop, stats=out.st)
        else:
            self.conv(a2, Co, Hh, Ww, c2.weight, Co, 3, bias=f32(c2.bias), resid=xa.buf, y_f32=out.buf, y_op=yop, stats=out.st)

        def bwd():
            g_out = self.gact(out)
            go = self.get_op(out)
            da2 = P.buf("d_a2", Nf * hw * Co * osz)
            self.dgrad(go, Co, Hh, Ww, c2.weight, Co, 3, out_op=da2)
            draw = None
            if has_skip:
                self.wgrad(a2, opd, Co, Co, Hh, Ww, go, Co, 3, 1, c2.weight)
                draw = P.buf("d_raw", Nf * hw * Ci * osz)
                self.dgrad(go, Co, Hh, Ww, sk.weight, Ci, 1, out_op=draw)
                self.wgrad(raw, opd, Ci, Ci, Hh, Ww, go, Co, 1, 1, sk.weight)
            else:
                self.wgrad(a2, opd, Co, Co, Hh, Ww, go, Co, 3, 1, c2.weight)  # identity residual: g_xa += g_out inside the last gn_bwd
            self.gn_bwd(h1_, None, gn2, self.film_off[id(rb)], da2, None, None, 1, last=True, dropf=dropf)
            gh = self.get_op(h1_)
            da1 = P.buf("d_a1", Nf * hw * Ci * osz)
            self.dgrad(gh, Co, Hh, Ww, c1.weight, Ci, 3, out_op=da1)
            self.wgrad(a1, opd, Ci, Ci, Hh, Ww, gh, Co, 3, 1, c1.weight)
            self.gn_bwd(xa, xb, gn, None, da1, None, draw, 1, last=True, dpass=None if has_skip else g_out)
        if self.train:
            P.tape.append(bwd)
        return out

    def attention(self, ab, x, want_op=False):
        P, B, T, Nf, osz, opd, f32, train = self.P, self.B, self.T, self.Nf, self.osz, self.opd, self.w.f32, self.train
        R, R_op, key = self.R, self.R_op, lambda which: (id(ab), which)
        Cc, Hh, Ww, hw = x.C, x.H, x.W, x.H * x.W
        ta, sa = ab.temporal_attention, ab.spatial_attention

        # Inference plans in bf16 mode: the GroupNorm of each half runs in the operand path of its qkv linear (fdm_norm_linear:
        # the normalised tensor is never written) and the proj_out epilogue recomputes the residual GN(x) from x and the
        # saved statistics (fdm_conv resid_norm) — 2 launches and 24 bytes per element less per attention block.
        def nl_ok(a_mode):
            if not self.use_tc or train:
                return False
            probe = N_.NormLinearArgs(B=B, T=T, HW=hw, K=Cc, Cout=3 * Cc, a_mode=a_mode)
            return bool(self.lib.fdm_norm_linear_supported(C.byref(probe)))

        def norm_qkv(src, a_mode, norm, lin, out, stats=None, tstats=None):
            P.op("fdm_norm_linear", N_.NormLinearArgs, x=src, stats=stats, tstats=tstats, gamma=f32(norm.weight),
                 beta=f32(norm.bias), w=self.w.fwd(lin.weight, True), bias=f32(lin.bias), y_op=out, B=B, T=T, HW=hw, K=Cc,
                 Cout=3 * Cc, a_mode=a_mode, eps=norm.eps)
            P.flops += 2 * Nf * hw * 3 * Cc * Cc

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
            self.conv(xn_op, Cc, Hh, Ww, ta.qkv.weight, 3 * Cc, 1, bias=f32(ta.qkv.bias), y_op=qkv)
        o = P.buf("ta_o", Nf * hw * Cc * osz)
        P.flops += 10 * T * T * Cc * B * hw  # QK^T, PV and the three contextual RPE einsums (rpe.py:72-83,144,166)
        ws_bytes = self.temporal_ws(Cc, ta.num_heads, hw) if (self.use_tc and not train) else None
        ws = P.buf("ta_ws", ws_bytes) if ws_bytes else None
        if ws is None and R[key("rpe_q")] is None:
            raise NativeShapeError(f"temporal attention: no kernel takes T={T}, HW={hw}, C={Cc}, heads={ta.num_heads}")
        # return_attn_weights=True plans: the tcgen05 kernels also accumulate the head-averaged attention weights — the maps
        # RPEAttention.forward logs (rpe.py:128-130) — into zero-initialised fp32 buffers
        t_mean = s_mean = None
        if self.collect_attn:
            if ws is None or not self.use_tc:
                raise NativeShapeError("attention-map logging is served by the tcgen05 attention kernels (bf16 mode)")
            t_mean = P.zeroed("ta_attn_mean", B * hw * T * T * 4)
            s_mean = P.zeroed("sa_attn_mean", Nf * hw * hw * 4)
            P.attn_maps["temporal"].append((t_mean, (B * hw, T, T)))
            P.attn_maps["spatial"].append((s_mean, (Nf, hw, hw)))
        P.op("fdm_attn_temporal", N_.AttnTemporalArgs, qkv=qkv, Rq=R[key("rpe_q")], Rk=R[key("rpe_k")],
             Rv=R[key("rpe_v")], mask=P.mask, out=o, B=B, T=T, HW=hw, C=Cc, heads=ta.num_heads,
             qkv_dtype=opd, out_dtype=opd, Rq_op=R_op.get(key("rpe_q")) if ws else None,
             Rk_op=R_op.get(key("rpe_k")) if ws else None, Rv_op=R_op.get(key("rpe_v")) if ws else None,
             workspace=ws, workspace_bytes=ws_bytes or 0, attn_mean=t_mean)
        y = self.new_act("ta_y", Cc, Hh, Ww)
        y.biases = (ta.proj_out.bias,)
        if t_fused:
            self.conv(o, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, bias=f32(ta.proj_out.bias), resid=x.buf, y_f32=y.buf, stats=y.st,
                      resid_norm=2, rn_T=T, rn_eps=ta.norm.eps, rn_tstats=tst, rn_gamma=f32(ta.norm.weight),
                      rn_beta=f32(ta.norm.bias))
        else:
            self.conv(o, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, bias=f32(ta.proj_out.bias), resid=xn, y_f32=y.buf, stats=y.st)
        # --- spatial: plain per-frame GroupNorm, attention over the pixels of each frame
        qkv2 = P.buf("sa_qkv", Nf * hw * 3 * Cc * osz)
        s_fused = nl_ok(1)
        if s_fused:
            yn = None
            norm_qkv(y.buf, 1, sa.norm, sa.qkv, qkv2, stats=y.st)
        else:
            yn = P.buf("sa_yn", Nf * hw * Cc * 4)
            yn_op = P.buf("sa_yn_op", Nf * hw * Cc * osz)
            self.gn_apply(y, sa.norm, yn_op, out_f32=yn, silu=0)
            self.conv(yn_op, Cc, Hh, Ww, sa.qkv.weight, 3 * Cc, 1, bias=f32(sa.qkv.bias), y_op=qkv2)
        o2 = P.buf("sa_o", Nf * hw * Cc * osz)
        P.flops += 4 * hw * hw * Cc * Nf
        # training: the tcgen05 forward also saves the log-sum-exp of every score row for the tcgen05 backward kernels
        sa_lse = P.buf("sa_lse", Nf * sa.num_heads * hw * 4) if (train and self.use_tc) else None
        P.op("fdm_attn_spatial", N_.AttnSpatialArgs, qkv=qkv2, out=o2, N=Nf, L=hw, C=Cc, heads=sa.num_heads,
             qkv_dtype=opd, out_dtype=opd, engine=0 if self.use_tc else 1, lse=sa_lse, attn_mean=s_mean)
        z = self.new_act("sa_z", Cc, Hh, Ww)
        z.biases = (sa.proj_out.bias,)
        if s_fused:
            self.conv(o2, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, bias=f32(sa.proj_out.bias), resid=y.buf, y_f32=z.buf,
                      y_op=self.with_op_copy(z) if want_op else None, stats=z.st, resid_norm=3, rn_eps=sa.norm.eps, rn_stats=y.st,
                      rn_gamma=f32(sa.norm.weight), rn_beta=f32(sa.norm.bias))
        else:
            self.conv(o2, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, bias=f32(sa.proj_out.bias), resid=yn, y_f32=z.buf,
                      y_op=self.with_op_copy(z) if want_op else None, stats=z.st)

        def bwd():
            pg, dRb = self.pg, self.dRb
            n_tok = Nf * hw
            # spatial half: z = proj(o2) + yn ; o2 = attn(qkv2) ; qkv2 = qkv(yn_op) ; yn = GN(y)
            g_z = self.gact(z)
            gz = self.get_op(z)
            do2 = P.buf("d_sa_o", n_tok * Cc * osz)
            self.dgrad(gz, Cc, Hh, Ww, sa.proj_out.weight, Cc, 1, out_op=do2)
            self.wgrad(o2, opd, Cc, Cc, Hh, Ww, gz, Cc, 1, 1, sa.proj_out.weight)
            dqkv2 = P.buf("d_sa_qkv", n_tok * 3 * Cc * osz)
            P.bflops += 10 * hw * hw * Cc * Nf
            P.op("fdm_attn_spatial_bwd", N_.AttnSpatialBwdArgs, qkv=qkv2, out=o2, dout=do2, dqkv=dqkv2,
                 lse=sa_lse if sa_lse is not None else P.at_lse, dsum=P.at_dsum, N=Nf, L=hw, C=Cc, heads=sa.num_heads,
                 dtype=opd, lse_from_forward=1 if sa_lse is not None else 0)
            P.at_rows = max(P.at_rows, Nf * sa.num_heads * hw)
            dyn = P.buf("d_sa_yn", n_tok * Cc * osz)
            self.dgrad(dqkv2, 3 * Cc, Hh, Ww, sa.qkv.weight, Cc, 1, out_op=dyn)
            self.wgrad(yn_op, opd, Cc, Cc, Hh, Ww, dqkv2, 3 * Cc, 1, 1, sa.qkv.weight, (sa.qkv.bias,))
            self.gn_bwd(y, None, sa.norm, None, dyn, g_z, None, 0, last=True)
            # temporal half: y = proj(o) + xn ; o = attn_rpe(qkv, R) ; qkv = qkv(xn_op) ; xn = temporalGN(x)
            g_y = self.gact(y)
            gy = self.get_op(y)
            do = P.buf("d_ta_o", n_tok * Cc * osz)
            self.dgrad(gy, Cc, Hh, Ww, ta.proj_out.weight, Cc, 1, out_op=do)
            self.wgrad(o, opd, Cc, Cc, Hh, Ww, gy, Cc, 1, 1, ta.proj_out.weight)
            dqkv = P.buf("d_ta_qkv", n_tok * 3 * Cc * osz)
            P.bflops += 25 * T * T * Cc * B * hw
            P.op("fdm_attn_temporal_bwd", N_.AttnTemporalBwdArgs, qkv=qkv, out=o, Rq=R[key("rpe_q")],
                 Rk=R[key("rpe_k")], Rv=R[key("rpe_v")], mask=P.mask, dout=do, dqkv=dqkv,
                 dRq=dRb[key("rpe_q")], dRk=dRb[key("rpe_k")], dRv=dRb[key("rpe_v")], lse=P.at_lse,
                 dsum=P.at_dsum, B=B, T=T, HW=hw, C=Cc, heads=ta.num_heads, dtype=opd)
            P.at_rows = max(P.at_rows, B * ta.num_heads * T * hw)
            dxn = P.buf("d_ta_xn", n_tok * Cc * osz)
            self.dgrad(dqkv, 3 * Cc, Hh, Ww, ta.qkv.weight, Cc, 1, out_op=dxn)
            self.wgrad(xn_op, opd, Cc, Cc, Hh, Ww, dqkv, 3 * Cc, 1, 1, ta.qkv.weight, (ta.qkv.bias,))
            P.op("fdm_temporal_gn_bwd", N_.TemporalGnBwdArgs, x=x.buf, gamma=f32(ta.norm.weight), dy_op=dxn, dy_f32=g_y,
                 gx=self.gact(x), dgamma=pg(ta.norm.weight), dbeta=pg(ta.norm.bias), B=B, T=T, HW=hw, C=Cc, op_dtype=opd,
                 accumulate=self.acc(x), eps=ta.norm.eps)
        if train:
            P.tape.append(bwd)
        return z

    def resample(self, layer, x, down, want_op=False):
        P, Nf, osz, opd, train = self.P, self.Nf, self.osz, self.opd, self.train
        cv = layer.op if down else layer.conv
        Ho, Wo = (x.H // 2, x.W // 2) if down else (x.H * 2, x.W * 2)
        out = self.new_act("down" if down else "up", x.C, Ho, Wo)
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
            self.conv(a, x.C, x.H, x.W, cv.weight, x.C, 3, upsample=1, bias=self.w.f32(cv.bias), y_f32=out.buf, stats=out.st,
                      y_op=self.with_op_copy(out) if want_op else None)
        elif (self.use_tc and self.tc_ok(x.C, 0, x.C, 3, 2 if down else 1, 0, Ho, Wo)) or (train and not down):
            if down and x.op is not None:
                a = x.op  # the producing conv already stored the bf16 operand copy
            else:
                # bf16 operand copy of the fp32 stream (nearest x2 upsample folded into the cast, unet.py:85), then tcgen05
                a = P.buf("resample_a", Nf * Hc * Wc * x.C * osz)
                P.op("fdm_cast", N_.CastArgs, x=x.buf, out=a, N=Nf, H=x.H, W=x.W, C=x.C, upsample=0 if down else 1,
                     op_dtype=opd, colsum=None, colsum2=None)
            self.conv(a, x.C, Hc, Wc, cv.weight, x.C, 3, stride=2 if down else 1, bias=self.w.f32(cv.bias), y_f32=out.buf,
                      stats=out.st, y_op=self.with_op_copy(out) if (want_op and not train) else None)
        else:
            # the CUDA-core engine gathers straight from the fp32 stream (stride 2 / folded nearest upsample)
            self.conv(x.buf, x.C, x.H, x.W, cv.weight, x.C, 3, stride=2 if down else 1, upsample=0 if down else 1,
                      bias=self.w.f32(cv.bias), y_f32=out.buf, stats=out.st, a_dtype=N_.F32)

        def bwd():
            Cc = x.C
            g_out = self.gact(out)
            go = self.get_op(out)
            if down:
                # dgrad of the stride-2 conv = stride-1 conv over the zero-inserted gradient, accumulated in place into g_x
                z_ = self.to_op(g_out, Cc, Ho, Wo, up=2)
                gx = self.gact(x)
                self.dgrad(z_, Cc, Hc, Wc, cv.weight, Cc, 3, out_f32=gx, resid=gx if self.acc(x) else None)
                if self.use_tc and a is not None:
                    # tcgen05 wgrad is stride-1: the zero-inserted gradient against the full-resolution input is the same sum
                    self.wgrad(a, opd, Cc, Cc, Hc, Wc, z_, Cc, 3, 1, cv.weight)
                else:
                    self.wgrad(a if a is not None else x.buf, opd if a is not None else N_.F32, Cc, Cc, Hc, Wc, go, Cc, 3, 2,
                               cv.weight)
            else:
                da = P.buf("d_up_a", Nf * Ho * Wo * Cc * osz)
                self.dgrad(go, Cc, Ho, Wo, cv.weight, Cc, 3, out_op=da)
                self.wgrad(a, opd, Cc, Cc, Ho, Wo, go, Cc, 3, 1, cv.weight)
                P.op("fdm_accum", N_.AccumArgs, src=da, dst=self.gact(x), N=Nf, H=x.H, W=x.W, C=Cc, pool=1, src_dtype=opd,
                     accumulate=self.acc(x))
        if train:
            P.tape.append(bwd)
        return out

    def run_stage(self, stage, h, skip=None, feeds_downsample=False):
        layers = list(stage)
        for li, layer in enumerate(layers):
            want_op = feeds_downsample and li == len(layers) - 1 and self.use_tc
            # inference: the phase-mode upsample conv reads the low-resolution bf16 operand — let the producing conv store it
            # (one more epilogue store instead of a cast launch)
            if (not self.train and h is not None and li + 1 < len(layers) and isinstance(layers[li + 1], Upsample)
                    and isinstance(layer, (ResBlock, FactorizedAttentionBlock))
                    and self.up_tc_ok(getattr(layer, "out_channels", h.C), h.H, h.W)):
                want_op = True
            if isinstance(layer, nn.Conv2d):
                h = self.stem(layer, want_op)
            elif isinstance(layer, ResBlock):
                h = self.res_block(layer, h, skip, want_op=want_op)
                skip = None
            elif isinstance(layer, FactorizedAttentionBlock):
                h = self.attention(layer, h, want_op=want_op)
            elif isinstance(layer, Downsample):
                h = self.resample(layer, h, True, want_op=want_op)
            elif isinstance(layer, Upsample):
                h = self.resample(layer, h, False, want_op=want_op)
            else:
                raise NotImplementedError(type(layer))
            self.P.taps[self.names[id(layer)]] = (h.buf, h.C, h.H, h.W)
        return h

    def body(self):
        P, m, H, W, Nf, Cin = self.P, self.m, self.H, self.W, self.Nf, self.m.in_channels
        # bf16 mode: the stem conv runs on tcgen05 over a bf16 copy of the network input, channels zero-padded to 8
        self.stem_tc = self.use_tc and self.tc_ok(8, 0, m.model_channels, 3, 1, 0, H, W) and Cin <= 8
        Cpad = 8 if self.stem_tc else 0
        self.xin = P.buf("xin", Nf * H * W * (Cpad * 2 if self.stem_tc else Cin * 4))
        P.op("fdm_input_prep", N_.InputPrepArgs, x=P.x, x0=P.x0, obs_mask=P.obs, xin=None if self.stem_tc else self.xin,
             xin_bf16=self.xin if self.stem_tc else None, N=Nf, C=Cin - 1, H=H, W=W, Cpad=Cpad)
        self.names = {id(mod): name for name, mod in m.named_modules()}
        h, hs = None, []
        in_stages = list(m.input_blocks)
        for si, stage in enumerate(in_stages):
            nxt = in_stages[si + 1] if si + 1 < len(in_stages) else None
            feeds = nxt is not None and len(nxt) == 1 and isinstance(nxt[0], Downsample)
            h = self.run_stage(stage, h, feeds_downsample=feeds)   # pushed as a U-Net skip
            hs.append(h)
        h = self.run_stage(m.middle_block, h)
        for stage in m.output_blocks:
            h = self.run_stage(stage, h, hs.pop())
        self.head(h)

    def head(self, h):
        P, m, H, W, Nf, osz, opd = self.P, self.m, self.H, self.W, self.Nf, self.osz, self.opd
        gn, cv = m.out[0], m.out[2]
        a = P.buf("head_a", Nf * H * W * h.C * osz)
        self.gn_apply(h, gn, a)
        self.conv(a, h.C, H, W, cv.weight, m.out_channels, 3, bias=self.w.f32(cv.bias), y_f32=P.eps, out_nchw=1)
        if not self.train:
            return
        Co_ = m.out_channels
        P.geps = P.buf("geps", Nf * Co_ * H * W * 4, True)
        P.at_rows = 1
        P.at_lse, P.at_dsum = P.buf("attn_lse", 256), P.buf("attn_dsum", 256)

        def bwd():
            pg = self.pg
            tc_head = self.use_tc and self.tc_ok(8, 0, h.C, 3, 1, 0, H, W) and Co_ <= 8
            Cp = 8 if tc_head else Co_
            ge_p = P.buf("geps_op", Nf * H * W * Cp * osz)
            P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge_p, N=Nf, C=Co_, H=H, W=W, Cpad=Cp, op_dtype=opd)
            ge = ge_p
            if Cp != Co_:
                ge = P.buf("geps_op_true", Nf * H * W * Co_ * osz)
                P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge, N=Nf, C=Co_, H=H, W=W, Cpad=Co_, op_dtype=opd)
            da = P.buf("d_head_a", Nf * H * W * h.C * osz)
            self.dgrad(ge_p, Cp, H, W, cv.weight, h.C, 3, out_op=da)
            if tc_head and h.C % 64 == 0:
                # same trick on the output side: the eps gradient zero-padded to 64 channels feeds the tcgen05 wgrad; the first
                # Co_ rows of its [64][C][3][3] result are the head's weight gradient
                ge64 = P.buf("geps_op64", Nf * H * W * 64 * osz)
                P.op("fdm_nchw_to_nhwc", N_.NchwToNhwcArgs, src=P.geps, dst=ge64, N=Nf, C=Co_, H=H, W=W, Cpad=64, op_dtype=opd)
                dw64 = P.buf("head_dw64", 64 * h.C * 9 * 4)
                self.wgrad(a, opd, h.C, h.C, H, W, ge64, 64, 3, 1, cv.weight, (), dw=dw64)
                P.bside.add(len(P.bops))  # consumes the side-stream wgrad's scratch: same stream
                P.op("fdm_sum_parts", N_.SumPartsArgs, parts=dw64, out=pg(cv.weight), part_stride=0, n=Co_ * h.C * 9,
                     count=1, accumulate=0)
                self.wgrad(None, opd, h.C, h.C, H, W, ge, Co_, 3, 1, cv.weight, (cv.bias,))
            else:
                self.wgrad(a, opd, h.C, h.C, H, W, ge, Co_, 3, 1, cv.weight, (cv.bias,))
            self.gn_bwd(h, None, gn, None, da, None, None, 1, last=True)
        P.tape.append(bwd)

    # ------------------------------------------------------------------ backward schedule, streams
    def backward(self):
        P = self.P
        P.cur = P.bops
        for emit in reversed(P.tape):
            emit()
        P.cur = P.ops
        # a fused operand copy is only valid if nothing writes that gradient afterwards
        grad_out_fields = ("gxa", "gxb", "dst", "y_f32", "gx")
        for idx, gbuf in self.fused_checks:
            for j in range(idx + 1, len(P.bops)):
                fn_j, _, f_j = P.bops[j]
                if fn_j == "fdm_gn_bwd" and f_j.get("phases") == 2:
                    continue  # parameter-gradient launch: does not write activation gradients
                if any(f_j.get(k) is gbuf for k in grad_out_fields):
                    raise AssertionError(f"backward schedule: {fn_j} (#{j}) writes a gradient after its operand copy was fused (#{idx})")
        P.grad_buckets = self.grad_buckets()
        P.at_lse.nbytes = P.at_dsum.nbytes = (P.at_rows * 4 + 255) // 256 * 256

    def grad_buckets(self):
        """Partition the flat parameter-gradient buffer into FDM_GRAD_BUCKETS (default 4) ranges of consecutive slots and find, for
        each, the backward launch after which it is final: [(first element, one past the last element, index of that launch)].
        The slots are in gradient-completion order (optim.completion_order), so the `done` indices ascend: bucket k can be
        all-reduced while launches done_k+1 ... run.  Every parameter must have a writer (DDP find_unused_parameters=False)."""
        P, params = self.P, self.params
        base, n = P.pgrad.data_ptr(), P.pgrad.numel()
        by_off = sorted((o, i) for i, o in enumerate(P.flat_offs))
        starts = [o for o, _ in by_off]
        last = [-1] * len(params)

        def note(v, j):
            if isinstance(v, th.Tensor) and base <= v.data_ptr() < base + 4 * n:
                i = by_off[bisect.bisect_right(starts, (v.data_ptr() - base) // 4) - 1][1]
                last[i] = max(last[i], j)
        for j, (_, _, f) in enumerate(P.bops):
            for v in P.field_values(f):
                note(v, j)
        names = [nm for nm, _ in self.m.named_parameters()]
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

    def streams(self):
        # The whole conditioning chain — timestep embedding, time MLP, FiLM / RPE time projections, RPENet tables: everything that
        # depends only on (t, frame_indices) — runs on a side stream and is joined before its first consumer on the main stream
        # (the first FiLM GroupNorm-apply, or the first temporal attention), so it overlaps input prep, stem and the first convs
        # instead of heading every step.  Inside a CUDA-graph capture the fork / join become graph edges.
        P = self.P
        cond_bufs = ({id(self.cond)} | {id(v) for v in self.R.values() if v is not None}
                     | {id(v) for v in self.R_op.values() if v is not None})

        def reads_cond(fields):
            for v in fields.values():
                b_ = v[0] if isinstance(v, tuple) else v
                if isinstance(b_, Buf) and id(b_) in cond_bufs:
                    return True
            return False
        if not self.train and P.side_end > P.side_begin:
            P.side_begin = P.temb_op
        P.join_at = next((i for i, (fn, _, f_) in enumerate(P.ops) if i >= P.side_end and reads_cond(f_)), len(P.ops))
        if th.device(self.device).type == "cuda" and P.side_end > P.side_begin and P.join_at >= P.side_end:
            P.side_stream = th.cuda.Stream(self.device)
            P.ev_fork, P.ev_join = th.cuda.Event(), th.cuda.Event()

"""
FlatAdamW — torch.optim.AdamW as the reference constructs it (train_util.py:127: `AdamW(self.master_params, lr=, weight_decay=)`),
restated over FLAT buffers (SURVEY §8f-2).

The native backward (engine._DenoiserFn) already returns every parameter gradient as a view of ONE flat fp32 buffer.  Here the
parameters, `exp_avg` and `exp_avg_sq` are flat buffers too (each parameter's `.data` is re-pointed to its 16-byte aligned slot;
`Parameter` identity, `state_dict()` keys / shapes and `load_state_dict` are unchanged), so an optimizer step is ONE kernel
launch (`fdm_adamw`) with ~20 us of host work, instead of torch's multi-tensor path over 390 tensors (~0.7 ms of GPU time and
~1 ms of host time per step — a quarter of the launch-bound cfg2 training step).  Optionally the EMA copies of the parameters
(`update_ema`, nn.py:55-65; up to two rates) are updated in the same pass.

Same update rule as torch (decoupled weight decay, bias correction, no amsgrad); `tests/test_gpu_parity.py` checks it against
torch.optim.AdamW step by step.  Gradients that do not come from the native backward (CPU path, torch DDP buckets, partial
graphs) are gathered into a flat buffer with one foreach copy first.  CUDA only: there is no CPU fallback.

`FlatAdamW(model.parameters(), ..., model=model, bind=False)` only adopts the model's flat layout (gradient-completion order, the
layout of the native backward's buffer: its per-parameter gradient views are then used in place, without a gather copy).
`FlatAdamW(model.parameters(), ..., model=model)` additionally BINDS the model's gradient path to the optimizer ("flat-gradient
mode": it becomes the `sink` of the model's `engine.GradRoute`): every `p.grad` becomes a persistent view of the optimizer's flat
gradient buffer, the native backward node takes ONE anchor tensor instead of the 390 parameters and hands its flat gradient over
with one (allreduce +) copy — or add, when several backwards run between `zero_grad()` calls (gradient accumulation).
`p.grad` stays readable / clippable as usual; torch DDP (per-parameter hooks) does not apply in this mode — use
`sharding.FlatGradDataParallel`.
"""
import ctypes as C

import torch as th

from . import _native as N_
from .engine import grad_route


def completion_order(names):
    """Permutation of the parameters (given by name, in model.named_parameters() order) into the order in which their gradients
    become FINAL in the native backward schedule (engine.py): head first, then output blocks / middle block / input blocks in
    reverse forward order, and last the conditioning path — time MLP, every ResBlock's FiLM projection (`emb_layers`) and every
    RPENet — whose gradients are only complete after the whole network has been walked.  The flat gradient / parameter / moment
    buffers use this order, so a bucket of consecutive slots is complete as soon as the backward passes one point, and its
    allreduce can overlap the rest of the backward (sharding.FlatGradDataParallel; reference: DDP buckets, train_util.py:118-125).
    Returns (order, n_early): `order[k]` = index of the parameter stored k-th; the last len(order) - n_early are the late ones."""
    def late(n):
        return n.startswith("time_embed.") or ".emb_layers." in n or ".rpe_net." in n

    def rank(n):
        parts = n.split(".")
        if parts[0] == "out":
            return (0, 0)
        if parts[0] == "output_blocks":
            return (1, -int(parts[1]))
        if parts[0] == "middle_block":
            return (2, 0)
        if parts[0] == "input_blocks":
            return (3, -int(parts[1]))
        return (4, 0)
    early = sorted((i for i, n in enumerate(names) if not late(n)), key=lambda i: rank(names[i]))  # stable within a block
    return early + [i for i, n in enumerate(names) if late(n)], len(early)


def flat_slots(params, order=None):
    """(offsets, total) of the 16-byte aligned slots of `params` in a flat fp32 buffer; `offsets[i]` belongs to params[i], slots
    are laid out in `order` (default: as given).  Shared by the native backward's gradient buffer (engine.py) and FlatAdamW, so
    their views line up."""
    offs, o = [0] * len(params), 0
    for i in (order if order is not None else range(len(params))):
        offs[i] = o
        o += (params[i].numel() + 3) // 4 * 4
    return offs, o


def model_flat_layout(model):
    """(parameters, offsets, total, order, n_early) of a model's flat layout in gradient-completion order."""
    named = list(model.named_parameters())
    order, n_early = completion_order([n for n, _ in named])
    params = [p for _, p in named]
    offs, total = flat_slots(params, order)
    return params, offs, total, order, n_early


class FlatAdamW(th.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, ema_rates=(), model=None, bind=True):
        params = list(params)
        if any(isinstance(p, dict) for p in params):
            raise NotImplementedError("FlatAdamW takes one parameter group (as train_util.py:127 builds it)")
        if len(ema_rates) > 2:
            raise NotImplementedError("up to two EMA rates are fused into the step")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        ps = self.param_groups[0]["params"]
        if not ps or not all(p.is_cuda and p.dtype == th.float32 for p in ps):
            raise RuntimeError("FlatAdamW runs on the sm_100a kernels only: fp32 CUDA parameters (there is no CPU fallback)")
        order = None
        if model is not None:
            mp = list(model.parameters())
            if len(mp) != len(ps) or any(a is not b for a, b in zip(mp, ps)):
                raise ValueError("flat-gradient mode needs exactly the model's parameters, in model.parameters() order")
            order = model_flat_layout(model)[3]  # gradient-completion order: the layout of the native backward's flat buffer
        self._offs, self._total = flat_slots(ps, order)
        dev = ps[0].device
        self.flat_p = th.zeros(self._total, device=dev)
        self.flat_m, self.flat_v = th.zeros_like(self.flat_p), th.zeros_like(self.flat_p)
        self._gather = th.zeros_like(self.flat_p)  # used when the gradients are not already views of one buffer
        with th.no_grad():
            for p, o in zip(ps, self._offs):
                slot = self.flat_p[o:o + p.numel()].view(p.shape)
                slot.copy_(p.data)
                p.data = slot  # same Parameter object, storage now inside the flat buffer
        self._views = lambda flat: [flat[o:o + p.numel()].view(p.shape) for p, o in zip(ps, self._offs)]
        self._g_views = self._views(self._gather)
        for p, m, v in zip(ps, self._views(self.flat_m), self._views(self.flat_v)):
            self.state[p] = {"step": th.zeros((), dtype=th.float32), "exp_avg": m, "exp_avg_sq": v}
        self._step = 0
        self.ema_rates = tuple(float(r) for r in ema_rates)
        self.flat_ema = [self.flat_p.clone() for _ in self.ema_rates]
        self.route = None  # the model's engine.GradRoute once bound
        if model is not None and bind:
            self.flat_g = th.zeros_like(self.flat_p)
            for p, gview in zip(ps, self._views(self.flat_g)):
                p.grad = gview  # persistent: the native backward refreshes flat_g, never these tensor objects
            self.anchor = th.zeros(1, device=dev, requires_grad=True)
            self._fresh = True
            self.route = grad_route(model)
            self.route.sink = self

    def receive(self, flat):
        """Called by the native backward node with the plan's flat gradient (same slot layout): copy, or add when accumulating."""
        if flat.numel() != self.flat_g.numel():
            raise RuntimeError("flat gradient layout mismatch between the training plan and FlatAdamW")
        if self._fresh:
            self.flat_g.copy_(flat)
            self._fresh = False
        else:
            self.flat_g.add_(flat)

    def zero_grad(self, set_to_none=True):
        if self.route is None:
            return super().zero_grad(set_to_none=set_to_none)
        self.flat_g.zero_()  # one memset: gradients that arrive through AccumulateGrad (CPU-style autograd path) add into the views
        self._fresh = True   # the native backward overwrites (copy) on its first hand-over, adds on later ones
        self.route.pending = False

    def ema_params(self, i):
        """Per-parameter views of the i-th EMA copy (same shapes / order as the parameters)."""
        return self._views(self.flat_ema[i])

    def _flat_grad(self, ps):
        if self.route is not None:
            return self.flat_g.data_ptr(), None
        g0 = ps[0].grad
        if g0 is None:
            raise RuntimeError("FlatAdamW.step(): parameter without a gradient (find_unused_parameters=False contract)")
        base = g0.data_ptr() - 4 * self._offs[0]
        if g0.is_contiguous() and g0.dtype == th.float32 and all(
                p.grad is not None and p.grad.data_ptr() == base + 4 * o for p, o in zip(ps, self._offs)):
            return base, None  # the native backward's flat buffer: use it in place
        th._foreach_copy_(self._g_views, [p.grad for p in ps])
        return self._gather.data_ptr(), self._gather

    @th.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with th.enable_grad():
                loss = closure()
        group = self.param_groups[0]
        ps = group["params"]
        if ps[0].data_ptr() != self.flat_p.data_ptr() + 4 * self._offs[0]:
            raise RuntimeError("a parameter's storage was replaced after FlatAdamW flattened it (.to() / .data = ...): rebuild the optimizer")
        g_ptr, _keep = self._flat_grad(ps)
        self._step += 1
        b1, b2 = group["betas"]
        a = N_.AdamwArgs(p=self.flat_p.data_ptr(), g=g_ptr, m=self.flat_m.data_ptr(), v=self.flat_v.data_ptr(),
                         ema0=self.flat_ema[0].data_ptr() if len(self.flat_ema) > 0 else None,
                         ema1=self.flat_ema[1].data_ptr() if len(self.flat_ema) > 1 else None,
                         n=self._total, lr=group["lr"], beta1=b1, beta2=b2, eps=group["eps"], weight_decay=group["weight_decay"],
                         bias_correction1=1.0 - b1 ** self._step, bias_correction2_sqrt=(1.0 - b2 ** self._step) ** 0.5,
                         ema_rate0=self.ema_rates[0] if len(self.ema_rates) > 0 else 0.0,
                         ema_rate1=self.ema_rates[1] if len(self.ema_rates) > 1 else 0.0)
        N_.check(N_.lib().fdm_adamw(C.byref(a), C.c_void_p(th.cuda.current_stream(self.flat_p.device).cuda_stream)), "fdm_adamw")
        # the kernel wrote the parameters through raw pointers: bump one tensor version so that version-keyed caches (the
        # inference engine's packed weights, DenoiserEngine.refresh_weights) notice the update
        ps[0].add_(0)
        return loss

    def state_dict(self):
        for st in self.state.values():
            st["step"].fill_(self._step)
        return super().state_dict()

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        ps = self.param_groups[0]["params"]
        with th.no_grad():  # torch replaced the per-parameter state tensors: copy them back into the flat buffers and re-point
            for p, m, v in zip(ps, self._views(self.flat_m), self._views(self.flat_v)):
                st = self.state[p]
                m.copy_(st["exp_avg"])
                v.copy_(st["exp_avg_sq"])
                self._step = int(st["step"])
                st["exp_avg"], st["exp_avg_sq"] = m, v

"""engine.GradRoute on CPU: every case of the gradient hand-over after the native backward (which graphs run, which buffers are
reduced, what the sink receives, what autograd gets back), driven through a stand-in plan and a stand-in sink.  No kernels run."""
import torch as th

from improved_diffusion.engine import GradRoute, Plan, grad_route
from improved_diffusion.optim import FlatAdamW

DEV = th.device("cpu")


class FakePlan:
    """What GradRoute.hand_over reads of a training plan: three parameters (3 elements padded to 4, 2x2, 2 padded to 4) in a
    12-slot flat gradient, one gradient bucket per parameter, and a backward that writes known values and records its runs."""
    backward_segments = Plan.backward_segments

    def __init__(self, log, buckets=((0, 4, 6), (4, 8, 10), (8, 12, 15))):
        self.log = log
        self.values = th.arange(1.0, 13.0)
        self.pgrad = th.zeros(12)
        self.grad_buckets = list(buckets)
        self.unflat = [th.empty(3), th.empty(1), th.empty(2, 2), th.empty(2), th.empty(2)]
        self.unflat_pick = [0, 2, 3]

    def run_graphed(self, which, device, seg=None):
        assert which == "bwd" and device == DEV
        self.log.append(("bwd", seg))
        if seg is None:
            self.pgrad.copy_(self.values)
            return
        lo, hi = seg
        if lo == 0:
            self.pgrad.zero_()
        for b_lo, b_hi, done in self.grad_buckets:  # the bucket that is final at the end of this segment
            if done + 1 == hi:
                self.pgrad[b_lo:b_hi] = self.values[b_lo:b_hi]

    def slots(self, t):
        return ((t.data_ptr() - self.pgrad.data_ptr()) // 4, (t.data_ptr() - self.pgrad.data_ptr()) // 4 + t.numel())


class FakeSink:
    """FlatAdamW's side of the hand-over on CPU tensors: its own receive / zero_grad code, with each receive recorded."""
    zero_grad = FlatAdamW.zero_grad

    def __init__(self, route, n, log):
        self.route, self.log = route, log
        self.flat_g, self._fresh = th.zeros(n), True
        self.anchor = th.zeros(1, requires_grad=True)
        route.sink = self

    def receive(self, flat):
        self.log.append(("receive", flat.clone()))
        FlatAdamW.receive(self, flat)


def make(sink=False, reduce=False, overlap=False, **plan_kw):
    """(route, plan, sink, log).  The reduces are the mean over two ranks of which the other one holds zeros: they halve."""
    log = []
    P = FakePlan(log, **plan_kw)
    route = GradRoute()
    s = FakeSink(route, P.pgrad.numel(), log) if sink else None

    def name(t):
        if t.data_ptr() == P.pgrad.data_ptr() and t.numel() == P.pgrad.numel():
            return "pgrad"
        return "flat_g" if s is not None and t is s.flat_g else "copy"

    def reduce_(flat):
        log.append(("reduce", name(flat)))
        flat.mul_(0.5)

    def reduce_async(view):
        rng = P.slots(view)
        log.append(("reduce_async", rng))

        def finish():
            log.append(("finish", rng))
            view.mul_(0.5)
        return finish
    if reduce:
        route.reduce = reduce_
    if overlap:
        route.reduce_async = reduce_async
    return route, P, s, log


def events(log):
    return [e if e[0] != "receive" else ("receive",) for e in log]


def views(P, scale):
    v = P.values * scale
    return (v[0:3], v[4:8].view(2, 2), v[8:10])


def assert_grads(got, want):
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.shape == b.shape and th.equal(a, b)


def test_no_sink_returns_per_parameter_views_of_a_copy():
    route, P, _, log = make()
    got = route.hand_over(P, DEV)
    assert events(log) == [("bwd", None)]
    assert_grads(got, views(P, 1.0))
    assert all(g.data_ptr() != P.pgrad.data_ptr() for g in got)  # autograd owns a copy; the plan's buffer is reused


def test_no_sink_reduces_the_copy_before_the_views():
    route, P, _, log = make(reduce=True, overlap=True)  # without a sink the bucketed exchange never runs
    got = route.hand_over(P, DEV)
    assert events(log) == [("bwd", None), ("reduce", "copy")]
    assert_grads(got, views(P, 0.5))
    assert th.equal(P.pgrad, P.values)


def test_sink_without_reduce_receives_the_plan_buffer():
    route, P, s, log = make(sink=True)
    assert route.hand_over(P, DEV) == (None,)
    assert events(log) == [("bwd", None), ("receive",)]
    assert th.equal(s.flat_g, P.values)
    assert route.hand_over(P, DEV) == (None,)  # a second backward before zero_grad() accumulates
    assert th.equal(s.flat_g, 2 * P.values) and route.pending is False


def test_no_sync_twice_then_sync_reduces_the_accumulated_total_once():
    route, P, s, log = make(sink=True, reduce=True, overlap=True)
    route.synced = False
    route.hand_over(P, DEV)
    assert route.pending is True
    route.hand_over(P, DEV)
    assert route.pending is True
    route.synced = True
    assert route.hand_over(P, DEV) == (None,)
    assert route.pending is False
    # the pending backward runs its whole graph (no buckets) and reduces the sink's total, not the plan's buffer
    assert events(log) == [("bwd", None), ("receive",)] * 3 + [("reduce", "flat_g")]
    assert th.equal(s.flat_g, 1.5 * P.values)


def test_zero_grad_clears_pending():
    route, P, s, log = make(sink=True, reduce=True)
    route.synced = False
    route.hand_over(P, DEV)
    assert route.pending is True
    s.zero_grad()
    assert route.pending is False and s._fresh and not s.flat_g.any()
    route.synced = True
    route.hand_over(P, DEV)  # a fresh synchronised backward: the plain single allreduce
    assert events(log)[2:] == [("bwd", None), ("reduce", "pgrad"), ("receive",)]


def test_bucketed_exchange_hands_every_bucket_over_once_in_completion_order():
    route, P, s, log = make(sink=True, reduce=True, overlap=True)
    assert route.hand_over(P, DEV) == (None,)
    segs = P.backward_segments()
    assert [(lo, hi) for lo, hi, _ in segs] == [(0, 7), (7, 11), (11, 16)]
    buckets = [(lo, hi) for lo, hi, _ in P.grad_buckets]
    want = []
    for (lo, hi, _), b in zip(segs, buckets):
        want += [("bwd", (lo, hi)), ("reduce_async", b)]
    want += [("finish", b) for b in buckets] + [("receive",)]
    assert events(log) == want
    received = log[-1][1]
    assert th.equal(received, 0.5 * P.values) and th.equal(s.flat_g, 0.5 * P.values)


def test_single_bucket_falls_back_to_one_graph_and_one_allreduce():
    route, P, s, log = make(sink=True, reduce=True, overlap=True, buckets=((0, 12, 15),))
    assert route.hand_over(P, DEV) == (None,)
    assert events(log) == [("bwd", None), ("reduce", "pgrad"), ("receive",)]
    assert th.equal(s.flat_g, 0.5 * P.values)


def test_sink_with_blocking_reduce():
    route, P, s, log = make(sink=True, reduce=True)
    assert route.hand_over(P, DEV) == (None,)
    assert events(log) == [("bwd", None), ("reduce", "pgrad"), ("receive",)]
    assert th.equal(s.flat_g, 0.5 * P.values)


def test_grad_route_is_created_once_per_module():
    m, other = th.nn.Linear(2, 2), th.nn.Linear(2, 2)
    r = grad_route(m)
    assert grad_route(m) is r and grad_route(other) is not r
    assert (r.sink, r.reduce, r.reduce_async, r.synced, r.pending) == (None, None, None, True, False)
    assert [n for n, _ in m.named_parameters()] == ["weight", "bias"] and "_grad_route" not in m.state_dict()

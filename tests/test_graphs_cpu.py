"""Host-side state machine of graphs.GraphedViewStep with the capture replaced by a recording stand-in (no GPU): first
visit eager, second visit captures, later visits replay; a changed guard or a replaced parameter drops every graph;
a failing capture leaves the view eager; least-recently-used graphs go first; accumulate adds into an existing .grad."""
import torch

from opengaussian_b200 import graphs
from opengaussian_b200._lib import OgsError


class _FakeGraph:
    def __init__(self, fn):
        self.fn = fn

    def replay(self):
        self.fn()


class _Step(graphs.GraphedViewStep):
    """Captures by running the loss once and remembering how to run it again into the same buffers."""
    fail_for = ()

    def _graphable(self):
        return True

    def _capture(self, view, sig):
        if view in self.fail_for:
            raise OgsError("not capturable")
        g = graphs._Graph()
        g.sig, g.pins = sig, []
        for p in self.params:
            p.grad = None
        loss = self.view_loss(view)
        loss.backward()
        g.loss = loss.detach().clone()
        g.grads = [p.grad for p in self.params]

        def again():
            fresh = torch.autograd.grad(self.view_loss(view), self.params)
            for buf, f in zip(g.grads, fresh):
                buf.copy_(f)
            g.loss.copy_(self.view_loss(view).detach())
        g.graph = _FakeGraph(again)
        self.captures += 1
        return g


def test_visit_sequence_guard_and_replacement():
    w = torch.tensor([1.0, 2.0, 3.0], requires_grad=True)
    version = [0]
    st = _Step(lambda v: (w * w).sum() * v, [w], guard=lambda: version[0])
    for visit, want in enumerate([dict(eager=1, captures=0, replays=0), dict(eager=1, captures=1, replays=1),
                                  dict(eager=1, captures=1, replays=2)]):
        loss = st(2.0)
        assert float(loss) == 28.0 and torch.equal(w.grad, 4.0 * w.detach())
        s = st.stats()
        assert {k: s[k] for k in want} == want, (visit, s)
    with torch.no_grad():
        w.mul_(2.0)                                   # an optimizer step: same tensor, the replay must see the new values
    assert float(st(2.0)) == 112.0 and torch.equal(w.grad, 4.0 * w.detach()) and st.stats()["replays"] == 3
    version[0] += 1                                   # the guard reports a change: start over
    st(2.0)
    assert st.stats()["graphs"] == 0 and st.stats()["eager"] == 2
    st(2.0)
    assert st.stats()["graphs"] == 1 and st.stats()["captures"] == 2
    w2 = w.detach().clone().requires_grad_(True)      # a REPLACED parameter
    st.params = [w2]
    st.view_loss = lambda v: (w2 * w2).sum() * v
    st(2.0)
    assert st.stats()["graphs"] == 0 and w2.grad is not None


def test_failed_capture_stays_eager_and_lru():
    w = torch.ones(2, requires_grad=True)
    st = _Step(lambda v: (w * v).sum(), [w], max_graphs=2)
    st.fail_for = (7.0,)
    for _ in range(4):
        assert float(st(7.0)) == 14.0
    assert st.stats() == dict(graphs=0, replays=0, captures=0, eager=4)
    for v in (1.0, 2.0, 3.0):
        st(v)
        st(v)
    assert st.stats()["graphs"] == 2 and 1.0 not in st._graphs and 3.0 in st._graphs     # least recently used dropped
    st(2.0)
    st(4.0)
    st(4.0)
    assert 2.0 in st._graphs and 3.0 not in st._graphs


def test_accumulate_adds_into_existing_grad():
    w = torch.tensor([1.0, -1.0], requires_grad=True)
    st = _Step(lambda v: (w * v).sum(), [w])
    for rep in range(3):                               # eager, capture + replay, replay
        st(1.0)
        first = w.grad.clone()
        st(5.0, accumulate=True)
        assert torch.equal(w.grad, first + 5.0), rep
    assert st.stats()["graphs"] == 2


def test_accumulate_in_any_order_across_eager_capture_and_replay():
    """A, B(acc), A(acc): a replayed view that finds its own earlier output in .grad must still add to it."""
    w = torch.tensor([1.0, -1.0], requires_grad=True)
    st = _Step(lambda v: (w * v).sum(), [w])
    for rep in range(4):                               # eager, capture + replay, replay, replay
        st(1.0)
        st(5.0, accumulate=True)
        st(1.0, accumulate=True)
        assert torch.equal(w.grad, torch.full((2,), 7.0)), (rep, w.grad)
    assert st.stats()["graphs"] == 2 and st.stats()["replays"] >= 6


def test_zero_grad_then_accumulate_every_view_in_changing_orders():
    """optimizer.zero_grad() (both forms) and then step(v, accumulate=True) for every view, in a new order each step --
    from the start, and after single-view steps (accumulate=False) have visited and captured every view."""
    w = torch.tensor([1.0, 2.0, -1.0], requires_grad=True)
    views = (1.0, 2.0, 3.0, 4.0)
    orders = [(0, 1, 2, 3), (3, 2, 1, 0), (1, 3, 0, 2), (2, 0, 3, 1), (0, 2, 1, 3), (3, 1, 2, 0)]
    for set_to_none in (False, True):
        for single_view_first in (False, True):
            w.grad = None
            st = _Step(lambda v: (w * w).sum() * v, [w])
            opt = torch.optim.SGD([w], lr=0.0)
            if single_view_first:
                for v in views + views:
                    st(v)
            for k, order in enumerate(orders):             # eager, capture, then replays
                opt.zero_grad(set_to_none=set_to_none)
                for i in order:
                    st(views[i], accumulate=True)
                assert torch.equal(w.grad, 2.0 * w.detach() * sum(views)), (set_to_none, single_view_first, k, w.grad)
            assert st.stats()["graphs"] == 4


def test_returned_loss_and_grad_outlive_later_replays():
    """A loss (or a .grad) the caller keeps is not overwritten by later steps, of the same view or another one."""
    w = torch.tensor([1.0, 2.0], requires_grad=True)
    st = _Step(lambda v: (w * w).sum() * v, [w])
    for _ in range(2):                                 # eager, capture: the graphs exist from here on
        st(1.0)
        st(2.0)
    kept = []
    for scale in (1.0, 2.0, 3.0):
        with torch.no_grad():
            w.copy_(torch.tensor([1.0, 2.0]) * scale)
        for v in (1.0, 2.0):
            loss = st(v)
            kept.append((loss, float(loss), w.grad, w.grad.clone()))
    assert st.stats()["replays"] >= 7
    for loss, value, grad, grad_value in kept:
        assert float(loss) == value and torch.equal(grad, grad_value)

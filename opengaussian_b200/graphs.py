"""One frozen-geometry training step per camera as a CUDA graph.

From Stage 1 on (train.py:431-436) a step of OpenGaussian's loop -- render() of one training camera
(gaussian_renderer/__init__.py:22-373), the SAM-mask statistics and losses (train.py:441-456), loss.backward()
(:497-498) -- is a fixed sequence of kernels over fixed addresses once the camera's geometry is resident
(rasterizer.ViewCache): about fourteen launches and 0.6 ms of GPU work at 1 M Gaussians, behind roughly 1 ms of
Python, ctypes and autograd bookkeeping.  ``GraphedViewStep`` captures that sequence once per camera (second visit)
and afterwards replays it with one launch; the host no longer bounds the step.

    step = GraphedViewStep(view_loss, [gaussians._ins_feat], guard=geometry_guard(gaussians))
    loss = step(view)            # visit 1: eager (fills the view cache); visit 2: capture + replay; then replay
    optimizer.step()             # reads gaussians._ins_feat.grad as usual

Contract (the usual one of CUDA graphs, stated once): ``view_loss(view)`` must be a function of the view, the
parameters' CURRENT VALUES and tensors that stay alive at the same address (camera matrices, SAM id maps, background);
its Python side effects happen only on the eager and the capturing visit.  Parameters are read in place, so optimizer
steps are seen; a parameter that is REPLACED by a new tensor (or any change the ``guard`` reports, e.g. the geometry's
version counters) drops the graphs and starts over.  Gradients are written, not accumulated: after the call
``p.grad`` is this view's gradient in a tensor of its own, as after an eager backward; ``step(view, accumulate=True)``
adds it to an existing ``.grad`` instead (the 2nd..Vth view of a multi-view step, in any order, or every view after
``optimizer.zero_grad(set_to_none=False)``).  The returned loss is a tensor of its own as well.  A replay's outputs
are copied out of the graph before the call returns (one read and one write of each gradient: 48 MB of traffic at
1 M Gaussians x 6 channels), so no ``.grad`` and no loss the caller holds is ever a graph's buffer -- which a later
replay of that graph, or of another graph whose intermediates share its memory, would overwrite.  That is also why
every view's graph can share one memory pool: the graphs never run concurrently and nothing they write outlives the
call, so the step keeps one set of intermediates instead of one per camera.  Camera matrices, like the parameters, are read in place: a camera edited in place needs ``reset()`` (or a
``guard`` that reports it).
Anything that cannot be captured -- a view whose geometry is not resident (cache disabled or over budget), trainable
geometry (the forward then has to read the frame's duplicate count back) -- runs eagerly, every time, with the same
results."""
import collections
import warnings
from typing import Callable, Hashable, Iterable, Optional

import torch

from . import rasterizer as _rz


def geometry_guard(pc) -> Callable[[], tuple]:
    """Guard for a GaussianModel-like object: the frozen parameters' storage, shape and version counters
    (scene/gaussian_model.py:66-74) plus the SH degree -- whatever makes rasterizer.ViewCache miss."""
    names = ("_xyz", "_scaling", "_rotation", "_opacity", "_features_dc", "_features_rest")

    def guard():
        return tuple(_rz._sig(getattr(pc, n, None)) for n in names) + (getattr(pc, "active_sh_degree", None),)
    return guard


class _Graph:
    __slots__ = ("graph", "loss", "grads", "sig", "pins")


class GraphedViewStep:
    def __init__(self, view_loss: Callable, params: Iterable[torch.Tensor], guard: Optional[Callable[[], Hashable]] = None,
                 key: Optional[Callable] = None, max_graphs: Optional[int] = None):
        self.view_loss = view_loss
        self.params = list(params)
        self.guard = guard or (lambda: None)
        self.key = key or (lambda v: v if isinstance(v, Hashable) else id(v))
        self.max_graphs = max_graphs
        self._graphs = collections.OrderedDict()     # view key -> _Graph (least recently used first)
        self._seen = set()                           # views that have had their eager visit under the current signature
        self._eager_only = set()                     # views whose capture failed: not tried again until the signature changes
        self._pool = None
        self._sig = None
        self.replays = self.captures = self.eager = 0

    def _signature(self):
        return (tuple((p.data_ptr(), tuple(p.shape), p.dtype, p.requires_grad) for p in self.params), self.guard())

    def reset(self):
        self._graphs.clear()
        self._seen.clear()
        self._eager_only.clear()

    def stats(self):
        return dict(graphs=len(self._graphs), replays=self.replays, captures=self.captures, eager=self.eager)

    def _graphable(self):
        return bool(self.params) and self.params[0].is_cuda

    def _eager(self, view, accumulate=False):
        if not accumulate:
            for p in self.params:
                p.grad = None
        loss = self.view_loss(view)
        loss.backward()
        self.eager += 1
        return loss.detach()

    def _capture(self, view, sig):
        dev = self.params[0].device
        if self._pool is None:
            self._pool = torch.cuda.graph_pool_handle()   # one pool for every view's graph (see the module docstring)
        for p in self.params:
            p.grad = None
        g = _Graph()
        g.graph = torch.cuda.CUDAGraph()
        g.sig = sig
        g.pins = []
        prev = _rz._CAPTURE_PINS.get(dev.index)
        _rz._CAPTURE_PINS[dev.index] = g.pins             # the rasterizer records the cache buffers the capture reads
        try:
            with warnings.catch_warnings():
                warnings.filterwarnings("ignore", message="The CUDA Graph is empty")   # a refused capture ends empty
                with torch.cuda.graph(g.graph, pool=self._pool):
                    loss = self.view_loss(view)
                    loss.backward()
                    g.loss = loss.detach()
        finally:
            if prev is None:
                _rz._CAPTURE_PINS.pop(dev.index, None)
            else:
                _rz._CAPTURE_PINS[dev.index] = prev
        g.grads = [p.grad for p in self.params]
        self.captures += 1
        return g

    def __call__(self, view, accumulate: bool = False) -> torch.Tensor:
        if not self._graphable():
            return self._eager(view, accumulate)
        sig = self._signature()
        if sig != self._sig:                # parameters replaced or geometry changed: every graph reads stale addresses
            self.reset()
            self._sig = sig
        k = self.key(view)
        g = self._graphs.get(k)
        if g is None:
            if k in self._eager_only or k not in self._seen:
                self._seen.add(k)
                return self._eager(view, accumulate)
            held = [p.grad for p in self.params] if accumulate else None     # the capture starts from .grad = None
            try:
                g = self._capture(view, sig)
            except (_rz._lib.OgsError, RuntimeError):
                self._eager_only.add(k)
                if self.params[0].is_cuda:
                    torch.cuda.synchronize(self.params[0].device)
                if held is not None:
                    for p, h in zip(self.params, held):
                        p.grad = h
                return self._eager(view, accumulate)
            if held is not None:
                for p, h in zip(self.params, held):
                    p.grad = h
            self._graphs[k] = g
            if self.max_graphs is not None:
                while len(self._graphs) > self.max_graphs:
                    self._graphs.popitem(last=False)
        else:
            self._graphs.move_to_end(k)
        g.graph.replay()
        self.replays += 1
        for p, gr in zip(self.params, g.grads):
            if gr is None:
                if not accumulate:
                    p.grad = None
            elif accumulate and p.grad is not None:
                p.grad.add_(gr)
            else:
                p.grad = gr.clone()
        return g.loss.clone()

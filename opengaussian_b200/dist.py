"""Multi-GPU plumbing (one process per GPU, torch.distributed; NCCL over NVLink on the B200 box,
gloo in the CPU tests).  The reference has no distributed code at all (SURVEY.md section 5); the
hot path shards in exactly two places (section 8e):

* rasterizer: over CAMERA VIEWS -- every rank renders its own views against a full replica of the
  Gaussians; per-parameter gradients are summed with all-reduce (`allreduce_gradients`);
* forward-only sweeps (construct_pseudo_ins_feat, the Stage-2.2 / Stage-3 association loops of
  train.py:676-681,755-760,846-856): over CAMERA VIEWS too, with no collective for the images; the per-view
  columns of `match_info [k1*k2, V, 3]` are merged once at the end (`merge_view_columns`) and the per-cluster
  object counts `iClusterSubNum [k1]` with one all-reduce(max) (`allreduce_max`);
* k-means: over POINTS -- every rank owns a contiguous shard, centres are replicated, and one
  all-reduce of the packed [k*D sums | k counts] buffer is done per Lloyd iteration
  (`shard_kmeans` switches a Quantize_kMeans instance into that mode; ids stay sharded,
  `gather_ids` collects them when a caller such as save_kmeans needs the full vector).

No collective is invented where the path does not exchange data: a single frame is never split
across GPUs.
"""
from typing import Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist


def world(group=None):
    if not dist.is_available() or not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def split_views(views: Sequence, group=None) -> List:
    """Round-robin shard of a view list: rank r gets views r, r+R, r+2R, ..."""
    r, w = world(group)
    return list(views[r::w])


def shard_range(n: int, group=None):
    """Contiguous [lo, hi) shard of n items for this rank (k-means points)."""
    r, w = world(group)
    per = (n + w - 1) // w
    return min(n, r * per), min(n, (r + 1) * per)


def _flat_layout(params):
    """Offsets (in floats) of every parameter's gradient in the step's flat buffer: the parameters in the given
    order, each slice aligned to 64 floats -- a function of the parameter SHAPES only, hence identical on every
    rank.  It is also the layout the rasterizer's backward carves its gradients from (rasterizer.py), so that
    buffer is reduced in place when the caller lists the parameters in the rasterizer's order."""
    offs, total = [], 0
    for p in params:
        offs.append(total)
        total += (p.numel() + 63) // 64 * 64
    span = offs[-1] + params[-1].numel() if params else 0
    return offs, span


def allreduce_gradients(params: Iterable[torch.Tensor], group=None, bucket_bytes: int = 1 << 30,
                        average: bool = False):
    """Sums .grad of every parameter across ranks with ONE collective over a flat fp32 buffer (split into
    `bucket_bytes` pieces only beyond that size: NVSwitch gives every peer full bandwidth, so buckets are sized for
    launch latency, not link count).  The collective sequence is RANK-INVARIANT: its element count comes from the
    parameter shapes alone (`_flat_layout`), and a parameter whose .grad is None on this rank -- a rank that had
    no view this step -- contributes zeros.  Afterwards every .grad is a view into the reduced buffer."""
    r, w = world(group)
    if w == 1:
        return
    params = [p for p in params if p.requires_grad]
    if not params:
        return
    offs, span = _flat_layout(params)
    flat = _coalesced_grads(params, offs, span)
    arena = _ARENAS.get(params[0].device.index) if params[0].is_cuda else None
    if arena is not None and arena.owns(flat, span):
        arena.all_reduce(span)                    # one kernel of ours: the NVSwitch reduces in flight
        if average:
            flat.div_(w)
        return
    packed = flat is None
    if packed:
        flat = torch.zeros(span, dtype=torch.float32, device=params[0].device)
        for p, o in zip(params, offs):
            if p.grad is not None:
                flat[o:o + p.numel()].copy_(p.grad.reshape(-1))
    step = max(1, bucket_bytes // 4)
    for lo in range(0, span, step):
        dist.all_reduce(flat[lo:lo + step], group=group)
    if average:
        flat.div_(w)
    if packed:
        for p, o in zip(params, offs):
            g = flat[o:o + p.numel()].view(p.shape)
            p.grad = g if p.dtype == torch.float32 else g.to(p.dtype)


def _coalesced_grads(params, offs=None, span=None) -> Optional[torch.Tensor]:
    """If every .grad is a contiguous fp32 view into ONE storage laid out exactly as `_flat_layout` says, returns
    that span as a flat tensor (the alignment gaps between the slices ride along), else None."""
    params = list(params)
    if offs is None:
        offs, span = _flat_layout(params)
    grads = [p.grad for p in params]
    if not grads or any(g is None or g.dtype != torch.float32 or not g.is_contiguous() for g in grads):
        return None
    st = grads[0].untyped_storage()
    base = grads[0].storage_offset()
    for g, o in zip(grads, offs):
        if g.untyped_storage().data_ptr() != st.data_ptr() or g.storage_offset() - base != o:
            return None
    if (base + span) * 4 > st.nbytes():
        return None
    return torch.empty(0, dtype=torch.float32, device=grads[0].device).set_(st, base, (span,))


_ARENAS = {}


class GradArena:
    """Symmetric-memory home of the step's gradient buffer + its all-reduce through the NVSwitch multicast mapping.

    The rasterizer's backward carves every parameter gradient out of ONE flat buffer (rasterizer.py); with an arena
    installed that buffer lives in memory that all ranks of the node map into one multicast address range
    (torch.distributed._symmetric_memory does the allocation and the rendezvous -- plumbing), and
    `allreduce_gradients` sums it with ONE kernel of libogs_b200 (csrc/nvls.cu: multimem.ld_reduce / multimem.st,
    the switch adds the ranks' copies in flight) bracketed by two stream-ordered cross-rank barriers, instead of a
    library all-reduce.  `kind` says what is in use; without multicast support the arena is not installed and the
    gradients go through torch.distributed as before."""

    def __init__(self, n_floats: int, group=None, device=None):
        from . import _lib
        from .rasterizer import set_grad_arena
        self._lib = _lib
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = world(group)
        self.kind = "torch.distributed all_reduce"
        self.buf = None
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.world == 1:
            return
        n = (int(n_floats) + 4 * self.world + 63) // 64 * 64
        ok = 1
        try:
            import torch.distributed._symmetric_memory as symm_mem
            buf = symm_mem.empty(n, dtype=torch.float32, device=self.device)
            hdl = symm_mem.rendezvous(buf, self.group)
            mc = int(hdl.multicast_ptr) if hdl.has_multicast_support else 0
            if mc == 0:
                ok = 0
        except Exception as e:      # noqa: BLE001  (no symmetric memory / multicast on this box)
            self.error = repr(e)
            ok = 0
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=group)
        if not all(flags):
            return
        buf.zero_()
        self.buf, self.hdl, self.mc = buf, hdl, mc
        self.kind = "one kernel: multimem.ld_reduce + multimem.st through the NVSwitch multicast mapping (ogs_multimem_allreduce_f32)"
        set_grad_arena(buf)
        _ARENAS[self.device.index] = self

    def enable(self, on: bool):
        """Installs / removes the arena as the home of the gradient buffer (it stays allocated either way)."""
        from .rasterizer import set_grad_arena
        if self.buf is None:
            return
        if on:
            set_grad_arena(self.buf)
            _ARENAS[self.device.index] = self
        else:
            set_grad_arena(None)
            _ARENAS.pop(self.device.index, None)

    def owns(self, flat: Optional[torch.Tensor], span: int) -> bool:
        return (self.buf is not None and flat is not None and flat.data_ptr() == self.buf.data_ptr()
                and span <= self.buf.numel())

    def all_reduce(self, n_floats: int, barriers: bool = True):
        """In-place sum over the ranks of the first n_floats of the arena, enqueued on the current stream.
        (barriers=False is a timing aid only: the result is then unordered against the other ranks' writes.)"""
        n = (int(n_floats) + 3) // 4 * 4
        if barriers:
            self.hdl.barrier(channel=0)             # every rank's gradients are written
        self._lib.launch("ogs_multimem_allreduce_f32", self.device, self.mc, n, self.rank, self.world)
        if barriers:
            self.hdl.barrier(channel=1)             # every slice has been stored everywhere

    def close(self):
        from .rasterizer import set_grad_arena
        if self.buf is not None:
            set_grad_arena(None)
            _ARENAS.pop(self.device.index, None)
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
            self.buf = None


def shard_kmeans(codebook, group=None, peer_reduce: bool = False):
    """Puts a Quantize_kMeans into sharded mode: its forward() then sees only this rank's points.
    peer_reduce=True (CUDA, one node): the per-pass all-reduce of the centroid partials is done by the library's own
    one-kernel reduction over NVLink peer memory (PeerReducer) instead of a torch.distributed call."""
    r, w = world(group)
    codebook.process_group = group
    codebook.distributed = w > 1
    if peer_reduce and w > 1:
        k1, k2 = codebook.num_clusters, codebook.leaf_num_clusters
        codebook.reducer = PeerReducer(max(k1 * (codebook.vec_dim + 1) * 4, k1 * k2 * (codebook.leaf_vec_dim + 1) * 8) + 256,
                                       group=group)
    return codebook


class PeerReducer:
    """In-place all-reduce(sum) of a small float32 / int64 CUDA tensor in ONE kernel over NVLink peer memory
    (C ABI ogs_peer_*, csrc/peer.cu): every rank pushes its vector into every rank's inbox, signals, waits, and sums
    the inbox in rank order (bit-identical results on all ranks).  ~5 us per call against ~45 us for a library
    collective of a few KB -- what the sharded k-means needs once per Lloyd pass (SURVEY.md 8e).  torch.distributed is
    only used once, to exchange the 64-byte memory handles.  If peer memory cannot be mapped (`kind == "nccl"`)
    the calls go to torch.distributed.all_reduce instead."""

    def __init__(self, max_bytes: int, group=None, device=None):
        import ctypes as C
        from . import _lib
        self.group = group
        self.rank, self.world = world(group)
        self.kind = "nccl"
        self.comm = None
        self._C, self._lib = C, _lib
        if self.world == 1:
            self.kind = "single"
            return
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        L = _lib.lib()
        handle = (C.c_char * 64)()
        comm = C.c_void_p()
        ok = 1
        with torch.cuda.device(self.device):
            rc = L.ogs_peer_comm_create(self.rank, self.world, int(max_bytes), C.byref(comm), handle)
        if rc != 0:
            ok = 0
        handles = [None] * self.world
        dist.all_gather_object(handles, (ok, bytes(handle)), group=group)
        if all(h[0] for h in handles):
            blob = b"".join(h[1] for h in handles)
            with torch.cuda.device(self.device):
                rc = L.ogs_peer_comm_connect(comm, blob)
            ok = 1 if rc == 0 else 0
        else:
            ok = 0
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=group)
        if all(flags):
            self.comm, self.kind = comm, "nvlink peer memory, one kernel (ogs_peer_allreduce)"
        elif comm:
            L.ogs_peer_comm_destroy(comm)

    def all_reduce(self, t: torch.Tensor):
        if self.world == 1:
            return t
        if self.comm is None:
            dist.all_reduce(t, group=self.group)
            return t
        if not t.is_contiguous() or t.dtype not in (torch.float32, torch.int64):
            raise self._lib.OgsError("PeerReducer.all_reduce needs a contiguous float32 or int64 tensor")
        self._lib.launch("ogs_peer_allreduce", t.device, self.comm, t.data_ptr(), t.numel(),
                         0 if t.dtype == torch.float32 else 1)
        return t

    def check(self):
        """Raises if a call timed out waiting for a peer (synchronises the current stream)."""
        if self.comm is not None:
            L = self._lib.lib()
            stream = self._C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            with torch.cuda.device(self.device):
                if L.ogs_peer_comm_error(self.comm, stream) != 0:
                    raise self._lib.OgsError("ogs_peer_allreduce: a rank did not arrive within the time-out")

    def close(self):
        if self.comm is not None:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)         # nobody unmaps while a peer may still push
            self._lib.lib().ogs_peer_comm_destroy(self.comm)
            self.comm = None


def bind_to_gpu_numa_node(local_rank: int) -> Optional[int]:
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, so that pinned host buffers (first touch)
    and the copy engine's reads stay on the GPU's own socket: with 8 ranks feeding ~25 GB/s each from one node the
    cross-socket link is what limits the end-to-end step.  Best effort: returns the node, or None if the topology
    cannot be read (then nothing changes)."""
    import os
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev_id = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def gather_ids(local_ids: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather of the sharded id vector (shards may differ in length)."""
    r, w = world(group)
    if w == 1:
        return local_ids
    n = torch.tensor([local_ids.numel()], dtype=torch.int64, device=local_ids.device)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n, group=group)
    m = int(max(int(s) for s in sizes))
    pad = torch.zeros(m, dtype=local_ids.dtype, device=local_ids.device)
    pad[:local_ids.numel()] = local_ids
    outs = [torch.zeros_like(pad) for _ in range(w)]
    dist.all_gather(outs, pad, group=group)
    return torch.cat([o[:int(s)] for o, s in zip(outs, sizes)])


def view_indices(n_views: int, group=None) -> List[int]:
    """Indices of the views `split_views` gives this rank (r, r+R, ...): the columns of a per-view table it owns."""
    r, w = world(group)
    return list(range(r, n_views, w))


def merge_view_columns(table: torch.Tensor, view_dim: int = 1, group=None) -> torch.Tensor:
    """Merges a per-view table whose columns were filled by the ranks that rendered those views
    (`match_info [k1*k2, V, 3]`, train.py:844-890; rank r owns the columns `view_indices(V)`): every rank ends up
    with the complete table.  Columns a rank does not own are ignored (they need not be zero)."""
    r, w = world(group)
    if w == 1:
        return table
    own = torch.zeros(table.shape[view_dim], dtype=torch.bool, device=table.device)
    own[r::w] = True
    shape = [1] * table.dim()
    shape[view_dim] = -1
    merged = torch.where(own.view(shape), table, torch.zeros_like(table)).contiguous()
    dist.all_reduce(merged, op=dist.ReduceOp.SUM, group=group)      # disjoint supports: the sum is a merge
    return merged


def allreduce_max(t: torch.Tensor, group=None) -> torch.Tensor:
    """Element-wise maximum over ranks, in place (`iClusterSubNum [k1]`, train.py:754,804: the largest number of
    objects any view saw in a coarse cluster)."""
    r, w = world(group)
    if w > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t


_SIDE_STREAMS = {}


def _side_streams(device, n):
    key = (str(device), n)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = [torch.cuda.Stream(device) for _ in range(n)]
    return _SIDE_STREAMS[key]


def render_views_backward(render_loss, views: Sequence, params: Iterable[torch.Tensor], group=None,
                          already_split: bool = False, streams: int = 1,
                          fuse_accumulate: bool = True, reduce: bool = True, lookahead: int = 1,
                          defer_capacity_check: bool = True) -> Optional[torch.Tensor]:
    """One view-parallel step: this rank renders ITS views (`render_loss(view) -> scalar loss`),
    backpropagates, and the parameter gradients of all ranks are summed.  Equivalent to one
    process rendering every view and summing the losses.

    ``streams > 1`` (CUDA only, experimental) round-robins the rank's views over that many side streams.
    Measured on B200 (1 M Gaussians, 1080p): +3 % at best -- the binning kernels' large CTAs do not get
    scheduled under a machine full of blend CTAs -- and occasional multi-millisecond allocator stalls,
    so the default stays 1.  Gradients still accumulate in ``.grad`` (autograd orders the accumulation
    across streams); the caller's stream waits for every side stream before the all-reduce.
    ``fuse_accumulate`` lets the rasterizer's backward add the 2nd..Vth view's gradients straight into the
    parameters' existing ``.grad`` inside its kernel (rasterizer.fuse_grad_accumulation) when the parameters
    are fed to the rasterizer directly (leaf inputs, e.g. the raw-parameter path).
    ``lookahead = 1`` (default) issues the forward of view v+1 BEFORE the backward of view v (forwards and backwards
    each stay in view order, so the gradients are summed in the same order): the rasterizer's forward makes the host
    wait for the frame's duplicate count, and with the previous view's backward still to be queued behind it the GPU
    always has more than a millisecond of work in its queue while the host catches up (without it the queue holds
    0.45 ms at that point and runs dry whenever the host needs longer).  Costs one extra forward state in memory.
    ``defer_capacity_check`` (default) removes that wait altogether by treating the step as a transaction: when no
    parameter holds a ``.grad`` on entry, the forwards run under ``rasterizer.deferred_capacity_check`` (buffers sized
    from the running estimate, nothing read back), and once every backward has been queued -- BEFORE the gradients
    meet any collective -- the frames' real counts are checked.  If one did not fit (a view with over 25 % more
    duplicates than any recent one: rare), the gradients are dropped and the rank's views are rendered again with the
    ordinary synchronous check; ``render_loss`` is then called a second time for those views, so it must be a function
    of the parameters and the view only (side effects happen twice)."""
    from .rasterizer import capacity_overflowed, deferred_capacity_check, fuse_grad_accumulation
    mine = views if already_split else split_views(views, group)
    params = list(params)
    total = None

    def finish(res):
        """render_loss may return a scalar loss, (outputs, grad_outputs) to be back-propagated as is, an already
        back-propagated (detached) loss, or a dict {"outputs", "grads", "loss" (detached, optional), "after"
        (callable run once the backward has been queued, optional)}."""
        if isinstance(res, dict):
            torch.autograd.backward(res["outputs"], res["grads"])
            if res.get("after") is not None:
                res["after"]()
            return res.get("loss")
        if isinstance(res, tuple):
            torch.autograd.backward(res[0], res[1])
            return None
        if res.requires_grad:
            res.backward()
        return res.detach()

    def run(v):
        return finish(render_loss(v))

    use_streams = streams > 1 and len(mine) > 1 and params and params[0].is_cuda
    if use_streams:
        dev = params[0].device
        cur = torch.cuda.current_stream(dev)
        side = _side_streams(dev, min(streams, len(mine)))
        parts = []
        for s in side:
            s.wait_stream(cur)
        for i, v in enumerate(mine):
            s = side[i % len(side)]
            with torch.cuda.stream(s):
                part = run(v)
                if part is not None:
                    parts.append(part)
        for s in side:
            cur.wait_stream(s)
        for p_ in parts:
            p_.record_stream(cur)
            total = p_ if total is None else total + p_
    else:
        def local_pass(defer):
            tot = None
            pending = []                  # forwards whose backward has not been issued yet (at most `lookahead`)
            with fuse_grad_accumulation(fuse_accumulate), deferred_capacity_check(defer):
                for v in list(mine) + [None] * max(0, lookahead):
                    if v is not None:
                        pending.append(render_loss(v))
                    if pending and (v is None or len(pending) > max(0, lookahead)):
                        part = finish(pending.pop(0))
                        if part is not None:
                            tot = part if tot is None else tot + part
                while pending:
                    part = finish(pending.pop(0))
                    if part is not None:
                        tot = part if tot is None else tot + part
            return tot

        defer = bool(defer_capacity_check and mine and params and params[0].is_cuda
                     and all(p.grad is None for p in params))
        total = local_pass(defer)
        if defer and capacity_overflowed(params[0].device):
            for p in params:
                p.grad = None
            total = local_pass(False)
    r, w = world(group)
    if not reduce:          # measurement aid: the step without its collectives (bench.py's exposed-collective figure)
        return total
    allreduce_gradients(params, group)
    if w > 1:
        # rank-invariant: a rank without views this step (fewer views than ranks) contributes a zero loss
        if total is None:
            dev = params[0].device if params else torch.device("cpu")
            total = torch.zeros((), dtype=torch.float32, device=dev)
        dist.all_reduce(total, group=group)
    return total

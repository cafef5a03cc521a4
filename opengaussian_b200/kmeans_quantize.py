"""Drop-in for ``scene/kmeans_quantize.py::Quantize_kMeans`` (reference :12-280): the two-level
k-means codebook of OpenGaussian stages 2.1 / 2.2, with the assign / centroid-sum / finalize /
gather work done by libogs_b200.so (kmeans.cu) instead of chunked torch.cdist + one-hot GEMMs.

Same constructor, same ``forward(gaussian, iteration, assign, mode, selected_leaf, pos_weight)``,
same public attributes (``centers, leaf_centers, iLeafSubNum, cls_ids, leaf_cls_ids, nn_index``
-- read/written by train.py:206-215,299,310,355,626 and save_kmeans train.py:62-100) with the same
dtypes (ids int64, centres float32).  Reproduced quirks of ``cluster_assign`` (:146-241):
``counts`` starts at 1e-6, gains 1e-6 per 10000-point chunk (``N // 10000 + 1`` chunks, the
strict ``i*chunk > N`` break) and is zeroed only where > 0.1, so empty clusters get centre 0;
leaf mode rewrites all ``leaf_num`` rows of the selected block although only
``iLeafSubNum[selected]`` compete; unassigned points carry the sentinel id ``k1*k2``; argmin ties
go to the lowest index.  ``update_centers`` (:58-78) discards its result in the reference, so the
non-assign call is a no-op on the centres here as well.

The padded index lists built by ``equalize_cluster_size`` (:89-144: ``cluster_ids, cluster_len,
max_cnt, excl_clusters, excl_cluster_ids``) only feed that discarded computation; they are
materialised lazily on first access.
"""
import torch

from . import _lib

CHUNK = 10000  # reference chunk size (:178); only its count matters (the eps added to counts)


def kmeans_assign(a, b, scale_b, centers, select_ids=None, selected=-1, id_offset=0, ids_out=None,
                  sums=None, counts=None):
    """One fused assign (+ optional centroid sums/counts accumulation) pass through the C ABI.
    a [N,Da] (+ b [N,Db] * scale_b) vs centers [k, Da+Db]; returns ids (int64 [N])."""
    a = a.detach()
    if a.dtype != torch.float32 or not a.is_contiguous():
        a = a.float().contiguous()
    if b is not None:
        b = b.detach()
        if b.dtype != torch.float32 or not b.is_contiguous():
            b = b.float().contiguous()
    centers = centers.detach().float().contiguous()
    N, Da = a.shape
    Db = 0 if b is None else b.shape[1]
    k = centers.shape[0]
    if a.device.type != "cuda":
        raise _lib.OgsError("k-means kernels need CUDA tensors (there is no CPU fallback)")
    if ids_out is None:
        ids_out = torch.empty(N, dtype=torch.int64, device=a.device)
    _lib.launch("ogs_kmeans_assign", a.device, N, _lib.ptr(a), Da, _lib.ptr(b), Db, float(scale_b), _lib.ptr(centers), k,
                _lib.ptr(select_ids), int(selected), int(id_offset), _lib.ptr(ids_out), _lib.ptr(sums), _lib.ptr(counts))
    return ids_out


def fixed_point_bits(n_points: int, max_abs: float) -> int:
    """Largest fix_bits <= 30 with max_abs * 2^fix_bits < 2^31 (the kernel's 32-bit partial words) and
    n_points * max_abs * 2^fix_bits < 2^62 (exact int64 centroid sums)."""
    import math
    e = max(0, math.floor(math.log2(float(max_abs))) + 1) if max_abs > 0 else 0
    n = max(1, math.ceil(math.log2(max(int(n_points), 1) + 1)))
    return int(max(0, min(30, 31 - e, 62 - n - e)))


def kmeans_assign_segmented(a, coarse_ids, seg_centers, seg_k, k2, ids_out=None, acc=None, fix_bits=30):
    """Fine level for ALL coarse clusters in one launch (C ABI ogs_kmeans_assign_segmented): point i competes among
    rows [c*k2, c*k2 + seg_k[c]) of seg_centers, c = coarse_ids[i]; ids_out[i] = c*k2 + argmin.  acc (int64
    [k1*k2*(D+1)], added to) receives the exact fixed-point centroid sums and counts."""
    a = a.detach()
    if a.dtype != torch.float32 or not a.is_contiguous():
        a = a.float().contiguous()
    if a.device.type != "cuda":
        raise _lib.OgsError("k-means kernels need CUDA tensors (there is no CPU fallback)")
    seg_centers = seg_centers.detach().float().contiguous()
    seg_k = seg_k.to(device=a.device, dtype=torch.int32).contiguous()
    coarse_ids = coarse_ids.to(torch.int64).contiguous()
    N, D = a.shape
    k1 = seg_k.numel()
    if seg_centers.shape[0] < k1 * k2 or seg_centers.shape[1] != D:
        raise _lib.OgsError(f"seg_centers must be [>= {k1 * k2}, {D}] (got {tuple(seg_centers.shape)})")
    if ids_out is None:
        ids_out = torch.full((N,), k1 * k2, dtype=torch.int64, device=a.device)
    if acc is not None and (acc.dtype != torch.int64 or acc.numel() < k1 * k2 * (D + 1) or not acc.is_contiguous()):
        raise _lib.OgsError("acc must be a contiguous int64 tensor of k1*k2*(D+1) elements")
    _lib.launch("ogs_kmeans_assign_segmented", a.device, N, _lib.ptr(a), D, _lib.ptr(coarse_ids), _lib.ptr(seg_centers),
                _lib.ptr(seg_k), k1, int(k2), _lib.ptr(ids_out), _lib.ptr(acc), int(fix_bits))
    return ids_out


class LloydWorkspace:
    """Device scratch of the one-launch Lloyd passes (ticket + per-CTA partial tables), zeroed once and reused."""

    def __init__(self, device, k=None, D=None, k1=None, k2=None):
        L = _lib.lib()
        n = L.ogs_kmeans_lloyd_workspace_bytes(k, D) if k1 is None else L.ogs_kmeans_lloyd_segmented_workspace_bytes(k1, k2, D)
        self.buf = torch.zeros((n + 3) // 4, dtype=torch.int32, device=device)


def lloyd_pass(a, b, scale_b, centers, counts_state, eps_add, ids_out, ws: LloydWorkspace, comm=None, k=None,
               select_ids=None, selected=-1, id_offset=0):
    """One Lloyd iteration in one launch (C ABI ogs_kmeans_lloyd_pass): `centers` [k_out, D] is updated in place from
    its first k rows; counts_state [k_out] carries the reference's count bookkeeping; comm = PeerReducer.comm when the
    points are sharded over GPUs."""
    k_out = centers.shape[0]
    k = k_out if k is None else k
    _lib.launch("ogs_kmeans_lloyd_pass", a.device, a.shape[0], _lib.ptr(a), a.shape[1], _lib.ptr(b),
                0 if b is None else b.shape[1], float(scale_b), _lib.ptr(centers), k, k_out, _lib.ptr(select_ids),
                int(selected), int(id_offset), _lib.ptr(ids_out), _lib.ptr(counts_state), float(eps_add), comm,
                _lib.ptr(ws.buf))


def lloyd_pass_segmented(a, coarse_ids, seg_centers, seg_k, k2, counts_state, ids_out, fix_bits, ws: LloydWorkspace,
                         comm=None, eps_add=1e-6):
    """One Lloyd pass of every coarse cluster's fine level in one launch (C ABI ogs_kmeans_lloyd_pass_segmented)."""
    _lib.launch("ogs_kmeans_lloyd_pass_segmented", a.device, a.shape[0], _lib.ptr(a), a.shape[1], _lib.ptr(coarse_ids),
                _lib.ptr(seg_centers), _lib.ptr(seg_k), seg_k.numel(), int(k2), _lib.ptr(ids_out), int(fix_bits),
                _lib.ptr(counts_state), float(eps_add), comm, _lib.ptr(ws.buf))


class _GatherStraightThrough(torch.autograd.Function):
    """_ins_feat_q = _ins_feat - _ins_feat.detach() + centres[ids][:, :D]  (reference :273-275)."""

    @staticmethod
    def forward(ctx, feat, centers, ids):
        f = feat.detach().float().contiguous()
        c = centers.detach().float().contiguous()
        out = torch.empty_like(f)
        _lib.launch("ogs_kmeans_gather_st", f.device, f.shape[0], _lib.ptr(f), f.shape[1], _lib.ptr(c), c.shape[1],
                    _lib.ptr(ids), _lib.ptr(out))
        return out

    @staticmethod
    def backward(ctx, g):
        return g, None, None


class Quantize_kMeans():
    def __init__(self, num_clusters=64, num_leaf_clusters=10, num_iters=10, dim=9, dim_leaf=6):
        self.num_clusters = num_clusters            # k1
        self.leaf_num_clusters = num_leaf_clusters  # k2
        self.num_kmeans_iters = num_iters
        self.vec_dim = dim                          # coarse level: ins_feat (6) + xyz (3)
        self.leaf_vec_dim = dim_leaf                # fine level: ins_feat only
        self.centers = torch.empty(0)               # [k1, 9]
        self.leaf_centers = torch.empty(0)          # [k1*k2+1, 6]
        self.iLeafSubNum = torch.empty(0)           # fine clusters actually used per coarse cluster
        self.cls_ids = torch.empty(0)               # coarse id per point (int64)
        self.leaf_cls_ids = torch.empty(0)          # fine id per point (int64)
        self.nn_index = torch.empty(0)

        self.max_cnt_th = 10000
        self._eq_cache = None                       # lazily built equalize_cluster_size products
        self._eq_mode = "root"
        # multi-GPU (SURVEY.md section 8e): points sharded over ranks, centres replicated; ONE
        # all-reduce of the packed [k*D sums | k counts] buffer per Lloyd iteration.  Set by
        # opengaussian_b200.dist.shard_kmeans(); None = single process (the reference's behaviour).
        self.process_group = None
        self.distributed = False
        self.reducer = None                         # dist.PeerReducer (in-kernel NVLink all-reduce) or None = torch.distributed
        self.pos_centers = torch.empty(0)

    # ------------------------------------------------------------------ lazily materialised lists
    def _equalized(self):
        if self._eq_cache is None:
            self._eq_cache = self._build_equalized(self._eq_mode)
        return self._eq_cache

    def _build_equalized(self, mode):
        """Index lists of the reference's equalize_cluster_size (:89-144), torch ops only."""
        nn_index = self.nn_index
        dev = nn_index.device
        num_clusters = self.num_clusters if mode == "root" else self.num_clusters * self.leaf_num_clusters + 1
        unq, n_unq = torch.unique(nn_index, return_counts=True)
        topk = min(100, len(n_unq))
        max_cnt_topk, topk_idx = torch.topk(n_unq, topk)
        max_cnt = max_cnt_topk[0]
        idx = 0
        excl = []
        while max_cnt > self.max_cnt_th:
            excl.append(unq[topk_idx[idx]])
            idx += 1
            if idx < topk:
                max_cnt = max_cnt_topk[idx]
            else:
                break
        excl = sorted(excl)
        excl_set = set(int(e) for e in excl)
        max_cnt_i = int(max_cnt)
        order = torch.argsort(nn_index, stable=True)
        counts = torch.bincount(nn_index.clamp(min=0), minlength=num_clusters)[:num_clusters]
        starts = torch.cumsum(counts, 0) - counts
        all_ids = torch.full((num_clusters, max_cnt_i), -1, dtype=torch.long, device=dev)
        excl_ids = []
        counts_c = counts.tolist()
        starts_c = starts.tolist()
        for i in range(num_clusters):
            members = order[starts_c[i]:starts_c[i] + counts_c[i]]
            if i in excl_set:
                excl_ids.append(members[max_cnt_i:])
                members = members[:max_cnt_i]
            all_ids[i, :members.numel()] = members
        return dict(cluster_ids=all_ids.reshape(-1), cluster_len=counts.to(torch.long).unsqueeze(1),
                    max_cnt=max_cnt, excl_clusters=excl, excl_cluster_ids=excl_ids, n_excl_cls=len(excl))

    cluster_ids = property(lambda self: self._equalized()["cluster_ids"])
    cluster_len = property(lambda self: self._equalized()["cluster_len"])
    max_cnt = property(lambda self: self._equalized()["max_cnt"])
    excl_clusters = property(lambda self: self._equalized()["excl_clusters"])
    excl_cluster_ids = property(lambda self: self._equalized()["excl_cluster_ids"])
    n_excl_cls = property(lambda self: self._equalized()["n_excl_cls"])

    # ------------------------------------------------------------------ reference API
    def get_dist(self, x, y, mode='sq_euclidean'):
        """Pairwise L2 distance [m, n] (reference :38-55).  Kept for API parity; the assign path
        never materialises this matrix."""
        return torch.cdist(x.unsqueeze(0).detach(), y.unsqueeze(0).detach())[0]

    def update_centers(self, feat, mode="root", selected_leaf=-1):
        """Reference :58-78 computes padded-gather sums into a local and discards them: no-op."""
        return None

    def equalize_cluster_size(self, mode="root"):
        self._eq_cache = None
        self._eq_mode = mode
        if mode == "root":
            self.cls_ids = self.nn_index
        elif mode == "leaf":
            self.leaf_cls_ids = self.nn_index

    def cluster_assign(self, feat, feat_scaled=None, mode="root", selected_leaf=-1, _split=None):
        """Lloyd iterations + final reassign (reference :146-241).  ``_split=(a, b, scale_b)`` lets
        forward() pass ins_feat and xyz separately so the [N,9] concatenation is never built."""
        if _split is not None:
            a, b, scale_b = _split
        else:
            a, b, scale_b = feat.detach(), None, 1.0
        dev = a.device
        N = a.shape[0]
        D = a.shape[1] + (0 if b is None else b.shape[1])
        k1, k2 = self.num_clusters, self.leaf_num_clusters

        def rows(idx):
            r = a[idx]
            return r if b is None else torch.cat([r, b[idx] * scale_b], 1)

        dist_on = self.distributed
        if dist_on:
            import torch.distributed as dist
            n_glob = torch.tensor([N], dtype=torch.int64, device=dev)
            dist.all_reduce(n_glob, group=self.process_group)
            N_global = int(n_glob)
        else:
            N_global = N
        if len(self.centers) == 0 and mode == "root":
            self.centers = rows(torch.randperm(N)[:k1].to(dev)).float()
            if dist_on:          # rank 0's draw wins
                dist.broadcast(self.centers, src=dist.get_global_rank(self.process_group, 0)
                               if self.process_group is not None else 0, group=self.process_group)
        if len(self.leaf_centers) == 0 and mode == "leaf":
            self.leaf_centers = rows(torch.randperm(N)[:k1 * k2 + 1].to(dev)).float()
            if dist_on:
                dist.broadcast(self.leaf_centers, src=dist.get_global_rank(self.process_group, 0)
                               if self.process_group is not None else 0, group=self.process_group)
            self.leaf_cls_ids = torch.ones(N, device=dev).to(torch.int64) * k1 * k2

        if mode == "root":
            k = k1
            n_eps = N_global // CHUNK + 1          # chunks visited per pass (strict '>' break, :193)
            centers = self.centers.detach().float().contiguous().to(dev)
            select, selected, id_offset = None, -1, 0
            ids = torch.empty(N, dtype=torch.int64, device=dev)
        elif mode == "leaf":
            k = k2
            n_eps = 1
            start_id = int(selected_leaf) * k2
            n_sub = int(self.iLeafSubNum[selected_leaf])
            self.leaf_centers = self.leaf_centers.detach().float().contiguous().to(dev)
            select, selected, id_offset = self.cls_ids, int(selected_leaf), start_id
            ids = self.leaf_cls_ids
        else:
            raise ValueError(mode)

        comm = self.reducer.comm if (dist_on and self.reducer is not None) else None
        if not dist_on or comm is not None:
            # ONE launch per Lloyd iteration (C ABI ogs_kmeans_lloyd_pass): assign + centroid sums + [all-reduce over
            # NVLink peer memory by the kernel's last CTA] + the reference's centre update, in place on `cur`
            if mode == "root":
                cur, k_in, eps_add = centers.clone(), k, n_eps * 1e-6
            else:
                cur, k_in, eps_add = self.leaf_centers[start_id:start_id + k2], n_sub, 1e-6
            ws = LloydWorkspace(dev, k=k_in, D=D)
            counts_state = torch.full((cur.shape[0],), 1e-6, dtype=torch.float32, device=dev)
            a_c = a if (a.dtype == torch.float32 and a.is_contiguous()) else a.float().contiguous()
            b_c = None if b is None else (b if (b.dtype == torch.float32 and b.is_contiguous()) else b.float().contiguous())
            for _ in range(self.num_kmeans_iters):
                lloyd_pass(a_c, b_c, scale_b, cur, counts_state, eps_add, ids, ws, comm, k_in, select, selected, id_offset)
            if mode == "root":
                centers = cur
        else:
            buf = torch.zeros(k * D + k, dtype=torch.float32, device=dev)   # [sums | counts]: one collective
            sums = buf[:k * D].view(k, D)
            cnt = buf[k * D:]
            counts_state = torch.full((k,), 1e-6, dtype=torch.float32, device=dev)
            for _ in range(self.num_kmeans_iters):
                buf.zero_()
                if mode == "root":
                    kmeans_assign(a, b, scale_b, centers, None, -1, 0, ids, sums, cnt)
                else:
                    cur = self.leaf_centers[start_id:start_id + n_sub]
                    # sums/counts rows beyond n_sub stay zero -> those centres become 0 / eps = 0 (:211)
                    kmeans_assign(a, b, scale_b, cur, select, selected, id_offset, ids, sums[:n_sub], cnt[:n_sub])
                self._all_reduce(buf)
                counts_state += cnt + n_eps * 1e-6
                new_centers = sums / counts_state.unsqueeze(-1)
                if mode == "root":
                    centers = new_centers
                else:
                    self.leaf_centers[start_id:start_id + k2] = new_centers
                counts_state[counts_state > 0.1] = 0.

        # final reassign with the new centres (:217-240)
        if mode == "root":
            self.centers = centers
            kmeans_assign(a, b, scale_b, centers, None, -1, 0, ids, None, None)
            self.nn_index = ids
        else:
            kmeans_assign(a, b, scale_b, self.leaf_centers[start_id:start_id + n_sub], select, selected, id_offset,
                          ids, None, None)
            self.leaf_cls_ids = ids
            self.nn_index = self.leaf_cls_ids
        self.equalize_cluster_size(mode=mode)

    def _all_reduce(self, t):
        if self.reducer is not None:
            self.reducer.all_reduce(t)
        else:
            import torch.distributed as dist
            dist.all_reduce(t, group=self.process_group)

    def cluster_assign_all_leaves(self, gaussian=None, feat=None):
        """The fine level of EVERY coarse cluster in one go: equivalent to
        ``for c in range(k1): self.forward(gaussian, it, assign=True, mode="leaf", selected_leaf=c)`` of the
        reference (scene/kmeans_quantize.py:196-214,233-238 per call; train.py:322-332 drives one cluster per
        training iteration), because the per-cluster Lloyd iterations never read each other's state.  One segmented
        launch per Lloyd pass over all N points (C ABI ogs_kmeans_assign_segmented) instead of k1 x (iters + 1)
        passes that each re-read all N coarse ids; exact integer centroid sums, one [k1*k2, D+1] all-reduce per
        pass when sharded.  Needs ``cls_ids`` (coarse ids) and ``iLeafSubNum``; initialises ``leaf_centers`` the way
        the reference does when they are empty."""
        a = (gaussian._ins_feat if feat is None else feat).detach()
        if a.dtype != torch.float32 or not a.is_contiguous():
            a = a.float().contiguous()
        dev, N, D = a.device, a.shape[0], a.shape[1]
        k1, k2 = self.num_clusters, self.leaf_num_clusters
        rows = k1 * k2
        if len(self.leaf_centers) == 0:
            self.leaf_centers = a[torch.randperm(N)[:rows + 1].to(dev)].float()
            if self.distributed:
                import torch.distributed as dist
                dist.broadcast(self.leaf_centers, src=dist.get_global_rank(self.process_group, 0)
                               if self.process_group is not None else 0, group=self.process_group)
        if len(self.leaf_cls_ids) != N:
            self.leaf_cls_ids = torch.ones(N, device=dev).to(torch.int64) * rows
        self.leaf_centers = self.leaf_centers.detach().float().contiguous().to(dev)
        seg_k = torch.as_tensor(self.iLeafSubNum).to(device=dev, dtype=torch.int32).contiguous()
        # exact sums need a bound on |x|: one host read per call (not per pass)
        stats = torch.stack([a.abs().max() if N > 0 else a.new_zeros(()), a.new_tensor(float(N))])
        if self.distributed:
            import torch.distributed as dist
            mx = stats[:1].clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=self.process_group)
            nn = stats[1:].clone()
            dist.all_reduce(nn, group=self.process_group)
            stats = torch.cat([mx, nn])
        max_abs, n_glob = (float(v) for v in stats.tolist())
        fix = fixed_point_bits(int(n_glob), max_abs)
        counts_state = torch.full((rows,), 1e-6, dtype=torch.float32, device=dev)
        ids = self.leaf_cls_ids
        comm = self.reducer.comm if (self.distributed and self.reducer is not None) else None
        coarse = self.cls_ids.to(torch.int64).contiguous()
        if not self.distributed or comm is not None:
            # ONE launch per Lloyd pass: segmented assign + exact sums + [integer all-reduce over NVLink peer memory by the
            # kernel's last CTA] + centre update of every block, in place on leaf_centers
            ws = LloydWorkspace(dev, D=D, k1=k1, k2=k2)
            for _ in range(self.num_kmeans_iters):
                lloyd_pass_segmented(a, coarse, self.leaf_centers, seg_k, k2, counts_state, ids, fix, ws, comm)
        else:
            acc = torch.zeros(rows * (D + 1), dtype=torch.int64, device=dev)
            for _ in range(self.num_kmeans_iters):
                acc.zero_()
                kmeans_assign_segmented(a, coarse, self.leaf_centers, seg_k, k2, ids, acc, fix)
                self._all_reduce(acc)
                _lib.launch("ogs_kmeans_finalize_fixed", dev, rows, D, _lib.ptr(acc), fix, 1e-6, _lib.ptr(counts_state),
                            _lib.ptr(self.leaf_centers))
        kmeans_assign_segmented(a, self.cls_ids, self.leaf_centers, seg_k, k2, ids, None, fix)
        self.leaf_cls_ids = ids
        self.nn_index = ids
        self.equalize_cluster_size(mode="leaf")
        if gaussian is not None:
            gaussian._ins_feat_q = _GatherStraightThrough.apply(gaussian._ins_feat, self.leaf_centers, self.nn_index)

    def rescale(self, feat, scale=None):
        if scale is None:
            return feat / (abs(feat).max(dim=0)[0] + 1e-8)
        return feat / (scale + 1e-8)

    def forward(self, gaussian, iteration, assign=False, mode="root", selected_leaf=-1, pos_weight=1.0):
        if mode == "root":
            split = (gaussian._ins_feat.detach(), gaussian._xyz.detach(), float(pos_weight))
        elif mode == "leaf":
            split = (gaussian._ins_feat.detach(), None, 1.0)
        else:
            raise ValueError(mode)
        if assign:
            self.cluster_assign(None, mode=mode, selected_leaf=selected_leaf, _split=split)
        else:
            self.update_centers(None, mode=mode, selected_leaf=selected_leaf)
        centers = self.centers if mode == "root" else self.leaf_centers
        gaussian._ins_feat_q = _GatherStraightThrough.apply(gaussian._ins_feat, centers, self.nn_index)

    __call__ = forward

    def replace_with_centers(self, gaussian):
        deg = gaussian._features_rest.shape[1]
        sampled_centers = torch.gather(self.centers, 0, self.nn_index.unsqueeze(-1).repeat(1, self.vec_dim))
        gaussian._features_rest = gaussian._features_rest - gaussian._features_rest.detach() + \
            sampled_centers.reshape(-1, deg, 3)

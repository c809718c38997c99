"""Row-sharded offline phase over G ranks (one process per GPU, torch.distributed / NCCL over NVLink).

BASELINE.json config 4: M pcore MCs x D dims, the pairwise eps-neighbourhood (predecon.py:161-188) is the
O(M^2 D) part.  Rank g owns the contiguous rows [g*R, (g+1)*R), R = ceil(M/G):

  stage 1 (local)   N(p) bit rows + |N(p)| for own rows, the pairs  ccb_off_neighbours  (kernel 4b)
                    inside the guard band settled with dnrm2
  stage 2 (local)   subspace preference masks w_p of own rows       ccb_off_subspace    (kernel 4c)
  all-gather        w_p masks of every row (M * 8 B)                NCCL all_gather_into_tensor
  stage 3 (local)   weighted-neighbour bit rows WN(p) of own rows   ccb_off_weighted    (kernel 4d)
  stage 4a (local)  own rows -> isolated flags + CSR row lengths     ccb_offc_rowinfo
  all-gather        isolated flags (M B), row lengths (M * 4 B)      NCCL all_gather_into_tensor
  stage 4b (local)  own rows' column lists into the global CSR       ccb_offc_fill
  all-reduce        the CSR (disjoint segments; sum = union)         NCCL all_reduce (nnz * 4 B)
  stage 4c (every rank, redundantly -- deterministic, so no broadcast is needed)
                    ordered cluster growth over the CSR              ccb_off_clusters_csr (kernel 4e)

Only the LISTS of the non-isolated microclusters travel (kilobytes to a few MB) -- the weighted-neighbour bit matrix
(M^2 / 8 bytes: 1.25 GB at M = 1e5) stays sharded; if the lists would be larger than a quarter of the bit matrix the
bit rows are all-gathered instead (ccb_off_clusters).  PyTorch is only plumbing here (device buffers, the NCCL
communicator); every stage is a kernel of this repo.
The compute backend is injectable so that the sharding / gather logic is testable on CPU with gloo.
"""
import ctypes as C

from . import _lib


class CudaStages:
    """The C-ABI stage functions on raw device pointers of torch tensors."""

    def __init__(self, device, dnrm2_ptr=None):
        import torch

        self.torch = torch
        self.device = device
        self.dev = torch.device("cuda", device)
        self.L = _lib.lib()
        self.dnrm2_ptr = dnrm2_ptr

    def stream(self):
        return self.torch.cuda.current_stream(self.dev).cuda_stream

    def empty(self, shape, dtype):
        return self.torch.zeros(shape, dtype=dtype, device=self.dev)

    def neighbours(self, cen, M, D, r0, r1, E, E2, nbr, cnt):
        n = C.c_int64()
        _lib.check(self.L.ccb_off_neighbours(self.device, self.stream(), cen.data_ptr(), M, D, r0, r1, E, E2,
                                             self.dnrm2_ptr, nbr.data_ptr(), cnt.data_ptr(), C.byref(n)))
        return n.value

    def subspace(self, cen, M, D, r0, r1, nbr, cnt, delta, submask):
        _lib.check(self.L.ccb_off_subspace(self.device, self.stream(), cen.data_ptr(), M, D, r0, r1, nbr.data_ptr(),
                                           cnt.data_ptr(), delta, submask.data_ptr()))

    def weighted(self, cen, M, D, r0, r1, nbr, submask_all, k, E2, wnbr):
        _lib.check(self.L.ccb_off_weighted(self.device, self.stream(), cen.data_ptr(), M, D, r0, r1, nbr.data_ptr(),
                                           submask_all.data_ptr(), k, E2, wnbr.data_ptr()))

    def _grow(self, M, call):
        """label / order / cl_off / n_cl of the cluster growth `call(label, order, cl_off, n_cl)`, read back"""
        t = self.torch
        label = t.empty(max(M, 1), dtype=t.int32, device=self.dev)
        order = t.empty(max(M, 1), dtype=t.int32, device=self.dev)
        cl_off = t.zeros(M + 2, dtype=t.int32, device=self.dev)
        ncl = t.zeros(1, dtype=t.int32, device=self.dev)
        _lib.check(call(label.data_ptr(), order.data_ptr(), cl_off.data_ptr(), ncl.data_ptr()))
        n = int(ncl.item())
        return label[:M].cpu().numpy(), order.cpu().numpy(), cl_off[:n + 1].cpu().numpy(), n

    def clusters(self, M, wnbr_all, core, submask_all, k, pi, csr_min_m=0):
        return self._grow(M, lambda *out: self.L.ccb_off_clusters(
            self.device, self.stream(), M, wnbr_all.data_ptr(), core.data_ptr(), submask_all.data_ptr(), k, pi, csr_min_m,
            *out))

    def rowinfo(self, wn_rows, M, r0, r1, iso, nnz):
        _lib.check(self.L.ccb_offc_rowinfo(self.device, self.stream(), wn_rows.data_ptr(), M, r0, r1, iso.data_ptr(),
                                           nnz.data_ptr()))

    def fill(self, wn_rows, M, r0, r1, iso_all, off_all, col):
        _lib.check(self.L.ccb_offc_fill(self.device, self.stream(), wn_rows.data_ptr(), M, r0, r1, iso_all.data_ptr(),
                                        off_all.data_ptr(), col.data_ptr()))

    def clusters_csr(self, M, off_all, col, iso_all, core, submask_all, k, pi):
        return self._grow(M, lambda *out: self.L.ccb_off_clusters_csr(
            self.device, self.stream(), M, off_all.data_ptr(), col.data_ptr(), iso_all.data_ptr(), core.data_ptr(),
            submask_all.data_ptr(), k, pi, *out))


def row_range(M, world, rank):
    R = (M + world - 1) // world
    r0 = min(M, rank * R)
    return R, r0, min(M, r0 + R)


def sharded_offline(stages, cen, core, M, D, k, pi, delta, E, E2, group=None, dist=None, timers=None):
    """Runs the offline phase row-sharded over the ranks of `group`.

    cen: [M, D] fp64 centroids (replicated on every rank), core: [M] uint8 core flags (replicated).
    Returns (label [M], order, cl_off, n_clusters, info) -- identical on every rank.
    """
    world = dist.get_world_size(group) if dist is not None else 1
    rank = dist.get_rank(group) if dist is not None else 0
    words = (M + 31) // 32
    R, r0, r1 = row_range(M, world, rank)
    torch = stages.torch
    nbr = stages.empty((R, words), torch.int32)
    cnt = stages.empty((R,), torch.int32)
    submask = stages.empty((R,), torch.int64)
    wn = stages.empty((R, words), torch.int32)
    import time

    def lap(name, t0):
        """optional per-stage wall time (device-synchronised); timers = {} collects seconds per stage"""
        if timers is None:
            return t0
        if hasattr(stages, "torch") and hasattr(stages.torch, "cuda") and stages.torch.cuda.is_available():
            stages.torch.cuda.synchronize()
        t1 = time.perf_counter()
        timers[name] = timers.get(name, 0.0) + (t1 - t0)
        return t1

    tq = lap("alloc", time.perf_counter()) if timers is not None else 0.0
    n_border = stages.neighbours(cen, M, D, r0, r1, E, E2, nbr, cnt)
    tq = lap("neighbours", tq)
    stages.subspace(cen, M, D, r0, r1, nbr, cnt, delta, submask)
    tq = lap("subspace", tq)
    if world > 1:
        sub_all = stages.empty((world * R,), torch.int64)
        dist.all_gather_into_tensor(sub_all, submask, group=group)
    else:
        sub_all = submask
    tq = lap("allgather_submask", tq)
    stages.weighted(cen, M, D, r0, r1, nbr, sub_all, k, E2, wn)
    tq = lap("weighted", tq)
    gather_bytes = int(world * R * 8) if world > 1 else 0
    exchange = "none"
    if world > 1 and hasattr(stages, "rowinfo"):
        # only the lists of the non-isolated microclusters travel; the bit matrix stays sharded
        iso = stages.empty((R,), torch.uint8)
        nnz = stages.empty((R,), torch.int32)
        stages.rowinfo(wn, M, r0, r1, iso, nnz)
        iso_all = stages.empty((world * R,), torch.uint8)
        nnz_all = stages.empty((world * R,), torch.int32)
        dist.all_gather_into_tensor(iso_all, iso, group=group)
        dist.all_gather_into_tensor(nnz_all, nnz, group=group)
        off_all = stages.empty((M + 1,), torch.int64)
        off_all[1:] = torch.cumsum(nnz_all[:M].to(torch.int64), dim=0)
        total = int(off_all[M].item())
        gather_bytes += int(world * R * 5)
        tq = lap("csr_rowinfo", tq)
        if total * 4 <= M * words:  # lists <= a quarter of the bit matrix
            col = stages.empty((max(total, 1),), torch.int32)
            stages.fill(wn, M, r0, r1, iso_all, off_all, col)
            dist.all_reduce(col, group=group)  # disjoint segments: the sum is the union
            gather_bytes += int(total * 4)
            tq = lap("csr_fill_allreduce", tq)
            label, order, cl_off, ncl = stages.clusters_csr(M, off_all, col, iso_all, core, sub_all, k, pi)
            tq = lap("clusters", tq)
            exchange = "csr"
    if exchange == "none":
        if world > 1:
            wn_all = stages.empty((world * R, words), torch.int32)
            dist.all_gather_into_tensor(wn_all, wn, group=group)
            gather_bytes += int(world * R * words * 4)
            exchange = "bitrows"
        else:
            wn_all = wn
        tq = lap("allgather_wn", tq)
        label, order, cl_off, ncl = stages.clusters(M, wn_all, core, sub_all, k, pi)
        tq = lap("clusters", tq)
    info = {"rows": (r0, r1), "rows_per_rank": R, "borderline_pairs": n_border,
            "gather_bytes": gather_bytes, "exchange": exchange,
            "neighbour_count": int(cnt[:max(r1 - r0, 0)].sum().item()) if r1 > r0 else 0}
    return label, order, cl_off, ncl, info

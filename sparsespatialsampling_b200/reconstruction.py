"""
How much of the original field a sampled grid keeps: the exported field is interpolated back onto the original points
and compared there (the reference leaves this to its post-processing scripts).

``ReconstructionError`` builds the interpolation tables of the other direction -- a KNN index over the sampled cell
centres, queried with the N original points; inverse-distance weights normalised per point, as in
``ExportData._build_knn_cache`` -- and hands every (original, sampled) window to ``s3_recon_error``, which reads the
original field once and never materialises the reconstruction:

    rec = ReconstructionError(s_cube, coordinates)
    stats = rec.error(original, sampled)                       # one window of snapshots
    stats = rec.error(original2, sampled2, stats=stats)        # the next window: appended / accumulated
    stats.relative_l2(), stats.max_abs, stats.rms()

``distributed=True`` mirrors ``ExportData``: rank 0 builds the tables and broadcasts them once, every rank passes its own
snapshot window (``parallel.snapshot_window``), and ``ErrorStats.gather()`` is the only exchange.
"""
from typing import Optional

import torch as pt

from . import _lib
from .export import KnnTables
from .interpolate import _rows_view
from .knn import KnnIndex, default_n_neighbors


def recon_error(original: pt.Tensor, sampled: pt.Tensor, tables: KnnTables, point_sq_err: Optional[pt.Tensor]):
    """One ``s3_recon_error`` launch: ``original`` ``[N, D, T]`` and ``sampled`` ``[Nc, D, T]`` fp32 device tensors (T
    contiguous, any row / component stride) -> ``(sq_err, sq_ref, max_abs)`` fp64 ``[D, T]``; ``sum_t e^2`` is added
    into ``point_sq_err`` fp64 ``[N, D]`` when it is given."""
    lib = _lib.load()
    n_comp, n_cols = original.size(1), original.size(2)
    o, _, _, o_row, o_comp = _rows_view(original)
    s, _, _, s_row, s_comp = _rows_view(sampled)
    sq_err = pt.empty((n_comp, n_cols), dtype=pt.float64, device=original.device)
    sq_ref = pt.empty_like(sq_err)
    max_abs = pt.empty_like(sq_err)
    dt = {pt.float32: _lib.S3_F32, pt.float64: _lib.S3_F64}
    with pt.cuda.device(original.device):
        _lib.check(lib.s3_recon_error(
            _lib.ptr(s, strided=True), dt.get(s.dtype, -1), s.size(0), n_comp, n_cols, s_row, s_comp,
            _lib.ptr(o, strided=True), dt.get(o.dtype, -1), o.size(0), o_row, o_comp,
            _lib.ptr(tables.idx_sorted), _lib.ptr(tables.w32_sorted), _lib.ptr(tables.out_row), tables.k,
            _lib.ptr(sq_err), _lib.ptr(sq_ref), _lib.ptr(max_abs), _lib.ptr(point_sq_err), _lib.stream_ptr()))
    return sq_err, sq_ref, max_abs


class ErrorStats:
    """Reconstruction error of the snapshots seen so far (fp64, on the device of the tables).

    ``sq_err`` / ``sq_ref`` / ``max_abs`` ``[D, T_seen]``: per component and snapshot, the sum over the original points
    of ``e^2`` and of ``original^2``, and the largest ``|e|``; ``point_sq_err`` ``[N, D]``: per original point (order of
    ``coordinates``) and component, the sum of ``e^2`` over the snapshots; ``n_snapshots`` = ``T_seen``. For errors on
    the grid side (``DMD.reconstruction_error``, ``svd.reconstruction_error``) ``sq_err`` / ``sq_ref`` are area-weighted
    and ``point_sq_err`` is per cell."""

    def __init__(self, n_points: int, n_comp: int, device, distributed: bool = False, group=None):
        self.sq_err = pt.zeros((n_comp, 0), dtype=pt.float64, device=device)
        self.sq_ref = pt.zeros_like(self.sq_err)
        self.max_abs = pt.zeros_like(self.sq_err)
        self.point_sq_err = pt.zeros((n_points, n_comp), dtype=pt.float64, device=device)
        self.n_snapshots = 0
        self._distributed = distributed
        self._group = group

    def relative_l2(self) -> pt.Tensor:
        """``[T_seen]``: ``||rec - original|| / ||original||`` per snapshot, over all points and components."""
        return pt.sqrt(self.sq_err.sum(0) / self.sq_ref.sum(0))

    def rms(self) -> pt.Tensor:
        """``[N, D]``: root mean square error of every original point over the snapshots seen."""
        return pt.sqrt(self.point_sq_err / self.n_snapshots)

    def gather(self) -> "ErrorStats":
        """Statistics of all ranks (``distributed=True``), on every rank: the per-snapshot arrays of the ranks'
        windows concatenated in rank order (windows may differ in length), the point maps summed. A copy of ``self``
        in a single process."""
        from .parallel import _active, allreduce_sum
        out = ErrorStats(self.point_sq_err.size(0), self.sq_err.size(0), self.sq_err.device)
        if not (self._distributed and _active(self._group)):
            out.sq_err, out.sq_ref, out.max_abs = self.sq_err.clone(), self.sq_ref.clone(), self.max_abs.clone()
            out.point_sq_err, out.n_snapshots = self.point_sq_err.clone(), self.n_snapshots
            return out
        import torch.distributed as dist
        world = dist.get_world_size(self._group)
        dev = self.sq_err.device
        n_local = pt.tensor([self.n_snapshots], dtype=pt.int64, device=dev)
        counts = [pt.empty_like(n_local) for _ in range(world)]
        dist.all_gather(counts, n_local, group=self._group)
        counts = [int(c.item()) for c in counts]
        t_max = max(counts)
        mine = pt.zeros((3, self.sq_err.size(0), t_max), dtype=pt.float64, device=dev)
        mine[0, :, :self.n_snapshots] = self.sq_err
        mine[1, :, :self.n_snapshots] = self.sq_ref
        mine[2, :, :self.n_snapshots] = self.max_abs
        parts = [pt.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=self._group)
        every = pt.cat([p[:, :, :c] for p, c in zip(parts, counts)], dim=2)
        out.sq_err, out.sq_ref, out.max_abs = (every[i].contiguous() for i in range(3))
        out.point_sq_err = allreduce_sum(self.point_sq_err.clone(), self._group)
        out.n_snapshots = sum(counts)
        return out


class ReconstructionError:
    def __init__(self, s_cube, coordinates: pt.Tensor, n_neighbors: int = None, device=None, distributed: bool = False,
                 group=None):
        """
        :param s_cube: the sampled grid (``SparseSpatialSampling`` or anything with ``centers`` / ``n_dimensions``)
        :param coordinates: ``[N, d]`` original points, the rows of the original field
        :param n_neighbors: cells per original point, ``default_n_neighbors(d)`` (8 in 2-D, 26 in 3-D) by default
        :param distributed: inside an initialised ``torch.distributed`` job: rank 0 builds the tables, every other rank
            receives them (one broadcast, ``KnnTables.share``)
        """
        _lib.require_cuda()
        self._device = pt.device(device) if device is not None else pt.device("cuda", pt.cuda.current_device())
        centers = s_cube.centers
        n_dim = getattr(s_cube, "n_dimensions", None) or centers.size(1)
        self.k = int(n_neighbors) if n_neighbors is not None else default_n_neighbors(n_dim)
        self.n_cells = int(centers.size(0))
        self.n_points = int(coordinates.size(0))
        if not 1 <= self.k <= 64:
            raise ValueError(f"n_neighbors must be in [1, 64], got {self.k}")
        if self.n_cells < self.k:
            raise ValueError(f"the grid has {self.n_cells} cells, fewer than n_neighbors = {self.k}")
        self._group = group
        self._rank, self._world = 0, 1
        if distributed:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
                self._rank, self._world = dist.get_rank(group), dist.get_world_size(group)
        self.tables = self._make_tables(centers, coordinates) if self._rank == 0 else None
        if self._world > 1:
            self.tables = KnnTables.share(self.tables, self._device, 0, group, n=self.n_points, k=self.k)

    def _make_tables(self, centers: pt.Tensor, coordinates: pt.Tensor) -> KnnTables:
        """KNN index over the cell centres, queried with the original points (rank 0 only)."""
        index = KnnIndex(centers, device=self._device)
        return KnnTables(index, coordinates, self.k)

    def _fields(self, original: Optional[pt.Tensor], sampled: pt.Tensor):
        """Both fields as ``[rows, D, T]`` fp32 device tensors, shapes checked against the grid and each other."""
        def as3(t, name):
            if t.dim() == 2:
                t = t.unsqueeze(1)
            if t.dim() != 3:
                raise ValueError(f"`{name}` must be [rows, D, T] or [rows, T], got {tuple(t.shape)}")
            if t.dtype != pt.float32:
                raise ValueError(f"`{name}` must be float32 (the export's default dtype), got {t.dtype}")
            return t.to(self._device)
        sampled = as3(sampled, "sampled")
        if sampled.size(0) != self.n_cells:
            raise ValueError(f"`sampled` has {sampled.size(0)} rows, the grid {self.n_cells} cells")
        if original is None:
            return None, sampled
        original = as3(original, "original")
        if original.size(0) != self.n_points:
            raise ValueError(f"`original` has {original.size(0)} rows, `coordinates` {self.n_points} points")
        if original.shape[1:] != sampled.shape[1:]:
            raise ValueError(f"`original` [.., D, T] = {tuple(original.shape[1:])} differs from `sampled` "
                             f"{tuple(sampled.shape[1:])}")
        return original, sampled

    def reconstruct(self, sampled: pt.Tensor) -> pt.Tensor:
        """The sampled field interpolated back onto the original points: ``[N, D, T]`` (``[N, T]`` for ``[Nc, T]``
        input) fp32 on the device, in the order of ``coordinates``."""
        _, s = self._fields(None, sampled)
        out = self.tables.interpolate(s, pt.float32)
        return out.squeeze(1) if sampled.dim() == 2 else out

    def error(self, original: pt.Tensor, sampled: pt.Tensor, stats: ErrorStats = None) -> ErrorStats:
        """Error of one window of snapshots: ``original`` ``[N, D, T]`` / ``[N, T]`` (rows in the order of
        ``coordinates``) against ``sampled`` ``[Nc, D, T]`` / ``[Nc, T]`` (what ``ExportData`` returned for the same
        snapshots). With ``stats`` from an earlier window, its snapshots are appended and the point map added into."""
        o, s = self._fields(original, sampled)
        if stats is None:
            stats = ErrorStats(self.n_points, o.size(1), self._device, self._world > 1, self._group)
        elif stats.point_sq_err.shape != (self.n_points, o.size(1)):
            raise ValueError(f"`stats` holds {tuple(stats.point_sq_err.shape)} points x components, this window "
                             f"{(self.n_points, o.size(1))}")
        sq_err, sq_ref, max_abs = recon_error(o, s, self.tables, stats.point_sq_err)
        stats.sq_err = pt.cat([stats.sq_err, sq_err], dim=1)
        stats.sq_ref = pt.cat([stats.sq_ref, sq_ref], dim=1)
        stats.max_abs = pt.cat([stats.max_abs, max_abs], dim=1)
        stats.n_snapshots += o.size(2)
        return stats

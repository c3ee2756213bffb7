"""
Volume-weighted SVD of the sampled snapshots on the GPU.

``compute_svd(data_matrix, cell_area, rank)`` keeps the signature and the return values ``(s, U, V)`` of the reference
(sparseSpatialSampling/utils.py:302-346): subtract the temporal mean, weight every cell by ``sqrt(cell_area)``, thin
SVD, un-weight the modes; vector fields ``[N_cells, D, T]`` are stacked to ``(N_cells * D, T)`` rows
(utils.py:337-338) and the modes reshaped back (utils.py:344-346).

The reference hands the weighted matrix to ``flowtorch.analysis.SVD`` (LAPACK ``gesdd`` through ``torch.linalg.svd``).
Here the tall-skinny problem is solved by the method of snapshots -- the data matrix is read twice and never copied:

    G = B^T B                 s3_svd_gram     tcgen05 tensor cores, 3xTF32 split, fp64 across K segments
    G = V diag(s^2) V^T       torch.linalg.eigh on the device, fp64, T x T (the only library call)
    U = (A - mean) V / s      s3_svd_project  (the sqrt(volume) scaling cancels against the un-weighting)

Differences to the reference, stated: ``data_matrix`` is NOT modified in place; singular values far below
``sqrt(eps_fp32) * s[0]`` lose relative accuracy (the Gram matrix squares the condition number), modes whose singular
value is below ``1e-6 * s[0]`` are returned as zeros; ``rank=None`` uses the optimal hard threshold of Gavish & Donoho
(2014) -- flowtorch's own ``opt_rank`` is not vendored with the reference (requirements.txt:5), so that case is
unpinned. There is no CPU fallback.
"""
import logging
import math
from typing import Tuple

import numpy as np
import torch as pt

from . import _lib

logger = logging.getLogger(__name__)

GRAM_METHODS = {"simt": 0, "tc3": 1, "tc": 2}


def optimal_rank(s: pt.Tensor, rows: int, cols: int) -> int:
    """Optimal hard threshold for singular values, unknown noise level (Gavish & Donoho 2014, eq. 5):
    rank = #{s_i > omega(beta) * median(s)}, omega(beta) ~ 0.56 b^3 - 0.95 b^2 + 1.82 b + 1.43, beta = min/max."""
    beta = min(rows, cols) / max(rows, cols)
    omega = 0.56 * beta ** 3 - 0.95 * beta ** 2 + 1.82 * beta + 1.43
    tau = omega * float(pt.median(s))
    return max(1, int((s > tau).sum()))


def _as_device_matrix(data_matrix: pt.Tensor, dev) -> pt.Tensor:
    a = data_matrix.detach()
    if a.dtype != pt.float32:
        a = a.to(pt.float32)
    if a.device != dev:
        a = a.pin_memory().to(dev, non_blocking=True) if a.device.type == "cpu" else a.to(dev)
    return a.contiguous()


def _field_on_device(data_matrix: pt.Tensor, cell_area: pt.Tensor, device):
    """Checks a ``[N_cells, T]`` / ``[N_cells, D, T]`` field and its cell areas and puts both on the compute device
    (``device``, else the field's CUDA device, else the current one): ``(a [N_cells * D, T] fp32, vol [N_cells] fp32,
    vol_div = D, compute device)``."""
    shape = tuple(data_matrix.shape)
    if len(shape) not in (2, 3):
        raise ValueError(f"data_matrix must be [N_cells, T] or [N_cells, D, T], got {shape}")
    if cell_area.numel() != shape[0]:
        raise ValueError(f"cell_area has {cell_area.numel()} entries for {shape[0]} cells")
    home = data_matrix.device
    dev = pt.device(device) if device is not None else (home if home.type == "cuda" else pt.device("cuda", pt.cuda.current_device()))
    vol_div = 1 if len(shape) == 2 else shape[1]
    a = _as_device_matrix(data_matrix, dev).reshape(shape[0] * vol_div, shape[-1])
    vol = cell_area.detach().reshape(-1).to(device=dev, dtype=pt.float32).contiguous()
    return a, vol, vol_div, dev


def row_means(a: pt.Tensor) -> pt.Tensor:
    """Temporal mean of every row of ``a`` ([M, T] fp32 on the device)."""
    lib = _lib.load()
    a = a.contiguous()                    # (a pitched export result is a strided view: the SVD kernels want dense rows)
    mean = pt.empty((a.size(0),), dtype=pt.float32, device=a.device)
    with pt.cuda.device(a.device):
        _lib.check(lib.s3_svd_row_means(_lib.ptr(a), a.size(0), a.size(1), _lib.ptr(mean), _lib.stream_ptr()))
    return mean


def gram(a: pt.Tensor, mean: pt.Tensor, vol: pt.Tensor, vol_div: int = 1, method: str = "tc3") -> pt.Tensor:
    """G[i, j] = sum_m vol[m // vol_div] (a[m, i] - mean[m]) (a[m, j] - mean[m]), fp64 [T, T]."""
    lib = _lib.load()
    a = a.contiguous()
    t = a.size(1)
    g = pt.empty((t, t), dtype=pt.float64, device=a.device)
    with pt.cuda.device(a.device):
        _lib.check(lib.s3_svd_gram(_lib.ptr(a), _lib.ptr(mean), _lib.ptr(vol), vol_div, a.size(0), t,
                                   GRAM_METHODS[method], _lib.ptr(g), _lib.stream_ptr()))
    return g


def project(a: pt.Tensor, mean: pt.Tensor, vs: pt.Tensor) -> pt.Tensor:
    """U = (a - mean[:, None]) @ vs, fp32 [M, r]."""
    lib = _lib.load()
    vs = vs.to(pt.float32).contiguous()
    a = a.contiguous()
    u = pt.empty((a.size(0), vs.size(1)), dtype=pt.float32, device=a.device)
    with pt.cuda.device(a.device):
        _lib.check(lib.s3_svd_project(_lib.ptr(a), _lib.ptr(mean), _lib.ptr(vs), a.size(0), a.size(1), vs.size(1),
                                      _lib.ptr(u), _lib.stream_ptr()))
    return u


def project_tc(a: pt.Tensor, mean: pt.Tensor, vol: pt.Tensor, vol_div: int, vs: pt.Tensor, method: str = "tc3") -> pt.Tensor:
    """The same projection on the tensor cores (``s3_svd_project_tc``): the rows are centred, weighted and split into
    TF32 planes exactly as for the Gram matrix, contracted with ``vs`` over t by tcgen05 MMAs (3xTF32 for ``"tc3"``)
    and un-weighted in the epilogue. fp32 [M, r]."""
    lib = _lib.load()
    vs = vs.to(pt.float32).contiguous()
    a = a.contiguous()
    u = pt.empty((a.size(0), vs.size(1)), dtype=pt.float32, device=a.device)
    with pt.cuda.device(a.device):
        _lib.check(lib.s3_svd_project_tc(_lib.ptr(a), _lib.ptr(mean), _lib.ptr(vol), vol_div, _lib.ptr(vs), a.size(0),
                                         a.size(1), vs.size(1), GRAM_METHODS[method], _lib.ptr(u), _lib.stream_ptr()))
    return u


LOWRANK_MAX_Q = 512


def lowrank_error(a: pt.Tensor, left: pt.Tensor, right_t: pt.Tensor, mean: pt.Tensor = None, vol: pt.Tensor = None,
                  vol_div: int = 1, row_sq_err: pt.Tensor = None):
    """Residual ``e = (a - mean[:, None]) - left @ right_t.T`` reduced without forming it (``s3_lowrank_error``: tcgen05
    3xTF32 product, fp64 epilogue, ``a`` read once). ``a`` fp32 ``[M, T]``, ``left`` ``[M, q]``, ``right_t`` ``[T, q]``,
    ``q <= 512``; ``mean`` ``[M]`` (``None`` = 0), ``vol`` ``[M / vol_div]`` (``None`` = 1). Returns ``(sq_err, sq_ref,
    max_abs)`` fp64 ``[vol_div, T]`` (volume-weighted sums of ``e^2`` and ``(a - mean)^2``, largest ``|e|``, per
    component ``m % vol_div``); ``sum_t e^2`` is added into ``row_sq_err`` fp64 ``[M]`` when it is given."""
    lib = _lib.load()
    for name, x in (("a", a), ("left", left), ("right_t", right_t), ("mean", mean), ("vol", vol)):
        if x is not None and x.dtype != pt.float32:
            raise ValueError(f"`{name}` must be float32, got {x.dtype}")
    m, t = a.shape
    if left.dim() != 2 or left.size(0) != m or right_t.dim() != 2 or right_t.size(0) != t or \
            right_t.size(1) != left.size(1):
        raise ValueError(f"left {tuple(left.shape)} / right_t {tuple(right_t.shape)} do not fit a {(m, t)} matrix")
    if row_sq_err is not None and (row_sq_err.dtype != pt.float64 or row_sq_err.numel() != m):
        raise ValueError("`row_sq_err` must be float64 with one entry per row")
    if vol_div < 1 or m % vol_div:
        raise ValueError(f"{m} rows are not a multiple of vol_div = {vol_div}")
    if mean is not None and mean.numel() != m:
        raise ValueError(f"`mean` has {mean.numel()} entries for {m} rows")
    if vol is not None and vol.numel() != m // vol_div:
        raise ValueError(f"`vol` has {vol.numel()} entries for {m // vol_div} cells ({m} rows / vol_div = {vol_div})")
    for name, x in (("left", left), ("right_t", right_t), ("mean", mean), ("vol", vol), ("row_sq_err", row_sq_err)):
        if x is not None and x.device != a.device:
            raise ValueError(f"`{name}` is on {x.device}, `a` on {a.device}")
    if a.device.type != "cuda":
        raise ValueError(f"`a` must be a CUDA tensor, got {a.device}")
    if row_sq_err is not None and not row_sq_err.is_contiguous():
        raise ValueError("`row_sq_err` must be contiguous (the kernel adds into it)")
    a, left, right_t = a.contiguous(), left.contiguous(), right_t.contiguous()
    mean = mean.contiguous() if mean is not None else None
    vol = vol.contiguous() if vol is not None else None
    sq_err = pt.empty((vol_div, t), dtype=pt.float64, device=a.device)
    sq_ref, max_abs = pt.empty_like(sq_err), pt.empty_like(sq_err)
    with pt.cuda.device(a.device):
        _lib.check(lib.s3_lowrank_error(_lib.ptr(a), m, t, _lib.ptr(mean), _lib.ptr(vol), vol_div, _lib.ptr(left),
                                        _lib.ptr(right_t), left.size(1), _lib.ptr(sq_err), _lib.ptr(sq_ref),
                                        _lib.ptr(max_abs), _lib.ptr(row_sq_err), _lib.stream_ptr()))
    return sq_err, sq_ref, max_abs


def _error_stats(a: pt.Tensor, left: pt.Tensor, right_t: pt.Tensor, mean, vol: pt.Tensor, vol_div: int):
    """``ErrorStats`` of one low-rank model of the whole matrix ``a`` (rows = cells x components)."""
    from .reconstruction import ErrorStats
    n_cells = a.size(0) // vol_div
    stats = ErrorStats(n_cells, vol_div, a.device)
    row = pt.zeros((a.size(0),), dtype=pt.float64, device=a.device)
    stats.sq_err, stats.sq_ref, stats.max_abs = lowrank_error(a, left, right_t, mean, vol, vol_div, row)
    stats.point_sq_err = row.reshape(n_cells, vol_div)
    stats.n_snapshots = a.size(1)
    return stats


def reconstruction_error(data_matrix: pt.Tensor, cell_area: pt.Tensor, s: pt.Tensor, U: pt.Tensor, V: pt.Tensor,
                         device=None):
    """
    Truncation error of a POD model from ``compute_svd``: the field is rebuilt from the row means and the triplets the
    caller passes (``s[:r]``, ``U[..., :r]``, ``V[:, :r]``), ``mean + U diag(s) V^T``, and compared with ``data_matrix``
    (the same ``[N_cells, T]`` / ``[N_cells, D, T]`` input) by ``s3_lowrank_error`` without materialising it. Returns
    ``ErrorStats``: area-weighted ``sq_err`` / ``sq_ref`` (``sq_ref`` = the centred field) and ``max_abs`` per component
    and snapshot, ``point_sq_err`` per cell and component. ``r <= 512``.
    """
    _lib.require_cuda()
    shape = tuple(data_matrix.shape)
    r = int(s.numel())
    if tuple(U.shape) != shape[:-1] + (r,) or tuple(V.shape) != (shape[-1], r):
        raise ValueError(f"U {tuple(U.shape)} / V {tuple(V.shape)} do not match {r} singular values of a {shape} field")
    if r > LOWRANK_MAX_Q:
        raise ValueError(f"at most {LOWRANK_MAX_Q} modes, got {r}")
    a, vol, vol_div, dev = _field_on_device(data_matrix, cell_area, device)
    n_cells = shape[0]
    left = (U.to(dev, pt.float64).reshape(n_cells * vol_div, r) * s.to(dev, pt.float64)[None, :]).float()
    return _error_stats(a, left, V.to(dev, pt.float32), row_means(a), vol, vol_div)


def compute_svd(data_matrix: pt.Tensor, cell_area: pt.Tensor, rank: int = None, method: str = "tc3",
                n_modes: int = None, device=None) -> Tuple[pt.Tensor, pt.Tensor, pt.Tensor]:
    """
    Weighted SVD of a field (utils.py:302-346).

    :param data_matrix: ``[N_cells, T]`` or ``[N_cells, D, T]``; host or device tensor (not modified)
    :param cell_area: area (2D) / volume (3D) of every cell, ``[N_cells]``
    :param rank: number of singular triplets to keep; ``None`` = optimal hard threshold
    :param method: Gram kernel, ``"tc3"`` (tensor cores, 3xTF32, default), ``"tc"`` (single TF32), ``"simt"`` (fp32 cores)
    :param n_modes: compute only the first ``n_modes`` columns of U (``s`` and ``V`` keep ``rank`` entries); used by
        ``write_svd_s_cube_to_file``, which writes only that many modes
    :return: ``(s [r], U [N_cells, r] | [N_cells, D, r], V [T, r])`` on the device of ``data_matrix``
    """
    _lib.require_cuda()
    if method not in GRAM_METHODS:
        raise ValueError(f"unknown Gram method '{method}', available: {sorted(GRAM_METHODS)}")
    shape = tuple(data_matrix.shape)
    home = data_matrix.device
    a, vol, vol_div, dev = _field_on_device(data_matrix, cell_area, device)
    n_cells = shape[0]

    mean = row_means(a)
    g = gram(a, mean, vol, vol_div, method)
    s_out, u, v_out = _factor(a, mean, g, rank, n_modes, a.size(0), vol, vol_div, method)
    if len(shape) == 3:
        u = u.reshape(n_cells, vol_div, u.size(-1))
    if home != dev:
        pt.cuda.synchronize(dev)
        return s_out.to(home), u.to(home), v_out.to(home)
    return s_out, u, v_out


EIG_METHOD = "auto"          # "auto": top-r subspace iteration when rank << T, else the full eigh; "eigh": always full


def top_eigenpairs(g: pt.Tensor, r: int, tol: float = 1e-7, max_iter: int = 40):
    """
    The ``r`` largest eigenpairs of the symmetric positive semi-definite ``g`` (fp64 ``[T, T]``) by blocked subspace
    iteration with a Rayleigh-Ritz step per sweep: ``Z = G Q`` (fp64 GEMM), ``H = Q^T Z`` (``b x b``), ``H = W diag(w)
    W^T``, ``Q <- orth(Z W)`` by Cholesky-QR (the Ritz rotation makes the columns of ``Z W`` nearly orthogonal, so the
    Cholesky factor is well conditioned). Block size ``b = r + max(8, r / 2)``. Stops when the residuals
    ``||G x_i - w_i x_i|| <= tol * w_i`` for the first ``r`` pairs (eigenvalue error <= residual^2 / gap, vector error
    <= residual / gap). Returns ``None`` -- the caller falls back to ``torch.linalg.eigh`` -- if ``r`` is not small
    against ``T``, or as soon as the observed contraction rate of the residuals says that ``max_iter`` sweeps will not
    do (slowly decaying spectra: a flat tail inside the first ``r`` pairs).
    A full ``eigh`` of a 2000 x 2000 Gram matrix takes 27.7 ms on a B200 (62 % of compute_svd at C5, VERDICT r1);
    the examples of the reference ask for 20-150 modes.
    """
    t = g.size(0)
    b = r + max(8, r // 2)
    if 4 * b > t:
        return None
    gen = pt.Generator(device=g.device).manual_seed(0)
    q = pt.randn((t, b), dtype=pt.float64, device=g.device, generator=gen)
    q, _ = pt.linalg.qr(g @ q)
    history = []
    for sweep in range(max_iter):
        z = g @ q
        h = q.T @ z
        if not bool(pt.isfinite(h).all()):
            return None
        try:
            w, rot = pt.linalg.eigh(0.5 * (h + h.T))
        except RuntimeError:                                   # the small solver gave up: let the full eigh decide
            return None
        w, rot = pt.flip(w, dims=(0,)), pt.flip(rot, dims=(1,))
        x, gx = q @ rot, z @ rot                               # Ritz vectors and G times them
        res = (gx - x * w.unsqueeze(0)).norm(dim=0)
        excess = float((res[:r] / (tol * w[:r].clamp_min(0.0) + 1e-13 * w[0])).max())
        if excess <= 1.0:
            return w[:r], x[:, :r]
        history.append(excess)
        if sweep == 0:
            # residuals contract by about lambda_(b+1) / lambda_i per sweep: without a gap between the r-th Ritz value and
            # the end of the block (a flat noise tail inside the requested pairs) 40 sweeps cannot deliver 1e-7 --
            # decided here, after one sweep, instead of iterating first
            if float(w[r - 1]) < 1.5 * float(w[-1].clamp_min(0.0)) or float(w[r - 1]) <= 0.0:
                return None
        if sweep >= 6:
            rate = (history[-1] / history[-4]) ** (1.0 / 3.0)          # contraction per sweep, last three sweeps
            if not np.isfinite(rate) or rate >= 0.98 or np.log(excess) / -np.log(rate) > (max_iter - 1 - sweep):
                return None
        # next basis: orth(G X). The columns of G X are ~ w_i x_i: normalise them, then Cholesky-QR twice; directions in
        # the (numerical) null space of G carry no information -- refresh them with random vectors
        nrm = gx.norm(dim=0)
        dead = nrm <= 1e-13 * nrm.max()
        y = gx / nrm.clamp_min(1e-300).unsqueeze(0)
        if bool(dead.any()):
            y[:, dead] = pt.randn((t, int(dead.sum())), dtype=pt.float64, device=g.device, generator=gen) / np.sqrt(t)
        for _ in range(2):
            chol, info = pt.linalg.cholesky_ex(y.T @ y)
            if int(info) != 0:
                y, _ = pt.linalg.qr(y)
                break
            y = pt.linalg.solve_triangular(chol, y.T, upper=False).T
        q = y
    return None


def eigenpairs(g: pt.Tensor, rank, r_max: int):
    """Eigenpairs of the symmetric Gram matrix ``g`` in descending order: the top ``min(rank, r_max)`` by subspace
    iteration when that converges (``EIG_METHOD = "auto"``, ``rank`` given), else all of them by ``torch.linalg.eigh``."""
    top = None
    if rank is not None and EIG_METHOD == "auto":
        top = top_eigenpairs(g, max(1, min(int(rank), r_max)))
    if top is not None:
        return top                                     # descending, only the pairs that were asked for
    lam, vec = pt.linalg.eigh(g)                       # ascending, fp64
    return pt.flip(lam, dims=(0,)), pt.flip(vec, dims=(1,))


def _factor(a: pt.Tensor, mean: pt.Tensor, g: pt.Tensor, rank, n_modes, rows_total: int, vol: pt.Tensor, vol_div: int,
            method: str):
    """Eigen-decomposition of the (summed) Gram matrix and projection of the rows held in ``a``."""
    t = a.size(1)
    r_max = min(rows_total, t)
    lam, vec = eigenpairs(g, rank, r_max)
    s_all = lam.clamp_min(0.0).sqrt()
    if rank is None:
        r = optimal_rank(s_all[:r_max], rows_total, t)
    else:
        r = max(1, min(int(rank), r_max))
    s = s_all[:r]
    v = vec[:, :r]
    r_u = r if n_modes is None else max(1, min(int(n_modes), r))
    live = s[:r_u] > 1e-6 * float(s_all[0]) if float(s_all[0]) > 0 else pt.zeros(r_u, dtype=pt.bool, device=a.device)
    inv_s = pt.where(live, 1.0 / s[:r_u].clamp_min(1e-300), pt.zeros_like(s[:r_u]))
    vs = v[:, :r_u] * inv_s.unsqueeze(0)
    u = project(a, mean, vs) if method == "simt" else project_tc(a, mean, vol, vol_div, vs, method)
    return s.to(pt.float32), u, v.to(pt.float32)


def compute_svd_sharded(data_local: pt.Tensor, cell_area_local: pt.Tensor, rank: int = None, method: str = "tc3",
                        n_modes: int = None, sharded_by: str = "cells", n_snapshots_total: int = None,
                        gather_modes: bool = False, group=None) -> Tuple[pt.Tensor, pt.Tensor, pt.Tensor]:
    """
    ``compute_svd`` over several GPUs, one process per GPU (SURVEY 8e, "SVD Gram").

    The contraction runs over the cells, so the cells are sharded: every rank centres, weights and contracts its own
    rows on the tensor cores, the ``T x T`` fp64 partial Gram matrices are summed with ONE all-reduce (32 MB at
    T = 2000), every rank factors the identical sum and projects its own rows. Nothing else crosses the links.

    :param data_local: ``sharded_by="cells"``: ``[n_local, T]`` / ``[n_local, D, T]``, the cells
        ``parallel.row_window(N_cells, world, rank)``; ``sharded_by="time"``: ``[N_cells, (D,) T_s]``, the snapshot
        window the sharded export left on this rank -- it is first transposed with ``parallel.time_to_row_shards``
    :param cell_area_local: areas / volumes of the local cells (``"cells"``) or of all cells (``"time"``)
    :param n_snapshots_total: T, required for ``sharded_by="time"``
    :param gather_modes: all-gather U so that every rank returns all cells (default: the local rows only)
    :return: ``(s [r], U [n_local | N_cells, (D,) r], V [T, r])`` on the device; ``s`` and ``V`` are identical on all ranks
    """
    from . import parallel
    _lib.require_cuda()
    if method not in GRAM_METHODS:
        raise ValueError(f"unknown Gram method '{method}', available: {sorted(GRAM_METHODS)}")
    if sharded_by not in ("cells", "time"):
        raise ValueError(f"sharded_by must be 'cells' or 'time', got '{sharded_by}'")
    if data_local.device.type != "cuda":
        raise ValueError("compute_svd_sharded expects the shard in device memory (one process per GPU)")
    dev = data_local.device
    area = cell_area_local.detach().reshape(-1)
    if sharded_by == "time":
        if n_snapshots_total is None:
            raise ValueError("sharded_by='time' needs n_snapshots_total")
        n_cells_total = data_local.size(0)
        if area.numel() != n_cells_total:
            raise ValueError(f"cell_area has {area.numel()} entries for {n_cells_total} cells")
        data_local = parallel.time_to_row_shards(data_local, n_snapshots_total, group)
        if data_local.size(0) != n_cells_total:        # more than one rank: keep the areas of the local rows
            import torch.distributed as dist
            r0, r1 = parallel.row_window(n_cells_total, dist.get_world_size(group), dist.get_rank(group))
            area = area[r0:r1]
    shape = tuple(data_local.shape)
    if len(shape) not in (2, 3):
        raise ValueError(f"data_local must be [n, T] or [n, D, T], got {shape}")
    if area.numel() != shape[0]:
        raise ValueError(f"cell_area has {area.numel()} entries for {shape[0]} local cells")
    n_local, t = shape[0], shape[-1]
    vol_div = 1 if len(shape) == 2 else shape[1]
    a = _as_device_matrix(data_local, dev).reshape(n_local * vol_div, t)
    vol = area.to(device=dev, dtype=pt.float32).contiguous()

    mean = row_means(a)
    g = gram(a, mean, vol, vol_div, method)
    counts = pt.tensor([a.size(0)], dtype=pt.int64, device=dev)
    parallel.allreduce_sum(g, group)
    parallel.allreduce_sum(counts, group)
    rows_total = int(counts.item())
    s_out, u, v_out = _factor(a, mean, g, rank, n_modes, rows_total, vol, vol_div, method)
    if len(shape) == 3:
        u = u.reshape(n_local, vol_div, u.size(-1))
    if gather_modes:
        u = parallel.gather_rows(u, rows_total // vol_div, group)
    return s_out, u, v_out


def svd_flops(m: int, t: int) -> float:
    """Useful floating point operations of the Gram contraction (full square, 2*M*T^2)."""
    return 2.0 * m * t * t

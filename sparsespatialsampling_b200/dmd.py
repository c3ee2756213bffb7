"""
Exact dynamic mode decomposition (Tu et al. 2014) of the sampled snapshots in the area-weighted inner product, the
third of the reference's post-processing analyses next to the error plots and the SVD (the reference takes it from
``flowtorch.analysis.DMD``, on the host).

With ``X~ = sqrt(w) X`` and ``X1 = X~[:, :-1]``, everything but the modes comes from the uncentred Gram matrix, so the
data matrix is read twice (Gram, modes) and never copied:

    G = X~^T X~                          s3_svd_gram with a zero mean (tcgen05, 3xTF32)
    G[:-1, :-1] = V S^2 V^T              top-r eigenpairs / eigh, fp64 (as compute_svd)
    A~ = S^-1 V^T G[:-1, 1:] V S^-1      r x r, fp64;  A~ Y = Y diag(lambda)   (torch.linalg.eig on the device)
    C = V S^-1 Y                         Phi = X[:, 1:] C
    b = (C^H G[1:, 1:] C)^-1 C^H G[1:, 0]   weighted least squares fit of the first snapshot
    Phi                                  s3_svd_project_tc with a zero mean, coefficients [0; Re C | Im C]

Differences to flowtorch's DMD, stated: the inner product is area-weighted (consistent with ``compute_svd``), the
amplitudes are the weighted least-squares fit of ``x0`` and the pairs are ordered by descending ``|b|``.
"""
import logging
import math

import torch as pt

from . import _lib, svd

logger = logging.getLogger(__name__)

MAX_ERROR_MODES = svd.LOWRANK_MAX_Q // 2


class DMD:
    """Result of ``compute_dmd``. Complex values are complex128 (``modes`` complex64), on the compute device.

    ``s`` ``[rank]`` singular values of the weighted ``X1``; ``eigvals`` ``[rank]`` discrete eigenvalues; ``eigvals_cont``
    = ``log(eigvals) / dt``, ``frequency`` = its imaginary part / 2 pi, ``growth_rate`` = its real part; ``amplitude``
    ``[rank]``; ``dynamics`` ``[rank, T]`` = ``amplitude[i] * eigvals[i] ** t``; ``modes`` ``[N_cells, n]`` or
    ``[N_cells, D, n]``, the first ``n = n_modes`` pairs. Pairs are ordered by descending ``|amplitude|``."""

    def __init__(self, s, eigvals, amplitude, modes, dt, n_snapshots, cell_area, shape):
        self.s = s
        self.rank = int(s.numel())
        self.dt = float(dt)
        self.eigvals = eigvals
        self.eigvals_cont = pt.log(eigvals) / dt
        self.frequency = self.eigvals_cont.imag / (2.0 * math.pi)
        self.growth_rate = self.eigvals_cont.real
        self.amplitude = amplitude
        steps = pt.arange(n_snapshots, dtype=pt.float64, device=eigvals.device)
        self.dynamics = amplitude[:, None] * pt.pow(eigvals[:, None], steps[None, :])
        self.modes = modes
        self._cell_area = cell_area
        self._shape = shape

    @property
    def n_modes(self) -> int:
        return int(self.modes.size(-1))

    def reconstruction_error(self, data_matrix: pt.Tensor):
        """How well the ``n_modes`` pairs reproduce ``data_matrix`` (the input of ``compute_dmd`` again):
        ``Re(modes @ dynamics[:n])`` against the snapshots, by ``s3_lowrank_error`` without forming either. Returns
        ``ErrorStats`` (area-weighted ``sq_err`` / ``sq_ref`` per component and snapshot, ``point_sq_err`` per cell)."""
        _lib.require_cuda()
        if tuple(data_matrix.shape) != self._shape:
            raise ValueError(f"data_matrix has shape {tuple(data_matrix.shape)}, the decomposition {self._shape}")
        n = self.n_modes
        if n > MAX_ERROR_MODES:
            raise ValueError(f"reconstruction_error supports at most {MAX_ERROR_MODES} modes, this DMD holds {n}")
        dev = self.modes.device
        n_cells, t = self._shape[0], self._shape[-1]
        vol_div = 1 if len(self._shape) == 2 else self._shape[1]
        a = svd._as_device_matrix(data_matrix, dev).reshape(n_cells * vol_div, t)
        phi = self.modes.reshape(n_cells * vol_div, n)
        dyn = self.dynamics[:n].T                                          # [T, n]
        left = pt.cat([phi.real, phi.imag], dim=1).float()
        right_t = pt.cat([dyn.real, -dyn.imag], dim=1).float()
        return svd._error_stats(a, left, right_t, None, self._cell_area, vol_div)


def _order(amplitude: pt.Tensor) -> pt.Tensor:
    """Descending |b|; |b| of a conjugate pair can differ in the last bits, so ties are judged at 1e-10 of the largest
    |b| and keep the order of ``eig``."""
    mag = amplitude.abs()
    scale = float(mag.max()) if mag.numel() else 0.0
    key = pt.round(mag / scale * 1e10) if scale > 0 else mag
    return pt.sort(-key, stable=True).indices


def compute_dmd(data_matrix: pt.Tensor, cell_area: pt.Tensor, dt: float, rank: int = None, n_modes: int = None,
                method: str = "tc3", device=None) -> DMD:
    """
    Exact DMD of a field in the area-weighted inner product.

    :param data_matrix: ``[N_cells, T]`` or ``[N_cells, D, T]`` snapshots (host or device, not modified), ``T >= 2``
    :param cell_area: area (2D) / volume (3D) of every cell, ``[N_cells]``
    :param dt: time between two snapshots, ``> 0``
    :param rank: truncation of the SVD of ``X1``; ``None`` = optimal hard threshold (as ``compute_svd``), clamped to
        ``T - 1``
    :param n_modes: number of modes to compute (the leading pairs by ``|b|``), default all ``rank``
    :param method: Gram kernel, as ``compute_svd``
    :return: ``DMD`` whose tensors stay on the compute device even for host input (unlike ``compute_svd``, which moves
        its results back): ``DMD.reconstruction_error`` contracts the modes there, and ``.cpu()`` is one call away
    """
    _lib.require_cuda()
    svd._check_method(method)
    shape = tuple(data_matrix.shape)
    if len(shape) not in (2, 3):
        raise ValueError(f"data_matrix must be [N_cells, T] or [N_cells, D, T], got {shape}")
    t = shape[-1]
    if t < 2:
        raise ValueError(f"DMD needs at least 2 snapshots, got {t}")
    if not dt > 0:
        raise ValueError(f"dt must be positive, got {dt}")
    a, vol, vol_div, dev = svd._field_on_device(data_matrix, cell_area, device)
    zero = pt.zeros((a.size(0),), dtype=pt.float32, device=dev)

    g = svd.gram(a, zero, vol, vol_div, method)
    s_all, vec, r = svd._spectrum(g[:-1, :-1], rank, a.size(0), t - 1)
    # the cutoff of compute_svd's modes: below 1e-6 sigma_0, S^-1 only amplifies the rounding of G (whose 1e-6 accuracy
    # holds for sigma^2, so singular values below about 1e-3 sigma_0 that are kept already carry that rounding)
    live = int((s_all[:r] > 1e-6 * float(s_all[0])).sum()) if float(s_all[0]) > 0 else 0
    if live < 1:
        raise ValueError("the snapshots are zero: there is nothing to decompose")
    if live < r:
        logger.warning(f"rank {r} reduced to {live}: the remaining singular values are below 1e-6 of the largest")
        r = live
    s = s_all[:r]
    vs = vec[:, :r] / s[None, :]                                            # V S^-1, fp64 [T-1, r]
    a_tilde = vs.T @ g[:-1, 1:] @ vs
    eigvals, y = pt.linalg.eig(a_tilde)
    c = vs.to(pt.complex128) @ y                                            # [T-1, r]
    g11 = g[1:, 1:].to(pt.complex128)
    h = c.conj().T @ g11 @ c
    rhs = c.conj().T @ g[1:, 0].to(pt.complex128)
    amplitude = pt.linalg.solve(h, rhs)
    order = _order(amplitude)
    eigvals, amplitude, c = eigvals[order], amplitude[order], c[:, order]

    n = r if n_modes is None else max(1, int(n_modes))
    if n > r:
        logger.warning(f"Number of modes is set to {n}, but found only {r} modes.")
        n = r
    coef = pt.zeros((t, 2 * n), dtype=pt.float32, device=dev)              # row 0: X[:, 0] is not in X[:, 1:]
    coef[1:, :n] = c[:, :n].real.float()
    coef[1:, n:] = c[:, :n].imag.float()
    u = svd._project(a, zero, vol, vol_div, coef, method)
    modes = pt.complex(u[:, :n], u[:, n:])
    modes = modes.reshape(shape[:-1] + (n,))
    return DMD(s, eigvals, amplitude, modes, dt, t, vol, shape)

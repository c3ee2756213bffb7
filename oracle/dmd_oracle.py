"""fp64 numpy exact DMD, the CPU reference of sparsespatialsampling_b200.dmd (kept apart from s3_oracle.py, which
restates the reference package)."""
import numpy as np


def compute_dmd(a, area, rank):
    """Exact DMD (Tu et al. 2014) in the area-weighted inner product, fp64, by a path independent of the Gram matrix:
    thin SVD of sqrt(w) X1, Atilde = U^T X~2 V S^-1, modes Phi = X2 V S^-1 Y (unweighted), amplitudes by weighted least
    squares of the first snapshot on the full Phi, pairs ordered by descending |b| (ties: eig order, judged at 1e-10).
    a: [N, T] or [N, D, T]. Returns (eigvals, amplitude, modes [N, (D,) r], s)."""
    a = np.asarray(a, dtype=np.float64)
    shape = a.shape
    d = 1 if a.ndim == 2 else shape[1]
    x = a.reshape(shape[0] * d, shape[-1])
    w = np.repeat(np.asarray(area, dtype=np.float64), d)
    sw = np.sqrt(w)[:, None]
    x1, x2 = sw * x[:, :-1], sw * x[:, 1:]
    u, s, vt = np.linalg.svd(x1, full_matrices=False)
    r = min(rank, s.size)
    u, s, v = u[:, :r], s[:r], vt[:r].T
    a_tilde = u.T @ x2 @ v / s[None, :]
    lam, y = np.linalg.eig(a_tilde)
    phi = x[:, 1:] @ (v / s[None, :]) @ y
    b = np.linalg.lstsq(sw * phi, sw[:, 0] * x[:, 0], rcond=None)[0]
    mag = np.abs(b)
    order = np.argsort(-np.round(mag / mag.max() * 1e10), kind="stable")
    lam, b, phi = lam[order], b[order], phi[:, order]
    return lam, b, phi.reshape(shape[:-1] + (r,)), s

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


def compute_dmd_torch(a, area, rank, block=65536):
    """The same exact DMD in fp64 with torch, on the device of ``a``, for sizes where the numpy oracle takes minutes
    (582 000 x 2000). Independent of the Gram matrix as well: QR of sqrt(w) X1 = Q R, SVD of the small R = U_r S V^T
    (so U = Q U_r), Atilde = U^T X~2 V S^-1, Phi = X2 V S^-1 Y, amplitudes by least squares (QR of sqrt(w) Phi) on the
    full Phi, the ordering of ``compute_dmd``. X~2 and Phi are formed ``block`` rows at a time from the fp32 input, so
    the large fp64 arrays are sqrt(w) X1, Q and the working copy that the QR keeps while it runs: 9.3 GB each at
    582 000 x 2000, about 28 GB on top of the input (an estimate from the sizes).
    a: fp32/fp64 tensor [N, T] or [N, D, T], area [N]. Returns torch (eigvals, amplitude, modes [N, (D,) r], s)."""
    import torch as pt
    shape = tuple(a.shape)
    d = 1 if a.dim() == 2 else shape[1]
    x = a.reshape(shape[0] * d, shape[-1])
    dev = x.device
    sw = area.to(dev, pt.float64).repeat_interleave(d).sqrt()
    q, r_fac = pt.linalg.qr(x[:, :-1].double().mul_(sw[:, None]))
    u_r, s, vt = pt.linalg.svd(r_fac)
    r = min(int(rank), s.numel())
    u_r, s, vs = u_r[:, :r], s[:r], vt[:r].T / s[:r][None, :]             # vs = V S^-1, [T-1, r]
    p = pt.empty((x.size(0), r), dtype=pt.float64, device=dev)             # X2 V S^-1
    for r0 in range(0, x.size(0), block):
        p[r0:r0 + block] = x[r0:r0 + block, 1:].double() @ vs
    a_tilde = u_r.T @ (q.T @ (p * sw[:, None]))
    del q
    lam, y = pt.linalg.eig(a_tilde)
    phi = p.to(pt.complex128) @ y
    qp, rp = pt.linalg.qr(phi * sw[:, None])
    b = pt.linalg.solve_triangular(rp, qp.conj().T @ (sw * x[:, 0].double()).to(pt.complex128)[:, None],
                                   upper=True)[:, 0]
    mag = b.abs()
    order = pt.sort(-pt.round(mag / mag.max() * 1e10), stable=True).indices
    lam, b, phi = lam[order], b[order], phi[:, order]
    return lam, b, phi.reshape(shape[:-1] + (r,)), s

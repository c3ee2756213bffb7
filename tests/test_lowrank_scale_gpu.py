"""s3_lowrank_error, the POD truncation error and compute_dmd at production sizes, against fp64 references computed
with torch on the same GPU, under tolerances that follow from an error model of the kernel.

Error model of ``s3_lowrank_error``. The fp64 reference is ``e = (a - mean) - left right_t^T``, formed from the same
fp32 inputs in row blocks of 65 536. The kernel differs from it in two ways only: the product is a 3xTF32 product
(hi hi + hi lo + lo hi, ``lo`` truncated to TF32 by the tensor core) accumulated in fp32 in TMEM, and ``e`` is rounded
to fp32 before it is squared and summed in fp64. Elementwise, the product error is at most

    delta[m, t] = (2^-19 + n_mma 2^-23) sum_j |left[m, j]| |right_t[t, j]|,   n_mma = 3 q_pad / 8,  q_pad = 32 ceil(q / 32)

The first term covers the split (``lo`` truncated to TF32 and the dropped ``lo lo`` term, about 1.25 2^-20 of
|x| |y|), the second one truncating fp32 add per MMA. The rounding of ``e`` adds 2^-24 (|e| + delta). By the triangle
inequality, for every component and column (``||.||_w`` the area-weighted norm over the rows of that component):

    | sqrt(sq_err) - ||e||_w | <= (1 + 2^-24) ||delta||_w + 2^-24 ||e||_w
    | max_abs - max |e| |      <= max (delta + 2^-24 (|e| + delta))
    the first bound unweighted for every row of ``row_sq_err``,  sq_ref within 1e-11 (fp64 sums in another order)

The bound holds for every input, not only for typical roundings, as long as the tensor core behaves as modelled:
products of TF32 operands exact, and one truncating fp32 add per MMA into the accumulator. A TF32 MMA aligns and
truncates its eight products and the accumulator internally, which is not literally one rounding; the model is that
this loses no more than one fp32 truncation of the sum of the magnitudes. It can fail: the residual of a
product of the operands rounded once to TF32 (``rna``, what a kernel that dropped the ``lo`` passes would compute)
exceeds it in every column at q = 20 and q = 100 once the residual is not far above the product error (levels
<= 1e-4 below; an fp32 emulation of the 3xTF32 product put the 1xTF32 deviation at about 20x the bound at q = 20 and
4x at q = 100 there). At q = 512 the ``n_mma`` term grows linearly in q while random-sign rounding errors grow like
sqrt(q), so there the bound is not claimed to separate the two.

Residual levels: ``a = fp32(mean + left right_t^T + eps N)`` with a unit-rms product, q = 20 and 100. ``delta``
dominates the bound (||delta||_w > ||e||_w) below eps of about 1e-5 at q = 20 and 5e-5 at q = 100 (it is a property
of the inputs: 0.95 and 0.49 at 1e-5 and 1e-4 respectively). That is the level below which the kernel's error
statistics are no longer guaranteed to one significant digit: its measurement floor.

Largest deviation / bound measured on one NVIDIA B200, power limit 1000 W: not measured.

Sizes reach the work distribution of the kernel: row tiles of 128 rows are dealt out in at most 1024 groups of
``ceil(n_rt / 1024)`` consecutive tiles, a CTA loops over groups ``blockIdx.x, +gridDim.x, ...``, and a group's
partials are read, added and written back tile by tile.

DMD: ``compute_dmd`` against ``oracle.dmd_oracle.compute_dmd_torch`` (QR of the weighted X1, no Gram matrix) on fields
of damped and growing oscillation pairs with exact eigenvalues. The Gram matrix of 3xTF32 is accurate to about
eps_G = 1e-6 of sigma_0^2 (DESIGN 3.3, 3.5). ``A~ = S^-1 V^T G[:-1, 1:] V S^-1`` turns an error E of G into
``V_i^T E V_j / (sigma_i sigma_j)``. At the rank of the signal every kept direction belongs to a signal pair, so a pair
whose singular values are about sigma_i gets ``eps_G (sigma_0 / sigma_i)^2`` for lambda, and that over the distance
``gap_i`` to the nearest other eigenvalue for its eigenvector and so for ``Phi b``. Those are the tolerances at that
rank. With noise directions kept (rank 50, 256) the same formula with sigma_j = sigma_noise would grow like
1 / sigma_noise and bound nothing; there a pair is held to the larger of the model's tolerance and fixed scales, 1e-4
for lambda (the scale of the small-grid tests) and 1e-3 for ``Phi b`` (``NOISE_RANK_TOL``). Beside a steady part the
model gives the pairs at sigma / sigma_0 = 1e-1, 1e-2 and 2e-3 lambda tolerances of 1e-4, 1e-2 and 0.25 and ``Phi b``
tolerances of about 3e-3, 0.2 and 5: it says nothing about the mode of the last two, only the measured deviations do.
Measured on one NVIDIA B200, power limit 1000 W: not measured.

Time and peak device memory of this file on one B200: not measured (budget: under 5 minutes, at most 60 GB of device memory).
"""
import time

import pytest
import torch as pt

from oracle import dmd_oracle

pytestmark = pytest.mark.gpu

BLOCK = 65536                    # rows per block of the fp64 references
U32 = 2.0 ** -24                 # unit roundoff of fp32


def _coef(q):
    """Relative product error of the 3xTF32 product with q terms, in units of sum_j |left| |right_t|."""
    q_pad = -(-q // 32) * 32
    return 2.0 ** -19 + 3 * q_pad / 8 * 2.0 ** -23


def _rna_tf32(x):
    """fp32 rounded to TF32 (10 explicit mantissa bits), to nearest with ties away from zero, as cvt.rna.tf32.f32."""
    bits = x.contiguous().view(pt.int32)
    return ((bits + 0x1000) & -0x2000).view(pt.float32)


_PEAK = [0]                      # peak device memory of the file, across the resets of the DMD tests


def _fold_peak():
    _PEAK[0] = max(_PEAK[0], pt.cuda.max_memory_allocated())


@pytest.fixture(scope="module", autouse=True)
def budget():
    """Wall time and peak device memory of the whole file (printed with -s)."""
    if not pt.cuda.is_available():
        yield
        return
    pt.cuda.synchronize()
    pt.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    pt.cuda.synchronize()
    _fold_peak()
    print(f"\n[test_lowrank_scale_gpu] {pt.cuda.get_device_name()}: {time.perf_counter() - t0:.1f} s, "
          f"peak {_PEAK[0] / 2 ** 30:.1f} GiB allocated")


def _reference(a, left, right_t, mean, vol, vol_div, tf32_only=False):
    """fp64 residual statistics and the error bound, ``BLOCK`` rows at a time (blocks hold whole cells).
    ``tf32_only``: also ``sum w e1^2`` of the residual of the 1xTF32 product, rounded to fp32 like the kernel's."""
    m, t = a.shape
    dev = a.device
    c = _coef(left.size(1))
    z = lambda: pt.zeros((vol_div, t), dtype=pt.float64, device=dev)
    ref = {k: z() for k in ("sq_err", "sq_ref", "sq_delta", "max_abs", "max_slack", "sq_err_1x")}
    ref["row_sq"] = pt.empty(m, dtype=pt.float64, device=dev)
    ref["row_sq_delta"] = pt.empty(m, dtype=pt.float64, device=dev)
    r64 = right_t.double()
    r64_abs = r64.abs()
    r1x = _rna_tf32(right_t).double() if tf32_only else None
    step = BLOCK - BLOCK % vol_div
    for r0 in range(0, m, step):
        r1 = min(r0 + step, m)
        nc = (r1 - r0) // vol_div
        w = vol[r0 // vol_div:r1 // vol_div].double() if vol is not None else pt.ones(nc, dtype=pt.float64, device=dev)
        wsum = lambda y: pt.einsum("n,nct->ct", w, y.view(nc, vol_div, t))
        cmax = lambda y: y.view(nc, vol_div, t).amax(0)
        x = a[r0:r1].double()
        if mean is not None:
            x -= mean[r0:r1].double()[:, None]
        l64 = left[r0:r1].double()
        e = x - l64 @ r64.T
        delta = (l64.abs() @ r64_abs.T).mul_(c)
        ref["sq_err"] += wsum(e * e)
        ref["sq_ref"] += wsum(x * x)
        ref["sq_delta"] += wsum(delta * delta)
        ref["row_sq"][r0:r1] = (e * e).sum(1)
        ref["row_sq_delta"][r0:r1] = (delta * delta).sum(1)
        ref["max_abs"] = pt.maximum(ref["max_abs"], cmax(e.abs()))
        ref["max_slack"] = pt.maximum(ref["max_slack"], cmax(delta + U32 * (e.abs() + delta)))
        if tf32_only:
            e1 = (x - _rna_tf32(left[r0:r1]).double() @ r1x.T).float().double()
            ref["sq_err_1x"] += wsum(e1 * e1)
        del x, e, delta, l64
    return ref


def _norm_bound(sq_e, sq_delta):
    return (1 + U32) * sq_delta.sqrt() + U32 * sq_e.sqrt()


def _check(got, ref, row=None):
    """Asserts the bounds of the module docstring; returns the largest deviation / bound of the three statistics."""
    sq_err, sq_ref, max_abs = got
    bound = _norm_bound(ref["sq_err"], ref["sq_delta"])
    dev = (sq_err.sqrt() - ref["sq_err"].sqrt()).abs()
    ratios = {"sq_err": float((dev / bound.clamp_min(1e-300)).max())}
    assert bool((dev <= bound).all()), ("sq_err", ratios["sq_err"])
    rel = float(((sq_ref - ref["sq_ref"]).abs() / ref["sq_ref"].clamp_min(1e-300)).max())
    assert rel <= 1e-11, ("sq_ref", rel)
    dev = (max_abs - ref["max_abs"]).abs()
    ratios["max_abs"] = float((dev / ref["max_slack"].clamp_min(1e-300)).max())
    assert bool((dev <= ref["max_slack"]).all()), ("max_abs", ratios["max_abs"])
    if row is not None:
        bound = _norm_bound(ref["row_sq"], ref["row_sq_delta"])
        dev = (row.sqrt() - ref["row_sq"].sqrt()).abs()
        ratios["row"] = float((dev / bound.clamp_min(1e-300)).max())
        assert bool((dev <= bound).all()), ("row_sq_err", ratios["row"])
    return ratios


def _inputs(m, t, q, vol_div, seed, eps=1e-3):
    """``a = fp32(mean + left right_t^T + eps N)``: a unit-rms product, a mean about 2 and areas 2^-8..2^-1."""
    g = pt.Generator(device="cuda").manual_seed(seed)
    left = pt.randn((m, q), device="cuda", generator=g) / q ** 0.5
    right_t = pt.randn((t, q), device="cuda", generator=g)
    mean = pt.randn((m,), device="cuda", generator=g) * 0.5 + 2.0
    vol = 2.0 ** -pt.randint(1, 9, (m // vol_div,), device="cuda", generator=g).float()
    a = pt.empty((m, t), dtype=pt.float32, device="cuda")
    r64 = right_t.double()
    for r0 in range(0, m, BLOCK):                      # in fp64, rounded once
        r1 = min(r0 + BLOCK, m)
        noise = pt.randn((r1 - r0, t), device="cuda", generator=g, dtype=pt.float64)
        a[r0:r1] = (left[r0:r1].double() @ r64.T).add_(mean[r0:r1].double()[:, None]).add_(noise, alpha=eps).float()
    return a, left, right_t, mean, vol


def _run(a, left, right_t, mean, vol, vol_div):
    from sparsespatialsampling_b200 import svd
    row = pt.zeros(a.size(0), dtype=pt.float64, device=a.device)
    return svd.lowrank_error(a, left, right_t, mean, vol, vol_div, row), row


CASES = [
    (131_072, 600, 32, 1),            # 1024 groups of one tile, about 7 groups per CTA
    (131_073, 600, 32, 1),            # 513 groups of two tiles, the last of one
    (582_000, 2000, 20, 1),           # C5: 910 groups of 5 tiles (the last of 2), 8 column tiles, the last ragged
    (582_000, 2000, 100, 1),
    (582_000, 2000, 512, 1),
    (582_000, 2001, 256, 3),          # 194 000 cells x 3: components straddle row tiles; t % 4 != 0: scalar loads
    (4_194_304, 256, 8, 1),           # 1024 groups of 32 tiles
]


@pytest.mark.parametrize("m,t,q,vol_div", CASES)
def test_lowrank_error_at_production_sizes(cuda, m, t, q, vol_div):
    from sparsespatialsampling_b200 import _lib
    a, left, right_t, mean, vol = _inputs(m, t, q, vol_div, seed=m + t + q)
    got, row = _run(a, left, right_t, mean, vol, vol_div)
    ratios = _check(got, _reference(a, left, right_t, mean, vol, vol_div), row)
    print(f"\n[lowrank] m {m} t {t} q {q} vol_div {vol_div}: deviation / bound {ratios}")
    if (m, t, q) == (582_000, 2000, 20):
        try:                                           # one CTA walks all 910 groups; 7 CTAs 130 each
            for cap in (1, 7):
                _lib.tune(19, cap)
                capped, row_c = _run(a, left, right_t, mean, vol, vol_div)
                assert all(pt.equal(x, y) for x, y in zip(got, capped)), cap
                assert pt.equal(row, row_c), cap
        finally:
            _lib.tune(19, 0)


LEVELS = [1e-2, 1e-3, 1e-4, 1e-5, 1e-6]


@pytest.mark.parametrize("q", [20, 100])
@pytest.mark.parametrize("eps", LEVELS)
def test_residual_levels(cuda, eps, q):
    """The residuals a well-resolved model leaves (1e-2..1e-3 of the signal) and below, where the Gram formula of the
    error has long lost them; a 1xTF32 product must fail the same bound wherever the residual is not far above its
    error."""
    m, t = 200_000, 600
    a, left, right_t, mean, vol = _inputs(m, t, q, 1, seed=q, eps=eps)
    got, row = _run(a, left, right_t, mean, vol, 1)
    ref = _reference(a, left, right_t, mean, vol, 1, tf32_only=True)
    ratios = _check(got, ref, row)
    floor = float((ref["sq_delta"] / ref["sq_err"]).sqrt().median())        # ||delta||_w / ||e||_w
    bound = _norm_bound(ref["sq_err"], ref["sq_delta"])
    tf32_ratio = (ref["sq_err_1x"].sqrt() - ref["sq_err"].sqrt()).abs() / bound
    print(f"\n[levels] eps {eps:g} q {q}: deviation / bound {ratios}, ||delta|| / ||e|| {floor:.3g}, "
          f"1xTF32 deviation / bound min {float(tf32_ratio.min()):.3g} median {float(tf32_ratio.median()):.3g}")
    if eps <= 1e-4:
        assert float(tf32_ratio.min()) > 1.0, float(tf32_ratio.min())
    if eps == 1e-4:                                    # the relative L2 error per snapshot, as a user reads it
        rel = (got[0] / got[1]).sqrt()
        rel_ref = (ref["sq_err"] / ref["sq_ref"]).sqrt()
        assert float((rel / rel_ref - 1).abs().max()) <= 1e-2


def _pod_field(m, t, seed, n_modes=5, noise=1e-3):
    """As tests/test_svd_scale_gpu.py: a few coherent modes, small noise and a large row mean."""
    g = pt.Generator(device="cuda").manual_seed(seed)
    time_ = pt.linspace(0, 2 * pt.pi, t + 1, device="cuda", dtype=pt.float64)[:-1]
    amp = 2.0 ** -pt.arange(n_modes, device="cuda", dtype=pt.float64)
    phase = pt.rand((n_modes, 1), device="cuda", generator=g, dtype=pt.float64)
    temporal = (amp[:, None] * pt.cos(pt.arange(1, n_modes + 1, device="cuda")[:, None] * time_[None, :] + phase)).float()
    a = pt.randn((m, t), device="cuda", generator=g).mul_(noise)
    a.addmm_(pt.randn((m, n_modes), device="cuda", generator=g), temporal)
    a.add_(pt.randn((m, 1), device="cuda", generator=g)).add_(3.0)
    return a


def test_pod_truncation_error_at_c5_size(cuda):
    """``svd.reconstruction_error`` of ``compute_svd``'s own triplets, 582 000 x 2000, r = 1 (the coherent modes left
    in the residual), 50 (noise only) and 512 (the kernel's largest q)."""
    from sparsespatialsampling_b200 import compute_svd, svd
    m, t = 582_000, 2000
    a = _pod_field(m, t, 11)
    vol = 2.0 ** -pt.randint(1, 9, (m,), device="cuda", generator=pt.Generator(device="cuda").manual_seed(12)).float()
    s, u, v = compute_svd(a, vol, rank=512)
    mean = svd.row_means(a)
    for r in (1, 50, 512):
        stats = svd.reconstruction_error(a, vol, s[:r], u[:, :r], v[:, :r])
        left = (u[:, :r].double() * s[:r].double()[None, :]).float()         # rounded once, as the call does
        ref = _reference(a, left, v[:, :r].contiguous(), mean, vol, 1)
        ratios = _check((stats.sq_err, stats.sq_ref, stats.max_abs), ref, stats.point_sq_err.reshape(-1))
        print(f"\n[pod] r {r}: deviation / bound {ratios}")


# ------------------------------------------------------------------------------------------------------------- DMD

PAIRS = ((-0.4, 3.0, 1.0), (0.3, 7.0, 0.5), (-0.2, 11.0, 0.25))     # (growth rate, frequency, amplitude)
TOL_GRAM = 1e-6                                                     # accuracy of the 3xTF32 Gram, of sigma_0^2


def _dmd_field(n_cells, d, t, pairs, steady=0.0, noise=1e-3, seed=0):
    """Oscillation pairs ``amp psi_i(x) Re(exp(i phi) lambda_i^k)`` with exact ``lambda_i = exp((s + 2 pi i f) dt)``,
    ``dt = 2 / T`` (so |s dt T| <= 0.8), on random points with areas 2^-7..2^0, an optional steady mode
    (``lambda = 1``), plus ``noise`` N(0, 1). Returns the fp32 field ``[n_cells, (d,) T]``, the areas, dt, the exact
    eigenvalues and, per mode, the two singular values of its weighted rank-2 (steady: rank-1) part."""
    g = pt.Generator(device="cuda").manual_seed(seed)
    f64 = dict(device="cuda", dtype=pt.float64)
    dd = 1 if d is None else d
    rows = n_cells * dd
    dt = 2.0 / t
    xy = pt.rand((n_cells, 2), generator=g, **f64).repeat_interleave(dd, 0)
    comp = (pt.arange(rows, device="cuda") % dd).double()
    area = 2.0 ** -pt.randint(0, 8, (n_cells,), device="cuda", generator=g).float()
    w = area.double().repeat_interleave(dd)
    k = pt.arange(t, **f64)
    cols_l, cols_r, lams, blocks = [], [], [], []
    if steady:
        cols_l.append(steady * (1.0 + 0.5 * pt.cos(pt.pi * xy[:, 0])) * (1.0 + comp))
        cols_r.append(pt.ones(t, **f64))
        lams.append(complex(1.0, 0.0))
        blocks.append(slice(0, 1))
    for i, (s, f, amp) in enumerate(pairs):
        lam = pt.exp(pt.tensor(complex(s, 2 * pt.pi * f) * dt, dtype=pt.complex128))
        psi = amp * pt.cos((i + 1) * pt.pi * xy[:, 0] + i * pt.pi * xy[:, 1]) * (1.0 + comp)
        phase = 2 * pt.pi * pt.rand(rows, generator=g, **f64)
        powk = lam.to("cuda") ** k
        cols_l += [psi * pt.cos(phase), -psi * pt.sin(phase)]
        cols_r += [powk.real, powk.imag]
        lams += [complex(lam), complex(lam.conj())]
        blocks.append(slice(len(cols_l) - 2, len(cols_l)))
    big_l, big_r = pt.stack(cols_l, 1), pt.stack(cols_r, 0)
    sigmas = []                                       # singular values of sqrt(w) L_b R_b: sqrt(eig(L^T W L R R^T))
    for b in blocks:
        lwl = big_l[:, b].T @ (w[:, None] * big_l[:, b])
        rr = big_r[b] @ big_r[b].T
        sigmas.append(pt.linalg.eigvals(lwl @ rr).real.clamp_min(0).sqrt().sort().values.cpu())
    a = pt.empty((rows, t), dtype=pt.float32, device="cuda")
    for r0 in range(0, rows, BLOCK):
        r1 = min(r0 + BLOCK, rows)
        a[r0:r1] = (big_l[r0:r1] @ big_r).add_(pt.randn((r1 - r0, t), generator=g, **f64), alpha=noise).float()
    shape = (n_cells, t) if d is None else (n_cells, d, t)
    return a.reshape(shape), area, dt, lams, sigmas


# With noise directions kept (rank 50, 256), a pair is held to the tolerance of the model or to these fixed scales (the
# scale of the small-grid tests for lambda, ten times it for Phi b), whichever is larger: the coupling to a noise
# direction of singular value sigma_n grows like 1 / sigma_n in the worst case, which would make any tolerance vacuous.
NOISE_RANK_TOL = (1e-4, 1e-3)


def _signal_margins(dmd, ref, lams, sigmas, area, dd, floor=(0.0, 0.0)):
    """Matches every exact eigenvalue to the nearest of the reference and of ``dmd``; returns, per signal eigenvalue,
    the deviations of lambda and of Phi b (weighted, relative) from the reference and their tolerances:
    ``eps_G (sigma_0 / sigma_i)^2`` for lambda, that over ``gap_i`` for Phi b, at least ``floor``."""
    lam_ref, b_ref, phi_ref, s_ref = ref
    lam_got = dmd.eigvals
    sigma0 = float(s_ref[0])
    sw = area.double().repeat_interleave(dd).sqrt()
    phi_ref = phi_ref.reshape(-1, phi_ref.size(-1))
    phi_got = dmd.modes.reshape(-1, dmd.modes.size(-1))
    sig_of = [sg[0] for sg in sigmas for _ in range(2 if sg.numel() == 2 else 1)]   # the smaller one of each part
    rows, used = [], set()
    for z, sigma_i in zip(lams, sig_of):
        z = pt.tensor(z, dtype=pt.complex128, device=lam_ref.device)
        j = int((lam_ref - z).abs().argmin())
        assert float((lam_ref[j] - z).abs()) <= 1e-2, (complex(z), complex(lam_ref[j]))      # the pair is resolved
        i = int((lam_got - lam_ref[j]).abs().argmin())
        assert i not in used
        used.add(i)
        model = TOL_GRAM * (sigma0 / float(sigma_i)) ** 2
        others = pt.cat([lam_ref[:j], lam_ref[j + 1:]])
        gap = float((others - lam_ref[j]).abs().min()) if others.numel() else 1.0
        want = phi_ref[:, j] * b_ref[j] * sw
        got = phi_got[:, i].to(pt.complex128) * dmd.amplitude[i] * sw
        rows.append(dict(lam=complex(z), sigma=float(sigma_i) / sigma0, exact=float((lam_ref[j] - z).abs()),
                         err_lam=float((lam_got[i] - lam_ref[j]).abs()), tol_lam=max(floor[0], model),
                         err_phi=float((got - want).norm() / want.norm()), tol_phi=max(floor[1], model / gap)))
    return rows


def _assert_margins(label, rows):
    for r in rows:
        print(f"[dmd] {label}: lambda {r['lam']:.6f} (sigma / sigma_0 {r['sigma']:.2g}, reference - exact "
              f"{r['exact']:.2g}): |dlambda| {r['err_lam']:.3g} (tol {r['tol_lam']:.3g}), "
              f"Phi b {r['err_phi']:.3g} (tol {r['tol_phi']:.3g})")
    for r in rows:
        assert r["err_lam"] <= r["tol_lam"], r
        assert r["err_phi"] <= r["tol_phi"], r


@pytest.mark.parametrize("name,n_cells,d,t,steady", [
    ("C5", 582_000, None, 2000, 0.0),
    ("C2 vector", 99_000, 3, 1000, 0.0),
    ("steady part", 99_000, None, 1000, 1.0),
])
def test_dmd_at_production_sizes(cuda, name, n_cells, d, t, steady):
    """At the rank of the signal (6 pairs' eigenvalues, 7 with the steady mode) under the model's tolerances, and at
    rank 50, where the noise pairs are decided by Gram rounding, for the signal pairs only. With the steady part, the
    fluctuation pairs sit at sigma / sigma_0 of about 1e-1, 1e-2 and 2e-3."""
    from sparsespatialsampling_b200 import compute_dmd
    pairs = ((-0.4, 3.0, 0.43), (0.3, 7.0, 0.022), (-0.2, 11.0, 0.0073)) if steady else PAIRS
    a, area, dt, lams, sigmas = _dmd_field(n_cells, d, t, pairs, steady=steady, seed=t)
    dd = 1 if d is None else d
    rows = {}
    for rank, floor in ((len(lams), (0.0, 0.0)), (50, NOISE_RANK_TOL)):
        dmd = compute_dmd(a, area, dt, rank=rank)
        assert dmd.rank == rank
        pt.cuda.synchronize()
        base = pt.cuda.memory_allocated()
        _fold_peak()
        pt.cuda.reset_peak_memory_stats()
        ref = dmd_oracle.compute_dmd_torch(a, area, rank)
        print(f"\n[dmd] {name}, rank {rank}: reference peak {(pt.cuda.max_memory_allocated() - base) / 2 ** 30:.1f} "
              f"GiB above the {base / 2 ** 30:.1f} GiB held before it")
        _fold_peak()
        rows[rank] = _signal_margins(dmd, ref, lams, sigmas, area, dd, floor)
        del dmd, ref
    for rank, r in rows.items():
        _assert_margins(f"{name}, rank {rank}", r)


def test_dmd_past_the_256_snapshot_padding_and_256_mode_error(cuda):
    """T = 257: the paired Gram pads to 512 columns. Rank 256 = T - 1: noise of 1e-2 supplies the singular values above
    the 1e-6 sigma_0 cutoff (about 1e-3 sigma_0, so their squares stay above the Gram rounding; at 1e-3 they would sit
    near it and the rank could drop), and ``reconstruction_error`` with all 256 pairs is q = 512, against ``X - Re(Phi dyn)`` in
    fp64 from the call's own modes and dynamics: ``[Re Phi | Im Phi] [Re dyn^T | -Im dyn^T]^T``."""
    from sparsespatialsampling_b200 import compute_dmd
    n_cells, t = 99_000, 257
    a, area, dt, lams, sigmas = _dmd_field(n_cells, None, t, PAIRS, noise=1e-2, seed=t)
    dmd = compute_dmd(a, area, dt, rank=256)
    assert dmd.rank == 256 and dmd.n_modes == 256
    ref = dmd_oracle.compute_dmd_torch(a, area, 256)
    rows = _signal_margins(dmd, ref, lams, sigmas, area, 1, NOISE_RANK_TOL)
    stats = dmd.reconstruction_error(a)
    phi = dmd.modes.reshape(n_cells, 256)
    dyn = dmd.dynamics.T
    left = pt.cat([phi.real, phi.imag], dim=1).float()
    right_t = pt.cat([dyn.real, -dyn.imag], dim=1).float()
    assert bool(pt.isfinite(right_t).all())
    ref_err = _reference(a, left, right_t, None, area, 1)
    ratios = _check((stats.sq_err, stats.sq_ref, stats.max_abs), ref_err, stats.point_sq_err.reshape(-1))
    print(f"[dmd] T = 257, 256 pairs: deviation / bound {ratios}, "
          f"relative L2 error max {float(stats.relative_l2().max()):.3g}")
    _assert_margins("T = 257", rows)

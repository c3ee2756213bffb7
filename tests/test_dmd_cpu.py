"""
Host logic of compute_dmd (no GPU): the Gram algebra, amplitudes, ordering and conjugate pairs against the fp64 numpy
oracle, the time step taken from write times, and the input checks. The kernels are replaced by fp64 torch stand-ins
with the same contract.
"""
import numpy as np
import pytest
import torch as pt

from oracle import dmd_oracle


def _gram(a, mean, vol, vol_div=1, method="tc3"):
    b = (a.double() - mean.double()[:, None]) * vol.double().repeat_interleave(vol_div).sqrt()[:, None]
    return b.T @ b


def _project_tc(a, mean, vol, vol_div, vs, method="tc3"):
    return ((a.double() - mean.double()[:, None]) @ vs.double()).float()


@pytest.fixture
def host(monkeypatch):
    from sparsespatialsampling_b200 import _lib, svd
    monkeypatch.setattr(_lib, "require_cuda", lambda: None)
    monkeypatch.setattr(svd, "gram", _gram)
    monkeypatch.setattr(svd, "project_tc", _project_tc)
    monkeypatch.setattr(svd, "EIG_METHOD", "eigh")


def _oscillations(n, t, d=None, noise=0.0, seed=0):
    """Three damped oscillations (six complex eigenvalues) on random points, fp32, plus optional noise."""
    rng = np.random.default_rng(seed)
    shape = (n,) if d is None else (n, d)
    dt = 0.01
    k = np.arange(t) * dt
    a = np.zeros(shape + (t,))
    for sigma, f, amp in ((-0.2, 3.0, 1.0), (0.1, 7.0, 0.5), (-0.5, 11.0, 0.25)):
        c, s = rng.standard_normal(shape), rng.standard_normal(shape)
        env = amp * np.exp(sigma * k)
        a += c[..., None] * env * np.cos(2 * np.pi * f * k) - s[..., None] * env * np.sin(2 * np.pi * f * k)
    a += noise * rng.standard_normal(a.shape)
    area = rng.random(n) + 0.5
    return a.astype(np.float32), area.astype(np.float32), dt


@pytest.mark.parametrize("d", [None, 2])
def test_gram_algebra_matches_the_oracle(host, d):
    from sparsespatialsampling_b200.dmd import compute_dmd
    a, area, dt = _oscillations(300, 80, d, noise=1e-3, seed=1)
    dmd = compute_dmd(pt.from_numpy(a), pt.from_numpy(area), dt, rank=6, device="cpu")
    lam, b, phi, s = dmd_oracle.compute_dmd(a, area, 6)
    assert dmd.rank == 6 and dmd.eigvals.dtype == pt.complex128 and dmd.modes.dtype == pt.complex64
    assert np.abs(dmd.s.numpy() - s).max() <= 1e-10 * s[0]
    # same pairs in the same order (descending |b|), conjugate pairs both kept
    assert np.abs(dmd.eigvals.numpy() - lam).max() <= 1e-10
    assert np.abs(np.abs(dmd.amplitude.numpy()) - np.abs(b)).max() <= 1e-10 * np.abs(b).max()
    assert np.all(np.diff(np.abs(b)) <= 1e-10 * np.abs(b).max())
    for z in lam[np.abs(lam.imag) > 1e-8]:
        assert np.abs(dmd.eigvals.numpy() - z.conj()).min() <= 1e-10
    # modes and amplitudes depend on the eigenvector scaling, their product does not
    got = (dmd.modes.numpy().astype(np.complex128) * dmd.amplitude.numpy())
    want = phi * b
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()        # fp32 modes
    # continuous-time quantities
    assert np.allclose(dmd.frequency.numpy(), np.angle(lam) / (2 * np.pi * dt), rtol=1e-10, atol=1e-10)
    assert np.allclose(dmd.growth_rate.numpy(), np.log(np.abs(lam)) / dt, rtol=1e-10, atol=1e-10)
    assert np.allclose(dmd.dynamics.numpy()[:, 5], dmd.amplitude.numpy() * dmd.eigvals.numpy() ** 5, rtol=1e-10)


@pytest.mark.parametrize("d,rank", [(None, 6), (3, 20)])
def test_torch_oracle_matches_the_numpy_oracle(d, rank):
    """The fp64 torch port (QR of the weighted X1, the reference of the GPU tests at production sizes) against the
    numpy oracle (SVD of the weighted X1), rank beyond the six signal pairs included, ``block`` smaller than M."""
    a, area, _ = _oscillations(400, 60, d, noise=1e-3, seed=4)
    lam, b, phi, s = dmd_oracle.compute_dmd(a, area, rank)
    lam_t, b_t, phi_t, s_t = dmd_oracle.compute_dmd_torch(pt.from_numpy(a), pt.from_numpy(area), rank, block=128)
    assert tuple(phi_t.shape) == phi.shape and phi_t.dtype == pt.complex128
    assert np.abs(s_t.numpy() - s[:rank]).max() <= 1e-12 * s[0]
    assert np.abs(lam_t.numpy() - lam).max() <= 1e-9
    got = phi_t.numpy() * b_t.numpy()
    want = phi * b
    assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()


def test_n_modes_and_rank_clamps(host, caplog):
    from sparsespatialsampling_b200.dmd import compute_dmd
    a, area, dt = _oscillations(200, 12, seed=2)
    a = a + 1e-3 * np.random.default_rng(0).standard_normal(a.shape).astype(np.float32)
    dmd = compute_dmd(pt.from_numpy(a), pt.from_numpy(area), dt, rank=50, n_modes=3, device="cpu")
    assert dmd.rank == 11 and dmd.n_modes == 3 and tuple(dmd.modes.shape) == (200, 3)    # rank <= T - 1
    with caplog.at_level("WARNING"):
        dmd = compute_dmd(pt.from_numpy(a), pt.from_numpy(area), dt, rank=4, n_modes=9, device="cpu")
    assert dmd.n_modes == 4 and "only 4 modes" in caplog.text


def test_input_checks(host):
    from sparsespatialsampling_b200.dmd import compute_dmd
    a, area, dt = _oscillations(50, 10, seed=3)
    a, area = pt.from_numpy(a), pt.from_numpy(area)
    with pytest.raises(ValueError, match="at least 2 snapshots"):
        compute_dmd(a[:, :1], area, dt, device="cpu")
    for bad in (0.0, -1.0):
        with pytest.raises(ValueError, match="dt must be positive"):
            compute_dmd(a, area, bad, device="cpu")
    with pytest.raises(ValueError, match="cell_area"):
        compute_dmd(a, area[:5], dt, device="cpu")
    with pytest.raises(ValueError, match="Gram method"):
        compute_dmd(a, area, dt, method="lapack", device="cpu")
    with pytest.raises(ValueError, match="N_cells"):
        compute_dmd(a[:, 0], area, dt, device="cpu")


def test_time_step_from_write_times():
    from sparsespatialsampling_b200.utils import uniform_time_step
    assert abs(uniform_time_step(["0.3", "0.1", "0.2", "0.4"]) - 0.1) <= 1e-15
    assert abs(uniform_time_step([1e-3 * i for i in range(1000)]) - 1e-3) <= 1e-12
    with pytest.raises(ValueError, match="uniformly"):
        uniform_time_step(["0.1", "0.2", "0.4"])
    with pytest.raises(ValueError, match="at least 2"):
        uniform_time_step(["0.1"])


def test_lowrank_error_refuses_mismatched_inputs():
    """Checks that run before the kernel is reached: wrong lengths would make it read past the end of a buffer."""
    from sparsespatialsampling_b200 import svd
    m, t, q = 12, 5, 3
    a, left, right_t = pt.zeros((m, t)), pt.zeros((m, q)), pt.zeros((t, q))
    with pytest.raises(ValueError, match="`mean` has 11 entries"):
        svd.lowrank_error(a, left, right_t, mean=pt.zeros(m - 1))
    with pytest.raises(ValueError, match="`vol` has 12 entries for 6 cells"):
        svd.lowrank_error(a, left, right_t, vol=pt.zeros(m), vol_div=2)
    with pytest.raises(ValueError, match="multiple of vol_div"):
        svd.lowrank_error(a, left, right_t, vol_div=5)
    with pytest.raises(ValueError, match="do not fit"):
        svd.lowrank_error(a, left[:, :2], right_t)
    with pytest.raises(ValueError, match="float32"):
        svd.lowrank_error(a, left.double(), right_t)
    with pytest.raises(ValueError, match="one entry per row"):
        svd.lowrank_error(a, left, right_t, row_sq_err=pt.zeros(m - 1, dtype=pt.float64))
    with pytest.raises(ValueError, match="CUDA tensor"):
        svd.lowrank_error(a, left, right_t)

"""Weighted SVD kernels at the sizes where their chunked and long-axis paths switch on, against fp64 references computed
with torch on the same GPU.

gram_tc / project_tc cut the matrix into TF32 planes of at most 2 GB (`plane_rows` rows); every later chunk adds into the
result. Tuning key 17 caps `plane_rows`, so that the chunk boundaries -- exact, ragged, inside the three components of a
vector field -- are reached at small sizes; one case (300 000 x 2000) chunks without it. Long snapshot axes (T up to the
16 384 the Gram entry point accepts) and the fp32 K-splits of the CUDA-core Gram kernel at C5 size are checked as well.
"""
import pytest
import torch as pt

pytestmark = pytest.mark.gpu

# tolerances of tests/test_svd_gpu.py::test_gram_matches_fp64, relative to sqrt(G_ii G_jj)
GRAM_TOL = {"simt": 2e-5, "tc3": 5e-6, "tc": 3e-3}
BLOCK = 65536                    # rows per block of the fp64 references


def _field(m, t, seed, n_modes=5, noise=1e-3):
    """[m, t] fp32 on the device: a few well separated coherent modes, small noise and a large row mean."""
    g = pt.Generator(device="cuda").manual_seed(seed)
    time = pt.linspace(0, 2 * pt.pi, t + 1, device="cuda", dtype=pt.float64)[:-1]
    amp = 2.0 ** -pt.arange(n_modes, device="cuda", dtype=pt.float64)
    phase = pt.rand((n_modes, 1), device="cuda", generator=g, dtype=pt.float64)
    temporal = (amp[:, None] * pt.cos(pt.arange(1, n_modes + 1, device="cuda")[:, None] * time[None, :] + phase)).float()
    a = pt.randn((m, t), device="cuda", generator=g).mul_(noise)          # in place: 4M x 256 is 4 GB
    a.addmm_(pt.randn((m, n_modes), device="cuda", generator=g), temporal)
    a.add_(pt.randn((m, 1), device="cuda", generator=g)).add_(3.0)
    return a


def _vol(n, seed):
    g = pt.Generator(device="cuda").manual_seed(seed + 1)
    return 2.0 ** -pt.randint(8, 16, (n,), device="cuda", generator=g).float()


def _centred_block(a, mean, vol, vol_div, r0, r1):
    """fp64 rows r0..r1 of B = sqrt(vol) (A - mean), the mean rounded to fp32 as the kernels use it."""
    rows = pt.arange(r0, r1, device=a.device) // vol_div
    return (a[r0:r1] - mean[r0:r1, None]).double() * vol[rows].double().sqrt()[:, None]


def _gram_ref(a, mean, vol, vol_div):
    t = a.size(1)
    g = pt.zeros((t, t), dtype=pt.float64, device=a.device)
    for r0 in range(0, a.size(0), BLOCK):
        b = _centred_block(a, mean, vol, vol_div, r0, min(r0 + BLOCK, a.size(0)))
        g += b.T @ b
    return g


def _gram_err(g, ref):
    """max_ij |G - G_ref| / sqrt(G_ref_ii G_ref_jj), row block by row block (T = 16 384 is 2 GB per matrix)."""
    d = pt.diag(ref).sqrt()
    err = 0.0
    for r0 in range(0, g.size(0), 2048):
        blk = (g[r0:r0 + 2048] - ref[r0:r0 + 2048]).abs() / (d[r0:r0 + 2048, None] * d[None, :]).clamp_min(1e-300)
        err = max(err, float(blk.max()))
    return err


def _tune(key, value):
    from sparsespatialsampling_b200 import _lib
    _lib.tune(key, value)


def _restore():
    _tune(17, 0)
    _tune(14, 1)
    _tune(10, 8)
    _tune(11, 128)


@pytest.mark.parametrize("vol_div", [1, 3])
@pytest.mark.parametrize("method", ["tc3", "tc", "tc3-single-cta", "tc-single-cta"])
@pytest.mark.parametrize("cap,ms", [(16, (624, 633)), (48, (1200, 1221)), (4096, (12288, 13287, 3000))])
def test_chunked_gram_matches_fp64(cuda, cap, ms, method, vol_div):
    """Planes of `cap` rows: chunks that divide m, a ragged last chunk, m below the cap. Caps 16 and 4096 are not
    multiples of 3, so the components of a D = 3 field straddle chunk boundaries."""
    from sparsespatialsampling_b200 import svd
    name = method.split("-")[0]
    try:
        _tune(17, cap)
        _tune(14, 0 if method.endswith("single-cta") else 1)
        for m in ms:
            a = _field(m, 300, m + cap)
            vol = _vol(m // vol_div, m)
            mean = svd.row_means(a)
            ref = _gram_ref(a, mean, vol, vol_div)
            g = svd.gram(a, mean, vol, vol_div, name)
            assert pt.equal(g, g.T)
            err = _gram_err(g, ref)
            assert err <= GRAM_TOL[name], (m, err)
    finally:
        _restore()


@pytest.mark.parametrize("cap,m,vol_div", [(128, 946, 1), (384, 1997, 1), (128, 1002, 3)])
@pytest.mark.parametrize("r", [1, 50, 256, 257, 300])
def test_chunked_projection_matches_fp64(cuda, cap, m, vol_div, r):
    from sparsespatialsampling_b200 import svd
    g = pt.Generator(device="cuda").manual_seed(r)
    a = _field(m, 200, m + r)
    vol = _vol(m // vol_div, r)
    w = pt.randn((200, r), device="cuda", generator=g)
    mean = svd.row_means(a)
    ref = (a - mean[:, None]).double() @ w.double()
    scale = float(ref.abs().max())
    try:
        _tune(17, cap)
        u3 = svd.project_tc(a, mean, vol, vol_div, w, "tc3")
        u1 = svd.project_tc(a, mean, vol, vol_div, w, "tc")
    finally:
        _restore()
    assert float((u3.double() - ref).abs().max()) <= 2e-5 * scale
    assert float((u1.double() - ref).abs().max()) <= 5e-3 * scale


def test_c5_sized_matrix_chunks_without_the_hook(cuda):
    """300 000 x 2000: t_pad = 2048, so the 2 GB planes hold 262 144 rows and both kernels run two chunks."""
    from sparsespatialsampling_b200 import svd
    m, t = 300_000, 2000
    a = _field(m, t, 7)
    vol = _vol(m, 7)
    mean = svd.row_means(a)
    ref = _gram_ref(a, mean, vol, 1)
    assert _gram_err(svd.gram(a, mean, vol, 1, "tc3"), ref) <= GRAM_TOL["tc3"]
    lam, vec = pt.linalg.eigh(ref)
    lam, vec = lam.flip(0).clamp_min(0), vec.flip(1)
    s_ref = lam.sqrt()
    s, u, v = svd.compute_svd(a, vol, rank=50)
    n_sig = 5                                            # the coherent modes of _field; the rest is the noise floor
    assert float(((s[:n_sig].double() - s_ref[:n_sig]).abs() / s_ref[:n_sig]).max()) <= 1e-4
    cos_v = (v[:, :n_sig].double() * vec[:, :n_sig]).sum(0).abs()
    assert float(cos_v.min()) >= 1 - 1e-4
    uw = pt.zeros((n_sig, n_sig), dtype=pt.float64, device="cuda")
    cross = pt.zeros(n_sig, dtype=pt.float64, device="cuda")
    for r0 in range(0, m, BLOCK):
        r1 = min(r0 + BLOCK, m)
        b = _centred_block(a, mean, vol, 1, r0, r1)
        u_ref = b @ (vec[:, :n_sig] / s_ref[:n_sig])                  # weighted reference modes, unit norm
        u_w = u[r0:r1, :n_sig].double() * vol[r0:r1].double().sqrt()[:, None]
        uw += u_w.T @ u_w
        cross += (u_w * u_ref).sum(0)
    assert float((uw - pt.eye(n_sig, dtype=pt.float64, device="cuda")).abs().max()) <= 1e-3
    assert float((cross.abs() / pt.diag(uw).sqrt()).min()) >= 1 - 1e-4


@pytest.mark.parametrize("t,m", [(1000, 3000), (2000, 2000), (2048, 2000), (2049, 1500), (4096, 1000), (16384, 600)])
def test_gram_long_snapshot_axis(cuda, t, m):
    from sparsespatialsampling_b200 import svd
    a = _field(m, t, t)
    vol = _vol(m, t)
    mean = svd.row_means(a)
    ref = _gram_ref(a, mean, vol, 1)
    g = svd.gram(a, mean, vol, 1, "tc3")
    assert _gram_err(g, ref) <= GRAM_TOL["tc3"]


def test_gram_rejects_too_many_snapshots(cuda):
    from sparsespatialsampling_b200 import svd, _lib
    a = pt.ones((2, 16385), device="cuda")
    mean = svd.row_means(a)
    with pytest.raises(_lib.S3Error, match="too many snapshots"):
        svd.gram(a, mean, pt.ones(2, device="cuda"), 1, "tc3")


@pytest.mark.parametrize("r", [32, 256])
@pytest.mark.parametrize("t", [2000, 8192, 16384])
def test_projection_long_snapshot_axis(cuda, t, r):
    """The tensor core truncates its fp32 accumulation, so project_tc bounds the chain per TMEM segment to 32 column
    groups (384 MMAs) and runs longer t ranges as launches that add into U. With one launch for the whole range
    (2 segments at r = 256) the error at T = 8192 / 16 384 was 3.2e-5 / 5.1e-5 of the largest entry (B200, 1000 W);
    with the split launches it is <= 8.3e-6 at every size here."""
    from sparsespatialsampling_b200 import svd
    m = 2000
    g = pt.Generator(device="cuda").manual_seed(t + r)
    a = pt.randn((m, t), device="cuda", generator=g) + 3.0
    vol = pt.rand((m,), device="cuda", generator=g) + 0.5
    w = pt.randn((t, r), device="cuda", generator=g)
    mean = svd.row_means(a)
    ref = (a - mean[:, None]).double() @ w.double()
    u = svd.project_tc(a, mean, vol, 1, w, "tc3")
    err = float((u.double() - ref).abs().max()) / float(ref.abs().max())
    assert err <= 2e-5, err


def test_gram_flushes_at_default_knobs(cuda):
    """4M x 256: one K-split covers ~220 TMEM segments, i.e. two fp64 flushes of 128 segments, in each of two chunks."""
    from sparsespatialsampling_b200 import svd
    m = 4 * 1024 * 1024
    a = _field(m, 256, 4)
    vol = _vol(m, 4)
    mean = svd.row_means(a)
    ref = _gram_ref(a, mean, vol, 1)
    assert _gram_err(svd.gram(a, mean, vol, 1, "tc3"), ref) <= GRAM_TOL["tc3"]


def test_simt_gram_at_c5_size(cuda):
    """The CUDA-core Gram kernel sums each of its K-splits in fp32 before the fp64 reduce. In 5 splits of 120 000 rows
    (the split count that fills the GPU) the error here was 5.8e-5; with splits of at most 8192 rows it is 1.5e-6
    (B200, 1000 W)."""
    from sparsespatialsampling_b200 import svd
    m, t = 600_000, 2000
    a = _field(m, t, 5)
    vol = _vol(m, 5)
    mean = svd.row_means(a)
    ref = _gram_ref(a, mean, vol, 1)
    err = _gram_err(svd.gram(a, mean, vol, 1, "simt"), ref)
    assert err <= GRAM_TOL["simt"], err

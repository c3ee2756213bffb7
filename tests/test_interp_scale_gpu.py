"""s3_interp_gather at production sizes against an fp64 reference computed with torch on the same GPU.

The suite's other interpolation tests use a few thousand cells, so the persistent part-warp kernel never starts a second
sweep there and most kernels are compared with each other only. Here the tables are real KnnTables on synthetic clouds
(Morton processing order, neighbouring cells sharing source rows) at the sizes of the time windows of a sharded export,
the part-warp kernel is driven through its sweep boundaries with a CTA cap (tuning key 15), and every result is compared
with the reference:
  fp32 result: |out - ref| <= 1e-5 * max_j |data[idx[c, j]]| for every element (the criterion of test_interp_gpu.py);
  fp64 result: bit-exact against fp64 products added one neighbour after the other (MODE 1, the reference's order).
"""
import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc

pytestmark = pytest.mark.gpu

RTOL_F32 = 1e-5
CHUNK = 8192                         # cells per block of the reference
SENTINEL = float("nan")
# defaults of the launch knobs these tests set (csrc/interp.cu)
KNOBS = {1: 8, 7: 0, 8: -1, 12: 0, 13: 0, 15: 0}


def _restore():
    from sparsespatialsampling_b200 import _lib
    for key, value in KNOBS.items():
        _lib.tune(key, value)


def _tune(spec):
    from sparsespatialsampling_b200 import _lib
    for kv in [s for s in spec.split(",") if s]:
        key, value = kv.split("=")
        _lib.tune(int(key), int(value))


def _ref_blocks(data, idx, w64):
    """(c0, c1, ref, scale) per block of cells: ref = sum_j w64[c, j] * data[idx[c, j]] with fp64 products added in
    neighbour order, scale = max_j |data[idx[c, j]]|."""
    idx = idx.long()
    for c0 in range(0, idx.size(0), CHUNK):
        c1 = min(c0 + CHUNK, idx.size(0))
        acc, scale = None, None
        for j in range(idx.size(1)):
            x = data[idx[c0:c1, j]]
            prod = w64[c0:c1, j].reshape((-1,) + (1,) * (x.dim() - 1)) * x.double()
            acc = prod if acc is None else acc + prod
            scale = x.abs() if scale is None else pt.maximum(scale, x.abs())
        yield c0, c1, acc, scale.double()


def _check(out, data, idx, w64, exact=False):
    """out (reference cell order) against the fp64 reference; fp32: the tolerance above, fp64: same bits."""
    for c0, c1, ref, scale in _ref_blocks(data, idx, w64):
        got = out[c0:c1]
        if exact:
            assert got.dtype == pt.float64 and pt.equal(got, ref), c0
        else:
            err = (got.double() - ref).abs()
            bad = ~(err <= RTOL_F32 * scale.clamp_min(1e-30))          # NaN (cells never written) counts as bad
            assert not bool(bad.any()), (c0, int(bad.sum()), float(pt.nan_to_num(err, nan=pt.inf).max()))


def _field(n, d, t, seed):
    """[n, d, t] fp32 on the device: a large per-point mean plus a unit fluctuation."""
    g = pt.Generator(device="cuda").manual_seed(seed)
    return 100.0 + 10.0 * pt.randn((n, 1, 1), device="cuda", generator=g) + pt.randn((n, d, t), device="cuda", generator=g)


def _pitched(x):
    from sparsespatialsampling_b200.interpolate import to_pitched
    return to_pitched(x)


def _fresh_pitched(nc, d, t, dtype=pt.float32):
    """Pitched result filled with the sentinel, padding included."""
    from sparsespatialsampling_b200.interpolate import alloc_snapshots
    out = alloc_snapshots(nc, d, t, dtype=dtype, device="cuda")
    out._base.fill_(SENTINEL)
    return out


def _padding_untouched(out, t):
    pad = out._base[..., t:]
    return pad.numel() == 0 or bool(pad.isnan().all())


class _Tables:
    def __init__(self, dim, n_points, n_cells, ks, seed):
        from sparsespatialsampling_b200.export import KnnTables
        from sparsespatialsampling_b200.knn import KnnIndex
        g = pt.Generator(device="cuda").manual_seed(seed)
        x = pt.rand((n_points, dim), device="cuda", generator=g, dtype=pt.float64)
        q = pt.rand((n_cells, dim), device="cuda", generator=g, dtype=pt.float64)
        index = KnnIndex(x)
        self.n_points = n_points
        self.by_k = {k: KnnTables(index, q, k) for k in ks}


@pytest.fixture(scope="module")
def c2_tables(cuda):
    """2-D: ~100k points, ~60k cells (a C2-sized export)."""
    return _Tables(2, 100_000, 60_000, (1, 8, 16), 2)


@pytest.fixture(scope="module")
def c4_tables(cuda):
    """3-D: ~200k points, ~30k cells, k = 26."""
    return _Tables(3, 200_000, 30_000, (26,), 3)


def test_reference_matches_the_oracle(c2_tables):
    """The GPU reference of this file against oracle.s3_oracle.interpolate on a random sample of cells: same bits."""
    tab = c2_tables.by_k[8]
    data = _field(c2_tables.n_points, 2, 125, 11)
    sample = pt.randperm(tab.n, generator=pt.Generator().manual_seed(1))[:200].cuda()
    idx, w64 = tab.idx[sample], tab.w64[sample]
    (_, _, ref, _), = list(_ref_blocks(data, idx, w64))
    want = orc.interpolate(w64.cpu().numpy(), idx.long().cpu().numpy(), data.cpu().numpy())
    assert np.array_equal(ref.cpu().numpy(), want)


@pytest.mark.parametrize("t", [125, 250, 500])
@pytest.mark.parametrize("d", [1, 2])
def test_c2_windows(c2_tables, d, t):
    """Time windows of a sharded C2 export (k = 8: the part-warp kernel, 8-12 sweeps at the default launch) on a pitched
    source; pitched result (32-byte aligned rows: 256-bit stores, padding untouched) and dense result, whose rows are
    16 / 8 / 4-byte aligned for T = 500 / 250 / 125 -- and the fp64 result."""
    tab = c2_tables.by_k[8]
    src = _pitched(_field(c2_tables.n_points, d, t, d * t))
    out = _fresh_pitched(tab.n, d, t)
    tab.interpolate(src, pt.float32, out=out)
    _check(out, src, tab.idx, tab.w64)
    assert _padding_untouched(out, t)
    dense = pt.full((tab.n, d, t), SENTINEL, device="cuda")
    tab.interpolate(src, pt.float32, out=dense)
    assert pt.equal(dense, out)
    out64 = pt.full((tab.n, d, t), SENTINEL, dtype=pt.float64, device="cuda")
    tab.interpolate(src, pt.float64, out=out64)
    _check(out64, src, tab.idx, tab.w64, exact=True)


@pytest.mark.parametrize("t", [64, 125, 250])
def test_c4_windows(c4_tables, t):
    """3-D windows: k = 26, D = 3 (the component loop of the part-warp kernel)."""
    tab = c4_tables.by_k[26]
    src = _pitched(_field(c4_tables.n_points, 3, t, t))
    out = _fresh_pitched(tab.n, 3, t)
    tab.interpolate(src, pt.float32, out=out)
    _check(out, src, tab.idx, tab.w64)
    assert _padding_untouched(out, t)
    out64 = pt.full((tab.n, 3, t), SENTINEL, dtype=pt.float64, device="cuda")
    tab.interpolate(src, pt.float64, out=out64)
    _check(out64, src, tab.idx, tab.w64, exact=True)


def _local_tables(n_src, n_cells, k, seed):
    """Tables like tests/test_interp_gpu.py::_local_case: cells in order share neighbours (a sliding window of 3k
    source rows), k distinct neighbours per cell, weights summing to one."""
    rng = np.random.default_rng(seed)
    base = np.sort(rng.integers(0, max(n_src - 3 * k, 1), n_cells))
    idx = np.stack([rng.permutation(3 * k)[:k] + b for b in base]).astype(np.int32)
    w = rng.random((n_cells, k))
    w /= w.sum(1, keepdims=True)
    return pt.from_numpy(idx).cuda(), pt.from_numpy(w).cuda()


@pytest.mark.parametrize("t", [100, 250])
@pytest.mark.parametrize("k", [33, 40, 64])
def test_many_neighbours(cuda, k, t):
    """k > 32: whole-warp cells with two table registers per lane (KR = 2) in the part-warp kernel, and fp32 with
    k > 32 on the warp-per-cell kernel."""
    from sparsespatialsampling_b200.interpolate import interp_gather
    idx, w64 = _local_tables(40_000, 20_000, k, k + t)
    src = _pitched(_field(40_000, 2, t, k * t))
    try:
        for spec in ("", "8=0"):
            _restore()
            _tune(spec)
            out = _fresh_pitched(idx.size(0), 2, t)
            interp_gather(src, idx, w64.float(), out=out)
            _check(out, src, idx, w64)
            assert _padding_untouched(out, t), spec
    finally:
        _restore()
    out64 = interp_gather(src, idx, w64, out_dtype=pt.float64)
    _check(out64, src, idx, w64, exact=True)


@pytest.mark.parametrize("t", [132, 500, 1004])
@pytest.mark.parametrize("k", [1, 8, 16])
def test_dense_kernel(c2_tables, k, t):
    """Dense fp32 rows that are 16- but not 32-byte aligned (T % 8 == 4): interp_dense_kernel."""
    tab = c2_tables.by_k[k]
    src = _field(c2_tables.n_points, 1, t, k + t)
    out = pt.full((tab.n, 1, t), SENTINEL, device="cuda")
    tab.interpolate(src, pt.float32, out=out)
    _check(out, src, tab.idx, tab.w64)


@pytest.mark.parametrize("t", [125, 250])
@pytest.mark.parametrize("d", [1, 2])
def test_scalar_path_on_the_reference_layout(c2_tables, d, t):
    """The reference's dense [N, D, T] layout with T % 4 != 0: one column per lane."""
    tab = c2_tables.by_k[8]
    src = _field(c2_tables.n_points, d, t, 7 * t + d)
    out = pt.full((tab.n, d, t), SENTINEL, device="cuda")
    tab.interpolate(src, pt.float32, out=out)
    _check(out, src, tab.idx, tab.w64)


def test_long_rows_wide_kernel(c2_tables):
    """T = 1000 on pitched rows: the 256-bit warp-per-cell kernel (contrast to the short windows)."""
    tab = c2_tables.by_k[8]
    src = _pitched(_field(c2_tables.n_points, 2, 1000, 1000))
    out = _fresh_pitched(tab.n, 2, 1000)
    tab.interpolate(src, pt.float32, out=out)
    _check(out, src, tab.idx, tab.w64)
    assert _padding_untouched(out, 1000)


# part-warp instantiations (csrc/interp.cu, launch_interp): lanes per cell (key 13) x table registers per lane (k) x
# load batch / resident CTAs per SM (KU 4 at 3 or 4 CTAs by key 12, KU 8 by key 7)
_PARTWARP = [(lpc, k, extra) for lpc, ks in ((16, (8, 26)), (32, (8, 40))) for k in ks
             for extra in ("12=3", "12=4", "7=8")]


@pytest.mark.parametrize("lpc,k,extra", _PARTWARP)
def test_partwarp_sweep_edges(cuda, lpc, k, extra):
    """With the part-warp kernel capped at 1, 2 and 3 CTAs (P part-warps), cell counts 3P - 1, 3P and 3P + 1: every
    part-warp takes three or four sweeps, the last one partial, and hands the (index, weight) pairs it fetched ahead over
    the sweep boundary. Against the reference and bit-identical to the warp-per-cell kernel."""
    from sparsespatialsampling_b200.interpolate import interp_gather
    t, d = 100, 2
    warps = 8
    idx_all, w_all = _local_tables(4000, 3 * 3 * warps * (32 // lpc) + 1, k, k + lpc)
    src = _pitched(_field(4000, d, t, k * lpc))
    try:
        for cap in (1, 2, 3):
            p = cap * warps * (32 // lpc)
            for n in (3 * p - 1, 3 * p, 3 * p + 1):
                idx, w64 = idx_all[:n].contiguous(), w_all[:n].contiguous()
                _restore()
                _tune("8=0")
                want = interp_gather(src, idx, w64.float())
                _tune(f"8=1,13={lpc},15={cap},{extra}")
                out = _fresh_pitched(n, d, t)
                interp_gather(src, idx, w64.float(), out=out)
                assert pt.equal(out, want), (cap, n)
                assert _padding_untouched(out, t), (cap, n)
                _check(out, src, idx, w64)
    finally:
        _restore()


@pytest.mark.parametrize("t", [250, 1000])
def test_host_path_against_fp64(c2_tables, t):
    """KnnTables.interpolate_host on a C2-sized pinned batch: one dense window (T = 250) and four pitched windows
    (T = 1000), rows staged by DMA and by the PCIe gather."""
    tab = c2_tables.by_k[8]
    dev_data = _field(c2_tables.n_points, 2, t, t + 1)
    host = dev_data.cpu().pin_memory()
    for gather in (False, True):
        out = pt.full((tab.n, 2, t), SENTINEL, pin_memory=True)
        tab.interpolate_host(host, out=out, gather=gather)
        _check(out.cuda(), dev_data, tab.idx, tab.w64)

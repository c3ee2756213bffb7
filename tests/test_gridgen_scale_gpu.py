"""Grid generation's KNN, gain and reduction kernels past their size thresholds, bit-exact against the CPU oracle.

The KNN index is a 32-ary box tree over 32-point leaves: up to 32^4 = 1 048 576 points it has 4 levels, one point more
gives it a 5th (32 769 -> 1 025 -> 33 -> 2 -> 1 nodes). The other KNN tests stay below 200k points, so the 5-level
search -- the index every 3-D production cloud uses -- is compared with the oracle only here:
  * kneighbors / predict / tables on random, clustered, lattice and degenerate clouds on both sides of the threshold,
    k = 1, 8, 26 and 32, with queries inside the cloud, on its bounding box, far outside and on cloud points;
  * lattice clouds with power-of-two spacing, where the k-th neighbour sits in a shell of exactly equidistant points:
    the tie-break (smaller original index) must survive pruning and the stack, and predict depends on it;
  * everything once more on the Morton curve (tuning key 30): the curve only changes the point order of the index;
  * s3_morton_order at 3M points (733 radix-sort tiles) against a numpy port of the curve key: sorted and stable;
  * s3_cells_gain (the refinement driver) against OracleTree._update_gain on 5-level indexes;
  * s3_sumsq / s3_leaf_sumsq past 256 block partials (10M elements).
One oracle search with k = 32 per cloud serves every k: its rows are ordered by (distance, index), so the first k
columns are the k-nearest result.
"""
import functools

import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc

pytestmark = pytest.mark.gpu

KS = (1, 8, 26, 32)
N4 = 32 ** 4                            # largest cloud with a 4-level index
H2 = 2.0 ** -10                         # lattice spacings: every coordinate and distance below is exact
H3 = 2.0 ** -7


@pytest.fixture(params=["hilbert", "morton"])
def curve(request, cuda):
    from sparsespatialsampling_b200 import _lib
    _lib.tune(30, 1 if request.param == "hilbert" else 0)
    yield request.param
    _lib.tune(30, 1)


def _lattice(shape, h, seed):
    grid = np.stack(np.meshgrid(*[np.arange(s) for s in shape], indexing="ij"), -1).reshape(-1, len(shape))
    X = grid.astype(np.float64) * h + 0.5
    return X[np.random.default_rng(seed).permutation(X.shape[0])]


def _cloud(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name in ("rand2_4", "rand2_5", "rand3_4", "rand3_5"):
        return rng.random((N4 + (name[-1] == "5"), int(name[4])))
    if name == "clustered3":                                   # anisotropic, CFD-like clustering towards a wall
        X = rng.random((1_300_000, 3))
        X[:, 1] = X[:, 1] ** 3 * 0.41
        X[:, 0] *= 2.2
        return X
    if name == "lattice2":
        return _lattice((1100, 1000), H2, 1)
    if name == "lattice3":
        return _lattice((104, 104, 104), H3, 2)
    if name == "flat3":                                        # zero bounding-box extent in z
        X = rng.random((N4 + 5000, 3))
        X[:, 2] = 0.375
        return X
    if name == "line3":                                        # evenly spaced on a line: ties between line points
        t = rng.permutation(N4 + 1).astype(np.float64) * 2.0 ** -20
        return np.stack([t, 0.5 * t, 0.25 * t], 1) + np.array([0.25, -0.5, 1.0])
    if name == "dup4":                                         # every point four times, 5 levels
        base = rng.random(((N4 + 4) // 4, 3))
        return np.tile(base, (4, 1))[rng.permutation(4 * base.shape[0])]
    raise KeyError(name)


def _queries(name, X):
    rng = np.random.default_rng(7 + len(name))
    d = X.shape[1]
    lo, hi = X.min(0), X.max(0)
    ext = np.where(hi > lo, hi - lo, 1.0)
    parts = [lo + rng.random((1000, d)) * (hi - lo),                           # inside
             X[rng.integers(0, X.shape[0], 100)]]                              # exact hits
    box = lo + rng.random((150, d)) * (hi - lo)                                # on the bounding box
    axis = rng.integers(0, d, 150)
    box[np.arange(150), axis] = np.where(rng.random(150) < 0.5, lo[axis], hi[axis])
    parts += [box, lo + (rng.random((100, d)) * 6.0 - 2.5) * ext]              # far outside
    if name.startswith("lattice"):
        h = H2 if d == 2 else H3
        shape = np.array([1100, 1000]) if d == 2 else np.array([104] * 3)
        cell = rng.integers(0, shape, (300, d)).astype(np.float64)
        cell[:30] = np.where(rng.random((30, d)) < 0.5, 0.0, shape - 1)        # lattice corners and faces
        parts.append(cell * h + 0.5)                                           # lattice points
        parts.append((cell + 0.5) * h + 0.5)                                   # cell midpoints (2^d / 3-D: 8 + 24 shell)
        parts.append((cell + rng.choice([0.25, 0.75], (300, d))) * h + 0.5)    # dyadic child centres
    if name in ("flat3", "line3"):
        near = X[rng.integers(0, X.shape[0], 200)] + rng.choice([-1.0, 0.0, 1.0], (200, d)) * 2.0 ** -21
        parts.append(near)                                                     # next to and between line / plane points
    return np.ascontiguousarray(np.concatenate(parts))


@functools.lru_cache(maxsize=None)
def _case(name):
    """(cloud, queries, values, oracle distances and indices for k = 32) of one named cloud, computed once per session."""
    X = _cloud(name)
    Q = _queries(name, X)
    y = np.random.default_rng(3).random(X.shape[0]) * 4.0 - 1.0
    d, i = orc.knn_search(X, Q, 32)
    return X, Q, y, d, i


CLOUDS = ["rand2_4", "rand2_5", "rand3_4", "rand3_5", "clustered3", "lattice2", "lattice3", "flat3", "line3", "dup4"]


@pytest.mark.parametrize("name", CLOUDS)
def test_knn_bit_exact_at_five_levels(cuda, curve, name):
    from sparsespatialsampling_b200.knn import KnnIndex
    X, Q, y, d_ref, i_ref = _case(name)
    index = KnnIndex(pt.from_numpy(X), pt.from_numpy(y))
    q = pt.from_numpy(Q)
    for k in KS:
        dist, idx = index.kneighbors(q, k)
        assert np.array_equal(idx.cpu().numpy(), i_ref[:, :k]), (name, k)
        assert np.array_equal(dist.cpu().numpy(), d_ref[:, :k]), (name, k)
        pred = index.predict(q, k).cpu().numpy()
        assert np.array_equal(pred, orc.idw_predict(d_ref[:, :k], i_ref[:, :k], y)), (name, k)
        t_idx, w32, w64 = index.tables(q, k)
        w_ref = orc.export_weights(d_ref[:, :k])
        assert np.array_equal(t_idx.cpu().numpy().astype(np.int64), i_ref[:, :k]), (name, k)
        if k == 8:
            assert np.array_equal(w64.cpu().numpy(), w_ref), (name, k)
        else:
            np.testing.assert_allclose(w64.cpu().numpy(), w_ref, rtol=1e-14)
        np.testing.assert_allclose(w32.cpu().numpy(), w_ref.astype(np.float32), rtol=2e-7)


def test_lattice_queries_hit_tie_shells(cuda):
    """The lattice queries reach the equidistant shells the tie-break has to resolve (guards the test data itself)."""
    for name, k, shell in (("lattice2", 8, 2 * H2 ** 2), ("lattice3", 26, 3 * H3 ** 2)):
        _, Q, _, d, _ = _case(name)
        kth = d[:, k - 1] ** 2
        # k-th neighbour of a lattice point: the sqrt(2) shell (2-D, 4 points) / the corner shell (3-D, 8 points);
        # k-th of a 3-D cell midpoint: the second shell of 24 points around the 8 nearest
        assert np.sum(np.isclose(kth, shell, rtol=0, atol=1e-18)) >= 100, name
        assert np.sum(d[:, k - 1] == d[:, k]) >= 300, name                   # the k-th and (k+1)-th are tied
    _, _, _, d, _ = _case("lattice3")
    assert np.sum(np.isclose(d[:, 25] ** 2, 11 * H3 ** 2 / 4, rtol=0, atol=1e-18)) >= 100


# ------------------------------------------------------------------------------------------------ curve key + sort
def _spread2(v):
    v = v & np.uint64(0xFFFFFFFF)
    for s, m in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F), (2, 0x3333333333333333),
                 (1, 0x5555555555555555)):
        v = (v | (v << np.uint64(s))) & np.uint64(m)
    return v


def _spread3(v):
    v = v & np.uint64(0x1FFFFF)
    for s, m in ((32, 0x001F00000000FFFF), (16, 0x001F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3),
                 (2, 0x1249249249249249)):
        v = (v | (v << np.uint64(s))) & np.uint64(m)
    return v


def _hilbert_transpose(x, bits):
    """Skilling's axes-to-transpose, vectorised over points (csrc/knn.cu hilbert_transpose)."""
    x = [a.copy() for a in x]
    q = 1 << (bits - 1)
    while q > 1:
        p, qq = np.uint64(q - 1), np.uint64(q)
        for i in range(len(x)):
            hit = (x[i] & qq) != 0
            if i == 0:
                x[0] = np.where(hit, x[0] ^ p, x[0])
            else:
                t = np.where(hit, np.uint64(0), (x[0] ^ x[i]) & p)
                x[0] = np.where(hit, x[0] ^ p, x[0] ^ t)
                x[i] = x[i] ^ t
        q >>= 1
    for i in range(1, len(x)):
        x[i] = x[i] ^ x[i - 1]
    t = np.zeros_like(x[0])
    q = 1 << (bits - 1)
    while q > 1:
        t = np.where((x[-1] & np.uint64(q)) != 0, t ^ np.uint64(q - 1), t)
        q >>= 1
    return [a ^ t for a in x]


def curve_key(X, curve):
    """numpy port of csrc/knn.cu morton_kernel: quantised bounding-box position, Morton or Hilbert key."""
    d = X.shape[1]
    bits = 31 if d == 2 else 21
    lo, hi = X.min(0), X.max(0)
    q = []
    for a in range(d):
        ext = hi[a] - lo[a]
        u = (X[:, a] - lo[a]) / ext if ext > 0.0 else np.zeros(X.shape[0])
        f = u * float(1 << bits)
        c = np.where(f <= 0.0, 0.0, f)
        c = np.minimum(c.astype(np.uint64), np.uint64((1 << bits) - 1))
        q.append(c)
    if curve == "hilbert":
        q = _hilbert_transpose(q, bits)
        if d == 2:
            return (_spread2(q[0]) << np.uint64(1)) | _spread2(q[1])
        return (_spread3(q[0]) << np.uint64(2)) | (_spread3(q[1]) << np.uint64(1)) | _spread3(q[2])
    if d == 2:
        return _spread2(q[0]) | (_spread2(q[1]) << np.uint64(1))
    return _spread3(q[0]) | (_spread3(q[1]) << np.uint64(1)) | (_spread3(q[2]) << np.uint64(2))


@pytest.mark.parametrize("dim", [2, 3])
def test_morton_order_is_a_stable_sort_of_the_curve_key(cuda, curve, dim):
    from sparsespatialsampling_b200 import _lib
    rng = np.random.default_rng(dim)
    n = 3_000_000                                               # 733 tiles of the radix sort
    base = rng.random((900_000, dim))
    base[:1000] = np.round(base[:1000] * 64) / 64              # exact values on the quantisation grid
    X = base[rng.integers(0, base.shape[0], n)]                # ~2.2 copies of every point: equal keys everywhere
    X[:5] = base.min(0) - 1.0                                  # bounding-box corners: the clamp at 0 and 2^bits - 1
    X[5:10] = base.max(0) + 1.0
    key = curve_key(X, curve)
    want = np.lexsort((np.arange(n), key))
    perm = pt.empty(n, dtype=pt.int32, device="cuda")
    lib = _lib.load()
    x = pt.from_numpy(X).cuda()
    _lib.check(lib.s3_morton_order(_lib.ptr(x), n, dim, _lib.ptr(perm), _lib.stream_ptr()))
    assert np.array_equal(perm.cpu().numpy().astype(np.int64), want)


# ------------------------------------------------------------------------------------------------ gain
GAIN_CELLS = {2: 240, 3: 150}
WIDTH = 1.0
GAIN0 = 0.0123


@functools.lru_cache(maxsize=None)
def _gain_case(name, k):
    """Cells (centre, level) on cloud `name` and the oracle's metric prediction at each centre and its 2^d children."""
    X, _, y, _, _ = _case(name)
    d = X.shape[1]
    rng = np.random.default_rng(11 * d + k)
    n = GAIN_CELLS[d]
    dirs = orc.DIRS_2D if d == 2 else orc.DIRS_3D
    level = rng.integers(2, 13, n)
    lo, hi = X.min(0), X.max(0)
    center = lo + rng.random((n, d)) * (hi - lo)
    center[:20] = X[rng.integers(0, X.shape[0], 20)]                        # centre on a cloud point
    if name.startswith("lattice"):
        # lattice centres: the children land on lattice points (level <= 8 in 2-D, <= 5 in 3-D) or on dyadic points
        # between them, equidistant from several cloud points
        h = H2 if d == 2 else H3
        shape = np.array([1100, 1000]) if d == 2 else np.array([104] * 3)
        center[20:120] = rng.integers(20, shape - 20, (100, d)) * h + 0.5
    else:
        # a child centre on a cloud point: centre = p - offset, kept where centre + offset gives p back exactly
        for t in range(20, 60):
            p, j = X[rng.integers(0, X.shape[0])], rng.integers(0, 2 ** d)
            off = dirs[j] * 0.25 * WIDTH / (2 ** int(level[t]))
            if np.array_equal((p - off) + off, p):
                center[t] = p - off
    q = np.concatenate([center[:, None, :], center[:, None, :] + dirs[None] * 0.25 * WIDTH / (2.0 ** level)[:, None, None]],
                       axis=1)
    dist, idx = orc.knn_search(X, q.reshape(-1, d), k)
    m = orc.idw_predict(dist, idx, y).reshape(n, 2 ** d + 1)
    zero_rows = int(np.sum(dist[:, 0] == 0.0))
    return center, level, m, zero_rows


@pytest.mark.parametrize("name,k,sdm_order", [("rand2_5", 8, 1), ("lattice2", 8, 1), ("rand3_5", 26, 0),
                                              ("rand3_5", 26, 1), ("lattice3", 26, 0), ("lattice3", 26, 1)])
def test_cells_gain_bit_exact_at_five_levels(cuda, name, k, sdm_order):
    from sparsespatialsampling_b200 import _lib
    from sparsespatialsampling_b200.knn import KnnIndex
    X, _, y, _, _ = _case(name)
    center, level, m, zero_rows = _gain_case(name, k)
    assert zero_rows >= 20                              # the indicator-weight rows of warp_idw_predict are exercised
    d, n = X.shape[1], center.shape[0]
    sdm = orc.sum_delta_metric(m, sdm_order)
    gain_ref = np.array([orc.gain_formula(int(level[t]), d, WIDTH, GAIN0, float(sdm[t])) for t in range(n)])
    metric_ref = m[:, 0]
    index = KnnIndex(pt.from_numpy(X), pt.from_numpy(y))
    lib = _lib.load()
    c_d = pt.from_numpy(center).cuda()
    l_d = pt.from_numpy(level.astype(np.int32)).cuda()
    rng = np.random.default_rng(n)
    cells = rng.permutation(n)[: n - 37]                                     # unsorted, with gaps
    first, count = 13, n - 30                                                # contiguous form
    for sel, args in ((cells, None), (np.arange(first, first + count), (first, count))):
        metric = pt.full((n,), float("nan"), dtype=pt.float64, device="cuda")
        gain = pt.full((n,), float("nan"), dtype=pt.float64, device="cuda")
        if args is None:
            cl = pt.from_numpy(cells.astype(np.int64)).cuda()
            _lib.check(lib.s3_cells_gain(index.handle, _lib.ptr(c_d), _lib.ptr(l_d), _lib.ptr(cl), 0, cl.numel(), k,
                                         WIDTH, GAIN0, sdm_order, _lib.ptr(metric), _lib.ptr(gain), _lib.stream_ptr()))
        else:
            _lib.check(lib.s3_cells_gain(index.handle, _lib.ptr(c_d), _lib.ptr(l_d), None, first, count, k, WIDTH,
                                         GAIN0, sdm_order, _lib.ptr(metric), _lib.ptr(gain), _lib.stream_ptr()))
        metric, gain = metric.cpu().numpy(), gain.cpu().numpy()
        assert np.array_equal(metric[sel], metric_ref[sel])
        assert np.array_equal(gain[sel], gain_ref[sel])
        rest = np.setdiff1d(np.arange(n), sel)
        assert np.isnan(metric[rest]).all() and np.isnan(gain[rest]).all()   # cells outside the call are untouched


# ------------------------------------------------------------------------------------------------ sums of squares
def _sumsq(lib_fn, *args):
    from sparsespatialsampling_b200 import _lib
    out = pt.empty(1, dtype=pt.float64, device="cuda")
    _lib.check(lib_fn(*args, _lib.ptr(out), _lib.stream_ptr()))
    return float(out.item())


@pytest.mark.parametrize("n", [10_000_000, 10_000_000 + 4097])
def test_sums_of_squares_past_256_partials(cuda, n):
    import math
    from sparsespatialsampling_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(n)
    flags = rng.integers(0, 4, n).astype(np.uint8)                 # bit 0 = leaf; the other bits must be ignored
    leaf = (flags & 1).astype(bool)
    f_d = pt.from_numpy(flags).cuda()
    # squares are small integers: every partial sum is an exact integer below 2^53 in any order
    xi = rng.integers(-3, 4, n).astype(np.float64)
    x_d = pt.from_numpy(xi).cuda()
    assert _sumsq(lib.s3_sumsq, _lib.ptr(x_d), n) == float(np.sum(xi * xi))
    assert _sumsq(lib.s3_leaf_sumsq, _lib.ptr(x_d), _lib.ptr(f_d), n) == float(np.sum((xi * xi)[leaf]))
    # general values: within 1e-13 of the correctly rounded sum, and the same bits on every call
    xg = rng.standard_normal(n) * np.exp(rng.uniform(-3, 3, n))
    x_d = pt.from_numpy(xg).cuda()
    ref_all, ref_leaf = math.fsum(xg * xg), math.fsum((xg * xg)[leaf])
    for fn, args, ref in ((lib.s3_sumsq, (_lib.ptr(x_d), n), ref_all),
                          (lib.s3_leaf_sumsq, (_lib.ptr(x_d), _lib.ptr(f_d), n), ref_leaf)):
        a, b = _sumsq(fn, *args), _sumsq(fn, *args)
        assert abs(a - ref) <= 1e-13 * ref
        assert np.float64(a).tobytes() == np.float64(b).tobytes()

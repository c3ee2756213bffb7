"""STL masks past one tile batch of the tiled kernel, and more STL bodies than the mask call pre-evaluates.

stl_inside_kernel (csrc/stl.cuh) lists at most 1024 tiles of 128 triangles at a time. A larger surface runs in batches
that carry the crossing parity (XOR) and the tolerance-band flag (OR) from batch to batch through global memory. The
other STL tests use at most 20 480 triangles, a single batch. Here an icosphere of 327 680 triangles (2 560 tiles,
3 batches) is tested; its triangles are stored in Morton order of their centroids, so the entry and the exit triangle
of many +x rays fall into different batches. Most points lie within a few tolerances of the surface.

cells_mask_kernel pre-evaluates at most four STL bodies with the tiled kernel (kMaxStlPre); a fifth and sixth take the
per-thread in_stl path inside the mask kernel. Six small bodies in one call cover the mapping between the two.
"""
import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc
from tests.stl_util import write_binary_stl, icosphere_triangles

pytestmark = pytest.mark.gpu

C = np.array([0.5, 0.45, 0.55])
R = 0.31


@pytest.fixture(scope="module")
def big_sphere(cuda, tmp_path_factory):
    from sparsespatialsampling_b200.geometry import GeometrySTL3D, CubeGeometry
    from sparsespatialsampling_b200.geometry.device import GeometryTable
    p = tmp_path_factory.mktemp("stl") / "sphere7.stl"
    write_binary_stl(p, icosphere_triangles(7, radius=R, center=tuple(C)))
    g = GeometrySTL3D("body", False, str(p))
    tab = GeometryTable([CubeGeometry("domain", True, [0, 0, 0], [1, 1, 1]), g], pt.device("cuda"))
    assert tab.stl_geoms == 2 and tab._stl_meta[1, 1] == 327_680          # 2 560 tiles: batches of 1024, 1024, 512
    return g, tab


def _shell_points(rng, n, tol):
    """~80 % within 4 tolerances of the sphere, the rest uniform in its bounding box grown by 2 %."""
    ns = n * 4 // 5
    v = rng.standard_normal((ns, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    shell = C + v * (R + tol * rng.uniform(-4.0, 4.0, ns))[:, None]
    box = C + (rng.random((n - ns, 3)) * 2.0 - 1.0) * R * 1.02
    return np.concatenate([shell, box])


def _both_paths(fn, tab):
    """fn(stl_geoms, stl_meta) -> uint8 tensor: the tiled pre-pass and the per-thread path."""
    return fn(tab.stl_geoms, tab.stl_meta).cpu().numpy(), fn(0, None).cpu().numpy()


def test_points_inside_across_tile_batches(big_sphere):
    from sparsespatialsampling_b200 import _lib
    g, tab = big_sphere
    lib = _lib.load()
    tol = g._tolerance
    pts = _shell_points(np.random.default_rng(0), 120_000, tol)
    d_pts = pt.from_numpy(pts).cuda()

    def run(stl_geoms, meta):
        ins = pt.empty(d_pts.size(0), dtype=pt.uint8, device="cuda")
        _lib.check(lib.s3_points_inside(_lib.ptr(d_pts), d_pts.size(0), 3, _lib.ptr(tab.hdr), _lib.ptr(tab.par), 1,
                                        _lib.ptr(ins), stl_geoms, meta, _lib.stream_ptr()))
        return ins

    tiled, per_thread = _both_paths(run, tab)
    assert np.array_equal(tiled, per_thread)
    got = tiled.astype(bool)
    # the CPU oracle on a subsample (it loops over every triangle per point)
    sub = np.random.default_rng(1).choice(pts.shape[0], 1500, replace=False)
    assert np.array_equal(got[sub], orc.points_inside(g, pts[sub]))
    # the analytic sphere away from the band; the facets of subdivision 7 lie within 3e-6 of it, the fp32 STL vertices
    # within 1e-7
    r = np.linalg.norm(pts - C, axis=1)
    inside, outside = r < R - 1e-5, r > R + tol + 1e-5
    assert got[inside].all() and not got[outside].any()
    assert inside.sum() > 30_000 and outside.sum() > 30_000
    band = ~inside & (r < R + tol - 1e-5)
    assert got[band].all() and band.sum() > 10_000                        # within tol of the surface counts as inside


@pytest.mark.parametrize("refine_mode", [0, 1])
def test_cells_mask_across_tile_batches(big_sphere, refine_mode):
    from sparsespatialsampling_b200 import _lib
    g, tab = big_sphere
    lib = _lib.load()
    rng = np.random.default_rng(10 + refine_mode)
    n = 12_000
    center = _shell_points(rng, n, g._tolerance * 4)
    level = rng.integers(5, 12, n).astype(np.int32)                       # half widths 2^-6 .. 2^-12 around the surface
    c_d, l_d = pt.from_numpy(center).cuda(), pt.from_numpy(level).cuda()
    cells = pt.from_numpy(rng.permutation(n)[: n - 500].astype(np.int64)).cuda()

    def run(stl_geoms, meta):
        inv = pt.empty(cells.numel(), dtype=pt.uint8, device="cuda")
        _lib.check(lib.s3_cells_mask(_lib.ptr(c_d), _lib.ptr(l_d), _lib.ptr(cells), 0, cells.numel(), 3, 1.0,
                                     _lib.ptr(tab.hdr), _lib.ptr(tab.par), tab.n, -1, refine_mode, 0, _lib.ptr(inv),
                                     None, None, stl_geoms, meta, _lib.stream_ptr()))
        return inv

    tiled, per_thread = _both_paths(run, tab)
    assert np.array_equal(tiled, per_thread)
    assert 0.1 < tiled.mean() < 0.9
    # the oracle's check_cell (GeometryObject._apply_mask of the nodes' inside flags) on a subsample of the cells
    sub = np.random.default_rng(2).choice(cells.numel(), 200, replace=False)
    c = cells.cpu().numpy()[sub]
    nodes = center[c][:, None, :] + orc.DIRS_3D[None] * 0.5 / (2.0 ** level[c])[:, None, None]
    assert ((nodes > 0.0) & (nodes < 1.0)).all()                         # the domain cube masks none of them
    inside = orc.points_inside(g, nodes.reshape(-1, 3)).reshape(-1, 8)
    want = [orc.apply_mask(inside[t], False, bool(refine_mode)) for t in range(sub.size)]
    assert np.array_equal(tiled[sub].astype(bool), want)


def test_nodes_mask_across_tile_batches(big_sphere):
    from sparsespatialsampling_b200 import _lib
    g, tab = big_sphere
    lib = _lib.load()
    rng = np.random.default_rng(20)
    n, nn = 8_000, 8
    h = 2.0 ** -rng.integers(7, 13, n)                                   # cell corners around points near the surface
    nodes = _shell_points(rng, n, g._tolerance)[:, None, :] + orc.DIRS_3D[None] * h[:, None, None]
    d_nodes = pt.from_numpy(nodes).cuda()
    for refine_mode in (0, 1):
        def run(stl_geoms, meta):
            inv = pt.empty(n, dtype=pt.uint8, device="cuda")
            _lib.check(lib.s3_nodes_mask(_lib.ptr(d_nodes), n, nn, 3, _lib.ptr(tab.hdr), _lib.ptr(tab.par), tab.n, 1,
                                         refine_mode, _lib.ptr(inv), stl_geoms, meta, _lib.stream_ptr()))
            return inv

        tiled, per_thread = _both_paths(run, tab)
        assert np.array_equal(tiled, per_thread)
        assert 0.05 < tiled.mean() < 0.95


def test_six_stl_bodies_in_one_mask_call(cuda, tmp_path):
    """Bodies 0-3 are pre-evaluated by the tiled kernel, 4 and 5 take the per-thread path; an analytic sphere between
    them shifts every STL body's slot away from its geometry index."""
    from sparsespatialsampling_b200 import _lib
    from sparsespatialsampling_b200.geometry import GeometrySTL3D, SphereGeometry
    from sparsespatialsampling_b200.geometry.device import GeometryTable
    centres = np.array([[0.2, 0.2, 0.2], [0.8, 0.2, 0.25], [0.2, 0.8, 0.3], [0.8, 0.8, 0.7], [0.5, 0.5, 0.8],
                        [0.3, 0.5, 0.65]])
    radii = [0.12, 0.1, 0.14, 0.11, 0.09, 0.08]
    geoms = []
    for i, (c, r) in enumerate(zip(centres, radii)):
        p = tmp_path / f"b{i}.stl"
        write_binary_stl(p, icosphere_triangles(2 + i % 2, radius=r, center=tuple(c)))
        geoms.append(GeometrySTL3D(f"b{i}", False, str(p)))
    geoms.insert(1, SphereGeometry("ball", False, [0.55, 0.2, 0.75], 0.1))
    stl_index = [0, 2, 3, 4, 5, 6]
    tab = GeometryTable(geoms, pt.device("cuda"))
    assert tab.stl_geoms == sum(1 << i for i in stl_index)
    lib = _lib.load()
    rng = np.random.default_rng(5)
    n = 3_000
    body = rng.integers(0, 7, n)
    all_c = np.concatenate([centres[:1], [[0.55, 0.2, 0.75]], centres[1:]])
    all_r = np.array([radii[0], 0.1] + radii[1:])
    v = rng.standard_normal((n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    center = all_c[body] + v * (all_r[body] * rng.uniform(0.5, 1.5, n))[:, None]
    level = rng.integers(3, 8, n).astype(np.int32)
    c_d, l_d = pt.from_numpy(center).cuda(), pt.from_numpy(level).cuda()
    nodes = center[:, None, :] + orc.DIRS_3D[None] * 0.5 / (2.0 ** level)[:, None, None]
    for refine_mode in (0, 1):
        def run(only_geom):
            inv = pt.empty(n, dtype=pt.uint8, device="cuda")
            _lib.check(lib.s3_cells_mask(_lib.ptr(c_d), _lib.ptr(l_d), None, 0, n, 3, 1.0, _lib.ptr(tab.hdr),
                                         _lib.ptr(tab.par), tab.n, only_geom, refine_mode, 0, _lib.ptr(inv), None, None,
                                         tab.stl_geoms, tab.stl_meta, _lib.stream_ptr()))
            return inv.cpu().numpy().astype(bool)

        # the oracle's check_cell per cell and body: GeometryObject._apply_mask of the body's inside flags
        want = np.zeros((len(geoms), n), dtype=bool)
        for gi, g in enumerate(geoms):
            inside = orc.points_inside(g, nodes.reshape(-1, 3)).reshape(n, 8)
            want[gi] = [orc.apply_mask(inside[t], g.keep_inside, bool(refine_mode)) for t in range(n)]
            assert np.array_equal(run(gi), want[gi]), (refine_mode, gi)
            assert 0 < want[gi].sum() < n // 5, (refine_mode, gi)
        assert np.array_equal(run(-1), want.any(axis=0)), refine_mode

"""
GPU parity of the refinement engine (SamplingTree.refine, s_cube.py:563-667):
  * against golden outputs of the REFERENCE itself (tests/golden/*.npz, made by tests/golden/make_golden.py),
  * against the CPU oracle on inputs that are not in the fixtures.
Bit-exact: leaf cells (centre bits, level, numbering), N_leaf per iteration, gains and metrics of the leaves, and -- from
the host-side pointer replay -- the vertex table and the faces (node numbering) of the reference.
Tolerance: metric_per_iter 1e-12 relative (the reference reduces the norm with torch, a different summation tree).
"""
import os
import pickle

import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc
from tests.golden.make_golden import case_definitions

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _run(case):
    import sparsespatialsampling_b200.geometry as geo
    from sparsespatialsampling_b200.s_cube import SamplingTree
    tree = SamplingTree(case["coords"], case["metric"], case["geoms"](geo), **case["kwargs"], sdm_order=1)
    tree.refine()
    return tree


@pytest.mark.parametrize("name", ["g2d_metric", "g2d_ncells", "g3d_metric", "g2d_delta", "g3d_delta", "g2d_delta_geo",
                                  "g2d_reltol", "g3d_delta_geo"])
def test_refine_matches_reference_golden(cuda, name):
    import sparsespatialsampling_b200.geometry as geo
    case = case_definitions(geo)[name]
    ref = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    tree = _run(case)
    info = tree.data_final_mesh
    assert info["n_cells"] == int(ref["n_cells"])
    assert info["iterations"] == int(ref["iterations"])
    assert info["cells_per_iter"] == ref["cells_per_iter"].tolist()
    assert list(tree._leaf_cells) == ref["leaf_index"].tolist()              # numbering + output order
    assert np.array_equal(tree.all_centers.numpy(), ref["centers"])          # fp64 bit-exact
    assert np.array_equal(tree.all_levels.numpy(), ref["levels"])
    assert tree.all_levels.dtype == pt.int64 and tuple(tree.all_levels.shape) == (int(ref["n_cells"]), 1)
    assert info["min_level"] == int(ref["min_level"]) and info["max_level"] == int(ref["max_level"])
    assert info["size_initial_cell"] == float(ref["width"])
    assert tree._gain0 == float(ref["gain0"])
    leaves = pt.tensor(ref["leaf_index"], device=tree._device)
    assert np.array_equal(tree._gain[leaves].cpu().numpy(), ref["leaf_gain"])
    assert np.array_equal(tree._metric_d[leaves].cpu().numpy(), ref["leaf_metric"])
    np.testing.assert_allclose(info["metric_per_iter"], ref["metric_per_iter"], rtol=1e-12)
    # vertex table and faces: identical to the reference's history-dependent node sharing (pointer replay on the host)
    assert tree.face_ids.dtype == pt.int32
    assert np.array_equal(tree.face_ids.numpy(), ref["faces"])
    assert np.array_equal(tree.all_nodes.numpy(), ref["vertices"])


@pytest.mark.parametrize("name", ["g2d_metric", "g3d_metric"])
def test_export_stage_on_reference_grid(cuda, name):
    # ExportData._build_knn_cache + interpolate_data (export.py:403-468) against the reference's own output
    import synth
    import sparsespatialsampling_b200.geometry as geo
    from sparsespatialsampling_b200.knn import KnnIndex
    from sparsespatialsampling_b200.interpolate import interp_gather
    case = case_definitions(geo)[name]
    ref = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    k = ref["knn_idx"].shape[1]
    idx, w32, w64 = KnnIndex(case["coords"]).tables(pt.from_numpy(ref["centers"]), k)
    assert np.array_equal(idx.cpu().numpy(), ref["knn_idx"])                 # KNN indices bit-exact
    np.testing.assert_allclose(w64.cpu().numpy(), ref["knn_w"], rtol=1e-14)
    field = synth.wake_field(case["coords"], 0, 12, 12, components=2).cuda()
    out32 = interp_gather(field, idx, w32).cpu().numpy()
    scale = np.abs(field.cpu().numpy()[ref["knn_idx"].astype(np.int64)]).max(axis=1)
    assert (np.abs(out32 - ref["interp"]) <= 1e-5 * np.maximum(scale, 1e-30)).all()   # stated fp32 tolerance
    out64 = interp_gather(field, idx, w64, out_dtype=pt.float64).cpu().numpy()
    np.testing.assert_allclose(out64, ref["interp"], rtol=1e-12, atol=1e-15)


def test_refine_matches_oracle_on_fresh_inputs(cuda):
    # inputs that are not in the fixtures: GPU path vs CPU oracle, same host
    import synth
    import sparsespatialsampling_b200.geometry as geo
    from sparsespatialsampling_b200.s_cube import SamplingTree
    x = synth.cylinder2d_cloud(9000, seed=11)
    m = synth.wake_metric(x)
    mk = lambda: [geo.CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
                  geo.SphereGeometry("cyl", False, synth.CYL2D["pos"], synth.CYL2D["radius"], refine=True,
                                     min_refinement_level=7)]
    kw = dict(uniform_level=5, min_metric=0.7, n_cells_iter_start=25, n_cells_iter_end=5)
    tree = SamplingTree(x, m, mk(), **kw, sdm_order=1)
    tree.refine()
    o = orc.OracleTree(x.numpy(), m.numpy(), mk(), **kw, sdm_order=1).refine()
    assert list(tree._leaf_cells) == o.leaf_order
    assert np.array_equal(tree.all_centers.numpy(), o.all_centers)
    assert np.array_equal(tree.all_levels.numpy(), o.all_levels)
    assert tree.data_final_mesh["cells_per_iter"] == o.n_cells_log
    np.testing.assert_allclose(tree.data_final_mesh["metric_per_iter"], o.metric_log, rtol=1e-12)


@pytest.mark.parametrize("fused", [1, 0])
def test_selection_order_matches_heapq(cuda, fused):
    # s3_select_topk == heapq.nlargest(k, leaves, key=(gain, -idx)) including exact gain ties; both implementations:
    # the single cooperative launch (default, k <= 8192) and the multi-kernel radix select + sort
    import heapq
    from sparsespatialsampling_b200 import _lib
    lib = _lib.load()
    _lib.check(lib.s3_select_set_fused(fused))
    rng = np.random.default_rng(0)
    for n, k in [(5000, 37), (5000, 5000), (100000, 2500), (7, 3), (3000, 1), (400000, 8192), (400000, 9000),
                 (1000, 1000), (300, 2)]:
        gain = rng.random(n)
        if n == 300:
            gain = -gain                                  # negative and mixed-sign gains keep their order
            gain[::7] = 1e-300
        gain[rng.integers(0, n, n // 3)] = 0.25          # many exact ties
        gain[rng.integers(0, n, n // 10)] = 0.0
        flags = (rng.random(n) < 0.7).astype(np.uint8)
        flags[:k] |= 1
        leaves = np.nonzero(flags & 1)[0]
        kk = min(k, leaves.size)
        ref = heapq.nlargest(kk, leaves.tolist(), key=lambda i: (gain[i], -i))
        g = pt.from_numpy(gain).cuda()
        f = pt.from_numpy(flags).cuda()
        out = pt.empty(kk, dtype=pt.int64, device="cuda")
        _lib.check(lib.s3_select_topk(_lib.ptr(g), _lib.ptr(f), n, kk, _lib.ptr(out), _lib.stream_ptr()))
        assert out.cpu().tolist() == ref, (n, k, fused)
    _lib.check(lib.s3_select_set_fused(1))


def test_facade_outputs_and_pickle(cuda, tmp_path):
    # SparseSpatialSampling.execute_grid_generation: attributes + files (sparse_spatial_sampling.py:116-146)
    import synth
    import sparsespatialsampling_b200 as s3
    x = synth.cylinder2d_cloud(3000, seed=5)
    m = synth.wake_metric(x)
    geoms = [s3.geometry.CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
             s3.geometry.SphereGeometry("cyl", False, synth.CYL2D["pos"], synth.CYL2D["radius"])]
    sc = s3.SparseSpatialSampling(x, m, geoms, str(tmp_path), "case", uniform_levels=4, min_metric=0.5,
                                  n_cells_iter_start=30)
    sc.execute_grid_generation()
    nc = sc.centers.shape[0]
    assert sc.centers.dtype == pt.float64 and sc.centers.shape == (nc, 2) and not sc.centers.is_cuda
    assert sc.faces.shape == (nc, 4) and sc.levels.shape == (nc, 1) and sc.vertices.shape[1] == 2
    assert sc.size_initial_cell == 2.2 and sc.n_dimensions == 2
    info = pt.load(os.path.join(tmp_path, "mesh_info_case.pt"), weights_only=False)
    for key in ["size_initial_cell", "n_cells_orig", "n_cells", "iterations", "min_level", "max_level",
                "metric_per_iter", "cells_per_iter", "t_total", "t_uniform", "t_renumbering", "t_geometry",
                "t_adaptive"]:
        assert key in info
    assert info["n_cells"] == nc
    again = pt.load(os.path.join(tmp_path, "s_cube_case.pt"), weights_only=False)
    assert pt.equal(again.centers, sc.centers) and again._sampling is None


def test_input_validation(cuda, tmp_path):
    import sparsespatialsampling_b200 as s3
    x = pt.rand(100, 2, dtype=pt.float64)
    dom = s3.geometry.CubeGeometry("domain", True, [0.0, 0.0], [1.0, 1.0])
    with pytest.raises(AssertionError):
        s3.SparseSpatialSampling(x, pt.rand(100, 1), [dom], str(tmp_path), "a")          # metric must be 1-D
    with pytest.raises(AssertionError):
        s3.SparseSpatialSampling(x, pt.rand(100), [], str(tmp_path), "a")               # no geometry
    with pytest.raises(AssertionError):
        body = s3.geometry.CubeGeometry("b", False, [0.0, 0.0], [1.0, 1.0])
        s3.SparseSpatialSampling(x, pt.rand(100), [body], str(tmp_path), "a")           # no domain
    with pytest.raises(ValueError):
        dom3 = s3.geometry.CubeGeometry("domain", True, [0.0, 0.0, 0.0], [1.0, 1.0, 1.0])
        s3.SparseSpatialSampling(x, pt.rand(100, dtype=pt.float64), [dom3], str(tmp_path), "a")   # dim mismatch


@pytest.mark.parametrize("name", ["C1", "C2"])
def test_full_size_configs_match_the_reference_run(cuda, name):
    """BASELINE.json configurations C1 (~20k points) and C2 (~100k points, the bench workload) at full size against a run
    of the reference itself (tests/golden/make_golden_configs.py: SHA-256 of centers / levels / faces / vertices, the
    per-iteration logs; the reference needed 64 s / 129 s with n_jobs=8 in the build container)."""
    import hashlib
    import synth
    import sparsespatialsampling_b200.geometry as geo
    from sparsespatialsampling_b200.s_cube import SamplingTree
    ref = np.load(os.path.join(GOLDEN, f"config_{name}.npz"))
    x = synth.cylinder2d_cloud(synth.CONFIGS[name][0], seed=0)
    assert x.shape[0] == int(ref["n_points"])
    geoms = [geo.CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
             geo.SphereGeometry("cylinder", False, synth.CYL2D["pos"], synth.CYL2D["radius"], refine=True)]
    tree = SamplingTree(x, synth.wake_metric(x), geoms, uniform_level=5, min_metric=0.75, sdm_order=1)
    tree.refine()
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    info = tree.data_final_mesh
    assert info["n_cells"] == int(ref["n_cells"]) and info["iterations"] == int(ref["iterations"])
    assert info["cells_per_iter"] == ref["cells_per_iter"].tolist()
    np.testing.assert_allclose(info["metric_per_iter"], ref["metric_per_iter"], rtol=1e-12)
    assert sha(np.asarray(list(tree._leaf_cells), dtype=np.int64)) == str(ref["leaf_index_sha"])
    assert sha(tree.all_centers.numpy()) == str(ref["centers_sha"])
    assert sha(tree.all_levels.numpy()) == str(ref["levels_sha"])
    assert str(tree.face_ids.numpy().dtype) == str(ref["faces_dtype"])
    assert sha(tree.face_ids.numpy()) == str(ref["faces_sha"])
    assert tree.all_nodes.shape[0] == int(ref["n_vertices"]) and sha(tree.all_nodes.numpy()) == str(ref["vertices_sha"])


def _edge_cases():
    rng = np.random.default_rng(0)
    x, m = rng.random((500, 2)), rng.random(500)
    x3, m3 = rng.random((300, 3)), rng.random(300)
    box2 = lambda g: [g.CubeGeometry("d", True, [0, 0], [1, 1])]
    box3 = lambda g: [g.CubeGeometry("d", True, [0, 0, 0], [1, 1, 1])]
    return {
        "plain_2d": (x, m, box2, dict(uniform_level=3, min_metric=0.7)),
        "uniform_level_1": (x, m, box2, dict(uniform_level=1, min_metric=0.5)),
        "n_cells_below_uniform_grid": (x, m, box2, dict(uniform_level=4, n_cells=50)),
        "cells_per_iter_above_leaf_count": (x, m, box2, dict(uniform_level=2, min_metric=0.6, n_cells_iter_start=10000)),
        "constant_metric": (x, np.ones(500), box2, dict(uniform_level=3, min_metric=0.9)),
        "12_points": (x[:12], m[:12], box2, dict(uniform_level=2, min_metric=0.5)),
        "as_many_points_as_neighbours": (x[:8], m[:8], box2, dict(uniform_level=2, min_metric=0.5)),
        "plain_3d": (x3, m3, box3, dict(uniform_level=2, min_metric=0.6)),
        "30_points_3d": (x3[:30], m3[:30], box3, dict(uniform_level=2, min_metric=0.5)),
        "metric_reached_after_uniform": (x, m, box2, dict(uniform_level=5, min_metric=0.05)),
        "body_covers_most_of_the_domain": (x, m, lambda g: [g.CubeGeometry("d", True, [0, 0], [1, 1]),
                                                           g.CubeGeometry("b", False, [0.1, 0.1], [0.9, 0.9])],
                                           dict(uniform_level=3, min_metric=0.5)),
        "two_domains_last_is_root": (x, m, lambda g: [g.CubeGeometry("d1", True, [0, 0], [1, 1]),
                                                     g.CubeGeometry("d2", True, [0.0, 0.0], [0.5, 0.5])],
                                     dict(uniform_level=3, min_metric=0.5)),
    }


@pytest.mark.parametrize("name", sorted(_edge_cases()))
def test_edge_configurations_match_oracle(cuda, name):
    # corner cases of the control flow (tiny clouds, degenerate schedules, stopping right after the uniform phase, the
    # root-cell rule with several domains): same leaves, levels and iteration log as the restatement of the reference
    import sparsespatialsampling_b200.geometry as geo
    from sparsespatialsampling_b200.s_cube import SamplingTree
    from oracle import s3_oracle as orc
    x, m, geoms, kw = _edge_cases()[name]
    tree = SamplingTree(pt.from_numpy(x), pt.from_numpy(m), geoms(geo), sdm_order=1, **kw)
    tree.refine()
    ref = orc.OracleTree(x, m, geoms(geo), sdm_order=1, **kw).refine()
    assert np.array_equal(tree.all_centers.numpy(), ref.all_centers)
    assert np.array_equal(tree.all_levels.numpy(), ref.all_levels)
    assert tree.data_final_mesh["cells_per_iter"] == ref.n_cells_log

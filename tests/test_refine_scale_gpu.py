"""The refinement loop (SamplingTree.refine) at production selection sizes, bit for bit against the CPU oracle.

The other end-to-end parity tests select at most ~100 cells per iteration. Production runs select thousands: C4 and C5
(10M points) select 0.001 * N = 10 000 cells per iteration, above the fused cooperative selection's limit of 8 192
(kFusedMaxSortK, csrc/refine.cu), so every iteration goes through the multi-kernel radix select (select_topk_multi),
and with a constant schedule that selection runs speculatively behind the mask pass of the previous iteration.

  A  3-D, metric mode, 9 000 cells per iteration: select_topk_multi, handed out speculatively; pure C oracle (its own
     brute-force KNN) with the topology replay; once more with the topology replayed synchronously
  B  3-D, n_cells mode, metric rounded to two decimals: selections of 896 and 5 376 (fused) and 12 000 (multi) in one
     run, 22 544 leaves tied at the cut of one iteration (ties resolved by index), a speculation dropped when the loop
     stops
  C  input of B with the multi-kernel selection for every k
  D  3-D, max_delta_level: the constraint closure and a geometry refinement to level 9, with the topology replay
  E  2-D, 400k points, C3 geometry: 87 iterations, wedge refinement
  F  3-D, pre_select: five uniform levels without a mask pass (parent lists 1 ... 4 096 through one pinned buffer)
  G  3-D, C5 geometry with a 1 280-triangle STL body inside the loop and in the geometry refinement

For every case the product and the oracle must agree on the selected cells of every iteration (order included), the
per-iteration logs, and the centre, level, gain, metric, leaf and invalid bits of EVERY cell (not only the leaves).

Except in A, the oracle's knn_predict is answered by the product's KnnIndex.predict while the oracle runs: the C oracle's
brute-force search would dominate the file's run time, and predict is held bit-exact to that search at these sizes by
test_gridgen_scale_gpu.py. test_device_knn_answers_the_oracles_queries_like_the_c_oracle re-checks it on a sample of
the queries the oracle issued in case B.
"""
import copy
import functools
import gc
import heapq
import time

import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc
from oracle.topology_oracle import OracleTopology

pytestmark = pytest.mark.gpu

D_LEVEL = 9                             # case D: cylinder refinement level, above the adaptive depth (8)
STL_SUBDIV = 3                          # case G: icosphere of 20 * 4^3 = 1 280 triangles

CASES = {
    #     cloud                          config  options                                                   C KNN  topology
    "A": (("cylinder3d", 40_000, None), "C4", dict(uniform_level=4, min_metric=2.5, n_cells_iter_start=9000), True, True),
    "B": (("cylinder3d", 100_000, 2), "C4", dict(uniform_level=4, n_cells=150_000, n_cells_iter_start=12_000,
                                                 n_cells_iter_end=2000), False, False),
    "D": (("cylinder3d", 60_000, None), "C4-D", dict(uniform_level=3, max_delta_level=True, n_cells=80_000,
                                                     n_cells_iter_start=3000), False, True),
    "E": (("airfoil2d", 400_000, None), "C3", dict(uniform_level=6, n_cells=100_000), False, False),
    "F": (("cylinder3d", 100_000, None), "C4", dict(uniform_level=5, pre_select=True, n_cells=60_000,
                                                    n_cells_iter_start=3000), False, False),
    "G": (("cylinder3d", 100_000, None), "C5", dict(uniform_level=5, n_cells=80_000, n_cells_iter_start=3000), False,
          False),
}
# product runs: case -> (oracle case, multi-kernel selection only, topology replayed synchronously)
RUNS = {"A": ("A", False, False), "A-sync": ("A", False, True), "B": ("B", False, False), "C": ("B", True, False),
        "D": ("D", False, False), "E": ("E", False, False), "F": ("F", False, False), "G": ("G", False, False)}


@functools.lru_cache(maxsize=None)
def _cloud(kind, n, decimals):
    import synth
    if kind == "airfoil2d":
        x = synth.airfoil2d_cloud(n, seed=0)
        m = synth.wake_metric(x, xc=1.0, yc=0.0)                    # wake centre of C3 (scripts/run_config.py)
    else:
        x = synth.cylinder3d_cloud(n, seed=0)
        m = synth.wake_metric(x, xc=0.8, yc=1.0)                    # wake centre of C4 / C5
    m = m.numpy()
    if decimals is not None:
        m = np.round(m, decimals)                                   # coarse levels: exact gain ties between leaves
    return x.numpy(), m


@functools.lru_cache(maxsize=None)
def _geometries(name):
    import tempfile
    from scripts.run_config import config
    if name == "C4-D":
        domain, cylinder = _geometries("C4")
        cylinder = copy.copy(cylinder)
        cylinder._min_refinement_level = D_LEVEL
        return domain, cylinder
    # the STL file is read by the constructor; the directory can go right after
    with tempfile.TemporaryDirectory() as tmp:
        return tuple(config(name, None, STL_SUBDIV, tmp)[1])


_ORIG_GEOMETRY_PARAMS = orc.geometry_params
_PARAMS = {}


def _geometry_params(g):
    """orc.geometry_params, built once per geometry (the geometries above live for the whole session)."""
    if id(g) not in _PARAMS:
        type_id, par, n_extra = _ORIG_GEOMETRY_PARAMS(g)
        _PARAMS[id(g)] = type_id, np.ascontiguousarray(par, dtype=np.float64), n_extra
    return _PARAMS[id(g)]


@functools.lru_cache(maxsize=None)
def _oracle(case):
    """Oracle run of a case: (OracleTree, cells left unselected but tied with the k-th selected cell per iteration,
    queries issued to knn_predict (substituted runs), wall time)."""
    (kind, n, dec), geo_name, kw, c_knn, topology = CASES[case]
    X, m = _cloud(kind, n, dec)
    ties, queries = [], []
    nlargest = heapq.nlargest

    def nlargest_spy(k, iterable, key):
        # the oracle's selection (s_cube.py:601-602); counts the leaves that tie with the k-th winner but lose on index
        leaves = list(iterable)
        out = nlargest(k, leaves, key=key)
        won = set(out)
        kth = key(out[-1])[0] if out else None
        ties.append(sum(1 for i in leaves if i not in won and key(i)[0] == kth))
        return out

    with pytest.MonkeyPatch.context() as mp:
        # the STL parameter block is thousands of floats: build it once per geometry instead of once per cell
        mp.setattr(orc, "geometry_params", _geometry_params)
        mp.setattr(heapq, "nlargest", nlargest_spy)
        if not c_knn:
            from sparsespatialsampling_b200.knn import KnnIndex
            index = KnnIndex(pt.from_numpy(X), pt.from_numpy(m))

            def predict(points, values, query, k):
                assert points.shape == X.shape and values.shape == m.shape
                q = np.ascontiguousarray(np.atleast_2d(query), dtype=np.float64)
                queries.append(q)
                return index.predict(pt.from_numpy(q), k).cpu().numpy()
            mp.setattr(orc, "knn_predict", predict)
        t0 = time.time()
        o = orc.OracleTree(X, m, list(_geometries(geo_name)), sdm_order=1, **kw,
                           topology=OracleTopology if topology else None).refine()
        wall = time.time() - t0
    return o, ties, queries, wall


@functools.lru_cache(maxsize=None)
def _product(run):
    """Product run: its final state of every cell, the per-iteration logs and what the spies saw."""
    from sparsespatialsampling_b200 import _lib
    from sparsespatialsampling_b200.s_cube import SamplingTree
    case, multi_only, sync_topology = RUNS[run]
    (kind, n, dec), geo_name, kw, _, _ = CASES[case]
    X, m = _cloud(kind, n, dec)
    lib = _lib.load()
    spy = dict(select=[], spec=[], parents=[])
    with pytest.MonkeyPatch.context() as mp:
        if sync_topology:
            mp.setattr(SamplingTree, "topology_async", False)
        tree = SamplingTree(pt.from_numpy(X), pt.from_numpy(m), list(_geometries(geo_name)), sdm_order=1, **kw)
        tree._selected_log = []
        select, mask, refine_cells = tree._select, tree._mask, tree._refine_cells

        def select_spy(k):
            spec = tree._spec_selection
            out = select(k)
            # (k after the leaf clamp, length of the speculation waiting for this call, whether it was handed out)
            spy["select"].append((min(k, len(tree._leaf_cells)), None if spec is None else len(spec), out is spec))
            return out

        def mask_spy(cells, refine_geometry, geometry_no):
            queued = tree._speculate_k
            out = mask(cells, refine_geometry, geometry_no)
            if queued and tree._spec_selection is not None:
                spy["spec"].append(len(tree._spec_selection))           # a selection queued behind this mask pass
            return out

        def refine_cells_spy(parents):
            out = refine_cells(parents)
            spy["parents"].append((len(parents), tree._pin_i64.data_ptr()))
            return out
        mp.setattr(tree, "_select", select_spy)
        mp.setattr(tree, "_mask", mask_spy)
        mp.setattr(tree, "_refine_cells", refine_cells_spy)
        _lib.check(lib.s3_select_set_fused(0 if multi_only else 1))
        try:
            t0 = time.time()
            tree.refine()
            wall = time.time() - t0
        finally:
            _lib.check(lib.s3_select_set_fused(1))
    nc = tree._n_cells
    res = dict(n_cells=nc, center=tree._center[:nc].cpu().numpy(), level=tree._level[:nc].cpu().numpy(),
               gain=tree._gain[:nc].cpu().numpy(), metric=tree._metric_d[:nc].cpu().numpy(),
               flags=tree._flags[:nc].cpu().numpy(), leaf_order=list(tree._leaf_cells), all_centers=tree.all_centers.numpy(),
               all_levels=tree.all_levels.numpy(), face_ids=tree.face_ids.numpy(), all_nodes=tree.all_nodes.numpy(),
               selected=tree._selected_log, info=dict(tree.data_final_mesh), spy=spy, wall=wall)
    del tree, select, mask, refine_cells
    gc.collect()                                                  # the spies close over the tree
    pt.cuda.empty_cache()
    return res


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


@pytest.mark.parametrize("run", list(RUNS))
def test_refine_matches_oracle_at_scale(cuda, run):
    case = RUNS[run][0]
    topology = CASES[case][4]
    o, _, _, t_oracle = _oracle(case)
    p = _product(run)
    print(f"\n[{run}] product {p['wall']:.1f} s, oracle {t_oracle:.1f} s, {p['n_cells']} cells, "
          f"{len(o.leaf_order)} leaves, selections {[len(s) for s in o.selected_log]}")
    # per iteration
    assert len(p["selected"]) == len(o.selected_log)
    for it, (a, b) in enumerate(zip(p["selected"], o.selected_log)):
        assert a == b, f"iteration {it}: selection differs"
    assert p["info"]["cells_per_iter"] == o.n_cells_log
    np.testing.assert_allclose(p["info"]["metric_per_iter"], o.metric_log, rtol=1e-12)
    # every cell, leaves or not
    n = len(o.center)
    assert p["n_cells"] == n
    assert np.array_equal(_bits(p["center"]), _bits(np.stack(o.center)))
    assert np.array_equal(p["level"], np.asarray(o.level))
    assert np.array_equal(_bits(p["gain"]), _bits(np.asarray(o.gain, dtype=np.float64)))
    assert np.array_equal(_bits(p["metric"]), _bits(np.asarray(o.metric, dtype=np.float64)))
    leaf = np.zeros(n, dtype=bool)
    leaf[list(o.leaf)] = True
    assert np.array_equal((p["flags"] & 1) != 0, leaf)
    assert np.array_equal((p["flags"] & 2) != 0, np.asarray(o.invalid))
    # final grid
    assert p["leaf_order"] == o.leaf_order
    assert np.array_equal(_bits(p["all_centers"]), _bits(o.all_centers))
    assert np.array_equal(p["all_levels"], o.all_levels)
    if topology:
        assert np.array_equal(p["face_ids"], o.face_ids)
        assert np.array_equal(_bits(p["all_nodes"]), _bits(o.all_nodes))


def test_cases_reach_the_paths_they_claim(cuda):
    """Guards the inputs above: each case reaches the path it is there for (sizes, speculation, ties, closure)."""
    k = lambda run: [s[0] for s in _product(run)["spy"]["select"]]
    # A: k = 9 000 through select_topk_multi, and a speculative selection handed out
    a = _product("A")["spy"]
    assert max(k("A")) > 8192
    assert any(consumed and n_spec == kk > 8192 for kk, n_spec, consumed in a["select"])
    # B: one run selects with both implementations; a speculation is dropped when the loop stops
    b = _product("B")["spy"]
    assert min(k("B")) <= 8192 < max(k("B"))
    assert len(b["spec"]) > sum(consumed for _, _, consumed in b["select"]) >= 1
    # every speculation that reaches _select has the size of the selection it stands for, and is handed out
    for run in RUNS:
        for kk, n_spec, consumed in _product(run)["spy"]["select"]:
            assert n_spec is None or (n_spec == kk and consumed), run
    # B: an iteration whose k-th selected gain equals the gain of a leaf left unselected (ties cut by index)
    _, ties, _, _ = _oracle("B")
    assert max(ties) > 0
    assert any(t > 0 and n > 8192 for t, n in zip(ties, k("B")))
    # D: the constraint closure added cells: more parents refined than cells selected in some iteration
    d = _product("D")
    adaptive = d["spy"]["parents"][3:3 + len(d["selected"])]
    assert any(n_par > len(sel) for (n_par, _), sel in zip(adaptive, d["selected"]))
    assert int(d["level"].max()) == D_LEVEL > max(int(d["level"][s].max()) for s in d["selected"]) + 1
    # F: no cell is masked, and several uniform levels with more than one parent write the same pinned buffer
    f = _product("F")
    uniform = f["spy"]["parents"][:5]
    assert [n_par for n_par, _ in uniform] == [1, 8, 64, 512, 4096]
    shared = [ptr for n_par, ptr in uniform if n_par > 1]
    assert max(shared.count(ptr) for ptr in shared) >= 2
    assert not (f["flags"] & 2).any()
    # G: the STL body invalidates cells during the loop and is refined afterwards
    g = _product("G")
    body = np.array([0.8, 1.0, np.pi * 0.1 / 2])
    invalid = (g["flags"] & 2) != 0
    assert (np.linalg.norm(g["center"][invalid] - body, axis=1) < 0.12).any()
    n_adaptive = g["info"]["cells_per_iter"][-1]
    assert len(g["leaf_order"]) > n_adaptive                    # the geometry refinement added leaves


def test_device_knn_answers_the_oracles_queries_like_the_c_oracle(cuda):
    """The substitution the oracle runs rely on: a sample of the queries case B issued, through the C oracle."""
    from sparsespatialsampling_b200.knn import KnnIndex
    (kind, n, dec), _, _, _, _ = CASES["B"]
    X, m = _cloud(kind, n, dec)
    _, _, queries, _ = _oracle("B")
    q = np.concatenate(queries)
    assert q.shape[0] > 1_000_000
    rng = np.random.default_rng(0)
    sample = q[np.sort(rng.choice(q.shape[0], 20_000, replace=False))]
    want = orc.idw_predict(*orc.knn_search(X, sample, 26), m)
    got = KnnIndex(pt.from_numpy(X), pt.from_numpy(m)).predict(pt.from_numpy(sample), 26).cpu().numpy()
    assert np.array_equal(_bits(got), _bits(want))

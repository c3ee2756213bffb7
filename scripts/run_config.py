"""
Runs one of the BASELINE.json configurations end to end on one GPU (grid generation + export interpolation) with
size-independent correctness checks, and prints one JSON line with the timings.

  python scripts/run_config.py C3 [--snapshots T] [--n-cells-max M]
  python scripts/run_config.py C4 [--snapshots T] [--n-cells-max M]
  python scripts/run_config.py C5 [--snapshots T] [--n-cells-max M]     (STL-masked body + weighted SVD of the export)

Checks (no reference run needed, all hold for any size):
  * KNN indices / weights of a random sample of cells equal the CPU oracle's brute-force search (bit-exact idx);
  * interpolated rows of that sample are within 1e-5 (relative to the largest gathered magnitude) of the oracle;
  * a constant field is reproduced (weights sum to one), the operator is linear;
  * every leaf cell passes the geometry masks of the oracle (sample), levels and centres are consistent with the
    integer lattice, faces reference valid vertices, per-cell corner coordinates equal centre +- width/2^(level+1).
"""
import argparse
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch as pt

import synth
import sparsespatialsampling_b200 as s3
from sparsespatialsampling_b200.export import KnnTables
from sparsespatialsampling_b200.knn import KnnIndex
from oracle import s3_oracle as orc


def fill_field(out: pt.Tensor, coords: pt.Tensor, n_total: int, comps: int, xc: float, yc: float, chunk: int = 16):
    """Closed-form wake written into out [N, comps, T] chunk by chunk (keeps the fp64 temporaries small)."""
    T = out.size(2)
    for t0 in range(0, T, chunk):
        t1 = min(t0 + chunk, T)
        out[:, :, t0:t1] = synth.wake_field(coords, t0, t1, n_total, comps, xc, yc)
    return out


def config(name: str, n_cells_max, stl_subdiv: int = 4, tmp_dir: str = None):
    """Cloud, geometries, wake centre and grid options of a configuration; C5 writes its STL body into ``tmp_dir``."""
    geo = s3.geometry
    if name == "C3":
        x = synth.airfoil2d_cloud(synth.CONFIGS["C3"][0], seed=0)
        geoms = [geo.CubeGeometry("domain", True, synth.AIRFOIL2D["lower"], synth.AIRFOIL2D["upper"]),
                 geo.TriangleGeometry("wedge", False, [[0.0, 0.0], [1.0, 0.06], [1.0, -0.06]], refine=True)]
        return x, geoms, dict(xc=1.0, yc=0.0), dict(uniform_levels=6, n_cells_max=n_cells_max or 100000)
    if name == "C4":
        x = synth.cylinder3d_cloud(synth.CONFIGS["C4"][0], seed=0)
        zmax = synth.CYL3D["upper"][2]
        geoms = [geo.CubeGeometry("domain", True, synth.CYL3D["lower"], synth.CYL3D["upper"]),
                 geo.CylinderGeometry3D("cylinder", False, [[0.8, 1.0, 0.0], [0.8, 1.0, zmax]], 0.05, refine=True)]
        return x, geoms, dict(xc=0.8, yc=1.0), dict(uniform_levels=5, n_cells_max=n_cells_max or 500000)
    if name == "C5":
        # same cloud as C4; the body is a closed triangulated surface (icosphere, 5120 triangles) read from an STL file
        from tests.stl_util import icosphere_triangles, write_binary_stl
        x = synth.cylinder3d_cloud(synth.CONFIGS["C5"][0], seed=0)
        zmax = synth.CYL3D["upper"][2]
        stl = os.path.join(tmp_dir, "c5_body.stl")
        write_binary_stl(stl, icosphere_triangles(stl_subdiv, 0.12, (0.8, 1.0, zmax / 2)))
        geoms = [geo.CubeGeometry("domain", True, synth.CYL3D["lower"], synth.CYL3D["upper"]),
                 geo.GeometrySTL3D("body", False, stl, refine=True)]
        return x, geoms, dict(xc=0.8, yc=1.0), dict(uniform_levels=5, n_cells_max=n_cells_max or 500000)
    raise SystemExit(f"unknown config {name}")


def main(tmp_dir: str):
    ap = argparse.ArgumentParser()
    ap.add_argument("name", choices=["C3", "C4", "C5"])
    ap.add_argument("--svd", action="store_true", help="weighted SVD of the exported matrix (always on for C5)")
    ap.add_argument("--snapshots", type=int, default=0)
    ap.add_argument("--n-cells-max", type=int, default=0)
    ap.add_argument("--sample", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--tune", default="", help="comma separated key=value pairs for s3x_tune (csrc/interp.cu), e.g. 2=1,3=0")
    ap.add_argument("--dense", action="store_true", help="the reference's dense [N, D, T] layout instead of 128-byte pitched rows")
    ap.add_argument("--stl-subdiv", type=int, default=4, help="C5: icosphere subdivisions of the STL body (4: 5120 triangles, 6: 81920)")
    ap.add_argument("--grid-only", action="store_true", help="stop after grid generation (timings only)")
    ap.add_argument("--e2e", action="store_true", help="also time the host-to-host export (256 snapshots): DMA vs row gather")
    args = ap.parse_args()
    dev = pt.device("cuda", 0)
    pt.cuda.set_device(dev)
    if args.tune:
        from sparsespatialsampling_b200 import _lib
        for kv in args.tune.split(","):
            key, val = kv.split("=")
            _lib.tune(int(key), int(val))
    x, geoms, wake, grid_kw = config(args.name, args.n_cells_max, args.stl_subdiv, tmp_dir)
    d = x.size(1)
    k = 8 if d == 2 else 26
    T = args.snapshots or synth.CONFIGS[args.name][1]
    xd = x.to(dev)
    metric = synth.wake_metric(xd, xc=wake["xc"], yc=wake["yc"]).cpu()

    # ---- grid generation
    t0 = time.time()
    sc = s3.SparseSpatialSampling(x, metric, geoms, tmp_dir, args.name.lower(), **grid_kw)
    t_setup = time.time() - t0
    sc.execute_grid_generation()
    info = sc.mesh_info
    nc = sc.centers.size(0)
    width = sc.size_initial_cell
    if args.grid_only:
        print(json.dumps({"config": args.name, "stl_triangles": 20 * 4 ** args.stl_subdiv if args.name == "C5" else None,
                          "n_points": int(x.size(0)), "n_cells": int(nc), "grid_gen_s": info["t_total"],
                          "t_uniform": info["t_uniform"], "t_adaptive": info["t_adaptive"], "t_geometry": info["t_geometry"],
                          "t_renumbering": info["t_renumbering"], "t_knn_build_gridgen": info["t_knn_build"],
                          "iterations": info["iterations"], "levels": [info["min_level"], info["max_level"]]}))
        return

    # grid consistency
    lv = sc.levels.squeeze(1).numpy()
    cen = sc.centers.numpy()
    half = width / 2.0 ** (lv + 1)
    verts = sc.vertices.numpy()
    faces = sc.faces.numpy().astype(np.int64)
    assert faces.min() >= 0 and faces.max() < verts.shape[0]
    dirs = orc.DIRS_2D if d == 2 else orc.DIRS_3D
    corner = verts[faces]                                               # [nc, 2^d, d]
    want = cen[:, None, :] + dirs[None, :, :] * half[:, None, None]
    assert np.abs(corner - want).max() <= 1e-12 * width
    # (the reference's renumbering keeps node ids outside [min, max] of the used ones, so unused vertices may remain)
    assert np.unique(faces).size <= verts.shape[0]
    # centres sit on the lattice of their level: (c - root_lo) / (width / 2^level) is a half-integer
    root_lo = np.asarray(geoms[0].center.numpy()) - width / 2
    frac = (cen - root_lo) / (width / 2.0 ** lv)[:, None]
    assert np.abs(frac - np.floor(frac) - 0.5).max() < 1e-6
    # no duplicate leaves
    assert np.unique(np.concatenate([lv[:, None], np.round(frac - 0.5)], axis=1), axis=0).shape[0] == nc
    # masks: every leaf is valid for the oracle (sample)
    rng = np.random.default_rng(0)
    sample = rng.choice(nc, size=min(args.sample, nc), replace=False)
    for c in sample[:200]:
        nodes = cen[c][None, :] + dirs * half[c]
        for g in geoms:
            assert not orc.check_cell(g, nodes, False), f"leaf {c} is invalid for geometry {g.name}"

    # ---- export tables + interpolation
    t0 = time.time()
    index = KnnIndex(xd)
    pt.cuda.synchronize()
    t_build = time.time() - t0
    t0 = time.time()
    tables = KnnTables(index, sc.centers.to(dev), k)
    pt.cuda.synchronize()
    t_tables = time.time() - t0
    d_ref, i_ref = orc.knn_search(x.numpy(), cen[sample], k)
    assert np.array_equal(tables.idx[pt.from_numpy(sample).to(dev)].cpu().numpy().astype(np.int64), i_ref)
    w_ref = orc.export_weights(d_ref)
    np.testing.assert_allclose(tables.w64[pt.from_numpy(sample).to(dev)].cpu().numpy(), w_ref, rtol=1e-13)

    from sparsespatialsampling_b200.interpolate import alloc_snapshots
    if args.dense:
        data = pt.empty((x.size(0), 1, T), dtype=pt.float32, device=dev)
        out = pt.empty((nc, 1, T), dtype=pt.float32, device=dev)
    else:
        data = alloc_snapshots(x.size(0), 1, T, device=dev)
        out = alloc_snapshots(nc, 1, T, device=dev)
    fill_field(data, xd, T, 1, wake["xc"], wake["yc"])
    tables.interpolate(data, pt.float32, out=out)
    pt.cuda.synchronize()
    e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        tables.interpolate(data, pt.float32, out=out)
    e1.record()
    pt.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    rows = data[pt.from_numpy(i_ref.reshape(-1)).to(dev)].cpu().numpy().reshape(len(sample), k, 1, T)
    ref = (w_ref[:, :, None, None] * rows).sum(1)
    scale = np.abs(rows).max(axis=1)
    got = out[pt.from_numpy(sample).to(dev)].cpu().numpy()
    assert (np.abs(got - ref) <= 1e-5 * np.maximum(scale, 1e-30)).all()
    # constant field and linearity on a thin slab
    slab = data[:, :, :8].contiguous()
    ones = pt.ones_like(slab)
    o1 = tables.interpolate(ones, pt.float32)
    assert (o1 - 1.0).abs().max().item() < 5e-6
    a = tables.interpolate(slab, pt.float32)
    b = tables.interpolate(slab * 2.0, pt.float32)
    normal = a.abs() > 1e-30          # power-of-two scaling commutes with rounding only outside the subnormal range
    if not pt.equal(b[normal], a[normal] * 2.0) or (b - 2.0 * a).abs().max().item() > 1e-37:
        bad = (b != a * 2.0) & normal
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"linearity violated at {int(bad.sum())} of {bad.numel()} values, e.g. {i}: "
                             f"{a[i].item()!r} {b[i].item()!r}; nan: {int(pt.isnan(a).sum())} {int(pt.isnan(b).sum())}")

    # ---- weighted SVD of the exported matrix (C5): device Gram vs an fp64 contraction, SVD identities
    svd_info = None
    if args.svd or args.name == "C5":
        from sparsespatialsampling_b200 import svd as s3svd
        del data
        a2 = out.reshape(nc, T).contiguous()
        area = pt.pow(width / pt.pow(2.0, sc.levels.to(device=dev, dtype=pt.float64).reshape(-1)), d).to(pt.float32)
        mean = s3svd.row_means(a2)
        times = {}
        for method in ("tc3", "tc", "simt"):
            g = s3svd.gram(a2, mean, area, 1, method)
            pt.cuda.synchronize()
            g0, g1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
            g0.record()
            g = s3svd.gram(a2, mean, area, 1, method)
            g1.record()
            pt.cuda.synchronize()
            times[method] = g0.elapsed_time(g1)
            if method == "tc3":
                g_tc3 = g
        # fp64 Gram in row chunks (the fp64 copy of the whole matrix would not be needed at once)
        g_ref = pt.zeros((T, T), dtype=pt.float64, device=dev)
        for r0 in range(0, nc, 65536):
            b = (a2[r0:r0 + 65536] - mean[r0:r0 + 65536, None]).double() * area[r0:r0 + 65536].sqrt().double()[:, None]
            g_ref += b.T @ b
        scale = pt.sqrt(pt.outer(pt.diag(g_ref), pt.diag(g_ref))).clamp_min(1e-300)
        gram_err = float(((g_tc3 - g_ref).abs() / scale).max())
        assert gram_err <= 5e-6, gram_err
        s3svd.compute_svd(a2, area, rank=50, n_modes=10)      # first call: one-time cuSOLVER initialisation
        pt.cuda.synchronize()
        t0 = time.time()
        s_val, u, v = s3svd.compute_svd(a2, area, rank=50, n_modes=10)
        pt.cuda.synchronize()
        t_svd = time.time() - t0
        lam = pt.linalg.eigvalsh(g_ref).flip(0).clamp_min(0).sqrt()[:50]
        big = lam > 1e-2 * lam[0]
        assert float(((s_val.double() - lam).abs() / lam)[big].max()) <= 1e-4
        # weighted modes are orthonormal (the synthetic wake has only a handful of coherent modes: check those)
        n_sig = max(1, min(10, int((lam > 1e-3 * lam[0]).sum())))
        uw = u[:, :n_sig].double() * area.sqrt().double()[:, None]
        ortho = float((uw.T @ uw - pt.eye(n_sig, dtype=pt.float64, device=dev)).abs().max())
        assert ortho <= 1e-3, ortho
        assert float((v.double().T @ v.double() - pt.eye(50, dtype=pt.float64, device=dev)).abs().max()) <= 1e-5
        flop = 2.0 * nc * T * T
        svd_info = {"matrix": [int(nc), T], "gram_ms": times, "gram_useful_tflops_tc3": flop / times["tc3"] / 1e9,
                    "gram_max_rel_err_vs_fp64": gram_err, "compute_svd_s_rank50_10_modes": t_svd,
                    "mode_orthonormality_err": ortho, "significant_modes": n_sig, "s_rel_err_top": float(((s_val.double() - lam).abs() / lam)[big].max())}

    # ---- host-to-host export of a 256-snapshot batch: pitched DMA of all rows vs PCIe gather of the referenced rows
    e2e_info = None
    if args.e2e:
        te = min(256, T)
        host = out.new_empty((x.size(0), 1, te), device="cpu").pin_memory()
        host.copy_(synth.wake_field(xd, 0, te, te, 1, wake["xc"], wake["yc"]))
        res_h, e2e_info = None, {"snapshots": te, "referenced_fraction": int(pt.unique(tables.idx_sorted).numel()) / x.size(0)}
        for label, g in (("dma", False), ("gather", True)):
            res_h = tables.interpolate_host(host, out=res_h, gather=g)
            pt.cuda.synchronize()
            t0 = time.time()
            for _ in range(3):
                tables.interpolate_host(host, out=res_h, gather=g)
            pt.cuda.synchronize()
            e2e_info[f"{label}_ms"] = (time.time() - t0) / 3 * 1e3
        want = tables.interpolate(host.to(dev), pt.float32).cpu()
        assert pt.equal(res_h, want)

    n_unique = int(pt.unique(tables.idx_sorted).numel())
    b_algo = n_unique * T * 4 + nc * T * 4 + nc * k * 8
    peak = 6542.7
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    if os.path.exists(p):
        peak = float(json.load(open(p))["hbm_gbs"])
    print(json.dumps({
        "config": args.name, "layout": "dense" if args.dense else "pitched", "tune": args.tune or None, "n_points": int(x.size(0)), "dim": d, "k": k, "snapshots": T, "n_cells": int(nc),
        "grid_gen_s": info["t_total"], "t_uniform": info["t_uniform"], "t_adaptive": info["t_adaptive"],
        "t_geometry": info["t_geometry"], "t_renumbering": info["t_renumbering"], "t_knn_build_gridgen": info["t_knn_build"],
        "setup_s": t_setup, "iterations": info["iterations"], "levels": [info["min_level"], info["max_level"]],
        "captured_metric": info["metric_per_iter"][-1], "export_knn_build_s": t_build, "export_tables_s": t_tables,
        "interp_ms": ms, "snapshot_points_per_s": nc * T / (ms * 1e-3), "unique_source_points": n_unique,
        "algorithmic_GBps": b_algo / (ms * 1e-3) / 1e9, "roofline_frac_of_measured": b_algo / (ms * 1e-3) / 1e9 / peak,
        "checks": "grid consistency, masks, knn idx/weights, interpolation tolerance, constant, linearity: ok",
        "svd": svd_info, "e2e_256_snapshots": e2e_info,
    }))


if __name__ == "__main__":
    # the STL body and the grid files are written to a directory of this run, removed at the end
    with tempfile.TemporaryDirectory(prefix="s3b200_cfg_") as tmp:
        main(tmp)

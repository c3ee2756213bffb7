"""
Reconstruction error of a sampled grid (ReconstructionError / s3_recon_error) on the C2 and C4 workloads, against the
unfused composition (``reconstruct`` followed by torch fp64 reductions) on the same inputs.

  python scripts/recon_bench.py [--workloads C2,C4] [--steps K] [--warmup W] [--out FILE]

  C2: the bench grid (bench.py: ~99k points, uniform level 5, min_metric 0.75), k = 8, T = 1000, p (D = 1) and U (D = 2),
      pitched layout.
  C4: the 10M-point 3-D cloud of scripts/scale_c4.py (n_cells_max 500 000), k = 26, T = 2000, the scalar wake field
      generated on the device. The unfused composition needs [N, D, T] fp32 and fp64 temporaries that do not fit beside
      the 80 GB field, so both are compared on the window T = [0, 500) there; the fused kernel is also timed on all T.

The sampled field is what the export computes (KnnTables over the original points, fp32). Per workload and field one
JSON line goes to stdout and is appended to ``--out``, with the card name and power limit read in the same run:
  tables_s        ReconstructionError construction: KNN index over the Nc centres, N queries, Morton order (wall clock);
  fused_ms        one s3_recon_error call (CUDA events, after warm-up; the working set is several times the 126 MB L2);
  B_algo          N*D*T*4 + U_c*D*T*4 + N*k*8 + N*D*16 bytes (original once, the U_c distinct referenced cells once, the
                  tables, the point map read and written), roofline_frac = B_algo / fused time / MEASURED_PEAKS hbm_gbs;
  extra_bytes     scratch written and read again (DESIGN.md 3.4): 2 * (n_blocks * D * T * 24 + n_tiles * N * D * 8), plus
                  2 * n_groups * D * T * 24 when there are more than 256 blocks;
  unfused_ms      reconstruct + torch fp64 reductions; parity of the two (max_abs bit-exact, sums within 1e-12).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch as pt

import synth
import sparsespatialsampling_b200 as s3
from bench import measured_peak, geometries, GRID_KW
from sparsespatialsampling_b200.export import KnnTables
from sparsespatialsampling_b200.interpolate import alloc_snapshots
from sparsespatialsampling_b200.knn import KnnIndex
from sparsespatialsampling_b200.reconstruction import recon_error

BLOCK, TILE, GROUP = 512, 256, 256           # csrc/interp.cu: kReconBlock, kReconTile, kReconGroup


def card():
    info = {"gpu": pt.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception:
        pass
    return info


def extra_bytes(n, d, t):
    n_blocks = -(-n // BLOCK)
    n_tiles = -(-t // TILE)
    n_groups = -(-n_blocks // GROUP)
    extra = 2 * (n_blocks * d * t * 24 + n_tiles * n * d * 8)
    if n_groups > 1:
        extra += 2 * n_groups * d * t * 24
    return extra


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    pt.cuda.synchronize()
    e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    pt.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def unfused(rec, original, sampled):
    """reconstruct, then torch fp64 reductions; in-place where possible so that C4 windows fit beside the field."""
    e = rec.reconstruct(sampled).double()
    e.sub_(original)
    max_abs = pt.linalg.vector_norm(e, float("inf"), dim=0)
    e.square_()
    sq_err, point = e.sum(0), e.sum(2)
    e.copy_(original)
    e.square_()
    return sq_err, e.sum(0), max_abs, point


def fused(rec, original, sampled, point):
    return recon_error(original, sampled, rec.tables, point)


def compare(rec, original, sampled, steps, warmup):
    """(fused ms, unfused ms, parity) on the same window."""
    point = pt.zeros((rec.n_points, original.size(1)), dtype=pt.float64, device=original.device)
    f = fused(rec, original, sampled, point)
    u = unfused(rec, original, sampled)
    rel = lambda a, b: float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())
    parity = {"max_abs_bit_exact": bool(pt.equal(f[2], u[2])), "sq_err_rel": rel(f[0], u[0]),
              "sq_ref_rel": rel(f[1], u[1]), "point_sq_err_rel": rel(point, u[3])}
    parity["ok"] = parity["max_abs_bit_exact"] and max(parity["sq_err_rel"], parity["sq_ref_rel"],
                                                       parity["point_sq_err_rel"]) <= 1e-12
    del u
    t_f = time_ms(lambda: fused(rec, original, sampled, point), steps, warmup)
    t_u = time_ms(lambda: unfused(rec, original, sampled), max(1, steps // 2), 1)
    return t_f, t_u, parity


def record(workload, field, rec, n, d, t, k, t_fused, extra_info, peak):
    u_c = int(pt.unique(rec.tables.idx_sorted).numel())
    b_algo = n * d * t * 4 + u_c * d * t * 4 + n * k * 8 + n * d * 16
    ex = extra_bytes(n, d, t)
    line = {"workload": workload, "field": field, "n_points": n, "n_cells": rec.n_cells, "k": k, "D": d, "T": t,
            "distinct_cells_referenced": u_c, "fused_ms": t_fused, "B_algo": b_algo,
            "algorithmic_GBps": b_algo / (t_fused * 1e-3) / 1e9, "hbm_gbs_peak": peak[0], "peak_source": peak[1],
            "roofline_frac": b_algo / (t_fused * 1e-3) / 1e9 / peak[0], "extra_bytes": ex,
            "extra_frac_of_B_algo": ex / b_algo}
    line.update(extra_info)
    return line


def run_c2(args, dev, tmp, peak, hw):
    n_snap = synth.CONFIGS["C2"][1]
    x = synth.cylinder2d_cloud(synth.CONFIGS["C2"][0], seed=0)
    xd = x.to(dev)
    sc = s3.SparseSpatialSampling(x, synth.wake_metric(xd).cpu(), geometries(s3.geometry), tmp, "c2",
                                  uniform_levels=GRID_KW["uniform_level"], min_metric=GRID_KW["min_metric"])
    sc.execute_grid_generation()
    export = KnnTables(KnnIndex(xd), sc.centers.to(dev), 8)
    s3.ReconstructionError(sc, xd, device=dev)                    # first construction: one-off module / pool set-up
    pt.cuda.synchronize()
    t0 = time.time()
    rec = s3.ReconstructionError(sc, xd, device=dev)
    pt.cuda.synchronize()
    t_tables = time.time() - t0
    lines = []
    for field, d in (("p", 1), ("U", 2)):
        original = alloc_snapshots(xd.size(0), d, n_snap, device=dev)
        original.copy_(synth.wake_field(xd, 0, n_snap, n_snap, d))
        sampled = alloc_snapshots(rec.n_cells, d, n_snap, device=dev)
        export.interpolate(original, pt.float32, out=sampled)
        t_f, t_u, parity = compare(rec, original, sampled, args.steps, args.warmup)
        lines.append(record("C2", field, rec, rec.n_points, d, n_snap, 8, t_f,
                            dict(layout="pitched", tables_s=t_tables, unfused_ms=t_u, unfused_T=n_snap,
                                 fused_over_unfused_speedup=t_u / t_f, parity=parity, **hw), peak))
        del original, sampled
    return lines


def run_c4(args, dev, tmp, peak, hw):
    from run_config import config, fill_field
    if args.points:
        synth.CONFIGS["C4"] = (args.points,) + tuple(synth.CONFIGS["C4"][1:])
    x, geoms, wake, grid_kw = config("C4", 0)
    n_snap, k, t_win = synth.CONFIGS["C4"][1], 26, 500
    xd = x.to(dev)
    sc = s3.SparseSpatialSampling(x, synth.wake_metric(xd, xc=wake["xc"], yc=wake["yc"]).cpu(), geoms, tmp, "c4",
                                  **grid_kw)
    sc.execute_grid_generation()
    original = alloc_snapshots(xd.size(0), 1, n_snap, device=dev)
    fill_field(original, xd, n_snap, 1, wake["xc"], wake["yc"])
    sampled = alloc_snapshots(sc.centers.size(0), 1, n_snap, device=dev)
    KnnTables(KnnIndex(xd), sc.centers.to(dev), k).interpolate(original, pt.float32, out=sampled)
    pt.cuda.synchronize()
    t0 = time.time()
    rec = s3.ReconstructionError(sc, xd, device=dev)
    pt.cuda.synchronize()
    t_tables = time.time() - t0
    point = pt.zeros((rec.n_points, 1), dtype=pt.float64, device=dev)
    t_full = time_ms(lambda: fused(rec, original, sampled, point), args.steps, args.warmup)
    t_f, t_u, parity = compare(rec, original[:, :, :t_win], sampled[:, :, :t_win], args.steps, args.warmup)
    n = rec.n_points
    u_c = int(pt.unique(rec.tables.idx_sorted).numel())
    b_win = n * t_win * 4 + u_c * t_win * 4 + n * k * 8 + n * 16
    return [record("C4", "p", rec, n, 1, n_snap, k, t_full,
                   dict(layout="pitched", tables_s=t_tables, unfused_T=t_win, window_fused_ms=t_f, unfused_ms=t_u,
                        window_roofline_frac=b_win / (t_f * 1e-3) / 1e9 / peak[0],
                        window_extra_frac_of_B_algo=extra_bytes(n, 1, t_win) / b_win,
                        fused_over_unfused_speedup=t_u / t_f, parity=parity, **hw), peak)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C2,C4")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--points", type=int, default=0, help="C4: smaller cloud for quick checks")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "recon_bench.jsonl"))
    args = ap.parse_args()
    dev = pt.device("cuda", 0)
    pt.cuda.set_device(dev)
    peak, hw = measured_peak(), card()
    runners = {"C2": run_c2, "C4": run_c4}
    with tempfile.TemporaryDirectory(prefix="s3b200_recon_") as tmp:
        for name in args.workloads.split(","):
            for line in runners[name](args, dev, tmp, peak, hw):
                print(json.dumps(line), flush=True)
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
            pt.cuda.empty_cache()


if __name__ == "__main__":
    main()

"""
compute_dmd phase times and the fused low-rank error kernel (s3_lowrank_error) against the unfused torch composition.

  python scripts/dmd_bench.py [--out FILE] [--reps N]

  phases: compute_dmd on C2-sized p ([99k, 1000]), C2-sized U ([99k, 2, 1000]) and a C5-sized [582k, 2000] matrix,
          random low-rank-plus-noise fields; Gram, eigen (eigh / eig / amplitude algebra) and modes timed separately
          with CUDA events after a warm-up call (rank 50, all modes).
  kernel: s3_lowrank_error on the C5-sized matrix at q in {20, 100, 256, 512}, mean and volume on, row map on.
          B_algo = m*t*4 + (m + t)*q*4 + m*4 + vol_div*t*24 + m*16; roofline_frac = B_algo / time / 7.7 TB/s.
          unfused = fp32 matmul left @ right_t^T, then fp64 reductions of (a - mean - L R^T) in torch, same inputs.
One JSON line per measurement goes to stdout and is appended to --out, with the card name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch as pt

from sparsespatialsampling_b200 import svd
from sparsespatialsampling_b200.dmd import compute_dmd

HBM_GBS = 7700.0


def card():
    info = {"gpu": pt.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception:
        pass
    return info


def timed(fn, reps):
    fn()
    pt.cuda.synchronize()
    t0, t1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        out = fn()
    t1.record()
    pt.cuda.synchronize()
    return t0.elapsed_time(t1) / reps, out


def field(n, d, t, seed):
    g = pt.Generator(device="cuda").manual_seed(seed)
    shape = (n, t) if d is None else (n, d, t)
    rows = n * (d or 1)
    a = (pt.randn((rows, 60), device="cuda", generator=g) @ pt.randn((60, t), device="cuda", generator=g)
         + 0.01 * pt.randn((rows, t), device="cuda", generator=g)).reshape(shape)
    return a, pt.rand((n,), device="cuda", generator=g) + 0.5


def phases(name, n, d, t, reps, emit):
    a, area = field(n, d, t, 1)
    rows = n * (d or 1)
    a2 = a.reshape(rows, t)
    zero = pt.zeros((rows,), device="cuda")
    vol_div = d or 1
    gram_ms, g = timed(lambda: svd.gram(a2, zero, area, vol_div), reps)
    total_ms, dmd = timed(lambda: compute_dmd(a, area, 0.01, rank=50), max(1, reps // 2))
    coef = pt.zeros((t, 2 * dmd.n_modes), device="cuda")
    modes_ms, _ = timed(lambda: svd.project_tc(a2, zero, area, vol_div, coef), reps)
    emit({"kind": "compute_dmd", "workload": name, "shape": list(a.shape), "rank": dmd.rank, "total_ms": total_ms,
          "gram_ms": gram_ms, "modes_ms": modes_ms, "eigen_ms": total_ms - gram_ms - modes_ms})
    del a, a2


def kernel(reps, emit):
    m, t = 582000, 2000
    a, area = field(m, None, t, 2)
    mean = svd.row_means(a)
    g = pt.Generator(device="cuda").manual_seed(3)
    for q in (20, 100, 256, 512):
        left = pt.randn((m, q), device="cuda", generator=g) / q
        right_t = pt.randn((t, q), device="cuda", generator=g)
        row = pt.zeros((m,), dtype=pt.float64, device="cuda")
        fused_ms, fused = timed(lambda: svd.lowrank_error(a, left, right_t, mean, area, 1, row), reps)

        def unfused():
            e = (a - mean[:, None]) - left @ right_t.T
            e64 = e.double()
            w = area.double()[:, None]
            x = (a.double() - mean.double()[:, None])
            return (w * e64 * e64).sum(0), (w * x * x).sum(0), e64.abs().max(0).values, (e64 * e64).sum(1)
        unfused_ms, ref = timed(unfused, max(1, reps // 4))
        b_algo = m * t * 4 + (m + t) * q * 4 + m * 4 + t * 24 + m * 16
        rel = float(((fused[0][0] - ref[0]).abs() / ref[1].clamp_min(1e-300)).max())
        emit({"kind": "lowrank_error", "m": m, "t": t, "q": q, "fused_ms": fused_ms, "B_algo": b_algo,
              "achieved_gbs": b_algo / fused_ms / 1e6, "roofline_frac": b_algo / fused_ms / 1e6 / HBM_GBS,
              "tf32x3_tflops": 6.0 * m * t * q / fused_ms / 1e9, "unfused_ms": unfused_ms,
              "speedup": unfused_ms / fused_ms, "max_rel_diff_sq_err": rel})
        del left, right_t, ref


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    info = card()

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    for name, n, d, t in (("C2 p", 99000, None, 1000), ("C2 U", 99000, 2, 1000), ("C5", 582000, None, 2000)):
        phases(name, n, d, t, args.reps, emit)
    kernel(args.reps, emit)


if __name__ == "__main__":
    main()

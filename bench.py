#!/usr/bin/env python
"""
bench.py -- headline benchmark of the S^3 hot path on B200.

Metric (BASELINE.json): snapshot-points interpolated per second (export-stage interpolation of every original
snapshot onto the sampled grid), with the grid-generation seconds and the HBM roofline fraction beside it.

Workload: C2 (cylinder2D_Re100-sized: ~100k points, 1000 snapshots, p[D=1] + U[D=2] export). One "step" = one pass of
the export interpolation over that batch. With N GPUs the SAME batch is sharded by snapshot window
(`parallel.snapshot_window`: rank r interpolates T/N snapshots of all cells) -- strong scaling; the sampled grid and
the KNN tables are computed on rank 0 and broadcast over NCCL once, there is no collective inside the step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl s3b200|reference] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...                     (one rank per GPU)

`--dump-outputs DIR` writes what the last timed step computed as DIR/p.npy [n, 1, T] and DIR/U.npy [n, 2, T] (float32)
for a fixed, seeded sample of n grid cells (at most 64 MB in all). The inputs are seeded, so two builds of the project
can be compared output for output.

`--impl reference` times the reference's own CPU `interpolate_data` (unmodified, from oracle/_ref; the oracle port if
that install is missing) with all host threads on the same workload.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch as pt

import synth

METRIC = "snapshot_points_interpolated_per_s"
UNIT = "snapshot-points/s"
WORKLOAD = "C2: cylinder2D_Re100-sized synthetic field (~100k pts, 1000 snapshots, p/U export)"
N_POINTS, N_SNAP = synth.CONFIGS["C2"][0], synth.CONFIGS["C2"][1]
GRID_KW = dict(uniform_level=5, min_metric=0.75)
K_NEIGHBORS = 8
L2_BYTES = 126e6
DUMP_BYTES = 64 * 10**6


def geometries(geo):
    return [geo.CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
            geo.SphereGeometry("cylinder", False, synth.CYL2D["pos"], synth.CYL2D["radius"], refine=True)]


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs. The region is a few milliseconds long, so
    NVML is polled directly from a thread (about one sample per millisecond); nvidia-smi -lms 200 is the fallback."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop, self._thread, self._how = threading.Event(), None, None

    def _poll_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            entry = visible.split(",")[self.index].strip() if visible else str(self.index)
            h = (pynvml.nvmlDeviceGetHandleByIndex(int(entry)) if entry.isdigit()
                 else pynvml.nvmlDeviceGetHandleByUUID(entry))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self._how = "nvml"
            self._ready.set()
            while not self._stop.is_set():
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                bits = int(reasons_fn(h))
                for name, bit in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
                time.sleep(0.0005)
        finally:
            pynvml.nvmlShutdown()

    def _poll_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self._how = "nvidia-smi"
        self._ready.set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            line = proc.stdout.readline()
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                try:
                    self.samples.append(float(parts[0]))
                    self.max_mhz = float(parts[1])
                except ValueError:
                    continue
                for nm, val in zip(names, parts[2:6]):
                    if val.lower().startswith("active"):
                        self.reasons.add(nm)
        proc.terminate()

    def _run(self):
        try:
            self._poll_nvml()
        except Exception:
            try:
                self._poll_smi()
            except Exception:
                self._ready.set()

    def __enter__(self):
        self._ready = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        self._ready.wait(timeout=10)
        self.samples.clear()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=3)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0, "how": self._how}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "how": self._how}


def algorithmic_bytes(n_unique, n_cells, k, comps, t, out_bytes=4):
    """SURVEY.md 8(d): unique source rows read once + result written once + the (idx, w) tables."""
    return n_unique * comps * t * 4 + n_cells * comps * t * out_bytes + n_cells * k * 8


def all_host_threads():
    """Lift a NUMA / torchrun restriction for the CPU legs: every core of the box, every torch intra-op thread."""
    n = os.cpu_count() or 1
    try:
        os.sched_setaffinity(0, range(n))
    except OSError:
        pass
    pt.set_num_threads(n)
    return n


def reference_gridgen_record():
    """The reference's own SamplingTree.refine() timed on a B200 host (scripts/ref_gridgen.py, run under gpurun) and in
    the build container (tests/golden/config_C2.npz) -- context for grid_gen_s; the grids are bit-identical
    (tests/test_gridgen_gpu.py)."""
    out = {}
    p = os.path.join(ROOT, "profiles", "r2_ref_gridgen_b200.json")
    if os.path.exists(p):
        with open(p) as f:
            out["b200_host"] = json.load(f)
    p = os.path.join(ROOT, "tests", "golden", "config_C2.npz")
    if os.path.exists(p):
        g = np.load(p)
        out["build_container_C2"] = {"t_total_s": float(g["reference_t_total"]), "n_cells": int(g["n_cells"]),
                                     "iterations": int(g["iterations"]), "where": "8 vCPU build container, n_jobs=8"}
    return out or None


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_interpolation(w64, idx64, fields, budget_s, full_t):
    """
    Time the reference's interpolate_data (export.py:446-468) on `fields` (list of [N, D, T] fp32 host tensors).
    Returns (callable(ts) -> seconds for one pass over the first ts snapshots, kind, description).
    """
    from oracle import reference
    ref = reference.load()
    if ref is not None:
        from sparseSpatialSampling.export import interpolate_data as fn
        kind, what = "reference", "sparseSpatialSampling.export.interpolate_data (unmodified reference, oracle/_ref)"
    else:
        from oracle import s3_oracle as orc
        fn = orc.interpolate_torch
        kind, what = "port", "oracle.interpolate_torch (port of export.py:446-468; oracle/_ref not installed)"

    def one_pass(ts):
        sl = [f[:, :, :ts].contiguous() for f in fields]
        t0 = time.time()
        for f in sl:
            fn(w64, idx64, f, 100000)
        return time.time() - t0
    return one_pass, kind, what


def pick_sample(one_pass, full_t, budget_s):
    """Largest snapshot count (multiple of 8, <= full_t) whose pass fits `budget_s`, from a 16-snapshot probe."""
    one_pass(8)
    probe = one_pass(16)
    rate = 16.0 / max(probe, 1e-6)
    ts = int(min(full_t, max(8, (rate * budget_s) // 8 * 8)))
    return ts


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = all_host_threads()
    from oracle import s3_oracle as orc

    class _G:      # tiny geometry shells with the attributes the oracle reads
        pass
    dom, cyl = _G(), _G()
    dom.type, dom.keep_inside, dom.refine, dom.min_refinement_level = "cube", True, False, None
    dom._lower_bound, dom._upper_bound = synth.CYL2D["lower"], synth.CYL2D["upper"]
    dom.main_width, dom.center = 2.2, np.array([1.1, 0.205])
    cyl.type, cyl.keep_inside, cyl.refine, cyl.min_refinement_level = "sphere", False, True, None
    cyl._position, cyl._radius = synth.CYL2D["pos"], synth.CYL2D["radius"]
    cyl.main_width, cyl.center = 0.05, np.array(synth.CYL2D["pos"])

    x = synth.cylinder2d_cloud(N_POINTS, seed=0)
    m = synth.wake_metric(x)
    # the sampled grid: oracle port of SamplingTree.refine (10 s); the reference itself needs minutes for this case and
    # produces the same grid -- checked here against the digest of the reference's own run (tests/golden)
    t0 = time.time()
    tree = orc.OracleTree(x.numpy(), m.numpy(), [dom, cyl], **GRID_KW, sdm_order=1).refine()
    t_grid = time.time() - t0
    nc = tree.all_centers.shape[0]
    same_grid = None
    gp = os.path.join(ROOT, "tests", "golden", "config_C2.npz")
    if os.path.exists(gp):
        same_grid = bool(hashlib.sha256(np.ascontiguousarray(tree.all_centers).tobytes()).hexdigest()
                         == str(np.load(gp)["centers_sha"]))
    # KNN cache exactly as ExportData._build_knn_cache (export.py:423-436)
    from sklearn.neighbors import NearestNeighbors
    t0 = time.time()
    dist, idx = NearestNeighbors(n_neighbors=K_NEIGHBORS, n_jobs=cores).fit(x.numpy()).kneighbors(tree.all_centers)
    w = 1.0 / pt.clamp(pt.from_numpy(dist), min=1e-12)
    w /= w.sum(axis=1, keepdim=True)
    t_knn = time.time() - t0
    idx = pt.from_numpy(idx)
    p = synth.wake_field(x, 0, N_SNAP, N_SNAP, 1)
    u = synth.wake_field(x, 0, N_SNAP, N_SNAP, 2)
    one_pass, kind, what = cpu_interpolation(w, idx, [p, u], None, N_SNAP)
    # the whole run (warm-up + K steps) has to end within a few minutes: bound the snapshots per step accordingly
    budget = 150.0 / max(args.steps + args.warmup, 1)
    ts = N_SNAP if args.full else pick_sample(one_pass, N_SNAP, budget)
    for _ in range(args.warmup):
        one_pass(ts)
    t0 = time.time()
    for _ in range(args.steps):
        one_pass(ts)
    dt = (time.time() - t0) / max(args.steps, 1)
    value = nc * 3 * ts / dt
    sample = (f"all {N_SNAP} snapshots of p and U per step" if ts == N_SNAP else
              f"{ts} of {N_SNAP} snapshots of p and U per step (cost is linear in T; bounded so that "
              f"{args.steps}+{args.warmup} steps end within minutes)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_points": int(x.shape[0]), "n_cells": int(nc), "k": K_NEIGHBORS,
                   "fields": "p[D=1] + U[D=2]", "snapshots_per_step": ts, "snapshots_total": N_SNAP,
                   "same_grid_as_reference_run": same_grid},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{sample}; {what}, torch CPU, {pt.get_num_threads()} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "grid_gen_s": t_grid, "grid_gen_note": "oracle port of SamplingTree.refine on the host (no process pool)",
        "grid_gen_reference": reference_gridgen_record(),
        "knn_tables_s": t_knn, "host_cores": os.cpu_count(),
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, tmp_dir):
    import torch.distributed as dist
    import sparsespatialsampling_b200 as s3
    from sparsespatialsampling_b200 import _lib
    from sparsespatialsampling_b200.export import ExportData, KnnTables
    from sparsespatialsampling_b200.interpolate import alloc_snapshots
    from sparsespatialsampling_b200.knn import KnnIndex
    from sparsespatialsampling_b200.parallel import bind_to_gpu_numa_node, broadcast_grid, snapshot_window

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # native libraries (NCCL's version banner) write to fd 1: keep stdout for the one JSON line
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    pt.cuda.set_device(local)
    dev = pt.device("cuda", local)
    # host cores + pinned buffers on the NUMA node of this rank's GPU (the e2e leg moves every byte over PCIe)
    numa_cores = None if args.no_numa_bind else bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    for kv in [t for t in args.tune.split(",") if t]:
        key, val = kv.split("=")
        _lib.tune(int(key), int(val))

    def barrier():
        if world > 1:
            dist.barrier()
        pt.cuda.synchronize()

    def max_over_ranks(v):
        t = pt.tensor([v], device=dev, dtype=pt.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- inputs (seeded, identical on every rank)
    x = synth.cylinder2d_cloud(N_POINTS, seed=0)
    xd = x.to(dev)
    metric = synth.wake_metric(xd).cpu()
    k = K_NEIGHBORS

    # ---- grid generation on rank 0 (replicas only: the loop is sequential), then broadcast grid + tables
    grid_info, t_grid_wall, grid_cold, sc, centers, tables, t_tables = None, None, None, None, None, None, None
    if rank == 0:
        # two runs: the first pays one-off costs of the process (module load, first cooperative launch, memory pools),
        # the second is the steady-state number reported as grid_gen_s; both produce the same grid
        for attempt in range(2):
            t0 = time.time()
            sc = s3.SparseSpatialSampling(x, metric, geometries(s3.geometry), tmp_dir, "c2", **{
                "uniform_levels": GRID_KW["uniform_level"], "min_metric": GRID_KW["min_metric"]})
            sc.execute_grid_generation()
            pt.cuda.synchronize()
            t_grid_wall = time.time() - t0
            grid_info = sc.mesh_info
            if attempt == 0:
                grid_cold = {"t_total": grid_info["t_total"], "wall_incl_setup_s": t_grid_wall}
        centers = sc.centers.to(dev)
        t0 = time.time()
        tables = KnnTables(KnnIndex(xd), centers, k)
        pt.cuda.synchronize()
        t_tables = time.time() - t0
    barrier()
    if world > 1:        # NCCL builds its broadcast channels on first use (20-35 ms on an 8-GPU box), per message
        # size class: not the tables' cost -- one untimed broadcast of the same size first
        KnnTables.share(tables, dev, src=0)
    barrier()
    b0, b1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
    b0.record()
    centers = broadcast_grid(centers, 2, dev, src=0)
    # NCCL over NVLink: every rank uses rank 0's tables (one packed broadcast; n, k known from the grid broadcast)
    tables = KnnTables.share(tables, dev, src=0, n=int(centers.size(0)), k=k)
    b1.record()
    barrier()
    bcast_ms = max_over_ranks(b0.elapsed_time(b1)) if world > 1 else 0.0
    n_cells = int(centers.size(0))
    n_unique = int(pt.unique(tables.idx_sorted).numel())

    # ---- this rank's snapshot window of the ONE batch, resident in HBM. Layout: rows padded to a multiple of 128 bytes
    # (interpolate.alloc_snapshots, DESIGN.md 2); the dense [N, D, T] layout of the reference is timed beside it
    t_lo, t_hi = snapshot_window(N_SNAP, world, rank)
    ts = t_hi - t_lo
    p_dense = synth.wake_field(xd, t_lo, t_hi, N_SNAP, 1)
    u_dense = synth.wake_field(xd, t_lo, t_hi, N_SNAP, 2)
    step_bytes = (p_dense.numel() + u_dense.numel()) * 4 + n_cells * 3 * ts * 4
    n_rot = int(min(8, max(1, -(-int(3 * L2_BYTES) // step_bytes))))      # rotate buffer sets so that re-use distance > L2

    def make_sets(pitched, out_dtype):
        sets = []
        for _ in range(n_rot):
            if pitched:
                p = alloc_snapshots(xd.size(0), 1, ts, device=dev, zero=True); p.copy_(p_dense)
                u = alloc_snapshots(xd.size(0), 2, ts, device=dev, zero=True); u.copy_(u_dense)
                op = alloc_snapshots(n_cells, 1, ts, dtype=out_dtype, device=dev)
                ou = alloc_snapshots(n_cells, 2, ts, dtype=out_dtype, device=dev)
            else:
                p, u = p_dense.clone(), u_dense.clone()
                op = pt.empty((n_cells, 1, ts), dtype=out_dtype, device=dev)
                ou = pt.empty((n_cells, 2, ts), dtype=out_dtype, device=dev)
            sets.append((p, u, op, ou))
        return sets

    def timed(sets, out_dtype, steps, warmup, clocks=False):
        def step(i):
            p, u, op, ou = sets[i % len(sets)]
            tables.interpolate(p, out_dtype, out=op)
            tables.interpolate(u, out_dtype, out=ou)
        for i in range(warmup):
            step(i)
        barrier()
        e0, e1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
        sampler = ClockSampler(local) if clocks else None
        if sampler:
            sampler.__enter__()
        barrier()
        pt.cuda.profiler.start()        # no-op unless run under `ncu --profile-from-start off`
        e0.record()
        for i in range(steps):
            step(i)
        e1.record()
        barrier()
        pt.cuda.profiler.stop()
        if sampler:
            sampler.__exit__()
        return max_over_ranks(e0.elapsed_time(e1)), (sampler.summary() if sampler else None)

    warmup = max(args.warmup, 3)
    sets = make_sets(True, pt.float32)
    launches0 = _lib.launch_count()
    ms_total, clocks = timed(sets, pt.float32, args.steps, warmup, clocks=True)
    launches = _lib.launch_count() - launches0 - 2 * warmup
    ms_step = ms_total / args.steps
    units_step = n_cells * 3 * N_SNAP                       # whole job: all ranks together interpolate the full batch
    # `value`: the K timed steps, as the bench contract defines it. The one-off broadcast of grid + tables (once per
    # ExportData object, whatever the number of fields / batches exported afterwards) is reported beside it, and as
    # `value_incl_table_broadcast` charged in full to these K steps.
    value = units_step / (ms_step * 1e-3)
    value_incl_bcast = units_step * args.steps / ((ms_total + bcast_ms) * 1e-3)
    out_p, out_u = sets[(args.steps - 1) % len(sets)][2:]          # the results of the last timed step
    check_p, check_u = out_p.clone(), out_u.clone()
    if args.dump_outputs:
        n_dump = min(n_cells, (DUMP_BYTES - 4096) // (3 * ts * 4))     # 4096: room for the two .npy headers
        rows = pt.from_numpy(np.sort(np.random.default_rng(0).choice(n_cells, n_dump, replace=False))).to(dev)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "p.npy"), out_p[rows].cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "U.npy"), out_u[rows].cpu().numpy())

    aux_steps = max(10, min(args.steps, 50))
    dense_sets = make_sets(False, pt.float32)
    ms_dense = timed(dense_sets, pt.float32, aux_steps, 3)[0] / aux_steps
    assert pt.equal(dense_sets[0][2], check_p) and pt.equal(dense_sets[0][3], check_u), "layouts disagree"
    del dense_sets
    f64_sets = make_sets(True, pt.float64)
    ms_f64 = timed(f64_sets, pt.float64, aux_steps, 3)[0] / aux_steps
    del f64_sets, sets

    # ---- end to end through the public API: this rank's host window in, host result out
    p_h = p_dense.cpu().pin_memory()
    u_h = u_dense.cpu().pin_memory()

    class _Grid:
        pass
    g = _Grid()
    g.n_dimensions, g.faces, g.vertices, g.levels = 2, None, None, None
    g.centers, g.metric, g.size_initial_cell = centers, metric, 2.2
    g.save_path, g.save_name, g.grid_name = tmp_dir, f"c2_rank{rank}", "grid"

    def e2e_run(async_host):
        exp = ExportData(g, write_times=[str(i) for i in range(N_SNAP)], write_files=False, device=dev,
                         async_host=async_host, distributed=world > 1)
        exp._tables_centers, exp._initialized_weights, exp._interpolated_metric = tables, True, True
        exp._stream_min_elements = 0

        def e2e_step():
            # host tensors in, host tensors out: ExportData streams windows of the time axis through the device
            # (pitched H2D copy | gather kernel | pitched D2H copy on three streams) and returns pinned host results
            exp.export(x, p_h, "p", n_snapshots_total=N_SNAP)
            r_p = exp._last_fields.centers
            exp.export(x, u_h, "U", n_snapshots_total=N_SNAP)
            r_u = exp.interpolated_fields.centers          # waits for all result copies
            return r_p, r_u
        for _ in range(3):           # the pinned result pool reaches its steady size (two buffers per field) here:
            res_p, res_u = e2e_step()    # the caller still holds the previous step's results when the next one starts
        assert not res_p.is_cuda and not res_u.is_cuda
        assert pt.equal(res_p, check_p.cpu()) and pt.equal(res_u, check_u.cpu()), "streamed export differs from the resident path"
        n = max(2, min(args.steps, 8))
        barrier()
        t0 = time.time()
        for _ in range(n):
            res_p, res_u = e2e_step()
        barrier()
        return max_over_ranks((time.time() - t0) * 1e3 / n), res_p, res_u
    e2e_ms, res_p, res_u = e2e_run(False)                 # default API semantics (fresh results, input released)
    e2e_async_ms, _, _ = e2e_run(True)
    e2e_value = units_step / (e2e_ms * 1e-3)
    # bytes that cross PCIe on THIS rank: the whole window with the DMA path, only the referenced source rows when
    # the ingest kernel gathers them (chosen when less than 60 % of the points are referenced; not the case on C2)
    h2d = (n_unique if n_unique < 0.6 * x.shape[0] else x.shape[0]) * 3 * ts * 4
    d2h = res_p.numel() * 4 + res_u.numel() * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- optional last stage of the path: sqrt(area)-weighted SVD of the exported p matrix [Nc, T_s] (rank 0 only)
    svd_info = None
    if not args.no_svd:
        from sparsespatialsampling_b200 import svd as s3svd
        area = pt.pow(2.2 / pt.pow(2.0, sc.levels.to(device=dev, dtype=pt.float64).reshape(-1)), 2).to(pt.float32)
        a2 = check_p.reshape(n_cells, ts).contiguous()
        mean = s3svd.row_means(a2)
        svd_ms = {}
        for method in ("tc3", "simt"):
            s3svd.gram(a2, mean, area, 1, method)
            pt.cuda.synchronize()
            g0, g1 = pt.cuda.Event(enable_timing=True), pt.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(3):
                s3svd.gram(a2, mean, area, 1, method)
            g1.record()
            pt.cuda.synchronize()
            svd_ms[method] = g0.elapsed_time(g1) / 3
        r = min(20, ts)
        s3svd.compute_svd(a2, area, rank=r)               # first call: one-time solver initialisation
        pt.cuda.synchronize()
        t0 = time.time()
        s_val, _, _ = s3svd.compute_svd(a2, area, rank=r)
        pt.cuda.synchronize()
        t_svd = time.time() - t0
        gram_flop = 2.0 * n_cells * ts * ts
        svd_info = {"matrix": [n_cells, ts], "gram_ms_tcgen05_3xtf32": svd_ms["tc3"],
                    "gram_ms_fp32_cuda_cores": svd_ms["simt"],
                    "gram_useful_tflops": gram_flop / (svd_ms["tc3"] * 1e-3) / 1e12,
                    "compute_svd_s": t_svd, "rank": r, "s0": float(s_val[0])}

    # ---- roofline of the dominant kernel (the interpolation kernel; a step is two launches of it), per GPU
    def b_algo(out_bytes=4):
        return (algorithmic_bytes(n_unique, n_cells, k, 1, ts, out_bytes) +
                algorithmic_bytes(n_unique, n_cells, k, 2, ts, out_bytes))
    peak, peak_src = measured_peak()
    achieved = b_algo() / (ms_step * 1e-3) / 1e9
    naive_bytes = sum(n_cells * k * comps * ts * 4 + n_cells * comps * ts * 4 + n_cells * k * 8 for comps in (1, 2))
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tp) and world == 1:
        with open(tp) as f:
            tj = json.load(f)
        traffic, traffic_src = tj.get("interp_dram_bytes_per_step"), tj.get("source")

    # ---- CPU baseline beside it (rank 0, N=1 only): the reference's own interpolate_data on all host cores
    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        cores = all_host_threads()
        w64 = tables.w64.cpu()
        idx64 = tables.idx.cpu().to(pt.int64)
        one_pass, kind, what = cpu_interpolation(w64, idx64, [p_h, u_h], None, N_SNAP)
        n_t = pick_sample(one_pass, N_SNAP, 8.0)
        reps = 2
        dt = min(one_pass(n_t) for _ in range(reps))
        cpu_baseline = {"value": n_cells * 3 * n_t / dt, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": f"{n_t} of {N_SNAP} snapshots of p and U (cost is linear in T), best of {reps} passes; "
                                  f"{what}, torch CPU, {pt.get_num_threads()} threads",
                        "seconds_per_pass": dt}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_points": int(x.shape[0]), "n_cells": n_cells, "k": k,
                   "fields": "p[D=1] + U[D=2]", "snapshots_total": N_SNAP, "snapshots_per_gpu": ts,
                   "unique_source_points": n_unique,
                   "layout": "[N, D, T] rows padded to a multiple of 128 bytes (interpolate.alloc_snapshots); the dense "
                             "reference layout is reported in roofline_dense_layout",
                   "l2_policy": f"{n_rot} rotating input/output buffer set(s): {step_bytes * n_rot / 1e6:.0f} MB touched "
                                f"between re-uses of a byte vs 126 MB L2",
                   "sharding": "one batch, snapshot window per rank (strong scaling); grid + KNN tables broadcast once "
                               "over NCCL before the timed steps (tables_broadcast_ms; value_incl_table_broadcast charges "
                               "it to the K timed steps)",
                   "tables_broadcast_ms": bcast_ms, "value_incl_table_broadcast": value_incl_bcast,
                   "host_cores_bound_to_gpu_numa_node": len(numa_cores) if numa_cores else None,
                   "tune": args.tune or None},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     # csrc/interp.cu launch_interp: rows of <= 768 columns (k <= 16) take the part-warp kernel
                     "kernel": "interp_warpcell_kernel" if ts > 768 else "interp_partwarp_kernel",
                     "per": "GPU (rank 0's window)",
                     "algorithmic_bytes_per_step": b_algo(), "frac_of_nominal_8TBs": achieved / 8000.0,
                     # SURVEY 8(d): what a gather without any cache re-use would move (every reference read from DRAM)
                     "naive_gather_bytes_per_step": naive_bytes,
                     "naive_gather_gbs": naive_bytes / (ms_step * 1e-3) / 1e9},
        # the same step on the reference's dense layout (T*4-byte row pitch: 3 rows in 4 start inside a cache line)
        "roofline_dense_layout": {"ms_per_step": ms_dense, "achieved": b_algo() / (ms_dense * 1e-3) / 1e9,
                                  "frac": b_algo() / (ms_dense * 1e-3) / 1e9 / peak, "unit": "GB/s"},
        # the reference's result dtype: fp64 weights, fp64 accumulation in the reference's order, fp64 result
        "roofline_fp64_out": {"ms_per_step": ms_f64, "achieved": b_algo(8) / (ms_f64 * 1e-3) / 1e9,
                              "frac": b_algo(8) / (ms_f64 * 1e-3) / 1e9 / peak, "unit": "GB/s",
                              "algorithmic_bytes_per_step": b_algo(8)},
        "cpu_baseline": cpu_baseline,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms, "bytes_are": "per rank",
                "api": "ExportData(distributed=N>1).export(pinned host window, n_snapshots_total) -> pinned host result; time windows pipelined over "
                       "H2D (pitched DMA, or a PCIe row gather when < 60 % of the points are referenced) / interpolation "
                       "kernel / D2H copy streams",
                "async_host_ms_per_step": e2e_async_ms,
                "pcie_gbs_per_rank": (h2d + d2h) / (e2e_ms * 1e-3) / 1e9},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "grid_gen_s": grid_info["t_total"] if grid_info else None,
        "grid_gen": None if grid_info is None else {
            "t_total": grid_info["t_total"], "t_uniform": grid_info["t_uniform"], "t_adaptive": grid_info["t_adaptive"],
            "t_geometry": grid_info["t_geometry"], "t_renumbering": grid_info["t_renumbering"],
            "t_knn_build": grid_info["t_knn_build"], "wall_incl_setup_s": t_grid_wall,
            "iterations": grid_info["iterations"], "n_cells": grid_info["n_cells"],
            "captured_metric": grid_info["metric_per_iter"][-1], "first_run_in_process": grid_cold},
        "knn_tables_s": t_tables,
        "svd": svd_info,
        "grid_gen_reference": reference_gridgen_record(),
    }
    sys.stdout.flush()
    os.dup2(stdout_fd, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="s3b200", choices=["s3b200", "reference"])
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--tune", default="", help="A/B harness: comma separated key=value pairs for s3x_tune (csrc/interp.cu)")
    ap.add_argument("--no-svd", action="store_true", help="skip the SVD stage report")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--full", action="store_true", help="reference arm: all snapshots per step whatever it takes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results (a seeded sample of cells) as DIR/p.npy and DIR/U.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl s3b200 in a single process")
    if args.impl == "reference":
        run_reference(args)
    else:
        # grid files written by the grid generation go to a directory of this run, removed at the end
        with tempfile.TemporaryDirectory(prefix="s3b200_bench_") as tmp_dir:
            run_ours(args, tmp_dir)


if __name__ == "__main__":
    main()

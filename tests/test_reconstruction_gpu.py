"""ReconstructionError / s3_recon_error against the existing fp32 gather and torch fp64 reductions on the same GPU.

The reference of every case is ``rec.reconstruct(sampled)`` (the gather kernel, fp32 FMA chain in neighbour order),
``e = rec.double() - original.double()`` and torch fp64 sums. The fused kernel computes the same fp32 products, so
``max_abs`` must be bit-exact; the sums are reduced in another order and agree within 1e-12 relative.
"""
import os
import socket

import numpy as np
import pytest
import torch as pt

from oracle import s3_oracle as orc

pytestmark = pytest.mark.gpu

RTOL = 1e-12
BLOCK = 512                          # points per block of the kernel (csrc/interp.cu kReconBlock)


class _Grid:
    def __init__(self, centers):
        self.centers = centers
        self.n_dimensions = centers.size(1)


def _points(n, dim, seed):
    g = pt.Generator().manual_seed(seed)
    return pt.rand((n, dim), generator=g, dtype=pt.float64)


_RECS = {}


def _rec(dim, k, n=5000, nc=1500):
    """ReconstructionError of a random cloud (n not a multiple of the block: the last block is partial). The KNN index
    returns at most 32 neighbours; wider tables (the kernel takes up to 64) are random rows of normalised weights in
    place of the KNN tables, with the same Morton processing order."""
    from sparsespatialsampling_b200 import ReconstructionError
    key = (dim, k, n, nc)
    if key not in _RECS:
        rec = ReconstructionError(_Grid(_points(nc, dim, 1 + dim)), _points(n, dim, 2 + dim), n_neighbors=min(k, 32))
        if k > 32:
            t = rec.tables
            g = pt.Generator(device=t.out_row.device).manual_seed(k)
            t.idx_sorted = pt.randint(0, nc, (n, k), generator=g, device=g.device, dtype=pt.int32)
            w = pt.rand((n, k), generator=g, device=g.device, dtype=pt.float64) + 0.1
            t.w64_sorted = w / w.sum(1, keepdim=True)
            t.w32_sorted = t.w64_sorted.float()
            t.k = rec.k = k
        _RECS[key] = rec
    return _RECS[key]


def _field(rows, d, t, layout, seed, dev):
    """A [rows, D, T] (or [rows, T]) fp32 field on the device in the given layout."""
    from sparsespatialsampling_b200.interpolate import alloc_snapshots
    g = pt.Generator(device=dev).manual_seed(seed)
    vals = pt.randn((rows, d, t), generator=g, device=dev, dtype=pt.float32)
    if layout == "pitched":
        out = alloc_snapshots(rows, d, t, device=dev)
        out.copy_(vals)
        return out
    if layout == "dense":
        return vals
    if layout == "2d":
        assert d == 1
        return vals[:, 0, :].contiguous()
    # a window x[:, :, t0:t0 + t] of a pitched batch of t + 16 snapshots
    t0 = int(layout[len("window"):])
    big = alloc_snapshots(rows, d, t + 16, device=dev)
    big.copy_(pt.randn((rows, d, t + 16), generator=g, device=dev, dtype=pt.float32))
    big[:, :, t0:t0 + t] = vals
    return big[:, :, t0:t0 + t]


def _reference(rec, original, sampled):
    r = rec.reconstruct(sampled)
    if r.dim() == 2:
        r, original = r.unsqueeze(1), original.unsqueeze(1)
    o = original.double()
    e = r.double() - o
    return (e * e).sum(0), (o * o).sum(0), e.abs().amax(0), (e * e).sum(2)


def _close(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype == pt.float64
    assert bool(((a - b).abs() <= RTOL * b.abs()).all()), float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())


def _check(stats, ref):
    sq_err, sq_ref, max_abs, point = ref
    assert pt.equal(stats.max_abs, max_abs)
    _close(stats.sq_err, sq_err)
    _close(stats.sq_ref, sq_ref)
    _close(stats.point_sq_err, point)


def _same_bits(a, b):
    for x, y in ((a.sq_err, b.sq_err), (a.sq_ref, b.sq_ref), (a.max_abs, b.max_abs), (a.point_sq_err, b.point_sq_err)):
        assert pt.equal(x, y)


def test_tables_equal_brute_force_knn(cuda):
    from sparsespatialsampling_b200 import ReconstructionError
    for dim, k, n, nc in ((2, 8, 3000, 700), (3, 26, 3000, 900)):
        centers, coords = _points(nc, dim, 10 + dim), _points(n, dim, 20 + dim)
        rec = ReconstructionError(_Grid(centers), coords)
        assert rec.k == k
        d_ref, i_ref = orc.knn_search(centers.numpy(), coords.numpy(), k)
        got = rec.tables.idx.cpu().numpy().astype(np.int64)
        for row in np.nonzero((got != i_ref).any(1))[0]:            # ties: the columns of one distance as sets
            for dv in np.unique(d_ref[row]):
                cols = d_ref[row] == dv
                assert set(got[row, cols]) == set(i_ref[row, cols]), row
        assert (got == i_ref).mean() > 0.99
        # weights: the export's rule, inverse distance normalised per point
        np.testing.assert_allclose(rec.tables.w64.cpu().numpy(), orc.export_weights(d_ref), rtol=1e-12)


@pytest.mark.parametrize("d,t,k,layout", [
    (1, 1, 8, "pitched"),
    (2, 7, 26, "dense"),
    (3, 250, 33, "pitched"),
    (1, 250, 8, "dense"),            # 1000-byte rows: no 256-bit path
    (2, 1000, 64, "pitched"),
    (1, 2000, 26, "2d"),
    (1, 7, 64, "2d"),
    (2, 250, 26, "window8"),         # 32-byte aligned window, T % 8 tail inside the pitch
    (3, 1000, 8, "window3"),         # misaligned window
    (2, 2000, 33, "dense"),
    (3, 2000, 8, "pitched"),
])
def test_error_matches_gather_and_torch(cuda, d, t, k, layout):
    dim = 2 if k == 8 else 3
    rec = _rec(dim, k)
    original = _field(rec.n_points, d, t, layout, 1, cuda)
    sampled = _field(rec.n_cells, d, t, layout, 2, cuda)
    stats = rec.error(original, sampled)
    assert stats.n_snapshots == t and stats.sq_err.shape == (d, t) and stats.point_sq_err.shape == (rec.n_points, d)
    _check(stats, _reference(rec, original, sampled))
    assert stats.relative_l2().shape == (t,) and stats.rms().shape == (rec.n_points, d)


def test_error_is_deterministic_and_independent_of_the_cta_cap(cuda):
    from sparsespatialsampling_b200 import _lib
    rec = _rec(3, 26)
    n_blocks = -(-rec.n_points // BLOCK)
    assert n_blocks == 10
    original = _field(rec.n_points, 2, 1000, "pitched", 3, cuda)
    sampled = _field(rec.n_cells, 2, 1000, "pitched", 4, cuda)
    first = rec.error(original, sampled)
    _same_bits(first, rec.error(original, sampled))
    try:
        for cap in (1, 4, 5, 6, 9, 10, 11):        # several blocks per CTA; around n_blocks / 2 and n_blocks
            _lib.tune(18, cap)
            _same_bits(first, rec.error(original, sampled))
    finally:
        _lib.tune(18, 0)


def test_windows_give_the_columns_of_the_whole_batch(cuda):
    rec = _rec(2, 8)
    original = _field(rec.n_points, 2, 1000, "pitched", 5, cuda)
    sampled = _field(rec.n_cells, 2, 1000, "pitched", 6, cuda)
    whole = rec.error(original, sampled)
    stats = None
    for t0, t1 in ((0, 333), (333, 700), (700, 1000)):
        stats = rec.error(original[:, :, t0:t1], sampled[:, :, t0:t1], stats=stats)
    assert stats.n_snapshots == 1000
    assert pt.equal(stats.sq_err, whole.sq_err) and pt.equal(stats.sq_ref, whole.sq_ref)
    assert pt.equal(stats.max_abs, whole.max_abs)
    _close(stats.point_sq_err, whole.point_sq_err)
    _close(stats.rms(), whole.rms())


def test_scale_3d_200k_points(cuda):
    rec = _rec(3, 26, n=200_000, nc=30_000)
    original = _field(rec.n_points, 1, 2000, "pitched", 7, cuda)
    sampled = _field(rec.n_cells, 1, 2000, "pitched", 8, cuda)
    stats = rec.error(original, sampled)
    _check(stats, _reference(rec, original, sampled))


def test_constant_field_reconstructs(cuda):
    rec = _rec(3, 26)
    levels = pt.linspace(-3.0, 5.0, 40, device=cuda, dtype=pt.float32)
    original = levels[None, None, :].expand(rec.n_points, 2, 40).contiguous()
    sampled = levels[None, None, :].expand(rec.n_cells, 2, 40).contiguous()
    stats = rec.error(original, sampled)
    assert float(stats.relative_l2().max()) <= 1e-6


def test_finer_grid_reconstructs_better(cuda, tmp_path):
    import synth
    from sparsespatialsampling_b200 import SparseSpatialSampling, ExportData, ReconstructionError
    from sparsespatialsampling_b200.geometry import CubeGeometry, SphereGeometry
    n, t = synth.CONFIGS["C1"][0], synth.CONFIGS["C1"][1]
    x = synth.cylinder2d_cloud(n, seed=0)
    field = synth.wake_field(x, 0, t, t, components=1)
    errors, cells = [], []
    for min_metric in (0.5, 0.9):
        geoms = [CubeGeometry("domain", True, synth.CYL2D["lower"], synth.CYL2D["upper"]),
                 SphereGeometry("cylinder", False, synth.CYL2D["pos"], synth.CYL2D["radius"], refine=True)]
        s_cube = SparseSpatialSampling(x, synth.wake_metric(x), geoms, str(tmp_path), f"m{min_metric}", "grid",
                                       uniform_levels=4, min_metric=min_metric)
        s_cube.execute_grid_generation()
        export = ExportData(s_cube, write_times=[str(i) for i in range(t)], write_files=False)
        export.export(x, field, "p")
        sampled = export.interpolated_fields.centers
        stats = ReconstructionError(s_cube, x).error(field, sampled)
        errors.append(float(stats.relative_l2().mean()))
        cells.append(s_cube.centers.size(0))
    assert cells[1] > cells[0]
    assert errors[1] < errors[0], errors


def test_errors(cuda):
    from sparsespatialsampling_b200 import ReconstructionError, _lib
    with pytest.raises(ValueError):
        ReconstructionError(_Grid(_points(20, 3, 0)), _points(100, 3, 1))             # 20 cells < k = 26
    with pytest.raises(ValueError):
        ReconstructionError(_Grid(_points(20, 2, 0)), _points(100, 2, 1), n_neighbors=21)
    rec = _rec(2, 8)
    o = _field(rec.n_points, 2, 10, "dense", 1, cuda)
    s = _field(rec.n_cells, 2, 10, "dense", 2, cuda)
    for bad_o, bad_s in ((o[:-1], s), (o, s[:-1]), (o[:, :1], s), (o[:, :, :9], s), (o.double(), s.double()),
                         (o, s.double())):
        with pytest.raises(ValueError):
            rec.error(bad_o, bad_s)
    with pytest.raises(ValueError):
        rec.reconstruct(s[:-1])
    # the C-ABI: fp64 fields are not supported, k must be in [1, 64]
    lib = _lib.load()
    t = rec.tables
    res = pt.empty((3, 2, 10), dtype=pt.float64, device=cuda)

    def call(k, dtype=_lib.S3_F32):
        return lib.s3_recon_error(
            _lib.ptr(s), dtype, rec.n_cells, 2, 10, 20, 10, _lib.ptr(o), dtype, rec.n_points, 20, 10,
            _lib.ptr(t.idx_sorted), _lib.ptr(t.w32_sorted), _lib.ptr(t.out_row), k, _lib.ptr(res[0]),
            _lib.ptr(res[1]), _lib.ptr(res[2]), None, _lib.stream_ptr())
    assert call(8) == 0
    assert call(0) != 0 and call(65) != 0
    assert call(8, _lib.S3_F64) == -3                                                  # S3_ERR_UNSUPPORTED
    assert b"fp32" in lib.s3_last_error()


# ---------------------------------------------------------------------------------------------------- two GPUs, NCCL
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, tmp):
    import torch.distributed as dist
    from sparsespatialsampling_b200 import ReconstructionError
    from sparsespatialsampling_b200.parallel import snapshot_window
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = pt.device("cuda", rank)
    pt.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    T = 301                                                      # unequal windows
    rec = ReconstructionError(_Grid(_points(1500, 3, 4)), _points(5000, 3, 5), device=dev, distributed=True)
    original = _field(rec.n_points, 2, T, "pitched", 1, dev)
    sampled = _field(rec.n_cells, 2, T, "pitched", 2, dev)
    t0, t1 = snapshot_window(T, world, rank)
    mid = (t0 + t1) // 2
    stats = rec.error(original[:, :, t0:mid], sampled[:, :, t0:mid])
    stats = rec.error(original[:, :, mid:t1], sampled[:, :, mid:t1], stats=stats)
    every = stats.gather()
    if rank == 0:
        single = ReconstructionError(_Grid(_points(1500, 3, 4)), _points(5000, 3, 5), device=dev).error(original, sampled)
        pt.save({"every": [every.sq_err.cpu(), every.sq_ref.cpu(), every.max_abs.cpu(), every.point_sq_err.cpu(),
                           every.n_snapshots],
                 "single": [single.sq_err.cpu(), single.sq_ref.cpu(), single.max_abs.cpu(),
                            single.point_sq_err.cpu(), single.n_snapshots]}, os.path.join(tmp, "out.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_error_two_gpus(cuda, tmp_path):
    import torch.multiprocessing as mp
    if pt.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r = pt.load(tmp_path / "out.pt")
    for a, b in zip(r["every"][:3], r["single"][:3]):
        assert pt.equal(a, b)
    _close(r["every"][3], r["single"][3])
    assert r["every"][4] == r["single"][4] == 301

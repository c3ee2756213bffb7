"""
world_size-2 gloo tests of the N>1 path (host logic only, no GPU): the product's ExportData in distributed mode -- rank 0
owns the KNN tables and broadcasts them, every rank interpolates and writes its own snapshot window -- gives the same
files as one process; the re-sharding and all-reduce of the sharded SVD.
"""
import os
import socket

import numpy as np
import torch as pt
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import s3_oracle as orc


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _cpu_gather(data, idx, weights, out=None, out_row=None, out_dtype=None):
    """Stand-in for the kernel launch (there is no GPU here): the same operator with torch CPU ops, so that everything
    AROUND the launch -- table broadcast, windows, part files, XDMF, Dataloader -- is the product's own code."""
    rows = data.reshape(data.size(0), -1).to(out_dtype)
    res = pt.zeros((idx.size(0), rows.size(1)), dtype=out_dtype)
    for j in range(idx.size(1)):                      # sequential over the neighbours: independent of the batch shape
        res += weights[:, j].to(out_dtype)[:, None] * rows[idx[:, j].long()]
    res = res.reshape((idx.size(0),) + tuple(data.shape[1:]))
    if out_row is not None:
        full = pt.empty_like(res)
        full[out_row.long()] = res
        res = full
    if out is not None:
        out.copy_(res)
        return out
    return res


def _case():
    rng = np.random.default_rng(0)                     # same data on every rank
    N, Nc, k, T = 400, 150, 8, 11
    return (rng, N, Nc, k, T, pt.from_numpy(rng.random((N, 2))), pt.from_numpy(rng.standard_normal((N, 2, T)).astype(np.float32)),
            pt.from_numpy(rng.standard_normal((N, 1, T)).astype(np.float32)))


class _Grid:
    pass


def _grid(rng, Nc, N, tmp):
    g = _Grid()
    g.n_dimensions, g.size_initial_cell = 2, 1.0
    g.centers = pt.from_numpy(rng.random((Nc, 2)))
    g.vertices = pt.from_numpy(rng.random((Nc + 30, 2)))
    g.faces = pt.from_numpy(rng.integers(0, Nc + 30, (Nc, 4)).astype(np.int32))
    g.levels = pt.from_numpy(rng.integers(1, 5, (Nc, 1)))
    g.metric = pt.from_numpy(rng.random(N))
    g.save_path, g.save_name, g.grid_name = tmp, "sharded", "grid"
    return g


def _worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from sparsespatialsampling_b200 import _lib, export
    from sparsespatialsampling_b200.parallel import snapshot_window
    _lib.require_cuda = lambda: None                  # host logic only
    export.interp_gather = _cpu_gather
    rng, N, Nc, k, T, x, u, p = _case()
    g = _grid(rng, Nc, N, tmp if world > 1 else os.path.join(tmp, "single"))
    idx0, w0 = pt.from_numpy(rng.integers(0, N, (Nc, k)).astype(np.int32)), pt.from_numpy(rng.random((Nc, k)))
    perm0 = pt.from_numpy(rng.permutation(Nc).astype(np.int32))

    class _Export(export.ExportData):
        def _make_tables(self, _coord):              # rank 0 only: the tables a device KNN search would produce
            t = export.KnnTables.__new__(export.KnnTables)
            t.n, t.k, t._inflight = Nc, k, []
            t.idx, t.w64 = idx0, w0
            t.out_row = perm0
            t.idx_sorted, t.w64_sorted = idx0[perm0.long()].contiguous(), w0[perm0.long()].contiguous()
            t.w32_sorted = t.w64_sorted.float()
            self._tables_centers = t

    times = [f"{0.5 * i:.1f}" for i in range(T)]
    exp = _Export(g, write_times=times, device="cpu", stream_host=False, distributed=world > 1)
    t0, t1 = snapshot_window(T, world, rank)
    mid = (t0 + t1) // 2                              # two batches per rank
    for field, data in (("U", u), ("p", p)):
        exp.export(x, data[:, :, t0:mid], field, n_snapshots_total=T)
        exp.export(x, data[:, :, mid:t1], field, n_snapshots_total=T)
    if world > 1:
        assert exp._tables_centers.n == Nc and pt.equal(exp._tables_centers.idx, idx0)      # every rank has rank 0's tables
        dist.barrier()
        dist.destroy_process_group()


def test_sharded_export_world_size_2_equals_single_process(tmp_path, monkeypatch):
    """ExportData(distributed=True) under gloo: table broadcast, snapshot windows, per-rank part files, one XDMF and the
    Dataloader that follows the part list -- against the same export done by one process."""
    from sparsespatialsampling_b200 import _lib, export
    from sparsespatialsampling_b200.data import Dataloader
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    # the single-process run happens in this process: the CPU stand-ins _worker installs must not outlive this test
    monkeypatch.setattr(_lib, "require_cuda", _lib.require_cuda)
    monkeypatch.setattr(export, "interp_gather", export.interp_gather)
    _worker(0, 1, 0, str(tmp_path))                                   # single process, same code
    assert sorted(os.listdir(tmp_path))[:3] == ["sharded.h5", "sharded.part1.h5", "sharded.xdmf"]
    many, one = Dataloader(str(tmp_path), "sharded.h5"), Dataloader(str(tmp_path / "single"), "sharded.h5")
    assert many.write_times == one.write_times and len(many.write_times) == 11
    assert many.field_names == one.field_names
    for f in ("p", "U"):
        assert pt.equal(many.load_snapshot(f), one.load_snapshot(f))
    assert pt.equal(many.metric, one.metric) and pt.equal(many.faces, one.faces)
    # the XDMF of the sharded run points every time step at the part that holds it
    xdmf = open(tmp_path / "sharded.xdmf").read()
    ref = open(tmp_path / "single" / "sharded.xdmf").read()
    assert xdmf.count("<Time Value=") == 11 and "sharded.part1.h5:/data/5.0/U_center" in xdmf
    assert "sharded.h5:/data/0.0/p_center" in xdmf and "part_files" not in xdmf
    assert xdmf.replace("sharded.part1.h5", "sharded.h5") == ref


def _svd_exchange_worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sparsespatialsampling_b200.parallel import (snapshot_window, row_window, time_to_row_shards, allreduce_sum,
                                                     gather_rows)
    rng = np.random.default_rng(1)                     # same data on every rank
    Nc, D, T = 37, 2, 13                               # odd sizes: unequal windows on both axes
    full = rng.standard_normal((Nc, D, T)).astype(np.float32)
    vol = rng.random(Nc) + 0.5
    t0, t1 = snapshot_window(T, world, rank)
    rows = time_to_row_shards(pt.from_numpy(full[:, :, t0:t1].copy()), T)
    r0, r1 = row_window(Nc, world, rank)
    assert np.array_equal(rows.numpy(), full[r0:r1])
    rows2d = time_to_row_shards(pt.from_numpy(full[:, 0, t0:t1].copy()), T)
    assert np.array_equal(rows2d.numpy(), full[r0:r1, 0])
    # local weighted Gram of the own rows (oracle arithmetic), summed over the ranks == Gram of the whole matrix
    g = pt.from_numpy(orc.weighted_gram(rows.numpy().reshape(-1, T), np.repeat(vol[r0:r1], D)))
    allreduce_sum(g)
    everything = gather_rows(rows, Nc)
    assert np.array_equal(everything.numpy(), full)
    np.save(os.path.join(tmp, f"gram{rank}.npy"), g.numpy())
    dist.barrier()
    dist.destroy_process_group()


def test_svd_exchange_world_size_3(tmp_path):
    """time -> cell re-sharding, all-reduce of the partial Gram matrices and the row gather of compute_svd_sharded."""
    world = 3
    mp.spawn(_svd_exchange_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    rng = np.random.default_rng(1)
    full = rng.standard_normal((37, 2, 13)).astype(np.float32)
    vol = rng.random(37) + 0.5
    ref = orc.weighted_gram(full.reshape(-1, 13), np.repeat(vol, 2))
    for r in range(world):
        g = np.load(tmp_path / f"gram{r}.npy")
        assert np.allclose(g, ref, rtol=1e-12, atol=1e-12)
        assert np.array_equal(g, np.load(tmp_path / "gram0.npy"))


def test_bind_to_gpu_numa_node_is_harmless_without_nvml():
    # no GPU / NVML in the CPU container: the helper must leave the affinity alone and say so
    from sparsespatialsampling_b200.parallel import bind_to_gpu_numa_node
    before = os.sched_getaffinity(0)
    cores = bind_to_gpu_numa_node(0)
    assert cores is None or set(cores) <= before
    if cores is None:
        assert os.sched_getaffinity(0) == before
    os.sched_setaffinity(0, before)


def test_row_and_snapshot_windows_partition_the_axis():
    from sparsespatialsampling_b200.parallel import snapshot_window, row_window
    for n, world in [(1000, 8), (13, 3), (5, 8), (0, 2)]:
        edges = [snapshot_window(n, world, r) for r in range(world)]
        assert edges[0][0] == 0 and edges[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(edges, edges[1:]))
        sizes = [b - a for a, b in edges]
        assert max(sizes) - min(sizes) <= 1
        assert edges == [row_window(n, world, r) for r in range(world)]

"""
world_size-2 gloo test of ReconstructionError(distributed=True), host logic only (no GPU): rank 0 builds the tables and
shares them, every rank passes its own (unequal) snapshot window in two calls, and ErrorStats.gather() gives every rank
what one process computes. Only the kernel launch is replaced, by a torch stand-in with the same contract.
"""
import os
import socket

import numpy as np
import torch as pt
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import s3_oracle as orc

N, NC, K, D, T = 400, 150, 8, 2, 11


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _cpu_recon_error(original, sampled, tables, point_sq_err):
    """Stand-in for the s3_recon_error launch: fp32 gather in neighbour order, fp64 error, every column reduced on
    its own (so that a column's results do not depend on the other columns of the call, as in the kernel)."""
    idx, w = tables.idx_sorted.long(), tables.w32_sorted
    r = pt.zeros((idx.size(0),) + tuple(sampled.shape[1:]), dtype=pt.float32)
    for j in range(idx.size(1)):
        r += w[:, j, None, None] * sampled[idx[:, j]]
    o = original[tables.out_row.long()].double()
    e = r.double() - o
    sq_err = pt.empty(original.shape[1:], dtype=pt.float64)
    sq_ref, max_abs = pt.empty_like(sq_err), pt.empty_like(sq_err)
    for d in range(original.size(1)):
        for t in range(original.size(2)):
            sq_err[d, t] = (e[:, d, t] * e[:, d, t]).sum()
            sq_ref[d, t] = (o[:, d, t] * o[:, d, t]).sum()
            max_abs[d, t] = e[:, d, t].abs().max()
    if point_sq_err is not None:
        point_sq_err[tables.out_row.long()] += (e * e).sum(2)
    return sq_err, sq_ref, max_abs


def _case():
    rng = np.random.default_rng(3)                     # same data on every rank
    return (pt.from_numpy(rng.random((NC, 2))), pt.from_numpy(rng.random((N, 2))),
            pt.from_numpy(rng.standard_normal((N, D, T)).astype(np.float32)),
            pt.from_numpy(rng.standard_normal((NC, D, T)).astype(np.float32)))


class _Grid:
    pass


def _run(rank, world, out_path):
    from sparsespatialsampling_b200 import reconstruction
    from sparsespatialsampling_b200.export import KnnTables
    from sparsespatialsampling_b200.parallel import snapshot_window
    centers, coords, original, sampled = _case()
    grid = _Grid()
    grid.centers, grid.n_dimensions = centers, 2

    class _Rec(reconstruction.ReconstructionError):
        def _make_tables(self, centers, coordinates):     # rank 0 only: the tables a device KNN search would produce
            dist_ref, idx = orc.knn_search(centers.numpy(), coordinates.numpy(), self.k)
            w64 = pt.from_numpy(orc.export_weights(dist_ref))
            perm = pt.from_numpy(np.random.default_rng(5).permutation(N).astype(np.int32))
            t = KnnTables.__new__(KnnTables)
            t.n, t.k, t._inflight = N, self.k, []
            t.idx, t.w64, t.out_row = pt.from_numpy(idx.astype(np.int32)), w64, perm
            t.idx_sorted, t.w64_sorted = t.idx[perm.long()].contiguous(), w64[perm.long()].contiguous()
            t.w32_sorted = t.w64_sorted.float()
            return t

    rec = _Rec(grid, coords, device="cpu", distributed=world > 1)
    assert rec.k == K and rec.tables.n == N
    t0, t1 = snapshot_window(T, world, rank)
    mid = (t0 + t1) // 2
    stats = rec.error(original[:, :, t0:mid], sampled[:, :, t0:mid])
    stats = rec.error(original[:, :, mid:t1], sampled[:, :, mid:t1], stats=stats)
    assert stats.n_snapshots == t1 - t0
    every = stats.gather()
    if rank == 0:
        pt.save({"stats": [every.sq_err, every.sq_ref, every.max_abs, every.point_sq_err, every.n_snapshots],
                 "tables": [rec.tables.idx_sorted, rec.tables.out_row, rec.tables.w32_sorted]}, out_path)
    else:
        pt.save({"tables": [rec.tables.idx_sorted, rec.tables.out_row, rec.tables.w32_sorted]}, out_path)


def _worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sparsespatialsampling_b200 import _lib, reconstruction
    _lib.require_cuda = lambda: None                  # host logic only
    reconstruction.recon_error = _cpu_recon_error
    _run(rank, world, os.path.join(tmp, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_error_world_size_2_equals_single_process(tmp_path, monkeypatch):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    from sparsespatialsampling_b200 import _lib, reconstruction
    monkeypatch.setattr(_lib, "require_cuda", lambda: None)
    monkeypatch.setattr(reconstruction, "recon_error", _cpu_recon_error)
    _run(0, 1, str(tmp_path / "single.pt"))
    one = pt.load(tmp_path / "single.pt")
    ranks = [pt.load(tmp_path / f"rank{r}.pt") for r in range(world)]
    for r in ranks:                                    # every rank works with rank 0's tables
        assert all(pt.equal(a, b) for a, b in zip(r["tables"], one["tables"]))
    got, want = ranks[0]["stats"], one["stats"]
    assert got[4] == want[4] == T
    for a, b in zip(got[:3], want[:3]):
        assert a.shape == (D, T) and pt.equal(a, b)
    # the point map: sums over other windows, summed over the ranks
    assert got[3].shape == (N, D) and bool((got[3] > 0).all()) and pt.allclose(got[3], want[3], rtol=1e-12, atol=0)

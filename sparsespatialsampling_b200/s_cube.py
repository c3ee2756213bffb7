"""
Refinement engine of S^3 on the GPU (host side).

``SamplingTree`` keeps the constructor, ``refine()`` and the result attributes of the reference class
(sparseSpatialSampling/s_cube.py:86-205, :563-667: ``all_centers, all_nodes, face_ids, all_levels, data_final_mesh``)
but holds the tree as a structure of arrays on the device instead of a graph of Python ``Cell`` objects:

=====================  ==========================================================================================
device (CUDA kernels)  child generation, KNN + inverse-distance metric prediction, gain, geometry masks, top-k
                       selection (radix select + sort), captured-metric reduction, vertex table
host (this file)       the sequential control flow of the reference (stopping criteria, cells per iteration,
                       geometry-refinement passes) and the *cell numbering*: the reference numbers new cells in
                       the iteration order of CPython sets (s_cube.py:603-606, :879), so the same set operations
                       are replayed here on plain integers -- a few thousand ints per iteration
=====================  ==========================================================================================

Per iteration the host reads back: the k selected cell indices, one invalid flag per new cell, one scalar
(sum of squared leaf metrics).
"""
import logging
from time import time
from typing import Union

import numpy as np
import torch as pt

from . import _lib
from .topology import Topology
from .knn import KnnIndex, default_n_neighbors
from .geometry.device import GeometryTable

logger = logging.getLogger(__name__)

FLAG_LEAF = 1
FLAG_INVALID = 2


def _initialize_time_dict() -> dict:
    return {"t_start_uniform": 0.0, "t_end_uniform": 0.0, "t_start_adaptive": 0.0, "t_start_geometry": 0.0,
            "t_end_geometry": 0.0, "t_start_renumber": 0.0, "t_end_renumber": 0.0}


def probe_sum_order_8() -> int:
    """
    Association order torch's CPU kernel uses for ``tensor[n, 8].sum(dim=1)`` in fp64 on THIS host -- the reference
    evaluates the 3-D ``sum_delta_metric`` with it (s_cube.py:229) and the order depends on the CPU capability.
    Returns the ``sdm_order`` code of ``s3_cells_gain`` (0 sequential, 1 four-lane).
    """
    g = pt.Generator().manual_seed(1234)
    a = pt.rand((4096, 8), dtype=pt.float64, generator=g) * pt.rand((4096, 1), dtype=pt.float64, generator=g) * 1e3
    ref = a.sum(dim=1)
    seq = a[:, 0].clone()
    for j in range(1, 8):
        seq = seq + a[:, j]
    lane4 = (((a[:, 0] + a[:, 4]) + (a[:, 1] + a[:, 5])) + (a[:, 2] + a[:, 6])) + (a[:, 3] + a[:, 7])
    if pt.equal(ref, lane4):
        return 1
    if pt.equal(ref, seq):
        return 0
    logger.warning("Could not identify torch's fp64 sum(dim=1) order on this host; using the four-lane order.")
    return 1


class SamplingTree(object):
    # queue the host-side topology replay on the library's worker thread whenever nothing reads it inside the loop
    topology_async = True

    def __init__(self, vertices: pt.Tensor, target: pt.Tensor, geometry_obj: list, n_cells: int = None,
                 uniform_level: int = 5, min_metric: float = 0.75, max_delta_level: bool = False,
                 n_cells_iter_start: int = None, n_cells_iter_end: int = None, n_jobs: int = 1,
                 relTol: Union[int, float] = 1e-3, reach_at_least: float = 0.75, pre_select: bool = False,
                 device=None, sdm_order: int = None):
        _lib.require_cuda()
        self._topo = None
        self._lib = _lib.load()
        self._device = pt.device(device) if device is not None else pt.device("cuda", pt.cuda.current_device())
        self._pre_select = pre_select
        self._n_jobs = n_jobs                       # accepted and ignored: the device does the work
        self._max_delta_level = max_delta_level
        self._geometry = geometry_obj
        self._n_cells = 0
        self._min_metric = min_metric
        self._n_cells_max = n_cells
        self._min_level = uniform_level
        self._current_min_level = 0
        self._current_max_level = 0
        # s_cube.py:147-156
        self._cells_per_iter_start = int(0.001 * vertices.size(0)) if n_cells_iter_start is None else n_cells_iter_start
        if self._cells_per_iter_start <= 0:
            self._cells_per_iter_start = 1
        self._cells_per_iter_end = self._cells_per_iter_start if n_cells_iter_end is None else n_cells_iter_end
        self._cells_per_iter = self._cells_per_iter_start
        self._cells_per_iter_last = 1e9
        self._reach_at_least = reach_at_least
        self._width = None
        self._n_dimensions = vertices.size(-1)
        self._k = default_n_neighbors(self._n_dimensions)
        self._nch = 2 ** self._n_dimensions
        self._sdm_order = probe_sum_order_8() if sdm_order is None else int(sdm_order)

        # KNN index over the original grid with the metric as regression target (s_cube.py:161-163)
        t0 = time()
        with pt.cuda.device(self._device):
            self._knn = KnnIndex(vertices, target, device=self._device)
        self._t_knn_build = time() - t0

        self._leaf_cells = set()
        self._n_cells_after_uniform = None
        self.all_nodes = None
        self.all_centers = None
        self.all_levels = None
        self.face_ids = None
        self._metric = []
        self._n_cells_log = []
        self._selected_log = None       # set to [] before refine() to record the selected cells per iteration
        self._n_cells_orig = target.size(0)
        self.data_final_mesh = {}
        self._times = _initialize_time_dict()
        if relTol is None:
            self._relTol = 1e-3 if n_cells is None else 10
        else:
            self._relTol = relTol

        # device state
        self._cap = 0
        self._center = self._level = self._gain = self._metric_d = self._flags = None
        self._levels_h = np.zeros(0, dtype=np.int32)
        self._invalid_h = np.zeros(0, dtype=bool)
        self._scalar = pt.zeros(1, dtype=pt.float64, device=self._device)
        # pinned staging of the per-iteration transfers: parent list up, (invalid flags, captured-metric sum) down with
        # ONE synchronisation per iteration
        self._pin_i64 = pt.empty(1024, dtype=pt.int64, pin_memory=True)
        self._pin_i64_copied = pt.cuda.Event()      # recorded behind the last host-to-device copy out of _pin_i64
        self._pin_u8 = pt.empty(8192, dtype=pt.uint8, pin_memory=True)
        self._pin_f64 = pt.empty(1, dtype=pt.float64, pin_memory=True)
        self._pin_sel = pt.empty(1024, dtype=pt.int64, pin_memory=True)
        self._sel_d = pt.empty(1024, dtype=pt.int64, device=self._device)
        self._stream_obj, self._stream_ptr, self._ptr_cache = None, None, {}
        self._mask_out = pt.empty(8192, dtype=pt.uint8, device=self._device)
        self._fuse_metric = False        # set by refine(): the next mask pass also evaluates the captured metric
        self._fused_sumsq = None
        self._speculate_k = 0            # set by refine(): the next mask pass also selects the cells of the NEXT iteration
        self._spec_selection = None
        self._geom_table = GeometryTable(self._geometry, self._device)

        self._create_first_cell()

        # ||target||_2 (s_cube.py:205), reduced on the device
        tgt = target.detach().to(device=self._device, dtype=pt.float64).contiguous()
        self._target_norm = float(np.sqrt(self._sumsq(tgt)))

    # ------------------------------------------------------------------------------------------ helpers
    def _stream(self):
        # the C-ABI calls of one refine() run are all queued on the stream that was current when it started
        # (torch.cuda.current_stream() costs ~15 us per call -- more than a small launch)
        if self._stream_obj is None:
            return _lib.stream_ptr()
        return self._stream_ptr

    def _enter_hot_loop(self) -> None:
        import ctypes
        pt.cuda.set_device(self._device)
        self._stream_obj = pt.cuda.current_stream(self._device)
        self._stream_ptr = ctypes.c_void_p(self._stream_obj.cuda_stream)

    def _p(self, name: str):
        """Device pointer of a cell array, cached until the arrays are re-allocated (``_reserve``)."""
        ptr = self._ptr_cache.get(name)
        if ptr is None:
            ptr = self._ptr_cache[name] = _lib.ptr(getattr(self, name))
        return ptr

    def _sumsq(self, x: pt.Tensor) -> float:
        with pt.cuda.device(self._device):
            _lib.check(self._lib.s3_sumsq(_lib.ptr(x), x.numel(), _lib.ptr(self._scalar), self._stream()))
        return self._scalar.item()

    def _reserve(self, n: int) -> None:
        """Grow the cell arrays to hold at least ``n`` cells (capacity doubling)."""
        if n <= self._cap:
            return
        new_cap = max(n, 2 * self._cap, 1024)
        d, dev = self._n_dimensions, self._device

        def grow(old, shape, dtype):
            new = pt.zeros(shape, dtype=dtype, device=dev)
            if old is not None:
                new[:old.size(0)] = old
            return new
        self._ptr_cache = {}
        self._center = grow(self._center, (new_cap, d), pt.float64)
        self._level = grow(self._level, (new_cap,), pt.int32)
        self._gain = grow(self._gain, (new_cap,), pt.float64)
        self._metric_d = grow(self._metric_d, (new_cap,), pt.float64)
        self._flags = grow(self._flags, (new_cap,), pt.uint8)
        lv = np.zeros(new_cap, dtype=np.int32)
        lv[:self._levels_h.size] = self._levels_h
        self._levels_h = lv
        iv = np.zeros(new_cap, dtype=bool)
        iv[:self._invalid_h.size] = self._invalid_h
        self._invalid_h = iv
        self._cap = new_cap

    # ------------------------------------------------------------------------------------------ root cell
    def _create_first_cell(self) -> None:
        # s_cube.py:338-397
        middle_ = None
        for g in self._geometry:
            if g.keep_inside:
                self._width = g.main_width
                middle_ = g.center
            if g.center.size(0) != self._n_dimensions:
                raise ValueError(f"The number of dimensions for geometry object '{g.name}' with dim = "
                                 f"{g.center.size(0)} is not matching the number of dimensions within the CFD grid "
                                 f"with dim = {self._n_dimensions}.")
        if middle_ is None:
            raise ValueError("No GeometryObject with 'keep_inside=True', representing the numerical domain, was found.")
        self._width = float(self._width)
        d = self._n_dimensions
        if d == 2:
            dirs = pt.tensor([[-1, -1], [-1, 1], [1, 1], [1, -1]], dtype=pt.float64)
        else:
            dirs = pt.tensor([[-1, -1, 1], [-1, 1, 1], [1, 1, 1], [1, -1, 1],
                              [-1, -1, -1], [-1, 1, -1], [1, 1, -1], [1, -1, -1]], dtype=pt.float64)
        centers_ = middle_.detach().cpu().unsqueeze(0).repeat(self._nch + 1, 1).type(pt.float64)
        centers_[1:, :] += dirs * 0.25 * self._width
        metric = self._knn.predict(centers_, self._k).cpu().numpy()

        # gain of the root: level 0, so (width/2)^d * sum |m0 - mi| (s_cube.py:375-381)
        sum_distances = sum([abs(metric[0] - metric[i]) for i in range(1, len(metric))])
        gain = pow(self._width / 2, d) * sum_distances
        if abs(gain - 0) < 1e-6:
            gain = 1.0
        self._gain0 = float(gain)

        self._reserve(1)
        self._center[0] = centers_[0].to(self._device)
        self._level[0] = 0
        self._gain[0] = self._gain0
        self._metric_d[0] = float(metric[0])
        self._flags[0] = FLAG_LEAF
        self._n_cells = 1
        self._leaf_cells.add(0)
        # without max_delta_level nothing reads the pointers before the final grid assembly
        self._topo = Topology(d, centers_[0].numpy(), self._width, asynchronous=self.topology_async and not self._max_delta_level)

    # ------------------------------------------------------------------------------------------ refinement
    def _refine_cells(self, parents: list) -> range:
        """
        Create the 2^d children of every cell in ``parents`` (in that order) and evaluate their gain
        (s_cube.py:865-902 with _update_gain :207-241); returns the index range of the new cells.
        """
        n_par = len(parents)
        first = self._n_cells
        n_new = n_par * self._nch
        self._reserve(first + n_new)
        par_h = np.asarray(parents, dtype=np.int64)
        if n_par > self._pin_i64.numel():
            self._pin_i64 = pt.empty(2 * n_par, dtype=pt.int64, pin_memory=True)
        # the previous copy out of the pinned buffer may still be queued: the mask pass synchronises the stream after
        # every refinement step, but with pre_select nothing does between two uniform levels
        self._pin_i64_copied.synchronize()
        self._pin_i64[:n_par].numpy()[:] = par_h
        par_d = self._pin_i64[:n_par].to(self._device, non_blocking=True)
        self._pin_i64_copied.record(self._stream_obj or pt.cuda.current_stream(self._device))
        if self._stream_obj is None:
            pt.cuda.set_device(self._device)
        _lib.check(self._lib.s3_cells_refine(self._p("_center"), self._p("_level"), self._p("_flags"), _lib.ptr(par_d),
                                             n_par, first, self._n_dimensions, self._width, self._stream()))
        _lib.check(self._lib.s3_cells_gain(self._knn.handle, self._p("_center"), self._p("_level"), None, first, n_new,
                                           self._k, self._width, self._gain0, self._sdm_order, self._p("_metric_d"),
                                           self._p("_gain"), self._stream()))
        self._levels_h[first:first + n_new] = np.repeat(self._levels_h[par_h] + 1, self._nch)
        if n_par:
            self._topo.refine(par_h.copy())                   # host replay of _assign_neighbors + _assign_indices
            self._current_max_level = max(self._current_max_level, int(self._levels_h[par_h].max()) + 1)

        # leaf-set bookkeeping exactly as the reference does it (s_cube.py:877-899, :243-251): the reference fills
        # `all_children` / `all_parents` parent by parent; the same insertion sequence in one call gives the same sets
        # (identical hash-table layout, hence identical iteration order further on)
        all_children = set(range(first, first + n_new))
        all_parents = set(parents)
        self._leaf_cells -= all_parents
        self._leaf_cells.update(all_children)
        self._n_cells += n_new
        return range(first, first + n_new)

    # ------------------------------------------------------------------------------------------ delta-level constraint
    def _check_nb(self, _cell_no: int) -> list:
        """
        Leaf neighbours of a cell (8 / 26 directions, reference order) with a lower level: refining the cell alone would
        create a level difference of two (s_cube.py:447-464), read from the host replay of the reference's own (possibly
        stale) neighbour pointers.
        """
        return self._topo.check_nb(_cell_no)

    def _check_constraint(self, nb_violating_constraint: set) -> set:
        # s_cube.py:466-506: transitive closure of the constraint over the neighbours that get refined as well
        new_cells_to_check = True if nb_violating_constraint else False
        while new_cells_to_check:
            tmp = set()
            for c in nb_violating_constraint:
                self._topo.refresh_siblings([c])              # s_cube.py:489-490
                tmp.update(self._check_nb(c))
            if not tmp or tmp.issubset(nb_violating_constraint):
                new_cells_to_check = False
            else:
                nb_violating_constraint.update(tmp)
        return nb_violating_constraint

    def _mask(self, cells, refine_geometry: bool, geometry_no) -> np.ndarray:
        """
        ``check_cell`` of all (or one) geometries for ``cells`` (a range of consecutive indices or a list);
        returns a bool array aligned with ``cells``. In normal mode the device state is updated as well.
        """
        n = len(cells)
        if n > self._mask_out.numel():
            self._mask_out = pt.empty(2 * n, dtype=pt.uint8, device=self._device)
        out = self._mask_out
        if isinstance(cells, range):
            cells_d, first = None, cells.start
        else:
            cells_d, first = pt.tensor(list(cells), dtype=pt.int64, device=self._device), 0
        only = -1 if geometry_no is None else int(geometry_no)
        apply = 0 if refine_geometry else 1
        tab = self._geom_table
        if self._stream_obj is None:
            pt.cuda.set_device(self._device)
        stream = self._stream()
        _lib.check(self._lib.s3_cells_mask(self._p("_center"), self._p("_level"), _lib.ptr(cells_d), first, n,
                                           self._n_dimensions, self._width, _lib.ptr(tab.hdr), _lib.ptr(tab.par),
                                           tab.n, only, int(refine_geometry), apply, _lib.ptr(out),
                                           self._p("_flags"), self._p("_gain"), tab.stl_geoms, tab.stl_meta, stream))
        fuse = self._fuse_metric and apply and not tab.custom
        if fuse:
            # the mask kernel has removed the invalid children from the leaves on the device: the captured metric
            # (s_cube.py:317-336) follows in the same stream and comes back with the flags -- one sync, not two
            _lib.check(self._lib.s3_leaf_sumsq(self._p("_metric_d"), self._p("_flags"), self._n_cells,
                                               _lib.ptr(self._scalar), stream))
        spec_k = self._speculate_k if (apply and not tab.custom) else 0
        if spec_k:
            # gains and leaf flags of the next iteration are final on the device at this point: its top-k selection
            # (s_cube.py:601-602) is queued here as well and returns with the same synchronisation. If the loop
            # stops instead, the result is dropped.
            if spec_k > self._sel_d.numel():
                self._sel_d = pt.empty(2 * spec_k, dtype=pt.int64, device=self._device)
            _lib.check(self._lib.s3_select_topk(self._p("_gain"), self._p("_flags"), self._n_cells, spec_k,
                                                _lib.ptr(self._sel_d), stream))
            if spec_k > self._pin_sel.numel():
                self._pin_sel = pt.empty(2 * spec_k, dtype=pt.int64, pin_memory=True)
            self._pin_sel[:spec_k].copy_(self._sel_d[:spec_k], non_blocking=True)
        if n > self._pin_u8.numel():
            self._pin_u8 = pt.empty(2 * n, dtype=pt.uint8, pin_memory=True)
        self._pin_u8[:n].copy_(out[:n], non_blocking=True)
        if fuse:
            self._pin_f64.copy_(self._scalar, non_blocking=True)
        (self._stream_obj or pt.cuda.current_stream(self._device)).synchronize()
        self._fuse_metric = False
        self._speculate_k = 0
        self._spec_selection = self._pin_sel[:spec_k].tolist() if spec_k else None
        self._fused_sumsq = float(self._pin_f64[0]) if fuse else None
        res = self._pin_u8[:n].numpy().astype(bool)          # (a copy: the pinned buffer is re-used)
        if tab.custom:
            res = self._mask_custom(cells, res, refine_geometry, only, apply)
        return res

    def _mask_custom(self, cells, res, refine_geometry, only, apply) -> np.ndarray:
        """Geometries without a device lowering: call their Python check_cell per cell, as the reference does."""
        idx = pt.tensor(list(cells), dtype=pt.int64, device=self._device)
        c = self._center[idx].cpu()
        lv = self._level[idx].cpu()
        d = self._n_dimensions
        dirs = pt.tensor([[-1, -1], [-1, 1], [1, 1], [1, -1]] if d == 2 else
                         [[-1, -1, 1], [-1, 1, 1], [1, 1, 1], [1, -1, 1], [-1, -1, -1], [-1, 1, -1], [1, 1, -1],
                          [1, -1, -1]], dtype=pt.float64)
        newly = []
        for t in range(len(res)):
            if res[t]:
                continue
            nodes = c[t].unsqueeze(0) + dirs * 0.5 * self._width / (2 ** int(lv[t]))
            for gi in self._geom_table.custom:
                if only >= 0 and gi != only:
                    continue
                if self._geometry[gi].check_cell(nodes, refine_geometry):
                    res[t] = True
                    newly.append(int(idx[t]))
                    break
        if apply and newly:
            ii = pt.tensor(newly, dtype=pt.int64, device=self._device)
            self._flags[ii] = FLAG_INVALID
            self._gain[ii] = 0.0
        return res

    def _remove_invalid_cells(self, _refined_cells, _refine_geometry: bool = False, _geometry_no=None):
        """
        s_cube.py:669-732. ``_refined_cells`` is a range (new cells) or a set (geometry refinement); returns ``None``
        or, in refine mode, the set of cells touching the geometry built the way the reference builds it.
        """
        if self._pre_select:
            # s_cube.py:1832-1836: with pre_select_cells=True the `elif g.check_cell(...)` branch is never taken,
            # so the reference marks no cell at all. Mirrored, not "fixed".
            return None
        if isinstance(_refined_cells, range):
            flags = self._mask(_refined_cells, _refine_geometry, _geometry_no)
            if not flags.any():
                return None                                      # no cell to drop (the common case): nothing to order
            order = list({c for c in _refined_cells})            # the reference passes a set comprehension
            lookup = dict(zip(_refined_cells, flags.tolist()))
            result = [c if lookup[c] else None for c in order]
        else:
            order = list(_refined_cells)
            flags = self._mask(order, _refine_geometry, _geometry_no)
            result = [c if f else None for c, f in zip(order, flags.tolist())]
        _idx = set(filter(None, result))
        if _idx == set():
            return None
        elif _refine_geometry:
            return _idx
        for c in _idx:
            self._invalid_h[c] = True
        self._topo.mark_invalid(list(_idx))                  # neighbour reset, s_cube.py:721-731
        self._leaf_cells -= _idx
        return None

    def _refine_uniform(self) -> None:
        # s_cube.py:508-561
        logger.info("Starting uniform refinement.")
        self._times["t_start_uniform"] = time()
        for j in range(self._min_level):
            logger.info(f"\r\tStarting iteration no. {j}, N_cells = {len(self._leaf_cells)}")
            parents = list(self._leaf_cells)
            new_cells = self._refine_cells(parents)
            self._topo.refresh_children(parents)             # second pass, s_cube.py:547-549
            self._current_min_level += 1
            self._remove_invalid_cells(new_cells)
        self._current_max_level = max(self._current_max_level, self._min_level)
        logger.info("Finished uniform refinement.")
        self._times["t_end_uniform"] = time()

    def _compute_captured_metric(self) -> bool:
        # s_cube.py:317-336; the prediction at a leaf centre is the cell's stored metric (s_cube.py:241)
        if self._fused_sumsq is not None:                # evaluated right behind the mask kernel of this iteration
            sumsq, self._fused_sumsq = self._fused_sumsq, None
        else:
            with pt.cuda.device(self._device):
                _lib.check(self._lib.s3_leaf_sumsq(self._p("_metric_d"), self._p("_flags"), self._n_cells,
                                                   _lib.ptr(self._scalar), self._stream()))
            sumsq = self._scalar.item()
        ratio = float(np.sqrt(sumsq)) / self._target_norm
        self._metric.append(ratio)
        return ratio < self._min_metric

    def _check_stopping_criteria(self) -> bool:
        # s_cube.py:263-284
        if self._n_cells_max is None:
            if len(self._metric) > 1 and self._metric[-1] / self._min_metric >= self._reach_at_least:
                return self._metric[-1] < self._min_metric and abs(self._metric[-1] - self._metric[-2]) > self._relTol
        else:
            if len(self._leaf_cells) / self._n_cells_max >= self._reach_at_least:
                _relStop = abs(self._cells_per_iter / self._n_cells_max - self._cells_per_iter_last / self._n_cells_max)
                return len(self._leaf_cells) < self._n_cells_max and _relStop > self._relTol
        return True

    def _compute_n_cells_per_iter(self) -> None:
        # s_cube.py:286-315
        if self._n_cells_max is None:
            _delta_x = self._min_metric - self._metric[0]
            _current_x = self._metric[-1]
        else:
            _delta_x = self._n_cells_max - self._n_cells_after_uniform
            _current_x = self._n_cells
        _delta_y = self._cells_per_iter_start - self._cells_per_iter_end
        _new = self._cells_per_iter_start - (_delta_y / _delta_x) * _current_x
        self._cells_per_iter_last = self._cells_per_iter
        self._cells_per_iter = int(_new) if _new > 1 else 1

    def _select(self, k: int) -> list:
        """heapq.nlargest(k, leaf_cells, key=(gain, -idx)) on the device (s_cube.py:601-602)."""
        k = min(k, len(self._leaf_cells))
        if k <= 0:
            return []
        spec, self._spec_selection = self._spec_selection, None
        if spec is not None and len(spec) == k:
            return spec                                  # selected behind the previous iteration's mask pass
        out = pt.empty((k,), dtype=pt.int64, device=self._device)
        with pt.cuda.device(self._device):
            _lib.check(self._lib.s3_select_topk(self._p("_gain"), self._p("_flags"), self._n_cells, k,
                                                _lib.ptr(out), self._stream()))
        return out.cpu().tolist()

    def refine(self) -> None:
        # s_cube.py:563-667
        logger.info("Starting grid generation.")
        self._enter_hot_loop()
        self._refine_uniform()
        iteration_count = 0
        self._n_cells_after_uniform = len(self._leaf_cells)
        if self._n_cells_max is None:
            self._compute_captured_metric()
        self._n_cells_log.append(len(self._leaf_cells))

        logger.info("Starting metric-based refinement.")
        self._times["t_start_adaptive"] = time()
        while self._check_stopping_criteria():
            if self._n_cells_max is None:
                logger.info(f"\r\tStarting iteration no. {iteration_count}, captured metric: "
                            f"{round(self._metric[-1] * 100, 2)} %, N_cells = {len(self._leaf_cells)}")
            else:
                logger.info(f"\r\tStarting iteration no. {iteration_count}, N_cells = {len(self._leaf_cells)}")
            if len(self._metric) >= 2:
                self._compute_n_cells_per_iter()

            _leaf_cells_sorted = self._select(min(self._cells_per_iter, self._n_cells))
            if self._selected_log is not None:
                self._selected_log.append(list(_leaf_cells_sorted))
            to_refine = set()
            if not self._max_delta_level:
                # s_cube.py:611 for every selected cell; nothing reads the pointers in between, so one call
                self._topo.refresh_siblings(list(_leaf_cells_sorted))
            for i in _leaf_cells_sorted:
                to_refine.add(i)
                if self._max_delta_level:
                    self._topo.refresh_siblings([i])          # s_cube.py:611
                    nb_to_refine_as_well = set(self._check_nb(i))
                    to_refine.update(self._check_constraint(nb_to_refine_as_well))
            self._fuse_metric = self._n_cells_max is None
            new_cells = self._refine_cells(list(to_refine))
            # the number of cells the next iteration selects is known already when cells_per_iter is constant and the
            # leaves cannot run out: min(cells_per_iter, n_cells, n_leaves) (s_cube.py:601 and heapq.nlargest)
            k_next = min(self._cells_per_iter, self._n_cells)
            constant = self._cells_per_iter_start == self._cells_per_iter_end or self._n_cells_max is not None
            if constant and len(self._leaf_cells) - len(new_cells) >= k_next > 0:
                self._speculate_k = k_next
            self._remove_invalid_cells(new_cells)
            self._fuse_metric = False
            self._speculate_k = 0

            if self._n_cells_max is None:
                self._compute_captured_metric()
            iteration_count += 1
            self._n_cells_log.append(len(self._leaf_cells))

        if self._n_cells_max is not None:
            self._compute_captured_metric()
        logger.info("Finished metric-based refinement.")

        self._refine_geometries()
        self._update_min_ref_level()
        self._resort_nodes_and_indices_of_grid()
        self._create_mesh_info(iteration_count)
        logger.info(self)
        if self._n_cells_max is not None and self._metric[-1] > 1:
            logger.info("Detected a captured metric > 100%. The current 'n_cells_max' can be reduced without further "
                        "loss of information for this metric field.")

    def _update_min_ref_level(self) -> None:
        leaves = np.fromiter(self._leaf_cells, dtype=np.int64, count=len(self._leaf_cells))
        self._current_min_level = max(self._current_min_level, int(self._levels_h[leaves].min()))

    # ------------------------------------------------------------------------------------------ geometry refinement
    def _refine_geometries(self) -> None:
        # s_cube.py:1538-1555
        geometries_to_refine = [idx for idx, g in enumerate(self._geometry) if g.refine]
        if geometries_to_refine:
            self._times["t_start_geometry"] = time()
            self._execute_geometry_refinement(geometries_to_refine)
            self._times["t_end_geometry"] = time()

    def _execute_geometry_refinement(self, _geometries: list) -> None:
        # s_cube.py:774-863
        logger.info("Starting geometry refinement.")
        for g in _geometries:
            logger.info(f"Starting refining geometry {self._geometry[g].name}.")
            found = self._remove_invalid_cells(self._leaf_cells, _refine_geometry=True, _geometry_no=g)
            if found is None:
                logger.warning("Could not find any cells to refine. Skipping geometry refinement.")
                logger.info("Finished geometry refinement.")
                return
            _all_cells = set(found)
            _global_min_level = min([int(self._levels_h[c]) for c in _all_cells])
            if self._geometry[g].min_refinement_level is None:
                _global_max_level = max([int(self._levels_h[c]) for c in _all_cells])
            else:
                _global_max_level = self._geometry[g].min_refinement_level
            logger.info(f"Found a minimum cell level of {_global_min_level}. Target level is {_global_max_level}.")

            while _global_max_level > _global_min_level:
                logger.info(f"\r\t\t\t\t\t\t\t\t\tRefining level {_global_min_level + 1} / {_global_max_level}.")
                to_refine, checked, refresh = set(), set(), []
                for i in _all_cells:
                    if i in checked:
                        continue
                    if self._levels_h[i] < _global_max_level:
                        to_refine.add(i)
                        if self._max_delta_level:             # s_cube.py:826
                            self._topo.refresh_siblings([i])
                        else:
                            refresh.append(i)                 # nothing reads the pointers inside this loop
                    if self._max_delta_level:
                        nb_to_refine_as_well = set(self._check_nb(i))
                        nb_to_refine_as_well.update(self._check_constraint(nb_to_refine_as_well))
                        to_refine.update(nb_to_refine_as_well)
                        checked.update(nb_to_refine_as_well)
                if refresh:
                    self._topo.refresh_siblings(refresh)
                new_cells = self._refine_cells(list(to_refine))
                _idx_new = {c for c in new_cells}
                # children are only tested against the geometry being refined (s_cube.py:850)
                self._remove_invalid_cells(new_cells, _geometry_no=g)
                found = self._remove_invalid_cells({i for i in _idx_new if not self._invalid_h[i]},
                                                   _refine_geometry=True, _geometry_no=g)
                if found is None:
                    # the reference would raise a TypeError here (set(None), s_cube.py:855); stop refining instead
                    logger.warning("No cell near the geometry left to refine.")
                    break
                _all_cells = set(found)
                _global_min_level += 1
        leaves = np.fromiter(self._leaf_cells, dtype=np.int64, count=len(self._leaf_cells))
        self._current_max_level = int(self._levels_h[leaves].max())
        logger.info("Finished geometry refinement.")

    # ------------------------------------------------------------------------------------------ final grid
    def _resort_nodes_and_indices_of_grid(self) -> None:
        # s_cube.py:734-772
        logger.info("Starting renumbering final mesh.")
        self._times["t_start_renumber"] = time()
        leaf_order = list(self._leaf_cells)                      # centers / levels: leaf-set order (:770-771)
        ascending = sorted(leaf_order)                           # faces: cell-list order (:748)
        if leaf_order != ascending:
            logger.warning("Leaf-set iteration order differs from ascending cell index; 'centers' and 'faces' follow "
                           "the reference's two different orders.")
        order_d = pt.tensor(leaf_order, dtype=pt.int64, device=self._device)
        # the reference's node table: shared ids from the replayed pointers, unused ids squeezed out (:750-771)
        self._topo.sync()
        faces, vertices, _ = self._topo.final()
        assert faces.shape[0] == len(leaf_order), "host topology and device cell state disagree on the leaf cells"
        self.face_ids = pt.from_numpy(faces)
        self.all_nodes = pt.from_numpy(vertices)
        self.all_centers = self._center[order_d].cpu()
        self.all_levels = self._level[order_d].to(pt.int64).cpu().unsqueeze(-1)
        self._topo = None                                     # native handle: not part of the pickled object
        self._times["t_end_renumber"] = time()

    def _create_mesh_info(self, counter: int) -> None:
        # s_cube.py:1557-1584 (same keys)
        m = self.data_final_mesh
        m["size_initial_cell"] = self._width
        m["n_cells_orig"] = self._n_cells_orig
        m["n_cells"] = len(self._leaf_cells)
        m["iterations"] = counter
        m["min_level"] = self._current_min_level
        m["max_level"] = self._current_max_level
        m["metric_per_iter"] = self._metric
        m["cells_per_iter"] = self._n_cells_log
        m["t_total"] = self._times["t_end_renumber"] - self._times["t_start_uniform"]
        m["t_uniform"] = self._times["t_end_uniform"] - self._times["t_start_uniform"]
        m["t_renumbering"] = self._times["t_end_renumber"] - self._times["t_start_renumber"]
        if self._times["t_end_geometry"] > 0:
            m["t_geometry"] = self._times["t_end_geometry"] - self._times["t_start_geometry"]
            m["t_adaptive"] = self._times["t_start_geometry"] - self._times["t_start_adaptive"]
        else:
            m["t_geometry"] = None
            m["t_adaptive"] = self._times["t_start_renumber"] - self._times["t_start_adaptive"]
        m["t_knn_build"] = self._t_knn_build

    def __len__(self):
        return self._n_cells

    def __str__(self) -> str:
        m = self.data_final_mesh
        message = [f"Finished refinement in {m['t_total']:2.4f} s ({m['iterations']} iterations).",
                   f"Time for uniform refinement: {m['t_uniform']:2.4f} s",
                   f"Time for metric-based refinement: {m['t_adaptive']:2.4f} s"]
        if m["t_geometry"] is not None:
            message += [f"Time for geometry refinement: {m['t_geometry']:2.4f} s"]
        message += [f"Time for renumbering the final mesh: {m['t_renumbering']:2.4f} s",
                    f"Number of cells: {len(self._leaf_cells)}", f"Minimum ref. level: {self._current_min_level}",
                    f"Maximum ref. level: {self._current_max_level}",
                    f"Captured metric of original grid: {self._metric[-1] * 100:.2f} %"]
        return "\n\t".join(message)

    @property
    def n_dimensions(self) -> int:
        return self._n_dimensions

    @property
    def width(self):
        return self._width

    @property
    def geometry(self) -> list:
        return self._geometry

"""
API facade of S^3: same constructor arguments, attributes and output files as the reference's
``SparseSpatialSampling`` (sparseSpatialSampling/sparse_spatial_sampling.py:20-186); the grid generation itself
runs on the GPU (``s_cube.SamplingTree``).
"""
import inspect
import logging
import textwrap
from os import makedirs, path
from os.path import join
from typing import Union

import torch as pt

from .s_cube import SamplingTree

logger = logging.getLogger(__name__)


class SparseSpatialSampling:
    def __init__(self, coordinates: pt.Tensor, metric: pt.Tensor, geometry_objects: list, save_path: str,
                 save_name: str, grid_name: str = "grid_s_cube", uniform_levels: int = 5,
                 n_cells_max: Union[int, float] = None, min_metric: float = 0.75, max_delta_level: bool = False,
                 n_cells_iter_start: int = None, n_cells_iter_end: int = None, n_jobs: int = 1,
                 relTol: Union[int, float] = 1e-3, reach_at_least: float = 0.75, pre_select_cells: bool = False):
        self.n_jobs = n_jobs
        self.coordinates = coordinates
        self.metric = metric
        self.save_path = save_path
        self.save_name = save_name
        self.grid_name = grid_name

        # results of the grid generation
        self.centers = None
        self.vertices = None
        self.faces = None
        self.n_dimensions = coordinates.squeeze().size(-1)
        self.size_initial_cell = None
        self.levels = None

        self._geometries = geometry_objects
        self._pre_select_cells = pre_select_cells
        self._level_bounds = int(uniform_levels)
        self._n_cells_max = n_cells_max if n_cells_max is None else int(n_cells_max)
        self._min_metric = min_metric
        self._max_delta_level = max_delta_level
        self._n_cells_iter_start = n_cells_iter_start if n_cells_iter_start is None else int(n_cells_iter_start)
        self._n_cells_iter_end = n_cells_iter_end if n_cells_iter_end is None else int(n_cells_iter_end)
        self._relTol = relTol
        self._reach_at_least = reach_at_least
        self._check_input()

        self._sampling = SamplingTree(self.coordinates, self.metric, self._geometries, n_cells=self._n_cells_max,
                                      uniform_level=self._level_bounds, min_metric=self._min_metric,
                                      max_delta_level=self._max_delta_level, n_cells_iter_end=self._n_cells_iter_end,
                                      n_cells_iter_start=self._n_cells_iter_start, n_jobs=self.n_jobs,
                                      relTol=self._relTol, reach_at_least=self._reach_at_least,
                                      pre_select=self._pre_select_cells)

    def execute_grid_generation(self) -> None:
        """Run S^3; afterwards ``centers, vertices, faces, levels, size_initial_cell`` are set (CPU tensors) and
        ``mesh_info_<save_name>.pt`` / ``s_cube_<save_name>.pt`` are written, as the reference does (:116-146)."""
        if not path.exists(self.save_path):
            makedirs(self.save_path)
        self._sampling.refine()
        pt.save(self._sampling.data_final_mesh, join(self.save_path, f"mesh_info_{self.save_name}.pt"))
        self.mesh_info = dict(self._sampling.data_final_mesh)
        self.levels = self._sampling.all_levels
        self.centers = self._sampling.all_centers
        self.vertices = self._sampling.all_nodes
        self.faces = self._sampling.face_ids
        self.size_initial_cell = self._sampling.data_final_mesh["size_initial_cell"]
        self._sampling = None
        pt.save(self, join(self.save_path, f"s_cube_{self.save_name}.pt"))

    def _check_input(self) -> None:
        """
        Argument validation with the reference's outcomes (sparse_spatial_sampling.py:148-186: which inputs are
        rejected, which are silently corrected), worded independently.
        """
        problems = []
        if self.metric.dim() != 1:
            problems.append(f"`metric` has shape {tuple(self.metric.shape)}; S^3 needs one value per point, i.e. a 1-D "
                            f"tensor with {self.coordinates.size(0)} entries")
        if not self._geometries:
            problems.append("`geometry_objects` is empty; pass at least the geometry that spans the numerical domain")
        elif not any(bool(g.keep_inside) for g in self._geometries):
            problems.append("none of the geometries has keep_inside=True, so nothing defines the numerical domain")
        if problems:
            raise AssertionError("invalid input for SparseSpatialSampling: " + "; ".join(problems))
        if self._n_cells_max is None and self._min_metric > 1:
            logger.warning("min_metric = %s exceeds 100 %% of the metric; using 1.0 instead.", self._min_metric)
            self._min_metric = 1
        if self._level_bounds <= 0:
            logger.warning("uniform_levels = %s is not a positive number of levels; using 1 instead.", self._level_bounds)
            self._level_bounds = 1
        if self._n_cells_max is not None:
            logger.warning("n_cells_max = %s is set: the refinement stops on the cell budget and ignores min_metric.",
                           self._n_cells_max)
        if self._pre_select_cells:
            # the reference's validity check (s_cube.py:1832-1836) never reaches the full geometry test when the
            # bounding-box pre-selection is on, so NO cell is masked at all; mirrored for parity, but say so
            logger.warning("pre_select_cells=True reproduces the reference's behaviour of skipping every geometry mask: "
                           "cells inside bodies / outside the domain stay in the grid and geometry refinement finds "
                           "nothing. Leave it False unless that is what you need.")


def list_geometries() -> None:
    """Log all available geometry classes with their one-line description (reference :190-212)."""
    from . import geometry
    from .geometry.base import GeometryObject
    classes = [obj for _, obj in inspect.getmembers(geometry, inspect.isclass)
               if issubclass(obj, GeometryObject) and obj is not GeometryObject]
    width = max(len(c.__name__) for c in classes)
    lines = ["\n\tAvailable geometry objects:", "\t---------------------------"]
    for c in sorted(classes, key=lambda c: c.__name__):
        desc = textwrap.shorten(getattr(c, "__short_description__", ""), width=100, placeholder="…")
        lines.append(f"\t\t- {c.__name__.ljust(width)} : {desc}")
    logger.info("\n".join(lines))

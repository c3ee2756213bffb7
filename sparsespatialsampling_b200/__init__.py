"""
s3-b200: the data-parallel hot path of Sparse Spatial Sampling (S^3) on NVIDIA B200 (sm_100a).

Same Python surface as the reference package ``sparseSpatialSampling`` for the grid generation
(``SparseSpatialSampling.execute_grid_generation``), the geometry objects' ``check_cell`` contract and the export
stage (``ExportData.export`` / ``interpolate_data``); the work is done by hand-written CUDA kernels behind the C-ABI
in ``include/s3b200.h``. There is no CPU fallback.
"""
import logging as _logging

from .sparse_spatial_sampling import SparseSpatialSampling, list_geometries
from .s_cube import SamplingTree
from .interpolate import interpolate_data, interp_gather
from .knn import KnnIndex
from .export import ExportData, Fields
from .data import Datawriter, Dataloader, XDMFWriter
from .svd import compute_svd, compute_svd_sharded
from .reconstruction import ReconstructionError, ErrorStats
from .dmd import compute_dmd, DMD
from .utils import write_svd_s_cube_to_file, write_dmd_s_cube_to_file, export_fields_batchwise, export_openfoam_fields
from . import geometry

_logging.getLogger(__name__).addHandler(_logging.NullHandler())

__version__ = "0.1.0"
__all__ = ["SparseSpatialSampling", "SamplingTree", "list_geometries", "interpolate_data", "interp_gather", "KnnIndex",
           "ExportData", "Fields", "Datawriter", "Dataloader", "XDMFWriter", "compute_svd", "compute_svd_sharded", "ReconstructionError", "ErrorStats",
           "compute_dmd", "DMD", "write_svd_s_cube_to_file", "write_dmd_s_cube_to_file", "export_fields_batchwise", "export_openfoam_fields",
           "geometry"]

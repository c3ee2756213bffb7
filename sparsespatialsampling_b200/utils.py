"""
Workflow helpers of the reference that sit on the accelerated path (sparseSpatialSampling/utils.py):
``compute_svd`` (utils.py:302-346) and ``write_svd_s_cube_to_file`` (utils.py:349-413), and the DMD counterpart
``write_dmd_s_cube_to_file``.

The OpenFOAM loaders of the reference (``load_foam_data``, ``load_original_Foam_fields``, ``export_openfoam_fields``,
utils.py:23-299) are file I/O through flowtorch and out of scope (SURVEY.md section 2).
"""
import logging
from typing import Union

from .data import Dataloader, Datawriter
from .dmd import compute_dmd
from .svd import compute_svd

logger = logging.getLogger(__name__)

__all__ = ["compute_svd", "write_svd_s_cube_to_file", "write_dmd_s_cube_to_file"]


def write_svd_s_cube_to_file(field_names: Union[list, str], load_dir: str, file_name: str, new_file: bool,
                             n_modes: int = None, rank=None, t_start: Union[int, float] = 0,
                             method: str = "tc3") -> None:
    """
    SVD of exported fields, written as ``<file_name>_<field>_svd.h5`` (+ XDMF): modes ``mode_1..n`` , ``V``, ``s``,
    ``cell_area`` in ``constant`` (utils.py:349-413). Same arguments as the reference plus ``method`` (Gram kernel).
    Only the ``n_modes`` modes that are written are projected on the device; ``s`` and ``V`` keep ``rank`` entries.
    """
    if type(field_names) is str:
        field_names = [field_names]

    for f in field_names:
        logger.info(f"Performing SVD for field {f}.")
        _name = f"{file_name}_{f}" if new_file else file_name
        dataloader = Dataloader(load_dir, f"{_name}.h5")
        _write_times = sorted([t for t in dataloader.write_times if float(t) >= t_start], key=lambda x: float(x))

        # data matrix of the field, SVD weighted with the cell areas
        s, U, V = compute_svd(dataloader.load_snapshot(f, _write_times), dataloader.weights, rank, method=method,
                              n_modes=n_modes)

        datawriter = Datawriter(load_dir, file_name + f"_{f}_svd.h5")
        datawriter.write_grid(dataloader)

        n_write = U.size(-1) if n_modes is None else n_modes
        if n_write > U.size(-1):
            logger.warning(f"Number of modes to write is set to {n_write}, but found only {U.size(-1)} modes to write.")
            n_write = U.size(-1)

        # each mode is written as an independent field
        for i in range(n_write):
            datawriter.write_data(f"mode_{i + 1}", group="constant", data=U[..., i].squeeze())

        # not referenced by the XDMF file
        datawriter.write_data("V", group="constant", data=V)
        datawriter.write_data("s", group="constant", data=s)
        datawriter.write_data("cell_area", group="constant", data=dataloader.weights)
        datawriter.write_xdmf_file()


def uniform_time_step(write_times) -> float:
    """Spacing of ``write_times``; a spacing that varies by more than 1e-6 of itself raises ``ValueError``."""
    times = sorted(float(t) for t in write_times)
    if len(times) < 2:
        raise ValueError(f"a time step needs at least 2 write times, got {len(times)}")
    steps = [b - a for a, b in zip(times[:-1], times[1:])]
    dt = (times[-1] - times[0]) / (len(times) - 1)
    if dt <= 0 or max(abs(d - dt) for d in steps) > 1e-6 * dt:
        raise ValueError(f"write times are not uniformly spaced (steps {min(steps)} .. {max(steps)}); pass dt")
    return dt


def write_dmd_s_cube_to_file(field_names: Union[list, str], load_dir: str, file_name: str, new_file: bool,
                             dt: float = None, n_modes: int = None, rank=None, t_start: Union[int, float] = 0,
                             method: str = "tc3") -> None:
    """
    DMD of exported fields (``compute_dmd``), written as ``<file_name>_<field>_dmd.h5`` (+ XDMF), arguments as
    ``write_svd_s_cube_to_file``; ``dt = None`` takes the spacing of the write times. The file format has no complex
    type, so ``constant`` holds real / imaginary pairs: ``mode_<i>_real`` / ``mode_<i>_imag`` (i = 1..n, ordered by
    ``|amplitude|``), ``eigvals_real`` / ``eigvals_imag``, ``amplitude_real`` / ``amplitude_imag``, and ``frequency``,
    ``growth_rate``, ``s``, ``cell_area``.
    """
    if type(field_names) is str:
        field_names = [field_names]

    for f in field_names:
        logger.info(f"Performing DMD for field {f}.")
        _name = f"{file_name}_{f}" if new_file else file_name
        dataloader = Dataloader(load_dir, f"{_name}.h5")
        _write_times = sorted([t for t in dataloader.write_times if float(t) >= t_start], key=lambda x: float(x))
        step = uniform_time_step(_write_times) if dt is None else dt
        dmd = compute_dmd(dataloader.load_snapshot(f, _write_times), dataloader.weights, step, rank=rank,
                          n_modes=n_modes, method=method)

        datawriter = Datawriter(load_dir, file_name + f"_{f}_dmd.h5")
        datawriter.write_grid(dataloader)
        modes = dmd.modes.cpu()
        for i in range(dmd.n_modes):
            datawriter.write_data(f"mode_{i + 1}_real", group="constant", data=modes[..., i].real.contiguous().squeeze())
            datawriter.write_data(f"mode_{i + 1}_imag", group="constant", data=modes[..., i].imag.contiguous().squeeze())
        for name in ("eigvals", "amplitude"):
            value = getattr(dmd, name).cpu()
            datawriter.write_data(f"{name}_real", group="constant", data=value.real.contiguous())
            datawriter.write_data(f"{name}_imag", group="constant", data=value.imag.contiguous())
        datawriter.write_data("frequency", group="constant", data=dmd.frequency.cpu())
        datawriter.write_data("growth_rate", group="constant", data=dmd.growth_rate.cpu())
        datawriter.write_data("s", group="constant", data=dmd.s.cpu())
        datawriter.write_data("cell_area", group="constant", data=dataloader.weights)
        datawriter.write_xdmf_file()


def export_fields_batchwise(datawriter, load_batch, fields: Union[list, str], batch_size: int = None) -> None:
    """
    The batch loop of the reference's ``export_openfoam_fields`` (utils.py:204-226) with the data source factored out:
    every field is exported in batches of ``batch_size`` snapshots, each batch is one ``ExportData.export`` call with
    ``n_snapshots_total = len(write_times)``, a batch whose data is ``None`` (field not available) is skipped.

    :param datawriter: ``ExportData`` object with ``write_times`` set
    :param load_batch: ``load_batch(field_name, write_times_of_the_batch) -> (coordinates, data | None)``, data
        ``[N, D, T_batch]`` (vector) or ``[N, 1, T_batch]`` (scalar) -- e.g. a reader of the solver's output. Host
        batches are staged through pinned memory and stream through the device while the next batch is being read.
    :param fields: field name or list of field names
    :param batch_size: snapshots per batch, ``None`` = all at once
    """
    if datawriter.write_times is None:
        raise ValueError("Couldn't find any ``write_times`` for export. Set ``datawriter.write_times`` first.")
    times = datawriter.write_times
    batch_size = batch_size if batch_size is not None else len(times)
    if type(fields) is str:
        fields = [fields]
    n_batches = len(times) // batch_size + (1 if len(times) % batch_size else 0)
    for f in fields:
        for counter, t in enumerate(range(0, len(times), batch_size), start=1):
            logger.info(f"Exporting batch {counter} / {n_batches}")
            coordinates, data = load_batch(f, times[t:t + batch_size])
            if data is not None:
                datawriter.export(coordinates, data, f, n_snapshots_total=len(times))


def export_openfoam_fields(datawriter, load_path: str, boundaries: list, batch_size: int = None,
                           fields: Union[list, str] = None) -> None:
    """
    Drop-in for the reference's ``export_openfoam_fields`` (utils.py:155-226). Reading OpenFOAM cases is delegated to
    ``flowtorch`` (``FOAMDataloader`` / ``mask_box``) exactly as the reference does; it is an optional dependency that is
    not part of this package -- without it an ``ImportError`` says so. The loop itself is ``export_fields_batchwise``.
    """
    try:
        from flowtorch.data import FOAMDataloader, mask_box
    except ImportError as e:
        raise ImportError("export_openfoam_fields reads the OpenFOAM case with flowtorch (as the reference does); "
                          "install flowtorch or use export_fields_batchwise with your own reader.") from e
    import torch as pt
    loader = FOAMDataloader(load_path)
    n_dim = datawriter.n_dimensions
    vertices = loader.vertices if n_dim == 3 else loader.vertices[:, :2]
    mask = mask_box(vertices, lower=boundaries[0], upper=boundaries[1])
    coord = pt.stack([pt.masked_select(vertices[:, d], mask) for d in range(n_dim)], dim=1)
    if datawriter.write_times is None:
        datawriter.write_times = [t for t in loader.write_times[1:]]
    if fields is None:
        fields = loader.field_names[datawriter.write_times[0]]

    def load_batch(field, times):
        # load_original_Foam_fields, utils.py:106-143, for one field
        try:
            size = loader.load_snapshot(field, times[0]).size()
        except ValueError:
            logger.warning(f"Field '{field}' is not available. Skipping field {field}.")
            return None, None
        scalar = len(size) == 1
        data = pt.zeros((coord.size(0), 1 if scalar else size[1], len(times)), dtype=pt.float32)
        m = mask if scalar else mask.unsqueeze(-1).expand(size)
        try:
            for i, t in enumerate(times):
                data[:, :, i] = pt.masked_select(loader.load_snapshot(field, t), m).reshape(coord.size(0), -1)
        except RuntimeError:
            logger.warning(f"Field '{field}' is does not match the size of the masked domain. Skipping field {field}.")
            return None, None
        return coord, data

    export_fields_batchwise(datawriter, load_batch, fields, batch_size)

"""Molecular-dynamics trajectory — drop-in for ``ramannoodle.dynamics.Trajectory``
(``ramannoodle/dynamics/_trajectory.py:16-109``).

Host (numpy) trajectories are stored wrapped (``apply_pbc``) like the reference, by default
in page-locked memory so that ``get_raman_spectrum`` streams them to the GPU at full PCIe
bandwidth.  A trajectory may also be created from a CUDA tensor, in which case it stays
resident in HBM (the wrap runs on the device) and evaluation involves no host transfer.
"""
from __future__ import annotations

import ctypes
from collections.abc import Sequence

import numpy as np

from . import _lib
from .abstract import Dynamics, PolarizabilityModel
from .exceptions import get_type_error, verify_ndarray_shape
from .spectrum import MDRamanSpectrum, PhononRamanSpectrum

RAMAN_TENSOR_CENTRAL_DIFFERENCE = 0.001  # ramannoodle/constants.py:248


def apply_pbc(positions):
    """``ramannoodle/structure/utils.py:13-29``: ``positions - positions // 1`` (host)."""
    try:
        return positions - positions // 1
    except TypeError as exc:
        raise get_type_error("positions", positions, "ndarray") from exc


class Trajectory(Dynamics, Sequence):
    """Positions time series (S,N,3) (fractional) plus a timestep (fs)."""

    def __init__(self, positions_ts, timestep: float, pin_memory: bool = True) -> None:
        verify_ndarray_shape("positions_ts", positions_ts, (None, None, 3))
        try:
            timestep = float(timestep)
        except TypeError as exc:
            raise get_type_error("timestep", timestep, "float") from exc
        if timestep <= 0:
            raise ValueError("timestep must be positive")
        self._timestep = timestep
        self._pinned_owner = None
        if _lib.is_torch_tensor(positions_ts):
            self._positions_ts = self._wrap_device(positions_ts, pin_memory)
        else:
            self._positions_ts = self._wrap_host(np.asarray(positions_ts), pin_memory)

    @classmethod
    def _from_wrapped(cls, positions: np.ndarray, timestep: float, pinned_owner=None) -> "Trajectory":
        """Adopts host positions that are already wrapped into [0,1) (``io.read_trajectory`` parses
        straight into a page-locked buffer) without another pass over them."""
        verify_ndarray_shape("positions_ts", positions, (None, None, 3))
        self = cls.__new__(cls)
        timestep = float(timestep)
        if timestep <= 0:
            raise ValueError("timestep must be positive")
        self._timestep = timestep
        self._pinned_owner = pinned_owner
        self._positions_ts = positions
        return self

    def _wrap_device(self, tensor, pin_memory: bool = True):
        import torch  # pylint: disable=import-outside-toplevel

        if not tensor.is_cuda:  # a CPU tensor is host data: same path (and pinned owner) as an ndarray
            return self._wrap_host(tensor.detach().cpu().numpy(), pin_memory)
        data = tensor.to(torch.float64).contiguous()
        out = torch.empty_like(data)
        device = int(data.device.index or 0)
        _lib.require_device(device)
        with torch.cuda.device(device):
            status = _lib.lib().rn_apply_pbc(ctypes.c_void_p(data.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                             data.numel(), _lib.current_stream(device))
        _lib.check(status, "rn_apply_pbc")
        return out

    def _wrap_host(self, positions: np.ndarray, pin_memory: bool) -> np.ndarray:
        """``apply_pbc(positions)`` into a fresh (page-locked, when a GPU is present) buffer.  float64
        input goes through the library's threaded ``rn_host_apply_pbc`` (bit-identical to
        ``positions - positions // 1``; numpy's ``floor_divide`` needs ~17 s for a 1M-frame,
        192-atom trajectory), anything else through numpy."""
        wrapped = None
        if pin_memory and positions.size > 0:
            try:
                import torch  # pylint: disable=import-outside-toplevel

                if torch.cuda.is_available():
                    owner = torch.empty(positions.shape, dtype=torch.float64, pin_memory=True)
                    wrapped = owner.numpy()
                    self._pinned_owner = owner
            except (ImportError, RuntimeError):
                wrapped = None
                self._pinned_owner = None
        if positions.dtype == np.float64 and positions.size > 0:
            source = np.ascontiguousarray(positions)
            if wrapped is None:
                wrapped = np.empty(positions.shape, dtype=np.float64)
            status = _lib.lib().rn_host_apply_pbc(ctypes.c_void_p(source.ctypes.data),
                                                  ctypes.c_void_p(wrapped.ctypes.data), source.size, 0)
            _lib.check(status, "rn_host_apply_pbc")
            return wrapped
        if wrapped is not None:
            np.floor_divide(positions, 1, out=wrapped)  # positions // 1
            np.subtract(positions, wrapped, out=wrapped)  # positions - positions // 1
            return wrapped
        return np.asarray(apply_pbc(positions), dtype=np.float64)

    @property
    def positions_ts(self) -> np.ndarray:
        """(A copy of) the wrapped positions time series, shape (S,N,3)."""
        if _lib.is_torch_tensor(self._positions_ts):
            return self._positions_ts.cpu().numpy()
        return self._positions_ts.copy()

    @property
    def timestep(self) -> float:
        return self._timestep

    @property
    def is_device_resident(self) -> bool:
        return _lib.is_torch_tensor(self._positions_ts)

    def get_raman_spectrum(self, polarizability_model: PolarizabilityModel) -> MDRamanSpectrum:
        """One ``calc_polarizabilities`` call over the whole trajectory, wrapped into an
        ``MDRamanSpectrum`` (``_trajectory.py:71-90``).  With this package's models the
        polarizability series stays on the GPU for ``measure``."""
        try:
            to_device = getattr(polarizability_model, "calc_polarizabilities_to_device", None)
            if to_device is not None and not self.is_device_resident:
                polarizability_ts = to_device(self._positions_ts)
            else:
                polarizability_ts = polarizability_model.calc_polarizabilities(self._positions_ts)
        except ValueError as exc:
            raise ValueError("polarizability_model and trajectory are incompatible") from exc
        return MDRamanSpectrum(polarizability_ts, self._timestep)

    def get_raman_spectra(self, polarizability_models) -> list:
        """Mask sweep (SURVEY.md §8f N3): one ``MDRamanSpectrum`` per model, all evaluated in a
        single pass over the trajectory (``pmodel.calc_polarizabilities_sweep``).  Equivalent to
        ``[self.get_raman_spectrum(m) for m in polarizability_models]``, which is how the
        reference evaluates ``get_masked_model`` copies (``_interpolation.py:697-708``)."""
        from .pmodel import calc_polarizabilities_sweep  # pylint: disable=import-outside-toplevel

        try:
            series = calc_polarizabilities_sweep(polarizability_models, self._positions_ts, to_device=True)
        except ValueError as exc:
            raise ValueError("polarizability_model and trajectory are incompatible") from exc
        return [MDRamanSpectrum(series[g], self._timestep) for g in range(series.shape[0])]

    def __len__(self) -> int:
        return int(self._positions_ts.shape[0])

    def __getitem__(self, key):
        try:
            item = self._positions_ts[key]
        except IndexError as exc:
            if "out of bounds" in str(exc) or "out of range" in str(exc):
                raise IndexError("trajectory index out of bounds") from exc
            raise exc
        return item.cpu().numpy() if _lib.is_torch_tensor(item) else item


class Phonons(Dynamics):
    """Harmonic lattice vibrations — drop-in for ``ramannoodle.dynamics.Phonons``
    (``ramannoodle/dynamics/_phonon.py:13-108``).

    The reference evaluates two S=1 batches per mode in a Python loop (``_phonon.py:93-106``);
    here the 2·M central-difference geometries are stacked into ONE ``calc_polarizabilities``
    call of shape (2M,N,3), so the whole phonon spectrum is a single kernel launch."""

    def __init__(self, ref_positions, wavenumbers, displacements) -> None:
        verify_ndarray_shape("ref_positions", ref_positions, (None, 3))
        verify_ndarray_shape("wavenumbers", wavenumbers, (None,))
        verify_ndarray_shape("displacements", displacements, (wavenumbers.size, ref_positions.shape[0], 3))
        self._ref_positions = ref_positions
        self._wavenumbers = wavenumbers
        self._displacements = displacements

    @property
    def ref_positions(self) -> np.ndarray:
        return self._ref_positions.copy()

    @property
    def wavenumbers(self) -> np.ndarray:
        return self._wavenumbers.copy()

    @property
    def displacements(self) -> np.ndarray:
        return self._displacements.copy()

    def get_raman_spectrum(self, polarizability_model: PolarizabilityModel) -> PhononRamanSpectrum:
        epsilon = self._displacements * RAMAN_TENSOR_CENTRAL_DIFFERENCE
        batch = np.concatenate([self._ref_positions[None] + epsilon, self._ref_positions[None] - epsilon])
        try:
            polarizabilities = polarizability_model.calc_polarizabilities(batch)
        except ValueError as exc:
            raise ValueError("polarizability_model and phonons are incompatible") from exc
        modes = self._wavenumbers.size
        raman_tensors = (polarizabilities[:modes] - polarizabilities[modes:]) / RAMAN_TENSOR_CENTRAL_DIFFERENCE
        return PhononRamanSpectrum(self._wavenumbers, np.asarray(raman_tensors))

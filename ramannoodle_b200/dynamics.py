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
from .spectrum import MDRamanSpectrum, PhononRamanSpectrum, _current_device, _get_plan, _is_integer, _window_batch

RAMAN_TENSOR_CENTRAL_DIFFERENCE = 0.001  # ramannoodle/constants.py:248


def apply_pbc(positions):
    """``ramannoodle/structure/utils.py:13-29``: ``positions - positions // 1`` (host)."""
    try:
        return positions - positions // 1
    except TypeError as exc:
        raise get_type_error("positions", positions, "ndarray") from exc


def _host_array(value):
    return value.detach().cpu().numpy() if _lib.is_torch_tensor(value) else np.asarray(value)


def _check_vdos_args(lattice, atom_groups, atom_weights, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_vdos``; returns the lattice (3,3), the group offsets (G+1,) and atoms of the
    groups as int64, and the weights (N,) or None, all contiguous host arrays."""
    verify_ndarray_shape("lattice", lattice, (3, 3))
    lattice = np.ascontiguousarray(_host_array(lattice), dtype=np.float64)
    if not np.all(np.isfinite(lattice)):
        raise ValueError("lattice contains non-finite values")
    if atom_groups is None:
        atom_groups = [range(num_atoms)]
    if isinstance(atom_groups, (str, bytes)) or not isinstance(atom_groups, (Sequence, np.ndarray)):
        raise get_type_error("atom_groups", atom_groups, "list")
    if len(atom_groups) == 0:
        raise ValueError("atom_groups is empty")
    offsets, atoms = [0], []
    for g, group in enumerate(atom_groups):
        if isinstance(group, (str, bytes)) or not isinstance(group, (Sequence, np.ndarray)):
            raise get_type_error(f"atom_groups[{g}]", group, "list")
        if len(group) == 0:
            raise ValueError(f"atom_groups[{g}] is empty")
        for atom in group:
            if not _is_integer(atom):
                raise get_type_error(f"atom_groups[{g}] entry", atom, "int")
            if not 0 <= atom < num_atoms:
                raise ValueError(f"atom_groups[{g}] has atom index {atom} out of range [0, {num_atoms})")
        if len(set(int(atom) for atom in group)) != len(group):
            raise ValueError(f"atom_groups[{g}] repeats an atom")
        atoms.extend(int(atom) for atom in group)
        offsets.append(len(atoms))
    weights = None
    if atom_weights is not None:
        verify_ndarray_shape("atom_weights", atom_weights, (num_atoms,))
        weights = np.ascontiguousarray(_host_array(atom_weights), dtype=np.float64)
        if not np.all(np.isfinite(weights)) or np.any(weights < 0):
            raise ValueError("atom_weights must be finite and >= 0")
    if num_frames < 2:
        raise ValueError("positions_ts must contain at least 2 frames")
    return lattice, np.asarray(offsets, dtype=np.int64), np.asarray(atoms, dtype=np.int64), weights


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

    def get_vdos_device(self, lattice, atom_groups=None, atom_weights=None):
        """``get_vdos`` with the result left on the GPU (two CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice, offsets, atoms, weights = _check_vdos_args(lattice, atom_groups, atom_weights, num_atoms, num_frames)
        import torch  # pylint: disable=import-outside-toplevel

        points = int(_lib.lib().rn_spectrum_num_points(num_frames))
        positions = self._positions_ts
        if not _lib.is_torch_tensor(positions):  # host (pinned) trajectory: one copy to the device
            positions = torch.from_numpy(np.ascontiguousarray(positions, dtype=np.float64)).to(
                f"cuda:{_current_device()}")
        device = int(positions.device.index or 0)
        num_groups = len(offsets) - 1
        with torch.cuda.device(device):
            wavenumbers = torch.empty(points, dtype=torch.float64, device=positions.device)
            intensities = torch.empty((num_groups, points), dtype=torch.float64, device=positions.device)
            if points > 0:
                slots = int(np.sum((np.diff(offsets) + 1) // 2))
                plan = _get_plan(num_frames, device, _window_batch(num_frames, slots))
                status = _lib.lib().rn_vdos(
                    plan.handle, ctypes.c_void_p(positions.data_ptr()), num_atoms, ctypes.c_void_p(lattice.ctypes.data),
                    None if weights is None else ctypes.c_void_p(weights.ctypes.data),
                    ctypes.c_void_p(offsets.ctypes.data), ctypes.c_void_p(atoms.ctypes.data), num_groups,
                    self._timestep, ctypes.c_void_p(wavenumbers.data_ptr()),
                    ctypes.c_void_p(intensities.data_ptr()), _lib.current_stream(device))
                _lib.check(status, "rn_vdos")
        return wavenumbers, intensities

    def get_vdos(self, lattice, atom_groups=None, atom_weights=None):
        """Vibrational density of states -> (wavenumbers, vdos), numpy arrays of shape (P,) and (G, P),
        P = ceil((S-1)/2) - 1.

        ``lattice`` is the (3,3) cell in Å with lattice vectors as rows (the convention of ``io.read_lattice``
        and the models).  ``atom_groups`` is a sequence of G non-empty sequences of atom indices in [0, N),
        without repeats inside a group (groups may overlap); the default is one group of all atoms.
        ``atom_weights`` (N,) are finite and >= 0 (masses give the mass-weighted VDOS); the default is ones.

        Row g is by definition ``sum_{i in group g} sum_c atom_weights[i] * calc_signal_spectrum(v[:, i, c],
        timestep)[1][1:]`` with the velocities ``v = (d @ lattice) / timestep`` (Å/fs) of the minimum-image
        steps ``d`` between consecutive frames: the power spectrum of the velocities, 0 cm^-1 bin dropped, no
        corrections.  The wavenumbers are those of ``MDRamanSpectrum(series of S frames, timestep).measure()``
        bit for bit, so VDOS and Raman peaks share the bins.  All groups run as one batched transform on the
        GPU.  A device-resident trajectory is read in place; a host trajectory is copied to the device once
        (its S·N·24 bytes must fit there).  Argument errors are raised before any device work.
        """
        wavenumbers, vdos = self.get_vdos_device(lattice, atom_groups, atom_weights)
        return wavenumbers.cpu().numpy(), vdos.cpu().numpy()

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

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


def _check_lattice(lattice) -> np.ndarray:
    """The (3,3) lattice as a contiguous float64 host array; raises for a wrong type, shape or a non-finite entry."""
    verify_ndarray_shape("lattice", lattice, (3, 3))
    lattice = np.ascontiguousarray(_host_array(lattice), dtype=np.float64)
    if not np.all(np.isfinite(lattice)):
        raise ValueError("lattice contains non-finite values")
    return lattice


def _check_atom_groups(atom_groups, num_atoms: int):
    """Validate G atom groups (default: one group of all atoms); returns the group offsets (G+1,) and the atoms of the
    groups (CSR) as contiguous int64 host arrays."""
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
    return np.asarray(offsets, dtype=np.int64), np.asarray(atoms, dtype=np.int64)


def _num_slots(offsets) -> int:
    """The slots of the groups with these offsets: the GPU pairs two memberships of a group per slot."""
    return int(np.sum((np.diff(offsets) + 1) // 2))


def _check_vdos_args(lattice, atom_groups, atom_weights, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_vdos``; returns the lattice (3,3), the group offsets (G+1,) and atoms of the
    groups as int64, and the weights (N,) or None, all contiguous host arrays."""
    lattice = _check_lattice(lattice)
    offsets, atoms = _check_atom_groups(atom_groups, num_atoms)
    weights = None
    if atom_weights is not None:
        verify_ndarray_shape("atom_weights", atom_weights, (num_atoms,))
        weights = np.ascontiguousarray(_host_array(atom_weights), dtype=np.float64)
        if not np.all(np.isfinite(weights)) or np.any(weights < 0):
            raise ValueError("atom_weights must be finite and >= 0")
    if num_frames < 2:
        raise ValueError("positions_ts must contain at least 2 frames")
    return lattice, offsets, atoms, weights


RDF_MAX_BINS = 4096  # one shared-memory histogram of the kernel


def _cell_widths(lattice: np.ndarray):
    """(V, w) of a (3,3) lattice: the volume V = |L_0 . (L_1 x L_2)| (exact for an orthorhombic cell, like the C entry's)
    and the perpendicular widths w_c = V / |L_{c+1} x L_{c+2}|, or None if V is 0."""
    cross = np.cross(lattice[[1, 2, 0]], lattice[[2, 0, 1]])
    volume = abs(float(np.dot(lattice[0], cross[0])))
    return volume, (volume / np.sqrt(np.sum(cross * cross, axis=1)) if volume > 0 else None)


def _check_rdf_args(lattice, r_max, num_bins, atom_groups, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_rdf`` in the order lattice, r_max, num_bins, atom_groups, frames; returns the
    lattice (3,3), r_max as a float, and the group offsets and atoms (CSR, int64)."""
    lattice = _check_lattice(lattice)
    volume, widths = _cell_widths(lattice)
    if not volume > 0:
        raise ValueError("lattice has zero cell volume")
    r_max = _check_cell_r_max(r_max, widths)
    _check_num_bins(num_bins)
    offsets, atoms = _check_atom_groups(atom_groups, num_atoms)
    if num_frames < 1:
        raise ValueError("positions_ts must contain at least 1 frame")
    return lattice, r_max, offsets, atoms


def _check_r_max_type(r_max) -> float:
    """r_max as a float; raises TypeError for a bool or a non-number."""
    if isinstance(r_max, (bool, np.bool_)) or not isinstance(r_max, (int, float, np.integer, np.floating)):
        raise get_type_error("r_max", r_max, "float")
    return float(r_max)


def _check_cell_r_max(r_max, widths) -> float:
    """The r_max of ``get_rdf`` and ``get_distinct_van_hove``: a float with 0 < r_max <= w_min / 2 for the
    perpendicular widths w of the cell."""
    r_max = _check_r_max_type(r_max)
    bound = 0.5 * float(np.min(widths))
    if not (np.isfinite(r_max) and 0 < r_max <= bound):
        raise ValueError(f"r_max must be finite and in (0, {bound:.6g}] Å, half the smallest perpendicular width "
                         f"of the cell (got {r_max})")
    return r_max


def _check_num_bins(num_bins):
    """The histogram bin count of ``get_rdf`` and ``get_van_hove``: an integer in 1..RDF_MAX_BINS."""
    if not _is_integer(num_bins):
        raise get_type_error("num_bins", num_bins, "int")
    if not 1 <= num_bins <= RDF_MAX_BINS:
        raise ValueError(f"num_bins must be in 1..{RDF_MAX_BINS} (got {num_bins})")


def _check_van_hove_args(lattice, lags, r_max, num_bins, atom_groups, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_van_hove`` in the order lattice, lags, r_max, num_bins, atom_groups, frames;
    returns the lattice (3,3), the lags (T,) as int64, r_max as a float, and the group offsets and atoms (CSR, int64)."""
    lattice = _check_lattice(lattice)
    volume, _ = _cell_widths(lattice)
    if not volume > 0:
        raise ValueError("lattice has zero cell volume")
    lags = _check_lags(lags, num_frames)
    r_max = _check_r_max_type(r_max)
    if not (np.isfinite(r_max) and r_max > 0):
        raise ValueError(f"r_max must be finite and > 0 (got {r_max})")
    _check_num_bins(num_bins)
    offsets, atoms = _check_atom_groups(atom_groups, num_atoms)
    if num_frames < 2:
        raise ValueError("positions_ts must contain at least 2 frames")
    return lattice, lags, r_max, offsets, atoms


def _check_lags(lags, num_frames: int) -> np.ndarray:
    """The lags of ``get_van_hove`` and ``get_distinct_van_hove``: T >= 1 strictly increasing integers in [0, S), as
    a contiguous int64 host array."""
    if isinstance(lags, (str, bytes)):
        raise get_type_error("lags", lags, "list")
    lags = np.asarray(_host_array(lags))
    if lags.ndim != 1:
        raise ValueError(f"lags must be 1-D (got shape {lags.shape})")
    if lags.size == 0:
        raise ValueError("lags is empty")
    if lags.dtype.kind not in "iu":
        raise get_type_error("lags", lags, "int")
    lags = lags.astype(np.int64)
    if np.any(np.diff(lags) <= 0):
        raise ValueError("lags must be strictly increasing")
    if lags[0] < 0 or lags[-1] >= num_frames:
        raise ValueError(f"lags must be in [0, {num_frames}) (got {int(lags[0])}..{int(lags[-1])})")
    return np.ascontiguousarray(lags)


def _check_distinct_van_hove_args(lattice, lags, r_max, num_bins, atom_groups, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_distinct_van_hove`` in the order lattice, lags, r_max, num_bins, atom_groups
    (valid lags imply a frame); returns the lattice (3,3), the lags (T,) as int64, r_max as a float, and the group
    offsets and atoms (CSR, int64)."""
    lattice = _check_lattice(lattice)
    volume, widths = _cell_widths(lattice)
    if not volume > 0:
        raise ValueError("lattice has zero cell volume")
    lags = _check_lags(lags, num_frames)
    r_max = _check_cell_r_max(r_max, widths)
    _check_num_bins(num_bins)
    offsets, atoms = _check_atom_groups(atom_groups, num_atoms)
    return lattice, lags, r_max, offsets, atoms


def _check_projection_args(lattice, vectors, num_atoms: int, num_frames: int):
    """Validate the arguments of ``get_projected_vdos``; returns the lattice (3,3) and the vectors (K,N,3) as
    contiguous float64 host arrays."""
    lattice = _check_lattice(lattice)
    verify_ndarray_shape("vectors", vectors, (None, None, 3))
    if vectors.shape[1] != num_atoms:
        raise ValueError(f"vectors has {vectors.shape[1]} atoms, the trajectory {num_atoms}")
    if vectors.shape[0] == 0:
        raise ValueError("vectors is empty")
    vectors = np.ascontiguousarray(_host_array(vectors), dtype=np.float64)
    if not np.all(np.isfinite(vectors)):
        raise ValueError("vectors contains non-finite values")
    if num_frames < 2:
        raise ValueError("positions_ts must contain at least 2 frames")
    return lattice, vectors


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
        positions, device = self._device_positions()
        num_groups = len(offsets) - 1
        with torch.cuda.device(device):
            wavenumbers = torch.empty(points, dtype=torch.float64, device=positions.device)
            intensities = torch.empty((num_groups, points), dtype=torch.float64, device=positions.device)
            if points > 0:
                plan = _get_plan(num_frames, device, _window_batch(num_frames, _num_slots(offsets)))
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

    def _device_positions(self):
        """The positions as a CUDA tensor and its device index: a device trajectory in place, a host (pinned) one
        copied once."""
        positions = self._positions_ts
        if not _lib.is_torch_tensor(positions):
            import torch  # pylint: disable=import-outside-toplevel

            positions = torch.from_numpy(np.ascontiguousarray(positions, dtype=np.float64)).to(
                f"cuda:{_current_device()}")
        return positions, int(positions.device.index or 0)

    def get_projected_vdos_device(self, lattice, vectors):
        """``get_projected_vdos`` with the result left on the GPU (two CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice, vectors = _check_projection_args(lattice, vectors, num_atoms, num_frames)
        import torch  # pylint: disable=import-outside-toplevel

        points = int(_lib.lib().rn_spectrum_num_points(num_frames))
        positions, device = self._device_positions()
        num_vectors = int(vectors.shape[0])
        with torch.cuda.device(device):
            wavenumbers = torch.empty(points, dtype=torch.float64, device=positions.device)
            intensities = torch.empty((num_vectors, points), dtype=torch.float64, device=positions.device)
            if points > 0:
                # a window's three sequences carry six modes
                plan = _get_plan(num_frames, device, _window_batch(num_frames, -(-num_vectors // 6)))
                status = _lib.lib().rn_projected_vdos(
                    plan.handle, ctypes.c_void_p(positions.data_ptr()), num_atoms, ctypes.c_void_p(lattice.ctypes.data),
                    ctypes.c_void_p(vectors.ctypes.data), num_vectors, self._timestep,
                    ctypes.c_void_p(wavenumbers.data_ptr()), ctypes.c_void_p(intensities.data_ptr()),
                    _lib.current_stream(device))
                _lib.check(status, "rn_projected_vdos")
        return wavenumbers, intensities

    def get_projected_vdos(self, lattice, vectors):
        """Power spectra of the velocities projected on K vectors -> (wavenumbers, rows), numpy arrays of shape
        (P,) and (K, P), P = ceil((S-1)/2) - 1.

        ``lattice`` is the (3,3) cell in Å with lattice vectors as rows.  ``vectors`` (K, N, 3), K >= 1, finite,
        numpy, a CPU or a CUDA tensor (read on the host); ``vectors[k, i]`` is a Cartesian 3-vector of atom i.

        Row k is by definition ``calc_signal_spectrum(q_k, timestep)[1][1:]`` of the projected velocity
        ``q_k[n] = sum_{i,c} vectors[k, i, c] * v[n, i, c]``, with the velocities ``v = (d @ lattice) /
        timestep`` (Å/fs) of the minimum-image steps ``d`` between consecutive frames, exactly as ``get_vdos``
        forms them: 0 cm^-1 bin dropped, no corrections.  The rows are in (Å/fs)^2 times the units of
        ``vectors`` squared; the wavenumbers are those of ``MDRamanSpectrum(series of S frames,
        timestep).measure()`` and ``get_vdos`` bit for bit.  A zero vector gives an exactly zero row.

        With ``Phonons.get_mode_vectors`` row k is the spectrum of the normal-mode velocity of mode k: its
        anharmonic frequency and linewidth.  Sum rule: for any 3N orthonormal vectors e_k (over all 3N
        coordinates) and ``vectors[k, i] = sqrt(m_i) e_{k,i}``, ``rows.sum(0)`` equals ``get_vdos(lattice,
        atom_weights=m)[1][0]`` up to rounding, since an orthogonal change of basis commutes with the DFT.

        The projection runs on the FP64 tensor pipe and the rows as one batched transform on the GPU.  A
        device-resident trajectory is read in place; a host trajectory is copied to the device once (its S·N·24
        bytes must fit there).  Argument errors are raised before any device work.
        """
        wavenumbers, rows = self.get_projected_vdos_device(lattice, vectors)
        return wavenumbers.cpu().numpy(), rows.cpu().numpy()

    def get_msd_device(self, lattice, atom_groups=None):
        """``get_msd`` with the result left on the GPU (two CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice = _check_lattice(lattice)
        offsets, atoms = _check_atom_groups(atom_groups, num_atoms)
        if num_frames < 2:
            raise ValueError("positions_ts must contain at least 2 frames")
        import torch  # pylint: disable=import-outside-toplevel

        lib = _lib.lib()
        positions, device = self._device_positions()
        num_groups = len(offsets) - 1
        with torch.cuda.device(device):
            lag_times = torch.arange(num_frames, dtype=torch.float64, device=positions.device) * self._timestep
            msd = torch.empty((num_groups, num_frames), dtype=torch.float64, device=positions.device)
            # a plan of S + 1 frames has M = S and L >= 2S - 1: a linear autocorrelation of S values
            plan = _get_plan(num_frames + 1, device, _window_batch(num_frames + 1, _num_slots(offsets)))
            status = lib.rn_msd(plan.handle, ctypes.c_void_p(positions.data_ptr()), num_atoms,
                                ctypes.c_void_p(lattice.ctypes.data), ctypes.c_void_p(offsets.ctypes.data),
                                ctypes.c_void_p(atoms.ctypes.data), num_groups, ctypes.c_void_p(msd.data_ptr()),
                                _lib.current_stream(device))
            _lib.check(status, "rn_msd")
        return lag_times, msd

    def get_msd(self, lattice, atom_groups=None):
        """Mean squared displacement -> (lag_times, msd), numpy arrays of shape (S,) and (G, S) in fs and Å².

        ``lattice`` and ``atom_groups`` are those of ``get_vdos``: the (3,3) cell in Å with lattice vectors as rows,
        and G non-empty sequences of atom indices in [0, N) without repeats inside a group (groups may overlap); the
        default is one group of all atoms.  ``lag_times`` is ``np.arange(S) * timestep``.

        The path of atom i is unwrapped with the minimum-image steps of ``get_vdos``: with the steps ``d`` between
        consecutive frames, their integer image shifts ``k = x[n+1] - x[n] - d`` and ``K(n) = sum_{j<n} k_j``,
        ``r_i(n) = (x_i(n) - x_i(0) - K_i(n)) @ lattice``.  Row g at lag m is by definition
        ``mean_{i in g} mean_{n < S-m} |r_i(n+m) - r_i(n)|^2``; ``msd[:, 0]`` is exactly 0.  Every lag comes from
        one FFT autocorrelation per pair of atoms on the GPU, so the rounding error at lag m is of the order of
        ``1e-16 * log2(S) * mean_i sum_n |r_i(n)|^2 / (S - m)``, largest at long lags, where few pairs are averaged.
        A device-resident trajectory is read in place; a host trajectory is copied to the device once (its S·N·24
        bytes must fit there).  Argument errors are raised before any device work.

        A diffusion coefficient in Å²/fs is the slope of a linear range of lags over 6, for example
        ``np.polyfit(lag_times[a:b], msd[g, a:b], 1)[0] / 6``.
        """
        lag_times, msd = self.get_msd_device(lattice, atom_groups)
        return lag_times.cpu().numpy(), msd.cpu().numpy()

    def get_rdf_device(self, lattice, r_max, num_bins, atom_groups=None):
        """``get_rdf`` with the result left on the GPU (two CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice, r_max, offsets, atoms = _check_rdf_args(lattice, r_max, num_bins, atom_groups, num_atoms,
                                                         num_frames)
        import torch  # pylint: disable=import-outside-toplevel

        lib = _lib.lib()
        positions, device = self._device_positions()
        num_groups = len(offsets) - 1
        num_bins = int(num_bins)
        radii = (np.arange(num_bins) + 0.5) * (r_max / num_bins)
        with torch.cuda.device(device):
            rdf = torch.empty((num_groups, num_groups, num_bins), dtype=torch.float64, device=positions.device)
            ws_bytes = int(lib.rn_rdf_workspace_size(num_groups, len(atoms), num_bins))
            workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=positions.device)
            status = lib.rn_rdf(ctypes.c_void_p(positions.data_ptr()), num_frames, num_atoms,
                                ctypes.c_void_p(lattice.ctypes.data), r_max, num_bins,
                                ctypes.c_void_p(offsets.ctypes.data), ctypes.c_void_p(atoms.ctypes.data), num_groups,
                                ctypes.c_void_p(rdf.data_ptr()), ctypes.c_void_p(workspace.data_ptr()),
                                _lib.current_stream(device))
            _lib.check(status, "rn_rdf")
            return torch.from_numpy(radii).to(positions.device), rdf

    def get_rdf(self, lattice, r_max, num_bins, atom_groups=None):
        """Radial distribution functions of atom groups -> (r, g), numpy arrays of shape (B,) and (G, G, B).

        ``lattice`` is the (3,3) cell in Å with lattice vectors as rows; ``atom_groups`` are those of ``get_vdos``: G
        non-empty sequences of atom indices in [0, N) without repeats inside a group (groups may overlap), by default
        one group of all atoms.  ``num_bins`` B is an integer in 1..4096, ``r_max`` a float in Å with
        ``0 < r_max <= w_min / 2``, w_c = V / |L_{c+1} x L_{c+2}| the perpendicular widths of the cell: below that
        bound at most one image of a pair lies within r_max and the component-wise minimum image finds it, so no sum
        over images is needed.  A single frame is a valid input.

        With width = r_max / B, ``r = (np.arange(B) + 0.5) * width`` are the bin centres and e_k = k * width the edges.
        For every group pair a <= b and every frame, each pair (i, j) counts into bin k = floor(|v| / width) when
        k < B, with ``v = (d - ceil(d - 0.5)) @ lattice`` and d = x_j - x_i: for a == b the pairs of list positions
        p < q count twice (ordered pairs), for a < b every i in a and j in b with i != j counts once.  Then
        ``g[a, b, k] = count[a, b, k] * V / (S * n_ab * shell_k)`` with V = |det lattice|, n_ab = |a| |b| - |a n b|
        the number of ordered pairs and shell_k = (4 pi / 3)(e_{k+1}^3 - e_k^3); a pair of groups with n_ab = 0 (a
        one-atom group with itself) gets a zero row, and ``g[b, a] == g[a, b]``.  The distances are evaluated in FP64
        with every product and sum rounded on its own, so the counts are exact integers, the same for every launch
        configuration and for host and device trajectories.

        The running coordination number of b around a is ``np.cumsum(g[a, b] * shell) * n_ab / (|a| * V)``, with
        shell the shell volumes above.  A device-resident trajectory is read in place; a host trajectory is copied to
        the device once (its S·N·24 bytes must fit there).  Argument errors are raised before any device work.
        """
        radii, rdf = self.get_rdf_device(lattice, r_max, num_bins, atom_groups)
        return radii.cpu().numpy(), rdf.cpu().numpy()

    def get_van_hove_device(self, lattice, lags, r_max, num_bins, atom_groups=None):
        """``get_van_hove`` with the result left on the GPU (four CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice, lags, r_max, offsets, atoms = _check_van_hove_args(lattice, lags, r_max, num_bins, atom_groups,
                                                                    num_atoms, num_frames)
        import torch  # pylint: disable=import-outside-toplevel

        lib = _lib.lib()
        positions, device = self._device_positions()
        num_groups, num_lags, num_bins = len(offsets) - 1, len(lags), int(num_bins)
        lag_times = np.asarray(lags, dtype=np.float64) * self._timestep
        radii = (np.arange(num_bins) + 0.5) * (r_max / num_bins)
        with torch.cuda.device(device):
            van_hove = torch.empty((num_groups, num_lags, num_bins), dtype=torch.float64, device=positions.device)
            moments = torch.empty((num_groups, num_lags, 2), dtype=torch.float64, device=positions.device)
            ws_bytes = int(lib.rn_van_hove_workspace_size(num_frames, len(atoms), num_groups, num_lags, num_bins))
            workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=positions.device)
            status = lib.rn_van_hove(ctypes.c_void_p(positions.data_ptr()), num_frames, num_atoms,
                                     ctypes.c_void_p(lattice.ctypes.data), ctypes.c_void_p(lags.ctypes.data), num_lags,
                                     r_max, num_bins, ctypes.c_void_p(offsets.ctypes.data),
                                     ctypes.c_void_p(atoms.ctypes.data), num_groups,
                                     ctypes.c_void_p(van_hove.data_ptr()), ctypes.c_void_p(moments.data_ptr()),
                                     ctypes.c_void_p(workspace.data_ptr()), _lib.current_stream(device))
            _lib.check(status, "rn_van_hove")
            return (torch.from_numpy(lag_times).to(positions.device), torch.from_numpy(radii).to(positions.device),
                    van_hove, moments)

    def get_van_hove(self, lattice, lags, r_max, num_bins, atom_groups=None):
        """Self part of the Van Hove correlation of atom groups -> (lag_times, r, g_s, moments), numpy arrays of shape
        (T,), (B,), (G, T, B) and (G, T, 2).

        ``lattice`` is the (3,3) cell in Å with lattice vectors as rows; ``atom_groups`` are those of ``get_vdos``: G
        non-empty sequences of atom indices in [0, N) without repeats inside a group (groups may overlap), by default
        one group of all atoms.  ``lags`` are T >= 1 strictly increasing integer frame lags in [0, S);
        ``lag_times = lags * timestep`` in fs.  ``r_max`` in Å is finite and > 0 (the paths are unwrapped, so it is not
        bounded by the cell) and ``num_bins`` B an integer in 1..4096; ``r`` are the bin centres of ``get_rdf``.

        The path of atom i is unwrapped as in ``get_msd``: with the minimum-image steps of ``get_vdos``, their integer
        image shifts and ``K(n)`` their running sum, ``r_i(n) = (x_i(n) - x_i(0) - K_i(n)) @ lattice``.  For lag t,
        every membership i of group g and every origin n < S - t, the displacement ``|r_i(n+t) - r_i(n)|`` counts into
        bin k = floor(|.| * B / r_max) when k < B, and ``g_s[g, t, k] = count / ((S - t) |g| shell_k)`` in Å^-3 with the
        shell volumes of ``get_rdf``: ``sum_k g_s * shell`` is the fraction of displacements shorter than r_max and
        ``4 pi r^2 g_s`` the radial density.  Lag 0 puts every count in bin 0.  The moments run over all displacements:
        ``moments[g, t] = (<rr>, <rr^2>)``, the means of ``|.|^2`` and ``|.|^4`` over the (S - t) |g| displacements;
        ``moments[..., 0]`` is the MSD of ``get_msd`` at those lags up to rounding.  The non-Gaussian parameter is
        ``alpha2 = 3 * moments[..., 1] / (5 * moments[..., 0] ** 2) - 1``: 0 for Gaussian diffusion and harmonic
        rattling, positive for hopping.

        The displacements are evaluated in FP64 with every product and sum rounded on its own, so the counts are exact
        integers; the moments are summed in an order fixed by S, the lags and the group sizes, so every result is the
        same bit for bit for host and device trajectories, repeated calls and a group computed alone or with others.
        A device-resident trajectory is read in place; a host trajectory is copied to the device once (its S·N·24
        bytes must fit there).  Argument errors are raised before any device work.
        """
        lag_times, radii, van_hove, moments = self.get_van_hove_device(lattice, lags, r_max, num_bins, atom_groups)
        return lag_times.cpu().numpy(), radii.cpu().numpy(), van_hove.cpu().numpy(), moments.cpu().numpy()

    def get_distinct_van_hove_device(self, lattice, lags, r_max, num_bins, atom_groups=None):
        """``get_distinct_van_hove`` with the result left on the GPU (three CUDA tensors)."""
        num_frames, num_atoms = int(self._positions_ts.shape[0]), int(self._positions_ts.shape[1])
        lattice, lags, r_max, offsets, atoms = _check_distinct_van_hove_args(lattice, lags, r_max, num_bins,
                                                                             atom_groups, num_atoms, num_frames)
        import torch  # pylint: disable=import-outside-toplevel

        lib = _lib.lib()
        positions, device = self._device_positions()
        num_groups, num_lags, num_bins = len(offsets) - 1, len(lags), int(num_bins)
        lag_times = np.asarray(lags, dtype=np.float64) * self._timestep
        radii = (np.arange(num_bins) + 0.5) * (r_max / num_bins)
        with torch.cuda.device(device):
            g_d = torch.empty((num_groups, num_groups, num_lags, num_bins), dtype=torch.float64,
                              device=positions.device)
            ws_bytes = int(lib.rn_distinct_van_hove_workspace_size(len(atoms), num_groups, num_lags, num_bins))
            workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=positions.device)
            status = lib.rn_distinct_van_hove(ctypes.c_void_p(positions.data_ptr()), num_frames, num_atoms,
                                              ctypes.c_void_p(lattice.ctypes.data), ctypes.c_void_p(lags.ctypes.data),
                                              num_lags, r_max, num_bins, ctypes.c_void_p(offsets.ctypes.data),
                                              ctypes.c_void_p(atoms.ctypes.data), num_groups,
                                              ctypes.c_void_p(g_d.data_ptr()), ctypes.c_void_p(workspace.data_ptr()),
                                              _lib.current_stream(device))
            _lib.check(status, "rn_distinct_van_hove")
            return torch.from_numpy(lag_times).to(positions.device), torch.from_numpy(radii).to(positions.device), g_d

    def get_distinct_van_hove(self, lattice, lags, r_max, num_bins, atom_groups=None):
        """Distinct part of the Van Hove correlation of atom groups -> (lag_times, r, g_d), numpy arrays of shape (T,),
        (B,) and (G, G, T, B).

        ``lattice``, ``r_max``, ``num_bins`` and ``atom_groups`` are those of ``get_rdf`` (``0 < r_max <= w_min / 2``,
        B in 1..4096, groups may overlap); ``r`` are its bin centres.  ``lags`` are T >= 1 strictly increasing integer
        frame lags in [0, S) and ``lag_times = lags * timestep`` in fs, as in ``get_van_hove``.

        For every ordered group pair (a, b), lag t, origin n < S - t and pair i in a, j in b with i != j, the
        minimum-image vector ``v = (d - ceil(d - 0.5)) @ lattice`` of ``d = x_j(n + t) - x_i(n)`` counts into bin
        k = floor(|v| * B / r_max) when k < B, and ``g_d[a, b, t, k] = count * V / ((S - t) * n_ab * shell_k)`` with the
        V, n_ab and shell_k of ``get_rdf``; a pair of groups with n_ab = 0 gets a zero row.  It is the probability of
        finding a b atom at distance r at time n + t from where an a atom was at time n, relative to an ideal gas.  The
        result is not mirrored: ``g_d[a, b, t]`` and ``g_d[b, a, t]`` are different sums for t > 0 (the first is the
        second of the time-reversed trajectory).

        At lag 0 it is the RDF: ``g_d[:, :, lags == 0]`` equals ``get_rdf(lattice, r_max, num_bins, atom_groups)[1]``
        bit for bit (unless a coordinate difference sits exactly on a ±1/2 wrap tie with r_max exactly at w_min / 2).
        At long lags it tends to 1 for an uncorrelated or diffusing species, and to the time-averaged site structure
        (the RDF of the average positions, broadened by the vibrations) for a crystal.  A peak of ``g_d[a, a, t]`` at
        r -> 0 that grows with t means that other atoms of a move into the sites a atoms left: site refilling and
        concerted hopping, as of Li in a superionic conductor; the decay of the shells towards 1 shows the cage
        relaxing.  For one species a, the total Van Hove function in Å^-3 is
        ``G(r, t) = g_s[a, t] + (|a| - 1) / V * g_d[a, a, t]`` with the ``g_s`` of ``get_van_hove`` on the same lags,
        r_max and bins.

        The distances are evaluated in FP64 with every product and sum rounded on its own, so the counts are exact
        integers, the same for every launch configuration, host and device trajectories, repeated calls and a group
        pair computed alone or with others.  A device-resident trajectory is read in place; a host trajectory is copied
        to the device once (its S·N·24 bytes must fit there).  Argument errors are raised before any device work.
        """
        lag_times, radii, g_d = self.get_distinct_van_hove_device(lattice, lags, r_max, num_bins, atom_groups)
        return lag_times.cpu().numpy(), radii.cpu().numpy(), g_d.cpu().numpy()

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

    def get_mode_vectors(self, lattice, atom_masses) -> np.ndarray:
        """Projection vectors of the normal modes for ``Trajectory.get_projected_vdos`` -> (M, N, 3) numpy array.

        ``lattice`` (3,3) in Å, lattice vectors as rows; ``atom_masses`` (N,) finite and > 0 (e.g. in amu).
        The stored displacements are eigenvectors divided by sqrt(m) in fractional coordinates, so the
        eigenvector of mode k is ``e_k = normalize(sqrt(m_i) * (displacements[k, i] @ lattice))`` over all 3N
        coordinates; the result is ``sqrt(m_i) * e_{k,i}``.  With these vectors row k of ``get_projected_vdos``
        is the power spectrum of the normal-mode velocity ``q_k = sum_i sqrt(m_i) e_{k,i} . v_i`` in
        amu (Å/fs)^2 for masses in amu.  The eigenvectors are not orthogonalised (degenerate pairs would mix
        arbitrarily); when they are orthonormal and complete, the rows add up to the mass-weighted
        ``get_vdos(lattice, atom_weights=atom_masses)``.  Raises ValueError for a mode of zero norm.
        """
        lattice = _check_lattice(lattice)
        num_atoms = self._ref_positions.shape[0]
        verify_ndarray_shape("atom_masses", atom_masses, (num_atoms,))
        masses = np.asarray(_host_array(atom_masses), dtype=np.float64)
        if not np.all(np.isfinite(masses)) or np.any(masses <= 0):
            raise ValueError("atom_masses must be finite and > 0")
        sqrt_m = np.sqrt(masses)[None, :, None]
        eigenvectors = sqrt_m * (np.asarray(self._displacements, dtype=np.float64) @ lattice)
        norms = np.sqrt(np.sum(eigenvectors * eigenvectors, axis=(1, 2)))
        zero = np.flatnonzero(norms == 0)
        if zero.size:
            raise ValueError(f"mode {zero[0]} has zero norm")
        return sqrt_m * (eigenvectors / norms[:, None, None])

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

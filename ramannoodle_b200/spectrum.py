"""MD Raman spectrum and smearing — drop-ins for ``ramannoodle.spectrum``.

``MDRamanSpectrum.measure`` (``ramannoodle/spectrum/_raman.py:241-309``),
``calc_signal_spectrum`` (``ramannoodle/spectrum/utils.py:95-124``) and
``convolve_spectrum`` (``ramannoodle/spectrum/utils.py:12-73``) keep their signatures, return
types and error messages; the arithmetic runs in the CUDA library.
"""
from __future__ import annotations

import ctypes
import threading
from collections import OrderedDict
from collections.abc import Sequence

import numpy as np

from . import _lib
from .abstract import RamanSpectrum
from .exceptions import get_type_error, shape_string, verify_ndarray, verify_ndarray_shape

BOLTZMANN_CONSTANT = 8.617333262e-5  # eV/K (ramannoodle/constants.py:249)


def _torch():
    import torch  # pylint: disable=import-outside-toplevel

    return torch


def _current_device() -> int:
    torch = _torch()
    if not torch.cuda.is_available():
        _lib.require_device(0)  # raises NativeLibraryError with the reason
    return int(torch.cuda.current_device())


class _Plan:
    """``rn_spectrum_plan`` for one series length on one device (``batch`` windows of that length)."""

    def __init__(self, num_frames: int, device: int, batch: int = 1) -> None:
        handle = ctypes.c_void_p()
        if batch == 1:
            _lib.check(_lib.lib().rn_spectrum_plan_create(num_frames, device, ctypes.byref(handle)),
                       "rn_spectrum_plan_create")
        else:
            _lib.check(_lib.lib().rn_spectrum_plan_create_batched(num_frames, batch, device, ctypes.byref(handle)),
                       "rn_spectrum_plan_create_batched")
        self.handle = handle

    def close(self) -> None:
        if getattr(self, "handle", None):
            _lib.lib().rn_spectrum_plan_destroy(self.handle)
            self.handle = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass


_PLAN_CACHE: "OrderedDict[tuple, _Plan]" = OrderedDict()
_PLAN_CACHE_SIZE = 4
_PLAN_CACHE_LOCK = threading.Lock()


def _get_plan(num_frames: int, device: int, batch: int = 1) -> _Plan:
    """A plan owns its work buffers, so it is shared only by calls that are ordered anyway: the same
    Python thread AND the same CUDA stream (two streams or two threads measuring series of the same length
    would otherwise race on the buffers)."""
    stream_id = 0
    try:
        import torch  # pylint: disable=import-outside-toplevel

        if torch.cuda.is_available():
            stream_id = int(torch.cuda.current_stream(device).cuda_stream)
    except (ImportError, RuntimeError):
        stream_id = 0
    key = (int(num_frames), int(device), stream_id, threading.get_ident(), int(batch))
    with _PLAN_CACHE_LOCK:
        return _get_plan_locked(key, num_frames, device, batch)


def _get_plan_locked(key, num_frames: int, device: int, batch: int = 1) -> _Plan:
    plan = _PLAN_CACHE.get(key)
    if plan is None:
        _lib.require_device(device)
        while len(_PLAN_CACHE) >= _PLAN_CACHE_SIZE:
            _, old = _PLAN_CACHE.popitem(last=False)
            old.close()
        # a plan of one window is built with the two-argument form the single-series callers have always used
        plan = _Plan(num_frames, device) if batch == 1 else _Plan(num_frames, device, batch)
        _PLAN_CACHE[key] = plan
    else:
        _PLAN_CACHE.move_to_end(key)
    return plan


def clear_plan_cache() -> None:
    with _PLAN_CACHE_LOCK:
        while _PLAN_CACHE:
            _, plan = _PLAN_CACHE.popitem()
            plan.close()


def get_bose_einstein_correction(wavenumbers, temperature):
    """``ramannoodle/spectrum/_raman.py:13-40`` (elementwise; evaluated on the host when
    called directly — inside ``measure`` the correction is fused into the GPU kernel)."""
    try:
        if temperature <= 0:
            raise ValueError(f"invalid temperature: {temperature} <= 0")
    except TypeError as exc:
        raise get_type_error("temperature", temperature, "float") from exc
    try:
        energy = wavenumbers * 29979245800.0 * 4.1357e-15  # in eV
        return 1 / (1 - np.exp(-energy / (BOLTZMANN_CONSTANT * temperature)))
    except TypeError as exc:
        raise get_type_error("wavenumbers", wavenumbers, "ndarray") from exc


def get_laser_correction(wavenumbers, laser_wavenumber):
    """``ramannoodle/spectrum/_raman.py:43-69``."""
    try:
        if laser_wavenumber <= 0:
            raise ValueError(f"invalid laser_wavenumber: {laser_wavenumber} <= 0")
    except TypeError as exc:
        raise get_type_error("laser_wavenumber", laser_wavenumber, "float") from exc
    try:
        return ((wavenumbers - laser_wavenumber) / 10000) ** 4 / wavenumbers
    except TypeError as exc:
        raise get_type_error("wavenumbers", wavenumbers, "ndarray") from exc


class MDRamanSpectrum(RamanSpectrum):
    """Molecular-dynamics Raman spectrum (``ramannoodle/spectrum/_raman.py:197-309``).

    ``polarizability_ts`` is an array with shape (S,3,3) — numpy, or a CUDA tensor left on the
    device by ``Trajectory.get_raman_spectrum``.
    """

    def __init__(self, polarizability_ts, timestep: float):
        verify_ndarray_shape("polarizability_ts", polarizability_ts, (None, 3, 3))
        self._polarizability_ts = polarizability_ts
        self._timestep = timestep

    @property
    def polarizability_ts(self) -> np.ndarray:
        """The (S,3,3) series as numpy (copied from the GPU on first access if needed)."""
        if _lib.is_torch_tensor(self._polarizability_ts):
            return self._polarizability_ts.detach().cpu().numpy()
        return self._polarizability_ts

    @property
    def timestep(self) -> float:
        return self._timestep

    def _num_frames(self) -> int:
        return int(self._polarizability_ts.shape[0])

    def _device_series(self):
        torch = _torch()
        series = self._polarizability_ts
        if _lib.is_torch_tensor(series):
            if not series.is_cuda:
                series = series.to(f"cuda:{_current_device()}")
            return series.to(torch.float64).contiguous()
        device = _current_device()
        return torch.from_numpy(np.ascontiguousarray(series, dtype=np.float64)).to(f"cuda:{device}")

    # pylint: disable=too-many-arguments,too-many-positional-arguments
    def measure_device(self, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                       bose_einstein_correction=False, temperature=300):
        """``measure`` with the result left on the GPU (two CUDA tensors)."""
        _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction, temperature)
        torch = _torch()
        series = self._device_series()
        num_frames = int(series.shape[0])
        if num_frames < 2:
            raise ValueError("polarizability_ts must contain at least 2 configurations")
        device = int(series.device.index or 0)
        points = int(_lib.lib().rn_spectrum_num_points(num_frames))
        with torch.cuda.device(device):
            wavenumbers = torch.empty(points, dtype=torch.float64, device=series.device)
            intensities = torch.empty(points, dtype=torch.float64, device=series.device)
            if points > 0:
                plan = _get_plan(num_frames, device)
                status = _lib.lib().rn_md_spectrum(
                    plan.handle, ctypes.c_void_p(series.data_ptr()), float(self._timestep),
                    1 if laser_correction else 0, float(laser_wavelength) if laser_correction else 0.0,
                    1 if bose_einstein_correction else 0, float(temperature) if bose_einstein_correction else 0.0,
                    ctypes.c_void_p(wavenumbers.data_ptr()), ctypes.c_void_p(intensities.data_ptr()),
                    _lib.current_stream(device))
                _lib.check(status, "rn_md_spectrum")
        return wavenumbers, intensities

    def measure(self, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                bose_einstein_correction=False, temperature=300):
        """Raw polycrystalline Raman spectrum -> (wavenumbers, intensities), numpy arrays of
        shape (ceil((S-1)/2) - 1,)."""
        wavenumbers, intensities = self.measure_device(orientation, laser_correction, laser_wavelength,
                                                       bose_einstein_correction, temperature)
        return wavenumbers.cpu().numpy(), intensities.cpu().numpy()

    # pylint: disable=too-many-arguments,too-many-positional-arguments,too-many-locals
    def measure_windows_device(self, window_frames, hop_frames=None, orientation="polycrystalline",
                               laser_correction=False, laser_wavelength=522, bose_einstein_correction=False,
                               temperature=300):
        """``measure_windows`` with the result left on the GPU (two CUDA tensors)."""
        hop = _check_window_args(window_frames, hop_frames, int(self._polarizability_ts.shape[0]))
        _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction, temperature)
        return _measure_windows(self._device_series(), self._timestep, int(window_frames), hop, laser_correction,
                                laser_wavelength, bose_einstein_correction, temperature)

    def measure_windows(self, window_frames, hop_frames=None, orientation="polycrystalline", laser_correction=False,
                        laser_wavelength=522, bose_einstein_correction=False, temperature=300):
        """Spectra of windows of the series -> (wavenumbers, intensities), numpy arrays of shape (P,) and
        (W, P), P = ceil((window_frames-1)/2) - 1.

        Window w covers frames [w*hop, w*hop + window_frames) with hop = ``hop_frames`` (default
        ``window_frames``: contiguous blocks, for block averages); a smaller hop gives overlapping windows
        (a spectrogram), a larger one leaves gaps.  W = 1 + (S - window_frames) // hop: trailing frames that
        do not fill a window are not used.  Row w is by definition
        ``MDRamanSpectrum(polarizability_ts[w*hop : w*hop + window_frames], timestep).measure(...)[1]``
        with the same keyword arguments, and the wavenumbers are those of that call.  All windows run as
        one batched transform on the GPU.
        """
        wavenumbers, intensities = self.measure_windows_device(window_frames, hop_frames, orientation,
                                                               laser_correction, laser_wavelength,
                                                               bose_einstein_correction, temperature)
        return wavenumbers.cpu().numpy(), intensities.cpu().numpy()


def _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction,
                        temperature) -> None:
    """The argument errors of ``measure`` (``_raman.py:241-309``)."""
    if orientation != "polycrystalline":
        raise NotImplementedError("only polycrystalline spectra are supported for now")
    if laser_correction:
        laser_wavenumber = 10000000 / laser_wavelength
        try:
            if laser_wavenumber <= 0:
                raise ValueError(f"invalid laser_wavenumber: {laser_wavenumber} <= 0")
        except TypeError as exc:
            raise get_type_error("laser_wavenumber", laser_wavenumber, "float") from exc
    if bose_einstein_correction:
        try:
            if temperature <= 0:
                raise ValueError(f"invalid temperature: {temperature} <= 0")
        except TypeError as exc:
            raise get_type_error("temperature", temperature, "float") from exc


def _is_integer(value) -> bool:
    return isinstance(value, (int, np.integer)) and not isinstance(value, (bool, np.bool_))


def _check_window_args(window_frames, hop_frames, num_frames: int) -> int:
    """Validate the window of ``measure_windows`` on a series of ``num_frames`` frames; returns the hop."""
    if not _is_integer(window_frames):
        raise get_type_error("window_frames", window_frames, "int")
    if hop_frames is not None and not _is_integer(hop_frames):
        raise get_type_error("hop_frames", hop_frames, "int")
    if not 2 <= window_frames <= num_frames:
        raise ValueError(f"invalid window_frames: {window_frames} (a window needs 2 to {num_frames} frames)")
    hop = int(window_frames) if hop_frames is None else int(hop_frames)
    if hop < 1:
        raise ValueError(f"invalid hop_frames: {hop_frames} < 1")
    return hop


def num_windows(num_frames: int, window_frames: int, hop_frames: int) -> int:
    """W = 1 + (S - window_frames) // hop: the windows ``measure_windows`` returns."""
    return 1 + (int(num_frames) - int(window_frames)) // int(hop_frames)


# Device memory the batch buffers of one windowed plan may take: the windows run in chunks of as many
# as fit.  Larger chunks need fewer launches; the work of a window does not change.  A cached plan keeps its
# buffers after the call returns, so up to _PLAN_CACHE_SIZE windowed plans (4 GiB) can stay allocated; the
# batch is rounded up to a power of two so that calls with similar window counts share one plan.
_WINDOW_BATCH_BYTES = 1 << 30
_MAX_WINDOW_BATCH = 65535  # gridDim.y of the windowed pack and combine


def _window_batch(window_frames: int, windows: int) -> int:
    """Windows per chunk: the smallest power of two >= ``windows``, capped by the budget.  Per window the plan
    holds 3 work sequences of L complex values, 3 rows of M powers, the pack's energy partials and a ticket
    (``create_plan`` in ``csrc/rn_spectrum.cu``)."""
    m = window_frames - 1
    log2l = 12  # the plan pads L up to at least 4096
    while (1 << log2l) < max(2 * m - 1, 4096):
        log2l += 1
    pack_blocks = (m + 255) // 256
    per_window = 16 * 3 * (1 << log2l) + 8 * 3 * m + 8 * (pack_blocks + 1) + 4
    rounded = 1 << max(0, int(windows) - 1).bit_length()
    return max(1, min(rounded, _WINDOW_BATCH_BYTES // per_window, _MAX_WINDOW_BATCH))


# pylint: disable=too-many-arguments,too-many-positional-arguments
def _measure_windows(series, timestep, window_frames: int, hop: int, laser_correction, laser_wavelength,
                     bose_einstein_correction, temperature):
    """``rn_md_spectrum_windows`` on a contiguous float64 CUDA series (arguments already checked)."""
    torch = _torch()
    num_frames = int(series.shape[0])
    windows = num_windows(num_frames, window_frames, hop)
    device = int(series.device.index or 0)
    points = int(_lib.lib().rn_spectrum_num_points(window_frames))
    with torch.cuda.device(device):
        wavenumbers = torch.empty(points, dtype=torch.float64, device=series.device)
        intensities = torch.empty((windows, points), dtype=torch.float64, device=series.device)
        if points > 0:
            plan = _get_plan(window_frames, device, _window_batch(window_frames, windows))
            status = _lib.lib().rn_md_spectrum_windows(
                plan.handle, ctypes.c_void_p(series.data_ptr()), num_frames, hop, float(timestep),
                1 if laser_correction else 0, float(laser_wavelength) if laser_correction else 0.0,
                1 if bose_einstein_correction else 0, float(temperature) if bose_einstein_correction else 0.0,
                ctypes.c_void_p(wavenumbers.data_ptr()), ctypes.c_void_p(intensities.data_ptr()),
                _lib.current_stream(device))
            _lib.check(status, "rn_md_spectrum_windows")
    return wavenumbers, intensities


def _check_cross_spectra(spectra):
    """Validate the spectra of ``measure_cross_spectra``; returns (list, frames, timestep)."""
    if isinstance(spectra, (str, bytes)) or not isinstance(spectra, Sequence):
        raise get_type_error("spectra", spectra, "list")
    spectra = list(spectra)
    if not spectra:
        raise ValueError("spectra is empty")
    for item in spectra:
        if not isinstance(item, MDRamanSpectrum):
            raise get_type_error("spectra", item, "MDRamanSpectrum")
    frames = spectra[0]._num_frames()  # pylint: disable=protected-access
    timestep = spectra[0].timestep
    for g, item in enumerate(spectra):
        if item._num_frames() != frames:  # pylint: disable=protected-access
            raise ValueError(f"spectra[{g}] has {item._num_frames()} frames, spectra[0] has {frames}")  # pylint: disable=protected-access
        if item.timestep != timestep:
            raise ValueError(f"spectra[{g}] has timestep {item.timestep}, spectra[0] has {timestep}")
    if frames < 2:
        raise ValueError("polarizability_ts must contain at least 2 configurations")
    return spectra, frames, timestep


def _consecutive(series) -> bool:
    """Whether the series are consecutive slices of one contiguous float64 CUDA array (one (G,S,3,3) block)."""
    first = series[0]
    step = first.numel() * first.element_size()
    torch = _torch()
    return all(t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.device == first.device
               and t.data_ptr() == first.data_ptr() + g * step for g, t in enumerate(series))


# pylint: disable=too-many-arguments,too-many-positional-arguments,too-many-locals
def measure_cross_spectra_device(spectra, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                                 bose_einstein_correction=False, temperature=300):
    """``measure_cross_spectra`` with the result left on the GPU (two CUDA tensors)."""
    spectra, frames, timestep = _check_cross_spectra(spectra)
    _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction, temperature)
    torch = _torch()
    series = [item._device_series() for item in spectra]  # pylint: disable=protected-access
    if not _consecutive(series):  # e.g. separate arrays: one (G,S,3,3) copy on the current device
        device = _current_device()
        series = list(torch.stack([t.to(f"cuda:{device}") for t in series]))
    num_series = len(series)
    device = int(series[0].device.index or 0)
    points = int(_lib.lib().rn_spectrum_num_points(frames))
    with torch.cuda.device(device):
        wavenumbers = torch.empty(points, dtype=torch.float64, device=series[0].device)
        intensities = torch.empty((num_series, num_series, points), dtype=torch.float64, device=series[0].device)
        if points > 0:
            plan = _get_plan(frames, device, num_series)
            status = _lib.lib().rn_md_cross_spectra(
                plan.handle, ctypes.c_void_p(series[0].data_ptr()), num_series, float(timestep),
                1 if laser_correction else 0, float(laser_wavelength) if laser_correction else 0.0,
                1 if bose_einstein_correction else 0, float(temperature) if bose_einstein_correction else 0.0,
                ctypes.c_void_p(wavenumbers.data_ptr()), ctypes.c_void_p(intensities.data_ptr()),
                _lib.current_stream(device))
            _lib.check(status, "rn_md_cross_spectra")
    return wavenumbers, intensities


def measure_cross_spectra(spectra, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                          bose_einstein_correction=False, temperature=300):
    """Cross spectra of G MD Raman spectra -> (wavenumbers, intensities), numpy arrays of shape (P,) and (G,G,P).

    ``spectra`` is a non-empty sequence of ``MDRamanSpectrum`` with the same frame count S >= 2 and the same
    timestep, typically the list ``Trajectory.get_raman_spectra(models)`` returns for masked copies of one
    model.  ``I[g,h]`` is ``spectra[g].measure(...)`` with the spectrum of every signal replaced by that of the
    symmetrised cross-correlation ``(correlate(sig_g, sig_h) + correlate(sig_h, sig_g)) / 2`` of the same
    signal of series g and series h: the same signals, weights, dropped 0 cm^-1 bin and corrections.  So
    ``I[g,h] == I[h,g]``, ``I[g,g]`` is ``spectra[g].measure(...)[1]`` bit for bit, and ``I`` is bilinear in the
    series.  Cross terms can be negative, and as large as ``sqrt(I[g,g] * I[h,h])``.

    Sum rule: when the masks partition the DOFs (copy g keeps only group g), the differences of the G series
    add up to those of the unmasked model, so ``I.sum(axis=(0, 1))`` is the total spectrum, and
    ``I_g = I[g].sum(axis=0)`` attributes it additively to the groups (``sum_g I_g`` is the total).

    All G spectra run as one batched transform on the GPU.  With ``ShardedMDRamanSpectrum`` inputs of a shared
    transform context every series is first assembled on every rank (an all-gather, a collective): every rank
    of the group must call this function with the same list in the same order; every rank returns the full
    result.
    """
    wavenumbers, intensities = measure_cross_spectra_device(spectra, orientation, laser_correction, laser_wavelength,
                                                            bose_einstein_correction, temperature)
    return wavenumbers.cpu().numpy(), intensities.cpu().numpy()


class PhononRamanSpectrum(RamanSpectrum):
    """Phonon-based first-order Raman spectrum (``ramannoodle/spectrum/_raman.py:72-194``).

    ``measure`` is O(M) elementwise work on M = 3N Raman tensors (a few hundred numbers), so it
    stays on the host with the reference's exact formulas; the data-parallel part of the phonon
    path — the 2·M central-difference polarizabilities — is batched onto the GPU by
    ``ramannoodle_b200.dynamics.Phonons.get_raman_spectrum`` (SURVEY.md §8f row N1)."""

    def __init__(self, phonon_wavenumbers, raman_tensors) -> None:
        verify_ndarray_shape("phonon_wavenumbers", phonon_wavenumbers, (None,))
        verify_ndarray_shape("raman_tensors", raman_tensors, (len(phonon_wavenumbers), 3, 3))
        self._phonon_wavenumbers = phonon_wavenumbers
        self._raman_tensors = raman_tensors

    @property
    def phonon_wavenumbers(self) -> np.ndarray:
        return self._phonon_wavenumbers.copy()

    @property
    def raman_tensors(self) -> np.ndarray:
        return self._raman_tensors.copy()

    # pylint: disable=too-many-arguments,too-many-positional-arguments
    def measure(self, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                bose_einstein_correction=False, temperature=300):
        if orientation != "polycrystalline":
            raise NotImplementedError("only polycrystalline spectra are supported for now")
        tensors = self._raman_tensors
        alpha_squared = ((tensors[:, 0, 0] + tensors[:, 1, 1] + tensors[:, 2, 2]) / 3.0) ** 2
        gamma_squared = (
            (tensors[:, 0, 0] - tensors[:, 1, 1]) ** 2
            + (tensors[:, 0, 0] - tensors[:, 2, 2]) ** 2
            + (tensors[:, 1, 1] - tensors[:, 2, 2]) ** 2
            + 6.0 * (tensors[:, 0, 1] ** 2 + tensors[:, 0, 2] ** 2 + tensors[:, 1, 2] ** 2)
        ) / 2.0
        intensities = 45.0 * alpha_squared + 7.0 * gamma_squared
        if laser_correction:
            laser_wavenumber = 10000000 / laser_wavelength
            intensities *= get_laser_correction(self._phonon_wavenumbers, laser_wavenumber)
        if bose_einstein_correction:
            intensities *= get_bose_einstein_correction(self._phonon_wavenumbers, temperature)
        return self._phonon_wavenumbers, intensities


def calc_signal_spectrum(signal, sampling_rate: float):
    """Spectrum of one real signal (``ramannoodle/spectrum/utils.py:95-124``): the
    positive-frequency Fourier transform of its autocorrelation; ceil(S/2) points."""
    verify_ndarray_shape("signal", signal, (None,))
    torch = _torch()
    device = _current_device()
    data = torch.from_numpy(np.ascontiguousarray(signal, dtype=np.float64)).to(f"cuda:{device}")
    length = int(data.shape[0])
    if length < 1:
        raise ValueError("signal is empty")
    points = (length + 1) // 2
    with torch.cuda.device(device):
        wavenumbers = torch.empty(points, dtype=torch.float64, device=data.device)
        intensities = torch.empty(points, dtype=torch.float64, device=data.device)
        plan = _get_plan(length + 1, device)
        status = _lib.lib().rn_signal_spectrum(plan.handle, ctypes.c_void_p(data.data_ptr()), float(sampling_rate),
                                               ctypes.c_void_p(wavenumbers.data_ptr()),
                                               ctypes.c_void_p(intensities.data_ptr()), _lib.current_stream(device))
        _lib.check(status, "rn_signal_spectrum")
    return wavenumbers.cpu().numpy(), intensities.cpu().numpy()


def _smearing_args(wavenumbers, function, width, out_wavenumbers, check_inputs):
    """The default output grid and the argument checks of ``convolve_spectrum`` (``utils.py:12-56``), in its
    order; ``check_inputs()`` checks wavenumbers and intensities between the grid and the width.  Returns
    (out_wavenumbers, kind).  The grid of CUDA wavenumbers is taken from their min/max on the device."""
    if out_wavenumbers is None:
        if _lib.is_torch_tensor(wavenumbers) and wavenumbers.is_cuda and wavenumbers.numel() > 0:
            # the default grid needs two numbers, not a copy of the spectrum
            low, high = (float(v) for v in _torch().aminmax(wavenumbers))
        else:
            wn_host = wavenumbers.detach().cpu().numpy() if _lib.is_torch_tensor(wavenumbers) else wavenumbers
            low, high = np.min(wn_host), np.max(wn_host)
        min_wavenumber = low - 100
        max_wavenumber = high + 100
        num_samples = int(np.rint(max_wavenumber - min_wavenumber))
        out_wavenumbers = np.linspace(min_wavenumber, max_wavenumber, num_samples)
    verify_ndarray_shape("out_wavenumbers", out_wavenumbers, (None,))
    check_inputs()
    try:
        if width <= 0:
            raise ValueError(f"invalid width: {width} <= 0")
    except TypeError as exc:
        raise get_type_error("width", width, "float") from exc
    verify_ndarray("out_wavenumbers", out_wavenumbers)
    if function not in ("gaussian", "lorentzian"):
        raise ValueError(f"unsupported convolution type: {function}")
    return out_wavenumbers, 0 if function == "gaussian" else 1


def _to_device(array, device: int):
    """A float64 contiguous copy of ``array`` on ``cuda:device``; such a tensor is returned as it is."""
    torch = _torch()
    if _lib.is_torch_tensor(array):
        return array.to(device=f"cuda:{device}", dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(array, dtype=np.float64)).to(f"cuda:{device}")


def _to_host(array):
    return array.detach().cpu().numpy() if _lib.is_torch_tensor(array) else array


def convolve_spectrum(wavenumbers, intensities, function: str = "gaussian", width: float = 5,
                      out_wavenumbers=None):
    """Smear a spectrum (``ramannoodle/spectrum/utils.py:12-73``); same defaults, output grid
    and error messages.  Accepts numpy arrays (or CUDA tensors) and returns numpy arrays."""
    torch = _torch()

    def check_inputs():
        verify_ndarray_shape("wavenumbers", wavenumbers, (None,))
        verify_ndarray_shape("intensities", intensities, (len(wavenumbers),))

    out_wavenumbers, kind = _smearing_args(wavenumbers, function, width, out_wavenumbers, check_inputs)

    device = _current_device()
    _lib.require_device(device)
    d_wn, d_in, d_out_wn = (_to_device(a, device) for a in (wavenumbers, intensities, out_wavenumbers))
    num_in, num_out = int(d_wn.shape[0]), int(d_out_wn.shape[0])
    with torch.cuda.device(device):
        d_out = torch.empty(num_out, dtype=torch.float64, device=d_wn.device)
        ws_bytes = int(_lib.lib().rn_convolve_workspace_size(num_in, num_out))
        workspace = torch.empty(max(ws_bytes // 8, 1), dtype=torch.float64, device=d_wn.device)
        status = _lib.lib().rn_convolve_spectrum(
            ctypes.c_void_p(d_wn.data_ptr()), ctypes.c_void_p(d_in.data_ptr()), num_in, kind, float(width),
            ctypes.c_void_p(d_out_wn.data_ptr()), num_out, ctypes.c_void_p(d_out.data_ptr()),
            ctypes.c_void_p(workspace.data_ptr()), _lib.current_stream(device))
        _lib.check(status, "rn_convolve_spectrum")
    return (_to_host(out_wavenumbers), d_out.cpu().numpy())


# Device memory the workspace of one convolve_spectra launch may take (chunks * rows * L partial sums): the rows
# run in consecutive blocks of as many as fit.  Every row does the same work whatever the block.
_SMEAR_BLOCK_BYTES = 1 << 30


def _smear_rows_per_block(num_rows: int, row_bytes: int) -> int:
    """Rows per launch of ``rn_convolve_spectra`` when each row takes ``row_bytes`` of workspace: all of them if
    they fit ``_SMEAR_BLOCK_BYTES``, else as many as fit, and at least one."""
    if row_bytes == 0:
        return max(1, num_rows)
    return max(1, min(num_rows, _SMEAR_BLOCK_BYTES // row_bytes))


def _smeared_layout(shape, num_out: int):
    """(rows, output shape) of ``convolve_spectra`` on intensities of ``shape`` (..., P)."""
    return int(np.prod(shape[:-1], dtype=np.int64)), tuple(shape[:-1]) + (int(num_out),)


def _convolve_rows(wavenumbers, intensities, function, width, out_wavenumbers):
    """``convolve_spectra``: (out_wavenumbers as given or built, the same on the device, (..., Q) CUDA tensor)."""
    torch = _torch()

    def check_inputs():
        verify_ndarray_shape("wavenumbers", wavenumbers, (None,))
        verify_ndarray("intensities", intensities)
        if len(intensities.shape) == 0 or intensities.shape[-1] != len(wavenumbers):
            raise ValueError(f"intensities has shape {shape_string(intensities.shape)}, wavenumbers has shape "
                             f"{shape_string(wavenumbers.shape)}: the last axis of intensities must be as long as "
                             "wavenumbers")

    out_wavenumbers, kind = _smearing_args(wavenumbers, function, width, out_wavenumbers, check_inputs)

    device = _current_device()
    _lib.require_device(device)
    d_wn, d_in, d_out_wn = (_to_device(a, device) for a in (wavenumbers, intensities, out_wavenumbers))
    num_in, num_out = int(d_wn.shape[0]), int(d_out_wn.shape[0])
    num_rows, out_shape = _smeared_layout(tuple(d_in.shape), num_out)
    rows_per_block = _smear_rows_per_block(num_rows, int(_lib.lib().rn_convolve_spectra_workspace_size(1, num_in,
                                                                                                       num_out)))
    with torch.cuda.device(device):
        d_out = torch.empty(out_shape, dtype=torch.float64, device=d_wn.device)
        ws_bytes = int(_lib.lib().rn_convolve_spectra_workspace_size(min(rows_per_block, num_rows), num_in, num_out))
        workspace = torch.empty(max(ws_bytes // 8, 1), dtype=torch.float64, device=d_wn.device)
        for first in range(0, num_rows, rows_per_block):
            rows = min(rows_per_block, num_rows - first)
            status = _lib.lib().rn_convolve_spectra(
                ctypes.c_void_p(d_wn.data_ptr()), ctypes.c_void_p(d_in.data_ptr() + 8 * first * num_in), rows,
                num_in, kind, float(width), ctypes.c_void_p(d_out_wn.data_ptr()), num_out,
                ctypes.c_void_p(d_out.data_ptr() + 8 * first * num_out), ctypes.c_void_p(workspace.data_ptr()),
                _lib.current_stream(device))
            _lib.check(status, "rn_convolve_spectra")
    return out_wavenumbers, d_out_wn, d_out


def convolve_spectra_device(wavenumbers, intensities, function: str = "gaussian", width: float = 5,
                            out_wavenumbers=None):
    """``convolve_spectra`` with the result left on the GPU: (out_wavenumbers (Q,), intensities (..., Q)),
    two CUDA tensors."""
    _, d_out_wn, d_out = _convolve_rows(wavenumbers, intensities, function, width, out_wavenumbers)
    return d_out_wn, d_out


def convolve_spectra(wavenumbers, intensities, function: str = "gaussian", width: float = 5,
                     out_wavenumbers=None):
    """Smear every row of a stack of spectra that share ``wavenumbers`` -> (out_wavenumbers (Q,),
    intensities (..., Q)), numpy arrays.

    ``intensities`` has shape (..., P) with P = len(wavenumbers): the (W, P) rows of ``measure_windows``, the
    (G, G, P) cross spectra of ``measure_cross_spectra``, or one (P,) spectrum; numpy, a CPU tensor or a CUDA
    tensor (contiguous float64 CUDA input is read in place).  Row ``idx`` of the result is by definition
    ``convolve_spectrum(wavenumbers, intensities[idx], function, width, out_wavenumbers)[1]``, bit for bit, and
    the default output grid is the one that call builds.  All rows run in two launches on the GPU, which
    evaluate each smearing factor once for a group of rows; the rows are split into consecutive blocks when
    the partial sums of all of them would take more than 1 GiB.  Argument errors are those of
    ``convolve_spectrum`` (a wrong last axis or a 0-d ``intensities`` names both shapes) and are raised before
    any output is allocated or kernel launched; only the default grid of CUDA wavenumbers reads their min and
    max on the device first, as ``convolve_spectrum`` does.
    """
    out_wavenumbers, _, d_out = _convolve_rows(wavenumbers, intensities, function, width, out_wavenumbers)
    return _to_host(out_wavenumbers), d_out.cpu().numpy()

"""Windowed MD Raman spectra (``MDRamanSpectrum.measure_windows``): every row against ``measure`` of its
slice on the GPU (bit for bit: each window runs the same arithmetic in the same order) and a subset
against the oracle (pointwise relative error <= 1e-8)."""
import ctypes

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib, synthetic

from gpu_helpers import INTENSITY_RTOL, to_cuda
from helpers import GOLDEN, pointwise_rel_err, state_from_tables

pytestmark = pytest.mark.gpu


def _series(frames, seed):
    rng = np.random.default_rng(seed)
    steps = np.arange(frames)[:, None, None]
    return (6.0 * np.eye(3)[None] + 0.05 * np.sin(0.013 * steps + rng.uniform(0, 6, (1, 3, 3)))
            + 0.01 * rng.normal(size=(frames, 3, 3)))


def _host(series):
    return series.detach().cpu().numpy() if isinstance(series, torch.Tensor) else series


# pylint: disable=too-many-arguments,too-many-positional-arguments
def _check(series, window, hop, timestep=1.0, oracle_rows=(0,), rows=None, **kwargs):
    """measure_windows against measure() of every slice (or of `rows`) and the oracle on `oracle_rows`."""
    host = _host(series)
    wn, inten = rb.MDRamanSpectrum(series, timestep).measure_windows(window, hop, **kwargs)
    step = window if hop is None else hop
    windows = 1 + (len(host) - window) // step
    points = int(_lib.lib().rn_spectrum_num_points(window))
    assert wn.shape == (points,) and inten.shape == (windows, points)
    for w in range(windows) if rows is None else rows:
        piece = host[w * step: w * step + window]
        want_wn, want = rb.MDRamanSpectrum(piece, timestep).measure(**kwargs)
        assert np.array_equal(wn, want_wn)
        assert np.array_equal(inten[w], want), f"window {w}"
    for w in oracle_rows:
        piece = host[w * step: w * step + window]
        ref_wn, ref = ora.md_measure(piece, timestep, **kwargs)
        assert np.array_equal(wn, ref_wn)
        assert pointwise_rel_err(inten[w], ref) <= INTENSITY_RTOL
    return wn, inten


@pytest.mark.parametrize("window", [100, 2049, 2050, 40_001])
def test_window_lengths_around_plan_shapes(window):
    """No strided level (L = 4096 up to 2049 frames), the first one-level length and a mid one-level size."""
    frames = 3 * window + 7
    _check(_series(frames, window), window, None, oracle_rows=(0, 2))
    _check(_series(frames, window + 1), window, window // 2 + 1, oracle_rows=(1,))


@pytest.mark.parametrize("hop", [1000, 400, 1500, 333])
def test_hop_equal_below_above_and_odd(hop):
    _check(_series(6001, hop), 1000, hop, oracle_rows=(0, 1))


def test_hop_one_many_windows():
    wn, inten = _check(_series(700, 11), 101, 1, oracle_rows=(0, 37, 599))
    assert inten.shape == (600, 49) and wn.shape == (49,)


def test_single_window_is_measure():
    alpha = _series(4097, 12)
    want_wn, want = rb.MDRamanSpectrum(alpha, 1.5).measure()
    wn, inten = rb.MDRamanSpectrum(alpha, 1.5).measure_windows(4097)
    assert np.array_equal(wn, want_wn) and np.array_equal(inten[0], want) and inten.shape == (1, len(want))


@pytest.mark.parametrize("corrections", [False, True])
def test_corrections_and_timestep(corrections):
    kwargs = dict(laser_correction=corrections, laser_wavelength=532, bose_einstein_correction=corrections,
                  temperature=250)
    _check(_series(5000, 13), 1200, 700, timestep=2.5, oracle_rows=(0, 5), **kwargs)


@pytest.mark.parametrize("kind", ["numpy", "cpu", "cuda"])
def test_series_types(kind):
    alpha = _series(3001, 14)
    series = {"numpy": alpha, "cpu": torch.from_numpy(alpha), "cuda": to_cuda(alpha)}[kind]
    _check(series, 500, 251, oracle_rows=(3,))


def test_two_level_window():
    """A window of 2^21 + 2 frames (chirp-z length 2^23, two strided levels), against measure() only."""
    window = (1 << 21) + 2
    alpha = to_cuda(_series(window + 7, 15))
    _check(alpha, window, 7, oracle_rows=())


def test_tiny_windows_have_no_points():
    alpha = _series(10, 16)
    for window in (2, 3):
        wn, inten = rb.MDRamanSpectrum(alpha, 1.0).measure_windows(window)
        assert wn.shape == (0,) and inten.shape == (10 // window, 0)
    wn, inten = rb.MDRamanSpectrum(alpha, 1.0).measure_windows(4, 3)
    assert wn.shape == (1,) and inten.shape == (3, 1)


def test_chunked_batches_through_cabi():
    """A plan of 3 windows runs W = 10 windows in four chunks; rn_md_spectrum also runs on that plan."""
    window, hop = 900, 301
    alpha = _series(window + 9 * hop + 5, 17)
    want_wn, want = rb.MDRamanSpectrum(alpha, 1.0).measure_windows(window, hop)
    lib = _lib.lib()
    handle = ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(window, 3, 0, ctypes.byref(handle)), "create_batched")
    try:
        series = to_cuda(alpha)
        points = len(want_wn)
        wn = torch.empty(points, dtype=torch.float64, device="cuda:0")
        inten = torch.full((10, points), float("nan"), dtype=torch.float64, device="cuda:0")
        stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
        _lib.check(lib.rn_md_spectrum_windows(handle, ctypes.c_void_p(series.data_ptr()), len(alpha), hop, 1.0, 0,
                                              0.0, 0, 0.0, ctypes.c_void_p(wn.data_ptr()),
                                              ctypes.c_void_p(inten.data_ptr()), stream), "windows")
        assert np.array_equal(wn.cpu().numpy(), want_wn) and np.array_equal(inten.cpu().numpy(), want)
        one_wn = torch.empty_like(wn)
        one = torch.empty_like(wn)
        piece = to_cuda(alpha[2 * hop: 2 * hop + window])
        _lib.check(lib.rn_md_spectrum(handle, ctypes.c_void_p(piece.data_ptr()), 1.0, 0, 0.0, 0, 0.0,
                                      ctypes.c_void_p(one_wn.data_ptr()), ctypes.c_void_p(one.data_ptr()), stream),
                   "rn_md_spectrum")
        assert np.array_equal(one.cpu().numpy(), want[2])
        assert lib.rn_md_spectrum_windows(handle, ctypes.c_void_p(series.data_ptr()), window - 1, hop, 1.0, 0, 0.0,
                                          0, 0.0, ctypes.c_void_p(wn.data_ptr()),
                                          ctypes.c_void_p(inten.data_ptr()), stream) == -1
        assert lib.rn_md_spectrum_windows(handle, ctypes.c_void_p(series.data_ptr()), len(alpha), 0, 1.0, 0, 0.0,
                                          0, 0.0, ctypes.c_void_p(wn.data_ptr()),
                                          ctypes.c_void_p(inten.data_ptr()), stream) == -1
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(handle)
    bad = ctypes.c_void_p()
    assert lib.rn_spectrum_plan_create_batched(window, 0, 0, ctypes.byref(bad)) == -1
    assert lib.rn_spectrum_plan_create_batched(window, 65536, 0, ctypes.byref(bad)) == -1


@pytest.mark.parametrize("window", [2000, 40_001])
def test_launch_count_matches_single_measure(window):
    alpha = to_cuda(_series(window * 6, 18))
    spectrum = rb.MDRamanSpectrum(alpha, 1.0)
    single = rb.MDRamanSpectrum(alpha[:window].contiguous(), 1.0)
    spectrum.measure_windows_device(window, window // 3)  # plans are created (and cached) here
    single.measure_device()
    torch.cuda.synchronize()
    before = _lib.launch_count()
    spectrum.measure_windows_device(window, window // 3)
    windowed = _lib.launch_count() - before
    before = _lib.launch_count()
    single.measure_device()
    assert windowed == _lib.launch_count() - before


def test_real_model_series():
    """Windows of the series of a real TiO2 model (25 DFT geometries) through Trajectory.get_raman_spectrum."""
    with np.load(f"{GOLDEN}/real_tio2.npz") as data:
        model = rb.InterpolationModel(state_from_tables(data, "k3"))
        spectrum = rb.Trajectory(data["positions"], 1.0).get_raman_spectrum(model)
        alpha = spectrum.polarizability_ts
        assert np.array_equal(spectrum.measure_windows(9, 4)[1],
                              rb.MDRamanSpectrum(alpha, 1.0).measure_windows(9, 4)[1])
        _check(alpha, 9, 4, oracle_rows=(0, 1, 2, 3, 4))
        _check(alpha, 12, None, oracle_rows=(0, 1), laser_correction=True, bose_einstein_correction=True)


def test_windows_of_get_raman_spectra():
    state = synthetic.make_model("LLZO", "art")
    model = rb.ARTModel(state)
    keep = np.flatnonzero(np.random.default_rng(3).random(state.num_dofs) < 0.5)
    positions = synthetic.make_trajectory("LLZO", 3000, seed=19)
    for resident in (False, True):
        trajectory = rb.Trajectory(to_cuda(positions) if resident else positions, 2.0)
        for spectrum in trajectory.get_raman_spectra([model, model.get_masked_model(keep)]):
            wn, inten = spectrum.measure_windows(1000, 500)
            alpha = spectrum.polarizability_ts
            for w in range(inten.shape[0]):
                want_wn, want = rb.MDRamanSpectrum(alpha[w * 500: w * 500 + 1000], 2.0).measure()
                assert np.array_equal(wn, want_wn) and np.array_equal(inten[w], want)
            ref_wn, ref = ora.md_measure(alpha[500:1500], 2.0)
            assert np.array_equal(wn, ref_wn) and pointwise_rel_err(inten[1], ref) <= INTENSITY_RTOL

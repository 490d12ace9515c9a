"""Batched smearing (``convolve_spectra``) on the GPU: every row against ``convolve_spectrum`` of that row bit for
bit (both functions, default and custom grids, row counts around the row group of the kernel, input lengths around
its input chunk, unsorted inputs, skipped tiles, NaN and Inf rows, the rows of ``measure_windows`` and of
``measure_cross_spectra``), against the oracle, linearity over the cross spectra, the input forms, the launch
count and the C entry's errors."""
import ctypes

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib
from ramannoodle_b200 import spectrum as sp

from gpu_helpers import to_cuda
from helpers import rel_err

pytestmark = pytest.mark.gpu

GROUP = 8        # kRows in csrc/rn_smear.cu
IN_CHUNK = 2048  # kInChunk
WIDTHS = {"gaussian": 2.0, "lorentzian": 6.0}


def _spectra(rows, length, seed, shuffle=False):
    """Wavenumbers spread over 1..3000 (sorted unless ``shuffle``) and rows of both signs."""
    rng = np.random.default_rng(seed)
    wn = np.sort(rng.uniform(1.0, 3000.0, length))
    if shuffle:
        wn = rng.permutation(wn)
    return wn, rng.normal(size=(rows, length)) * rng.uniform(0.5, 2.0, (rows, 1))


def _singles(wn, rows, function, width, grid=None):
    """convolve_spectrum of every row of a (B, P) stack -> (out_wavenumbers, (B, Q))."""
    out = [rb.convolve_spectrum(wn, row, function, width, grid) for row in rows]
    return out[0][0], np.stack([o[1] for o in out])


def _check_rows(wn, rows, function, width, grid=None):
    got_wn, got = rb.convolve_spectra(wn, rows, function, width, grid)
    want_wn, want = _singles(wn, rows.reshape(-1, rows.shape[-1]), function, width, grid)
    assert np.array_equal(got_wn, want_wn)
    assert got.shape == rows.shape[:-1] + (len(got_wn),)
    flat = got.reshape(-1, len(got_wn))
    for b in range(flat.shape[0]):
        assert np.array_equal(flat[b], want[b], equal_nan=True), f"row {b}"
    return got_wn, got


@pytest.mark.parametrize("length", [2 * IN_CHUNK - 1, 2 * IN_CHUNK, 2 * IN_CHUNK + 1])
@pytest.mark.parametrize("rows", [1, GROUP - 1, GROUP, GROUP + 1, 2 * GROUP + 3])
@pytest.mark.parametrize("function", ["gaussian", "lorentzian"])
def test_rows_bit_identical_to_single_calls(function, rows, length):
    wn, inten = _spectra(rows, length, 100 * rows + length)
    _check_rows(wn, inten, function, WIDTHS[function])
    _check_rows(wn, inten, function, WIDTHS[function], np.linspace(-150.0, 3200.0, 2777))


@pytest.mark.parametrize("function", ["gaussian", "lorentzian"])
def test_unsorted_input(function):
    wn, inten = _spectra(2 * GROUP + 3, 2 * IN_CHUNK + 1, 7, shuffle=True)
    _check_rows(wn, inten, function, WIDTHS[function])
    _check_rows(wn, inten, function, WIDTHS[function], np.linspace(500.0, 900.0, 401))


def test_one_spectrum_has_the_shape_of_convolve_spectrum():
    wn, inten = _spectra(1, 3000, 9)
    for function in WIDTHS:
        got_wn, got = rb.convolve_spectra(wn, inten[0], function, 5)
        want_wn, want = rb.convolve_spectrum(wn, inten[0], function, 5)
        assert got.shape == want.shape == want_wn.shape
        assert np.array_equal(got_wn, want_wn) and np.array_equal(got, want)


def _synthetic_series(frames, seed, count=None):
    device = torch.device("cuda:0")
    gen = torch.Generator(device).manual_seed(seed)
    lead = () if count is None else (count,)
    steps = torch.arange(frames, dtype=torch.float64, device=device)[:, None, None]
    phase = torch.rand(lead + (1, 3, 3), dtype=torch.float64, device=device, generator=gen) * 6
    noise = torch.randn(lead + (frames, 3, 3), dtype=torch.float64, device=device, generator=gen)
    return 6.0 * torch.eye(3, dtype=torch.float64, device=device) + 0.05 * torch.sin(0.013 * steps + phase) \
        + 0.01 * noise


def test_spectrogram_rows_of_measure_windows():
    """W = 1997 windows of 2000 frames at hop 500 over 1e6 frames, device inputs."""
    wn, inten = rb.MDRamanSpectrum(_synthetic_series(1_000_000, 1), 1.0).measure_windows_device(2000, 500)
    assert inten.shape == (1997, 999)
    for function in WIDTHS:
        got_wn, got = rb.convolve_spectra_device(wn, inten, function, 5)
        for w in range(inten.shape[0]):
            want_wn, want = rb.convolve_spectrum(wn, inten[w], function, 5)
            assert np.array_equal(want, got[w].cpu().numpy()), f"{function} window {w}"
        assert np.array_equal(got_wn.cpu().numpy(), want_wn)


def test_cross_spectra_rows_and_linearity():
    """(G, G, P) cross spectra with negative cross rows; the smeared rows add up to the smeared total."""
    series = _synthetic_series(20_001, 2, count=3)
    spectra = [rb.MDRamanSpectrum(series[g], 1.0) for g in range(3)]
    wn, cross = rb.measure_cross_spectra(spectra)
    off = cross[~np.eye(3, dtype=bool)]
    assert np.any(off < 0)
    for function in WIDTHS:
        got_wn, got = _check_rows(wn, cross, function, 5)
        _, total = rb.convolve_spectrum(wn, cross.sum(axis=(0, 1)), function, 5)
        summed = got.sum(axis=(0, 1))
        assert np.max(np.abs(summed - total)) <= 1e-12 * np.max(np.abs(total))
        assert got_wn.shape == total.shape


def test_skipping_case_with_five_rows():
    """The skipping case of test_smearing_many_points_with_tile_skipping with 5 rows."""
    rng = np.random.default_rng(8)
    wn = np.sort(rng.uniform(1.0, 4000.0, 30_000))
    inten = rng.uniform(0.0, 2.0, (5, 30_000))
    grid = np.linspace(-100.0, 4100.0, 1500)
    for function, width in (("gaussian", 2.0), ("lorentzian", 6.0)):
        _, got = _check_rows(wn, inten, function, width, grid)
        d_wn, d_in, d_grid = to_cuda(wn), to_cuda(inten), to_cuda(grid)
        dx = d_wn[None, :] - d_grid[:, None]
        if function == "gaussian":
            factor = (1 / width) * (1 / np.sqrt(2 * np.pi)) * torch.exp(-(dx**2) / (2 * width**2))
        else:
            factor = (1 / np.pi) * (0.5 * width / (dx**2 + (0.5 * width) ** 2))
        for b in range(5):
            ref = (factor * d_in[b][None, :]).sum(dim=1).cpu().numpy()
            assert rel_err(got[b], ref) <= 1e-12


def test_non_finite_rows():
    """A NaN in row 2 and an Inf in row 12 turn skipping off for their groups; every row is still its single
    call bit for bit (NaN positions included)."""
    wn, inten = _spectra(2 * GROUP + 3, 3 * IN_CHUNK, 11)
    inten[2, 5000] = np.nan
    inten[12, 100] = np.inf
    for function in WIDTHS:
        _, got = _check_rows(wn, inten, function, WIDTHS[function])
        assert np.isnan(got[2]).any() and not np.isnan(got[0]).any() and not np.isnan(got[GROUP]).any()
        assert not np.isfinite(got[12]).all()


def test_against_the_oracle():
    wn, inten = _spectra(5, 300, 12)
    for function in WIDTHS:
        for grid in (None, np.linspace(0.0, 3100.0, 517)):
            got_wn, got = rb.convolve_spectra(wn, inten, function, 4.0, grid)
            for b in range(5):
                want_wn, want = ora.convolve_spectrum(wn, inten[b], function, 4.0, grid)
                assert np.array_equal(got_wn, want_wn)
                assert rel_err(got[b], want) <= 1e-12


def test_input_forms_give_the_same_bits(monkeypatch):
    wn, inten = _spectra(2 * GROUP + 3, 5000, 13)
    want_wn, want = rb.convolve_spectra(wn, inten)
    for form in (torch.from_numpy(inten), to_cuda(inten)):
        got_wn, got = rb.convolve_spectra(wn, form)
        assert np.array_equal(got_wn, want_wn) and np.array_equal(got, want)
    got_wn, got = rb.convolve_spectra(to_cuda(wn), to_cuda(inten), out_wavenumbers=to_cuda(want_wn))
    assert np.array_equal(got_wn, want_wn) and np.array_equal(got, want)

    lib = _lib.lib()
    calls = []
    original = lib.rn_convolve_spectra

    def spy(*args):
        calls.append(args)
        return original(*args)

    monkeypatch.setattr(lib, "rn_convolve_spectra", spy)
    d_in = to_cuda(inten)
    _, got = rb.convolve_spectra_device(wn, d_in)
    assert len(calls) == 1 and calls[0][1].value == d_in.data_ptr()  # read in place, not copied
    assert np.array_equal(got.cpu().numpy(), want)

    calls.clear()
    row_bytes = int(lib.rn_convolve_spectra_workspace_size(1, len(wn), len(want_wn)))
    monkeypatch.setattr(sp, "_SMEAR_BLOCK_BYTES", 5 * row_bytes)
    _, got = rb.convolve_spectra_device(wn, d_in)
    assert [c[2] for c in calls] == [5, 5, 5, 4]
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("rows", [1, 8, 1997])
def test_two_launches_whatever_the_row_count(rows):
    wn, inten = _spectra(rows, 999, 14)
    d_wn, d_in = to_cuda(wn), to_cuda(inten)
    rb.convolve_spectra_device(d_wn, d_in)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    rb.convolve_spectra_device(d_wn, d_in)
    assert _lib.launch_count() - before == 2


def test_c_entry_errors():
    lib = _lib.lib()
    wn, inten = _spectra(3, 100, 15)
    d_wn, d_in, d_grid = to_cuda(wn), to_cuda(inten), to_cuda(np.linspace(0.0, 3000.0, 300))
    d_out = torch.full((3, 300), 7.0, dtype=torch.float64, device="cuda:0")
    workspace = torch.empty(int(lib.rn_convolve_spectra_workspace_size(3, 100, 300)) // 8, dtype=torch.float64,
                            device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    ptr = [ctypes.c_void_p(t.data_ptr()) for t in (d_wn, d_in, d_grid, d_out, workspace)]

    def call(rows, kind=0, width=5.0, num_in=100):
        return lib.rn_convolve_spectra(ptr[0], ptr[1], rows, num_in, kind, width, ptr[2], 300, ptr[3], ptr[4],
                                       stream)

    assert call(-1) == -1 and "negative number of rows" in _lib.last_error()
    assert call(3, kind=2) == -1 and "unsupported convolution type: 2" in _lib.last_error()
    assert call(3, width=0.0) == -1 and "invalid width" in _lib.last_error()
    assert call(3, num_in=-1) == -1
    before = _lib.launch_count()
    assert call(0) == 0
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert torch.all(d_out == 7.0)
    assert call(3) == 0
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), _singles(wn, inten, "gaussian", 5.0, d_grid.cpu().numpy())[1])
    assert call(3, num_in=0) == 0  # no input points: zeros
    torch.cuda.synchronize()
    assert torch.all(d_out == 0.0)

"""``convolve_spectra``: argument errors (those of ``convolve_spectrum``, raised before any device work), the
row-block split of the workspace at its edges and the output layout.  No GPU needed."""
import re

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from ramannoodle_b200 import spectrum as sp

WN = np.array([1.0, 2.0, 3.0])
ROWS = np.ones((4, 3))


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    """Any device work fails the test: argument errors must come first."""
    def fail(*_args, **_kwargs):
        raise AssertionError("device work before the argument check")

    monkeypatch.setattr(sp, "_current_device", fail)
    monkeypatch.setattr(sp._lib, "require_device", fail)  # pylint: disable=protected-access
    monkeypatch.setattr(sp, "_to_device", fail)


@pytest.mark.parametrize("call", [rb.convolve_spectra, rb.convolve_spectra_device])
def test_argument_errors(call, no_device):  # pylint: disable=unused-argument
    with pytest.raises(ValueError, match="invalid width: -1 <= 0"):
        call(WN, ROWS, "gaussian", -1)
    with pytest.raises(ValueError, match="invalid width: 0 <= 0"):
        call(WN, ROWS, "lorentzian", 0)
    with pytest.raises(TypeError, match="width should have type float, not str"):
        call(WN, ROWS, "gaussian", "5")
    with pytest.raises(ValueError, match="unsupported convolution type: blah"):
        call(WN, ROWS, "blah", 3)
    with pytest.raises(TypeError, match="out_wavenumbers should have type ndarray, not list"):
        call(WN, ROWS, "gaussian", 5, [1.0, 2.0])
    with pytest.raises(ValueError, match=r"out_wavenumbers has wrong shape: \(2,2\) != \(_,\)"):
        call(WN, ROWS, "gaussian", 5, np.ones((2, 2)))
    with pytest.raises(TypeError, match="wavenumbers should have type ndarray, not list"):
        call([1.0, 2.0, 3.0], ROWS, "gaussian", 5, WN)
    with pytest.raises(TypeError, match="intensities should have type ndarray, not list"):
        call(WN, [[0, 3, 0]], "gaussian", 5)
    with pytest.raises(ValueError, match=r"intensities has shape \(4,2\), wavenumbers has shape \(3,\)"):
        call(WN, np.ones((4, 2)), "gaussian", 5)
    with pytest.raises(ValueError, match=r"intensities has shape \(3,4\), wavenumbers has shape \(3,\)"):
        call(WN, np.ones((3, 4)), "gaussian", 5)
    with pytest.raises(ValueError, match=r"intensities has shape \(\), wavenumbers has shape \(3,\)"):
        call(WN, np.float64(2.0), "gaussian", 5)
    with pytest.raises(ValueError, match=r"intensities has shape \(2,2,2\), wavenumbers has shape \(3,\)"):
        call(WN, torch.ones((2, 2, 2), dtype=torch.float64), "gaussian", 5)


def test_errors_match_convolve_spectrum(no_device):  # pylint: disable=unused-argument
    """The checks the two functions share give the same exception and message for a 1-D spectrum."""
    cases = [(WN, WN, "gaussian", -1, None), (WN, WN, "x", 3, None), (WN, WN, "gaussian", "5", None),
             (WN, WN, "gaussian", 5, [1.0]), (WN, WN, "gaussian", 5, np.ones((1, 2))), ([1.0], WN, "gaussian", 5, WN),
             (WN, [0, 3, 0], "gaussian", 5, None)]
    for args in cases:
        with pytest.raises((TypeError, ValueError)) as single:
            rb.convolve_spectrum(*args)
        with pytest.raises(single.type, match=f"^{re.escape(str(single.value))}$"):
            rb.convolve_spectra(*args)


def test_row_block_split_at_the_budget(monkeypatch):
    split = sp._smear_rows_per_block  # pylint: disable=protected-access
    budget = sp._SMEAR_BLOCK_BYTES  # pylint: disable=protected-access
    assert budget == 1 << 30
    assert split(1, 10**12) == 1  # one row always runs, whatever it needs
    assert split(1, 8) == 1
    assert split(1997, 8 * 16_878) == 1997  # a measure_windows spectrogram fits one block
    assert split(8, budget // 8) == 8  # exactly at the budget
    assert split(9, budget // 8) == 8  # one row over it
    assert split(3, budget) == 1
    assert split(3, budget + 1) == 1
    assert split(5, 0) == 5  # nothing to sum (no input or no output points)
    monkeypatch.setattr(sp, "_SMEAR_BLOCK_BYTES", 100)
    assert split(10, 30) == 3


def test_layout_of_rows():
    layout = sp._smeared_layout  # pylint: disable=protected-access
    assert layout((7,), 5) == (1, (5,))  # one spectrum: the (Q,) shape of convolve_spectrum
    assert layout((1997, 999), 1199) == (1997, (1997, 1199))
    assert layout((4, 4, 99), 300) == (16, (4, 4, 300))
    assert layout((0, 3), 10) == (0, (0, 10))
    assert layout((2, 3), 0) == (2, (2, 0))

"""``MDRamanSpectrum.measure_windows``: argument errors (raised before any device work), and the number of
windows, points and windows per chunk at the edges.  No GPU needed."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import spectrum as sp
from ramannoodle_b200.distributed import ShardedMDRamanSpectrum


def _spectra():
    alpha = np.random.default_rng(0).normal(size=(30, 3, 3))
    return rb.MDRamanSpectrum(alpha, 1.0), ShardedMDRamanSpectrum(alpha, 1.0)


@pytest.mark.parametrize("which", [0, 1])
def test_window_argument_errors(which):
    spectrum = _spectra()[which]
    for call in (spectrum.measure_windows, spectrum.measure_windows_device):
        with pytest.raises(TypeError, match="window_frames should have type int, not float"):
            call(10.0)
        with pytest.raises(TypeError, match="window_frames should have type int, not bool"):
            call(True)
        with pytest.raises(TypeError, match="window_frames should have type int, not str"):
            call("10")
        with pytest.raises(TypeError, match="hop_frames should have type int, not float"):
            call(10, 2.5)
        with pytest.raises(ValueError, match=r"invalid window_frames: 1 \(a window needs 2 to 30 frames\)"):
            call(1)
        with pytest.raises(ValueError, match=r"invalid window_frames: 31 \(a window needs 2 to 30 frames\)"):
            call(31)
        with pytest.raises(ValueError, match="invalid hop_frames: 0 < 1"):
            call(10, 0)
        with pytest.raises(ValueError, match="invalid hop_frames: -3 < 1"):
            call(np.int64(10), np.int32(-3))


@pytest.mark.parametrize("which", [0, 1])
def test_measure_argument_errors_match_measure(which):
    spectrum = _spectra()[which]
    with pytest.raises(NotImplementedError, match="only polycrystalline spectra are supported for now"):
        spectrum.measure_windows(10, orientation="single crystal")
    with pytest.raises(ValueError, match="invalid temperature: -1 <= 0"):
        spectrum.measure_windows(10, bose_einstein_correction=True, temperature=-1)
    with pytest.raises(TypeError, match="temperature should have type float, not str"):
        spectrum.measure_windows(10, bose_einstein_correction=True, temperature="hot")
    with pytest.raises(ValueError, match="invalid laser_wavenumber"):
        spectrum.measure_windows(10, laser_correction=True, laser_wavelength=-5)


def test_windows_and_points_at_the_edges():
    assert sp.num_windows(30, 30, 30) == 1
    assert sp.num_windows(30, 30, 1) == 1
    assert sp.num_windows(30, 2, 2) == 15
    assert sp.num_windows(30, 3, 3) == 10
    assert sp.num_windows(31, 3, 3) == 10  # a trailing frame that fills no window is not used
    assert sp.num_windows(30, 2, 1) == 29
    assert sp.num_windows(30, 10, 25) == 1
    assert sp.num_windows(1_000_000, 2000, 500) == 1997
    from ramannoodle_b200 import _lib

    num_points = _lib.lib().rn_spectrum_num_points
    assert [num_points(s) for s in (2, 3, 4, 5, 30)] == [0, 0, 1, 1, 14]


def test_window_batch_budget():
    # windows of up to 2049 frames use a 4096-point transform: 196608 work bytes per window and more
    per_window = 16 * 3 * 4096 + 8 * 3 * 1999 + 8 * 9 + 4
    assert sp._window_batch(2000, 1997) == 2048  # pylint: disable=protected-access  (rounded up to a power of two)
    assert sp._window_batch(2000, 1025) == 2048  # pylint: disable=protected-access  (the same plan)
    assert sp._window_batch(2000, 1) == 1  # pylint: disable=protected-access
    assert sp._window_batch(2000, 10**6) == (1 << 30) // per_window  # pylint: disable=protected-access
    assert sp._window_batch(2, 10**7) <= 65535  # pylint: disable=protected-access
    assert sp._window_batch(10**7, 3) == 1  # pylint: disable=protected-access
    assert sp._window_batch(1_000_001, 10) == 8  # pylint: disable=protected-access  (2^21-point transforms)

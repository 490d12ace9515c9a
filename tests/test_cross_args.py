"""Cross spectra without a GPU: the oracle's ``md_cross_measure`` against ``md_measure`` (diagonal bit for bit,
off-diagonal against the polarization identity), and the argument errors of ``measure_cross_spectra``, raised
before any device work."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib
from ramannoodle_b200.distributed import ShardedMDRamanSpectrum

from cross_oracle import md_cross_measure

CORRECTIONS = [{}, dict(laser_correction=True, laser_wavelength=532, bose_einstein_correction=True, temperature=250)]


def _series(frames, seed):
    rng = np.random.default_rng(seed)
    steps = np.arange(frames)[:, None, None]
    return (6.0 * np.eye(3)[None] + 0.05 * np.sin(0.013 * steps + rng.uniform(0, 6, (1, 3, 3)))
            + 0.01 * rng.normal(size=(frames, 3, 3)))


@pytest.mark.parametrize("kwargs", CORRECTIONS)
@pytest.mark.parametrize("frames", [5, 64, 301])
def test_oracle_diagonal_is_md_measure(frames, kwargs):
    series = [_series(frames, seed) for seed in range(3)]
    wn, cross = md_cross_measure(series, 1.5, **kwargs)
    assert cross.shape == (3, 3, len(wn))
    for g, alpha in enumerate(series):
        want_wn, want = ora.md_measure(alpha, 1.5, **kwargs)
        assert np.array_equal(wn, want_wn)
        assert np.array_equal(cross[g, g], want)


@pytest.mark.parametrize("kwargs", CORRECTIONS)
def test_oracle_off_diagonal_is_the_polarization_identity(kwargs):
    """I_gh = (I[alpha_g + alpha_h] - I_gg - I_hh) / 2, to the identity's own cancellation error."""
    series = [_series(401, 10), _series(401, 11), 0.3 * _series(401, 12)[::-1].copy()]
    _, cross = md_cross_measure(series, 2.0, **kwargs)
    for g in range(3):
        for h in range(g + 1, 3):
            _, both = ora.md_measure(series[g] + series[h], 2.0, **kwargs)
            identity = (both - cross[g, g] - cross[h, h]) / 2
            assert np.array_equal(cross[g, h], cross[h, g])
            assert np.all(np.abs(cross[g, h] - identity) <= 1e-12 * (cross[g, g] + cross[h, h]))


def test_oracle_sum_rule_of_a_split_series():
    """Series whose differences add up to those of a total: the G x G cross spectra add up to its spectrum."""
    parts = [_series(257, 20), _series(257, 21), _series(257, 22)]
    _, cross = md_cross_measure(parts, 1.0)
    _, total = ora.md_measure(parts[0] + parts[1] + parts[2], 1.0)
    scale = np.sum(np.sqrt(np.abs(np.diagonal(cross, axis1=0, axis2=1))), axis=1) ** 2
    assert np.all(np.abs(cross.sum(axis=(0, 1)) - total) <= 1e-12 * scale)


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("call", [rb.measure_cross_spectra, rb.measure_cross_spectra_device])
def test_argument_errors_before_device_work(call, no_device):  # pylint: disable=unused-argument
    alpha = _series(30, 0)
    one, two = rb.MDRamanSpectrum(alpha, 1.0), ShardedMDRamanSpectrum(alpha, 1.0)
    with pytest.raises(TypeError, match="spectra should have type list, not int"):
        call(5)
    with pytest.raises(TypeError, match="spectra should have type list, not str"):
        call("spectra")
    with pytest.raises(TypeError, match="spectra should have type list, not MDRamanSpectrum"):
        call(one)
    with pytest.raises(TypeError, match="spectra should have type MDRamanSpectrum, not ndarray"):
        call([one, alpha])
    with pytest.raises(ValueError, match="spectra is empty"):
        call([])
    with pytest.raises(ValueError, match=r"spectra\[1\] has 20 frames, spectra\[0\] has 30"):
        call([one, rb.MDRamanSpectrum(alpha[:20], 1.0)])
    with pytest.raises(ValueError, match=r"spectra\[2\] has timestep 2.0, spectra\[0\] has 1.0"):
        call((one, two, rb.MDRamanSpectrum(alpha, 2.0)))
    with pytest.raises(ValueError, match="polarizability_ts must contain at least 2 configurations"):
        call([rb.MDRamanSpectrum(alpha[:1], 1.0)] * 2)
    with pytest.raises(NotImplementedError, match="only polycrystalline spectra are supported for now"):
        call([one, two], orientation="single crystal")
    with pytest.raises(ValueError, match="invalid temperature: -1 <= 0"):
        call([one, two], bose_einstein_correction=True, temperature=-1)
    with pytest.raises(TypeError, match="temperature should have type float, not str"):
        call([one], bose_einstein_correction=True, temperature="hot")
    with pytest.raises(ValueError, match="invalid laser_wavenumber"):
        call([one, two], laser_correction=True, laser_wavelength=-5)
    with pytest.raises(AssertionError, match="device work"):  # valid arguments reach the device
        call([one, two])

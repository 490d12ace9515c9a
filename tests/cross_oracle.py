"""CPU oracle of cross spectra (``measure_cross_spectra``): ``md_measure`` of ``oracle/numpy_port.py`` with every
``calc_signal_spectrum(sig)`` replaced by the spectrum of the symmetrised cross-correlation of the same signal of
two series.  No reference counterpart; written with the reference's own calls (``scipy.signal.correlate``,
``scipy.fftpack.fft/fftfreq``) in the structure of ``md_measure``.  Test infrastructure only."""
import numpy as np
import scipy.fftpack
import scipy.signal

from oracle.numpy_port import calc_signal_spectrum, get_bose_einstein_correction, get_laser_correction


def calc_cross_signal_spectrum(signal_a, signal_b, sampling_rate):
    """``calc_signal_spectrum`` of two signals: the autocorrelation is replaced by the symmetrised
    cross-correlation ``(correlate(a, b) + correlate(b, a)) / 2`` (no reference counterpart; equal to
    ``calc_signal_spectrum(a)`` bit for bit when ``b is a``)."""
    correlation = (scipy.signal.correlate(signal_a, signal_b, "full")
                   + scipy.signal.correlate(signal_b, signal_a, "full")) / 2
    correlation = correlation[(len(correlation) - 1) // 2:]
    wavenumbers = (
        scipy.fftpack.fftfreq(correlation.size, sampling_rate)
        * 33.35640951981521
        * 1e3
    )
    intensities = np.real(scipy.fftpack.fft(correlation))
    return wavenumbers[wavenumbers >= 0], intensities[wavenumbers >= 0]


def md_cross_measure(series_list, timestep, laser_correction=False, laser_wavelength=522,
                     bose_einstein_correction=False, temperature=300):
    """Cross spectra ``I_gh`` of G (S,3,3) series -> wavenumbers (P,), intensities (G,G,P): ``md_measure``
    with every ``calc_signal_spectrum(sig)`` replaced by ``calc_cross_signal_spectrum(sig_g, sig_h)``.
    ``I_gg`` is ``md_measure`` of series g bit for bit."""
    diffs = [np.diff(series, axis=0) for series in series_list]
    wavenumbers, _ = calc_signal_spectrum(diffs[0][:, 0, 0], timestep)
    wavenumbers = wavenumbers[1:]
    rows = []
    for a in diffs:
        row = []
        for b in diffs:
            def spec(sig_a, sig_b):
                return calc_cross_signal_spectrum(sig_a, sig_b, timestep)[1]

            alpha2 = (1 / 9) * spec(a[:, 0, 0] + a[:, 1, 1] + a[:, 2, 2], b[:, 0, 0] + b[:, 1, 1] + b[:, 2, 2])
            gamma2 = (
                (1 / 2) * spec(a[:, 0, 0] - a[:, 1, 1], b[:, 0, 0] - b[:, 1, 1])
                + (1 / 2) * spec(a[:, 1, 1] - a[:, 2, 2], b[:, 1, 1] - b[:, 2, 2])
                + (1 / 2) * spec(a[:, 2, 2] - a[:, 0, 0], b[:, 2, 2] - b[:, 0, 0])
                + 3 * spec(a[:, 0, 1], b[:, 0, 1])
                + 3 * spec(a[:, 1, 2], b[:, 1, 2])
                + 3 * spec(a[:, 0, 2], b[:, 0, 2])
            )
            intensities = 45.0 * alpha2 + 7.0 * gamma2
            intensities = intensities[1:]
            if laser_correction:
                laser_wavenumber = 10000000 / laser_wavelength
                intensities *= get_laser_correction(wavenumbers, laser_wavenumber)
            if bose_einstein_correction:
                intensities *= get_bose_einstein_correction(wavenumbers, temperature)
            row.append(intensities)
        rows.append(row)
    return wavenumbers, np.array(rows).reshape(len(diffs), len(diffs), len(wavenumbers))

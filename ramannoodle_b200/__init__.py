"""ramannoodle_b200 — B200-native (sm_100a) MD-Raman hot path for ramannoodle.

Drop-in replacements for the three subsystems on the path
(``PolarizabilityModel.calc_polarizabilities`` of ``InterpolationModel``/``ARTModel``,
``Trajectory.get_raman_spectrum``, ``MDRamanSpectrum.measure`` + ``convolve_spectrum``),
implemented as hand-written CUDA behind the C-ABI in ``include/ramannoodle_b200.h``.
"""
from .abstract import Dynamics, PolarizabilityModel, RamanSpectrum
from .dynamics import Phonons, Trajectory
from .exceptions import NativeLibraryError, UserError
from .dropin import install, uninstall
from .pmodel import ARTModel, InterpolationModel, accelerate, calc_polarizabilities_sweep
from .spectrum import (MDRamanSpectrum, PhononRamanSpectrum, calc_signal_spectrum, convolve_spectra,
                       convolve_spectra_device, convolve_spectrum, get_bose_einstein_correction, get_laser_correction,
                       measure_cross_spectra, measure_cross_spectra_device)
from .state import ModelState

__all__ = [
    "ARTModel", "Dynamics", "InterpolationModel", "MDRamanSpectrum", "ModelState", "NativeLibraryError",
    "Phonons", "PhononRamanSpectrum", "PolarizabilityModel", "RamanSpectrum", "Trajectory", "UserError", "accelerate", "calc_signal_spectrum", "install", "uninstall",
    "convolve_spectrum", "get_bose_einstein_correction", "get_laser_correction", "measure_cross_spectra",
    "measure_cross_spectra_device", "convolve_spectra", "convolve_spectra_device",
]

"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares,
the host-side spline packing (B-spline -> piecewise polynomial) matches scipy, and the
Python drop-in layer validates arguments like the reference.  No GPU compute is issued."""
import ctypes
import os
import re

import numpy as np
import pytest
from scipy.interpolate import BSpline, make_interp_spline

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic
from ramannoodle_b200.exceptions import NativeLibraryError, shape_string

from helpers import REPO


def _declared_symbols():
    header = open(os.path.join(REPO, "include", "ramannoodle_b200.h"), encoding="utf-8").read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    return sorted(set(re.findall(r"\b(rn_[a-z0-9_]+)\s*\(", header)))


def test_library_exports_every_declared_symbol():
    names = _declared_symbols()
    assert len(names) >= 20
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in names:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
    assert sorted(_lib.PROTOTYPES) == names, "python prototypes and header disagree"
    _lib.lib()


def test_python_prototypes_match_header_arity():
    """Every ctypes prototype takes as many arguments as the header's declaration (a mismatch would
    only show up as a crash on the GPU box)."""
    header = open(os.path.join(REPO, "include", "ramannoodle_b200.h"), encoding="utf-8").read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declarations = dict(re.findall(r"\b(rn_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S))
    assert sorted(declarations) == sorted(_lib.PROTOTYPES)
    for name, params in declarations.items():
        params = " ".join(params.split())
        count = 0 if params in ("", "void") else params.count(",") + 1
        assert count == len(_lib.PROTOTYPES[name][1]), f"{name}: header has {count} parameters"


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device the product path must fail loudly, not fall back."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    state = synthetic.make_model("TiO2", "art", num_dofs=6)
    with pytest.raises(NativeLibraryError, match="no CPU fallback"):
        rb.ARTModel(state).calc_polarizabilities(synthetic.make_trajectory("TiO2", 4))
    with pytest.raises(NativeLibraryError):
        rb.MDRamanSpectrum(np.zeros((10, 3, 3)), 1.0).measure()
    with pytest.raises(NativeLibraryError):
        rb.convolve_spectrum(np.arange(1.0, 5.0), np.ones(4))


def _pp_eval(t, c, k, x):
    """Evaluate through rn_bspline_to_pp exactly like the dense kernel's epilogue."""
    n = c.shape[0]
    breaks = np.zeros(n)
    x0 = np.zeros(n)
    coefs = np.zeros(n * (k + 1) * 9)
    pieces = _lib.lib().rn_bspline_to_pp(
        ctypes.c_void_p(t.ctypes.data), len(t), ctypes.c_void_p(np.ascontiguousarray(c.reshape(n, 9)).ctypes.data),
        k, ctypes.c_void_p(breaks.ctypes.data), ctypes.c_void_p(x0.ctypes.data), ctypes.c_void_p(coefs.ctypes.data))
    assert pieces >= 1
    coefs = coefs[: pieces * (k + 1) * 9].reshape(pieces, k + 1, 9)
    out = np.empty((len(x), 9))
    for i, xv in enumerate(x):
        p = int(np.sum(xv >= breaks[: pieces - 1]))
        dx = xv - x0[p]
        r = coefs[p, k].copy()
        for m in range(k - 1, -1, -1):
            r = r * dx + coefs[p, m]
        out[i] = r
    return pieces, out


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("n", [2, 3, 5, 6, 9])
def test_piecewise_polynomial_matches_scipy(k, n):
    """Spline packing (rn_model_create's B-spline -> local power basis, 80-bit arithmetic)
    reproduces BSpline(..., extrapolate=True) to rounding, including at knots and outside."""
    if n <= k:
        pytest.skip("needs n >= k+1")
    rng = np.random.default_rng(31 * k + n)
    xs = np.sort(rng.uniform(-0.25, 0.25, n))
    spline = make_interp_spline(xs, rng.normal(size=(n, 3, 3)), k=k, bc_type=None)
    probe = np.concatenate([rng.uniform(-0.3, 0.3, 300), xs, spline.t, [-2.0, 2.0]])
    pieces, got = _pp_eval(spline.t, spline.c, k, probe)
    want = BSpline(spline.t, spline.c, k, extrapolate=True)(probe).reshape(-1, 9)
    assert pieces == len(np.unique(spline.t[k:n + 1])) - 1
    scale = np.max(np.abs(want))
    assert np.max(np.abs(got - want)) <= 1e-12 * scale


def test_art_spline_is_one_linear_piece():
    spline = make_interp_spline(np.array([-0.1, 0.1]), np.arange(18.0).reshape(2, 3, 3), k=1, bc_type=None)
    assert list(spline.t) == [-0.1, -0.1, 0.1, 0.1]
    pieces, got = _pp_eval(spline.t, spline.c, 1, np.array([-0.1, 0.0, 0.1, 5.0]))
    assert pieces == 1
    assert np.allclose(got[1], np.arange(4.5, 13.5, 1.0))


def test_repeated_interior_knots_and_bad_tables():
    t = np.array([0.0, 0.0, 0.0, 0.5, 0.5, 1.0, 1.0, 1.0])  # double interior knot, k=2 -> n=5
    c = np.random.default_rng(0).normal(size=(5, 3, 3))
    probe = np.array([-0.3, 0.0, 0.2, 0.5, 0.7, 1.0, 1.4])
    pieces, got = _pp_eval(t, c, 2, probe)
    want = BSpline(t, c, 2, extrapolate=True)(probe).reshape(-1, 9)
    assert pieces == 2
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    out = np.zeros(64)
    bad = _lib.lib().rn_bspline_to_pp(ctypes.c_void_p(t.ctypes.data), 8, ctypes.c_void_p(c.ctypes.data), 9,
                                      ctypes.c_void_p(out.ctypes.data), ctypes.c_void_p(out.ctypes.data),
                                      ctypes.c_void_p(out.ctypes.data))
    assert bad < 0 and "degree" in _lib.last_error()


def test_state_tables_roundtrip():
    state = synthetic.make_model("STO", "mixed", num_dofs=30, masked_fraction=0.2)
    tables = state.tables()
    assert tables["basis"].shape == (30, 405) and tables["degree"].tolist() == [1 + (j % 3) for j in range(30)]
    assert tables["knot_off"][-1] == len(tables["knots"]) and tables["coefs"].shape == (tables["coef_off"][-1], 9)
    assert np.array_equal(tables["weight"], 1.0 - state.mask)
    before = state.fingerprint()
    state.mask = ~state.mask
    assert state.fingerprint() != before


def test_argument_validation_matches_reference_messages():
    """Validation happens before any device work, so it is checkable on a CPU box."""
    state = synthetic.make_model("TiO2", "art", num_dofs=6)
    model = rb.ARTModel(state)
    with pytest.raises(TypeError, match="positions should have type ndarray, not list"):
        model.calc_polarizabilities([1, 2, 3])
    with pytest.raises(ValueError, match=re.escape("positions has wrong shape: (2,5,3) != (_,108,3)")):
        model.calc_polarizabilities(np.zeros((2, 5, 3)))
    with pytest.raises(ValueError, match=re.escape("mask has wrong shape: (3,) != (6,)")):
        model.mask = np.zeros(3, dtype=bool)
    sto = synthetic.make_trajectory("STO", 3)
    with pytest.raises(ValueError, match="timestep must be positive"):
        rb.Trajectory(sto, 0)
    with pytest.raises(TypeError, match="timestep should have type float, not list"):
        rb.Trajectory(sto, [1])
    with pytest.raises(TypeError, match="positions_ts should have type ndarray, not list"):
        rb.Trajectory([[1.0]], 1.0)
    with pytest.raises(ValueError, match=re.escape("polarizability_ts has wrong shape: (4,3) != (_,3,3)")):
        rb.MDRamanSpectrum(np.zeros((4, 3)), 1.0)
    with pytest.raises(NotImplementedError, match="only polycrystalline spectra are supported for now"):
        rb.MDRamanSpectrum(np.zeros((4, 3, 3)), 1.0).measure(orientation="xx")
    with pytest.raises(ValueError, match="invalid width: 0 <= 0"):
        rb.convolve_spectrum(np.arange(1.0, 4.0), np.ones(3), "gaussian", 0)
    with pytest.raises(ValueError, match="invalid temperature: 0 <= 0"):
        rb.get_bose_einstein_correction(np.arange(1.0, 4.0), 0)
    with pytest.raises(TypeError, match="temperature should have type float, not list"):
        rb.get_bose_einstein_correction(np.arange(1.0, 4.0), [])
    with pytest.raises(ValueError, match="invalid laser_wavenumber: -1 <= 0"):
        rb.get_laser_correction(np.arange(1.0, 4.0), -1)
    assert shape_string((None, 3)) == "(_,3)" and shape_string((5,)) == "(5,)"
    traj = rb.Trajectory(np.array([[[1.25, -0.25, 0.5]]]), 1, pin_memory=False)
    assert np.array_equal(traj.positions_ts, [[[0.25, 0.75, 0.5]]]) and traj.timestep == 1.0 and len(traj) == 1


def test_multi_gpu_entry_argument_errors():
    """The broadcast and routed evaluation forms and the shared-spectrum ``measure_device`` reject bad
    arguments before any device work."""
    import types

    from ramannoodle_b200.distributed import ShardedMDRamanSpectrum

    model = rb.ARTModel(synthetic.make_model("TiO2", "art", num_dofs=6))
    positions = synthetic.make_trajectory("TiO2", 4)
    for count in (0, 9):
        with pytest.raises(ValueError, match="between 1 and 8 output pointers are required"):
            model.calc_polarizabilities_multi(positions, [0] * count)
        with pytest.raises(ValueError, match="between 1 and 8 ranks"):
            model.calc_polarizabilities_routed(positions, 0, [0] * count, 0, 64, 32)
    with pytest.raises(ValueError, match="phased evaluation needs an HBM-resident trajectory block"):
        model.calc_polarizabilities_routed(positions, 0, [0, 0], 0, 64, 32, stripe=64, phase=0)
    spectrum = ShardedMDRamanSpectrum(None, 1.0, context=types.SimpleNamespace(generation=0), bounds=(0, 4))
    with pytest.raises(NotImplementedError, match="only polycrystalline spectra are supported for now"):
        spectrum.measure_device(orientation="xx")
    with pytest.raises(ValueError, match="invalid laser_wavenumber: -10000000.0 <= 0"):
        spectrum.measure_device(laser_correction=True, laser_wavelength=-1)
    with pytest.raises(ValueError, match="invalid temperature: 0 <= 0"):
        spectrum.measure_device(bose_einstein_correction=True, temperature=0)
    with pytest.raises(TypeError, match="temperature should have type float, not list"):
        spectrum.measure_device(bose_einstein_correction=True, temperature=[])


def test_corrections_match_oracle():
    from oracle import numpy_port as ora

    wn = np.linspace(1.0, 3500.0, 500)
    assert np.array_equal(rb.get_bose_einstein_correction(wn, 300), ora.get_bose_einstein_correction(wn, 300))
    assert np.array_equal(rb.get_laser_correction(wn, 1e7 / 532), ora.get_laser_correction(wn, 1e7 / 532))


def test_trajectory_accepts_cpu_tensors():
    """A CPU torch tensor is host data: wrapped like an ndarray (ADVICE r1: ``_wrap_device`` called the
    instance method ``_wrap_host`` unbound and raised TypeError)."""
    import torch

    positions = np.random.default_rng(0).uniform(-1.5, 2.5, size=(4, 5, 3))
    trajectory = rb.Trajectory(torch.from_numpy(positions), 1.0, pin_memory=False)
    assert not trajectory.is_device_resident
    assert np.array_equal(np.asarray(trajectory.positions_ts), positions - positions // 1)


def test_spectrum_plans_are_not_shared_across_threads():
    """Plans own work buffers: the cache key includes the thread (and the CUDA stream), so two threads
    measuring series of the same length never get the same plan object."""
    import threading

    from ramannoodle_b200 import spectrum

    created = []

    class FakePlan:
        def __init__(self, num_frames, device):
            created.append((num_frames, device, threading.get_ident()))

        def close(self):
            pass

    original_plan, original_require = spectrum._Plan, _lib.require_device  # pylint: disable=protected-access
    spectrum._Plan, _lib.require_device = FakePlan, lambda device=0: {}  # pylint: disable=protected-access
    try:
        spectrum.clear_plan_cache()
        first = spectrum._get_plan(1000, 0)  # pylint: disable=protected-access
        assert spectrum._get_plan(1000, 0) is first  # pylint: disable=protected-access
        other = []
        worker = threading.Thread(target=lambda: other.append(spectrum._get_plan(1000, 0)))  # pylint: disable=protected-access
        worker.start()
        worker.join()
        assert other[0] is not first and len(created) == 2
    finally:
        spectrum._Plan, _lib.require_device = original_plan, original_require  # pylint: disable=protected-access
        spectrum._PLAN_CACHE.clear()  # pylint: disable=protected-access

"""Cross spectra (``measure_cross_spectra``) on the GPU: the diagonal against ``measure`` bit for bit, symmetry,
the off-diagonal against the oracle at the Cauchy-Schwarz scale sqrt(I_gg I_hh), the sum rule of masks that
partition the DOFs of real models, the no-copy and stacked inputs, the launch count and the C entry's errors."""
import ctypes

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib, synthetic

from cross_oracle import md_cross_measure
from gpu_helpers import to_cuda
from helpers import GOLDEN, state_from_tables

pytestmark = pytest.mark.gpu

CROSS_RTOL = 1e-8
CORRECTIONS = dict(laser_correction=True, laser_wavelength=532, bose_einstein_correction=True, temperature=250)


def _series(frames, seed):
    rng = np.random.default_rng(seed)
    steps = np.arange(frames)[:, None, None]
    return (6.0 * np.eye(3)[None] + 0.05 * np.sin(0.013 * steps + rng.uniform(0, 6, (1, 3, 3)))
            + 0.01 * rng.normal(size=(frames, 3, 3)))


def _host(series):
    return series.detach().cpu().numpy() if isinstance(series, torch.Tensor) else series


def _check_diagonal(spectra, wn, cross, **kwargs):
    """I[g,g] is measure() of spectrum g bit for bit; I[g,h] is I[h,g] bit for bit."""
    count = len(spectra)
    assert cross.shape == (count, count, len(wn))
    for g, spectrum in enumerate(spectra):
        want_wn, want = spectrum.measure(**kwargs)
        assert np.array_equal(wn, want_wn)
        assert np.array_equal(cross[g, g], want), f"row ({g},{g})"
        for h in range(count):
            assert np.array_equal(cross[g, h], cross[h, g]), f"rows ({g},{h}) and ({h},{g})"


def _check_oracle(series_list, timestep, wn, cross, **kwargs):
    ref_wn, ref = md_cross_measure([_host(s) for s in series_list], timestep, **kwargs)
    assert np.array_equal(wn, ref_wn)
    diag = np.abs(np.diagonal(ref, axis1=0, axis2=1)).T  # (G, P)
    scale = np.sqrt(diag[:, None, :] * diag[None, :, :])
    assert np.all(np.abs(cross - ref) <= CROSS_RTOL * scale)


def _check(series_list, timestep=1.0, oracle=True, **kwargs):
    spectra = [rb.MDRamanSpectrum(s, timestep) for s in series_list]
    wn, cross = rb.measure_cross_spectra(spectra, **kwargs)
    _check_diagonal(spectra, wn, cross, **kwargs)
    if oracle:
        _check_oracle(series_list, timestep, wn, cross, **kwargs)
    return wn, cross


@pytest.mark.parametrize("frames", [100, 2049, 2050, 40_001])
def test_lengths_around_plan_shapes(frames):
    """No strided level (L = 4096 up to 2049 frames), the first one-level length and a mid one-level size."""
    _check([_series(frames, frames + g) for g in range(3)])


@pytest.mark.parametrize("count", [1, 2, 3, 5])
def test_series_counts(count):
    _check([_series(1000, 30 + g) for g in range(count)], timestep=0.5)


@pytest.mark.parametrize("corrections", [False, True])
def test_corrections_and_timestep(corrections):
    kwargs = CORRECTIONS if corrections else {}
    _check([_series(3001, 40), _series(3001, 41), 0.2 * _series(3001, 42)[::-1].copy()], timestep=2.5, **kwargs)


@pytest.mark.parametrize("kind", ["numpy", "cpu", "cuda"])
def test_series_types(kind):
    alphas = [_series(1501, 50 + g) for g in range(3)]
    convert = {"numpy": lambda a: a, "cpu": torch.from_numpy, "cuda": to_cuda}[kind]
    _check([convert(a) for a in alphas])


def _species_groups(model, atomic_numbers):
    """DOF indexes per species: the atom a DOF's basis vector moves most."""
    basis = np.stack([np.abs(np.asarray(v)).reshape(-1, 3).max(axis=1) for v in model.cart_basis_vectors])
    owner = np.asarray(atomic_numbers)[np.argmax(basis, axis=1)]
    return [np.flatnonzero(owner == z).tolist() for z in sorted(set(owner.tolist()))]


def _check_sum_rule(model, groups, positions, timestep, **kwargs):
    """Copy g keeps only group g: sum_gh I_gh is the spectrum of the unmasked model."""
    num_dofs = len(model.cart_basis_vectors)
    assert sorted(j for group in groups for j in group) == list(range(num_dofs))
    copies = [model.get_masked_model([j for j in range(num_dofs) if j not in set(group)]) for group in groups]
    trajectory = rb.Trajectory(positions, timestep)
    spectra = trajectory.get_raman_spectra(copies)
    wn, cross = rb.measure_cross_spectra(spectra, **kwargs)
    _check_diagonal(spectra, wn, cross, **kwargs)
    total_wn, total = trajectory.get_raman_spectrum(model).measure(**kwargs)
    assert np.array_equal(wn, total_wn)
    scale = np.sum(np.sqrt(np.abs(np.diagonal(cross, axis1=0, axis2=1))), axis=1) ** 2
    assert np.all(np.abs(cross.sum(axis=(0, 1)) - total) <= CROSS_RTOL * scale)
    _check_oracle([s.polarizability_ts for s in spectra], timestep, wn, cross, **kwargs)
    return cross


@pytest.mark.parametrize("corrections", [False, True])
def test_sum_rule_real_tio2_art_by_species(corrections):
    kwargs = CORRECTIONS if corrections else {}
    with np.load(f"{GOLDEN}/real_tio2.npz") as data:
        state = state_from_tables(data, "art")
    state.atomic_numbers = [int(z) for z in synthetic.load_structure("TiO2")["atomic_numbers"]]
    model = rb.ARTModel(state)
    groups = [model.get_dof_indexes("Ti"), model.get_dof_indexes("O")]
    assert groups == _species_groups(model, state.atomic_numbers)[::-1]
    _check_sum_rule(model, groups, synthetic.make_trajectory("TiO2", 3001, seed=5), 1.0, **kwargs)


def test_sum_rule_sto_cubic_by_species():
    state = synthetic.make_model("STO", "cubic")
    model = rb.InterpolationModel(state)
    groups = _species_groups(model, synthetic.load_structure("STO")["atomic_numbers"])
    assert len(groups) == 3
    _check_sum_rule(model, groups, synthetic.make_trajectory("STO", 2001, seed=6), 1.0)


def test_no_copy_and_stacked_paths_are_bit_identical():
    state = synthetic.make_model("LLZO", "art")
    model = rb.ARTModel(state)
    rng = np.random.default_rng(3)
    copies = [model.get_masked_model(np.flatnonzero(rng.random(state.num_dofs) < 0.5)) for _ in range(4)]
    spectra = rb.Trajectory(to_cuda(synthetic.make_trajectory("LLZO", 4001, seed=7)), 1.0).get_raman_spectra(copies)
    series = [s._polarizability_ts for s in spectra]  # pylint: disable=protected-access
    step = series[0].numel() * 8
    assert all(t.data_ptr() == series[0].data_ptr() + g * step for g, t in enumerate(series))  # one (G,S,3,3) block
    wn, cross = rb.measure_cross_spectra_device(spectra)
    separate = [rb.MDRamanSpectrum(t.clone(), 1.0) for t in reversed(series)][::-1]
    wn2, cross2 = rb.measure_cross_spectra_device(separate)
    wn3, cross3 = rb.measure_cross_spectra_device(spectra)
    assert torch.equal(wn, wn2) and torch.equal(cross, cross2)
    assert torch.equal(wn, wn3) and torch.equal(cross, cross3)


def test_launch_count_does_not_grow_with_the_series_count():
    alpha = to_cuda(np.stack([_series(20_001, 60 + g) for g in range(8)]))
    counts = []
    for count in (2, 8):
        spectra = [rb.MDRamanSpectrum(alpha[g], 1.0) for g in range(count)]
        rb.measure_cross_spectra_device(spectra)  # plans are created (and cached) here
        torch.cuda.synchronize()
        before = _lib.launch_count()
        rb.measure_cross_spectra_device(spectra)
        counts.append(_lib.launch_count() - before)
    single = rb.MDRamanSpectrum(alpha[0], 1.0)
    single.measure_device()
    before = _lib.launch_count()
    single.measure_device()
    assert counts[0] == counts[1] == _lib.launch_count() - before + 1  # + the cross-energy kernel


def test_c_entry_errors():
    frames = 500
    lib = _lib.lib()
    alpha = to_cuda(np.stack([_series(frames, 70 + g) for g in range(3)]))
    points = int(lib.rn_spectrum_num_points(frames))
    wn = torch.empty(points, dtype=torch.float64, device="cuda:0")
    inten = torch.empty((3, 3, points), dtype=torch.float64, device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    handle = ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(frames, 2, 0, ctypes.byref(handle)), "create_batched")
    try:
        def call(plan, src, count, wn_ptr, int_ptr):
            return lib.rn_md_cross_spectra(plan, src, count, 1.0, 0, 0.0, 0, 0.0, wn_ptr, int_ptr, stream)

        src, wn_ptr, int_ptr = (ctypes.c_void_p(t.data_ptr()) for t in (alpha, wn, inten))
        assert call(handle, src, 3, wn_ptr, int_ptr) == -1  # batch 2 < G = 3
        assert call(handle, src, 0, wn_ptr, int_ptr) == -1
        assert call(None, src, 2, wn_ptr, int_ptr) == -1
        assert call(handle, None, 2, wn_ptr, int_ptr) == -1
        assert call(handle, src, 2, None, int_ptr) == -1
        assert call(handle, src, 2, wn_ptr, None) == -1
        assert lib.rn_md_cross_spectra(handle, src, 2, 0.0, 0, 0.0, 0, 0.0, wn_ptr, int_ptr, stream) == -1
        assert call(handle, src, 2, wn_ptr, int_ptr) == 0  # the same plan runs G = 2
        torch.cuda.synchronize()
        want = rb.measure_cross_spectra([rb.MDRamanSpectrum(alpha[g], 1.0) for g in range(2)])[1]
        assert np.array_equal(inten.cpu().numpy().reshape(-1)[:4 * points].reshape(2, 2, points), want)
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(handle)

"""CPU checks of the drop-in layer around LIVE reference objects (needs /root/reference; skipped on the
GPU box, where tests/test_gpu_install.py drives the same code through a stand-in package):
``ModelState.from_reference`` / ``accelerate`` on models the unmodified reference built, the fingerprint
that re-packs a mutated model, and ``install()`` / ``uninstall()`` of the four patched entry points."""
import os

import numpy as np
import pytest

import ramannoodle_b200 as rb
from oracle.ref_bootstrap import REFERENCE_ROOT, import_reference, reference_available
from ramannoodle_b200 import dropin as rb_install
from ramannoodle_b200 import synthetic
from ramannoodle_b200.exceptions import NativeLibraryError
from ramannoodle_b200.state import ModelState

from helpers import GOLDEN

pytestmark = pytest.mark.skipif(not reference_available(), reason="reference tree not present")


@pytest.fixture(scope="module")
def ref():
    return import_reference()


def _tio2_reference_model(order, art=False):
    """The reference's own construction path on its real TiO2 DFT data (identity symmetry stub)."""
    import warnings

    import ramannoodle.io.generic as generic_io
    from ramannoodle.pmodel._art import ARTModel
    from ramannoodle.pmodel._interpolation import InterpolationModel

    data_dir = os.path.join(REFERENCE_ROOT, "test", "data", "TiO2")
    structure = generic_io.read_ref_structure(f"{data_dir}/phonons_OUTCAR", file_format="outcar")
    _, ref_pol = generic_io.read_positions_and_polarizability(f"{data_dir}/ref_eps_OUTCAR", file_format="outcar")
    model = (ARTModel if art else InterpolationModel)(structure, ref_pol)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for atom in ("Ti5", "O43"):
            for direction in "xyz":
                if art:
                    files = [f"{data_dir}/{atom}_{s}{direction}_eps_OUTCAR" for s in ("0.1", "m0.1")]
                    model.add_art_from_files(files, file_format="outcar")
                else:
                    files = [f"{data_dir}/{atom}_{s}{direction}_eps_OUTCAR" for s in ("0.1", "0.2", "m0.1", "m0.2")]
                    model.add_dof_from_files(files, file_format="outcar", interpolation_order=order)
    return model


@pytest.mark.parametrize("order", [1, 2, 3])
def test_from_reference_on_a_live_model_matches_the_goldens(ref, order):
    """The tables packed from a live reference model equal the ones the committed goldens were made from."""
    model = _tio2_reference_model(order)
    tables = ModelState.from_reference(model).tables()
    with np.load(f"{GOLDEN}/real_tio2.npz") as data:
        for key, value in tables.items():
            assert np.array_equal(value, data[f"k{order}_{key}"]), key
    wrapped = rb.accelerate(model)
    assert type(wrapped) is rb.InterpolationModel and wrapped.num_atoms == 108
    assert wrapped.state.atomic_numbers == [int(z) for z in model._ref_structure.atomic_numbers]  # pylint: disable=protected-access


def test_accelerate_art_model_and_dof_indexes(ref):
    model = _tio2_reference_model(1, art=True)
    wrapped = rb.accelerate(model)
    assert type(wrapped) is rb.ARTModel
    with np.load(f"{GOLDEN}/real_tio2.npz") as data:
        for key, value in wrapped.state.tables().items():
            assert np.array_equal(value, data[f"art_{key}"]), key
    # get_dof_indexes: same answers (and order) as the reference, for indexes, symbols and mixtures
    for query in (5, 43, [5, 43], "Ti", "O", ["Ti", 43], [43, 43, "O"], 0):
        assert wrapped.get_dof_indexes(query) == model.get_dof_indexes(query), query
    masked = wrapped.get_masked_model(wrapped.get_dof_indexes("Ti"))
    assert np.array_equal(masked.mask, model.get_masked_model(model.get_dof_indexes("Ti")).mask)
    with pytest.raises(TypeError, match="atom_symbols should have type list, not int"):
        wrapped.state.get_atom_indexes(5)


def test_live_fingerprint_tracks_every_mutation(ref):
    from scipy.interpolate import make_interp_spline

    model = _tio2_reference_model(1, art=True)
    last = [rb_install.live_fingerprint(model)]
    seen = set(last)

    def changed():  # against the previous state, which is what the cache compares with
        fingerprint = rb_install.live_fingerprint(model)
        fresh = fingerprint != last[0]
        last[0] = fingerprint
        seen.add(fingerprint)
        return fresh

    assert not changed()
    mask = model.mask
    mask[2] = True
    model.mask = mask  # the setter the reference documents (_interpolation.py:174-189)
    assert changed()
    model._mask[3] = True  # pylint: disable=protected-access  (in-place edit of the live array)
    assert changed()
    model.unmask()
    assert changed()
    spline = make_interp_spline(x=[-0.1, 0.1], y=np.zeros((2, 3, 3)), k=1, bc_type=None)
    model._cart_basis_vectors.append(np.zeros((108, 3)))  # pylint: disable=protected-access
    model._interpolations.append(spline)  # pylint: disable=protected-access
    model._mask = np.append(model._mask, False)  # pylint: disable=protected-access
    assert changed()
    model._interpolations[-1] = make_interp_spline(x=[-0.2, 0.2], y=np.ones((2, 3, 3)), k=1, bc_type=None)  # pylint: disable=protected-access
    assert changed()
    model._ref_polarizability = model._ref_polarizability + 1.0  # pylint: disable=protected-access
    assert changed()
    copy = model.get_masked_model([0, 1])  # deep copy: different lists, different mask
    assert rb_install.live_fingerprint(copy) not in seen


def test_accelerated_cache_repacks_after_mutation(ref):
    model = _tio2_reference_model(1, art=True)
    first = rb_install.accelerated(model)
    assert rb_install.accelerated(model) is first
    mask = model.mask
    mask[[1, 4]] = True
    model.mask = mask
    second = rb_install.accelerated(model)
    assert second is not first and np.array_equal(second.mask, mask)
    with np.load(f"{GOLDEN}/real_tio2.npz") as data:
        assert np.array_equal(second.state.tables()["weight"], 1.0 - data["art_masked_mask"])
    clone = model.get_masked_model([0])
    assert rb_install.accelerated(clone) is not second


def test_install_patches_and_restores(ref):
    import torch

    from ramannoodle.dynamics._trajectory import Trajectory
    from ramannoodle.pmodel._art import ARTModel
    from ramannoodle.pmodel._interpolation import InterpolationModel
    from ramannoodle.spectrum import utils
    from ramannoodle.spectrum._raman import MDRamanSpectrum

    originals = (InterpolationModel.calc_polarizabilities, Trajectory.get_raman_spectrum, MDRamanSpectrum.measure,
                 utils.convolve_spectrum)
    patched = rb.install()
    try:
        assert patched == ["ramannoodle.pmodel._interpolation.InterpolationModel.calc_polarizabilities",
                           "ramannoodle.dynamics._trajectory.Trajectory.get_raman_spectrum",
                           "ramannoodle.spectrum._raman.MDRamanSpectrum.measure",
                           "ramannoodle.spectrum.utils.convolve_spectrum"]
        assert InterpolationModel.calc_polarizabilities is not originals[0]
        assert ARTModel.calc_polarizabilities is InterpolationModel.calc_polarizabilities  # inherited
        assert utils.convolve_spectrum is rb.convolve_spectrum
        rb.install()  # idempotent: the originals are remembered once
        if not torch.cuda.is_available():
            # no CPU fallback behind the patched entries either
            model = _tio2_reference_model(1, art=True)
            positions = synthetic.make_trajectory("TiO2", 4)
            with pytest.raises(NativeLibraryError):
                model.calc_polarizabilities(positions)
            with pytest.raises(NativeLibraryError):
                Trajectory(positions, 1.0).get_raman_spectrum(model)
            with pytest.raises(NativeLibraryError):
                MDRamanSpectrum(np.zeros((8, 3, 3)), 1.0).measure()
            # argument errors keep the reference's types and messages
            with pytest.raises(TypeError, match="positions should have type ndarray, not list"):
                model.calc_polarizabilities([1, 2])
            with pytest.raises(ValueError, match=r"positions has wrong shape: \(4,5,3\) != \(_,108,3\)"):
                model.calc_polarizabilities(np.zeros((4, 5, 3)))
            with pytest.raises(ValueError, match="polarizability_model and trajectory are incompatible"):
                Trajectory(np.zeros((4, 5, 3)), 1.0).get_raman_spectrum(model)
    finally:
        rb.uninstall()
    assert (InterpolationModel.calc_polarizabilities, Trajectory.get_raman_spectrum, MDRamanSpectrum.measure,
            utils.convolve_spectrum) == originals

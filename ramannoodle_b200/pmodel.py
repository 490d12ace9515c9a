"""Drop-in evaluators for the reference's ``InterpolationModel`` / ``ARTModel``.

The public method is the reference's plugin entry,
``calc_polarizabilities(positions_batch) -> (S,3,3)`` (``ramannoodle/abstract.py:13-29``,
``ramannoodle/pmodel/_interpolation.py:191-252``) with the same error behaviour.  The entry
BASELINE.json's north_star names, ``get_polarizability(cart_displacements)``, is provided as
well (it starts at ``_interpolation.py:233``).  Model *construction* stays in the
reference: build the model there (``add_dof*``, ``add_art*``), then wrap it with
``InterpolationModel.from_reference(model)`` (or ``ramannoodle_b200.accelerate(model)``).

numpy in -> numpy out; a CUDA ``torch.Tensor`` in -> a CUDA tensor out (no host round trip).
All arithmetic runs in the CUDA library; there is no CPU fallback.
"""
from __future__ import annotations

import copy
import ctypes

import numpy as np

from . import _lib
from .abstract import PolarizabilityModel
from .exceptions import UserError, get_shape_error, get_type_error, verify_ndarray_shape
from .state import ModelState


def _ptr(array: np.ndarray) -> ctypes.c_void_p:
    return ctypes.c_void_p(array.ctypes.data)


class _DeviceModel:
    """Owns one ``rn_model`` handle (``include/ramannoodle_b200.h: rn_model_create``)."""

    def __init__(self, state: ModelState, device: int, force_dense: bool) -> None:
        tables = state.tables()
        self.device = device
        handle = ctypes.c_void_p()
        flags = _lib.RN_MODEL_FORCE_DENSE if force_dense else _lib.RN_MODEL_DEFAULT
        status = _lib.lib().rn_model_create(
            _ptr(state.ref_positions), state.num_atoms, _ptr(state.lattice), _ptr(tables["basis"]),
            state.num_dofs, _ptr(tables["degree"]), _ptr(tables["knot_off"]), _ptr(tables["knots"]),
            _ptr(tables["coef_off"]), _ptr(tables["coefs"]), _ptr(tables["weight"]),
            _ptr(state.ref_polarizability), device, flags, ctypes.byref(handle))
        _lib.check(status, "rn_model_create")
        self.handle = handle
        info = (ctypes.c_int64 * 8)()
        _lib.check(_lib.lib().rn_model_info(self.handle, info), "rn_model_info")
        self.info = {"num_atoms": info[0], "num_dofs": info[1], "affine_dofs": info[2], "dense_dofs": info[3],
                     "dense_degree": info[4], "device": info[5], "tma_affine": bool(info[6]),
                     "dense_max_pieces": info[7]}

    def close(self) -> None:
        if getattr(self, "handle", None):
            _lib.lib().rn_model_destroy(self.handle)
            self.handle = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass


class InterpolationModel(PolarizabilityModel):
    """GPU evaluator holding the state of a reference ``InterpolationModel``.

    Parameters
    ----------
    state
        The evaluation state (see ``ModelState``).
    device
        CUDA device index; defaults to torch's current device.
    force_dense
        Evaluate linear DOFs through the dense DMMA projection too (no affine collapse).
    """

    def __init__(self, state: ModelState, device: int | None = None, force_dense: bool = False) -> None:
        self._state = state
        self._device = device
        self._force_dense = bool(force_dense)
        self._native: _DeviceModel | None = None
        self._native_key = None

    # -- construction -------------------------------------------------------------------
    @classmethod
    def from_reference(cls, model, device: int | None = None, force_dense: bool = False):
        """Wrap a model built with the reference package (state is snapshotted)."""
        return cls(ModelState.from_reference(model), device=device, force_dense=force_dense)

    # -- mirrored properties (``_interpolation.py:117-189``) ------------------------------
    @property
    def state(self) -> ModelState:
        return self._state

    @property
    def num_atoms(self) -> int:
        return self._state.num_atoms

    @property
    def ref_polarizability(self) -> np.ndarray:
        return self._state.ref_polarizability.copy()

    @property
    def is_dummy_model(self) -> bool:
        return self._state.is_dummy_model

    @property
    def cart_basis_vectors(self) -> list:
        return copy.deepcopy(self._state.basis_vectors)

    @property
    def mask(self) -> np.ndarray:
        return self._state.mask.copy()

    @mask.setter
    def mask(self, value) -> None:
        verify_ndarray_shape("mask", value, self._state.mask.shape)
        self._state.mask = np.asarray(value, dtype=bool)

    def unmask(self) -> None:
        """``_interpolation.py:710-712``."""
        self._state.mask = np.zeros(self._state.mask.shape, dtype=bool)

    def get_masked_model(self, dof_indexes_to_mask):
        """``_interpolation.py:697-708``: a copy with the given DOFs masked."""
        result = copy.deepcopy(self)
        new_mask = result.mask
        new_mask[:] = False
        new_mask[dof_indexes_to_mask] = True
        result.mask = new_mask
        return result

    def calc_polarizabilities_masked(self, positions_batch, masks, to_device: bool = False):
        """Polarizabilities ``(G,S,3,3)`` of this model under each of the ``G`` masks (rows of a
        ``(G,J)`` bool array; True = DOF masked, as the ``mask`` property) in one pass over
        ``positions_batch`` — what evaluating ``G`` ``get_masked_model`` copies returns."""
        masks = np.asarray(masks)
        if masks.ndim != 2 or masks.shape[1] != self._state.mask.shape[0]:
            raise get_shape_error("masks", masks, f"(_,{self._state.mask.shape[0]})")
        copies = []
        for row in masks:
            clone = copy.deepcopy(self)
            clone.mask = np.asarray(row, dtype=bool)
            copies.append(clone)
        return calc_polarizabilities_sweep(copies, positions_batch, to_device=to_device)

    def __deepcopy__(self, memo):
        clone = type(self)(copy.deepcopy(self._state, memo), device=self._device, force_dense=self._force_dense)
        return clone

    def path_info(self) -> dict:
        """Which kernels this model runs through (affine collapse / dense projection)."""
        return dict(self._native_model().info)

    # -- native handle --------------------------------------------------------------------
    def _resolve_device(self, tensor=None) -> int:
        if tensor is not None:
            return int(tensor.device.index if tensor.device.index is not None else 0)
        if self._device is not None:
            return int(self._device)
        try:
            import torch  # pylint: disable=import-outside-toplevel

            if torch.cuda.is_available():
                return int(torch.cuda.current_device())
        except ImportError:
            pass
        return 0

    def _native_model(self, device: int | None = None) -> _DeviceModel:
        if device is None:
            device = self._resolve_device()
        key = (device, self._state.fingerprint())
        if self._native is None or self._native_key != key:
            _lib.require_device(device)
            if self._native is not None:
                self._native.close()
            self._native = _DeviceModel(self._state, device, self._force_dense)
            self._native_key = key
        return self._native

    # -- evaluation -----------------------------------------------------------------------
    def _check_dummy(self) -> None:
        # zip(..., strict=True) over unequal lists raises ValueError in the reference, which a
        # dummy model reports as UserError (_interpolation.py:245-250; test_art.py:367-369)
        if len(self._state.splines) != len(self._state.basis_vectors):
            if self._state.is_dummy_model:
                raise UserError("dummy model cannot calculate polarizabilities")
            raise ValueError("basis vectors and interpolations have different lengths")

    def calc_polarizabilities(self, positions_batch):
        """Return polarizabilities (S,3,3) for fractional positions (S,N,3)."""
        if _lib.is_torch_tensor(positions_batch):
            return self._eval_tensor(positions_batch, wrap=True, name="positions")
        _, positions, device, _ = _eval_inputs([self], positions_batch)
        alpha = np.empty((positions.shape[0], 3, 3), dtype=np.float64)
        native = self._native_model(device)
        status = _lib.lib().rn_calc_polarizabilities_host(native.handle, _ptr(positions), positions.shape[0],
                                                          _ptr(alpha), None, 0)
        _lib.check(status, "rn_calc_polarizabilities_host")
        return alpha

    def calc_polarizabilities_to_device(self, positions_batch: np.ndarray):
        """Host positions in, polarizabilities left on the GPU (a CUDA tensor): the path
        ``Trajectory.get_raman_spectrum`` uses so the series never round-trips to the host."""
        import torch  # pylint: disable=import-outside-toplevel

        if not isinstance(positions_batch, np.ndarray):
            raise get_type_error("positions", positions_batch, "ndarray")
        _, positions, device, _ = _eval_inputs([self], positions_batch)
        native = self._native_model(device)
        alpha = torch.empty((positions.shape[0], 3, 3), dtype=torch.float64, device=f"cuda:{device}")
        torch.cuda.synchronize(device)
        status = _lib.lib().rn_calc_polarizabilities_host(native.handle, _ptr(positions), positions.shape[0], None,
                                                          ctypes.c_void_p(alpha.data_ptr()), 0)
        _lib.check(status, "rn_calc_polarizabilities_host")
        return alpha

    def calc_polarizabilities_multi(self, positions_batch, output_ptrs) -> None:
        """Evaluate ``positions_batch`` (numpy, streamed from the host, or a CUDA tensor) and store
        the (S,3,3) rows to every device pointer in ``output_ptrs`` (ints): ``output_ptrs[0]`` is
        the local series, the others the same buffer on peer GPUs (symmetric memory over NVLink),
        all pre-offset to this rank's first frame.  The kernels write the peers' rows themselves —
        the all-gather is fused into the evaluation (``rn_calc_polarizabilities_multi``)."""
        count = len(output_ptrs)
        if not 1 <= count <= 8:
            raise ValueError("between 1 and 8 output pointers are required")
        outputs = (ctypes.c_void_p * count)(*[ctypes.c_void_p(int(ptr)) for ptr in output_ptrs])
        _, positions, device, is_tensor = _eval_inputs([self], positions_batch)
        native = self._native_model(device)
        if is_tensor:
            import torch  # pylint: disable=import-outside-toplevel

            with torch.cuda.device(device):
                status = _lib.lib().rn_calc_polarizabilities_multi(
                    native.handle, ctypes.c_void_p(positions.data_ptr()), int(positions.shape[0]), outputs, count,
                    _lib.current_stream(device))
            _lib.check(status, "rn_calc_polarizabilities_multi")
            return
        # the pipeline's private streams start after the work already enqueued on the current stream
        # (e.g. the cross-rank barrier in front of this call)
        status = _lib.lib().rn_calc_polarizabilities_host_multi(native.handle, _ptr(positions), positions.shape[0],
                                                                outputs, count, 0, _lib.current_stream(device))
        _lib.check(status, "rn_calc_polarizabilities_host_multi")

    # pylint: disable=too-many-arguments,too-many-positional-arguments
    def routed_phases_supported(self, positions_batch, first_frame: int, stripe: int) -> bool:
        """Whether ``calc_polarizabilities_routed(..., stripe=stripe, phase=0|1)`` can evaluate this block
        (``rn_routed_phases_supported``: a purely linear model on the TMA path, HBM-resident 16-byte aligned
        rows, block bounds on multiples of 16 frames)."""
        if stripe <= 0 or not _lib.is_torch_tensor(positions_batch) or not positions_batch.is_cuda:
            return False
        import torch  # pylint: disable=import-outside-toplevel

        if positions_batch.dtype != torch.float64 or not positions_batch.is_contiguous() or self.is_dummy_model:
            return False
        native = self._native_model(self._resolve_device(positions_batch))
        return bool(_lib.lib().rn_routed_phases_supported(native.handle, ctypes.c_void_p(positions_batch.data_ptr()),
                                                          int(positions_batch.shape[0]), int(first_frame), int(stripe)))

    def calc_polarizabilities_routed(self, positions_batch, local_ptr: int, peer_series, first_frame: int,
                                     period: int, width: int, stripe: int = 0, phase: int = -1) -> None:
        """Evaluate this rank's block and route the rows for the shared multi-GPU spectrum
        (``rn_calc_polarizabilities_routed``): rows go to ``local_ptr`` (this rank's block inside its own
        full series buffer) and, written by the kernels over NVLink, to the series buffers
        ``peer_series[r]`` (base pointers, 0 for this rank) of the ranks whose spectrum stage consumes them —
        row ``n`` to ranks ``(n % period) // width`` and ``((n - 1) % period) // width``.
        ``phase`` 0 / 1 (with ``stripe``; CUDA tensors only, ``routed_phases_supported``): one half of the
        pipelined schedule, ``rn_calc_polarizabilities_routed_phase``."""
        world = len(peer_series)
        if not 1 <= world <= 8:
            raise ValueError("between 1 and 8 ranks")
        peers = (ctypes.c_void_p * world)(*[ctypes.c_void_p(int(ptr)) if ptr else None for ptr in peer_series])
        if phase >= 0 and not _lib.is_torch_tensor(positions_batch):
            raise ValueError("phased evaluation needs an HBM-resident trajectory block")
        _, positions, device, is_tensor = _eval_inputs([self], positions_batch)
        native = self._native_model(device)
        routing = (ctypes.c_void_p(int(local_ptr)), peers, world, int(first_frame), int(period), int(width))
        if not is_tensor:
            status = _lib.lib().rn_calc_polarizabilities_host_routed(
                native.handle, _ptr(positions), positions.shape[0], *routing, 0, _lib.current_stream(device))
            _lib.check(status, "rn_calc_polarizabilities_host_routed")
            return
        import torch  # pylint: disable=import-outside-toplevel

        data, num_frames = ctypes.c_void_p(positions.data_ptr()), int(positions.shape[0])
        with torch.cuda.device(device):
            if phase >= 0:
                status = _lib.lib().rn_calc_polarizabilities_routed_phase(
                    native.handle, data, num_frames, *routing, int(stripe), int(phase), _lib.current_stream(device))
            else:
                status = _lib.lib().rn_calc_polarizabilities_routed(native.handle, data, num_frames, *routing,
                                                                    _lib.current_stream(device))
        _lib.check(status, "rn_calc_polarizabilities_routed")

    def get_polarizability(self, cart_displacements):
        """Polarizabilities from precomputed Cartesian displacements (S,N,3) or (S,3N) in Å
        (what ``_interpolation.py:217-223`` produces)."""
        if _lib.is_torch_tensor(cart_displacements):
            return self._eval_tensor(cart_displacements, wrap=False, name="cart_displacements")
        if not isinstance(cart_displacements, np.ndarray):
            raise get_type_error("cart_displacements", cart_displacements, "ndarray")
        import torch  # pylint: disable=import-outside-toplevel

        device = self._resolve_device()
        _lib.require_device(device)
        tensor = torch.from_numpy(np.ascontiguousarray(cart_displacements, dtype=np.float64)).to(f"cuda:{device}")
        return self._eval_tensor(tensor, wrap=False, name="cart_displacements").cpu().numpy()

    def _eval_tensor(self, tensor, wrap: bool, name: str):
        import torch  # pylint: disable=import-outside-toplevel

        _, data, device, _ = _eval_inputs([self], tensor, name=name, flat=not wrap)
        native = self._native_model(device)
        num_frames = int(data.shape[0])
        with torch.cuda.device(device):
            alpha = torch.empty((num_frames, 3, 3), dtype=torch.float64, device=data.device)
            entry = _lib.lib().rn_calc_polarizabilities if wrap else _lib.lib().rn_get_polarizability
            status = entry(native.handle, ctypes.c_void_p(data.data_ptr()), num_frames,
                           ctypes.c_void_p(alpha.data_ptr()), _lib.current_stream(device))
        _lib.check(status, "rn_calc_polarizabilities" if wrap else "rn_get_polarizability")
        return alpha


def _eval_inputs(models, positions_batch, name: str = "positions", flat: bool = False):
    """Validated inputs of an evaluation of ``models`` (one structure; one model, or the models of a sweep) on
    ``positions_batch``: (models, contiguous float64 positions, device, is_tensor).

    Checks, before any device work and in this order: the models, the type (ndarray or CUDA tensor), the
    shape (S,N,3) (``flat``: (S,3N) as well), dummy models.  The device is the tensor's, or for numpy input
    the one ``models[0]`` resolves."""
    models = list(models)
    if len(models) == 0:
        raise ValueError("at least one model is required")
    if len(models) > 64:
        raise ValueError("at most 64 models per sweep")
    for model in models:
        if not isinstance(model, InterpolationModel):
            raise get_type_error("models", model, "InterpolationModel")
    num_atoms = models[0].num_atoms
    if any(model.num_atoms != num_atoms for model in models):
        raise ValueError("models of a sweep must describe the same structure")
    is_tensor = _lib.is_torch_tensor(positions_batch)
    if is_tensor:
        if not positions_batch.is_cuda:
            raise get_type_error(name, positions_batch, "ndarray or CUDA tensor")
    elif not isinstance(positions_batch, np.ndarray):
        raise get_type_error(name, positions_batch, "ndarray")
    shape = tuple(positions_batch.shape)
    if not (len(shape) == 3 and shape[1:] == (num_atoms, 3)) and not (
            flat and len(shape) == 2 and shape[1] == 3 * num_atoms):
        raise get_shape_error(name, positions_batch, f"(_,{num_atoms},3)")
    for model in models:
        model._check_dummy()  # pylint: disable=protected-access
    if is_tensor:
        import torch  # pylint: disable=import-outside-toplevel

        data = positions_batch.to(torch.float64).contiguous()
        device = models[0]._resolve_device(data)  # pylint: disable=protected-access
    else:
        data = np.ascontiguousarray(positions_batch, dtype=np.float64)
        device = models[0]._resolve_device()  # pylint: disable=protected-access
    return models, data, device, is_tensor


def calc_polarizabilities_sweep(models, positions_batch, to_device: bool = False):
    """Evaluate several models of ONE structure (typically ``get_masked_model`` copies,
    ``_interpolation.py:697-708``) on the same positions in one pass: returns ``(G,S,3,3)``.

    A host trajectory crosses PCIe once; purely linear models (every ``ARTModel``) are contracted
    together by one kernel (``rn_calc_polarizabilities_sweep``), other models run one after the other
    on the resident positions.  Each slice equals ``models[g].calc_polarizabilities(positions_batch)``.
    numpy in -> numpy out (a CUDA tensor if ``to_device``); CUDA tensor in -> CUDA tensor out."""
    import torch  # pylint: disable=import-outside-toplevel

    models, data, device, is_tensor = _eval_inputs(models, positions_batch)
    count = len(models)
    num_frames = int(data.shape[0])
    natives = [model._native_model(device) for model in models]  # pylint: disable=protected-access
    handles = (ctypes.c_void_p * count)(*[native.handle for native in natives])
    with torch.cuda.device(device):
        alpha = torch.empty((count, num_frames, 3, 3), dtype=torch.float64, device=f"cuda:{device}")
        if num_frames == 0:
            return alpha if (is_tensor or to_device) else alpha.cpu().numpy()
        outputs = (ctypes.c_void_p * count)(*[ctypes.c_void_p(alpha[g].data_ptr()) for g in range(count)])
        if is_tensor:
            status = _lib.lib().rn_calc_polarizabilities_sweep(handles, count, ctypes.c_void_p(data.data_ptr()),
                                                               num_frames, outputs, _lib.current_stream(device))
            _lib.check(status, "rn_calc_polarizabilities_sweep")
            return alpha
        torch.cuda.synchronize(device)
        status = _lib.lib().rn_calc_polarizabilities_host_sweep(handles, count, _ptr(data), num_frames, outputs, 0)
        _lib.check(status, "rn_calc_polarizabilities_host_sweep")
    return alpha if to_device else alpha.cpu().numpy()


# pylint: disable=too-many-arguments,too-many-positional-arguments,too-many-locals
def calc_polarizabilities_sweep_routed(models, positions_batch, local_ptrs, peer_series, first_frame: int,
                                       period: int, width: int, chunk_frames: int = 0) -> None:
    """Mask sweep of this rank's block for the shared multi-GPU spectrum
    (``rn_calc_polarizabilities_sweep_routed``): model g's rows go to ``local_ptrs[g]`` (this rank's block
    inside its own series buffer of mask g) and, written by the kernels over NVLink, to
    ``peer_series[g][r]`` (base pointers of mask g's series buffer on rank r, 0 for this rank) for the
    ranks that consume them, as in ``InterpolationModel.calc_polarizabilities_routed``.  A host block
    crosses PCIe once for all models (in chunks of ``chunk_frames``, 0 = automatic)."""
    import torch  # pylint: disable=import-outside-toplevel

    models, data, device, is_tensor = _eval_inputs(models, positions_batch)
    count = len(models)
    if len(local_ptrs) != count or len(peer_series) != count:
        raise ValueError("one local pointer and one row of peer pointers per model are required")
    world = len(peer_series[0])
    if not 1 <= world <= 8 or any(len(row) != world for row in peer_series):
        raise ValueError("between 1 and 8 ranks, the same number for every model")
    natives = [model._native_model(device) for model in models]  # pylint: disable=protected-access
    handles = (ctypes.c_void_p * count)(*[native.handle for native in natives])
    outputs = (ctypes.c_void_p * count)(*[ctypes.c_void_p(int(ptr)) for ptr in local_ptrs])
    peers = (ctypes.c_void_p * (count * world))(*[ctypes.c_void_p(int(ptr)) if ptr else None
                                                  for row in peer_series for ptr in row])
    num_frames = int(data.shape[0])
    with torch.cuda.device(device):
        stream = _lib.current_stream(device)
        if is_tensor:
            status = _lib.lib().rn_calc_polarizabilities_sweep_routed(
                handles, count, ctypes.c_void_p(data.data_ptr()), num_frames, outputs, peers, world, int(first_frame),
                int(period), int(width), stream)
        else:
            status = _lib.lib().rn_calc_polarizabilities_host_sweep_routed(
                handles, count, _ptr(data), num_frames, outputs, peers, world, int(first_frame), int(period),
                int(width), int(chunk_frames), stream)
    _lib.check(status, "rn_calc_polarizabilities_sweep_routed")


class ARTModel(InterpolationModel):
    """Atomic-Raman-tensor model (``ramannoodle/pmodel/_art.py:48``): evaluation is inherited
    unchanged; every DOF is one linear piece, so it runs through the affine kernel."""

    def get_dof_indexes(self, atom_indexes_or_symbols) -> list:
        """DOF indexes of certain atoms (``ramannoodle/pmodel/_art.py:335-365``): integers are atom
        indexes, strings atom symbols (mixtures allowed).  A DOF belongs to an atom when its basis
        vector moves that atom (``not np.allclose(direction, 0, atol=1e-5)``); the result keeps the
        reference's order (atoms in ``set`` order, DOFs ascending) so that
        ``get_masked_model(get_dof_indexes("Ti"))`` reads like the masking tutorial."""
        if not isinstance(atom_indexes_or_symbols, list):
            atom_indexes_or_symbols = [atom_indexes_or_symbols]
        atom_indexes = []
        for item in atom_indexes_or_symbols:
            if isinstance(item, str):
                atom_indexes += self._state.get_atom_indexes(item)
            else:
                atom_indexes += [item]
        atom_indexes = list(set(atom_indexes))
        if not self._state.basis_vectors:
            return []
        basis = np.stack([np.asarray(v, dtype=np.float64).reshape(self.num_atoms, 3) for v in self._state.basis_vectors])
        moves = ~np.all(np.abs(basis) <= 1e-5, axis=2)  # (J,N): allclose(direction, 0, atol=1e-5, rtol irrelevant at 0)
        dof_indexes = []
        for atom_index in atom_indexes:
            dof_indexes += [int(j) for j in np.nonzero(moves[:, atom_index])[0]]
        return dof_indexes


def accelerate(model, device: int | None = None, force_dense: bool = False) -> InterpolationModel:
    """Wrap a reference ``InterpolationModel``/``ARTModel`` for GPU evaluation.  The state is
    SNAPSHOTTED: later changes to the reference object (``add_dof``, ``mask = ...``) are not seen —
    wrap again, or use ``ramannoodle_b200.install()``, which tracks the live object."""
    cls = ARTModel if type(model).__name__ == "ARTModel" else InterpolationModel
    return cls.from_reference(model, device=device, force_dense=force_dense)

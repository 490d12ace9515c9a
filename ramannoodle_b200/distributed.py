"""Frame sharding across GPUs (one process per GPU, ``torch.distributed``).

``calc_polarizabilities`` has no cross-frame term, so frames shard naturally: rank r evaluates the
contiguous block ``shard_bounds(S, G, r)`` with the model tables replicated
(``ramannoodle/pmodel/_interpolation.py:191-252``).  ``MDRamanSpectrum.measure``
(``ramannoodle/spectrum/_raman.py:241-309``) is global in S; here its single chirp-z transform is
SHARED by the ranks (decimation in frequency at rank level, ``csrc/rn_spectrum.cu``):

1. the evaluation kernels store every row of the (S,3,3) series straight to the rank whose spectrum
   stage consumes it (peer stores over NVLink into symmetric memory; every row has one or two
   destinations, so the series is never all-gathered).  Optionally (RN_DIST_OVERLAP=1, off by default: measured
   slower) HBM-resident blocks of purely linear models are evaluated in two launches — first the frames the
   first half of every rank's pack reads — with that half of the pack on a second stream under the second launch;
2. ``pack`` (np.diff, signal packing, chirp, G-point DFT over the blocks) stores residue r into rank
   r's work buffer; 3. every rank runs its local length-L/G convolution and stores the result to the
   ranks owning the output residues (mirror-symmetric ownership: the owner of bin m also owns bin M - m);
   4. ``final`` finishes the intensities of its bin pairs and stores them to every rank; 5. every rank copies
   them out (``finish``).  Device-side barriers separate the steps; there is no
   NCCL collective on the path.  ``polarizability_ts`` all-gathers the series lazily when read.

Without symmetric memory (CPU tensors, gloo, other backends) the local block is evaluated, one
``all_gather_into_tensor`` assembles the series and every rank runs the single-GPU ``measure``.
"""
from __future__ import annotations

import ctypes
import os
import warnings

from . import _lib
from .abstract import Dynamics
from .dynamics import Trajectory
from .spectrum import MDRamanSpectrum, _check_measure_args, _check_window_args, _measure_windows


def shard_bounds(num_frames: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous block [start, stop) of rank ``rank``: blocks of ceil(S/G) frames."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("invalid rank/world_size")
    block = -(-num_frames // world_size)
    start = min(rank * block, num_frames)
    return start, min(start + block, num_frames)


def transform_group_size(world_size: int) -> int:
    """Ranks that share the chirp-z transform: the largest power of two <= min(world, 8); the other
    ranks evaluate their frames and receive the spectrum."""
    if world_size < 1:
        raise ValueError("invalid world_size")
    group = 1
    while group * 2 <= min(world_size, 8):
        group *= 2
    return group


def route_owner(frame: int, period: int, width: int) -> int:
    """Rank whose ``pack`` stage consumes difference signal ``frame`` (it needs rows ``frame`` and
    ``frame + 1`` of the series): ``include/ramannoodle_b200.h: rn_spectrum_dist_route``."""
    return (frame % period) // width


def allgather_series(local_series, num_frames: int, group=None):
    """All-gather per-rank (S_r,3,3) blocks into the full (S,3,3) series on every rank.

    One collective: blocks are padded to ceil(S/G) frames so a single
    ``all_gather_into_tensor`` (NCCL over NVLink on GPUs, gloo in CPU tests) suffices; the
    padding of the tail rank is dropped afterwards.
    """
    import torch  # pylint: disable=import-outside-toplevel
    import torch.distributed as dist  # pylint: disable=import-outside-toplevel

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    block = -(-num_frames // world)
    start, stop = shard_bounds(num_frames, world, rank)
    if tuple(local_series.shape) != (stop - start, 3, 3):
        raise ValueError(f"rank {rank}: local series has shape {tuple(local_series.shape)}, "
                         f"expected {(stop - start, 3, 3)}")
    if world == 1:
        return local_series
    padded = local_series
    if stop - start != block:
        padded = torch.zeros((block, 3, 3), dtype=local_series.dtype, device=local_series.device)
        padded[: stop - start] = local_series
    full = torch.empty((world * block, 3, 3), dtype=local_series.dtype, device=local_series.device)
    dist.all_gather_into_tensor(full, padded.contiguous(), group=group)
    return full[:num_frames]


class SymmetricMemoryUnavailable(RuntimeError):
    """Symmetric memory (peer-mapped buffers over NVLink) cannot be used by this process group."""


_UNAVAILABLE_WARNED = False


def _all_ranks_agree(ok: bool, device, group) -> bool:
    """True only if ``ok`` holds on every rank (a rank-local failure must not split the ranks between
    two different collective schedules)."""
    import torch  # pylint: disable=import-outside-toplevel
    import torch.distributed as dist  # pylint: disable=import-outside-toplevel

    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    return bool(int(flag.item()))


class _SharedContext:
    """Everything the shared spectrum of one (S, device, group) needs: the dist plan and ONE symmetric
    allocation holding this rank's full-layout series buffers, work buffer, receive buffer and power
    buffer (cached: allocation and rendezvous are collectives).

    ``slots`` series buffers of ``align(S*72)`` bytes each lie at the start of the allocation, one per
    model of a mask sweep (``ShardedTrajectory.get_raman_spectra``); the work, receive and power buffers
    are shared by all slots: the spectra of the slots are measured one after the other on one stream,
    with barriers between the steps, like two ``measure()`` calls on one spectrum."""

    def __init__(self, num_frames: int, device, group, slots: int = 1) -> None:
        import torch  # pylint: disable=import-outside-toplevel
        import torch.distributed as dist  # pylint: disable=import-outside-toplevel

        self.num_frames = int(num_frames)
        self.slots = int(slots)
        self.device = device
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        index = int(device.index if device.index is not None else torch.cuda.current_device())
        lib = _lib.lib()
        handle = ctypes.c_void_p()
        _lib.check(lib.rn_spectrum_plan_create_dist(self.num_frames, index, self.world, self.rank, ctypes.byref(handle)),
                   "rn_spectrum_plan_create_dist")
        self.plan = handle
        sizes = [ctypes.c_int64() for _ in range(3)]
        _lib.check(lib.rn_spectrum_dist_sizes(self.plan, *[ctypes.byref(v) for v in sizes]), "rn_spectrum_dist_sizes")
        period, width = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(lib.rn_spectrum_dist_route(self.plan, ctypes.byref(period), ctypes.byref(width)),
                   "rn_spectrum_dist_route")
        self.period, self.width = int(period.value), int(width.value)
        self.transform_ranks = self.period // self.width
        stripe = ctypes.c_int64()
        _lib.check(lib.rn_spectrum_dist_stripe(self.plan, ctypes.byref(stripe)), "rn_spectrum_dist_stripe")
        self.stripe = int(stripe.value)
        self.phased = {}             # (model id, block pointer) -> every rank can evaluate in two phases
        self.packed_generation = -1  # generation whose first pack half is already running on the side stream
        self.pack_event = None

        def align(nbytes: int) -> int:
            return (nbytes + 255) // 256 * 256

        self.series_bytes = align(self.num_frames * 72)
        series_bytes = self.slots * self.series_bytes
        self.offsets = {"series": 0, "work": series_bytes, "recv": series_bytes + align(sizes[0].value),
                        "spectrum": series_bytes + align(sizes[0].value) + align(sizes[1].value)}
        total = self.offsets["spectrum"] + align(sizes[2].value)
        pg = group if group is not None else dist.group.WORLD
        ok = True
        self.buffer = self.handle = None
        try:
            import torch.distributed._symmetric_memory as symm_mem  # pylint: disable=import-outside-toplevel

            self.buffer = symm_mem.empty(total // 8, dtype=torch.float64, device=device)
            self.handle = symm_mem.rendezvous(self.buffer, group=pg.group_name)
        except (RuntimeError, ImportError, AttributeError, NotImplementedError) as exc:
            ok = False
            self.error = exc
        if not _all_ranks_agree(ok, device, group):
            self.close()
            raise SymmetricMemoryUnavailable(str(getattr(self, "error", "another rank could not allocate symmetric memory")))
        self.generation = 0
        self._side_streams = None
        # RN_DIST_OVERLAP=1: evaluate in two launches and run the first half of the pack (NVLink-bound) on a
        # second stream under the second launch (HBM-bound), module docstring step 1.  Measured on 4 x B200
        # (1M LLZO frames per GPU): the spectrum stage drops from 0.445 to 0.394 ms as intended, but the
        # evaluation in two launches with a barrier between them costs 0.94 instead of 0.85 ms — 1.322 against
        # 1.281 ms per step, whichever kernel is enqueued first — so it is off by default.
        self.overlap = os.environ.get("RN_DIST_OVERLAP", "0") == "1"
        # RN_DIST_PIPELINE=1: one stream per packed sequence (pack -> barrier -> convolution), so that the
        # NVLink-bound stores of one sequence can overlap the FP64-bound passes of another.  Measured on
        # 4 x B200 (1M frames per GPU): 1.254 ms/step against 1.262 ms with one launch for the three
        # sequences — the per-sequence launches fill the SMs worse (512 tiles = 1.15 waves) and need two
        # more barriers, which eats the overlap; off by default.
        self.pipeline = os.environ.get("RN_DIST_PIPELINE", "0") == "1"
        self.local_base = int(self.buffer.data_ptr())
        self.peer_bases = [int(self.handle.buffer_ptrs[r]) for r in range(self.world)]

    def ptr(self, rank: int, name: str, slot: int = 0) -> int:
        return self.peer_bases[rank] + self.offsets[name] + (slot * self.series_bytes if name == "series" else 0)

    def table(self, name: str, count: int):
        return (ctypes.c_void_p * count)(*[ctypes.c_void_p(self.ptr(r, name)) for r in range(count)])

    def series_view(self, start: int, stop: int, slot: int = 0):
        """This rank's rows [start, stop) of its own series buffer ``slot`` as a (n,3,3) tensor."""
        base = slot * self.series_bytes // 8
        return self.buffer[base + start * 9: base + stop * 9].view(stop - start, 3, 3)

    def barrier(self, channel: int = 0) -> None:
        self.handle.barrier(channel=channel)

    def side_streams(self, device):
        """Two extra streams (high priority: their pack kernels should get SMs as soon as some free up)."""
        import torch  # pylint: disable=import-outside-toplevel

        if self._side_streams is None:
            self._side_streams = [torch.cuda.Stream(device=device, priority=-1) for _ in range(2)]
        return self._side_streams

    def pack_stream(self, device):
        """The stream of the overlapped first pack half (default priority, see ShardedTrajectory)."""
        import torch  # pylint: disable=import-outside-toplevel

        if getattr(self, "_pack_stream", None) is None:
            self._pack_stream = torch.cuda.Stream(device=device)
        return self._pack_stream

    def close(self) -> None:
        if getattr(self, "plan", None):
            _lib.lib().rn_spectrum_plan_destroy(self.plan)
            self.plan = None

    def __del__(self) -> None:
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass


_SHARED: dict = {}


def _shared_context(num_frames: int, device, group, slots: int = 1):
    """The cached ``_SharedContext`` with at least ``slots`` series buffers, or None if symmetric memory is
    unavailable (every rank agrees)."""
    import torch.distributed as dist  # pylint: disable=import-outside-toplevel

    global _UNAVAILABLE_WARNED  # pylint: disable=global-statement
    pg = group if group is not None else dist.group.WORLD
    key = (int(num_frames), str(device), pg.group_name)
    if key in _SHARED and (_SHARED[key] is None or _SHARED[key].slots >= slots):
        return _SHARED[key]
    try:
        ctx = _SharedContext(num_frames, device, group, slots)
    except SymmetricMemoryUnavailable as exc:
        if not _UNAVAILABLE_WARNED:
            warnings.warn(f"symmetric memory unavailable ({exc}); using the all-gather path", RuntimeWarning)
            _UNAVAILABLE_WARNED = True
        ctx = None
    _SHARED.clear()  # one live context: its buffers are as large as the series
    _SHARED[key] = ctx
    return ctx


def clear_shared_contexts() -> None:
    for ctx in _SHARED.values():
        if ctx is not None:
            ctx.close()
    _SHARED.clear()


class ShardedMDRamanSpectrum(MDRamanSpectrum):
    """``MDRamanSpectrum`` of a frame-sharded series.

    With a shared context (NCCL group + symmetric memory) the rows sit where the shared transform
    needs them and ``measure`` runs steps 2-5 of the module docstring; ``polarizability_ts`` gathers
    the series on first access.  Otherwise every rank holds the whole series (all-gather path) and
    ``measure`` is the single-GPU one.
    """

    def __init__(self, polarizability_ts, timestep: float, group=None, context=None, generation: int = 0,
                 bounds=None, slot: int = 0):
        if context is None:
            super().__init__(polarizability_ts, timestep)
        else:  # the local block only; the full series is assembled on demand
            self._polarizability_ts = None
            self._timestep = timestep
        self._group = group
        self._context = context
        self._generation = generation
        self._bounds = bounds
        self._slot = slot

    def _check_live(self) -> None:
        if self._context.generation != self._generation:
            raise RuntimeError("the shared series buffer was overwritten by a later get_raman_spectrum() call; "
                               "measure() / polarizability_ts must be used before evaluating again")

    @property
    def local_polarizability_ts(self):
        """This rank's (S_r,3,3) block of the series (a CUDA tensor)."""
        if self._context is None:
            start, stop = self._bounds if self._bounds else (0, len(self._polarizability_ts))
            return self._polarizability_ts[start:stop]
        self._check_live()
        return self._context.series_view(*self._bounds, self._slot)

    def _gathered(self):
        if self._polarizability_ts is None:
            self._check_live()
            self._polarizability_ts = allgather_series(self.local_polarizability_ts, self._context.num_frames,
                                                       self._group).clone()
        return self._polarizability_ts

    def _num_frames(self) -> int:
        return int(self._context.num_frames) if self._context is not None else super()._num_frames()

    def _device_series(self):
        """The whole series on this rank's GPU (with a shared context: gathered, a collective on first use)."""
        return self._gathered() if self._context is not None else super()._device_series()

    @property
    def polarizability_ts(self):
        """The whole (S,3,3) series as numpy (a collective on first access: every rank must read it)."""
        if self._context is not None:
            return self._gathered().cpu().numpy()
        return MDRamanSpectrum.polarizability_ts.fget(self)

    # pylint: disable=too-many-arguments,too-many-positional-arguments
    def measure_windows_device(self, window_frames, hop_frames=None, orientation="polycrystalline",
                               laser_correction=False, laser_wavelength=522, bose_einstein_correction=False,
                               temperature=300):
        """``MDRamanSpectrum.measure_windows_device`` of the whole series; every rank returns all W rows.

        With a shared context the series is first assembled on every rank (an all-gather on first use, as
        for ``polarizability_ts``): every rank of the group must call it.  The windows then run on the
        local GPU."""
        if self._context is None:
            return super().measure_windows_device(window_frames, hop_frames, orientation, laser_correction,
                                                  laser_wavelength, bose_einstein_correction, temperature)
        hop = _check_window_args(window_frames, hop_frames, int(self._context.num_frames))
        _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction, temperature)
        return _measure_windows(self._gathered(), self._timestep, int(window_frames), hop, laser_correction,
                                laser_wavelength, bose_einstein_correction, temperature)

    # pylint: disable=too-many-arguments,too-many-positional-arguments,too-many-locals
    def measure_device(self, orientation="polycrystalline", laser_correction=False, laser_wavelength=522,
                       bose_einstein_correction=False, temperature=300):
        import torch  # pylint: disable=import-outside-toplevel

        if self._context is None:
            return super().measure_device(orientation, laser_correction, laser_wavelength,
                                          bose_einstein_correction, temperature)
        _check_measure_args(orientation, laser_correction, laser_wavelength, bose_einstein_correction, temperature)
        ctx = self._context
        self._check_live()
        if ctx.num_frames < 2:
            raise ValueError("polarizability_ts must contain at least 2 configurations")
        lib = _lib.lib()
        device = int(ctx.device.index or 0)
        points = int(lib.rn_spectrum_num_points(ctx.num_frames))
        with torch.cuda.device(device):
            wavenumbers = torch.empty(points, dtype=torch.float64, device=ctx.device)
            intensities = torch.empty(points, dtype=torch.float64, device=ctx.device)
            if points == 0:
                return wavenumbers, intensities
            stream = _lib.current_stream(device)
            group = ctx.transform_ranks
            series_ptr = ctypes.c_void_p(ctx.ptr(ctx.rank, "series", self._slot))
            work_ptr = ctypes.c_void_p(ctx.ptr(ctx.rank, "work"))
            if ctx.pipeline:
                # The three packed sequences are independent transforms: sequence s runs pack -> barrier ->
                # convolution on its own stream, the packs one after the other, so that the NVLink-bound
                # stores of one sequence (pack, last inverse pass) overlap the FP64-bound passes of another.
                current = torch.cuda.current_stream(device)
                start = torch.cuda.Event()
                start.record(current)
                packed = None
                finished = []
                for seq, lane in enumerate([current] + ctx.side_streams(device)):
                    if seq > 0:
                        lane.wait_event(start)
                        lane.wait_event(packed)
                    with torch.cuda.stream(lane):
                        lane_stream = ctypes.c_void_p(lane.cuda_stream)
                        _lib.check(lib.rn_spectrum_dist_pack(ctx.plan, series_ptr, ctx.table("work", group),
                                                             ctx.table("spectrum", ctx.world), ctx.world, seq, -1,
                                                             lane_stream), "rn_spectrum_dist_pack")
                        packed = torch.cuda.Event()
                        packed.record(lane)
                        ctx.barrier(channel=1 + seq)  # residue blocks of sequence `seq` have landed everywhere
                        _lib.check(lib.rn_spectrum_dist_transform(ctx.plan, work_ptr, ctx.table("recv", group), seq,
                                                                  lane_stream), "rn_spectrum_dist_transform")
                        if seq > 0:
                            done = torch.cuda.Event()
                            done.record(lane)
                            finished.append(done)
                for done in finished:
                    current.wait_event(done)
            else:
                # the first half of the pack may already be under way (ShardedTrajectory overlapped it with the
                # evaluation of the frames the second half needs)
                half_done = ctx.packed_generation == self._generation
                if half_done:
                    torch.cuda.current_stream(device).wait_event(ctx.pack_event)
                    ctx.packed_generation = -1  # the transform runs in place: a second measure() packs everything
                _lib.check(lib.rn_spectrum_dist_pack(ctx.plan, series_ptr, ctx.table("work", group),
                                                     ctx.table("spectrum", ctx.world), ctx.world, -1,
                                                     1 if half_done else -1, stream), "rn_spectrum_dist_pack")
                ctx.barrier()  # every residue of every block has landed in the work buffers
                _lib.check(lib.rn_spectrum_dist_transform(ctx.plan, work_ptr, ctx.table("recv", group), -1, stream),
                           "rn_spectrum_dist_transform")
            ctx.barrier()  # every rank holds all residues of the bin pairs it owns (and every energy share)
            spectrum_ptr = ctypes.c_void_p(ctx.ptr(ctx.rank, "spectrum"))
            transforms = ctx.rank < group
            status = lib.rn_spectrum_dist_final(
                ctx.plan, ctypes.c_void_p(ctx.ptr(ctx.rank, "recv")), spectrum_ptr, ctx.table("spectrum", ctx.world),
                ctx.world, float(self._timestep), 1 if laser_correction else 0,
                float(laser_wavelength) if laser_correction else 0.0, 1 if bose_einstein_correction else 0,
                float(temperature) if bose_einstein_correction else 0.0,
                ctypes.c_void_p(wavenumbers.data_ptr()) if transforms else None, stream)
            _lib.check(status, "rn_spectrum_dist_final")
            ctx.barrier()  # the finished intensities of every owner have landed on every rank
            _lib.check(lib.rn_spectrum_dist_finish(ctx.plan, spectrum_ptr, float(self._timestep),
                                                   None if transforms else ctypes.c_void_p(wavenumbers.data_ptr()),
                                                   ctypes.c_void_p(intensities.data_ptr()), stream),
                       "rn_spectrum_dist_finish")
        return wavenumbers, intensities


class ShardedTrajectory(Dynamics):
    """The local frame block of a trajectory that is sharded over the ranks of a process group.

    Parameters
    ----------
    local_positions_ts
        (fractional) (S_r,N,3) block of this rank, frames ``shard_bounds(num_frames, G, r)``;
        numpy (host) or CUDA tensor (HBM-resident).
    timestep
        (fs)
    num_frames
        Total number of frames S over all ranks.
    """

    def __init__(self, local_positions_ts, timestep: float, num_frames: int, group=None) -> None:
        import torch.distributed as dist  # pylint: disable=import-outside-toplevel

        self._local = Trajectory(local_positions_ts, timestep)
        self._num_frames = int(num_frames)
        self._group = group
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        start, stop = shard_bounds(self._num_frames, world, rank)
        if len(self._local) != stop - start:
            raise ValueError(f"rank {rank} holds {len(self._local)} frames, expected {stop - start}")

    @property
    def local(self) -> Trajectory:
        return self._local

    @property
    def num_frames(self) -> int:
        return self._num_frames

    def get_raman_spectrum(self, polarizability_model, shared: bool = True) -> MDRamanSpectrum:
        """Evaluate the local block; returns a ``ShardedMDRamanSpectrum``.

        ``shared=True`` (default; CUDA + NCCL groups of at most 8 ranks with this package's models):
        the rows are routed to the ranks that consume them and ``measure`` runs one chirp-z transform
        shared by the ranks.  The spectrum object refers to buffers that the next ``get_raman_spectrum``
        call of the same size overwrites.  Otherwise, or if symmetric memory is unavailable: one
        ``all_gather_into_tensor`` assembles the series on every rank."""
        if shared:
            spectrum = self._get_raman_spectrum_shared(polarizability_model)
            if spectrum is not None:
                return spectrum
        return self._allgather_spectrum(self._local.get_raman_spectrum(polarizability_model))

    def get_raman_spectra(self, polarizability_models, shared: bool = True) -> list:
        """Mask sweep (``Trajectory.get_raman_spectra``) of the sharded trajectory: one
        ``ShardedMDRamanSpectrum`` per model, all evaluated in one pass over the local block; equal to
        ``[self.get_raman_spectrum(m) for m in polarizability_models]`` with each spectrum measured before the
        next is evaluated.

        ``shared=True``: the rows of model g are routed into series slot g of the shared context, and every
        spectrum's ``measure`` runs the chirp-z transform shared by the ranks on its slot.  The G spectra stay
        valid together — measured in any order, any number of times — until the next ``get_raman_spectrum`` /
        ``get_raman_spectra`` call of the same size.  Otherwise, or if symmetric memory is unavailable: the
        local block is swept and one ``all_gather_into_tensor`` per model assembles the series on every rank."""
        models = list(polarizability_models)
        if shared:
            spectra = self._get_raman_spectra_shared(models)
            if spectra is not None:
                return spectra
        return [self._allgather_spectrum(local) for local in self._local.get_raman_spectra(models)]

    def _allgather_spectrum(self, local: MDRamanSpectrum) -> ShardedMDRamanSpectrum:
        """All-gather path: the spectrum of the whole series assembled from this rank's ``local`` spectrum."""
        import torch  # pylint: disable=import-outside-toplevel
        import torch.distributed as dist  # pylint: disable=import-outside-toplevel

        series = local._polarizability_ts  # pylint: disable=protected-access
        if not _lib.is_torch_tensor(series):
            series = torch.from_numpy(series)
        full = allgather_series(series, self._num_frames, self._group)
        bounds = shard_bounds(self._num_frames, dist.get_world_size(self._group), dist.get_rank(self._group))
        return ShardedMDRamanSpectrum(full, self._local.timestep, self._group, bounds=bounds)

    def _get_raman_spectra_shared(self, models):
        import torch  # pylint: disable=import-outside-toplevel
        import torch.distributed as dist  # pylint: disable=import-outside-toplevel

        from .pmodel import InterpolationModel, calc_polarizabilities_sweep_routed  # pylint: disable=import-outside-toplevel

        # anything the sweep rejects (no models, more than 64, foreign models) raises on the all-gather path
        if not 1 <= len(models) <= 64 or not all(isinstance(m, InterpolationModel) for m in models):
            return None
        if not torch.cuda.is_available() or dist.get_backend(self._group) != "nccl":
            return None
        world, rank = dist.get_world_size(self._group), dist.get_rank(self._group)
        if world == 1 or world > 8 or self._num_frames < 2:
            return None
        positions = self._local._positions_ts  # pylint: disable=protected-access
        device = positions.device if hasattr(positions, "data_ptr") else torch.device("cuda", torch.cuda.current_device())
        ctx = _shared_context(self._num_frames, device, self._group, slots=len(models))
        if ctx is None:
            return None
        start, stop = shard_bounds(self._num_frames, world, rank)
        local_ptrs = [ctx.ptr(rank, "series", g) + start * 72 for g in range(len(models))]
        peers = [[0 if r == rank else ctx.ptr(r, "series", g) for r in range(world)] for g in range(len(models))]
        if ctx.pack_event is not None:  # a first pack half that no measure() waited for still reads the buffers
            torch.cuda.current_stream(device).wait_event(ctx.pack_event)
            ctx.pack_event = None
        try:
            calc_polarizabilities_sweep_routed(models, positions, local_ptrs, peers, start, ctx.period, ctx.width)
        except ValueError as exc:
            raise ValueError("polarizability_model and trajectory are incompatible") from exc
        ctx.generation += 1
        ctx.barrier()  # every rank's rows of every mask have landed where they are consumed
        return [ShardedMDRamanSpectrum(None, self._local.timestep, self._group, context=ctx, generation=ctx.generation,
                                       bounds=(start, stop), slot=g) for g in range(len(models))]

    def _phased(self, ctx, model, positions, start: int) -> bool:
        """True if EVERY rank can evaluate its block in the two phases of the overlapped schedule (decided
        once per model and block: the answer is a collective)."""
        if not ctx.overlap or ctx.stripe <= 0 or ctx.pipeline or not hasattr(positions, "data_ptr"):
            return False
        supported = getattr(model, "routed_phases_supported", None)
        if supported is None:
            return False
        key = (id(model), int(positions.data_ptr()), tuple(positions.shape))
        if key not in ctx.phased:
            ctx.phased.clear()
            ctx.phased[key] = _all_ranks_agree(bool(supported(positions, start, ctx.stripe)), ctx.device, self._group)
        return ctx.phased[key]

    def _get_raman_spectrum_shared(self, polarizability_model):
        import torch  # pylint: disable=import-outside-toplevel
        import torch.distributed as dist  # pylint: disable=import-outside-toplevel

        routed = getattr(polarizability_model, "calc_polarizabilities_routed", None)
        if routed is None or not torch.cuda.is_available() or dist.get_backend(self._group) != "nccl":
            return None
        world, rank = dist.get_world_size(self._group), dist.get_rank(self._group)
        if world == 1 or world > 8 or self._num_frames < 2:
            return None
        positions = self._local._positions_ts  # pylint: disable=protected-access
        device = positions.device if hasattr(positions, "data_ptr") else torch.device("cuda", torch.cuda.current_device())
        ctx = _shared_context(self._num_frames, device, self._group)
        if ctx is None:
            return None
        start, stop = shard_bounds(self._num_frames, world, rank)
        peers = [0 if r == rank else ctx.ptr(r, "series") for r in range(world)]
        local_ptr = ctx.ptr(rank, "series") + start * 72
        phased = self._phased(ctx, polarizability_model, positions, start)
        generation = ctx.generation + 1
        if ctx.pack_event is not None:  # a first pack half that no measure() waited for still reads the buffers
            torch.cuda.current_stream(device).wait_event(ctx.pack_event)
            ctx.pack_event = None
        try:
            if phased:
                # Two launches: first the frames the first half of every rank's pack reads, then the others.  After
                # a barrier the pack's first half (NVLink-bound) runs on a side stream under the second launch
                # (HBM-bound); ``measure`` packs the other half.
                routed(positions, local_ptr, peers, start, ctx.period, ctx.width, stripe=ctx.stripe, phase=0)
                ctx.barrier()  # the rows of the first halves have landed on every rank
                current = torch.cuda.current_stream(device)
                landed = torch.cuda.Event()
                landed.record(current)
                # the evaluation is enqueued FIRST and the pack stream has no priority over it: the evaluation's
                # CTAs (one per SM, most of its shared memory) are placed first and the pack's CTAs fill in beside
                # them — the other way round the pack's thousand small CTAs occupy the SMs and the evaluation waits
                routed(positions, local_ptr, peers, start, ctx.period, ctx.width, stripe=ctx.stripe, phase=1)
                side = ctx.pack_stream(device)
                side.wait_event(landed)
                group = ctx.transform_ranks
                _lib.check(_lib.lib().rn_spectrum_dist_pack(
                    ctx.plan, ctypes.c_void_p(ctx.ptr(rank, "series")), ctx.table("work", group),
                    ctx.table("spectrum", world), world, -1, 0, ctypes.c_void_p(side.cuda_stream)), "rn_spectrum_dist_pack")
                ctx.pack_event = torch.cuda.Event()
                ctx.pack_event.record(side)
                ctx.packed_generation = generation
            else:
                routed(positions, local_ptr, peers, start, ctx.period, ctx.width)
        except ValueError as exc:
            raise ValueError("polarizability_model and trajectory are incompatible") from exc
        ctx.generation = generation
        ctx.barrier()  # every rank's rows have landed where they are consumed
        return ShardedMDRamanSpectrum(None, self._local.timestep, self._group, context=ctx,
                                      generation=ctx.generation, bounds=(start, stop))

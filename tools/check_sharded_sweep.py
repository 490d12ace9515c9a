"""Multi-GPU parity check of mask sweeps on frame-sharded trajectories (launch with torchrun, one rank per GPU;
tests/test_gpu_multi_sweep.py does): ShardedTrajectory.get_raman_spectra -> routed sweep evaluation -> one
shared chirp-z transform per mask, against the CPU oracle on the full trajectory, against per-mask
get_raman_spectrum, and against the single-GPU Trajectory.get_raman_spectra on the gathered trajectory.
The spectra are measured in reverse order and twice; a later evaluation must invalidate them."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from oracle import numpy_port as ora  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.distributed import ShardedTrajectory, shard_bounds  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
device = torch.device(f"cuda:{local}")
dist.init_process_group("nccl", device_id=device)
ok = True
big_frames = int(os.environ.get("RN_CHECK_BIG_FRAMES", "600000"))


def species_masks(model, structure):
    """One masked copy per species (the masking tutorial): the DOFs that move that species' atoms are masked."""
    numbers = synthetic.load_structure(structure)["atomic_numbers"]
    finder = rb.ARTModel(model.state)  # get_dof_indexes only reads the basis vectors
    return [model.get_masked_model(finder.get_dof_indexes([int(a) for a in np.flatnonzero(numbers == z)]))
            for z in np.unique(numbers)]


def gathered(sharded, frames):
    """The full trajectory on this rank (a CUDA tensor)."""
    positions = sharded.local._positions_ts  # pylint: disable=protected-access
    block = positions if hasattr(positions, "data_ptr") else torch.from_numpy(positions).to(device)
    start, stop = shard_bounds(frames, world, rank)
    per = -(-frames // world)
    padded = torch.zeros((per,) + tuple(block.shape[1:]), dtype=torch.float64, device=device)
    padded[: stop - start] = block
    full = torch.empty((world * per,) + tuple(block.shape[1:]), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(full, padded)
    return full[:frames]


def check_case(label, models, positions, frames, timestep, oracle):
    global ok  # pylint: disable=global-statement
    start, stop = shard_bounds(frames, world, rank)
    if oracle:
        want = []
        for model in models:
            state = model.state
            omodel = ora.OracleModel(state.ref_positions, state.lattice, state.ref_polarizability,
                                     list(state.basis_vectors), list(state.splines), state.mask)
            alpha = ora.calc_polarizabilities(omodel, ora.trajectory_positions(positions))
            want.append((alpha,) + tuple(ora.md_measure(alpha, timestep, laser_correction=True,
                                                         bose_einstein_correction=True)))
    for resident, shared in ((False, True), (True, True), (True, False), (False, False)):
        block = positions[start:stop] if isinstance(positions, np.ndarray) else positions[start:stop].cpu().numpy()
        if resident:
            block = torch.from_numpy(block).to(device)
        sharded = ShardedTrajectory(block, timestep, frames)
        spectra = sharded.get_raman_spectra(models, shared=shared)
        used = all(getattr(s, "_context", None) is not None for s in spectra)
        measured = {}
        for g in reversed(range(len(models))):
            measured[g] = spectra[g].measure_device(laser_correction=True, bose_einstein_correction=True)
        again = {g: spectra[g].measure_device(laser_correction=True, bose_einstein_correction=True)
                 for g in reversed(range(len(models)))}
        series = [spectra[g].polarizability_ts for g in range(len(models))]
        single = rb.Trajectory(gathered(sharded, frames), timestep).get_raman_spectra(models)
        lines = []
        for g, model in enumerate(models):
            wn, inten = (t.cpu().numpy() for t in measured[g])
            repeat = all(torch.equal(a, b) for a, b in zip(measured[g], again[g]))
            swn, sint = single[g].measure(laser_correction=True, bose_einstein_correction=True)
            salpha = single[g].polarizability_ts
            e_s = float(np.max(np.abs(series[g] - salpha)) / np.max(np.abs(salpha)))
            e_si = float(np.max(np.abs(inten - sint) / np.abs(sint)))
            good = repeat and np.array_equal(wn, swn) and e_si <= 1e-8 and e_s <= 1e-13
            if oracle:
                alpha_w, wn_w, int_w = want[g]
                e_a = float(np.max(np.abs(series[g] - alpha_w)) / np.max(np.abs(alpha_w)))
                e_i = float(np.max(np.abs(inten - int_w) / np.abs(int_w)))
                good = good and e_a <= 1e-10 and e_i <= 1e-8 and np.array_equal(wn, wn_w)
            else:
                e_a = e_i = float("nan")
            # the same as evaluating the masks one by one, each measured before the next is evaluated
            one = sharded.get_raman_spectrum(model, shared=shared)
            own, oint = one.measure(laser_correction=True, bose_einstein_correction=True)
            good = good and np.array_equal(own, wn) and float(np.max(np.abs(oint - inten) / np.abs(oint))) <= 1e-8
            lines.append((g, good, e_a, e_i, e_s, e_si))
        # the evaluations above replaced the shared series: every spectrum of the sweep must refuse to measure
        stale = True
        for spectrum in spectra if used else []:
            try:
                spectrum.measure()
                stale = False
            except RuntimeError:
                pass
        for g, good, e_a, e_i, e_s, e_si in lines:
            good = good and stale
            ok = ok and good
            print(f"rank {rank}/{world} {label} S={frames} resident={resident} shared={shared} (used={used}) mask {g}: "
                  f"alpha {e_a:.1e} intensity {e_i:.1e} vs single GPU {e_s:.1e} / {e_si:.1e} ok={good}", flush=True)
        del spectra, sharded, single


cases = [("LLZO/art", "LLZO", "art", None, 5001), ("STO/cubic", "STO", "cubic", None, 1237),
         ("TiO2/art", "TiO2", "art", None, 40)]
for label, structure, kind, dofs, frames in cases:
    state = synthetic.make_model(structure, kind, num_dofs=dofs)
    model = (rb.ARTModel if kind == "art" else rb.InterpolationModel)(state, device=local)
    check_case(label, species_masks(model, structure), synthetic.make_trajectory(structure, frames, seed=99), frames,
               1.0, oracle=True)

# a large case with an uneven tail: strided levels in the local transforms, rows routed across many tiles
state = synthetic.make_model("LLZO", "art")
model = rb.ARTModel(state, device=local)
frames = big_frames + 7
positions = synthetic.make_trajectory_cuda("LLZO", frames, device, seed=1000)
check_case("LLZO/art", species_masks(model, "LLZO"), positions, frames, 0.5, oracle=False)

flag = torch.tensor([1 if ok else 0], device=device)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) == 1 else 1)

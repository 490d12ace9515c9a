"""Multi-GPU check of cross spectra of frame-sharded mask sweeps (launch with torchrun, one rank per GPU;
tests/test_gpu_multi_cross.py does): ShardedTrajectory.get_raman_spectra(models) followed by
measure_cross_spectra on every rank, with the shared transform context and with the all-gather fallback,
against measure_cross_spectra of the gathered series on one GPU (bit for bit) and the CPU oracle
(|I_gh - ref_gh| <= 1e-8 sqrt(ref_gg ref_hh)).  At world 1 every call takes the single-GPU path."""
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

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from cross_oracle import md_cross_measure  # noqa: E402  pylint: disable=wrong-import-position

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
device = torch.device(f"cuda:{local}")
dist.init_process_group("nccl", device_id=device)
ok = True
KWARGS = dict(laser_correction=True, laser_wavelength=532, bose_einstein_correction=True, temperature=300)


# pylint: disable=too-many-locals
def check_case(label, model, masks, positions, timestep):
    global ok  # pylint: disable=global-statement
    frames = len(positions)
    start, stop = shard_bounds(frames, world, rank)
    models = [model.get_masked_model(mask) for mask in masks]
    alpha_want = []
    for masked in models:
        state = masked.state
        omodel = ora.OracleModel(state.ref_positions, state.lattice, state.ref_polarizability,
                                 list(state.basis_vectors), list(state.splines), state.mask)
        alpha_want.append(ora.calc_polarizabilities(omodel, ora.trajectory_positions(positions)))
    ref_wn, ref = md_cross_measure(alpha_want, timestep, **KWARGS)
    diag = np.abs(np.diagonal(ref, axis1=0, axis2=1)).T
    scale = np.sqrt(diag[:, None, :] * diag[None, :, :])
    for resident, shared in ((False, True), (True, True), (True, False)):
        block = positions[start:stop]
        if resident:
            block = torch.from_numpy(block).to(device)
        spectra = ShardedTrajectory(block, timestep, frames).get_raman_spectra(models, shared=shared)
        used = getattr(spectra[0], "_context", None) is not None
        wn, cross = rb.measure_cross_spectra(spectra, **KWARGS)  # collective with a shared context
        alphas = [s.polarizability_ts for s in spectra]
        swn, scross = rb.measure_cross_spectra([rb.MDRamanSpectrum(a, timestep) for a in alphas], **KWARGS)
        good = cross.shape == (len(models), len(models), len(wn)) and np.array_equal(wn, swn) \
            and np.array_equal(cross, scross) and np.array_equal(wn, ref_wn)
        e_a = max(float(np.max(np.abs(a - w)) / np.max(np.abs(w))) for a, w in zip(alphas, alpha_want))
        e_i = float(np.max(np.abs(cross - ref) / scale))
        good = good and e_a <= 1e-10 and e_i <= 1e-8
        ok = ok and good
        print(f"rank {rank}/{world} {label} S={frames} G={len(models)} resident={resident} shared={shared} "
              f"(used={used}): alpha {e_a:.1e} cross {e_i:.1e} ok={good}", flush=True)


state = synthetic.make_model("LLZO", "art")
llzo = rb.ARTModel(state, device=local)
rng = np.random.default_rng(4)
check_case("LLZO/art", llzo, [np.flatnonzero(rng.random(state.num_dofs) < 0.5) for _ in range(3)],
           synthetic.make_trajectory("LLZO", 5001, seed=99), 1.0)
state = synthetic.make_model("TiO2", "art")
dofs = np.arange(state.num_dofs)
check_case("TiO2/art", rb.ARTModel(state, device=local), [dofs[dofs % 2 == 0], dofs[dofs % 2 == 1]],
           synthetic.make_trajectory("TiO2", 2403, seed=98), 0.5)

flag = torch.tensor([1 if ok else 0], device=device)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) == 1 else 1)

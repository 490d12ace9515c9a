"""Multi-GPU check of windowed spectra on frame-sharded trajectories (launch with torchrun, one rank per GPU;
tests/test_gpu_multi_windows.py does): ShardedTrajectory.get_raman_spectrum(...).measure_windows on every rank,
with the shared transform context and with the all-gather fallback, against MDRamanSpectrum.measure_windows
of the gathered series on one GPU (bit for bit) and the CPU oracle per window (1e-8).  At world 1 every call
takes the single-GPU path."""
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
KWARGS = dict(laser_correction=True, laser_wavelength=532, bose_einstein_correction=True, temperature=300)


# pylint: disable=too-many-locals
def check_case(label, model, positions, timestep, window, hop, oracle_rows):
    global ok  # pylint: disable=global-statement
    frames = len(positions)
    start, stop = shard_bounds(frames, world, rank)
    state = model.state
    omodel = ora.OracleModel(state.ref_positions, state.lattice, state.ref_polarizability,
                             list(state.basis_vectors), list(state.splines), state.mask)
    alpha_want = ora.calc_polarizabilities(omodel, ora.trajectory_positions(positions))
    step = window if hop is None else hop
    want = {w: ora.md_measure(alpha_want[w * step: w * step + window], timestep, **KWARGS) for w in oracle_rows}
    for resident, shared in ((False, True), (True, True), (True, False)):
        block = positions[start:stop]
        if resident:
            block = torch.from_numpy(block).to(device)
        spectrum = ShardedTrajectory(block, timestep, frames).get_raman_spectrum(model, shared=shared)
        used = getattr(spectrum, "_context", None) is not None
        wn, inten = spectrum.measure_windows(window, hop, **KWARGS)  # collective with a shared context
        alpha = spectrum.polarizability_ts
        swn, sint = rb.MDRamanSpectrum(alpha, timestep).measure_windows(window, hop, **KWARGS)
        windows = 1 + (frames - window) // step
        good = inten.shape == (windows, len(wn)) and np.array_equal(wn, swn) and np.array_equal(inten, sint)
        e_a = float(np.max(np.abs(alpha - alpha_want)) / np.max(np.abs(alpha_want)))
        e_i = 0.0
        for w, (wn_w, int_w) in want.items():
            good = good and np.array_equal(wn, wn_w)
            e_i = max(e_i, float(np.max(np.abs(inten[w] - int_w) / np.abs(int_w))))
        good = good and e_a <= 1e-10 and e_i <= 1e-8
        ok = ok and good
        print(f"rank {rank}/{world} {label} S={frames} window={window} hop={hop} W={windows} resident={resident} "
              f"shared={shared} (used={used}): alpha {e_a:.1e} intensity {e_i:.1e} ok={good}", flush=True)


state = synthetic.make_model("LLZO", "art")
check_case("LLZO/art", rb.ARTModel(state, device=local), synthetic.make_trajectory("LLZO", 5001, seed=99), 1.0,
           1000, 333, (0, 6, 12))
state = synthetic.make_model("TiO2", "art")
check_case("TiO2/art", rb.ARTModel(state, device=local), synthetic.make_trajectory("TiO2", 2403, seed=98), 0.5,
           600, None, (0, 3))

flag = torch.tensor([1 if ok else 0], device=device)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag) == 1 else 1)

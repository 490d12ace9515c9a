"""Mean squared displacement, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_msd_device(lattice, groups): every group on the batched autocorrelation path;
  B = the torch composition a user writes without A: device minimum-image steps, torch.cumsum for the unwrapped
      Cartesian path, torch.fft.rfft / irfft at n = 2^p >= 2S - 1 for the autocorrelation, the cumulative-sum term
      and the group means.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call (median of
REPEATS); the peak device memory of each is torch.cuda.max_memory_allocated over one call, above what was allocated
before it.  Kernel times come from separate torch.profiler passes over one call of each.  Workloads: (a) LLZO,
192 atoms, S = 1e6, species groups, with a random walk added to the Li atoms; (b) TiO2, 108 atoms, S = 1e5, one
group; (c) LLZO, S = 1e5, per-atom groups.  The transform rate is 3 * slots * L points over the time of A's
transform passes (level and tile kernels).  On (a) A is also run on eight atoms of each species and checked against
the numpy oracle (tests/msd_oracle.py, FFT form) with the bound of the tests, and MSD(1) of the diffusing Li atoms
against their mean squared minimum-image step.
python tools/run_msd.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.spectrum import clear_plan_cache  # noqa: E402
from msd_oracle import error_ratio, msd_fft  # noqa: E402  pylint: disable=wrong-import-position

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r09_msd.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
LI_STEP = 0.01  # Å per frame and Cartesian component of the Li random walk of (a)


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def composition(positions, lattice, timestep, groups):
    """What a user writes today, on the device: (lag_times (S,), msd (G,S))."""
    frames, num_atoms = positions.shape[0], positions.shape[1]
    d = torch.diff(positions, dim=0)
    d = d - torch.ceil(d - 0.5)
    r = torch.zeros_like(positions)
    torch.cumsum(d @ torch.as_tensor(lattice, device=positions.device), dim=0, out=r[1:])
    del d
    n = 1 << int(2 * frames - 1).bit_length()
    spectrum = torch.fft.rfft(r.view(frames, 3 * num_atoms), n=n, dim=0)
    power = spectrum.real.square() + spectrum.imag.square()
    del spectrum
    c = torch.fft.irfft(power, n=n, dim=0)[:frames].view(frames, num_atoms, 3).sum(dim=2)  # (S,N)
    del power
    prefix = torch.zeros((frames + 1, num_atoms), dtype=torch.float64, device=positions.device)
    torch.cumsum(r.square().sum(dim=2), dim=0, out=prefix[1:])
    lags = torch.arange(frames, device=positions.device)
    per_atom = (prefix[frames - lags] + (prefix[frames:] - prefix[lags]) - 2 * c) / (frames - lags)[:, None]
    per_atom[0] = 0.0
    rows = torch.stack([per_atom[:, torch.as_tensor(list(g), device=positions.device)].mean(dim=1) for g in groups])
    return lags.to(torch.float64) * timestep, rows


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


def peak_bytes(fn):
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    result = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - before
    del result
    return int(peak)


def kernel_ms(fn):
    """Device time per kernel name of one fn() call (torch.profiler, a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile  # pylint: disable=import-outside-toplevel

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    times = {}
    for event in prof.key_averages():
        value = float(getattr(event, "self_device_time_total", getattr(event, "self_cuda_time_total", 0.0)))
        if value > 0:
            times[event.key] = times.get(event.key, 0.0) + value / 1000.0
    return times


def kernel_total(times):
    return sum(v for k, v in times.items() if not k.startswith(("Memcpy", "Memset")))


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def transform_length(frames):
    """L of the plan of S + 1 frames: the smallest power of two >= max(2S - 1, 4096)."""
    log2l = 12
    while (1 << log2l) < max(2 * frames - 1, 4096):
        log2l += 1
    return 1 << log2l


def make_positions(structure, frames, diffusing_z):
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=31)
    if diffusing_z is None:
        return positions
    geom = synthetic.load_structure(structure)
    walkers = torch.as_tensor(np.flatnonzero(geom["atomic_numbers"] == diffusing_z), device=device)
    gen = torch.Generator(device=device)
    gen.manual_seed(32)
    walk = torch.randn((frames, len(walkers), 3), generator=gen, device=device, dtype=torch.float64) * LI_STEP
    walk = torch.cumsum(walk, dim=0) @ torch.as_tensor(np.linalg.inv(geom["lattice"]), device=device)
    moved = positions[:, walkers] + walk
    positions[:, walkers] = moved - torch.floor(moved)
    return positions


def accuracy(trajectory, lattice, numbers):
    """Eight atoms of each species at full length against the numpy oracle; MSD(1) of the Li atoms."""
    species = [np.flatnonzero(numbers == z)[:8] for z in np.unique(numbers)]
    atoms = np.concatenate(species)
    host = trajectory._positions_ts[:, torch.as_tensor(atoms, device=device)].cpu().numpy()  # pylint: disable=protected-access
    local = [list(range(8 * g, 8 * g + len(s))) for g, s in enumerate(species)]
    _, got = (t.cpu().numpy() for t in trajectory.get_msd_device(lattice, [s.tolist() for s in species]))
    _, want = msd_fft(host, lattice, 1.0, local)
    ratio = error_ratio(got, want, host, lattice, local)
    li = list(np.unique(numbers)).index(3)
    d = np.diff(host[:, local[li]], axis=0)
    d = d - np.ceil(d - 0.5)
    step = float(np.mean(np.sum((d @ lattice) ** 2, axis=2)))
    return {"oracle_atoms": atoms.tolist(), "max_error_over_scale": ratio,
            "li_msd1": float(got[li, 1]), "li_mean_squared_step": step,
            "li_msd1_rel_err": abs(float(got[li, 1]) - step) / step,
            "li_msd_last_lag": float(got[li, -1])}


def run(name, structure, frames, grouping, diffusing_z=None):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    num_atoms = len(numbers)
    if grouping == "species":
        groups = [np.flatnonzero(numbers == z).tolist() for z in np.unique(numbers)]
    elif grouping == "per_atom":
        groups = [[i] for i in range(num_atoms)]
    else:
        groups = [list(range(num_atoms))]
    positions = make_positions(structure, frames, diffusing_z)
    trajectory = rb.Trajectory(positions, 1.0)
    stored = trajectory._positions_ts  # pylint: disable=protected-access
    new = lambda: trajectory.get_msd_device(lattice, groups)  # noqa: E731
    old = lambda: composition(stored, lattice, 1.0, groups)  # noqa: E731
    new()
    old()  # warm-up: plans, kernel modules, cuFFT plans
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    a_peak, b_peak = peak_bytes(new), peak_bytes(old)
    slots = sum((len(g) + 1) // 2 for g in groups)
    a_kernels = kernel_ms(new)
    b_kernels = kernel_ms(old)
    transform_ms = sum(v for k, v in a_kernels.items() if "level_kernel" in k or "tile_kernel" in k)
    points = 3 * slots * transform_length(frames)
    _, got = (t.cpu().numpy() for t in new())
    _, ref = (t.cpu().numpy() for t in old())
    gm = np.abs(got - ref)
    result = {
        "workload": name, "structure": structure, "atoms": num_atoms, "frames": frames, "groups": len(groups),
        "slots": slots, "transform_length": transform_length(frames),
        "msd_ms": stats(a_ms), "torch_ms": stats(b_ms), "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "msd_peak_bytes": a_peak, "torch_peak_bytes": b_peak,
        "msd_kernel_ms_total": kernel_total(a_kernels), "msd_kernel_ms": a_kernels,
        "msd_transform_ms": transform_ms, "transform_points": points,
        "transform_rate_points_per_s": points / (transform_ms * 1e-3),
        "torch_kernel_ms_total": kernel_total(b_kernels), "torch_kernel_ms": b_kernels,
        "torch_max_abs_dev": float(np.max(gm)), "torch_max_abs_dev_over_row_max": float(
            np.max(gm / np.max(np.abs(got), axis=1, keepdims=True))),
        "msd_runs_ms": a_ms, "torch_runs_ms": b_ms,
    }
    if diffusing_z is not None:
        result["accuracy"] = accuracy(trajectory, lattice, numbers)
    print(json.dumps({k: v for k, v in result.items() if not k.endswith(("runs_ms", "kernel_ms"))}), flush=True)
    del trajectory, positions, stored
    clear_plan_cache()
    torch.cuda.empty_cache()
    return result


card, power = gpu_info()
results = [
    run("(a) LLZO, species groups, Li diffusing", "LLZO", 1_000_000, "species", diffusing_z=3),
    run("(b) TiO2, one group", "TiO2", 100_000, "all"),
    run("(c) LLZO, per-atom groups", "LLZO", 100_000, "per_atom"),
]
record = {"what": "Trajectory.get_msd_device (A) against the torch composition (B: device minimum-image steps, "
                  "torch.cumsum, torch.fft.rfft/irfft at n = 2^p, the cumulative-sum term and group means); CUDA events "
                  "around each call, A and B alternated, medians of the repeats; peak memory from "
                  "torch.cuda.max_memory_allocated over one call; kernel times from separate torch.profiler passes over "
                  "one call of each; trajectories HBM-resident float64, timestep 1 fs",
          "gpu": card, "power_limit": power, "repeats": repeats, "li_step_angstrom": LI_STEP, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)

"""Self Van Hove correlation, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_van_hove_device(lattice, lags, r_max, num_bins, groups): per membership chunk a count, scan,
      unwrap and histogram launch, and one finishing launch;
  B = the chunked torch composition a user writes without A: the cumsum unwrap of the image shifts, then per lag and
      chunk of origins the (origins, N, 3) difference tensor, its norms, per-group torch.bincount and the moment sums.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call (median of
REPEATS); the peak device memory of each is torch.cuda.max_memory_allocated over one call, above what was allocated
before it.  Kernel times come from a separate torch.profiler pass over one call of A.  Workloads:
  (a) LLZO, 192 atoms, S = 1e5, the four species groups, Li random walk, 64 log-spaced lags in [1, S/2], r_max 10 Å,
      B = 500;
  (b) LLZO, S = 1e6, the Li group (56 atoms), Li random walk, 100 log-spaced lags up to S/10, r_max 12 Å, B = 600: the
      paths take 56 x 1e6 x 24 B = 1.34 GB, more than the 1 GiB budget, so A runs two membership chunks;
  (c) TiO2, 108 atoms, S = 1e5, one group, lags 1..32, r_max 1 Å, B = 1000: the rattling atoms put nearly every
      displacement in a few bins (the contended histogram).
Rates: displacements per second over the call and over the histogram kernel.  Ceilings of profiles/fp64_peaks.json: a
design that reads each 24-byte partner r(n+t) from HBM is bound at read_ldg128 / 24 B; the FP64 issue rate (DFMA rate,
one instruction per cycle slot) over FP64_PER_DISPLACEMENT instructions bounds the arithmetic.
python tools/run_van_hove.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r11_van_hove.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
# FP64-pipe instructions of one displacement: 3 DSUB, 3 DMUL and 2 DADD for rr, 1 DMUL and 2 DADD for the moments, the
# r_max test; one within r_max adds the square root (MUFU.RSQ64H, 4 DFMA and 4 DMUL), the scale, the bin test and the
# floor (the count of rn_rdf's binning).
FP64_PER_DISPLACEMENT = 12
FP64_PER_BINNED = 11
LI_STEP = 0.01  # Å per frame and Cartesian component of the Li random walk (tools/run_msd.py)
CHUNK_ELEMENTS = 1 << 24  # origins x atoms per step of the torch composition


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def peaks():
    with open(os.path.join(REPO, "profiles", "fp64_peaks.json"), encoding="utf-8") as handle:
        data = json.load(handle)
    return float(data["dfma_tflops"]) * 1e12 / 2, float(data["read_ldg128_gbs"]) * 1e9


def make_positions(structure, frames, diffusing_z):
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=51)
    if diffusing_z is None:
        return positions
    geom = synthetic.load_structure(structure)
    walkers = torch.as_tensor(np.flatnonzero(geom["atomic_numbers"] == diffusing_z), device=device)
    gen = torch.Generator(device=device)
    gen.manual_seed(52)
    walk = torch.randn((frames, len(walkers), 3), generator=gen, device=device, dtype=torch.float64) * LI_STEP
    walk = torch.cumsum(walk, dim=0) @ torch.as_tensor(np.linalg.inv(geom["lattice"]), device=device)
    moved = positions[:, walkers] + walk
    positions[:, walkers] = moved - torch.floor(moved)
    return positions


def composition(positions, lattice, lags, r_max, num_bins, groups):
    """What a user writes today, on the device: (g_s (G, T, B), moments (G, T, 2))."""
    frames = positions.shape[0]
    atoms = sorted({a for g in groups for a in g})
    column = {a: i for i, a in enumerate(atoms)}
    x = positions[:, atoms]
    step = x[1:] - x[:-1]
    shifts = torch.cumsum(torch.ceil(step - 0.5), dim=0)
    r = torch.cat([torch.zeros_like(x[:1]), (x[1:] - x[:1]) - shifts]) @ torch.as_tensor(lattice, device=device)
    del step, shifts
    index = [torch.as_tensor([column[a] for a in g], device=device) for g in groups]
    inv = num_bins / r_max
    edges = torch.arange(num_bins + 1, dtype=torch.float64, device=device) * (r_max / num_bins)
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    counts = torch.zeros((len(groups), len(lags), num_bins), dtype=torch.int64, device=device)
    sums = torch.zeros((len(groups), len(lags), 2), dtype=torch.float64, device=device)
    chunk = max(1, CHUNK_ELEMENTS // len(atoms))
    for ti, t in enumerate(lags):
        for n0 in range(0, frames - t, chunk):
            n1 = min(frames - t, n0 + chunk)
            rr = torch.sum((r[n0 + t:n1 + t] - r[n0:n1]) ** 2, dim=2)
            k = torch.floor(torch.sqrt(rr) * inv)
            for g, cols in enumerate(index):
                sub, kg = rr[:, cols], k[:, cols]
                sums[g, ti, 0] += sub.sum()
                sums[g, ti, 1] += (sub * sub).sum()
                counts[g, ti] += torch.bincount(kg[kg < num_bins].to(torch.int64), minlength=num_bins)
    sizes = torch.as_tensor([len(g) for g in groups], device=device, dtype=torch.float64)
    norm = (frames - torch.as_tensor(lags, device=device, dtype=torch.float64))[None, :] * sizes[:, None]
    return counts / (norm[:, :, None] * shell), sums / norm[:, :, None]


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


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def log_lags(low, high, count):
    """count distinct integers from low to high, log-spaced: the rounded geometric sequence, made longer until its
    distinct values number count."""
    num = count
    while True:
        lags = np.unique(np.rint(np.geomspace(low, high, num)).astype(np.int64))
        if len(lags) >= count:
            return lags
        num += 1


def run(name, structure, frames, grouping, lags, r_max, num_bins, diffusing_z, fp64_per_s, read_per_s):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    if grouping == "species":
        groups = [np.flatnonzero(numbers == z).tolist() for z in np.unique(numbers)]
    elif grouping == "li":
        groups = [np.flatnonzero(numbers == 3).tolist()]
    else:
        groups = [list(range(len(numbers)))]
    lags = [int(t) for t in lags]
    trajectory = rb.Trajectory(make_positions(structure, frames, diffusing_z), 1.0)
    stored = trajectory._positions_ts  # pylint: disable=protected-access
    new = lambda: trajectory.get_van_hove_device(lattice, lags, r_max, num_bins, groups)  # noqa: E731
    old = lambda: composition(stored, lattice, lags, r_max, num_bins, groups)  # noqa: E731
    new()
    old()  # warm-up: kernel modules, torch kernels
    before = rb._lib.launch_count()  # pylint: disable=protected-access
    new()
    torch.cuda.synchronize()
    launches = rb._lib.launch_count() - before  # pylint: disable=protected-access
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    a_peak, b_peak = peak_bytes(new), peak_bytes(old)
    a_kernels = kernel_ms(new)
    hist_ms = sum(v for k, v in a_kernels.items() if "vh_histogram_kernel" in k)
    _, _, got_g, got_m = (t.cpu().numpy() for t in new())
    ref_g, ref_m = (t.cpu().numpy() for t in old())
    sizes = np.array([len(g) for g in groups], dtype=np.float64)
    displacements = float(sizes.sum() * np.sum(frames - np.array(lags)))
    edges = np.arange(num_bins + 1) * (r_max / num_bins)
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    norm = (frames - np.array(lags))[None, :] * sizes[:, None]
    binned = float(np.rint(got_g * norm[:, :, None] * shell).sum())
    fp64 = FP64_PER_DISPLACEMENT * displacements + FP64_PER_BINNED * binned
    result = {
        "workload": name, "structure": structure, "atoms": len(numbers), "frames": frames, "groups": len(groups),
        "memberships": int(sizes.sum()), "lags": len(lags), "r_max": r_max, "num_bins": num_bins,
        "launches": launches, "membership_chunks": (launches - 1) // 4,
        "van_hove_ms": stats(a_ms), "torch_ms": stats(b_ms), "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "van_hove_peak_bytes": a_peak, "torch_peak_bytes": b_peak,
        "van_hove_kernel_ms": a_kernels, "histogram_kernel_ms": hist_ms,
        "displacements": displacements, "displacements_within_r_max": binned,
        "displacements_per_s_call": displacements / (np.median(a_ms) * 1e-3),
        "displacements_per_s_kernel": displacements / (hist_ms * 1e-3),
        "hbm_partner_bound_displacements_per_s": read_per_s / 24,
        "fp64_issue_bound_displacements_per_s": fp64_per_s * displacements / fp64,
        "fp64_share_of_dfma_rate": fp64 / (hist_ms * 1e-3) / fp64_per_s,
        "torch_g_s_max_rel_dev": float(np.max(np.abs(got_g - ref_g) / np.maximum(np.abs(got_g), 1e-300))),
        "torch_bins_differing": int(np.sum(got_g != ref_g)),
        "torch_moments_max_rel_dev": float(np.max(np.abs(got_m - ref_m) / np.maximum(np.abs(got_m), 1e-300))),
        "van_hove_runs_ms": a_ms, "torch_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith(("runs_ms", "kernel_ms"))}), flush=True)
    del trajectory, stored
    torch.cuda.empty_cache()
    return result


card, power = gpu_info()
fp64_rate, read_rate = peaks()
results = [
    run("(a) LLZO, species groups, Li diffusing", "LLZO", 100_000, "species", log_lags(1, 50_000, 64), 10.0, 500, 3,
        fp64_rate, read_rate),
    run("(b) LLZO, Li group, Li diffusing", "LLZO", 1_000_000, "li", log_lags(1, 100_000, 100), 12.0, 600, 3,
        fp64_rate, read_rate),
    run("(c) TiO2, one group", "TiO2", 100_000, "all", np.arange(1, 33), 1.0, 1000, None, fp64_rate, read_rate),
]
record = {"what": "Trajectory.get_van_hove_device (A) against the chunked torch composition (B: cumsum unwrap, per lag "
                  "and chunk of origins the difference tensor, norms, per-group torch.bincount and moment sums); CUDA "
                  "events around each call, A and B alternated, medians of the repeats; peak memory from "
                  "torch.cuda.max_memory_allocated over one call; kernel times from a separate torch.profiler pass "
                  "over one call of A; trajectories HBM-resident float64",
          "gpu": card, "power_limit": power, "repeats": repeats, "fp64_instructions_per_s": fp64_rate,
          "read_bytes_per_s": read_rate, "fp64_per_displacement": FP64_PER_DISPLACEMENT,
          "fp64_per_binned_displacement": FP64_PER_BINNED, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)

"""Radial distribution functions, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_rdf_device(lattice, r_max, num_bins, groups): one histogram launch and one finishing launch;
  B = the chunked torch composition a user writes without A: per group pair and chunk of frames the
      (frames, |a|, |b|, 3) difference tensor, the minimum-image wrap, the product with the lattice, the norms, the
      pair mask and torch.bincount, then the same normalisation.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call (median of
REPEATS); the peak device memory of each is torch.cuda.max_memory_allocated over one call, above what was allocated
before it.  Kernel times come from a separate torch.profiler pass over one call of A.  Workloads: (a) LLZO, 192 atoms,
S = 1e5, the four species groups, r_max = w_min/2, B = 400; (b) LLZO_2x2x2, 1536 atoms, S = 1e4, species groups,
r_max = 12.5 Å, B = 1000; (c) TiO2, 108 atoms, S = 1e5, one group, r_max = 4.8 Å, B = 200.
Rates: pair distances per second count N(N-1)/2 pairs per frame (the species groups partition the atoms); the FP64
rate counts FP64-pipe instructions per pair read from the SASS of rdf_histogram_kernel on its [0, 1] path
(FP64_PER_PAIR for every pair, FP64_PER_BINNED_PAIR more for a pair within r_max), over the histogram kernel's time,
as a share of the DFMA issue rate of profiles/fp64_peaks.json.
python tools/run_rdf.py [OUT.json] [REPEATS]"""
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

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r10_rdf.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
# FP64-pipe instructions of one pair on the [0, 1] path (cuobjdump -sass of rn_rdf.o): the wrap takes two DADD, up to
# two DSETP and one DADD per component (15), the lattice product and |v|^2 12 DMUL and 8 DADD, the r_max test one DSETP;
# a pair within r_max adds the square root (MUFU.RSQ64H, 4 DFMA and 4 DMUL), the scale, the bin test and the floor.
FP64_PER_PAIR = 36
FP64_PER_BINNED_PAIR = 11
CHUNK_ELEMENTS = 1 << 22  # frames x |a| x |b| per step of the torch composition


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def dfma_rate():
    with open(os.path.join(REPO, "profiles", "fp64_peaks.json"), encoding="utf-8") as handle:
        peaks = json.load(handle)
    return float(peaks["dfma_tflops"]) * 1e12 / 2  # two FLOPs per DFMA


def half_width(lattice):
    volume = abs(np.dot(lattice[0], np.cross(lattice[1], lattice[2])))  # as get_rdf computes it
    return min(volume / np.linalg.norm(np.cross(lattice[(c + 1) % 3], lattice[(c + 2) % 3])) for c in range(3)) / 2


def composition(positions, lattice, r_max, num_bins, groups):
    """What a user writes today, on the device: (r (B,), g (G, G, B))."""
    frames = positions.shape[0]
    lat = torch.as_tensor(lattice, device=positions.device)
    inv = num_bins / r_max
    width = r_max / num_bins
    edges = torch.arange(num_bins + 1, dtype=torch.float64, device=positions.device) * width
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    volume = abs(float(np.linalg.det(lattice)))
    index = [torch.as_tensor(np.asarray(g), device=positions.device) for g in groups]
    G = len(groups)
    g_out = torch.zeros((G, G, num_bins), dtype=torch.float64, device=positions.device)
    for a in range(G):
        for b in range(a, G):
            ia, ib = index[a], index[b]
            mask = torch.triu(torch.ones((len(ia), len(ib)), dtype=torch.bool, device=positions.device), 1) \
                if a == b else ia[:, None] != ib[None, :]
            counts = torch.zeros(num_bins, dtype=torch.int64, device=positions.device)
            step = max(1, CHUNK_ELEMENTS // (len(ia) * len(ib)))
            for f0 in range(0, frames, step):
                x = positions[f0:f0 + step]
                d = x[:, ib][:, None, :, :] - x[:, ia][:, :, None, :]
                d = d - torch.ceil(d - 0.5)
                r = torch.linalg.vector_norm(d @ lat, dim=3)
                k = torch.floor(r * inv)[:, mask]
                counts += torch.bincount(k[k < num_bins].to(torch.int64), minlength=num_bins)
            n_ab = len(ia) * len(ib) - int(torch.isin(ia, ib).sum())
            if n_ab > 0:
                g_out[a, b] = counts * (2 if a == b else 1) * volume / (frames * n_ab * shell)
                g_out[b, a] = g_out[a, b]
    return (torch.arange(num_bins, dtype=torch.float64, device=positions.device) + 0.5) * width, g_out


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


def run(name, structure, frames, grouping, r_max, num_bins, dfma_per_s):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    num_atoms = len(numbers)
    if grouping == "species":
        groups = [np.flatnonzero(numbers == z).tolist() for z in np.unique(numbers)]
    else:
        groups = [list(range(num_atoms))]
    r_max = half_width(lattice) if r_max is None else r_max
    trajectory = rb.Trajectory(synthetic.make_trajectory_cuda(structure, frames, device, seed=41), 1.0)
    stored = trajectory._positions_ts  # pylint: disable=protected-access
    new = lambda: trajectory.get_rdf_device(lattice, r_max, num_bins, groups)  # noqa: E731
    old = lambda: composition(stored, lattice, r_max, num_bins, groups)  # noqa: E731
    new()
    old()  # warm-up: kernel modules, torch kernels
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    a_peak, b_peak = peak_bytes(new), peak_bytes(old)
    a_kernels = kernel_ms(new)
    hist_ms = sum(v for k, v in a_kernels.items() if "rdf_histogram_kernel" in k)
    r, got = (t.cpu().numpy() for t in new())
    _, ref = (t.cpu().numpy() for t in old())
    # pairs within r_max, from the counts behind g (exact integers after rounding)
    volume = abs(np.linalg.det(lattice))
    edges = np.arange(num_bins + 1) * (r_max / num_bins)
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    sizes = np.array([len(g) for g in groups], dtype=np.float64)
    n_ab = sizes[:, None] * sizes[None, :] - np.diag(sizes)
    ordered = np.rint(got * (frames * n_ab)[:, :, None] * shell / volume).sum()
    pairs = frames * num_atoms * (num_atoms - 1) / 2
    binned = ordered / 2
    fp64 = FP64_PER_PAIR * pairs + FP64_PER_BINNED_PAIR * binned
    result = {
        "workload": name, "structure": structure, "atoms": num_atoms, "frames": frames, "groups": len(groups),
        "group_pairs": len(groups) * (len(groups) + 1) // 2, "r_max": r_max, "num_bins": num_bins,
        "rdf_ms": stats(a_ms), "torch_ms": stats(b_ms), "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "rdf_peak_bytes": a_peak, "torch_peak_bytes": b_peak,
        "rdf_kernel_ms": a_kernels, "histogram_kernel_ms": hist_ms,
        "pairs": pairs, "pairs_within_r_max": binned,
        "pairs_per_s_call": pairs / (np.median(a_ms) * 1e-3), "pairs_per_s_kernel": pairs / (hist_ms * 1e-3),
        "fp64_instructions": fp64, "fp64_instructions_per_s": fp64 / (hist_ms * 1e-3),
        "fp64_share_of_dfma_rate": fp64 / (hist_ms * 1e-3) / dfma_per_s,
        "torch_max_rel_dev": float(np.max(np.abs(got - ref) / np.maximum(np.abs(got), 1e-300))),
        "torch_bins_differing": int(np.sum(got != ref)),
        "rdf_runs_ms": a_ms, "torch_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith(("runs_ms", "kernel_ms"))}), flush=True)
    del trajectory, stored
    torch.cuda.empty_cache()
    return result


card, power = gpu_info()
rate = dfma_rate()
results = [
    run("(a) LLZO, species groups", "LLZO", 100_000, "species", None, 400, rate),
    run("(b) LLZO_2x2x2, species groups", "LLZO_2x2x2", 10_000, "species", 12.5, 1000, rate),
    run("(c) TiO2, one group", "TiO2", 100_000, "all", 4.8, 200, rate),
]
record = {"what": "Trajectory.get_rdf_device (A) against the chunked torch composition (B: per group pair and chunk of "
                  "frames the difference tensor, minimum-image wrap, lattice product, norms, pair mask and "
                  "torch.bincount); CUDA events around each call, A and B alternated, medians of the repeats; peak "
                  "memory from torch.cuda.max_memory_allocated over one call; kernel times from a separate "
                  "torch.profiler pass over one call of A; trajectories HBM-resident float64",
          "gpu": card, "power_limit": power, "repeats": repeats, "dfma_per_s": rate,
          "fp64_per_pair": FP64_PER_PAIR, "fp64_per_binned_pair": FP64_PER_BINNED_PAIR, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)

"""Cross spectra of G series, timed on one GPU (S = 1e6 frames):
  A = measure_cross_spectra_device(spectra): all G x G spectra in one batched transform;
  B = G measure_device calls (the diagonal only);
  C = the polarization identity a user would write without A: G(G+1)/2 measure_device calls, on each series and
      on the summed series alpha_g + alpha_h (summed on the GPU), then I_gh = (I[g+h] - I_gg - I_hh) / 2.
A, B and C run alternately in one process after warm-ups and are timed with CUDA events around the whole call
(median of REPEATS).  Kernel times come from a separate torch.profiler pass over one A call.  Workloads: a real
sweep (LLZO ARTModel, one mask per species keeping only that species, G = 4) and synthetic series (G = 2, 4, 8).
For the real sweep the largest deviation of A and of C from the CPU oracle is recorded at the scale
sqrt(I_gg I_hh) of each cross term.
python tools/run_cross.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.spectrum import clear_plan_cache  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from cross_oracle import md_cross_measure  # noqa: E402  pylint: disable=wrong-import-position

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r05_cross.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
FRAMES = 1_000_000
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def synthetic_series(count, frames, seed):
    gen = torch.Generator(device).manual_seed(seed)
    steps = torch.arange(frames, dtype=torch.float64, device=device)[None, :, None, None]
    phase = torch.rand((count, 1, 3, 3), dtype=torch.float64, device=device, generator=gen) * 6
    noise = torch.randn((count, frames, 3, 3), dtype=torch.float64, device=device, generator=gen)
    return 6.0 * torch.eye(3, dtype=torch.float64, device=device) + 0.05 * torch.sin(0.013 * steps + phase) \
        + 0.01 * noise


def cross(spectra):
    return rb.measure_cross_spectra_device(spectra)[1]


def diagonal(spectra):
    return [s.measure_device()[1] for s in spectra]


def polarization(spectra):
    """G(G+1)/2 measure_device calls: the diagonal, then every pair through the spectrum of the summed series."""
    count = len(spectra)
    diag = [s.measure_device()[1] for s in spectra]
    rows = [[None] * count for _ in range(count)]
    for g in range(count):
        rows[g][g] = diag[g]
        for h in range(g + 1, count):
            both = rb.MDRamanSpectrum(spectra[g]._polarizability_ts + spectra[h]._polarizability_ts,  # pylint: disable=protected-access
                                      spectra[g].timestep).measure_device()[1]
            rows[g][h] = rows[h][g] = (both - diag[g] - diag[h]) / 2
    return torch.stack([torch.stack(row) for row in rows])


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


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


def deviation(result, ref):
    diag = np.abs(np.diagonal(ref, axis1=0, axis2=1)).T
    scale = np.sqrt(diag[:, None, :] * diag[None, :, :])
    return float(np.max(np.abs(result - ref) / scale))


def run(name, spectra, oracle_series=None):
    count = len(spectra)
    for _ in range(2):  # warm-up: plans, kernel modules
        cross(spectra)
        diagonal(spectra)
        polarization(spectra)
    a_ms, b_ms, c_ms = [], [], []
    for _ in range(repeats):
        a_ms.append(timed(lambda: cross(spectra)))
        b_ms.append(timed(lambda: diagonal(spectra)))
        c_ms.append(timed(lambda: polarization(spectra)))
    result = {"workload": name, "frames": FRAMES, "series": count, "cross_ms": stats(a_ms), "diagonal_ms": stats(b_ms),
              "polarization_loop_ms": stats(c_ms), "cross_kernel_ms": kernel_ms(lambda: cross(spectra)),
              "cross_runs_ms": a_ms, "diagonal_runs_ms": b_ms, "polarization_runs_ms": c_ms}
    a = cross(spectra)
    diag = torch.stack(diagonal(spectra))
    result["diagonal_bit_identical"] = bool(torch.equal(torch.diagonal(a, dim1=0, dim2=1).T, diag))
    if oracle_series is not None:
        _, ref = md_cross_measure(oracle_series, spectra[0].timestep)
        result["max_deviation_from_oracle"] = {"cross": deviation(a.cpu().numpy(), ref),
                                               "polarization_loop": deviation(polarization(spectra).cpu().numpy(), ref)}
    print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms")}), flush=True)
    return result


results = []
state = synthetic.make_model("LLZO", "art")
state.atomic_numbers = [int(z) for z in synthetic.load_structure("LLZO")["atomic_numbers"]]
model = rb.ARTModel(state)
species = ["Li", "La", "Zr", "O"]
groups = [set(model.get_dof_indexes(symbol)) for symbol in species]
copies = [model.get_masked_model([j for j in range(state.num_dofs) if j not in group]) for group in groups]
positions = synthetic.make_trajectory("LLZO", FRAMES, seed=11)
sweep = rb.Trajectory(torch.from_numpy(positions).to(device), 1.0).get_raman_spectra(copies)
del positions
results.append(run("LLZO art, one mask per species (Li, La, Zr, O)", sweep,
                   [s.polarizability_ts for s in sweep]))
del sweep
for count in (2, 4, 8):
    series = synthetic_series(count, FRAMES, count)
    results.append(run(f"synthetic, G = {count}", [rb.MDRamanSpectrum(series[g], 1.0) for g in range(count)]))
    del series
    clear_plan_cache()
    torch.cuda.empty_cache()

card, power = gpu_info()
record = {"what": "measure_cross_spectra_device (A) against G measure_device calls (B, diagonal only) and the "
                  "polarization-identity loop of G(G+1)/2 measure_device calls (C); CUDA events around each call, "
                  "A, B and C alternated, medians of the repeats; kernel times from a separate torch.profiler pass "
                  "over one A call; series HBM-resident float64",
          "gpu": card, "power_limit": power, "repeats": repeats, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)

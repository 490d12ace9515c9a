#!/usr/bin/env python
"""Benchmark of the MD-Raman hot path (BASELINE.json metric: MD frames/s, polarizability +
spectrum, at 1/2/4/8 B200 vs the reference CPU path; % of roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload c3|c4|c5|c2|c1|c3dense] [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic trajectory block that is already resident in
HBM: ``calc_polarizabilities`` over every frame of the rank's block and ``MDRamanSpectrum.measure``
on the whole series.  N>1 is launched with torchrun (one process per GPU): frames are sharded, the
evaluation kernels route every row of the series to the rank whose spectrum stage consumes it, and
the ranks share ONE chirp-z transform (ramannoodle_b200/distributed.py).  Prints ONE JSON line (the
last line of stdout).

Workloads (BASELINE.json configs): "c3" (default) = configs[2], ARTModel of 192-atom LLZO, 1M frames
per GPU (weak scaling; the config north_star's target is quoted on); "c4" = configs[3], 10M LLZO
frames in total sharded over the ranks (strong); "c5" = configs[4], 1536-atom supercell, 4600 DOFs,
1M frames in total (strong); "c1", "c2" the small single-GPU configs.

After the timed region every run checks ITS OWN output against the CPU oracle (``parity`` in the
JSON line): random frame blocks of the series per rank (<= 1e-10) and the whole spectrum on rank 0
(<= 1e-8).

``--dump-outputs DIR`` writes what the last timed step returned on rank 0 as float64 ``.npy`` files:
``polarizability_ts`` (rank 0's frames), ``wavenumbers`` and ``intensities``.  The inputs are seeded, so
two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # name: (structure, kind, frames, "weak" = frames per GPU | "strong" = frames in total, description)
    "c1": ("TiO2", "art", 10_000, "weak", "ARTModel rutile TiO2 (108 atoms, 324 DOFs), 10k-frame synthetic trajectory"),
    "c2": ("STO", "cubic", 100_000, "weak", "InterpolationModel cubic BSpline, SrTiO3 (135 atoms, 405 DOFs), 100k frames"),
    "c3": ("LLZO", "art", 1_000_000, "weak", "ARTModel LLZO (192 atoms, 576 DOFs), 1M-frame synthetic trajectory per GPU"),
    "c4": ("LLZO", "art", 10_000_000, "strong", "ARTModel LLZO (192 atoms, 576 DOFs), 10M-frame synthetic trajectory sharded over the GPUs"),
    "c5": ("LLZO_2x2x2", "cubic4600", 1_000_000, "strong",
           "InterpolationModel (cubic BSpline) of the 1536-atom LLZO 2x2x2 supercell, 4600 DOFs, 1M frames sharded over the GPUs"),
    "c3dense": ("LLZO", "art", 200_000, "weak", "LLZO ARTModel forced through the dense DMMA projection, 200k frames per GPU"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames (per GPU for weak workloads, in total for strong ones)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=8192, help="frames in the CPU-baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (b200 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def workload_frames(args, world):
    """(frames on this launch's ranks in total, scaling)"""
    _, _, frames, scaling, _ = WORKLOADS[args.workload]
    if args.frames > 0:
        frames = args.frames
    total = frames * world if scaling == "weak" else frames
    return total, scaling


# --------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x0000000000000004: "sw_power_cap", 0x0000000000000008: "hw_slowdown",
        0x0000000000000020: "sw_thermal_slowdown", 0x0000000000000040: "hw_thermal_slowdown",
        0x0000000000000080: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
        except Exception:  # pylint: disable=broad-except
            self._nvml = None

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # pylint: disable=broad-except
                pass
            self._stop.wait(0.002)

    def start(self):
        if self._nvml is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peaks() -> tuple[float, str]:
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path, encoding="utf-8") as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp64_peak() -> tuple[float, str]:
    path = os.path.join(REPO, "profiles", "fp64_peaks.json")
    if os.path.exists(path):
        with open(path, encoding="utf-8") as fh:
            return float(json.load(fh)["dmma_m8n8k4_tflops"]), "measured (profiles/fp64_peaks.json, DMMA m8n8k4)"
    return 37.0, "fallback (tools/fp64_peaks.cu, earlier run)"


def ncu_traffic(kernel: str, workload: str):
    """DRAM bytes of the dominant kernel from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep)."""
    path = os.path.join(REPO, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path, encoding="utf-8") as fh:
            return json.load(fh).get(f"{kernel}:{workload}")
    return None


DUMP_ARRAY_BYTES = 16 << 20  # per array: three arrays stay well under 64 MB


def dump_outputs(directory, outputs):
    """Write each array of ``outputs`` as ``directory/<name>.npy`` in float64.  An array larger than
    DUMP_ARRAY_BYTES keeps a fixed, seeded sample of its rows (ascending), the same for every run with
    the same number of rows."""
    import torch

    os.makedirs(directory, exist_ok=True)
    for name, array in outputs.items():
        array = torch.as_tensor(array)
        rows = int(array.shape[0])
        keep = max(1, DUMP_ARRAY_BYTES // (8 * int(np.prod(array.shape[1:]))))
        if rows > keep:
            index = np.sort(np.random.default_rng(0).choice(rows, size=keep, replace=False))
            array = array[torch.from_numpy(index).to(array.device)]
        np.save(os.path.join(directory, f"{name}.npy"), array.to(torch.float64).cpu().numpy())


def build_state(structure, kind):
    from ramannoodle_b200 import synthetic

    if kind == "cubic4600":
        return synthetic.make_model(structure, "cubic", num_dofs=4600)
    return synthetic.make_model(structure, kind)


def oracle_model(state):
    from oracle import numpy_port as ora

    return ora.OracleModel(ref_positions=state.ref_positions, lattice=state.lattice,
                           ref_polarizability=state.ref_polarizability, basis_vectors=list(state.basis_vectors),
                           splines=list(state.splines), mask=state.mask)


# --------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle numpy port on the host cores
# --------------------------------------------------------------------------------------
_WORKER = {}


def _cpu_init(structure, kind):
    _WORKER["model"] = oracle_model(build_state(structure, kind))
    _WORKER["structure"] = structure


def _cpu_chunk(args):
    first, count = args
    from oracle import numpy_port as ora
    from ramannoodle_b200 import synthetic

    positions = synthetic.make_trajectory(_WORKER["structure"], count, seed=1000, first_frame=first)
    t0 = time.perf_counter()
    alpha = ora.calc_polarizabilities(_WORKER["model"], positions)
    return alpha, time.perf_counter() - t0


class CpuPath:
    """The reference's CPU path (oracle numpy/scipy port, statement for statement) as a timed step:
    ``calc_polarizabilities`` on a bounded frame sample split over worker processes (linear in S, so
    extrapolated to the workload's S) + ``md_measure`` on a series of the workload's FULL length
    (the sample's series tiled; O(S log S), not extrapolated up to `measure_cap` frames)."""

    def __init__(self, structure, kind, processes):
        self.structure, self.kind, self.processes = structure, kind, processes
        self.pool = None
        if processes > 1:
            import multiprocessing as mp

            self.pool = mp.get_context("fork").Pool(processes, initializer=_cpu_init, initargs=(structure, kind))
        else:
            _cpu_init(structure, kind)

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()

    def step(self, sample, total_frames, measure_cap=2_500_000):
        from oracle import numpy_port as ora

        per = max(1, sample // self.processes)
        jobs = [(i * per, per) for i in range(self.processes)]
        results = self.pool.map(_cpu_chunk, jobs) if self.pool is not None else [_cpu_chunk(jobs[0])]
        alpha = np.concatenate([r[0] for r in results])
        frames = per * self.processes
        # workers run concurrently: the stage takes as long as the slowest worker's evaluation
        t_poly = max(r[1] for r in results) * (total_frames / frames)
        measured = min(total_frames, measure_cap)
        series = np.resize(alpha, (measured, 3, 3))
        t1 = time.perf_counter()
        ora.md_measure(series, 1.0)
        t_meas = time.perf_counter() - t1
        if measured < total_frames:  # O(S log S) beyond the cap
            t_meas *= (total_frames * np.log2(total_frames)) / (measured * np.log2(measured))
        return total_frames / (t_poly + t_meas), {
            "sample_frames": frames, "t_polarizability_s_extrapolated": round(t_poly, 3),
            "measure_frames": measured, "t_measure_s": round(t_meas, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    structure, kind, _, _, desc = WORKLOADS[args.workload]
    kind = "art" if args.workload == "c3dense" else kind
    total_frames, scaling = workload_frames(args, world)
    cores = os.cpu_count() or 1
    # a bounded sample per step so that warmup + steps end within a few minutes
    per_worker = 512 if kind != "cubic4600" else 32
    sample = (cores if kind != "cubic4600" else min(cores, 16)) * per_worker
    workers = cores if kind != "cubic4600" else min(cores, 16)  # each worker holds the 170 MB basis
    path = CpuPath(structure, kind, workers)
    try:
        for _ in range(max(0, args.warmup)):
            path.step(max(cores * 16, sample // 8), total_frames, measure_cap=min(total_frames, 200_000))
        rates, detail = [], None
        t0 = time.perf_counter()
        for _ in range(max(1, args.steps)):
            rate, detail = path.step(sample, total_frames)
            rates.append(rate)
    finally:
        path.close()
    wall = time.perf_counter() - t0
    value = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": "md_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": len(rates), "warmup": max(0, args.warmup), "ms_per_step": 1e3 * total_frames / value,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}", "total_frames": total_frames, "wall_s": round(wall, 1)},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": workers, "kind": "port",
                         "sample": f"per step: oracle numpy/scipy port (statement-for-statement restatement of the "
                                   f"pure-Python reference) — calc_polarizabilities on {detail['sample_frames']} frames "
                                   f"of the same synthetic workload, frame-chunked over {cores} processes and "
                                   f"extrapolated linearly to {total_frames} frames, + md_measure on a "
                                   f"{detail['measure_frames']}-frame series; {detail}"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------
# parity of the run's own output against the oracle
# --------------------------------------------------------------------------------------
def check_parity(state, structure, trajectory, spectrum, wn, inten, first_frame, rank, world, blocks, block_frames):
    """Random frame blocks of this rank's series against the oracle (<= 1e-10), and on rank 0 the whole
    spectrum against md_measure on the gathered series (<= 1e-8)."""
    import torch
    import torch.distributed as dist

    from oracle import numpy_port as ora

    omodel = oracle_model(state)
    local = spectrum.local_polarizability_ts if hasattr(spectrum, "local_polarizability_ts") else spectrum._polarizability_ts  # pylint: disable=protected-access
    frames = int(local.shape[0])
    rng = np.random.default_rng(77 + rank)
    block_frames = min(block_frames, frames)
    starts = sorted({0, frames - block_frames} | {int(v) for v in rng.integers(0, frames - block_frames + 1, size=blocks)})
    worst, checked = 0.0, 0
    for start in starts:
        pos = trajectory.positions_ts_block(start, start + block_frames) if hasattr(trajectory, "positions_ts_block") \
            else trajectory._positions_ts[start:start + block_frames]  # pylint: disable=protected-access
        pos = pos.cpu().numpy() if hasattr(pos, "cpu") else np.asarray(pos)
        want = ora.calc_polarizabilities(omodel, pos)
        got = local[start:start + block_frames].cpu().numpy()
        worst = max(worst, float(np.max(np.abs(got - want)) / np.max(np.abs(want))))
        checked += block_frames
    series = spectrum.polarizability_ts  # N > 1: gathers the series (a collective; every rank takes part)
    stats = torch.tensor([worst, float(checked)], dtype=torch.float64, device=wn.device)
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        worst, checked = float(mx[0]), float(stats[1])
    result = {"alpha_rel": worst, "alpha_tol": 1e-10, "frames_checked": int(checked),
              "alpha_blocks_per_rank": len(starts), "first_frame_rank0": first_frame}
    if rank == 0:
        t0 = time.perf_counter()
        want_wn, want_int = ora.md_measure(series, 1.0)
        got_wn, got_int = wn.cpu().numpy(), inten.cpu().numpy()
        result.update({"intensity_rel": float(np.max(np.abs(got_int - want_int) / np.abs(want_int))),
                       "intensity_tol": 1e-8, "wavenumbers_equal": bool(np.array_equal(got_wn, want_wn)),
                       "spectrum_points": int(want_int.shape[0]), "oracle_measure_s": round(time.perf_counter() - t0, 1)})
        result["ok"] = bool(result["alpha_rel"] <= 1e-10 and result["intensity_rel"] <= 1e-8 and result["wavenumbers_equal"])
    return result


# --------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import ramannoodle_b200 as rb
    from ramannoodle_b200 import _lib, synthetic
    from ramannoodle_b200.distributed import ShardedTrajectory, shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _lib.require_device(local_rank)

    structure, kind, _, _, desc = WORKLOADS[args.workload]
    total_frames, scaling = workload_frames(args, world)
    start, stop = shard_bounds(total_frames, world, rank)
    frames = stop - start
    force_dense = args.workload == "c3dense"
    state = build_state(structure, kind)
    model = (rb.ARTModel if kind == "art" else rb.InterpolationModel)(state, device=local_rank, force_dense=force_dense)
    num_atoms = state.num_atoms
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=1000 + rank, first_frame=start)
    trajectory = rb.Trajectory(positions, 1.0)  # HBM-resident (wrap runs on the device)
    del positions
    info = model.path_info()
    # N > 1: the public multi-GPU API (frames sharded, rows routed over NVLink, one shared transform)
    sharded = ShardedTrajectory(trajectory._positions_ts, 1.0, total_frames) if world > 1 else None  # pylint: disable=protected-access

    def evaluate():
        return sharded.get_raman_spectrum(model) if world > 1 else trajectory.get_raman_spectrum(model)

    def step():
        spectrum = evaluate()
        return spectrum, spectrum.measure_device()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        spectrum, (wn, inten) = step()
    barrier()

    # ---- timed region: K steps, CUDA events, max over ranks ----
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = _lib.launch_count()
    sampler.start()
    barrier()
    ev0.record()
    for _ in range(args.steps):
        spectrum, (wn, inten) = step()
    ev1.record()
    barrier()
    clocks = sampler.stop()
    launches = _lib.launch_count() - launches0
    elapsed_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([elapsed_ms, float(launches)], dtype=torch.float64, device=device)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        elapsed_ms, launches = float(tmax[0]), int(t[1])
    ms_per_step = elapsed_ms / args.steps
    value = total_frames / (ms_per_step * 1e-3)

    if args.dump_outputs and rank == 0:
        local = spectrum.local_polarizability_ts if world > 1 else spectrum._polarizability_ts  # pylint: disable=protected-access
        dump_outputs(args.dump_outputs, {"polarizability_ts": local, "wavenumbers": wn, "intensities": inten})

    # ---- parity of the timed step's own output (outside the timed region) ----
    parity = None
    if not args.no_parity:
        dense = info["dense_dofs"] > 0
        parity = check_parity(state, structure, trajectory, spectrum, wn, inten, start, rank, world,
                              blocks=4, block_frames=(64 if num_atoms > 1000 else (512 if dense else 2048)))

    # ---- per-stage device times (same stream, CUDA events) for the roofline ----
    reps = max(5, min(args.steps, 20))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    acc = np.zeros(3)
    for _ in range(reps):
        # local evaluation alone (the roofline numerator), then the sharded path, then measure.
        # A primer launch of the same evaluation runs first: the timed launches are enqueued while it
        # executes, so the events bracket kernel time, not the host's launch latency.
        trajectory.get_raman_spectrum(model)
        evs[0].record()
        staged = trajectory.get_raman_spectrum(model)
        evs[1].record()
        if world > 1:
            staged = sharded.get_raman_spectrum(model)
        evs[2].record()
        staged.measure_device()
        evs[3].record()
        torch.cuda.synchronize()
        acc += [evs[0].elapsed_time(evs[1]), evs[1].elapsed_time(evs[2]), evs[2].elapsed_time(evs[3])]
    stage = dict(zip(["polarizability_ms", "polarizability_routed_ms", "spectrum_ms"], (acc / reps).round(4).tolist()))
    shared_transform = bool(world > 1 and getattr(staged, "_context", None) is not None)

    # ---- smearing (convolve_spectrum, gaussian, width 5, default output grid) on the run's own spectrum ----
    convolve = None
    barrier()  # the other ranks idle while rank 0 smears (no competing host / NVLink traffic)
    if rank == 0 and int(wn.shape[0]) > 0:
        rb.convolve_spectrum(wn, inten, "gaussian", 5)
        dt = float("inf")
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out_wn, _ = rb.convolve_spectrum(wn, inten, "gaussian", 5)
            torch.cuda.synchronize()
            dt = min(dt, time.perf_counter() - t0)
        evals = float(wn.shape[0]) * float(out_wn.shape[0])
        convolve = {"ms": dt * 1e3, "in_points": int(wn.shape[0]), "out_points": int(out_wn.shape[0]),
                    "kernel_evaluations": evals, "evaluations_per_s": evals / dt,
                    "note": "convolve_spectrum(gaussian, width=5, default grid), device inputs -> numpy output, best of 3; "
                            "(input chunk, output tile) pairs beyond 39 widths are skipped (exactly 0 in fp64)"}

    barrier()
    hbm_peak, hbm_src = measured_peaks()
    if info["dense_dofs"] == 0:
        alg_bytes = (24 * num_atoms + 72) * frames  # read positions once, write alpha once (SURVEY.md §8d)
        achieved = alg_bytes / (stage["polarizability_ms"] * 1e-3) / 1e9
        kernel_name = "affine_tma_kernel" if info["tma_affine"] else "affine_generic_kernel"
        roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "peak_source": hbm_src,
                    "algorithmic_bytes_per_frame": 24 * num_atoms + 72,
                    "traffic": ncu_traffic(kernel_name, args.workload)}
    else:
        peak_tf, peak_src = fp64_peak()
        flops = 2.0 * 3 * num_atoms * info["dense_dofs"] * frames
        achieved = flops / (stage["polarizability_ms"] * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "dense_kernel_tp", "achieved": achieved, "peak": peak_tf,
                    "unit": "TFLOP/s", "frac": achieved / peak_tf, "peak_source": peak_src + " (FP64 tensor pipe)",
                    "algorithmic_flops_per_frame": 2 * 3 * num_atoms * info["dense_dofs"],
                    "traffic": ncu_traffic("dense_kernel_tp", args.workload)}

    # ---- end to end through the public API with host buffers (H2D + D2H inside the timed region) ----
    e2e = None
    host_bytes = frames * num_atoms * 24
    if not args.no_e2e and host_bytes <= (12 << 30):
        host_traj = rb.Trajectory(trajectory.positions_ts, 1.0)  # pinned host copy (wrap is idempotent)
        assert not host_traj.is_device_resident
        host_sharded = ShardedTrajectory(host_traj._positions_ts, 1.0, total_frames) if world > 1 else None  # pylint: disable=protected-access

        def e2e_step():
            # chunked H2D overlapped with evaluation (and, N > 1, with the routed peer stores);
            # rank 0 copies the spectrum to the host, the other ranks keep theirs on the device
            spec = (host_sharded if world > 1 else host_traj).get_raman_spectrum(model)
            return spec.measure() if rank == 0 else spec.measure_device()

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            wn_h, inten_h = e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        tt = torch.tensor([dt], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": total_frames / float(tt[0]), "unit": "frames/s",
               "h2d_bytes_per_step": int(total_frames * num_atoms * 24),
               "d2h_bytes_per_step": int(2 * 8 * wn_h.shape[0]),  # (wavenumbers, intensities) on rank 0
               "ms_per_step": float(tt[0]) * 1e3, "steps": args.e2e_steps,
               "api": "Trajectory(host pinned).get_raman_spectrum(model).measure() -> numpy (N > 1: ShardedTrajectory; "
                      "the spectrum is copied to the host on rank 0)"}
        del host_traj

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = args.cpu_sample if num_atoms < 1000 else 64
        path = CpuPath(structure, "art" if force_dense else kind, 1)
        rate, detail = path.step(sample, total_frames)
        cpu_baseline = {"value": rate, "unit": "frames/s", "cores": 1, "kind": "port",
                        "sample": f"oracle numpy/scipy port, single process (as the reference ships): calc_polarizabilities "
                                  f"on {detail['sample_frames']} frames of the same synthetic workload extrapolated linearly "
                                  f"to {total_frames}, + md_measure on a {detail['measure_frames']}-frame series: {detail}"}

    if rank == 0:
        line = {
            "metric": "md_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "frames_per_gpu": frames, "total_frames": total_frames,
                       "atoms": num_atoms, "dofs": state.num_dofs, "path": info,
                       "l2": "inputs larger than L2 (no flush needed)" if frames * num_atoms * 24 > 2 * 126e6
                             else "inputs smaller than L2: cache-resident between steps",
                       "stages": stage, "shared_transform": shared_transform},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks, "e2e": e2e, "parity": parity,
            "convolve": convolve, "gpu_launches": int(launches),
        }
        sys.stdout.flush()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

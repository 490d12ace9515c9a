"""Per-phase device times of the shared multi-GPU spectrum (launch with torchrun): evaluation + routed
peer stores, pack, transform, final, combine and the barriers between them, CUDA events on rank 0's
stream (every rank runs the same schedule).  python -m torch.distributed.run ... tools/dist_breakdown.py [FRAMES_PER_GPU]"""
import ctypes
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import _lib, synthetic  # noqa: E402
from ramannoodle_b200.distributed import ShardedTrajectory, shard_bounds  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
device = torch.device(f"cuda:{local}")
dist.init_process_group("nccl", device_id=device)
per_gpu = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
total = per_gpu * world
start, stop = shard_bounds(total, world, rank)
state = synthetic.make_model("LLZO", "art")
model = rb.ARTModel(state, device=local)
block = synthetic.make_trajectory_cuda("LLZO", stop - start, device, seed=1000 + rank, first_frame=start)
sharded = ShardedTrajectory(block, 1.0, total)
spectrum = sharded.get_raman_spectrum(model)
spectrum.measure_device()
ctx = spectrum._context  # pylint: disable=protected-access
lib = _lib.lib()
stream = _lib.current_stream(local)
points = int(lib.rn_spectrum_num_points(total))
wn = torch.empty(points, dtype=torch.float64, device=device)
inten = torch.empty(points, dtype=torch.float64, device=device)
group = ctx.transform_ranks
peers = [0 if r == rank else ctx.ptr(r, "series") for r in range(world)]
positions = sharded.local._positions_ts  # pylint: disable=protected-access

phases = {
    "eval_routed": lambda: model.calc_polarizabilities_routed(positions, ctx.ptr(rank, "series") + start * 72, peers,
                                                              start, ctx.period, ctx.width),
    "barrier_0": ctx.barrier,
    "pack": lambda: lib.rn_spectrum_dist_pack(ctx.plan, ctypes.c_void_p(ctx.ptr(rank, "series")), ctx.table("work", group),
                                                 ctx.table("spectrum", world), world, -1, -1, stream),
    "barrier_1": ctx.barrier,
    "transform": lambda: lib.rn_spectrum_dist_transform(ctx.plan, ctypes.c_void_p(ctx.ptr(rank, "work")), ctx.table("recv", group), -1, stream),
    "barrier_2": ctx.barrier,
    "final": lambda: lib.rn_spectrum_dist_final(ctx.plan, ctypes.c_void_p(ctx.ptr(rank, "recv")), ctypes.c_void_p(ctx.ptr(rank, "spectrum")),
                                                ctx.table("spectrum", world), world, 1.0, 0, 0.0, 0, 0.0,
                                                ctypes.c_void_p(wn.data_ptr()) if rank < group else None, stream),
    "barrier_3": ctx.barrier,
    "finish": lambda: lib.rn_spectrum_dist_finish(ctx.plan, ctypes.c_void_p(ctx.ptr(rank, "spectrum")), 1.0,
                                                  None if rank < group else ctypes.c_void_p(wn.data_ptr()),
                                                  ctypes.c_void_p(inten.data_ptr()), stream),
}
names = list(phases)
reps = 20
acc = {name: 0.0 for name in names}
for it in range(reps + 3):
    events = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
    dist.barrier()
    torch.cuda.synchronize()
    events[0].record()
    for index, name in enumerate(names):
        phases[name]()
        events[index + 1].record()
    torch.cuda.synchronize()
    if it >= 3:
        for index, name in enumerate(names):
            acc[name] += events[index].elapsed_time(events[index + 1]) / reps
# barrier alone, back to back
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(100):
    ctx.barrier()
e1.record()
torch.cuda.synchronize()
acc["barrier_back_to_back"] = e0.elapsed_time(e1) / 100
acc["total"] = sum(acc[name] for name in names)
out = torch.tensor([acc[k] for k in acc], dtype=torch.float64, device=device)
gathered = [torch.empty_like(out) for _ in range(world)]
dist.all_gather(gathered, out)
if rank == 0:
    table = {k: [round(float(g[i]), 4) for g in gathered] for i, k in enumerate(acc)}
    print(json.dumps({"world": world, "frames_per_gpu": per_gpu, "lean": os.environ.get("RN_FFT_LEAN", "0"),
                      "ms_by_rank": table}), flush=True)
dist.destroy_process_group()

"""Multi-GPU parity check of OPEN scenes (particle sources, motored / free bodies, removal), under torchrun on a box
with >= 2 GPUs:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tests/mgpu_open_check.py                       # SC_TRANSPORT=p2p for the direct NVLink transport

Every rank runs its strip of the scene; rank 0 also runs the whole scene as one rank (world_size 1, bit-identical to
`Crate(noise="counter")`, tests/test_strips_open_gpu.py).  The gathered N-rank state must equal it bit for bit.  Cases:
wave_machine (600 ticks, fp64) and stirring_cup (400 ticks, fp64) as recorded, and the synthetic wave_tank at about
4M particles for 200 ticks (mixed precision), whose max_particles is set so that the emission clamp may bind from
about tick 100 on: the device time per tick (CUDA events on the launch stream, no host wait) is reported separately
for ticks with and without the scene-count all-reduce, on N GPUs and on one.  Prints one line per check and exits
non-zero on failure."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import world_from_freerun  # noqa: E402
from sand_crate_b200.scenes import wave_tank  # noqa: E402
from sand_crate_b200.strips import StripDomain, even_cuts  # noqa: E402

SEED = 5


def timed_run(dom, ticks, stream):
    """Step `ticks` ticks; per tick the device time between two events on the launch stream, and whether the tick took
    the scene count (ticks of the last 10 % and the first 10 are left out of the means: start-up and drain)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(ticks + 1)]
    counted = []
    ev[0].record(stream)
    for t in range(ticks):
        before = dom.scene_counts
        dom.physics_tick()
        ev[t + 1].record(stream)
        counted.append(dom.scene_counts > before)
    stream.synchronize()
    ms = np.array([ev[t].elapsed_time(ev[t + 1]) for t in range(ticks)])
    keep = np.arange(ticks) >= 10
    with_c, without = keep & np.array(counted), keep & ~np.array(counted)
    return {"ticks_with_count": int(np.sum(counted)),
            "ms_with_count": round(float(ms[with_c].mean()), 4) if with_c.any() else None,
            "ms_without_count": round(float(ms[without].mean()), 4) if without.any() else None}


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    transport = os.environ.get("SC_TRANSPORT", "nccl")
    n_tank = int(os.environ.get("SC_TANK_PARTICLES", 4_000_000))
    ok = True
    if rank == 0:
        print(f"[mgpu-open] {torch.cuda.get_device_name(local)} x {world}, transport={transport}", flush=True)

    def shipped(name):
        w, _ = world_from_freerun(name)
        return w, None, None

    def tank():
        w, p, v = wave_tank(n_tank)
        c = w.coefficients
        s = w.particle_sources[0]
        c["max_particles"] = int(n_tank + 100 * s["flow"] * c["dt"])   # the clamp may bind from about tick 100
        return w, p, v

    cases = [("wave_machine", shipped, 600, "f64"), ("stirring_cup", shipped, 400, "f64"), ("wave_tank", tank, 200, "mixed")]
    for name, make, ticks, precision in cases:
        w, pos, vel = make(name) if make is shipped else make()
        cuts = None
        if name == "wave_machine":   # through the liquid that pools at the floor (rows 78 .. 100)
            cuts = even_cuts(78, 24, world)
        dom = StripDomain(w, pos, vel, rank=rank, world_size=world, precision=precision, noise="counter",
                          noise_seed=SEED, device=local, stream=stream.cuda_stream, transport=transport, cuts=cuts,
                          slack=2.0)
        timing = timed_run(dom, ticks, stream)
        st = dom.status()
        uid, gp, gv = dom.gather()
        info = [None] * world
        dist.all_gather_object(info, (st, timing, dom.halo_rows))
        dom.close()
        if rank == 0:
            single = StripDomain(w, pos, vel, rank=0, world_size=1, precision=precision, noise="counter",
                                 noise_seed=SEED, device=local, stream=stream.cuda_stream)
            t1 = timed_run(single, ticks, stream)
            suid, sp, sv = single.gather()
            single.close()
            same = np.array_equal(uid, suid) and np.array_equal(gp, sp) and np.array_equal(gv, sv)
            flags = any(s["overflow"] or s["too_far"] for s, _, _ in info)
            print(f"[mgpu-open] {name} n={len(suid)} ticks={ticks} {precision} ranks={world} halo={info[0][2]}: "
                  f"bit-identical to one GPU = {same}; flags = {flags}; local = {[s['n_local'] for s, _, _ in info]}",
                  flush=True)
            print("[mgpu-open]   tick time " + json.dumps({"gpus": world, **info[0][1], "one_gpu": t1}), flush=True)
            ok = ok and same and not flags and len(suid) > 0
    res = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(res, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(res.item()) else 1)


if __name__ == "__main__":
    main()

"""Throughput of ensembles against separate Crates stepped in turn.

    python profiles/scripts/ensemble_throughput.py [--ticks 200] [--warmup 300] [--out FILE]

Scenes: wave_machine and stirring_cup (the recorded configs of tests/golden), mixed precision, counter noise, seed
replicas M in {1, 8, 48, 256, 1024}.  Per M: wall-clock ms per tick of Ensemble.physics_tick() over a window of
`--ticks` ticks that ends in a device synchronize (after `--warmup` ticks: both scenes' sources are still running or
just finished, so the live counts are the shipped configs' working sizes), the same for M separate Crates stepped in
turn (M <= 48), particle-steps/s (the sum of the members' live counts after each tick of the window, read after the
window from a second, identical and deterministic run of the window's ticks), launches per tick (sc_launch_count) and
the host waits the window's ticks made (sc_sync_count, without the synchronize that closes the window).  The device name
and power limit are read in the same run.  Needs a B200.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import world_from_freerun  # noqa: E402
from sand_crate_b200 import Crate, Ensemble  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return name, power


def time_ensemble(world, M, warmup, ticks):
    ens = Ensemble(world, M, precision="mixed", noise="counter")
    try:
        for _ in range(warmup):
            ens.physics_tick()
        ens.synchronize()
        l0, s0 = ens.launch_count(), ens.sync_count()
        t0 = time.perf_counter()
        for _ in range(ticks):
            ens.physics_tick()
        launches, syncs = ens.launch_count() - l0, ens.sync_count() - s0   # (before the window's own synchronize)
        ens.synchronize()
        dt = time.perf_counter() - t0
    finally:
        ens.close()
    # the same window again, reading the live counts after every tick (outside any timing)
    ens = Ensemble(world, M, precision="mixed", noise="counter")
    try:
        for _ in range(warmup):
            ens.physics_tick()
        steps = 0
        for _ in range(ticks):
            ens.physics_tick()
            steps += int(ens.particle_counts().sum())
    finally:
        ens.close()
    return {"ms_per_tick": 1e3 * dt / ticks, "particle_steps_per_s": steps / dt, "launches_per_tick": launches / ticks,
            "host_waits": syncs, "particles_per_tick": steps / ticks}


def time_crates(world, M, warmup, ticks):
    crates = [Crate(world, precision="mixed", noise="counter", noise_seed=s) for s in range(M)]
    try:
        for _ in range(warmup):
            for c in crates:
                c.physics_tick()
        for c in crates:
            c._ctx.synchronize()
        t0 = time.perf_counter()
        for _ in range(ticks):
            for c in crates:
                c.physics_tick()
        for c in crates:
            c._ctx.synchronize()
        return {"ms_per_tick": 1e3 * (time.perf_counter() - t0) / ticks}
    finally:
        for c in crates:
            c.close()


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--members", default="1,8,48,256,1024")
    ap.add_argument("--separate-max", type=int, default=48, help="largest M also timed as separate Crates")
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    name, power = device_info()
    lines = [f"# ensemble throughput on {name}, power limit {power}; mixed precision, counter noise, seed replicas; "
             f"{a.warmup} warm-up ticks, {a.ticks}-tick windows ending in a device synchronize"]
    results = []
    for scene in ("wave_machine", "stirring_cup"):
        world, _ = world_from_freerun(scene)
        for M in [int(x) for x in a.members.split(",")]:
            r = {"scene": scene, "M": M, "device": name, "power_limit": power}
            r["ensemble"] = time_ensemble(world, M, a.warmup, a.ticks)
            if M <= a.separate_max:
                r["separate_crates"] = time_crates(world, M, a.warmup, a.ticks)
                r["separate_over_ensemble"] = r["separate_crates"]["ms_per_tick"] / r["ensemble"]["ms_per_tick"]
            results.append(r)
            print(json.dumps(r), flush=True)
    lines += [json.dumps(r) for r in results]
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

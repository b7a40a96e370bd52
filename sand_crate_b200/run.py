"""Headless runner: `python -m sand_crate_b200.run config/stirring_cup.yaml --ticks 1200 --out run.npz`

The reference's only entry point opens a PyGame window (`src/main.py:19-23` -> `Playback.run_live_simulation`,
playback.py:51-65) and can only record rendered frames (GIF/AVI, playback.py:109-138; the particle dumps at 112-113
are commented out).  This runner drives the same `Crate(world_config).physics_tick()` loop without a display and
records what a renderer needs - positions, pressures and wall segments every `--every` ticks - so a run made on a GPU
box can be replayed anywhere (SURVEY.md section 8(f) row 2).  Output: one compressed .npz with
`ticks`, `count[t]`, `offsets[t + 1]`, `pos` (sum(count) x 2), `pressure`, `segments` (T x S x 2 x 2), `config_yaml`.

Sweeps (the shape of the reference's `src/main.py`, which runs one config under a grid of coefficient variants):
`--sweep sweep.yaml` (a mapping coefficient -> list of values; their Cartesian product) and / or `--replicas K` (K noise
seeds of each variant) run every variant as one member of a single `Ensemble`.  `--out DIR` then writes one recording
per member, `DIR/member_<m>.npz` in the format above (`load_recording` reads each), and `DIR/members.json` with each
member's overrides and seed.  The summary's ms_per_tick and particle_steps_per_sec cover the whole run, its ticks
enqueued back to back and closed by one synchronize (recorded ticks included, as for a single run; each tick's member
counts are copied on the device for the particle-step total); profiles/scripts/ensemble_throughput.py times windows
without recording.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import yaml

from . import Crate, Ensemble, load_config
from .ensemble import sweep_members


def run(config_path, ticks=None, every=10, out=None, precision="f64", noise="reference", device=0, quiet=False):
    cfg = load_config(config_path)
    ticks = int(ticks if ticks is not None else cfg.playback_config.ticks_to_record)
    crate = Crate(cfg.world_config, precision=precision, noise=noise, device=device)
    rec_ticks, counts, pos, prs, segs = [], [], [], [], []
    t0 = time.perf_counter()
    steps = 0
    for tick in range(1, ticks + 1):
        crate.physics_tick()
        steps += crate.particle_count if noise == "reference" else 0
        if out and (tick % every == 0 or tick == ticks):
            rec_ticks.append(tick)
            counts.append(crate.particle_count)
            pos.append(crate.particles.copy())
            prs.append(crate.particles_pressure.copy())
            segs.append(crate.segments.copy())
    n_final = crate.particle_count  # synchronises
    elapsed = time.perf_counter() - t0
    summary = {"config": str(config_path), "ticks": ticks, "particles_final": int(n_final),
               "seconds": round(elapsed, 3), "ms_per_tick": round(1e3 * elapsed / max(ticks, 1), 4),
               "precision": precision, "noise": noise}
    if steps:
        summary["particle_steps_per_sec"] = round(steps / elapsed, 1)
    if out:
        save_recording(out, config_path, rec_ticks, counts, pos, prs, segs, summary)
        summary["out"] = str(out)
    if not quiet:
        print(json.dumps(summary))
    crate.close()
    return summary


def save_recording(out, config_path, rec_ticks, counts, pos, prs, segs, summary):
    offsets = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
    with open(config_path) as f:
        config_yaml = f.read()
    np.savez_compressed(out, ticks=np.array(rec_ticks), count=np.array(counts), offsets=offsets,
                        pos=np.concatenate(pos) if pos else np.zeros((0, 2)),
                        pressure=np.concatenate(prs) if prs else np.zeros(0), segments=np.array(segs),
                        config_yaml=np.array(config_yaml), summary=np.array(json.dumps(summary)))


def load_sweep(path):
    with open(path) as f:
        sweep = yaml.safe_load(f) or {}
    if not isinstance(sweep, dict):
        raise ValueError(f"{path}: a sweep file is a mapping from coefficient to a list of values")
    return sweep


def run_ensemble(config_path, sweep=None, replicas=1, ticks=None, every=10, out=None, precision="f64", noise="counter",
                 device=0, quiet=False):
    """Every member of `sweep` x `replicas` (ensemble.sweep_members) as one Ensemble.  members.json is written before
    the device is touched, so a run that cannot start still documents what it was asked to run."""
    cfg = load_config(config_path)
    ticks = int(ticks if ticks is not None else cfg.playback_config.ticks_to_record)
    overrides, seeds = sweep_members(sweep, replicas)
    if out:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "members.json"), "w") as f:
            json.dump([{"member": m, "overrides": o, "seed": s} for m, (o, s) in enumerate(zip(overrides, seeds))], f,
                      indent=1)
    import torch   # a device buffer for the members' live counts of every tick
    ens = Ensemble(cfg.world_config, overrides, seeds=seeds, precision=precision, noise=noise, device=device)
    M = len(overrides)
    frames = [([], [], [], [], []) for _ in range(M)]   # ticks, counts, pos, prs, segments per member
    live = torch.zeros((max(ticks, 1), M), dtype=torch.int32, device=f"cuda:{device}")
    torch.cuda.synchronize(device)
    # one window over the whole run, closed by one synchronize, as `run` times it: the ticks are enqueued back to back
    # (each tick's counts are copied on the device, no host wait); recorded ticks read the state, which waits
    t0 = time.perf_counter()
    for tick in range(1, ticks + 1):
        ens.physics_tick()
        ens.member_counts_to(live[tick - 1])
        if out and (tick % every == 0 or tick == ticks):
            for m in range(M):
                mv = ens.member(m)
                f = frames[m]
                f[0].append(tick); f[1].append(mv.particle_count); f[2].append(mv.particles.copy())
                f[3].append(mv.particles_pressure.copy()); f[4].append(ens.segments.copy())
    ens.synchronize()
    elapsed = time.perf_counter() - t0
    steps = int(live[:ticks].sum())
    counts = ens.particle_counts()
    summary = {"config": str(config_path), "ticks": ticks, "members": M, "particles_final": int(counts.sum()),
               "seconds": round(elapsed, 3), "ms_per_tick": round(1e3 * elapsed / max(ticks, 1), 4),
               "particle_steps_per_sec": round(steps / elapsed, 1) if elapsed > 0 else None,
               "precision": precision, "noise": noise}
    if out:
        for m in range(M):
            f = frames[m]
            save_recording(os.path.join(out, f"member_{m}.npz"), config_path, f[0], f[1], f[2], f[3], f[4],
                           dict(summary, member=m, overrides=overrides[m], seed=seeds[m]))
        summary["out"] = str(out)
    if not quiet:
        print(json.dumps(summary))
    ens.close()
    return summary


def load_recording(path):
    """Frames of a recording made by `run`: yields (tick, positions, pressures, segments)."""
    z = np.load(path, allow_pickle=False)
    off = z["offsets"]
    for k, tick in enumerate(z["ticks"]):
        yield int(tick), z["pos"][off[k]:off[k + 1]], z["pressure"][off[k]:off[k + 1]], z["segments"][k]


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("config")
    ap.add_argument("--ticks", type=int, default=None, help="default: playback.ticks_to_record of the config")
    ap.add_argument("--every", type=int, default=10, help="record every N ticks")
    ap.add_argument("--out", default=None)
    ap.add_argument("--precision", default="f64", choices=["f64", "mixed"])
    ap.add_argument("--noise", default=None, choices=["reference", "counter", "none"],
                    help="default: reference; counter for a sweep (an ensemble cannot take the reference stream)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--sweep", default=None, help="YAML mapping coefficient -> list of values: run their product")
    ap.add_argument("--replicas", type=int, default=None, help="noise seeds per variant (0 .. K - 1)")
    a = ap.parse_args(argv)
    if a.sweep is None and a.replicas is None:
        return run(a.config, a.ticks, a.every, a.out, a.precision, a.noise or "reference", a.device)
    if a.noise == "reference":
        ap.error("--sweep / --replicas run one Ensemble, whose noise is counter or none")
    return run_ensemble(a.config, load_sweep(a.sweep) if a.sweep else None, a.replicas or 1, a.ticks, a.every, a.out,
                        a.precision, a.noise or "counter", a.device)


if __name__ == "__main__":
    main(sys.argv[1:])

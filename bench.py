#!/usr/bin/env python
"""bench.py - particle-steps/sec of the SandCrate step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--particles P] [--scene dam_break|box_fill|dam_break_wide]
    python bench.py --dump-outputs DIR ...      # also write the state after the last timed step as DIR/*.npy
    python bench.py --impl reference ...        # the reference's CPU step on the host cores (same scene mapping)

One "step" = one `physics_tick` over the whole synthetic scene.
  N = 1: dam-break, 1M particles (BASELINE.json configs[2]).
  N > 1: one scene cut into horizontal strips of cell rows, one rank per GPU; default box-fill, 2M particles per GPU
         (configs[3]: 16M on 8 GPUs); `--scene dam_break_wide --particles 8000000` = configs[4] (64M on 8 GPUs).
The scene is first RELAXED for `--relax` ticks (default 100, SURVEY.md section 8(d): part of the scene, never timed and
independent of --warmup), then W warm-up ticks, then K timed ticks.  Timed with CUDA events on the stream the kernels
are launched on; L2 is flushed between timed steps.  Prints ONE JSON line.

--dump-outputs DIR: what the caller of the timed path holds after the last timed step, in float64, rows in ascending
uid (the particle's insertion index): uid.npy, positions.npy, velocities.npy and, on one GPU, pressure.npy.  Where
those would exceed DUMP_BYTES (64 MB, headers included), only the rows of a fixed, seeded sample of uids are written.
The scene is seeded, so the same arguments give the same inputs on every run and two builds can be compared file by
file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle_steps_per_sec"
UNIT = "particle-steps/s"
# SURVEY.md section 8(d): algorithmic bytes per particle per kernel for the mixed layout (pos f64x2, vel f32x2, id, p, s,
# cell id), each record moved once per kernel.  These are the figures `roofline.achieved` is computed from.
SURVEY_BYTES = {"prepass_wall_key": 20, "place": 14, "rank_gather": 56, "density": 28, "force_integrate": 60}
DEFAULT_PARTICLES = 1_000_000
DUMP_BYTES = 64_000_000   # all files of --dump-outputs together: 64 MB, so also under 64 MiB
NPY_HEADER_BYTES = 4096   # allowance per file; np.save writes a 128-byte header for these arrays
DUMP_SEED = 0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload(a, world_size):
    """(scene name, particles per GPU, total particles) - ONE mapping for both arms."""
    if world_size == 1:
        return a.scene, a.particles, a.particles
    default = a.scene == "dam_break" and a.particles == DEFAULT_PARTICLES
    scene = "box_fill" if default else a.scene
    per_gpu = a.mgpu_particles if a.particles == DEFAULT_PARTICLES else a.particles
    return scene, per_gpu, per_gpu * world_size


def scene_params(world):
    c = world.coefficients
    return dict(dt=c["dt"], particle_radius=c["particle_radius"], wall_collision_decay=c["wall_collision_decay"],
                pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                gravity_x=c["gravity"][0], gravity_y=c["gravity"][1])


def coeff_vec(world):
    p = scene_params(world)
    return np.array([p[k] for k in ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier",
                                    "ignored_pressure", "collider_noise_level", "viscosity", "surface_smoothing",
                                    "target_pressure", "gravity_x", "gravity_y")])


def dump_sample(n_total, cols, budget=DUMP_BYTES):
    """The uids (of 0 .. n_total - 1) whose rows --dump-outputs writes, so that uid.npy plus one float64 file per
    array of `cols` (name -> per-particle array) stays within `budget` bytes, headers included: None (all of them)
    when every row fits, else a sorted sample drawn with DUMP_SEED, the same on every run and every rank."""
    row_bytes = 8 * (1 + sum(int(np.prod(v.shape[1:])) for v in cols.values()))
    k = (budget - NPY_HEADER_BYTES * (1 + len(cols))) // row_bytes
    if n_total <= k:
        return None
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n_total, size=k, replace=False))


def select_rows(uid, cols, sample):
    """The rows of the per-particle arrays `cols` (aligned with `uid`) whose uid is in `sample`, in ascending uid."""
    order = np.argsort(uid, kind="stable")
    if sample is not None:
        order = order[np.isin(uid[order], sample)]
    return uid[order], {name: v[order] for name, v in cols.items()}


def merge_rows(parts):
    """One (uid, cols) in ascending uid from the (uid, cols) of every rank."""
    return select_rows(np.concatenate([p[0] for p in parts]),
                       {k: np.concatenate([p[1][k] for p in parts]) for k in parts[0][1]}, None)


def write_dump(out_dir, uid, cols):
    os.makedirs(out_dir, exist_ok=True)
    for name, v in {"uid": uid, **cols}.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(v, dtype=np.float64))


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
            # nvidia-smi takes a few hundred ms to come up and the timed region is short: wait for its first line
            t0 = time.perf_counter()
            while time.perf_counter() - t0 < 5.0 and os.path.getsize(self.path) == 0:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons = [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9 or not f[1].isdigit():
                    continue
                sm.append(int(f[1]))
                out["sm_max_mhz"] = int(f[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm = sm[1:] if len(sm) > 2 else sm   # the first line predates the load
            out["sm_mhz"] = float(np.median(sm))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ---- CPU arms ---------------------------------------------------------------------------------------------------
def oracle_port_run(scene, n, relax, warmup, steps=None, budget_s=None):
    """The oracle port (oracle/step_oracle.c; OpenMP over particles for the force loops, scalar neighbor search) on an
    n-particle instance of `scene`: `relax` + `warmup` untimed ticks, then `steps` timed ticks (or as many as fit
    `budget_s`).  Returns (particle-steps/s, ticks, seconds, threads)."""
    from oracle import oracle as O
    from sand_crate_b200.scenes import SCENES
    world, pos, vel = SCENES[scene](n)
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    cv = coeff_vec(world)
    kin = np.zeros((1, 5))
    tick = 0

    def one():
        nonlocal pos, vel, tick
        out = O.step(cv, pos, vel, seg, [4], kin, noise_mode=1, tkey=O.tick_key(0, tick), want_all=False)
        pos, vel = out["pos_out"], out["vel_out"]
        tick += 1
    for _ in range(relax + warmup):
        one()
    t0 = time.perf_counter()
    ticks = 0
    while True:
        one()
        ticks += 1
        el = time.perf_counter() - t0
        if (steps is not None and ticks >= steps) or (budget_s is not None and (el > budget_s or ticks >= 200)):
            break
    return n * ticks / el, ticks, el, O.num_threads()


def _numpy_reference_job(args):
    """One process: the UNMODIFIED reference `Crate.physics_tick()` (shipped under baseline/_ref, loaded through
    oracle/ref_shim.py) on a synthetic block of n particles.  Returns (n, ticks, seconds)."""
    root, scene, n, ticks = args
    os.environ["SANDCRATE_REFERENCE_ROOT"] = root
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"   # the reference is single-threaded by construction; keep BLAS from pretending otherwise
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    from sand_crate_b200.scenes import SCENES
    ref = ref_shim.load_reference()
    world, pos, vel = SCENES[scene](n)
    cfg = ref.load_config(os.path.join(ref.config_dir, "wave_machine.yaml"))
    wc = cfg.world_config
    wc.rigid_bodies = world.rigid_bodies
    wc.particle_sources = []
    wc.coefficients = dict(world.coefficients)
    crate = ref.Crate(wc)
    crate.particles = pos.copy()
    crate.particle_velocities = vel.copy()
    crate.particles_pressure = np.zeros(len(pos))
    crate.physics_tick()   # warm
    t0 = time.perf_counter()
    for _ in range(ticks):
        crate.physics_tick()
    return n, ticks, time.perf_counter() - t0


def numpy_reference_block(scene):
    """BASELINE.md section 4 / SURVEY.md section 8(d): the reference's own NumPy step timed on THIS box's host cores:
    one core at P = 1k / 10k / 100k, and all cores as independent replicas (the step has no intra-tick parallelism)."""
    root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(root, "src", "crate", "crate.py")):
        return {"unavailable": "baseline/_ref/ (a copy of the reference tree made by __graft_entry__.build()) is absent"}
    import multiprocessing as mp
    ctxmp = mp.get_context("spawn")
    out = {"impl": "David-Taub/sand_crate src/crate/crate.py Crate.physics_tick(), unmodified, via oracle/ref_shim.py",
           "unit": UNIT, "one_core": {}}
    try:
        with ctxmp.Pool(1) as pool:
            for n, ticks in ((1_000, 5), (10_000, 3), (100_000, 1)):
                n_, t_, s_ = pool.apply(_numpy_reference_job, ((root, scene, n, ticks),))
                out["one_core"][str(n)] = {"value": n_ * t_ / s_, "ticks": t_, "seconds": round(s_, 3)}
        cores = os.cpu_count() or 1
        with ctxmp.Pool(cores) as pool:
            t0 = time.perf_counter()
            res = pool.map(_numpy_reference_job, [(root, scene, 10_000, 2)] * cores)
            wall = time.perf_counter() - t0
        out["all_cores_replicas"] = {"cores": cores, "particles_per_replica": 10_000, "ticks": 2,
                                     "value": sum(n * t / s for n, t, s in res), "wall_s_incl_startup": round(wall, 2)}
    except Exception as e:  # the block is informative; the arm's own value does not depend on it
        out["error"] = f"{type(e).__name__}: {e}"
    return out


def run_reference_arm(a):
    """`--impl reference`: the reference's CPU implementation of the path on this box's host cores, same scene mapping
    as the GPU arm.  The arm's value is the oracle port (all OpenMP threads) on a bounded sample of the workload; the
    unmodified NumPy reference, which is ~350x slower per core, is timed beside it (`numpy_reference`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    scene, per_gpu, n_total = workload(a, max(world_size, a.gpus))
    n = a.cpu_particles
    value, ticks, el, cores = oracle_port_run(scene, n, min(a.relax, 5), a.warmup, steps=a.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * el / ticks, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{scene} {n_total} particles (CPU sample: {n} particles; cost per particle is flat in P)",
                   "scene": scene, "particles_total": n_total, "particles_per_gpu": per_gpu},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{scene} {n} particles x {ticks} ticks, oracle/step_oracle.c, {cores} OpenMP threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host": {"cpu_count": os.cpu_count()},
    }
    if not a.no_numpy_reference and world_size == 1:   # once per round is enough: it does not depend on N
        line["numpy_reference"] = numpy_reference_block(scene)
    emit(line)


def emit(line: dict) -> None:
    """The ONE JSON line, written to the process's original stdout (see main: libraries such as NCCL print banners
    to fd 1, so everything else is sent to stderr)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def load_traffic():
    """ncu `dram__bytes_read.sum + dram__bytes_write.sum` per launch and the same capture's kernel durations
    (profiles/traffic.json, written by profiles/ncu_summary.py from the committed ncu CSV of this bench command)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # anything a library prints to stdout from here on goes to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed ticks (default 200; 20 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up ticks (default 10; 3 with --impl reference)")
    ap.add_argument("--relax", type=int, default=100, help="untimed relaxation ticks that are part of the scene")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="dam_break", choices=["dam_break", "box_fill", "dam_break_wide"])
    ap.add_argument("--particles", type=int, default=DEFAULT_PARTICLES, help="particles (per GPU when --gpus > 1)")
    ap.add_argument("--precision", default="mixed", choices=["mixed", "f64"])
    ap.add_argument("--transport", default="auto", choices=["auto", "nccl", "p2p"], help="strip exchange: NCCL send/recv or "
                    "direct NVLink stores into the neighbor's symmetric-memory buffer")
    ap.add_argument("--rebalance-every", type=int, default=250, help="strips: first work-weighted re-cut of the partition "
                    "after N ticks (0 = never); the interval then adapts to how far the cuts were found from their targets "
                    "and to what a re-cut costs (it drains the stream: histogram to the host, all-reduce)")
    ap.add_argument("--rebalance-fixed", action="store_true", help="strips: re-cut every --rebalance-every ticks exactly")
    ap.add_argument("--halo-rows", type=int, default=4)
    ap.add_argument("--mgpu-particles", type=int, default=2_000_000, help="particles per GPU when --gpus > 1")
    ap.add_argument("--cpu-particles", type=int, default=200_000)
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numpy-reference", action="store_true")
    ap.add_argument("--no-weak-baseline", action="store_true", help="N > 1: skip the same-scene 1-GPU baseline on rank 0")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state after the last timed step as DIR/<name>.npy "
                    "(float64, at most 64 MB in all; see the module docstring)")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        if a.dump_outputs:
            ap.error("--dump-outputs applies to the GPU arm")
        if a.steps is None:  # the GPU arm's default would keep the CPU arm busy for minutes; about one is enough
            a.steps = 20
        a.warmup = 3 if a.warmup is None else max(a.warmup, 1)
        return run_reference_arm(a)
    a.steps = 200 if a.steps is None else a.steps
    a.warmup = 10 if a.warmup is None else max(a.warmup, 3)

    import torch
    import torch.distributed as dist
    from sand_crate_b200 import Crate, _lib
    from sand_crate_b200.scenes import SCENES, scene_chunks

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    numa = None
    if world_size > 1:
        # each rank's host buffers on the socket its GPU hangs off (the e2e leg is PCIe-bound; see bind_to_gpu_numa_node)
        from sand_crate_b200.strips import bind_to_gpu_numa_node
        numa = bind_to_gpu_numa_node(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # a non-default torch stream: the library launches on it and torch.cuda.Event records on it (handle 0, the
    # legacy default stream, would make sc_create open a private stream that torch events cannot see)
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    precision = _lib.PRECISION_MIXED if a.precision == "mixed" else _lib.PRECISION_F64
    scene, n, n_total = workload(a, world_size)
    flush = None if a.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def single_gpu_context(scene_name, count):
        world_, pos_, vel_ = SCENES[scene_name](count)
        c_ = _lib.Context(count, precision, local_rank, stream)
        c_.set_params(**scene_params(world_))
        seg = np.array(world_.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
        c_.set_walls(seg, [4], np.zeros((1, 5)))
        c_.set_noise(_lib.NOISE_COUNTER, 0)
        c_.set_state(pos_, vel_)
        return world_, c_

    def timed_pass(ctx_, step_fn_, profile, sync_all=True):
        """K steps, each bracketed by CUDA events on the launch stream, L2 flushed (untimed) before each."""
        ctx_.profile_enable(profile)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
        barrier() if sync_all else torch.cuda.synchronize()
        w0 = time.perf_counter()
        for e0, e1 in ev:
            if flush is not None:
                flush.fill_(1)          # untimed: evicts the previous step's lines from the 126 MB L2
            e0.record()
            step_fn_()
            e1.record()
        barrier() if sync_all else torch.cuda.synchronize()
        w = time.perf_counter() - w0
        ms = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
        kern = ctx_.profile_read() if profile else {}
        ctx_.profile_enable(False)
        return float(ms.sum()), w, kern

    dom = None
    if world_size == 1:
        world, ctx = single_gpu_context(scene, n)
        step_fn = ctx.step
    else:
        from sand_crate_b200.strips import StripDomain
        world, chunks = scene_chunks(scene, n_total)
        dom = StripDomain(world, rank=rank, world_size=world_size, precision=a.precision, noise="counter",
                          device=local_rank, stream=stream, transport=a.transport,
                          rebalance_every=a.rebalance_every, chunks=chunks, halo_rows=a.halo_rows,
                          adaptive_rebalance=not a.rebalance_fixed,
                          check_every=0)   # the device flags are reported in the line (`strips`), not raised mid-run
        ctx = dom.ctx
        step_fn = dom.physics_tick

    for _ in range(a.relax + a.warmup):   # relaxation is part of the scene; then W warm-up ticks
        step_fn()
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launch_count()
    # pass 1 = THE timed region (value, ms_per_step): plain launches, nothing but the step kernels on the stream
    total_ms, wall, _ = timed_pass(ctx, step_fn, False)
    launches = ctx.launch_count() - launches0
    dumped = None
    if a.dump_outputs:   # read back now: the passes below step the scene further
        if dom is None:
            pos_d, vel_d, prs_d = ctx.get_state()
            uid_d, cols = ctx.get_uids(), {"positions": pos_d, "velocities": vel_d, "pressure": prs_d}
        else:
            pos_d, vel_d, uid_d = ctx.dist_get_owned()
            cols = {"positions": pos_d, "velocities": vel_d}
        dumped = select_rows(uid_d, cols, dump_sample(n_total, cols))
        if world_size > 1:   # only rank 0 writes
            parts = [None] * world_size if rank == 0 else None
            dist.gather_object(dumped, parts, dst=0)
            dumped = merge_rows(parts) if rank == 0 else None
    # pass 2 = the same K steps again with a CUDA-event pair around every kernel launch (per-kernel durations for
    # the roofline); the extra event records stretch the gaps between kernels, so its step time is not the headline
    total_ms_prof, _, kernels = timed_pass(ctx, step_fn, True)
    clocks = sampler.stop()
    status = {"overflow": False, "too_far": False, "n_local": ctx.particle_count()} if dom is None else dom.status()
    n_live = status["n_local"]
    n_pairs = ctx.last_pair_count()
    mean_pairs = n_pairs / max(n_live, 1)   # directed pairs per local particle of the last tick (ghosts included)
    untiled = ctx.untiled_blocks()

    t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = n_total * a.steps / (total_ms_max * 1e-3)
    per_rank = None
    if world_size > 1:
        per_rank = [None] * world_size
        dist.all_gather_object(per_rank, {"rank": rank, "n_local": int(n_live), "ms_per_step": total_ms / a.steps,
                                          "overflow": bool(status["overflow"]), "too_far": bool(status["too_far"]),
                                          "rows": [int(dom.row_lo), int(dom.row_hi)], "mean_pairs": mean_pairs,
                                          "host_affinity": numa})

    # ---- N > 1: the same per-GPU workload on ONE GPU, inside this invocation, as the weak-scaling baseline ---------
    # (only for box-fill: a dam break of 1/N the particles in the same box is a different column - fewer, larger
    # particles, another hydrostatic load - not 1/N of the work)
    weak = None
    if world_size > 1 and not a.no_weak_baseline and scene == "box_fill":
        if rank == 0:
            _, c1 = single_gpu_context(scene, n)
            for _ in range(a.relax + a.warmup):
                c1.step()
            ms1, _, _ = timed_pass(c1, c1.step, False, sync_all=False)
            weak = ms1 / a.steps
            c1.close()
        barrier()

    # ---- e2e: the public API with host buffers: upload state, tick, read the result back, every step ----------
    if dom is None:
        crate = Crate(world, precision=a.precision, noise="counter", device=local_rank, capacity=n, stream=stream)
        hp = torch.empty((n, 2), dtype=torch.float64, pin_memory=True).numpy()
        hv = torch.empty((n, 2), dtype=torch.float64, pin_memory=True).numpy()
        gp, gv, _ = ctx.get_state(want_pressure=False)
        hp[:], hv[:] = gp, gv

        def e2e_step():
            crate.set_particles(hp, hv)
            crate.physics_tick()
            return crate.particles
        e2e_api = "Crate.set_particles(host, page-locked) -> physics_tick() -> Crate.particles (host, page-locked)"
    else:
        gp, gv, uid0 = dom.ctx.dist_get_owned()
        m = len(uid0)
        hp = torch.empty((m, 2), dtype=torch.float64, pin_memory=True).numpy()
        hv = torch.empty((m, 2), dtype=torch.float64, pin_memory=True).numpy()
        hp[:], hv[:] = gp, gv
        del gp, gv

        def e2e_step():
            dom.ctx.set_state_uids(hp, hv, uid0)
            dom.physics_tick()
            return dom.ctx.dist_get_owned(want_vel=False, want_uid=False, reuse=True)[0]
        e2e_api = ("Context.set_state_uids(host, page-locked) -> StripDomain.physics_tick() -> "
                   "dist_get_owned (positions, host, page-locked), per rank")
    for _ in range(3):
        out_pos = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        out_pos = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_total * a.e2e_steps / float(t.item())
    assert np.isfinite(out_pos).all()
    h2d = torch.tensor([float(hp.nbytes + hv.nbytes), float(out_pos.nbytes)], device="cuda", dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(h2d)
    h2d_bytes, d2h_bytes = int(h2d[0].item()), int(h2d[1].item())

    if dumped is not None and rank == 0:
        write_dump(a.dump_outputs, *dumped)
    if rank == 0:
        peak, peak_src = peaks()
        top = max((k for k in kernels if k in SURVEY_BYTES), key=lambda k: kernels[k]["ms"], default="density")
        k = kernels.get(top, {"launches": 1, "ms": float("nan")})
        k_ms = k["ms"] / max(k["launches"], 1)
        achieved = SURVEY_BYTES[top] * n_live / (k_ms * 1e-3) / 1e9
        traffic_all = load_traffic()
        tr = traffic_all.get(top) if isinstance(traffic_all.get(top), dict) else None
        per_kernel = {}
        for name, v in kernels.items():
            ms = v["ms"] / max(v["launches"], 1)
            per_kernel[name] = {"ms": round(ms, 5), "launches_per_step": round(v["launches"] / a.steps, 2)}
            if name in SURVEY_BYTES:
                gbs = SURVEY_BYTES[name] * n_live / (ms * 1e-3) / 1e9
                per_kernel[name]["algo_gbs"] = round(gbs, 1)
                per_kernel[name]["frac"] = round(gbs / peak, 4)
        step_ms = total_ms_max / a.steps
        if dom is None:
            parallelism = "single GPU"
        else:
            how = ("direct NVLink stores into the neighbor's symmetric-memory buffer + release/acquire flags (no NCCL call "
                   "per tick)" if dom.transport == "p2p" else "NCCL send/recv (batch_isend_irecv)")
            parallelism = (f"{world_size} horizontal strips of cell rows, halo + migration exchange with rank+-1 every "
                           f"tick by {how}; halo {dom.halo_rows} rows, wire buffer {dom.wire_capacity} records, work-weighted "
                           f"re-cut, interval " + (f"fixed at {a.rebalance_every}" if a.rebalance_fixed else
                                                  f"adaptive from {a.rebalance_every or 'never'} (now {dom.rebalance_every})"))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 forces / f64 positions" if a.precision == "mixed" else "f64", "data": "synthetic",
            "config": {"workload": f"{scene} {n_total} particles ({n} per GPU), closed unit box, counter noise 0.1, "
                                   f"{a.relax} relaxation ticks before the warm-up",
                       "scene": scene, "particles_total": n_total, "particles_per_gpu": n, "relax_ticks": a.relax,
                       "local_particles_rank0": n_live, "mean_pairs_per_particle": round(mean_pairs, 3),
                       "untiled_density_blocks": untiled,
                       "parallelism": parallelism,
                       "l2": "flushed between timed steps (256 MiB write)" if flush is not None else "not flushed",
                       "timing": "CUDA events per step on the launch stream, summed; max over ranks"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "steps": a.e2e_steps, "api": e2e_api},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None if tr is None else tr.get("dram_bytes"),
                         "peak_source": peak_src, "algorithmic_bytes_per_particle": SURVEY_BYTES[top],
                         "algorithmic_bytes_per_launch": SURVEY_BYTES[top] * n_live, "kernel_ms": k_ms,
                         "traffic_source": None if tr is None else {
                             k2: tr.get(k2) for k2 in ("ncu_csv", "ncu_kernel_us", "particles", "note")},
                         "whole_step": {"survey_bytes_per_particle": 178,
                                        "achieved": 178 * n_live / (step_ms * 1e-3) / 1e9,
                                        "frac": 178 * n_live / (step_ms * 1e-3) / 1e9 / peak}},
            "kernels": per_kernel,
            "wall_s_timed_region": wall,
            "ms_per_step_with_per_kernel_events": total_ms_prof / a.steps,
        }
        if numa is not None:
            line["config"]["host_affinity_rank0"] = numa
        if per_rank is not None:
            nl = [p["n_local"] for p in per_rank]
            line["strips"] = {"n_local_min": min(nl), "n_local_max": max(nl),
                              "imbalance": round(max(nl) / (sum(nl) / len(nl)), 4),
                              "overflow": any(p["overflow"] for p in per_rank),
                              "too_far": any(p["too_far"] for p in per_rank), "per_rank": per_rank,
                              "recuts_tick_shift_interval_idleus_tickus": dom.rebalance_log[-12:], "recuts": len(dom.rebalance_log)}
        if weak is not None:
            line["weak_baseline_1gpu_ms"] = weak
            line["efficiency_same_scene"] = weak / step_ms
            line["config"]["weak_baseline"] = (f"{scene} {n} particles on one GPU (rank 0), same relaxation, warm-up, "
                                               f"steps and L2 flush, inside this invocation")
        if not a.no_cpu_baseline and world_size == 1:
            v, ticks, el, cores = oracle_port_run(a.scene, a.cpu_particles, 1, 1, budget_s=15.0)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{a.scene} {a.cpu_particles} particles x {ticks} ticks in {el:.1f}s, oracle/step_oracle.c, {cores} "
                          f"OpenMP threads (neighbor search scalar).  The unmodified NumPy reference is timed by "
                          f"`bench.py --impl reference` (numpy_reference block)."}
        emit(line)
    if world_size > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

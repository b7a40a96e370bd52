import glob
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def step_goldens():
    return sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, "step_*.npz")))


def neighbor_case_tags():
    g = golden("neighbors_cases.npz")
    return sorted({k.split("__")[0] for k in g.files})


def world_from_freerun(name):
    from sand_crate_b200 import WorldConfig
    g = golden(f"freerun_{name}.npz")
    w = json.loads(str(g["world_json"]))
    return WorldConfig(rigid_bodies=w["rigid_bodies"], particle_sources=w["particle_sources"],
                       coefficients=w["coefficients"]), g


def params_from_coeffs(c):
    """golden `coeffs` 11-vector (oracle.ref_shim.coefficients_of) -> sc_params keyword dict."""
    names = ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier", "ignored_pressure",
             "collider_noise_level", "viscosity", "surface_smoothing", "target_pressure", "gravity_x", "gravity_y")
    return {n: float(v) for n, v in zip(names, c)}


def aggregates(pos, vel, prs):
    """The bulk quantities the free-run drift bounds are stated on (SURVEY.md section 8(c), "1000-step free run")."""
    pos, vel, prs = np.asarray(pos), np.asarray(vel), np.asarray(prs)
    return {"count": int(len(pos)), "com_x": float(pos[:, 0].mean()), "com_y": float(pos[:, 1].mean()),
            "kinetic": float(0.5 * (vel ** 2).sum()), "mean_speed": float(np.sqrt((vel ** 2).sum(1)).mean()),
            "p_mean": float(prs.mean()), "p_max": float(prs.max())}


def oracle_counter_run(world, seed, ticks, precision_f32_vel=False):
    """The drop-in `Crate`'s production mode (counter noise, counter sources) re-stated end to end on the oracle, with
    no product code on the path except the rigid-body host logic: per tick create_new_particles (counter stream,
    oracle.emit_counter) -> body motion -> remove -> step.  Yields (tick, pos, vel, pressure) after every tick."""
    from oracle import oracle as O
    from sand_crate_b200.rigid_body import build_rigid_bodies
    c = world.coefficients
    cv = np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                   c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                   c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)
    bodies = build_rigid_bodies(world.rigid_bodies)
    pos, vel = np.zeros((0, 2)), np.zeros((0, 2))
    uid = np.zeros(0, np.uint32)
    next_uid = 0
    for tick in range(ticks):
        # sources (crate.py:138-147); identities advance by the drawn counts, like the library's
        drawn = [O.source_count(O.source_uniform(seed, tick, q, 0), s["flow"], c["dt"])
                 if s["active_ticks"] > tick else 0 for q, s in enumerate(world.particle_sources)]
        new_pos, new_vel = O.emit_counter(seed, tick, world.particle_sources, c["dt"], len(pos), c["max_particles"])
        room, ids = max(int(c["max_particles"]) - len(pos), 0), []
        for n in drawn:
            a = min(n, room)
            ids.append(np.arange(next_uid, next_uid + a, dtype=np.uint32))
            next_uid += n
            room -= a
        pos, vel = np.vstack((pos, new_pos)), np.vstack((vel, new_vel))
        uid = np.concatenate([uid] + ids)
        for b in bodies:
            b.apply_velocity(c["dt"])
        pos, vel, mask = O.remove_particles(pos, vel, c["particle_radius"])
        uid = uid[~mask]
        seg = np.vstack([b.segments for b in bodies]).reshape(-1, 4)
        out = O.step(cv, pos, vel, seg, np.array([len(b) for b in bodies], np.int32),
                     np.array([b.kinematics() for b in bodies]).reshape(-1, 5), noise_mode=1,
                     tkey=O.tick_key(seed, tick), uid=uid, want_all=True)
        pos, vel = out["pos_out"], out["vel_out"]
        yield tick + 1, pos, vel, out["pressure"]

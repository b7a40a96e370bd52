"""Open scenes on strips, CPU side: particle sources, motored bodies and removal across ranks over `torch.distributed`
(gloo, world sizes 2 to 4), the device work done by the oracle-backed test double.  The N-rank run of a shipped config
must reproduce the one-domain oracle run of the same config bit for bit: the scene-wide emission clamp (owned counts
summed by an all-reduce), identities taken from the scene-wide counter, each particle emitted by the rank that owns its
row.  The host rules (when the clamp may bind, even cuts of an empty scene) are tested on their own."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import world_from_freerun
from oracle import oracle as O
from oracle_strips_backend import OpenOracleContext
from sand_crate_b200.strips import INT64_MAX, INT64_MIN, StripDomain, emission_may_clamp, even_cuts, world_rows

SEED = 11


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _world(name, max_particles=None):
    world, _ = world_from_freerun(name)
    if max_particles is not None:
        world.coefficients["max_particles"] = max_particles
    return world


def oracle_one_domain(world, ticks):
    """The Crate's counter mode on the whole scene, restated on the oracle (conftest.oracle_counter_run, with the
    identities kept): (uid, pos, vel) after `ticks` ticks, and the ticks in which the host bound could not rule the
    max_particles clamp out."""
    from sand_crate_b200.rigid_body import build_rigid_bodies
    c = world.coefficients
    cv = np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                   c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                   c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)
    bodies = build_rigid_bodies(world.rigid_bodies)
    pos, vel, uid = np.zeros((0, 2)), np.zeros((0, 2)), np.zeros(0, np.uint32)
    next_uid, bound, may_clamp = 0, 0, 0
    for tick in range(ticks):
        drawn = [O.source_count(O.source_uniform(SEED, tick, q, 0), s["flow"], c["dt"])
                 if s["active_ticks"] > tick else 0 for q, s in enumerate(world.particle_sources)]
        if sum(drawn):
            may_clamp += emission_may_clamp(bound, sum(drawn), c["max_particles"])
            bound += sum(drawn)
        new_pos, new_vel = O.emit_counter(SEED, tick, world.particle_sources, c["dt"], len(pos), c["max_particles"])
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
                     tkey=O.tick_key(SEED, tick), uid=uid, want_all=False)
        pos, vel = out["pos_out"], out["vel_out"]
    return uid, pos, vel, may_clamp


def _worker(rank, world_size, port, name, max_particles, ticks, cuts, recut, out_dir):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        dom = StripDomain(_world(name, max_particles), rank=rank, world_size=world_size, precision="f64",
                          noise="counter", noise_seed=SEED, context_factory=OpenOracleContext,
                          tensor_device=torch.device("cpu"), cuts=cuts, rebalance_every=recut,
                          adaptive_rebalance=False)
        dom.step(ticks)
        uid, p, v = dom.gather()
        counts = [None] * world_size
        dist.all_gather_object(counts, (dom.scene_counts, dom.status()["too_far"], dom.halo_rows))
        if rank == 0:
            np.savez(os.path.join(out_dir, "out.npz"), uid=uid, pos=p, vel=v, counts=np.array(counts, np.int64))
    finally:
        dist.destroy_process_group()


CASES = [  # config, max_particles (None: the config's), ticks, world size, cuts, re-cut interval
    pytest.param("stirring_cup", None, 90, 2, None, 0, id="stirring_cup-2-even"),
    pytest.param("stirring_cup", 40, 60, 4, None, 0, id="stirring_cup-4-clamp"),
    pytest.param("wave_machine", None, 40, 3, [INT64_MIN, 80, 92, INT64_MAX], 0, id="wave_machine-3-through-source"),
    pytest.param("wave_machine", 200, 40, 2, None, 10, id="wave_machine-2-clamp-recut"),
]


@pytest.mark.parametrize("name,max_particles,ticks,world_size,cuts,recut", CASES)
def test_open_scene_on_strips_matches_one_domain(tmp_path, name, max_particles, ticks, world_size, cuts, recut):
    mp.spawn(_worker, args=(world_size, _free_port(), name, max_particles, ticks, cuts, recut, str(tmp_path)),
             nprocs=world_size, join=True)
    got = np.load(tmp_path / "out.npz")
    uid, pos, vel, may_clamp = oracle_one_domain(_world(name, max_particles), ticks)
    assert len(uid) > 0
    assert np.array_equal(got["uid"], uid), (len(got["uid"]), len(uid))
    assert np.array_equal(got["pos"], pos) and np.array_equal(got["vel"], vel)
    counts = got["counts"]
    assert (counts[:, 0] == may_clamp).all(), (counts[:, 0], may_clamp)   # one collective per such tick, every rank
    assert (may_clamp > 0) == (max_particles is not None)
    # the paddle's touch boxes overlap the box corner's: more than 2 contacts per particle, a 6-row halo
    assert not counts[:, 1].any() and (counts[:, 2] == {"stirring_cup": 4, "wave_machine": 6}[name]).all()


def test_emission_may_clamp_rule():
    assert not emission_may_clamp(0, 14, 4000) and not emission_may_clamp(3986, 14, 4000)
    assert emission_may_clamp(3987, 14, 4000) and emission_may_clamp(5000, 1, 4000)
    assert not emission_may_clamp(0, 0, 0)


def test_even_cuts_of_an_empty_scene():
    row0, nrows = world_rows(0.005)
    for n in (1, 2, 3, 4):
        cuts = even_cuts(row0, nrows, n)
        assert len(cuts) == n + 1 and cuts[0] == INT64_MIN and cuts[-1] == INT64_MAX
        inner = [row0] + cuts[1:-1] + [row0 + nrows]
        assert max(np.diff(inner)) - min(np.diff(inner)) <= 1


def test_wave_tank_scales_like_the_other_scenes():
    """The synthetic open scene: a bed of n particles, dt scaled with d, one source running 0.5 s of physical time, the
    clamp binding halfway through the source's run, and wave_machine's paddle (whose walls need a 6-row halo)."""
    from sand_crate_b200 import _lib
    from sand_crate_b200.rigid_body import build_rigid_bodies, wall_arrays
    from sand_crate_b200.scenes import wave_tank
    for n in (20_000, 80_000):
        world, pos, vel = wave_tank(n)
        c, s = world.coefficients, world.particle_sources[0]
        d = 2 * c["particle_radius"]
        assert pos.shape == (n, 2) and not vel.any()
        assert pos.min() > 0.5 * d and pos.max() < 1 - 0.5 * d and pos[:, 1].min() > 0.55
        assert c["dt"] == pytest.approx(0.002 * d / 0.01)
        assert s["active_ticks"] == round(0.5 / c["dt"]) and c["max_particles"] == int(n + 0.25 * s["flow"])
        assert [next(iter(b)) for b in world.rigid_bodies] == ["fixed", "motored"]
        assert _lib.dist_halo_rows(wall_arrays(build_rigid_bodies(world.rigid_bodies))[0], c["particle_radius"]) == 6

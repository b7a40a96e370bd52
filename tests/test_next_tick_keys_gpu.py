"""The force kernel computes the next tick's cell keys (NextKeys, sc_pair.cuh): the next tick then launches no
pre-pass.  Those keys must be the bits the pre-pass would have produced, and every call that changes what they depend
on must take them back (drop_keys, sc_api.cu).  A get_state -> set_state_uids round trip before a tick changes
nothing the tick computes, but it drops the keys: so a straight run (keys carried from tick to tick) and a run with a
round trip before every tick (pre-pass every tick) must agree bit for bit.  pytest -m gpu, B200 only."""
import numpy as np
import pytest

from oracle import oracle as O
from sand_crate_b200 import _lib
from sand_crate_b200.scenes import dam_break

pytestmark = pytest.mark.gpu


def _coeff_vec(c):
    return np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                     c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                     c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)


def _ctx(world, pos, vel, precision, seed=3):
    c = world.coefficients
    ctx = _lib.Context(len(pos), precision)
    ctx.set_params(dt=c["dt"], particle_radius=c["particle_radius"], wall_collision_decay=c["wall_collision_decay"],
                   pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                   collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                   surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                   gravity_x=c["gravity"][0], gravity_y=c["gravity"][1])
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64).reshape(-1, 4)
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))
    ctx.set_noise(_lib.NOISE_COUNTER, seed)
    ctx.set_state(pos, vel)
    return ctx, seg


def _push_again(ctx, world, seg):
    """What a Crate does every tick: the same coefficients and walls again.  Byte-identical values keep the keys."""
    c = world.coefficients
    ctx.set_params(dt=c["dt"], particle_radius=c["particle_radius"], wall_collision_decay=c["wall_collision_decay"],
                   pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                   collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                   surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                   gravity_x=c["gravity"][0], gravity_y=c["gravity"][1])
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))


def _wall_contacts(ctx):
    n = ctx.particle_count()
    return int(np.count_nonzero(ctx.get_wall_counts(n)))


@pytest.mark.parametrize("precision", [_lib.PRECISION_F64, _lib.PRECISION_MIXED])
def test_keys_carried_by_the_force_kernel_equal_the_pre_pass(precision):
    world, pos, vel = dam_break(100_000)
    straight, seg = _ctx(world, pos, vel, precision)
    tripped, _ = _ctx(world, pos, vel, precision)
    contacts = 0
    for tick in range(200):
        gp, gv, _ = tripped.get_state()
        tripped.set_state_uids(gp, gv, tripped.get_uids())   # drops the keys: this tick runs its own pre-pass
        for ctx in (straight, tripped):
            _push_again(ctx, world, seg)
            ctx.set_tick(tick)
            ctx.step()
        if tick % 50 == 49:
            contacts = max(contacts, _wall_contacts(straight))
    assert contacts > 100, "the scene must exercise the hard-wall fix"
    a, b = straight.get_state(), tripped.get_state()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(straight.get_uids(), tripped.get_uids())


def test_launches_per_tick():
    world, pos, vel = dam_break(100_000)
    ctx, seg = _ctx(world, pos, vel, _lib.PRECISION_MIXED)
    for tick in range(3):
        _push_again(ctx, world, seg)
        ctx.set_tick(tick)
        ctx.step()

    def launches_of_one_tick(tick):
        ctx.set_tick(tick)
        before = ctx.launch_count()
        ctx.step()
        return ctx.launch_count() - before

    assert launches_of_one_tick(3) == 5       # scan, place, rank + gather, density, force (+ next tick's keys)
    gp, gv, _ = ctx.get_state()               # a readback keeps the keys
    assert launches_of_one_tick(4) == 5
    ctx.set_state_uids(gp, gv, ctx.get_uids())
    assert launches_of_one_tick(5) == 6       # the pre-pass again
    assert launches_of_one_tick(6) == 6       # (the tick after a state change computes no keys for the next)
    assert launches_of_one_tick(7) == 5


def test_moved_wall_after_carried_keys_matches_oracle():
    """Keys carried into a tick whose walls moved would be stale: set_walls with a new segment takes them back."""
    world, pos, vel = dam_break(20_000)
    ctx, seg = _ctx(world, pos, vel, _lib.PRECISION_F64, seed=7)
    cv = _coeff_vec(world.coefficients)
    r = world.coefficients["particle_radius"]
    for tick in range(4):
        ctx.set_tick(tick)
        ctx.step()
    gp, gv, _ = ctx.get_state()
    uid = ctx.get_uids()
    moved = seg.copy()
    moved[3] = [0.0, 1.0 - 2.2 * r, 1.0, 1.0 - 2.2 * r]   # the floor (gravity is +y), raised under the bottom row
    ctx.set_walls(moved, [len(moved)], np.zeros((1, 5)))
    ctx.set_tick(4)
    before = ctx.launch_count()
    ctx.step()
    assert ctx.launch_count() - before == 6
    keep = (gp >= -r).all(1) & (gp <= 1 + r).all(1)
    ref = O.step(cv, gp[keep], gv[keep], moved, [len(moved)], np.zeros((1, 5)), noise_mode=1,
                 tkey=O.tick_key(7, 4), uid=uid[keep], want_all=True)
    assert np.count_nonzero(ref["wall_count"]) > 50
    p, v, prs = ctx.get_state()
    assert np.array_equal(p, ref["pos_out"]) and np.array_equal(v, ref["vel_out"])
    assert np.array_equal(prs, ref["pressure"])


def test_particles_leaving_the_box_match_oracle():
    """Particles in the two bottom corners of the box, outside both walls and beyond their touch distance: gravity
    (+y) carries them out of the box after a few ticks, and the ones started on top of each other scatter first.  From
    the third tick on, the key pass that drops them (no key, no count) is the force kernel's.  A count left above zero
    would shift the next tick's cells and break the bits."""
    world, pos, vel = dam_break(20_000)
    c = world.coefficients
    r, dt, g = c["particle_radius"], c["dt"], c["gravity"][1]
    corner = [[x, 1 + 0.98 * r] for k in range(8) for x in (1 + 0.96 * r, -0.96 * r)]
    up = [[0.0, -g * dt * (1 + 2.5 * k)] for k in range(8) for _ in range(2)]
    pos = np.concatenate((pos, np.array(corner)))
    vel = np.concatenate((vel, np.array(up)))
    ctx, seg = _ctx(world, pos, vel, _lib.PRECISION_F64, seed=11)
    cv = _coeff_vec(c)
    rp, rv, uid = pos.copy(), vel.copy(), np.arange(len(pos), dtype=np.uint32)
    removed_late = 0
    for tick in range(60):
        _push_again(ctx, world, seg)
        ctx.set_tick(tick)
        ctx.step()
        keep = (rp >= -r).all(1) & (rp <= 1 + r).all(1)       # remove_particles, crate.py:149-159
        if tick >= 2:
            removed_late += int(len(keep) - keep.sum())
        rp, rv, uid = rp[keep], rv[keep], uid[keep]
        out = O.step(cv, rp, rv, seg, [len(seg)], np.zeros((1, 5)), noise_mode=1, tkey=O.tick_key(11, tick), uid=uid,
                     want_all=True)
        rp, rv = out["pos_out"], out["vel_out"]
    assert removed_late >= 3, "particles must leave while the force kernel computes the keys"
    assert ctx.particle_count() == len(uid)
    gp, gv, gprs = ctx.get_state()
    assert np.array_equal(ctx.get_uids(), uid)
    assert np.array_equal(gp, rp) and np.array_equal(gv, rv) and np.array_equal(gprs, out["pressure"])

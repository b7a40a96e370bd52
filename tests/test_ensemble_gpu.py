"""Ensembles on the device: every member of an `Ensemble` is bit-identical - positions, velocities, pressures, local
uids and count - to a separate `Crate` with that member's coefficients and noise seed, in both precisions and both noise
modes an ensemble runs; plus the model's refusals."""
import copy

import numpy as np
import pytest

from conftest import oracle_counter_run, world_from_freerun
from sand_crate_b200 import Crate, Ensemble, SandCrateError, WorldConfig, _lib
from sand_crate_b200.scenes import dam_break

pytestmark = pytest.mark.gpu

VARIANTS8 = [{}, {"viscosity": 4}, {"pressure_amplifier": 20}, {"collider_noise_level": 0.0},
             {"surface_smoothing": 50, "target_pressure": -1}, {"gravity": [0.5, 7.0]},
             {"wall_collision_decay": 0.6, "ignored_pressure": 0.2}, {"max_particles": 1500}]


def with_coeffs(world, override):
    c = copy.deepcopy(dict(world.coefficients))
    c.update(override)
    return WorldConfig(rigid_bodies=copy.deepcopy(world.rigid_bodies),
                       particle_sources=copy.deepcopy(world.particle_sources), coefficients=c)


def crate_state(crate):
    pos, vel, prs = crate._ctx.get_state()
    return pos, vel, prs, crate._ctx.get_uids(), crate.particle_count


def assert_member_equal(ens, m, crate, where=""):
    mv = ens.member(m)
    pos, vel, prs, uid, n = crate_state(crate)
    assert mv.particle_count == n, (where, m, mv.particle_count, n)
    for name, a, b in (("pos", mv.particles, pos), ("vel", mv.particle_velocities, vel),
                       ("pressure", mv.particles_pressure, prs), ("uid", mv.uids, uid)):
        assert a.shape == b.shape and np.array_equal(a.view(np.uint8), np.ascontiguousarray(b).view(np.uint8)), \
            f"{where}: member {m} {name} differs from its separate run"


def run_and_compare(world, overrides, seeds, ticks, every, precision="mixed", noise="counter", states=None,
                    edit=None):
    """Step an Ensemble and one Crate per member side by side; compare every `every` ticks and at the end.
    `states`: per-member (pos, vel) to start from; `edit`: (tick, member, name, value) applied to both."""
    ens = Ensemble(world, overrides, seeds=seeds, precision=precision, noise=noise)
    if isinstance(overrides, int):
        overrides = [{}] * overrides
    crates = [Crate(with_coeffs(world, o), precision=precision, noise=noise, noise_seed=s)
              for o, s in zip(overrides, seeds)]
    try:
        if states is not None:
            ens.set_particles([p for p, _ in states], [v for _, v in states])
            for c, (p, v) in zip(crates, states):
                c.set_particles(p, v)
        for t in range(1, ticks + 1):
            if edit and edit[0] == t - 1:
                setattr(ens.member(edit[1]), edit[2], edit[3])
                setattr(crates[edit[1]], edit[2], edit[3])
            ens.physics_tick()
            for c in crates:
                c.physics_tick()
            if t % every == 0 or t == ticks:
                for m, c in enumerate(crates):
                    assert_member_equal(ens, m, c, f"tick {t}")
        return ens, crates
    finally:
        ens.close()
        for c in crates:
            c.close()


@pytest.mark.parametrize("precision", ["mixed", "f64"])
@pytest.mark.parametrize("noise", ["counter", "none"])
def test_wave_machine_sweep(precision, noise):
    """8 coefficient variants x 2 seeds: sources, the moving paddle, the W1b quirk and CCD, per-member clamps."""
    world, _ = world_from_freerun("wave_machine")
    overrides = [o for o in VARIANTS8 for _ in (0, 1)]
    seeds = [s for _ in VARIANTS8 for s in (3, 11)]
    run_and_compare(world, overrides, seeds, 300, 25, precision, noise)


def test_stirring_cup_drains():
    """Starts empty, sources for 200 ticks, the cup drains: removal in every member."""
    world, _ = world_from_freerun("stirring_cup")
    overrides = [{}, {"viscosity": 2}, {"pressure_amplifier": 50}, {"gravity": [0, 15.0]},
                 {"collider_noise_level": 0.3}, {"max_particles": 300}]
    run_and_compare(world, overrides, [5] * 6, 1200, 100)


def test_max_particles_clamp_per_member():
    """The clamp binds in some members (small max_particles) and not in others, each against its own count."""
    world, _ = world_from_freerun("wave_machine")
    overrides = [{"max_particles": 300}, {}, {"max_particles": 1000}, {"max_particles": 57}]
    ens, crates = run_and_compare(world, overrides, [1, 1, 2, 2], 200, 40)


def _spray(n, seed):
    r = np.random.default_rng(seed)
    return r.uniform(0.02, 0.98, (n, 2)), r.normal(0, 0.3, (n, 2))


def _band_over_dense_row(d, seed):
    """1400 particles packed into one cell row and 60 in the sparse row above it: a block of the sparse row has a
    previous-row window beyond the staging buffer, so it runs pass-through."""
    r = np.random.default_rng(seed)
    y0 = (np.floor(0.5 / d) + 0.5) * d
    dense = np.stack((r.uniform(0.05, 0.95, 1400), y0 + r.uniform(0.1, 0.3, 1400) * d), 1)
    sparse = np.stack((r.uniform(0.05, 0.95, 60), y0 + r.uniform(0.7, 0.9, 60) * d + d), 1)
    pos = np.concatenate((dense, sparse))
    return pos, np.zeros_like(pos)


def test_members_of_different_sizes_straddle_blocks():
    """Members of very different sizes: 256-blocks of the tiled kernels straddle member boundaries, and both kinds of
    block do - staged and pass-through.  The block kinds of tick 1 are predicted from the sorted cell keys (every
    particle is clear of the walls, so its key is floor(y / d), floor(x / d) in its member's grid) and the device's
    pass-through count must equal the prediction."""
    from test_pair_records_gpu import SC_TILE, tile_windows_np
    world, _, _ = dam_break(3000)
    d = 2 * world.coefficients["particle_radius"]
    # two sparse members side by side (a straddle whose windows stage), dense-row bands next to others (straddles whose
    # windows do not), a tiny and an empty member
    empty = (np.zeros((0, 2)), np.zeros((0, 2)))
    sizes = [_spray(700, 1), _spray(300, 2), _band_over_dense_row(d, 1), _spray(5, 4), empty,
             _band_over_dense_row(d, 3), _spray(900, 5)]
    sizes = [(p, np.zeros_like(p)) for p, _ in sizes]
    M = len(sizes)
    overrides = [{"max_particles": 3000}] * M
    ens = Ensemble(world, overrides, seeds=list(range(M)))
    crates = [Crate(with_coeffs(world, o), precision="mixed", noise="counter", noise_seed=s)
              for s, o in enumerate(overrides)]
    try:
        ens.set_particles([p for p, _ in sizes], [v for _, v in sizes])
        for c, (p, v) in zip(crates, sizes):
            c.set_particles(p, v)
        for t in range(1, 31):
            ens.physics_tick()
            for c in crates:
                c.physics_tick()
            if t == 1:
                row_min, col_min, nrows, ncols = ens._ctx.grid()
                ncs = (nrows // M) * ncols
                keys = np.concatenate([m * ncs + (np.floor(p[:, 1] / d).astype(np.int64) - row_min) * ncols
                                       + np.floor(p[:, 0] / d).astype(np.int64) - col_min
                                       for m, (p, _) in enumerate(sizes)])
                keys = np.sort(keys)
                w = tile_windows_np(keys, M * ncs, ncols)
                b0 = np.arange(0, len(keys), SC_TILE)
                straddle = keys[b0] // ncs != keys[np.minimum(b0 + SC_TILE, len(keys)) - 1] // ncs
                assert ens.untiled_blocks() == int((~w["staged"]).sum())
                assert (straddle & ~w["staged"]).any() and (straddle & w["staged"]).any()
            if t in (1, 10, 30):
                for m, c in enumerate(crates):
                    assert_member_equal(ens, m, c, f"tick {t}")
    finally:
        ens.close()
        for c in crates:
            c.close()


def test_max_particles_raised_mid_run():
    """Raising one member's max_particles past what the context was sized for grows the context, identities kept, and
    the member stays bit-identical to a Crate edited the same way: one with room for it and one with the default
    capacity, which grows its own context, so both growth paths must keep the identities."""
    world, _ = world_from_freerun("wave_machine")
    overrides = [{"max_particles": 300}, {"max_particles": 300}, {"max_particles": 500}]
    ens = Ensemble(world, overrides, seeds=[1, 2, 3])
    crates = [Crate(with_coeffs(world, o), precision="mixed", noise="counter", noise_seed=s, capacity=4000)
              for o, s in zip(overrides, [1, 2, 3])]
    grown = Crate(with_coeffs(world, overrides[1]), precision="mixed", noise="counter", noise_seed=2)
    try:
        cap0 = ens._ctx.capacity
        for t in range(1, 201):
            if t == 61:
                ens.member(1).max_particles = 3000
                crates[1].max_particles = grown.max_particles = 3000
            ens.physics_tick()
            for c in crates + [grown]:
                c.physics_tick()
            if t % 40 == 0:
                for m, c in enumerate(crates):
                    assert_member_equal(ens, m, c, f"tick {t}")
                assert_member_equal(ens, 1, grown, f"tick {t}, grown Crate")
        assert ens._ctx.capacity > cap0 and ens.member(1).particle_count > 300
        assert grown._ctx.capacity > 300
    finally:
        ens.close()
        for c in crates + [grown]:
            c.close()


def test_member_starts_above_its_max_particles():
    """A member whose state starts above its max_particles: no emission gets in until removal takes it below, and the
    context holds it (its sources' clamp is against its own count)."""
    world, _ = world_from_freerun("wave_machine")
    start, _ = _spray(800, 7)
    overrides = [{"max_particles": 300}, {"max_particles": 300}]
    states = [(start, np.zeros_like(start)), (start[:10], np.zeros((10, 2)))]
    run_and_compare(world, overrides, [4, 5], 80, 20, states=states)


def test_emission_past_capacity_is_refused_before_launch():
    """On the C ABI, an emission whose members' clamps could let the counts outgrow the capacity is refused with the
    cause named, before anything is launched (no particle is dropped on the device)."""
    world, _ = world_from_freerun("wave_machine")
    params = dict(dt=0.002, particle_radius=0.005, wall_collision_decay=0.2, pressure_amplifier=30,
                  ignored_pressure=0.3, collider_noise_level=0.1, viscosity=8, surface_smoothing=100,
                  target_pressure=-2, gravity_x=0, gravity_y=9.8)
    ctx = _lib.Context(100, _lib.PRECISION_MIXED)
    try:
        ctx.set_noise(_lib.NOISE_COUNTER, 0)
        ctx.ens_configure(2, 12)
        ctx.ens_set_params([params, params], [0, 1])
        pos, _ = _spray(60, 3)
        ctx.ens_set_state(pos, np.zeros_like(pos), [60, 0])
        rec = [(0.5, 0.5, 0.1, 0.0, 0.0, 0.0, 0, 0)]
        ctx.ens_emit_particles(rec, [[0], [40]], [100, 100])        # bounds 60 + 40: fits
        launches = ctx.launch_count()
        with pytest.raises(SandCrateError, match="capacity"):
            ctx.ens_emit_particles(rec, [[0], [1]], [100, 100])     # member 1 could reach 41: 101 > 100
        assert ctx.launch_count() == launches
        assert list(ctx.ens_member_counts()) == [60, 40]
    finally:
        ctx.close()


def test_member_drained_to_zero():
    """One member loses every particle (they start outside the box, so the first removal takes them all) while the
    others continue."""
    world, pos, vel = dam_break(2000)
    states = [(pos, vel), (pos + [0.0, 1.5], vel), (pos, vel)]
    overrides = [{}, {}, {"viscosity": 3}]
    ens = Ensemble(world, overrides, seeds=[0, 0, 0])
    crates = [Crate(with_coeffs(world, o), precision="mixed", noise="counter") for o in overrides]
    try:
        ens.set_particles([p for p, _ in states], [v for _, v in states])
        for c, (p, v) in zip(crates, states):
            c.set_particles(p, v)
        for t in range(1, 41):
            ens.physics_tick()
            for c in crates:
                c.physics_tick()
        assert ens.member(1).particle_count == 0
        for m, c in enumerate(crates):
            assert_member_equal(ens, m, c, "tick 40")
    finally:
        ens.close()
        for c in crates:
            c.close()


def test_dam_break_100k_four_members():
    world, pos, vel = dam_break(100_000)
    overrides = [{}, {"viscosity": 2}, {"pressure_amplifier": 40}, {"collider_noise_level": 0.0}]
    run_and_compare(world, overrides, [0, 1, 2, 3], 50, 25, states=[(pos, vel)] * 4)


def test_single_member_equals_plain_context():
    world, _ = world_from_freerun("wave_machine")
    run_and_compare(world, 1, [7], 200, 50)


def test_64_replicas():
    world, _ = world_from_freerun("wave_machine")
    run_and_compare(world, [{}] * 64, list(range(64)), 100, 50)


def test_f64_member_matches_oracle():
    """fp64: member 1 of a sweep is bit for bit the oracle's counter-mode run with its coefficients."""
    world, _ = world_from_freerun("wave_machine")
    overrides = [{"viscosity": 4}, {"pressure_amplifier": 20, "surface_smoothing": 60}, {}]
    ens = Ensemble(world, overrides, seeds=[2, 9, 4], precision="f64")
    try:
        check = {50, 100, 150}
        for tick, pos, vel, prs in oracle_counter_run(with_coeffs(world, overrides[1]), 9, 150):
            ens.physics_tick()
            if tick in check:
                mv = ens.member(1)
                assert np.array_equal(mv.particles, pos) and np.array_equal(mv.particle_velocities, vel), tick
                assert np.array_equal(mv.particles_pressure, prs), tick
    finally:
        ens.close()


def test_live_edit_one_member():
    """Changing member 2's viscosity at tick 50 equals a separate run edited at tick 50; the others are untouched."""
    world, _ = world_from_freerun("wave_machine")
    run_and_compare(world, [{}, {"viscosity": 5}, {}, {"pressure_amplifier": 20}], [1, 2, 3, 4], 120, 30,
                    edit=(50, 2, "viscosity", 3.5))


def test_no_host_wait_and_launches_of_one_context():
    """16 members of wave_machine with sources for 3000 ticks: no host wait, and the launches of a single context."""
    world, _ = world_from_freerun("wave_machine")
    ens = Ensemble(world, 16)
    crate = Crate(world, precision="mixed", noise="counter", noise_seed=0)
    try:
        ens.physics_tick()
        crate.physics_tick()
        s0, l0, c0 = ens.sync_count(), ens.launch_count(), crate._ctx.launch_count()
        for _ in range(3000):
            ens.physics_tick()
            crate.physics_tick()
        assert ens.sync_count() - s0 == 0
        assert ens.launch_count() - l0 == crate._ctx.launch_count() - c0
        assert int(ens.particle_counts().min()) > 0
    finally:
        ens.close()
        crate.close()


def test_refusals():
    world, _ = world_from_freerun("wave_machine")
    with pytest.raises(ValueError, match="dt differs"):
        Ensemble(world, [{}, {"dt": 0.001}])
    with pytest.raises(ValueError, match="particle_radius differs"):
        Ensemble(world, [{}, {"particle_radius": 0.004}])
    free, _ = world_from_freerun("free_body")
    with pytest.raises(ValueError, match="free body"):
        Ensemble(free, [{}, {"gravity": [0, 5.0]}])
    with pytest.raises(ValueError, match="reference"):
        Ensemble(world, 2, noise="reference")
    ens = Ensemble(world, 2)
    try:
        with pytest.raises(SandCrateError, match="ensemble"):
            ens._ctx.dist_configure(0, 2, 0, 50, 4, 1000)
        with pytest.raises(SandCrateError, match="ensemble"):
            ens._ctx.set_monitor(True)
        with pytest.raises(SandCrateError, match="SC_NOISE_HOST"):
            ens._ctx.set_noise(_lib.NOISE_HOST, 0)
        with pytest.raises(ValueError, match="shared"):
            ens.member(1).dt = 0.001
    finally:
        ens.close()
    ens = Ensemble(world, 2, member_uid_bits=10)   # 1024 identities; the source draws ~14 a tick
    try:
        with pytest.raises(SandCrateError, match="identities exhausted"):
            for _ in range(200):
                ens.physics_tick()
        assert ens.tick < 100
    finally:
        ens.close()
    small = with_coeffs(world, {"particle_radius": 0.0005, "max_particles": 1})
    with pytest.raises(SandCrateError, match="too many cells"):
        Ensemble(small, 5000, member_uid_bits=10)

"""CPU tests of the host-side mirror of the reference interface: config schema, rigid bodies, particle sources and
the `Crate` tick protocol.  The GPU context is replaced by the oracle-backed test double (tests/oracle_backend.py)
so the whole-run comparison against the reference's recorded trajectories runs without a GPU."""
import numpy as np
import pytest
import yaml

import sand_crate_b200
from conftest import golden, world_from_freerun
from oracle_backend import OracleContext
from sand_crate_b200 import Crate, config_from_dict, crate as crate_mod
from sand_crate_b200.rigid_body import build_rigid_bodies, rotate_degrees
from sand_crate_b200.scenes import box_fill, dam_break


@pytest.fixture
def oracle_backend(monkeypatch):
    monkeypatch.setattr(crate_mod._lib, "Context", OracleContext)


def test_config_schema_roundtrip(tmp_path):
    world, _ = world_from_freerun("stirring_cup")
    raw = {"playback": {"save_recording": True, "ticks_to_record": 1200, "recording_output_dir_path": "../data",
                        "screen_x": 1000, "screen_y": 1000},
           "world": {"coefficients": world.coefficients, "particle_sources": world.particle_sources,
                     "rigid_bodies": world.rigid_bodies}}
    path = tmp_path / "cfg.yaml"
    path.write_text(yaml.safe_dump(raw))
    cfg = sand_crate_b200.load_config(path)
    assert cfg.world_config.coefficients == world.coefficients
    assert cfg.playback_config.ticks_to_record == 1200
    assert config_from_dict(raw).world_config.rigid_bodies == world.rigid_bodies


def test_rotate_degrees_quarter_turns_are_exact():
    assert rotate_degrees(1.0, 2.0, 90) == (-2.0, 1.0)
    assert rotate_degrees(1.0, 2.0, -90) == (2.0, -1.0)
    assert rotate_degrees(1.0, 2.0, 180) == (-1.0, -2.0)
    x, y = rotate_degrees(1.0, 0.0, -12)
    assert abs(x - np.cos(np.radians(12))) < 1e-15 and abs(y + np.sin(np.radians(12))) < 1e-15


@pytest.mark.parametrize("name", ["stirring_cup", "wave_machine"])
def test_rigid_bodies_follow_the_reference(name):
    """Placement (scale -> rotate -> translate) and the linearised motored motion, against recorded segments."""
    world, g = world_from_freerun(name)
    bodies = build_rigid_bodies(world.rigid_bodies)
    dt = world.coefficients["dt"]
    ticks = [int(t) for t in g["ticks"]]
    for tick in range(1, max(ticks) + 1):
        for b in bodies:
            b.apply_velocity(dt)
        if tick in ticks:
            seg = np.vstack([b.segments for b in bodies])
            assert np.array_equal(seg, g[f"segments_t{tick}"]), tick


@pytest.mark.parametrize("name,last", [("stirring_cup", 1200), ("wave_machine", 500), ("free_body", 60)])
def test_crate_protocol_reproduces_reference_trajectory(oracle_backend, name, last):
    """Sources + RNG protocol + body motion + removal, whole run, bit for bit (step = oracle test double).
    stirring_cup over its full 1200 ticks; wave_machine to tick 500 here (its full 3000 ticks run on the GPU,
    tests/test_gpu_parity.py::test_crate_free_run_bit_exact, and in tests/make_spread.py when it is regenerated)."""
    world, g = world_from_freerun(name)
    crate = Crate(world)
    for tick in range(1, last + 1):
        crate.physics_tick()
        if f"pos_t{tick}" in g.files:
            assert crate.tick == tick
            assert crate.particle_count == len(g[f"pos_t{tick}"])
            assert np.array_equal(crate.particles, g[f"pos_t{tick}"]), tick
            assert np.array_equal(crate.particle_velocities, g[f"vel_t{tick}"]), tick
            assert np.array_equal(crate.particles_pressure, g[f"pressure_t{tick}"]), tick
            assert np.array_equal(crate.segments, g[f"segments_t{tick}"]), tick


def test_crate_surface(oracle_backend):
    world, _ = world_from_freerun("stirring_cup")
    crate = Crate(world)
    assert set(crate.editable_coefficients()) == set(world.coefficients)
    assert crate.diameter == 2 * world.coefficients["particle_radius"]
    assert crate.segments.shape == (6, 2, 2) and crate.particle_count == 0 and crate.tick == 0
    crate.viscosity = crate.viscosity * 1.1            # live edit, playback.py:221-226
    crate.gravity = np.array([0.0, -9.81])              # playback.py:151-153
    crate.physics_tick()
    assert crate._ctx.params["viscosity"] == pytest.approx(8.8) and crate._ctx.params["gravity_y"] == -9.81
    assert "Tick: 1" in crate.debug_prints and "viscosity" in crate.debug_prints
    assert crate.debug_arrows == []


def test_crate_grows_capacity(oracle_backend):
    world, _ = world_from_freerun("stirring_cup")
    crate = Crate(world, capacity=8)
    for _ in range(6):
        crate.physics_tick()
    assert crate.particle_count > 8 and crate._ctx.capacity >= crate.particle_count


@pytest.mark.parametrize("maker,n", [(dam_break, 20000), (box_fill, 10000)])
def test_synthetic_scenes(maker, n):
    world, pos, vel = maker(n)
    c = world.coefficients
    d = 2 * c["particle_radius"]
    assert pos.shape == (n, 2) and vel.shape == (n, 2) and not vel.any()
    assert pos.min() > 0.5 * d and pos.max() < 1 - 0.5 * d                 # inside the box, off the walls
    assert c["dt"] == pytest.approx(0.002 * d / 0.01) and c["max_particles"] == n
    # lattice spacing 0.75 d: about 1.8 particles per d x d cell where the liquid is
    cells = np.floor(pos / d).astype(np.int64)
    occ = np.unique(cells[:, 0] * 100000 + cells[:, 1], return_counts=True)[1]
    assert 1.5 < occ.mean() < 2.1


def test_headless_runner_records_the_reference_trajectory(oracle_backend, tmp_path):
    """sand_crate_b200.run: the display-less replacement of main.py / Playback (SURVEY 8(f) row 2)."""
    from sand_crate_b200 import run as runner
    world, g = world_from_freerun("stirring_cup")
    cfg = {"playback": {"save_recording": False, "ticks_to_record": 20, "recording_output_dir_path": ".",
                        "screen_x": 10, "screen_y": 10},
           "world": {"coefficients": world.coefficients, "particle_sources": world.particle_sources,
                     "rigid_bodies": world.rigid_bodies}}
    path = tmp_path / "cup.yaml"
    path.write_text(yaml.safe_dump(cfg))
    out = tmp_path / "run.npz"
    summary = runner.run(path, every=5, out=out, quiet=True)
    assert summary["ticks"] == 20 and summary["particles_final"] == len(g["pos_t20"])
    frames = {t: (p, prs, seg) for t, p, prs, seg in runner.load_recording(out)}
    assert sorted(frames) == [5, 10, 15, 20]
    for t in (5, 20):
        assert np.array_equal(frames[t][0], g[f"pos_t{t}"]) and np.array_equal(frames[t][1], g[f"pressure_t{t}"])
        assert np.array_equal(frames[t][2], g[f"segments_t{t}"])


@pytest.mark.parametrize("name,last", [("stirring_cup", 80), ("wave_machine", 40)])
def test_force_monitor_overlay_matches_reference(oracle_backend, name, last):
    """ForceMonitor (utils/force_monitor.py): EMA of the mean |dv| per force section, against the reference's own."""
    world, g = world_from_freerun(name)
    crate = Crate(world, monitor=True)
    for tick in range(1, last + 1):
        crate.physics_tick()
        if f"monitor_t{tick}" in g.files:
            got = np.array([crate.force_monitor.context_to_velocity[k] for k in crate_mod.FORCE_SECTIONS])
            assert np.allclose(got, g[f"monitor_t{tick}"], rtol=1e-11, atol=1e-15), tick
    assert "Forces" in crate.debug_prints and "tension" in crate.force_monitor.report()


def test_binomial_inverse_cdf_against_scipy():
    """The emission count of the counter-stream sources: Binomial(flow, dt) through its inverse CDF."""
    from scipy.stats import binom
    from sand_crate_b200.particle_source import binomial_inverse_cdf
    rs = np.random.RandomState(5)
    for trials, p in ((2000, 0.002), (7000, 0.002), (50, 0.3)):
        u = rs.rand(3000)
        got = np.array([binomial_inverse_cdf(x, trials, p) for x in u])
        want = binom.ppf(u, trials, p).astype(int)
        assert (got != want).mean() < 2e-3          # equal except where u sits within rounding of a CDF step
        assert abs(got.mean() - trials * p) < 0.15 * np.sqrt(trials * p)
    assert binomial_inverse_cdf(0.0, 10, 0.5) == 0 and binomial_inverse_cdf(1.0, 10, 0.5) == 10


def test_counter_sources_host_protocol(oracle_backend):
    """Production mode of the drop-in Crate (counter noise, device-side sources): the host protocol - counter-stream
    emission counts, sc_emit_particles, body motion, step - against an end-to-end restatement on the oracle."""
    from conftest import oracle_counter_run
    world, _ = world_from_freerun("wave_machine")
    crate = Crate(world, noise="counter", noise_seed=11)
    for tick, pos, vel, prs in oracle_counter_run(world, 11, 60):
        crate.physics_tick()
        if tick % 20 == 0:
            assert crate.particle_count == len(pos) > 0
            assert np.array_equal(crate.particles, pos) and np.array_equal(crate.particle_velocities, vel)
    # the max_particles clamp (crate.py:143): a tiny cap is reached and never exceeded
    world2, _ = world_from_freerun("wave_machine")
    world2.coefficients["max_particles"] = 100
    crate = Crate(world2, noise="counter", noise_seed=11)
    for tick, pos, vel, prs in oracle_counter_run(world2, 11, 30):
        crate.physics_tick()
    assert crate.particle_count == len(pos) == 100
    assert np.array_equal(crate.particles, pos)


def _same_crates(a, b, tick):
    assert a.particle_count == b.particle_count, tick
    assert np.array_equal(a._ctx.get_uids(), b._ctx.get_uids()), tick
    assert np.array_equal(a.particles, b.particles), tick
    assert np.array_equal(a.particle_velocities, b.particle_velocities), tick


def _wave_machine(max_particles):
    import copy
    world, _ = world_from_freerun("wave_machine")
    c = copy.deepcopy(dict(world.coefficients))
    c["max_particles"] = max_particles
    return sand_crate_b200.WorldConfig(rigid_bodies=world.rigid_bodies, particle_sources=world.particle_sources,
                                       coefficients=c)


def test_crate_growth_keeps_identities_counter_noise(oracle_backend):
    """A Crate that grows its context keeps every uid and the next one: counter noise is keyed on uids, so a grown
    Crate and one with room from the start stay identical.  The clamp binds before the raise, so the emission leaves
    gaps in the identities that the next uid must jump over."""
    grown = Crate(_wave_machine(300), noise="counter", noise_seed=2)
    roomy = Crate(_wave_machine(300), noise="counter", noise_seed=2, capacity=4000)
    clamped = False
    for tick in range(1, 91):
        if tick == 61:
            clamped = grown.particle_count == 300
            grown.max_particles = roomy.max_particles = 3000
        grown.physics_tick()
        roomy.physics_tick()
        _same_crates(grown, roomy, tick)
    assert clamped and grown._ctx.capacity > 300 and grown.particle_count > 300


def test_crate_growth_through_set_particles_keeps_identities(oracle_backend):
    rs = np.random.RandomState(4)
    pos = 0.2 + 0.6 * rs.rand(400, 2)
    grown = Crate(_wave_machine(500), noise="counter", noise_seed=5, capacity=64)
    roomy = Crate(_wave_machine(500), noise="counter", noise_seed=5, capacity=4000)
    for c in (grown, roomy):
        c.set_particles(pos)                     # beyond the capacity of `grown`: it grows here ...
    for tick in range(1, 61):
        if tick == 31:
            grown.max_particles = roomy.max_particles = 2000   # ... and again here, after clamped emissions
        grown.physics_tick()
        roomy.physics_tick()
        _same_crates(grown, roomy, tick)
    assert grown._ctx.capacity > 500 and grown.particle_count > 500


def test_crate_growth_keeps_identities_reference_noise(oracle_backend):
    world, _ = world_from_freerun("stirring_cup")
    grown = Crate(world, capacity=8)
    states = []
    for _ in range(40):
        grown.physics_tick()
        states.append((grown._ctx.get_uids(), grown.particles.copy(), grown.particle_velocities.copy()))
    roomy = Crate(world, capacity=4000)           # (each Crate reseeds the global stream the sources draw from)
    for tick, (uid, pos, vel) in enumerate(states, 1):
        roomy.physics_tick()
        assert np.array_equal(roomy._ctx.get_uids(), uid), tick
        assert np.array_equal(roomy.particles, pos) and np.array_equal(roomy.particle_velocities, vel), tick
    assert grown._ctx.capacity > 8

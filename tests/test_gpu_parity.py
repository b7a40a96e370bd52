"""GPU parity tests (pytest -m gpu, B200 only).  Everything goes through the C ABI (sand_crate_b200._lib.Context ->
libsandcrate.so); the oracle is only the checker.

Bars (SURVEY.md section 8(c)):
  * cell rows, sorted order, neighbor lists (order + 20-trim): bit-exact, both precision modes.  The lists come from
    `get_neighbors`, which re-runs the untiled count kernel; the tiled density kernel's own lists and vectors are
    checked in tests/test_pair_records_gpu.py through `get_pair_records`
  * fp64 parity mode: positions, velocities, pressures, surface normals bit-exact per step
  * mixed mode (fp64 positions, fp32 forces): per step from the same inputs,
      max|dv| <= 1e-5 * max(max|v|, 1)   and   max|dpos| <= 1e-5 * d
"""
import numpy as np
import pytest

from conftest import golden, neighbor_case_tags, params_from_coeffs, step_goldens, world_from_freerun
from oracle import oracle as O
from sand_crate_b200 import Crate, _lib
from sand_crate_b200.scenes import box_fill, dam_break

pytestmark = pytest.mark.gpu

REL_TOL_F32 = 1e-5
# bound on the error of the per-tick velocity INCREMENT of the production arithmetic, relative to the largest
# increment of the tick: max|dv_gpu - dv_ref| / max|dv_ref| with dv = v_out - v_in (VERDICT r1 item 6)
INCREMENT_TOL_F32 = 1e-5


def v_floor(coeffs_or_world):
    """Velocity scale below which a relative velocity error is meaningless, tied to the scene: 1 % of a particle
    diameter per tick (0.01 d / dt) - NOT a constant like 1.0, which is 20x the speeds of a scene at rest."""
    if hasattr(coeffs_or_world, "coefficients"):
        c = coeffs_or_world.coefficients
        return 0.01 * 2 * c["particle_radius"] / c["dt"]
    return 0.01 * 2 * float(coeffs_or_world[1]) / float(coeffs_or_world[0])


def increment_error(v_gpu, v_ref, v_in):
    dv_ref = v_ref - v_in
    return float(np.abs((v_gpu - v_in) - dv_ref).max() / np.abs(dv_ref).max())


def make_ctx(g, precision, noise_mode, capacity=None, seed=0):
    ctx = _lib.Context(capacity or max(len(g["pos_in"]), 1), precision)
    ctx.set_params(**params_from_coeffs(g["coeffs"]))
    ctx.set_walls(g["segments"], g["body_len"], g["body_kin"])
    ctx.set_noise(noise_mode, seed)
    ctx.set_state(g["pos_in"], g["vel_in"])
    return ctx


# ---- layer-2 functions ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", neighbor_case_tags())
def test_detect_particle_collisions_bit_exact(tag):
    g = golden("neighbors_cases.npz")
    ctx = _lib.Context(16)
    rows, order, counts, idx = ctx.detect_particle_collisions(g[f"{tag}__pts"], float(g[f"{tag}__d"]))
    assert np.array_equal(rows, g[f"{tag}__rows"])
    assert np.array_equal(order, g[f"{tag}__order"])
    assert np.array_equal(counts, g[f"{tag}__counts"])
    assert np.array_equal(idx, g[f"{tag}__idx"])


def test_points_to_segments_distance_bit_exact():
    g = golden("geometry_cases.npz")
    ctx = _lib.Context(16)
    for k in ("row", "rnd"):
        near, dist = ctx.points_to_segments_distance(g[f"{k}_p"], g[f"{k}_segs"])
        assert np.array_equal(near, g[f"{k}_near"]) and np.array_equal(dist, g[f"{k}_dist"])
    _, dist = ctx.points_to_segments_distance(g["row_p"], g["row_segs"])
    for i in range(5):
        for j in range(35):
            assert dist[j, i] == abs(j - i)  # the reference's own known-answer test (test_distance.py:16-25)


# ---- one tick against the recorded reference ---------------------------------------------------------------
@pytest.mark.parametrize("name", step_goldens())
def test_step_f64_reference_noise_bit_exact(name):
    g = golden(name)
    ctx = make_ctx(g, _lib.PRECISION_F64, _lib.NOISE_HOST)
    n, n_pairs = ctx.step_begin()
    assert n == len(g["pos_search"]) and n_pairs == len(g["noise"])
    pos_search, rows, order = ctx.get_search(n)
    counts, idx = ctx.get_neighbors(n)
    assert np.array_equal(pos_search, g["pos_search"])
    assert np.array_equal(rows, g["rows_sorted"]) and np.array_equal(order, g["order"])
    assert np.array_equal(counts, g["nbr_count"])
    flat = np.concatenate([idx[i, :counts[i]] for i in range(n)]) if n_pairs else np.zeros(0, np.int32)
    assert np.array_equal(flat, g["nbr_idx"])
    ctx.step_finish(g["noise"])
    pos, vel, prs = ctx.get_state()
    assert np.array_equal(prs, g["pressure"])
    assert np.array_equal(ctx.get_tension(n), g["tension_vec"])
    assert np.array_equal(vel, g["vel_out"])
    assert np.array_equal(pos, g["pos_out"])


@pytest.mark.parametrize("name", step_goldens())
def test_step_mixed_reference_noise_within_tolerance(name):
    g = golden(name)
    ctx = make_ctx(g, _lib.PRECISION_MIXED, _lib.NOISE_HOST)
    n, n_pairs = ctx.step_begin()
    _, rows, order = ctx.get_search(n)
    counts, idx = ctx.get_neighbors(n)
    assert np.array_equal(rows, g["rows_sorted"]) and np.array_equal(order, g["order"])  # search is fp64 in both modes
    assert np.array_equal(counts, g["nbr_count"])
    flat = np.concatenate([idx[i, :counts[i]] for i in range(n)]) if n_pairs else np.zeros(0, np.int32)
    assert np.array_equal(flat, g["nbr_idx"])           # the LISTS (order + trim), not only their lengths
    ctx.step_finish(g["noise"])
    pos, vel, prs = ctx.get_state()
    d = 2 * float(g["coeffs"][1])
    # the recorded inputs are fp64; mixed mode stores velocities in fp32, so compare against the oracle run on
    # the fp32-rounded input velocities (what the device actually holds)
    vin = g["vel_in"].astype(np.float32).astype(np.float64)
    ref = O.step(g["coeffs"], g["pos_in"], vin, g["segments"], g["body_len"], g["body_kin"], noise_mode=2,
                 noise=g["noise"])
    vscale = max(np.abs(ref["vel_out"]).max(), v_floor(g["coeffs"]))
    assert np.abs(vel - ref["vel_out"]).max() <= REL_TOL_F32 * vscale
    assert np.abs(pos - ref["pos_out"]).max() <= REL_TOL_F32 * d
    assert np.abs(prs - ref["pressure"]).max() <= 1e-5 * max(ref["pressure"].max(), 1.0)
    if n:
        err = increment_error(vel, ref["vel_out"], vin)
        print(f"{name}: increment error {err:.2e}")
        assert err <= INCREMENT_TOL_F32, err


@pytest.mark.parametrize("name", ["step_stirring_cup_t150.npz", "step_wave_machine_t300.npz"])
@pytest.mark.parametrize("precision", [_lib.PRECISION_F64, _lib.PRECISION_MIXED])
def test_step_counter_noise(name, precision):
    """Production noise: device counter-based uniforms == the oracle's restatement of the same hash."""
    g = golden(name)
    ctx = make_ctx(g, precision, _lib.NOISE_COUNTER, seed=1234)
    ctx.set_tick(77)
    ctx.step()
    pos, vel, prs = ctx.get_state()
    vin = g["vel_in"] if precision == _lib.PRECISION_F64 else g["vel_in"].astype(np.float32).astype(np.float64)
    ref = O.step(g["coeffs"], g["pos_in"], vin, g["segments"], g["body_len"], g["body_kin"], noise_mode=1,
                 tkey=O.tick_key(1234, 77))
    if precision == _lib.PRECISION_F64:
        assert np.array_equal(prs, ref["pressure"]) and np.array_equal(vel, ref["vel_out"])
        assert np.array_equal(pos, ref["pos_out"])
    else:
        d = 2 * float(g["coeffs"][1])
        assert np.abs(vel - ref["vel_out"]).max() <= REL_TOL_F32 * max(np.abs(ref["vel_out"]).max(), v_floor(g["coeffs"]))
        assert np.abs(pos - ref["pos_out"]).max() <= REL_TOL_F32 * d
        err = increment_error(vel, ref["vel_out"], vin)   # the tiled production kernels (device noise)
        print(f"{name}: increment error {err:.2e}")
        assert err <= INCREMENT_TOL_F32, err


def test_step_no_noise_bit_exact():
    g = golden("step_wave_machine_t300.npz")
    ctx = make_ctx(g, _lib.PRECISION_F64, _lib.NOISE_NONE)
    ctx.step()
    pos, vel, prs = ctx.get_state()
    ref = O.step(g["coeffs"], g["pos_in"], g["vel_in"], g["segments"], g["body_len"], g["body_kin"], noise_mode=0)
    assert np.array_equal(vel, ref["vel_out"]) and np.array_equal(pos, ref["pos_out"])
    assert np.array_equal(ctx.get_wall_counts(len(pos)), ref["wall_count"])


# ---- the drop-in object, whole runs ---------------------------------------------------------------------------
@pytest.mark.parametrize("name,last", [("stirring_cup", 1200), ("wave_machine", 3000), ("free_body", 60)])
def test_crate_free_run_bit_exact(name, last):
    """`Crate(world_config).physics_tick()` x N == the reference's trajectory, bit for bit (fp64 + reference RNG), over
    the configs' FULL length (`ticks_to_record`: config/stirring_cup.yaml:3 = 1200, config/wave_machine.yaml:3 = 3000):
    sources running and stopped (tick 200 / 500), the cup draining, removal, the paddle over ~7 periods."""
    world, g = world_from_freerun(name)
    crate = Crate(world)
    checked = 0
    for tick in range(1, last + 1):
        crate.physics_tick()
        if f"pos_t{tick}" in g.files:
            assert crate.particle_count == len(g[f"pos_t{tick}"])
            assert np.array_equal(crate.particles, g[f"pos_t{tick}"]), tick
            assert np.array_equal(crate.particle_velocities, g[f"vel_t{tick}"]), tick
            assert np.array_equal(crate.particles_pressure, g[f"pressure_t{tick}"]), tick
            checked += 1
    assert checked == len(g["ticks"]) and int(g["ticks"].max()) == last


@pytest.mark.parametrize("name", ["stirring_cup", "wave_machine"])
def test_mixed_free_run_vs_reference_aggregates(name):
    """Production arithmetic (fp32 forces) against the REFERENCE's trajectory over the configs' full length.  Single
    trajectories decorrelate within ~50 ticks (SURVEY.md section 0 item 4), so the bar is on aggregates, with the SURVEY
    section 8(c) bounds - count 1 %, centre of mass 1e-2, kinetic energy 10 %, max pressure 25 % - each widened to twice
    the reference's OWN spread under a 1e-13 perturbation where that is larger (tests/golden/spread_*.json,
    tests/make_spread.py)."""
    import json
    import os
    from conftest import GOLDEN, aggregates
    spread = json.load(open(os.path.join(GOLDEN, f"spread_{name}.json")))
    world, g = world_from_freerun(name)
    crate = Crate(world, precision="mixed", noise="reference")
    r = world.coefficients["particle_radius"]
    last = max(int(t) for t in spread["reference"])
    report = []
    for tick in range(1, last + 1):
        crate.physics_tick()
        if str(tick) not in spread["reference"]:
            continue
        pos, vel, prs = crate.particles, crate.particle_velocities, crate.particles_pressure
        assert np.isfinite(pos).all() and np.isfinite(vel).all()
        # (a particle may sit outside [-r, 1 + r] after a tick: remove_particles runs at the START of the next one)
        assert pos.min() >= -r - 0.1 and pos.max() <= 1 + r + 0.1
        got, ref, sp = aggregates(pos, vel, prs), spread["reference"][str(tick)], spread["max_abs_spread"][str(tick)]
        assert ref["count"] == len(g[f"pos_t{tick}"])
        bounds = {"count": 0.01 * ref["count"], "com_x": 1e-2, "com_y": 1e-2, "kinetic": 0.10 * ref["kinetic"],
                  "p_max": 0.25 * ref["p_max"]}
        for k, b in bounds.items():
            tol = max(b, 2 * sp[k])
            report.append((tick, k, got[k], ref[k], tol))
            assert abs(got[k] - ref[k]) <= tol, (tick, k, got[k], ref[k], tol, sp[k])
    print("\n".join(f"t={t} {k}: mixed {a:.5g} reference {b:.5g} (allowed +-{c:.3g})" for t, k, a, b, c in report))


def test_headless_runner_on_gpu_records_the_reference_trajectory(tmp_path):
    """sand_crate_b200.run (the display-less replacement of main.py / Playback, playback.py:109-118) on a real
    context: the recorded frames of 80 ticks of stirring_cup are the reference's own (freerun goldens)."""
    import yaml
    from sand_crate_b200 import run as runner
    world, g = world_from_freerun("stirring_cup")
    cfg = {"playback": {"save_recording": False, "ticks_to_record": 80, "recording_output_dir_path": ".",
                        "screen_x": 10, "screen_y": 10},
           "world": {"coefficients": world.coefficients, "particle_sources": world.particle_sources,
                     "rigid_bodies": world.rigid_bodies}}
    path = tmp_path / "cup.yaml"
    path.write_text(yaml.safe_dump(cfg))
    out = tmp_path / "run.npz"
    summary = runner.run(path, every=5, out=out, quiet=True)
    assert summary["ticks"] == 80 and summary["particles_final"] == len(g["pos_t80"])
    frames = {t: (p, prs, seg) for t, p, prs, seg in runner.load_recording(out)}
    assert sorted(frames) == list(range(5, 81, 5))
    for t in (5, 20, 40, 80):
        assert np.array_equal(frames[t][0], g[f"pos_t{t}"]) and np.array_equal(frames[t][1], g[f"pressure_t{t}"])
        assert np.array_equal(frames[t][2], g[f"segments_t{t}"])


def test_device_sources_match_oracle_and_never_synchronise():
    """(f1) Production mode end to end: counter-stream sources generated ON THE DEVICE (sc_emit_particles), counter noise,
    fp64 arithmetic - bit-identical to the same protocol re-stated on the oracle (tests/conftest.py::oracle_counter_run),
    and not one host synchronisation per tick while the sources are running."""
    from conftest import oracle_counter_run
    world, _ = world_from_freerun("wave_machine")
    crate = Crate(world, precision="f64", noise="counter", noise_seed=11)
    syncs0 = crate._ctx.sync_count()
    ref = {}
    for tick, pos, vel, prs in oracle_counter_run(world, 11, 150):
        crate.physics_tick()
        if tick in (50, 150):
            ref[tick] = (pos, vel, prs)
            if tick == 50:
                assert crate._ctx.sync_count() == syncs0, "a tick with active sources made the host wait"
                assert np.array_equal(crate.particles, pos) and np.array_equal(crate.particle_velocities, vel)
    assert crate.particle_count == len(ref[150][0]) > 500
    assert np.array_equal(crate.particles, ref[150][0]) and np.array_equal(crate.particle_velocities, ref[150][1])
    assert np.array_equal(crate.particles_pressure, ref[150][2])
    crate.close()


def test_wave_machine_full_length_counter_mode_without_a_sync():
    """config/wave_machine.yaml over its full 3000 ticks in the production mode (mixed precision, device noise, device
    sources): the host never waits for the GPU inside the run."""
    world, _ = world_from_freerun("wave_machine")
    crate = Crate(world, precision="mixed", noise="counter")
    syncs0 = crate._ctx.sync_count()
    for _ in range(3000):
        crate.physics_tick()
    assert crate._ctx.sync_count() == syncs0
    pos = crate.particles
    assert 2500 < crate.particle_count <= world.coefficients["max_particles"] and np.isfinite(pos).all()
    crate.close()


def test_crate_counter_mode_runs_and_stays_in_box():
    world, _ = world_from_freerun("wave_machine")
    crate = Crate(world, precision="mixed", noise="counter")
    for _ in range(300):
        crate.physics_tick()
    pos = crate.particles
    r = world.coefficients["particle_radius"]
    assert crate.particle_count > 1500 and np.isfinite(pos).all()
    assert pos.min() >= -r and pos.max() <= 1 + r


# ---- synthetic scenes: GPU vs oracle at sizes the oracle finishes in seconds ------------------------------------
def _scene_ctx(world, pos, vel, precision, noise_mode, seed=0):
    c = world.coefficients
    ctx = _lib.Context(len(pos), precision)
    ctx.set_params(dt=c["dt"], particle_radius=c["particle_radius"], wall_collision_decay=c["wall_collision_decay"],
                   pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                   collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                   surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                   gravity_x=c["gravity"][0], gravity_y=c["gravity"][1])
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))
    ctx.set_noise(noise_mode, seed)
    ctx.set_state(pos, vel)
    return ctx, seg


def _coeff_vec(c):
    return np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                     c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                     c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)


@pytest.mark.parametrize("maker,n", [(dam_break, 100_000), (box_fill, 60_000)])
def test_scene_f64_matches_oracle_over_steps(maker, n):
    """5 consecutive ticks, state NOT re-synchronised: fp64 mode stays bit-identical to the oracle."""
    world, pos, vel = maker(n)
    ctx, seg = _scene_ctx(world, pos, vel, _lib.PRECISION_F64, _lib.NOISE_COUNTER, seed=5)
    cv = _coeff_vec(world.coefficients)
    rp, rv = pos.copy(), vel.copy()
    for tick in range(5):
        ctx.set_tick(tick)
        ctx.step()
        out = O.step(cv, rp, rv, seg, [len(seg)], np.zeros((1, 5)), noise_mode=1, tkey=O.tick_key(5, tick),
                     want_all=(tick == 4))
        rp, rv = out["pos_out"], out["vel_out"]
    gp, gv, gprs = ctx.get_state()
    assert np.array_equal(gp, rp) and np.array_equal(gv, rv) and np.array_equal(gprs, out["pressure"])
    counts, idx = ctx.get_neighbors(n)
    assert np.array_equal(counts, out["nbr_count"]) and np.array_equal(idx, out["nbr_idx_padded"])


@pytest.mark.parametrize("maker,n,ticks", [(dam_break, 100_000, (3, 50, 200)), (box_fill, 60_000, (3, 30))])
def test_scene_mixed_per_step_tolerance(maker, n, ticks):
    """Per-step error of the production mode (tiled kernels, counter noise), state re-synchronised from the oracle
    (SURVEY 8(c)): at each listed tick the GPU takes ONE step from the oracle's state and is compared with the oracle's
    next state - absolute velocity / position error, the error of the velocity increment, and the neighbor lists."""
    world, pos, vel = maker(n)
    cv = _coeff_vec(world.coefficients)
    d = 2 * world.coefficients["particle_radius"]
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    tick = 0
    for stop in ticks:
        while tick < stop:  # the oracle carries the scene forward (velocities kept fp32-representable)
            out = O.step(cv, pos, vel, seg, [4], np.zeros((1, 5)), noise_mode=1, tkey=O.tick_key(0, tick), want_all=False)
            pos, vel = out["pos_out"], out["vel_out"].astype(np.float32).astype(np.float64)
            tick += 1
        ctx, _ = _scene_ctx(world, pos, vel, _lib.PRECISION_MIXED, _lib.NOISE_COUNTER)
        ctx.set_tick(tick)
        ctx.step()
        gp, gv, _ = ctx.get_state()
        ref = O.step(cv, pos, vel, seg, [4], np.zeros((1, 5)), noise_mode=1, tkey=O.tick_key(0, tick), want_all=True)
        assert np.abs(gv - ref["vel_out"]).max() <= REL_TOL_F32 * max(np.abs(ref["vel_out"]).max(), v_floor(world))
        assert np.abs(gp - ref["pos_out"]).max() <= REL_TOL_F32 * d
        err = increment_error(gv, ref["vel_out"], vel)
        print(f"{maker.__name__} {n} tick {tick}: increment error {err:.2e}, max|v| {np.abs(ref['vel_out']).max():.3g}")
        assert err <= INCREMENT_TOL_F32, (tick, err)
        counts, idx = ctx.get_neighbors(len(pos))
        assert np.array_equal(counts, ref["nbr_count"]) and np.array_equal(idx, ref["nbr_idx_padded"])
        ctx.close()


def test_tiled_density_pass_through_blocks():
    """The tiled density kernel's pass-through path (a block whose three windows do not fit the staging buffer: sparse
    spray right above dense rows) really runs, and gives the per-step tolerance and the exact neighbor lists."""
    import ctypes as C
    from sand_crate_b200.scenes import _world
    d = 1.0e-3
    s = 0.75 * d
    rs = np.random.RandomState(1)
    # a shallow pool: 1200 particles per cell row, 40 rows
    nx, ny = 1200, 40
    xs = np.tile(0.05 + (np.arange(nx) + 0.5) * s, ny)
    ys = np.repeat(1.0 - d - (np.arange(ny) + 0.5) * s, nx)
    pool = np.stack((xs, ys), 1) + (rs.rand(nx * ny, 2) - 0.5) * 0.1 * s
    # spray: one particle every other cell row above the pool
    k = np.arange(400)
    spray = np.stack((0.1 + 0.8 * rs.rand(len(k)), pool[:, 1].min() - d * (1.5 + 2 * k)), 1)
    spray = spray[spray[:, 1] > 2 * d]
    pos = np.concatenate((pool, spray))
    vel = rs.randn(*pos.shape) * 0.05
    world = _world(len(pos), d)
    ctx, seg = _scene_ctx(world, pos, vel, _lib.PRECISION_MIXED, _lib.NOISE_COUNTER)
    ctx.set_tick(0)
    ctx.step()
    assert ctx.untiled_blocks() > 0, "the scene must push at least one block onto the pass-through path"
    gp, gv, _ = ctx.get_state()
    cv = _coeff_vec(world.coefficients)
    ref = O.step(cv, pos, vel.astype(np.float32).astype(np.float64), seg, [4], np.zeros((1, 5)), noise_mode=1,
                 tkey=O.tick_key(0, 0), want_all=True)
    assert np.abs(gv - ref["vel_out"]).max() <= REL_TOL_F32 * max(np.abs(ref["vel_out"]).max(), v_floor(world))
    assert np.abs(gp - ref["pos_out"]).max() <= REL_TOL_F32 * d
    assert increment_error(gv, ref["vel_out"], vel.astype(np.float32).astype(np.float64)) <= INCREMENT_TOL_F32
    counts, idx = ctx.get_neighbors(len(pos))
    assert np.array_equal(counts, ref["nbr_count"]) and np.array_equal(idx, ref["nbr_idx_padded"])


def test_free_run_is_reproducible():
    """Two runs of the same scene give the same bits (regression: non-coherent loads under programmatic dependent
    launch made fp64 free runs differ from run to run, see sc_common.cuh)."""
    world, _ = world_from_freerun("wave_machine")
    for precision in ("f64", "mixed"):
        got = []
        for _ in range(3):
            np.random.seed(99)
            crate = Crate(world, precision=precision, noise="counter")
            for _ in range(150):
                crate.physics_tick()
            got.append((crate.particles.copy(), crate.particle_velocities.copy()))
            crate.close()
        for p, v in got[1:]:
            assert np.array_equal(p, got[0][0]) and np.array_equal(v, got[0][1]), precision


def test_crate_readback_is_page_locked_and_refilled_in_place():
    """`Crate.particles` and friends are read once per attribute per tick into page-locked buffers that are refilled in
    place (like the reference, whose arrays are updated in place); `Context.get_state()` keeps handing out fresh arrays."""
    world, _ = world_from_freerun("wave_machine")
    np.random.seed(3)
    crate = Crate(world, precision="mixed", noise="counter")
    for _ in range(20):
        crate.physics_tick()
    p1 = crate.particles
    assert crate.particles is p1                      # cached within the tick
    keep = p1.copy()
    fresh, _, _ = crate._ctx.get_state(want_vel=False, want_pressure=False)
    assert np.array_equal(fresh, keep) and not np.shares_memory(fresh, p1)
    crate.physics_tick()
    p2 = crate.particles
    assert np.shares_memory(p1[:1], p2[:1]) or len(p2) != len(p1)   # same buffer again
    assert not np.array_equal(p2[:len(keep)], keep[:len(p2)])        # and it now holds the new tick
    assert len(crate.particle_velocities) == len(p2) == len(crate.particles_pressure)
    # the page-locked memory belongs to the arrays, not to the context: what was handed out stays readable after close()
    # (it used to be freed under the caller's feet)
    last = p2.copy()
    crate.close()
    import gc
    gc.collect()
    assert np.array_equal(p2, last) and np.array_equal(p1[:len(last)], last[:len(p1)])


def test_mixed_mode_drift_stays_bounded_over_1000_ticks():
    """North-star bar for the production mode: over 1000 ticks of wave_machine (sources, moving paddle, removal) the
    mixed-precision run and the fp64 run - same counter noise - keep the same particle count and the same bulk state.
    Individual trajectories decorrelate (the system is chaotic and noised), so the bound is on aggregates."""
    world, _ = world_from_freerun("wave_machine")
    runs = {}
    for precision in ("f64", "mixed"):
        np.random.seed(1234)   # the sources draw from the global stream (particle_source.py)
        crate = Crate(world, precision=precision, noise="counter")
        for _ in range(1000):
            crate.physics_tick()
        runs[precision] = (crate.particle_count, crate.particles.copy(), crate.particle_velocities.copy(),
                           crate.particles_pressure.copy())
        crate.close()
    (n64, p64, v64, q64), (n32, p32, v32, q32) = runs["f64"], runs["mixed"]
    r = world.coefficients["particle_radius"]
    assert abs(n64 - n32) <= 0.01 * n64 and n64 > 1500   # removal at the rim may differ by a few particles
    m = min(n64, n32)
    assert np.isfinite(p32).all() and np.isfinite(v32).all() and p32.min() >= -r and p32.max() <= 1 + r
    assert np.abs(p64.mean(0) - p32.mean(0)).max() < 0.02            # centre of mass: within 2 % of the box
    assert abs(np.sqrt((v64 ** 2).sum(1)).mean() - np.sqrt((v32 ** 2).sum(1)).mean()) < 0.15 * max(
        np.sqrt((v64 ** 2).sum(1)).mean(), 0.05)                    # mean speed
    assert abs(q64.mean() - q32.mean()) < 0.15 * max(q64.mean(), 0.1)  # mean pressure
    hist64 = np.histogram(p64[:, 1], bins=10, range=(0, 1))[0]
    hist32 = np.histogram(p32[:, 1], bins=10, range=(0, 1))[0]
    assert np.abs(hist64 - hist32).max() < 0.05 * m                  # vertical density profile


# ---- size-independent properties at the benchmark size ----------------------------------------------------------
def test_dam_break_1m_properties():
    n = 1_000_000
    world, pos, vel = dam_break(n)
    ctx, _ = _scene_ctx(world, pos, vel, _lib.PRECISION_MIXED, _lib.NOISE_COUNTER)
    ctx.step(3)
    p1, v1, prs = ctx.get_state()
    assert ctx.particle_count() == n and np.isfinite(p1).all() and np.isfinite(v1).all()
    r = world.coefficients["particle_radius"]
    assert p1.min() >= -r and p1.max() <= 1 + r
    # the sorted order the last search produced really is np.lexsort((x, floor(y / d))) of the search positions
    ps, rows, order = ctx.get_search(n)
    d = 2 * r
    want = np.lexsort((ps[:, 0], np.floor(ps[:, 1] / d).astype(np.int64)))
    assert np.array_equal(order, want)
    assert np.array_equal(rows, np.floor(ps[order, 1] / d).astype(np.int64))
    # neighbor lists: untrimmed lists are symmetric and hold exactly the pairs within one diameter
    counts, idx = ctx.get_neighbors(n)
    assert counts.max() <= 20
    sample = np.random.RandomState(0).choice(n, 2000, replace=False)
    for i in sample:
        nb = idx[i, :counts[i]]
        dist = np.sqrt(((ps[nb] - ps[i]) ** 2).sum(1))
        assert (dist <= d).all()
        if counts[i] < 20:
            for j in nb:
                if counts[j] < 20:
                    assert i in idx[j, :counts[j]]
    # determinism: a second context fed the same inputs produces the same bits
    ctx2, _ = _scene_ctx(world, pos, vel, _lib.PRECISION_MIXED, _lib.NOISE_COUNTER)
    ctx2.step(3)
    p2, v2, _ = ctx2.get_state()
    assert np.array_equal(p1, p2) and np.array_equal(v1, v2)


# ---- edge cases -------------------------------------------------------------------------------------------------
def test_empty_and_single_particle():
    g = golden("step_stirring_cup_t150.npz")
    ctx = _lib.Context(8)
    ctx.set_params(**params_from_coeffs(g["coeffs"]))
    ctx.set_walls(g["segments"], g["body_len"], g["body_kin"])
    ctx.set_noise(_lib.NOISE_NONE)
    ctx.step()                                   # P = 0
    assert ctx.particle_count() == 0
    ctx.set_state(np.array([[0.5, 0.3]]), np.array([[0.1, -0.2]]))
    ctx.step()
    pos, vel, prs = ctx.get_state()
    ref = O.step(g["coeffs"], [[0.5, 0.3]], [[0.1, -0.2]], g["segments"], g["body_len"], g["body_kin"])
    assert np.array_equal(pos, ref["pos_out"]) and np.array_equal(vel, ref["vel_out"]) and prs[0] == 0


def test_removal_append_and_identity():
    """remove_particles (crate.py:149-159) is stable; appended rows come last; rows keep their identity."""
    g = golden("step_stirring_cup_t150.npz")
    pos, vel = g["pos_in"].copy(), g["vel_in"].copy()
    pos[[3, 50, 200]] = [[-0.2, 0.5], [0.5, 1.2], [1.0051, 0.5]]           # outside [-r, 1 + r]
    ctx = _lib.Context(1000)
    ctx.set_params(**params_from_coeffs(g["coeffs"]))
    ctx.set_walls(g["segments"], g["body_len"], g["body_kin"])
    ctx.set_noise(_lib.NOISE_COUNTER, 9)
    ctx.set_state(pos, vel)
    ctx.step()
    keep = np.ones(len(pos), bool)
    keep[[3, 50, 200]] = False
    uid = np.arange(len(pos), dtype=np.uint32)[keep]
    ref = O.step(g["coeffs"], pos[keep], vel[keep], g["segments"], g["body_len"], g["body_kin"], noise_mode=1,
                 tkey=O.tick_key(9, 0), uid=uid)
    gp, gv, _ = ctx.get_state()
    assert ctx.particle_count() == keep.sum()
    assert np.array_equal(ctx.get_uids(), uid)
    assert np.array_equal(gp, ref["pos_out"]) and np.array_equal(gv, ref["vel_out"])
    extra = np.array([[0.4, 0.4], [0.41, 0.4]])
    ctx.append_particles(extra, np.zeros((2, 2)))
    gp2, _, _ = ctx.get_state()
    assert np.array_equal(gp2[:-2], gp) and np.array_equal(gp2[-2:], extra)
    assert ctx.get_uids()[-2:].tolist() == [len(pos), len(pos) + 1]


def test_pile_up_in_one_cell_and_trim():
    """Hundreds of particles in a single cell (in-cell rank sort, 20-trim everywhere), duplicates included."""
    rs = np.random.RandomState(4)
    pts = 0.5 + rs.rand(700, 2) * 0.004
    pts[100:120] = pts[100]                      # exact duplicates: ties broken by original index
    ctx = _lib.Context(16)
    rows, order, counts, idx = ctx.detect_particle_collisions(pts, 0.01)
    r2, o2, c2, i2 = O.detect_particle_collisions(pts, 0.01)
    assert np.array_equal(order, o2) and np.array_equal(counts, c2) and np.array_equal(idx, i2)
    assert (counts == 20).all()


def test_errors_are_loud():
    ctx = _lib.Context(4)
    with pytest.raises(_lib.SandCrateError, match="sc_set_params"):
        ctx.step()
    g = golden("step_stirring_cup_t150.npz")
    ctx.set_params(**params_from_coeffs(g["coeffs"]))
    with pytest.raises(_lib.SandCrateError, match="capacity"):
        ctx.set_state(g["pos_in"], g["vel_in"])
    with pytest.raises(_lib.SandCrateError, match="SC_MAX_SEGMENTS"):
        ctx.set_walls(np.zeros((40, 4)), [40], np.zeros((1, 5)))
    ctx.set_noise(_lib.NOISE_HOST)
    ctx.set_state(g["pos_in"][:4], g["vel_in"][:4])
    with pytest.raises(_lib.SandCrateError, match="sc_step_begin"):
        ctx.step()


def test_recut_histogram_counts_every_owned_particle_once():
    """sc_dist_row_histogram (the strip re-cutter's input): per cell row, the summed weight `base + pair count` of the
    particles in it.  Before the first tick there are no pair counts (weight = base); after ticks the total must be
    base * n + the directed pair count, and each row's weight must lie between base and base + 20 per particle."""
    import os
    import torch
    base = int(os.environ.get("SC_WORK_BASE", "2"))
    world, pos, vel = dam_break(60000)
    c = world.coefficients
    d = 2 * c["particle_radius"]
    stream = torch.cuda.Stream()
    ctx = _lib.Context(len(pos) + 1024, _lib.PRECISION_MIXED, 0, stream.cuda_stream)
    ctx.set_params(**{k: float(c[k]) for k in ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier",
                                               "ignored_pressure", "collider_noise_level", "viscosity",
                                               "surface_smoothing", "target_pressure")},
                   gravity_x=float(c["gravity"][0]), gravity_y=float(c["gravity"][1]))
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))
    ctx.set_noise(_lib.NOISE_COUNTER, 3)
    ctx.set_state_uids(pos, vel, np.arange(len(pos), dtype=np.uint32))
    ctx.dist_configure(0, 1, -(1 << 62), 1 << 62, 4, 1024)
    row0, nrows = int(np.floor(-2 * c["particle_radius"] / d)) - 1, int(np.ceil(1.0 / d)) + 4
    rows = np.clip(np.floor(pos[:, 1] / d).astype(np.int64) - row0, 0, nrows - 1)
    hist = ctx.dist_row_histogram(row0, nrows)
    assert np.array_equal(hist, base * np.bincount(rows, minlength=nrows).astype(np.uint64))
    for tick in range(3):
        ctx.set_tick(tick)
        ctx.step()
    hist = ctx.dist_row_histogram(row0, nrows).astype(np.int64)
    pairs = ctx.last_pair_count()            # before sc_dist_get_owned, which ends the validity of the tick's lists
    assert pairs > 3 * len(pos)
    narrow = ctx.dist_row_histogram(row0 + 100, 30).astype(np.int64)
    p, _, uid = ctx.dist_get_owned()
    assert len(uid) == len(pos)
    count = np.bincount(np.clip(np.floor(p[:, 1] / d).astype(np.int64) - row0, 0, nrows - 1), minlength=nrows)
    assert hist.sum() == base * len(p) + pairs, (hist.sum(), base * len(p), pairs)
    assert np.all(hist >= base * count) and np.all(hist <= (base + 20) * count)
    assert (hist > base * count).sum() > 20, "the pair counts must be in the weights"
    # a narrow window: rows outside it are clamped into its first / last bin, nothing is lost
    assert narrow.sum() == hist.sum() and np.array_equal(narrow[1:-1], hist[101:129])


def test_pending_unpack_admits_only_the_step():
    """sc_dist_unpack only records the receive buffers; the next step's pre-pass appends the records.  In between, the
    particle arrays and the device count lack them, so calls that read or change the state are refused - and the step
    then appends the neighbor's migrant as an owned particle and its halos as ghosts."""
    import torch
    from sand_crate_b200.strips import HALO_ROWS, INT64_MIN
    world, pos, vel = dam_break(4000, height=0.4)
    pos = pos - [0.0, 0.5]      # the column (y in 0.58 .. 0.99) lifted, so the neighbor's rows above it lie in the box
    c = world.coefficients
    r, d = c["particle_radius"], 2 * c["particle_radius"]
    ctx = _lib.Context(len(pos) + 1024, _lib.PRECISION_F64)
    ctx.set_params(**{k: float(c[k]) for k in _lib.PARAM_FIELDS[:9]},
                   gravity_x=float(c["gravity"][0]), gravity_y=float(c["gravity"][1]))
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))
    ctx.set_noise(_lib.NOISE_COUNTER, 3)
    ctx.set_state_uids(pos, vel, np.arange(len(pos), dtype=np.uint32))
    row_hi = int(np.floor(pos[:, 1] / d).max()) + 20      # an upper neighbor far above every particle, no lower one
    assert (row_hi + 2) * d < 1
    wire_cap = 256
    ctx.dist_configure(0, 2, INT64_MIN, row_hi, HALO_ROWS, wire_cap)
    ctx.step()
    p0, _, uid0 = ctx.dist_get_owned()
    removed = int(((p0 < -r) | (p0 > 1 + r)).any(axis=1).sum())   # what the next step's removal pass drops
    nbytes = _lib.wire_bytes(wire_cap)
    rec = np.dtype([("px", "f8"), ("py", "f8"), ("vx", "f8"), ("vy", "f8"), ("uid", "u4"), ("kind", "u4")])
    recs = np.array([(0.3, (row_hi - 2 + 0.5) * d, 0.0, 0.0, 1_000_000, 0),    # MIGRANT into this strip
                     (0.6, (row_hi + 0.5) * d, 0.0, 0.0, 1_000_001, 1),        # HALO rows of the neighbor
                     (0.7, (row_hi + 1.5) * d, 0.0, 0.0, 1_000_002, 1)], dtype=rec)
    raw = np.zeros(nbytes, np.uint8)
    raw[:16].view(np.uint32)[:] = [len(recs), 0, 0, 0]
    raw[16:16 + rec.itemsize * len(recs)].view(rec)[:] = recs
    send_hi, recv_hi = torch.zeros(nbytes, dtype=torch.uint8, device="cuda"), torch.from_numpy(raw).cuda()
    torch.cuda.synchronize()                              # written on torch's stream, used on the context's
    ctx.dist_pack(None, send_hi)
    ctx.dist_unpack(None, recv_hi)
    for call in (ctx.particle_count, lambda: ctx.dist_status(None, send_hi), ctx.dist_get_owned,
                 lambda: ctx.set_state_uids(pos, vel, np.arange(len(pos), dtype=np.uint32))):
        with pytest.raises(_lib.SandCrateError, match="unpack"):
            call()
    ctx.step()
    _, _, uid1 = ctx.dist_get_owned()
    assert 1_000_000 in uid1 and len(uid1) == len(uid0) - removed + 1
    assert ctx.dist_status()["n_local"] == len(uid0) - removed + 3


# ---- multi-GPU: strip decomposition over NCCL (needs >= 2 GPUs; skipped on a 1-GPU box) -------------------------
def test_strips_two_gpus_bit_identical_to_single_gpu():
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run tests/mgpu_check.py under torchrun on a multi-GPU box)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29517", os.path.join(root, "tests", "mgpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert res.stdout.count("bit-identical to single GPU = True") == 4, res.stdout


def test_force_monitor_on_gpu_matches_reference():
    """The force kernel's monitor mode (sc_set_monitor) reproduces the reference's ForceMonitor overlay."""
    from sand_crate_b200.crate import FORCE_SECTIONS
    world, g = world_from_freerun("wave_machine")
    crate = Crate(world, monitor=True, profile=True)
    for tick in range(1, 41):
        crate.physics_tick()
        if f"monitor_t{tick}" in g.files:
            got = np.array([crate.force_monitor.context_to_velocity[k] for k in FORCE_SECTIONS])
            assert np.allclose(got, g[f"monitor_t{tick}"], rtol=1e-10, atol=1e-15), tick
            assert np.array_equal(crate.particles, g[f"pos_t{tick}"])  # monitor mode does not change the physics
    text = crate.debug_prints
    assert "Forces" in text and "Timing" in text and "force_integrate" in text

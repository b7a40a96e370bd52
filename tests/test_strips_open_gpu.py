"""Open scenes on strips on ONE GPU: N strips of a scene as N contexts in lockstep on one stream (the driver of
tests/test_strips_gpu.py, extended by the phases of StripDomain.physics_tick that open scenes add), against one context
of the whole scene (`Crate(noise="counter")`, itself pinned to the oracle).  Particle sources, motored and free bodies
and removal run on every rank; the scene-count all-reduce of the emission clamp becomes a torch sum of the ranks'
device words on the shared stream.  Owned state gathered by uid must be bit-identical to the one context every 25
ticks.  Also: emission into a neighbor's halo rows (the pack must cover the appended tail), walls with more than two
contacts per particle (the halo follows the wall-fix reach), and the library's refusals of a halo that is too shallow."""
import numpy as np
import pytest
import torch

from conftest import world_from_freerun
from oracle import oracle as O
from sand_crate_b200 import Crate, WorldConfig, _lib
from sand_crate_b200.scenes import UNIT_BOX, box_fill
from sand_crate_b200.strips import INT64_MAX, INT64_MIN, StripDomain, emission_may_clamp
from test_strips_gpu import Lockstep, _assert_same_particles

SEED = 5
CHECK_EVERY = 25


class OpenLockstep(Lockstep):
    """Lockstep (test_strips_gpu.py) over StripDomain's own tick phases: advance_scene, draw_emission, count_owned +
    the sum over the ranks (instead of the all-reduce), emit, re-cut / slide, pack, exchange, unpack, step,
    finish_tick."""

    def __init__(self, world, nranks, *, pos=None, vel=None, precision="f64", direct=False, rebalance_every=0,
                 cuts=None, halo_rows=None, slack=2.0):
        self.stream = torch.cuda.Stream()
        self.n, self.t, self.every = nranks, 0, rebalance_every
        self.doms = []
        try:
            for k in range(nranks):
                self.doms.append(StripDomain(world, pos, vel, rank=k, world_size=nranks, precision=precision,
                                             noise="counter", noise_seed=SEED, stream=self.stream.cuda_stream,
                                             rebalance_every=rebalance_every, cuts=cuts, adaptive_rebalance=False,
                                             check_every=0, halo_rows=halo_rows, slack=slack))
        except Exception:
            self.close()
            raise
        self.cap = self.doms[0].wire_capacity
        self.recuts, self.collectives = 0, 0
        self.direct = direct
        if direct:
            self.slot = (_lib.wire_bytes(self.cap) + 15) // 16 * 16
            with self._on_stream():
                self.inbox = [torch.zeros(2 * self.slot + 16, dtype=torch.uint8, device="cuda") for _ in self.doms]

    def tick(self):
        for d in self.doms:
            d.advance_scene()
        records, may_clamp = self.doms[0].draw_emission()
        assert all(d.draw_emission() == (records, may_clamp) for d in self.doms[1:])
        count = None
        if may_clamp:
            words = [d.count_owned() for d in self.doms]
            with self._on_stream():
                count = torch.stack(words).sum(0, dtype=torch.int32)
            self.collectives += 1
        for d in self.doms:
            d.emit(records, count)
        self.begin()   # re-cut (histograms summed here) and slide
        self.pack()
        self.exchange()
        self.unpack()
        for d in self.doms:
            d.ctx.step()
            d.finish_tick()
        self.t += 1

    def close(self):
        for d in self.doms:
            d.close()


def _crate(world, precision, pos=None, vel=None):
    c = Crate(world, precision=precision, noise="counter", noise_seed=SEED)
    if pos is not None:
        c.set_particles(pos, vel)
    return c


def _crate_state(c):
    return c._ctx.get_uids(), np.array(c.particles), np.array(c.particle_velocities)


def _run_against_crate(ls, crate, ticks):
    """Step both; at every 25th tick (and the last) the gathered strips must equal the one context bit for bit."""
    checked = 0
    for t in range(1, ticks + 1):
        ls.tick()
        crate.physics_tick()
        if t % CHECK_EVERY == 0 or t == ticks:
            uid, p, v, _ = ls.gather()
            _assert_same_particles(uid, p, v, *_crate_state(crate), f"tick {t}: {ls.n} strips vs one context")
            checked += 1
    flagged = [(k, s) for k, s in enumerate(ls.status()) if s["overflow"] or s["too_far"]]
    assert not flagged, f"device flags raised: {flagged}"
    return checked


def _may_clamp_ticks(world, ticks, n0=0):
    """Ticks in which the host bound cannot rule the max_particles clamp out (counted independently of strips.py's
    bookkeeping, from the oracle's restatement of the counter stream)."""
    c, bound, k = world.coefficients, n0, 0
    for tick in range(ticks):
        drawn = sum(O.source_count(O.source_uniform(SEED, tick, q, 0), s["flow"], c["dt"])
                    for q, s in enumerate(world.particle_sources) if s["active_ticks"] > tick)
        if drawn:
            k += emission_may_clamp(bound, drawn, c["max_particles"])
            bound += drawn
    return k


def _world(name, max_particles=None):
    world, _ = world_from_freerun(name)
    if max_particles is not None:
        world.coefficients["max_particles"] = max_particles
    return world


# ---- 1. the shipped configs -------------------------------------------------------------------------------------------
CASES = [  # config, max_particles, ticks, strips, precision, transport, cuts, re-cut interval
    pytest.param("wave_machine", None, 600, 2, "f64", "copy", [INT64_MIN, 88, INT64_MAX], 0, id="wave_machine-2-f64-copy"),
    pytest.param("wave_machine", None, 600, 3, "mixed", "direct", [INT64_MIN, 80, 92, INT64_MAX], 0,
                 id="wave_machine-3-mixed-direct"),
    pytest.param("wave_machine", None, 600, 2, "mixed", "copy", None, 50, id="wave_machine-2-mixed-copy-recut50"),
    pytest.param("stirring_cup", None, 400, 2, "f64", "direct", None, 0, id="stirring_cup-2-f64-direct"),
    pytest.param("stirring_cup", None, 400, 3, "mixed", "copy", None, 0, id="stirring_cup-3-mixed-copy"),
    pytest.param("stirring_cup", 150, 400, 3, "f64", "copy", None, 0, id="stirring_cup-3-f64-clamp150"),
    pytest.param("wave_machine", 1500, 400, 2, "mixed", "direct", [INT64_MIN, 88, INT64_MAX], 0,
                 id="wave_machine-2-mixed-direct-clamp1500"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,max_particles,ticks,nranks,precision,transport,cuts,recut", CASES)
def test_shipped_config_on_strips_bit_identical_to_one_context(name, max_particles, ticks, nranks, precision,
                                                                transport, cuts, recut):
    """wave_machine (the source runs and stops at tick 500, the paddle moves; its walls need a 6-row halo) and
    stirring_cup (starts empty, motored cup, draining removal); with max_particles lowered the clamp binds while the
    sources run and particles are removed, and the scene count is taken exactly in the ticks the host bound says."""
    world = _world(name, max_particles)
    ls = OpenLockstep(world, nranks, precision=precision, direct=transport == "direct", cuts=cuts,
                      rebalance_every=recut)
    crate = _crate(world, precision)
    try:
        assert ls.doms[0].halo_rows == {"wave_machine": 6, "stirring_cup": 4}[name]
        assert _run_against_crate(ls, crate, ticks) >= ticks // CHECK_EVERY
        assert ls.collectives == _may_clamp_ticks(world, ticks) == ls.doms[0].scene_counts
        if max_particles is not None:
            assert ls.collectives > 0
        if recut:
            assert ls.recuts == (ticks - 1) // recut
    finally:
        ls.close()
        crate.close()


# ---- 2. a source whose square straddles the cuts: emission into the neighbors' halo rows -----------------------------
def _straddling_world():
    c = dict(world_from_freerun("wave_machine")[0].coefficients, max_particles=6000)
    src = {"radius": 0.12, "position": [0.5, 0.5], "velocity": [0.0, 0.5], "flow": 30000, "noise": 0.2,
           "active_ticks": 150}
    return WorldConfig(rigid_bodies=[UNIT_BOX], particle_sources=[src], coefficients=c)


@pytest.mark.gpu
@pytest.mark.parametrize("nranks,precision,transport", [(2, "f64", "copy"), (3, "f64", "direct"), (3, "mixed", "copy")])
def test_source_straddling_cuts_bit_identical(nranks, precision, transport):
    """The emission square covers rows 44 .. 55 and the cuts pass through it, so a particle emitted by the top rank
    can lie within a halo of its cut in the tick it appears: only the pack of that same tick makes it a halo of the rank
    below.  The arrays are in the last sort order then, and the appended tail lies outside the top rank's boundary
    zone [0, A), so the pack must reach the tail explicitly."""
    world = _straddling_world()
    cuts = [INT64_MIN, 50, INT64_MAX] if nranks == 2 else [INT64_MIN, 46, 54, INT64_MAX]
    ls = OpenLockstep(world, nranks, precision=precision, direct=transport == "direct", cuts=cuts)
    crate = _crate(world, precision)
    try:
        _run_against_crate(ls, crate, 5)
        owners = {k for k, d in enumerate(ls.doms) if len(d.owned()[0])}
        assert owners == set(range(nranks)), "every strip must have received emitted particles"
        _run_against_crate(ls, crate, 195)
    finally:
        ls.close()
        crate.close()


# ---- 3. a free body falling across a cut -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "mixed"])
def test_free_body_falling_across_a_cut(precision):
    """The recorded free_body config: a free bar (centre y = 0.75) falls under gravity while a source pours; the cut
    at row 80 lies below it, so the bar crosses into the lower strip.  From tick 104 on the bar crosses the floor,
    where its walls need a 6-row halo: the caller passes it."""
    world = _world("free_body")
    ls = OpenLockstep(world, 2, precision=precision, cuts=[INT64_MIN, 80, INT64_MAX], halo_rows=6)
    crate = _crate(world, precision)
    try:
        _run_against_crate(ls, crate, 150)
        bar = [b for b in ls.doms[0].bodies if b.kind == "free"][0]
        assert bar.segments[:, :, 1].min() > 0.8, "the bar must have fallen across the cut"
        assert all(np.array_equal(b.segments, c.segments) for d in ls.doms for b, c in zip(d.bodies, crate.rigid_bodies))
    finally:
        ls.close()
        crate.close()


# ---- 4. walls with more than two contacts per particle -----------------------------------------------------------------
def _fan_world(n=17000, spokes=6):
    """box_fill with a fixed fan of `spokes` segments meeting at (0.5, 0.52): near its hub a particle touches every
    spoke, so the wall fix can move it by several rows."""
    world, pos, vel = box_fill(n)
    hub, arm = np.array([0.5, 0.52]), 0.06
    fan = [[hub.tolist(), (hub + arm * np.array([np.cos(a), np.sin(a)])).tolist()]
           for a in np.linspace(0, 2 * np.pi, spokes, endpoint=False) + 0.3]
    world.rigid_bodies = [UNIT_BOX, {"fixed": {"name": "fan", "segments": fan}}]
    return world, pos, vel


def _oracle_run(world, pos, vel, ticks):
    from sand_crate_b200.rigid_body import build_rigid_bodies, wall_arrays
    c = world.coefficients
    cv = np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                   c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                   c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)
    seg, bl, bk = wall_arrays(build_rigid_bodies(world.rigid_bodies))
    uid = np.arange(len(pos), dtype=np.uint32)
    for tick in range(ticks):
        pos, vel, mask = O.remove_particles(pos, vel, c["particle_radius"])
        uid = uid[~mask]
        out = O.step(cv, pos, vel, seg.reshape(-1, 4), np.array(bl, np.int32), bk, noise_mode=1,
                     tkey=O.tick_key(SEED, tick), uid=uid, want_all=False)
        pos, vel = out["pos_out"], out["vel_out"]
    return uid, pos, vel


@pytest.mark.gpu
def test_fan_near_a_cut_takes_the_deeper_halo():
    """Six spokes within a few rows of the cut at row 52: sc_debug_walls reports >= 5 contacts, the default halo is
    2 + 2 ceil(V / 2) rows, and 3 strips in fp64 are bit-identical to one context and equal to the oracle."""
    world, pos, vel = _fan_world()
    d = 2 * world.coefficients["particle_radius"]
    ticks = 60
    ls = OpenLockstep(world, 3, pos=pos, vel=vel, precision="f64", cuts=[INT64_MIN, 52, 70, INT64_MAX])
    crate = _crate(world, "f64", pos, vel)
    try:
        V = ls.doms[0].ctx.debug_walls()["contacts"]
        assert V >= 5 and ls.doms[0].halo_rows == 2 + 2 * ((V + 1) // 2) > 4
        near = np.abs(np.floor(pos[:, 1] / d) - 52) <= 6
        assert near.sum() > 500
        _run_against_crate(ls, crate, ticks)
        uid, p, v, _ = ls.gather()
    finally:
        ls.close()
        crate.close()
    _assert_same_particles(uid, p, v, *_oracle_run(world, pos, vel, ticks), "3 strips vs the oracle", bitwise=False)


@pytest.mark.gpu
def test_halo_too_shallow_for_the_fan_is_refused():
    """halo_rows = 4 under the fan: sc_dist_configure refuses (naming the halo needed) and nothing runs."""
    world, pos, vel = _fan_world()
    from sand_crate_b200.rigid_body import build_rigid_bodies, wall_arrays
    need = _lib.dist_halo_rows(wall_arrays(build_rigid_bodies(world.rigid_bodies))[0], world.coefficients["particle_radius"])
    assert need == 8
    with pytest.raises(_lib.SandCrateError, match=f"halo_rows >= {need}"):
        OpenLockstep(world, 2, pos=pos, vel=vel, halo_rows=4, cuts=[INT64_MIN, 52, INT64_MAX])
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_motored_body_outgrowing_the_halo_is_refused_mid_run():
    """A motored segment slides into the box's corner: at tick 0 its walls need 4 halo rows, once its touch box
    overlaps both walls of the corner (3 contacts) they need 6.  sc_set_walls refuses that tick with a library error;
    the device has not faulted (the stream still synchronises and the strips still read back)."""
    c = dict(world_from_freerun("stirring_cup")[0].coefficients)
    slider = {"motored": {"name": "slider", "segments": [[[0.3, 0.99], [0.4, 0.99]]],
                          "velocity_func": "lambda t: np.array([-1.0, 0.0])"}}
    world = WorldConfig(rigid_bodies=[UNIT_BOX, slider], particle_sources=[], coefficients=c)
    _, pos, vel = box_fill(17000)
    ls = OpenLockstep(world, 2, pos=pos, vel=vel, cuts=[INT64_MIN, 60, INT64_MAX])
    try:
        assert ls.doms[0].halo_rows == 4
        with pytest.raises(_lib.SandCrateError, match="halo_rows >= 6"):
            for _ in range(400):
                ls.tick()
        assert 100 < ls.t < 400
        ls.stream.synchronize()
        uid, _, _, _ = ls.gather()
        assert len(uid) > 0
    finally:
        ls.close()


# ---- 5. one rank ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,precision,ticks", [("wave_machine", "mixed", 300), ("stirring_cup", "f64", 250)])
def test_one_rank_equals_crate(name, precision, ticks):
    """world_size = 1 through StripDomain.physics_tick itself: bit-identical to Crate(noise="counter")."""
    world = _world(name)
    stream = torch.cuda.Stream()
    dom = StripDomain(world, rank=0, world_size=1, precision=precision, noise="counter", noise_seed=SEED,
                      stream=stream.cuda_stream)
    crate = _crate(world, precision)
    try:
        for t in range(1, ticks + 1):
            dom.physics_tick()
            crate.physics_tick()
            if t % CHECK_EVERY == 0:
                _assert_same_particles(*dom.owned(), *_crate_state(crate), f"tick {t}: one rank vs Crate")
        assert dom.scene_counts == _may_clamp_ticks(world, ticks)
    finally:
        dom.close()
        crate.close()

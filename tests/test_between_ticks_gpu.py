"""The calls between ticks against an oracle model of a context.  The tick carries state from one tick to the next in
host-side flags (the next tick's keys, a clean grid, tick parity, the carried count, the pressure readback, ...); a
wrong transition gives no crash and no NaN, only a tick that runs on stale keys, walls or counts.  A seeded generator
draws sequences of calls - readbacks, taps, diagnostics, coefficient / wall / noise / tick edits, state changes,
sources, steps of every form and calls the library must refuse - and sends each to the library and to `ModelContext`,
the fp64 oracle restating what every call should do:

* fp64: every readback and tap equals the model bit for bit;
* mixed precision: every step is checked against the oracle run from the state read just before it (DESIGN.md
  section 2 bars), every tap and count exactly;
* both: the same sequence replayed with every call that must change nothing removed reaches byte-identical states,
  and a step after a window of such calls launches exactly the 5 kernels of a keyed tick, while a window with a call
  that changes what the keys depend on gives the 6 or 7 of a pre-pass / cold start.

Then the Crate-level checks: a Crate that grows its context keeps its particles' identities.  pytest -m gpu, B200."""
import copy
from collections import Counter

import numpy as np
import pytest

from conftest import world_from_freerun
from oracle import oracle as O
from oracle_backend import OracleContext
from sand_crate_b200 import Crate, WorldConfig, _lib
from sand_crate_b200 import crate as crate_mod
from sand_crate_b200._lib import SandCrateError
from sand_crate_b200.particle_source import build_particle_sources
from sand_crate_b200.rigid_body import build_rigid_bodies, wall_arrays
from sand_crate_b200.scenes import dam_break
from test_walls_gpu import contact_bound_np, grow_box

pytestmark = pytest.mark.gpu

COEFFS = ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier", "ignored_pressure",
          "collider_noise_level", "viscosity", "surface_smoothing", "target_pressure", "gravity_x", "gravity_y")


def contact_bound(seg, r):
    seg = np.asarray(seg, np.float64).reshape(-1, 4)
    return contact_bound_np([grow_box(*s, r * 1.2) for s in seg]) if len(seg) else 1


class ModelContext(OracleContext):
    """What a context should do between ticks, on the fp64 oracle.  Keeps the last tick's full oracle output (or the
    open split step's search) to answer the taps.  Pressure: what the last tick computed for each row, 0 for every row
    once set_state / append / emit changed the particle set (OracleContext), untouched by every other call."""

    def __init__(self, capacity):
        super().__init__(capacity)
        self.last = None            # O.step(..., want_all=True) of the last tick / of the open split step's search
        self.search = False         # the library holds a search state its taps can read
        self.in_step = False
        self.contacts = 1           # wall contacts the cell grid has room for (sc_set_walls / sc_set_params re-grid)
        self.regrids = Counter()
        self.changed = True         # parameters, walls or noise changed since the last step: sc_debug_rerun refuses
        self.removed = 0            # particles the last step removed
        self.step_mode = 0          # effective noise mode of the last step
        self.monitor_on = self.monitor_valid = False

    def _effective_mode(self):
        return self.noise_mode if self.params["collider_noise_level"] != 0 else 0

    def set_params(self, **kw):
        kw = {k: float(kw[k]) for k in COEFFS}
        if self.params == kw:
            return
        regrid = self.params is None or kw["particle_radius"] != self.params["particle_radius"]
        self.params, self.changed = kw, True
        if regrid:
            if self.walls is not None:
                self.contacts = max(self.contacts, contact_bound(self.walls[0], kw["particle_radius"]))
            self.search = False
            self.regrids["radius"] += 1

    def set_walls(self, segments, body_len, body_kin):
        new = (np.array(segments, np.float64).reshape(-1, 4), np.array(body_len, np.int32),
               np.array(body_kin, np.float64).reshape(-1, 5))
        if self.walls is not None and all(a.shape == b.shape and np.array_equal(a, b) for a, b in zip(new, self.walls)):
            return
        self.walls, self.changed = new, True
        v = contact_bound(new[0], self.params["particle_radius"])
        if v > self.contacts:
            self.contacts, self.search = v, False
            self.regrids["walls"] += 1

    def set_noise(self, mode, seed=0):
        if (mode, seed) != (self.noise_mode, self.seed):
            self.changed = True
        super().set_noise(mode, seed)

    def set_state(self, pos, vel):
        super().set_state(pos, vel)
        self.search = False

    def append_particles(self, pos, vel):
        super().append_particles(pos, vel)
        self.search = False

    def emit_particles(self, records, max_particles):
        if records:
            super().emit_particles(records, max_particles)
            self.search = False

    def step_begin(self):
        before = len(self.pos)
        self._sort_by_identity()
        self._remove()
        self.removed = before - len(self.pos)
        seg, bl, bk = self.walls
        self.last = O.step(self._coeffs(), self.pos, self.vel, seg, bl, bk, noise_mode=0) if len(self.pos) else None
        self.search, self.in_step = True, True
        return len(self.pos), 0 if self.last is None else int(self.last["nbr_count"].sum())

    def step_finish(self, noise=None):
        seg, bl, bk = self.walls
        mode = self._effective_mode()
        if len(self.pos):
            out = O.step(self._coeffs(), self.pos, self.vel, seg, bl, bk, noise_mode=mode, noise=noise,
                         tkey=O.tick_key(self.seed, self.tick), uid=self.uid & np.uint32(0x7FFFFFFF))
            self.pos, self.vel, self.prs = out["pos_out"], out["vel_out"], out["pressure"]
            self.last = out
        self.tick += 1
        self.in_step, self.changed, self.step_mode = False, False, mode
        self.monitor_valid = self.monitor_on

    def rerun_ok(self):
        return self.search and not self.in_step and not self.changed and len(self.pos) > 0 and self.step_mode != 2


# ---- the scene ----------------------------------------------------------------------------------------------------
def _scene():
    world, pos, vel = dam_break(1800)
    c = world.coefficients
    r, g, dt = c["particle_radius"], c["gravity"][1], c["dt"]
    # particles in the two bottom corners, outside both walls: gravity (+y) carries them out of the box within a few
    # ticks (removal while the force kernel computes the keys), and the stacked ones give the 20-trim
    corner = [[x, 1 + 0.98 * r] for k in range(4) for x in (1 + 0.96 * r, -0.96 * r)]
    up = [[0.0, -g * dt * (1 + 2.5 * k)] for k in range(4) for _ in range(2)]
    rs = np.random.RandomState(1)
    a, s = 2 * np.pi * rs.rand(24), 0.9 * r * np.sqrt(rs.rand(24))      # 24 particles within one diameter
    stack = np.array([0.3, 0.7]) + np.stack((s * np.cos(a), s * np.sin(a)), 1)
    pos = np.concatenate((pos, corner, stack))
    vel = np.concatenate((vel, up, np.zeros((24, 2))))
    params = {"dt": c["dt"], "particle_radius": r, "wall_collision_decay": c["wall_collision_decay"],
              "pressure_amplifier": c["pressure_amplifier"], "ignored_pressure": c["ignored_pressure"],
              "collider_noise_level": c["collider_noise_level"], "viscosity": c["viscosity"],
              "surface_smoothing": c["surface_smoothing"], "target_pressure": c["target_pressure"],
              "gravity_x": float(c["gravity"][0]), "gravity_y": float(c["gravity"][1])}
    box = np.array(world.rigid_bodies[0]["fixed"]["segments"], np.float64).reshape(-1, 4)
    wave, _ = world_from_freerun("wave_machine")
    bodies = build_rigid_bodies(wave.rigid_bodies)
    for b in bodies:
        b.apply_velocity(wave.coefficients["dt"])
    wseg, wbl, wkin = wall_arrays(bodies)
    hub = np.array([0.5, 1.0])     # a fan on the floor: 6 segments and the floor share a point (a larger grid)
    fan = [np.concatenate((hub, hub + 0.3 * np.array([np.cos(a), -np.sin(a)]))) for a in np.linspace(0.3, 2.8, 6)]
    moved = box.copy()
    moved[3] = [0.0, 1.0 - 2.2 * r, 1.0, 1.0 - 2.2 * r]
    walls = {"box": (box, [4], np.zeros((1, 5))), "moved": (moved, [4], np.zeros((1, 5))),
             "fewer": (box[:3], [3], np.zeros((1, 5))), "none": (np.zeros((0, 4)), [], np.zeros((0, 5))),
             "wave": (np.asarray(wseg, np.float64).reshape(-1, 4), list(wbl), wkin),
             "fan": (np.vstack([box] + fan), [4, 6], np.array([[0.0, 0, 0, 0, 0], [0.01, -0.02, 0.5, 0.5, 1.0]]))}
    sources = build_particle_sources(wave.particle_sources)
    return params, pos, vel, walls, sources


NOOPS = ("get_state", "get_uids", "particle_count", "synchronize", "last_pair_count", "taps", "pair_records", "grid",
         "debug_walls", "untiled_blocks", "rerun", "profile", "monitor", "same_params", "same_walls", "same_tick",
         "standalone")
REFUSALS = ("refuse_set_state_cap", "refuse_append_cap", "refuse_body_len", "refuse_host_step", "refuse_finish")
PHYSICS = ("params", "walls", "noise", "tick", "set_state", "set_state_uids", "append", "emit", "step", "step_n",
           "split_host", "split", "empty")
# calls that always change what the next tick's keys depend on (drop_keys); set_params / set_walls do when their bytes
# change and a re-run when it runs (op_*); set_noise and set_tick never do
KEY_DROPS = {"set_state", "set_state_uids", "append", "emit", "empty"}
WALLS = ("fan", "moved", "fewer", "none", "wave", "box")
IN_STEP = ("get_state", "get_uids", "append", "emit", "set_state", "step", "walls", "fan", "radius")
SCENE_TARGETS = ("wall contacts", "removed while keyed", "binding clamp", "20-trim", "regrid radius", "regrid walls",
                 "clamp not binding", "max below count", "append to capacity", "append 0")


def draw_sequence(seed, length=150):
    """Every kind once, in a seeded order, then seeded draws; steps between them so the calls sit between ticks."""
    rs = np.random.RandomState(seed)
    kinds = list(NOOPS + REFUSALS + PHYSICS)
    once = kinds + ["emit", "emit", "append", "append"]      # each of their three modes at least once
    seq = [once[i] for i in rs.permutation(len(once))]
    weights = np.array([3.0 if k in ("step", "split", "split_host") else 1.0 for k in kinds])
    seq += [kinds[i] for i in rs.choice(len(kinds), length - len(seq), p=weights / weights.sum())]
    out = []
    for k, kind in enumerate(seq):
        out.append((kind, int(rs.randint(1 << 30))))
        if k % 3 == 2:
            out.append(("step", int(rs.randint(1 << 30))))
    return out


class Runner:
    def __init__(self, precision, capacity, full):
        self.precision, self.full = precision, full
        self.params, self.pos0, self.vel0, self.walls, self.sources = _scene()
        self.lib = _lib.Context(capacity, precision)
        self.model = ModelContext(capacity)
        self.cap = capacity
        self.drawn, self.reached = Counter(), Counter()
        self.checkpoints = []
        self.dropped, self.keyed = True, False     # a key drop since the last step / the last step computed keys
        self.launch_checks = Counter()
        self.param_i = self.walls_i = self.emit_i = self.append_i = 0
        self.f64 = precision == _lib.PRECISION_F64
        for on in (self.lib, self.model):
            on.set_params(**self.params)
            on.set_walls(*self.walls["box"])
            on.set_noise(_lib.NOISE_COUNTER, 3)
        if full:   # taps before the first step
            for call in (lambda: self.lib.get_search(1), lambda: self.lib.get_neighbors(1)):
                with pytest.raises(SandCrateError, match="no search state"):
                    call()
        self.both("set_state", self.pos0, self.vel0)

    def both(self, name, *args, **kw):
        out = getattr(self.lib, name)(*args, **kw)
        getattr(self.model, name)(*args, **kw)
        return out

    def refused(self, entry, call):
        with pytest.raises(SandCrateError, match=entry):
            call()

    # ---- checks ----
    def check_state(self, want_pos=True, want_vel=True, want_pressure=True, reuse=False):
        m = self.model
        p, v, q = self.lib.get_state(want_pos=want_pos, want_vel=want_vel, want_pressure=want_pressure, reuse=reuse)
        assert self.lib.particle_count() == len(m.pos)
        assert np.array_equal(self.lib.get_uids(), m.uid)
        if want_pressure:
            assert np.array_equal(q, m.prs, equal_nan=True)
        if self.f64:
            assert want_pos is False or np.array_equal(p, m.pos, equal_nan=True)
            assert want_vel is False or np.array_equal(v, m.vel, equal_nan=True)

    def check_taps(self):
        m = self.model
        if not m.search:
            for call in (self.lib.get_search, self.lib.get_neighbors, self.lib.get_wall_counts):
                self.refused("no search state", lambda: call(self.cap))
            return
        last = m.last
        n = 0 if last is None else len(last["nbr_count"])
        if n == 0:
            return
        ps, rows, order = self.lib.get_search(n)
        d = 2 * m.params["particle_radius"]
        assert np.array_equal(ps, last["pos_search"], equal_nan=True)
        want = np.lexsort((ps[:, 0], np.floor(ps[:, 1] / d).astype(np.int64)))
        assert np.array_equal(order, want) and np.array_equal(rows, np.floor(ps[want, 1] / d).astype(np.int64))
        counts, idx = self.lib.get_neighbors(n)
        assert np.array_equal(counts, last["nbr_count"]) and np.array_equal(idx, last["nbr_idx_padded"])
        wc = self.lib.get_wall_counts(n)
        assert np.array_equal(wc, last["wall_count"])
        if wc.any():
            self.reached["wall contacts"] += 1
        if counts.max() == 20:
            self.reached["20-trim"] += 1
        if not m.in_step and self.f64:
            assert np.array_equal(self.lib.get_tension(n), last["tension_vec"], equal_nan=True)

    def step_check(self, before, kind):
        """Mixed precision: the step from the state read just before it, against the oracle with the DESIGN.md section 2
        bars; the model then takes the library's state, so later checks are exact again."""
        m = self.model
        p, v, q = self.lib.get_state()
        uid = self.lib.get_uids()
        assert np.array_equal(uid, m.uid) and len(p) == len(m.pos)
        if kind == "step" and before is not None and len(p):
            bp, bv, buid = before
            keep = np.isin(buid, uid)
            dv_ref = m.vel - bv[keep]
            d, dt = 2 * m.params["particle_radius"], m.params["dt"]
            assert np.array_equal(np.isnan(p), np.isnan(m.pos)) and np.array_equal(np.isnan(v), np.isnan(m.vel))
            assert np.nanmax(np.abs(p - m.pos), initial=0) <= 1e-5 * d
            assert np.nanmax(np.abs(v - m.vel), initial=0) <= 1e-5 * max(np.nanmax(np.abs(m.vel), initial=0), 0.01 * d / dt)
            dv_err = np.nanmax(np.abs((v - bv[keep]) - dv_ref), initial=0)
            assert dv_err <= 1e-5 * max(np.nanmax(np.abs(dv_ref), initial=0), 1e-300)
        else:
            m.last = None if kind != "step" else m.last
        m.pos, m.vel, m.prs = p, v, q

    def checkpoint(self):
        p, v, q = self.lib.get_state()
        self.checkpoints.append((p, v, q, self.lib.get_uids(), self.lib.particle_count()))

    # ---- the calls ----
    def run(self, seq):
        for k, (kind, seed) in enumerate(seq):
            if self.full or kind in PHYSICS:
                self.drawn[kind] += 1
                getattr(self, "op_" + kind)(np.random.RandomState(seed))
                if kind in KEY_DROPS:
                    self.dropped = True
            if k % 8 == 7:
                self.checkpoint()
        self.checkpoint()

    def pre_step(self):
        if self.f64 or not self.full:
            return None
        p, v, _ = self.lib.get_state()
        uid = self.lib.get_uids()
        m = self.model
        m.pos, m.vel, m.uid = p, v, uid
        return p, v, uid

    def post_step(self, keyed_step):
        """The step's bookkeeping: did it compute the next tick's keys, and did it remove particles while it ran on
        keys carried from the step before."""
        m = self.model
        if keyed_step and m.removed:
            self.reached["removed while keyed"] += 1
        self.keyed = len(m.pos) > 0 and not self.dropped
        self.dropped = False

    def op_step(self, rs):
        m = self.model
        if m.noise_mode == _lib.NOISE_HOST and m.params["collider_noise_level"] != 0:
            return self.op_split_host(rs)
        before = self.pre_step()
        carried = self.keyed and not self.dropped
        n = len(m.pos)
        start = self.lib.launch_count()
        self.both("step")
        launches = self.lib.launch_count() - start
        if self.keyed and n:
            # the last step computed keys: a window of calls that change nothing keeps them (5 launches), a call that
            # changes what they depend on takes them back (pre-pass: 6; and a cold start after a re-grid: 7)
            if carried:
                assert launches == 5
            else:
                assert launches in (6, 7)
            self.launch_checks[launches] += 1
        self.post_step(carried)
        if not self.f64 and self.full:
            self.step_check(before, "step")
        if self.full:
            self.check_taps()

    def op_step_n(self, rs):
        if self.model.noise_mode == _lib.NOISE_HOST and self.model.params["collider_noise_level"] != 0:
            return self.op_split_host(rs)
        k = int(rs.randint(2, 4))
        self.pre_step()
        self.lib.step(k)
        for _ in range(k):
            self.model.step()
            self.post_step(False)
        if not self.f64 and self.full:
            self.step_check(None, "step_n")

    def _split(self, rs, host):
        m = self.model
        if host:
            self.both("set_noise", _lib.NOISE_HOST, 0)
            if m.params["collider_noise_level"] == 0:
                self.op_params(rs, name="collider_noise_level")
        before = self.pre_step()
        carried = self.keyed and not self.dropped
        n, k = self.lib.step_begin()
        want = m.step_begin()
        if self.f64 or self.full:   # (a lean mixed replay is not resynchronised: its model drifts)
            assert (n, k) == want
        if self.full:
            self.check_taps()
            for what in IN_STEP:
                self.drawn["in_step_" + what] += 1
                self.in_step_refusal(what)
        noise = rs.rand(k, 2) if host else None
        self.lib.step_finish(noise)
        m.step_finish(noise)
        self.post_step(carried)
        if not self.f64 and self.full:
            self.step_check(before, "step")
        if self.full:
            self.check_taps()
        if host:
            self.both("set_noise", _lib.NOISE_COUNTER if rs.rand() < 0.7 else _lib.NOISE_NONE, int(rs.randint(5)))

    def in_step_refusal(self, what):
        L, m = self.lib, self.model
        one = np.full((1, 2), 0.5)
        calls = {"get_state": ("sc_get_state", L.get_state), "get_uids": ("sc_get_uids", L.get_uids),
                 "append": ("sc_append_particles", lambda: L.append_particles(one, one * 0)),
                 "emit": ("sc_emit_particles", lambda: L.emit_particles([self.sources[0].emit_record(0, 3)], 10 ** 6)),
                 "set_state": ("sc_set_state", lambda: L.set_state(one, one * 0)),
                 "step": ("sc_step", L.step),
                 "walls": ("sc_set_walls", lambda: L.set_walls(*self.other_walls("moved"))),
                 "fan": ("sc_set_walls", lambda: L.set_walls(*self.other_walls("fan"))),
                 "radius": ("sc_set_params", lambda: L.set_params(**dict(m.params,
                                                                        particle_radius=m.params["particle_radius"] * 1.01)))}
        entry, call = calls[what]
        self.refused(entry, call)

    def other_walls(self, name):
        """walls `name`, or the box when they are the current ones"""
        cur = self.model.walls[0]
        w = self.walls[name]
        same = w[0].shape == cur.shape and np.array_equal(w[0], cur)
        return self.walls["box"] if same else w

    def op_split_host(self, rs):
        self._split(rs, True)

    def op_split(self, rs):
        self._split(rs, False)

    def op_empty(self, rs):
        """An empty context steps (the count is carried in the scan tail), then particles arrive."""
        self.both("set_state", np.zeros((0, 2)), np.zeros((0, 2)))
        self.op_step(rs)
        if rs.rand() < 0.5:
            self.op_append(rs, rows=int(rs.randint(1, 300)))
        else:
            self.op_emit(rs, mode="free")
        if self.full:
            self.check_state()

    # configuration
    def op_params(self, rs, name=None):
        """Three coefficients per call, in turn (particle_radius first: a re-grid), or `name` alone."""
        m = self.model
        p = dict(m.params)
        names = [name] if name else [COEFFS[(1 + self.param_i + q) % len(COEFFS)] for q in range(3)]
        self.param_i += 0 if name else 3
        for name in names:
            base = self.params[name]
            if name == "collider_noise_level":
                p[name] = 0.0 if p[name] != 0 else base
            elif name == "particle_radius":
                p[name] = base * 1.04 if p[name] == base else base
            elif name == "gravity_x":
                p[name] = 0.0 if p[name] != 0 else 2.0
            else:
                p[name] = base * (0.8 + 0.4 * rs.rand())
        regrids = sum(m.regrids.values())
        self.dropped |= p != m.params
        self.both("set_params", **p)
        if sum(m.regrids.values()) > regrids:
            self.reached["regrid radius"] += 1
            if self.full:
                self.check_after_regrid()

    def op_walls(self, rs):
        """The wall sets in turn: the fan first (a re-grid), then a moved segment, fewer, none, wave_machine's, the box."""
        m = self.model
        w = self.other_walls(WALLS[self.walls_i % len(WALLS)])
        self.walls_i += 1
        before = m.regrids["walls"]
        self.dropped |= not (w[0].shape == m.walls[0].shape and np.array_equal(w[0], m.walls[0]) and
                             np.array_equal(np.asarray(w[2]).reshape(-1, 5), m.walls[2]))
        self.both("set_walls", *w)
        if m.regrids["walls"] > before:
            self.reached["regrid walls"] += 1
            if self.full:
                self.check_after_regrid()

    def check_after_regrid(self):
        """A re-grid keeps the pressures (defect: they read 0); the taps refuse, their cell boundaries are gone."""
        self.check_state()
        self.check_taps()

    def op_noise(self, rs):
        mode = [_lib.NOISE_COUNTER, _lib.NOISE_NONE][rs.randint(2)]
        self.both("set_noise", mode, int(rs.randint(1, 9)))

    def op_tick(self, rs):
        self.both("set_tick", max(0, self.model.tick + int(rs.randint(-5, 20))))

    # state
    def op_set_state(self, rs):
        keep = rs.rand(len(self.pos0)) < 0.9
        self.both("set_state", self.pos0[keep], self.vel0[keep])

    def op_set_state_uids(self, rs):
        keep = rs.rand(len(self.pos0)) < 0.9
        n = int(keep.sum())
        uid = np.sort(rs.choice(3 * n, n, replace=False)).astype(np.uint32)
        self.both("set_state_uids", self.pos0[keep], self.vel0[keep], uid)

    def op_append(self, rs, rows=None):
        n = len(self.model.pos)
        room = self.cap - n
        if rows is None:   # in turn: none, some, exactly up to the capacity
            rows = [0, int(rs.randint(1, max(room, 1) + 1)), room][self.append_i % 3]
            self.append_i += 1
        rows = min(rows, room)
        pos = 0.05 + 0.9 * rs.rand(rows, 2)
        vel = 0.1 * (rs.rand(rows, 2) - 0.5)
        self.both("append_particles", pos, vel)
        if rows == room:
            self.reached["append to capacity"] += 1
        if rows == 0:
            self.reached["append 0"] += 1

    def op_emit(self, rs, mode=None):
        m = self.model
        n = len(m.pos)
        cnt = int(rs.randint(5, 60))
        recs = [self.sources[0].emit_record(0, cnt)]
        if mode is None:   # in turn: the clamp binding, max_particles below the count, the clamp not binding
            mode = ["bind", "below", "free"][self.emit_i % 3]
            self.emit_i += 1
        if mode == "free" and n + cnt > self.cap:
            mode = "bind"
        if mode == "bind" and n + cnt // 2 > self.cap:
            mode = "below"
        if mode == "free":
            mx = n + cnt + int(rs.randint(0, 5))
            self.reached["clamp not binding"] += 1
        elif mode == "bind":
            mx = n + cnt // 2
            self.reached["binding clamp"] += 1
        else:
            mx = max(n - 5, 0)
            self.reached["max below count"] += 1
        self.both("emit_particles", recs, min(mx, self.cap))

    # must change nothing
    def op_get_state(self, rs):
        w = rs.rand(3) < 0.5
        self.check_state(bool(w[0]), bool(w[1]), bool(w[2]), reuse=bool(rs.rand() < 0.5))

    def op_get_uids(self, rs):
        assert np.array_equal(self.lib.get_uids(), self.model.uid)

    def op_particle_count(self, rs):
        assert self.lib.particle_count() == len(self.model.pos)

    def op_synchronize(self, rs):
        self.lib.synchronize()

    def op_last_pair_count(self, rs):
        m = self.model
        want = int(m.last["nbr_count"].sum()) if m.search and m.last is not None else 0
        got = self.lib.last_pair_count()
        if self.f64 or m.last is not None:
            assert got == want

    def op_taps(self, rs):
        self.check_taps()

    def op_pair_records(self, rs):
        m = self.model
        if m.search and m.last is not None and len(m.last["nbr_count"]):
            counts, rows, _ = self.lib.get_pair_records(len(m.last["nbr_count"]))
            assert np.array_equal(counts, m.last["nbr_count"]) and np.array_equal(rows, m.last["nbr_idx_padded"])

    def op_grid(self, rs):
        self.lib.grid()

    def op_debug_walls(self, rs):
        assert self.lib.debug_walls()["contacts"] == self.model.contacts

    def op_untiled_blocks(self, rs):
        self.lib.untiled_blocks()

    def op_rerun(self, rs):
        got = self.lib._L.sc_debug_rerun(self.lib._h, int(4 + rs.randint(2)), 2)
        assert (got >= 0) == self.model.rerun_ok()
        self.dropped |= got >= 0      # the re-run takes back the next tick's keys (include/sandcrate.h)

    def op_profile(self, rs):
        self.lib.profile_enable(bool(rs.rand() < 0.5))
        self.lib.profile_read()

    def op_monitor(self, rs):
        m = self.model
        if m.monitor_valid and m.monitor_on and m.last is not None and len(m.pos):
            sums, n = self.lib.get_monitor()
            assert n == len(m.pos)
            if self.f64:
                assert np.allclose(sums / n, m.last["force_monitor"], rtol=1e-10, atol=1e-15)
        on = bool(rs.rand() < 0.6)
        self.lib.set_monitor(on)
        m.monitor_on = on

    def op_same_params(self, rs):
        self.both("set_params", **self.model.params)

    def op_same_walls(self, rs):
        self.both("set_walls", *self.model.walls)

    def op_same_tick(self, rs):
        self.both("set_tick", self.model.tick)

    def op_standalone(self, rs):
        pts = rs.rand(50, 2)
        rows, order, counts, idx = self.lib.detect_particle_collisions(pts, 0.1)
        assert np.array_equal(order, np.lexsort((pts[:, 0], np.floor(pts[:, 1] / 0.1))))
        self.lib.points_to_segments_distance(pts, self.walls["box"][0])

    # must be refused, and change nothing
    def op_refuse_set_state_cap(self, rs):
        big = np.full((self.cap + 1, 2), 0.5)
        self.refused("sc_set_state", lambda: self.lib.set_state(big, big * 0))

    def op_refuse_append_cap(self, rs):
        rows = self.cap - len(self.model.pos) + 1
        pos = np.full((rows, 2), 0.5)
        self.refused("sc_append_particles", lambda: self.lib.append_particles(pos, pos * 0))

    def op_refuse_body_len(self, rs):
        seg, _, _ = self.walls["fan"]
        kin = np.array([[0.3, -0.2, 1.0, 0.5, 0.5], [0.1, 0.1, 0.1, 0.1, 0.1]])
        self.refused("body_len does not sum to S", lambda: self.lib.set_walls(seg, [4, 5], kin))

    def op_refuse_host_step(self, rs):
        m = self.model
        if m.params["collider_noise_level"] == 0:
            return
        mode = m.noise_mode
        self.both("set_noise", _lib.NOISE_HOST, m.seed)
        self.refused("sc_step", self.lib.step)
        self.both("set_noise", mode, m.seed)

    def op_refuse_finish(self, rs):
        self.refused("sc_step_finish", lambda: self.lib.step_finish(None))


CASES = [(_lib.PRECISION_F64, 2311, 11), (_lib.PRECISION_MIXED, 2053, 12)]


@pytest.mark.parametrize("precision,capacity,seed", CASES, ids=["f64", "mixed"])
def test_call_sequences_against_the_model(precision, capacity, seed):
    seq = draw_sequence(seed)
    full = Runner(precision, capacity, full=True)
    full.run(seq)
    for kind in NOOPS + REFUSALS + PHYSICS + tuple("in_step_" + w for w in IN_STEP):
        assert full.drawn[kind] > 0, f"the sequence never drew {kind}"
    for target in SCENE_TARGETS:
        assert full.reached[target] > 0, f"the sequence never reached: {target}"
    assert full.launch_checks[5] > 0 and full.launch_checks[6] + full.launch_checks[7] > 0
    # the same sequence without the calls that must change nothing: byte-identical at every shared checkpoint
    lean = Runner(precision, capacity, full=False)
    lean.run(seq)
    assert len(lean.checkpoints) == len(full.checkpoints)
    for a, b in zip(full.checkpoints, lean.checkpoints):
        for x, y in zip(a, b):
            assert np.asarray(x).tobytes() == np.asarray(y).tobytes()
    full.lib.close()
    lean.lib.close()


# ---- Crate level ----------------------------------------------------------------------------------------------------
def _wave_machine(max_particles):
    world, _ = world_from_freerun("wave_machine")
    c = copy.deepcopy(dict(world.coefficients))
    c["max_particles"] = max_particles
    return WorldConfig(rigid_bodies=world.rigid_bodies, particle_sources=world.particle_sources, coefficients=c)


@pytest.mark.parametrize("precision", ["f64", "mixed"])
def test_grown_crate_keeps_identities(precision):
    """Counter noise is keyed on uids: a Crate that grows its context when max_particles is raised stays identical to
    one with room from the start, tick for tick."""
    grown = Crate(_wave_machine(300), precision=precision, noise="counter", noise_seed=2)
    roomy = Crate(_wave_machine(300), precision=precision, noise="counter", noise_seed=2, capacity=4000)
    for tick in range(1, 121):
        if tick == 61:
            assert grown.particle_count == 300          # the clamp bound: the identities have gaps
            grown.max_particles = roomy.max_particles = 3000
        grown.physics_tick()
        roomy.physics_tick()
        assert np.array_equal(grown._ctx.get_uids(), roomy._ctx.get_uids()), tick
        assert np.array_equal(grown.particles, roomy.particles), tick
        assert np.array_equal(grown.particle_velocities, roomy.particle_velocities), tick
    assert grown._ctx.capacity > 300


def test_crate_with_live_edits_matches_the_oracle_crate(monkeypatch):
    """A script that reads every attribute and edits every coefficient between ticks - particle_radius, max_particles up
    and down, gravity among them - gives bit for bit the oracle-backed Crate's results in fp64."""
    def script(crate):
        seen = []
        base = dict(crate.world_config.coefficients)
        for tick in range(1, 121):
            if tick == 20:
                crate.viscosity = base["viscosity"] * 1.3
                crate.pressure_amplifier = base["pressure_amplifier"] * 0.9
            if tick == 30:
                crate.particle_radius = base["particle_radius"] * 1.05
                crate.gravity = np.array([1.0, 9.0])
            if tick == 40:
                crate.max_particles = 200
            if tick == 55:
                crate.max_particles = 3000
                crate.collider_noise_level = 0.0
                crate.surface_smoothing = base["surface_smoothing"] * 1.1
            if tick == 70:
                crate.particle_radius = base["particle_radius"]
                crate.collider_noise_level = base["collider_noise_level"]
                crate.wall_collision_decay = 0.3
                crate.ignored_pressure = 0.25
                crate.target_pressure = -1.5
                crate.dt = base["dt"] * 0.9
            crate.physics_tick()
            seen.append((crate.particle_count, crate.particles.copy(), crate.particle_velocities.copy(),
                         crate.particles_pressure.copy(), crate.segments.copy(), crate._ctx.get_uids()))
            crate.debug_prints
        return seen

    gpu = script(Crate(_wave_machine(300), noise="counter", noise_seed=4))
    monkeypatch.setattr(crate_mod._lib, "Context", OracleContext)
    ref = script(Crate(_wave_machine(300), noise="counter", noise_seed=4))
    for tick, (a, b) in enumerate(zip(gpu, ref), 1):
        for x, y in zip(a, b):
            assert np.array_equal(x, y), tick


def test_reference_noise_crate_growth_keeps_identities():
    world, _ = world_from_freerun("stirring_cup")
    grown = Crate(world, capacity=8)
    seen = []
    for _ in range(40):
        grown.physics_tick()
        seen.append((grown._ctx.get_uids(), grown.particles.copy()))
    roomy = Crate(world, capacity=4000)
    for tick, (uid, pos) in enumerate(seen, 1):
        roomy.physics_tick()
        assert np.array_equal(roomy._ctx.get_uids(), uid) and np.array_equal(roomy.particles, pos), tick
    assert grown._ctx.capacity > 8

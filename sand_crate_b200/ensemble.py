"""`Ensemble` - M variants of one scene (a coefficient sweep, seed replicas) stepped as members of ONE context.

    from sand_crate_b200 import Ensemble
    ens = Ensemble(world_config, [{"viscosity": 4}, {"viscosity": 8}], seeds=[0, 0])
    ens.physics_tick()
    ens.member(1).particles

One launch sequence per tick whatever M is (DESIGN.md section 12): the members' cell grids are stacked into one grid,
their uids carry the member in their high bits, and each member's coefficients and noise seed sit in a device table.
Every member is bit-identical to a `Crate` of the same precision and noise mode with that member's coefficients and
`noise_seed` - the same bar as fp64 parity and strips.

The members share `dt`, `particle_radius` and the walls (body motion depends on time and dt only, so it is evaluated
once per tick); `gravity` may differ only when the config has no free body (a free body falls with gravity, so its
walls would differ).  Modes: precision "f64" or "mixed"; noise "counter" or "none" ("reference" draws from the one
global NumPy stream of the process, which cannot be split between members).
"""
from __future__ import annotations

import copy
import itertools

import numpy as np

from . import _lib
from .crate import _NOISES, _PRECISIONS
from .load_config import WorldConfig  # noqa: F401 (type of world_config)
from .particle_source import build_particle_sources, counter_records
from .rigid_body import (FixedRigidBody, MotoredRigidBody, advance_bodies, apply_gravity_to_free_bodies,
                         build_rigid_bodies, wall_arrays)

SHARED = ("dt", "particle_radius")
# identity bits of a member by default: enough to number 16 x max_particles particles created over a member's life
UID_HEADROOM = 16


def default_uid_bits(max_particles, members: int) -> int:
    """B = the bits that number UID_HEADROOM x the largest member's max_particles (at least 10), so a member may create
    that many particles over its life; the readback map then takes 4 M 2^B bytes.  Raises when M members of B bits do
    not fit below 2^31."""
    need = max(UID_HEADROOM * max(int(x) for x in max_particles), 1 << 10)
    bits = (need - 1).bit_length()
    if (members << bits) > (1 << 31):
        raise ValueError(f"{members} members of {bits} identity bits do not fit 31-bit uids; pass member_uid_bits")
    return bits


def pack_uid(member: int, local, uid_bits: int):
    return (np.uint32(member) << np.uint32(uid_bits)) | np.asarray(local, np.uint32)


def unpack_uid(uid, uid_bits: int):
    """(member, local uid) of global uids."""
    uid = np.asarray(uid, np.uint32)
    return uid >> np.uint32(uid_bits), uid & np.uint32((1 << uid_bits) - 1)


def sweep_members(sweep: dict | None = None, replicas: int = 1):
    """The members of a sweep: the Cartesian product of `sweep` (coefficient -> list of values, in the mapping's
    order, the last coefficient varying fastest) times `replicas` seeds (innermost).  Returns (overrides, seeds)."""
    sweep = sweep or {}
    for k, v in sweep.items():
        if not isinstance(v, (list, tuple)) or not v:
            raise ValueError(f"sweep: {k!r} must map to a non-empty list of values")
    if int(replicas) < 1:
        raise ValueError("replicas must be >= 1")
    overrides, seeds = [], []
    for combo in itertools.product(*sweep.values()):
        for r in range(int(replicas)):
            overrides.append(dict(zip(sweep.keys(), combo)))
            seeds.append(r)
    return overrides, seeds


def member_coefficients(world_config: WorldConfig, members):
    """One full coefficient dict per member (the config's, overridden), checked against the ensemble model: raises
    ValueError naming the coefficient, member or free body that breaks it."""
    base = world_config.coefficients
    overrides = [{} for _ in range(members)] if isinstance(members, int) else [dict(o) for o in members]
    if not overrides:
        raise ValueError("an ensemble needs at least one member")
    coeffs = []
    for m, o in enumerate(overrides):
        for k in o:
            if k not in base:
                raise ValueError(f"member {m}: {k!r} is not a coefficient of this config")
        c = copy.deepcopy(dict(base))
        c.update(o)
        coeffs.append(c)
    for k in SHARED:
        for m, c in enumerate(coeffs):
            if float(c[k]) != float(coeffs[0][k]):
                raise ValueError(f"{k} differs between member 0 and member {m}: the members of an ensemble share {k}")
    free = [b for b in build_rigid_bodies(world_config.rigid_bodies)
            if not isinstance(b, (FixedRigidBody, MotoredRigidBody))]
    if free:
        for m, c in enumerate(coeffs):
            if list(map(float, c["gravity"])) != list(map(float, coeffs[0]["gravity"])):
                raise ValueError(f"gravity differs between member 0 and member {m}, but the free body "
                                 f"{free[0].name or 'free'!r} falls with gravity: the members would not share walls")
    return coeffs


def _sc_params(c) -> dict:
    g = c["gravity"]
    return dict(dt=c["dt"], particle_radius=c["particle_radius"], wall_collision_decay=c["wall_collision_decay"],
                pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                gravity_x=g[0], gravity_y=g[1])


def member_emission(sources, seeds, tick: int, dt: float):
    """The emission of one tick for every member: (records, counts) with `records` the `sc_source` tuples of the
    sources that emit in at least one member and counts[m, k] the count member m drew for records[k] from its own
    counter stream (`counter_records` with its seed), or (None, None) when no member emits."""
    per = [{r[7]: r for r in counter_records(sources, int(s), tick, dt)} for s in seeds]
    idx = sorted(set().union(*[p.keys() for p in per]))
    if not idx:
        return None, None
    records = [next(p[q] for p in per if q in p) for q in idx]
    counts = np.array([[p[q][6] if q in p else 0 for q in idx] for p in per], np.int32)
    return records, counts


class EnsembleMember:
    """Read view of member m with the drop-in attributes of a `Crate`: `particles`, `particle_velocities`,
    `particles_pressure`, `particle_count`, `uids` (local), and every coefficient - live-editable like `Crate`'s, except
    the shared ones."""

    def __init__(self, ens: "Ensemble", m: int) -> None:
        object.__setattr__(self, "_ens", ens)
        object.__setattr__(self, "_m", m)

    def _rows(self, key):
        st = self._ens._state()
        return st[key][st["off"][self._m]:st["off"][self._m + 1]]

    @property
    def particles(self):
        return self._rows("pos")

    @property
    def particle_velocities(self):
        return self._rows("vel")

    @property
    def particles_pressure(self):
        return self._rows("prs")

    @property
    def uids(self):
        return unpack_uid(self._rows("uid"), self._ens.uid_bits)[1]

    @property
    def particle_count(self) -> int:
        return int(self._ens.particle_counts()[self._m])

    @property
    def seed(self) -> int:
        return int(self._ens.seeds[self._m])

    @property
    def tick(self) -> int:
        return self._ens.tick

    @property
    def segments(self):
        return self._ens.segments

    def __getattr__(self, name):
        c = self._ens._coeffs[self._m]
        if name in c:
            return np.array(c[name]) if name == "gravity" else c[name]
        raise AttributeError(name)

    def __setattr__(self, name, value):
        c = self._ens._coeffs[self._m]
        if name not in c:
            raise AttributeError(f"{name!r} is not a coefficient")
        if name in SHARED:
            raise ValueError(f"{name} is shared by all members of an ensemble")
        trial = [dict(x) for x in self._ens._coeffs]
        trial[self._m][name] = value.tolist() if isinstance(value, np.ndarray) else value
        member_coefficients(self._ens.world_config, trial)   # e.g. per-member gravity with a free body
        c[name] = trial[self._m][name]   # pushed with the next tick, like Crate's


class Ensemble:
    def __init__(self, world_config: WorldConfig, members, *, seeds=None, precision: str = "mixed",
                 noise: str = "counter", device: int = 0, stream: int | None = None,
                 member_uid_bits: int | None = None) -> None:
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
        if noise not in ("counter", "none"):
            raise ValueError(f"noise={noise!r}: an ensemble runs noise 'counter' or 'none' - the reference stream "
                             "('reference') is one global NumPy stream per process and cannot be split between members")
        self._coeffs = member_coefficients(world_config, members)
        M = len(self._coeffs)
        if seeds is None:   # replicas: one seed each; a sweep: Crate's default seed for every variant
            seeds = list(range(M)) if isinstance(members, int) else [0] * M
        if len(seeds) != M:
            raise ValueError(f"{len(seeds)} seeds for {M} members")
        self.world_config, self.precision, self.noise = world_config, precision, noise
        self.members, self.seeds = M, [int(s) for s in seeds]
        self.uid_bits = int(member_uid_bits) if member_uid_bits is not None else default_uid_bits(
            [c["max_particles"] for c in self._coeffs], M)
        self.tick = 0
        self.rigid_bodies = build_rigid_bodies(world_config.rigid_bodies)
        self.particle_sources = build_particle_sources(world_config.particle_sources)
        self._device, self._stream = device, stream
        # per member: an upper bound of its live count (the rule of sc_ens_emit_particles) and its next local uid
        self._bound = np.zeros(M, np.int64)
        self._next = np.zeros(M, np.int64)
        self._ctx = None
        self._cache: dict = {}
        self._open(sum(max(int(c["max_particles"]), 1) for c in self._coeffs))

    def _open(self, capacity: int) -> None:
        self._ctx = _lib.Context(capacity, _PRECISIONS[self.precision], self._device, self._stream)
        try:
            self._ctx.set_noise(_NOISES[self.noise], 0)
            self._ctx.ens_configure(self.members, self.uid_bits)
            self._push_params()
        except Exception:
            self.close()
            raise

    def _ensure_capacity(self, bound, keep: bool = True) -> None:
        """A context with room for the members' count bounds.  When they outgrow it, the new context takes room for
        every member's max(bound, max_particles) at once, so a raised max_particles costs one move, not one per tick.
        Growing moves the state - positions, velocities, every member's identities and next uid - to the new context,
        so each member continues exactly as it would have (its results do not depend on where its particles sit in the
        arrays)."""
        if int(np.sum(bound)) <= self._ctx.capacity:
            return
        maxp = np.array([max(int(c["max_particles"]), 1) for c in self._coeffs], np.int64)
        need = int(np.maximum(bound, maxp).sum())
        if keep:
            pos, vel, _, off = self._ctx.ens_get_state(want_pressure=False)
            uid = self._ctx.get_uids()
        self._cache = {}
        self._ctx.close()
        self._open(int(need))
        if keep:
            self._ctx.ens_set_state(pos, vel, np.diff(off), uid, self._next)

    # ---- state -------------------------------------------------------------------------------------------------
    @property
    def dt(self) -> float:
        return float(self._coeffs[0]["dt"])

    @property
    def segments(self) -> np.ndarray:
        if not self.rigid_bodies:
            return np.zeros((0, 2, 2))
        return np.vstack([body.segments for body in self.rigid_bodies])

    def member(self, m: int) -> EnsembleMember:
        if not 0 <= m < self.members:
            raise IndexError(m)
        return EnsembleMember(self, m)

    def particle_counts(self) -> np.ndarray:
        if "counts" not in self._cache:
            self._cache["counts"] = self._ctx.ens_member_counts()
        return self._cache["counts"]

    def member_counts_to(self, counts_dev) -> None:
        """Enqueue the members' live counts into the M uint32 device words `counts_dev` (a device address or a tensor):
        no host wait."""
        self._ctx.ens_member_counts(counts_dev, want_host=False)

    def set_particles(self, particles, velocities=None) -> None:
        """The whole state: one (n_m x 2) array per member (velocities likewise, or None for zero)."""
        pos = [np.asarray(p, np.float64).reshape(-1, 2) for p in particles]
        vel = [np.zeros_like(p) for p in pos] if velocities is None else [
            np.asarray(v, np.float64).reshape(-1, 2) for v in velocities]
        if len(pos) != self.members:
            raise ValueError(f"{len(pos)} particle sets for {self.members} members")
        counts = np.array([len(p) for p in pos], np.int64)
        self._ensure_capacity(counts, keep=False)
        self._push_params()
        self._ctx.ens_set_state(np.vstack(pos), np.vstack(vel), counts)
        self._bound, self._next = counts.copy(), counts.copy()
        self._cache = {}

    def _state(self) -> dict:
        if "pos" not in self._cache:
            pos, vel, prs, off = self._ctx.ens_get_state()
            self._cache.update(pos=pos, vel=vel, prs=prs, off=off, uid=self._ctx.get_uids())
        return self._cache

    # ---- the tick ----------------------------------------------------------------------------------------------
    def physics_tick(self) -> None:
        """Crate.physics_tick for every member: sources (each member's own stream), body motion (once), coefficient
        push, one step of all members."""
        records, counts = member_emission(self.particle_sources, self.seeds, self.tick, self.dt)
        if records:
            maxp = np.array([max(int(c["max_particles"]), 0) for c in self._coeffs], np.int64)
            drawn = counts.sum(1).astype(np.int64)
            # a member's clamp lets its count grow to at most max(P, min(P + drawn, max_particles)); max_particles is
            # live-editable and a state may start above it, so the context grows before the clamps could outgrow it
            bound = np.maximum(self._bound, np.minimum(self._bound + drawn, maxp))
            self._ensure_capacity(bound)
            self._push_params()
            self._ctx.set_tick(self.tick)
            self._ctx.ens_emit_particles(records, counts, maxp)
            self._bound = bound
            self._next += drawn
        advance_bodies(self.rigid_bodies, self.dt)
        self._push_params()
        self._ctx.set_walls(*wall_arrays(self.rigid_bodies))
        self._ctx.set_tick(self.tick)
        self._ctx.step()
        apply_gravity_to_free_bodies(self.rigid_bodies, self.dt, np.asarray(self._coeffs[0]["gravity"], np.float64))
        self._cache = {}
        self.tick += 1

    def _push_params(self) -> None:
        self._ctx.ens_set_params([_sc_params(c) for c in self._coeffs], self.seeds)

    # ---- measurement -------------------------------------------------------------------------------------------
    def synchronize(self) -> None:
        self._ctx.synchronize()

    def launch_count(self) -> int:
        return self._ctx.launch_count()

    def sync_count(self) -> int:
        return self._ctx.sync_count()

    def untiled_blocks(self) -> int:
        return self._ctx.untiled_blocks()

    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None:
            self._cache = {}
            self._ctx.close()
            self._ctx = None

"""`Crate` - drop-in for the reference's simulation step object (`src/crate/crate.py:19-371`).

Same constructor (`Crate(world_config)`), same `physics_tick()`, same attributes the front end reads
(`particles`, `particle_velocities`, `particles_pressure`, `segments`, `particle_radius`, `gravity`, `tick`,
`particle_count`, `debug_prints`, `debug_arrows`, every `world.coefficients` key as a live-editable attribute),
but the tick itself runs as sm_100a CUDA kernels behind the C ABI of `include/sandcrate.h`.  There is no NumPy
or CPU implementation of the step in this package: without the CUDA library and a B200 the constructor raises.

What stays on the host (inputs of the GPU step, O(#bodies) per tick): rigid-body motion, which evaluates the YAML
lambda strings, and - in the reference-stream mode only - the particle sources, which consume the reference's global
NumPy RNG (SURVEY.md section 2, rows "Rigid bodies" and "Particle sources").  In the counter mode the sources run on
the device (`sc_emit_particles`) and a tick never waits for the GPU.

Modes (keyword-only, the defaults reproduce the reference bit for bit):
  precision  "f64"   fp64 kernels, reference summation orders        | "mixed"  fp64 positions, fp32 forces
  noise      "reference"  per-pair collider noise drawn from the global `np.random` stream exactly where the
                          reference draws it (crate.py:168-170); costs one host round trip per tick
             "counter"    counter-based device noise keyed on (seed, tick, uid_i, uid_j); no host round trip
             "none"       noise term skipped
"""
from __future__ import annotations

import numpy as np
import yaml

from . import _lib
from .load_config import WorldConfig
from .particle_source import build_particle_sources, counter_records
from .rigid_body import advance_bodies, apply_gravity_to_free_bodies, build_rigid_bodies, wall_arrays

_PRECISIONS = {"f64": _lib.PRECISION_F64, "mixed": _lib.PRECISION_MIXED}
_NOISES = {"reference": _lib.NOISE_HOST, "counter": _lib.NOISE_COUNTER, "none": _lib.NOISE_NONE}


FORCE_SECTIONS = ("tension", "gravity", "pressure", "viscosity", "wall_bounce", "continuous_collision")


class ForceMonitor:
    """The reference's diagnostic overlay (utils/force_monitor.py:13-37): per force section of the tick
    (crate.py:110-124) an exponential moving average, decay 0.8, of the mean |dv| the section caused.  The six sums
    come from the force kernel's monitor mode (`sc_set_monitor`); enabling it costs six atomics per particle."""

    DECAY = 0.80

    def __init__(self) -> None:
        self.context_to_velocity: dict = {}

    def update(self, sums, count: int) -> None:
        if count == 0:  # force_monitor.py:28-29
            return
        for name, total in zip(FORCE_SECTIONS, sums):
            prev = self.context_to_velocity.get(name, 0)
            self.context_to_velocity[name] = prev * self.DECAY + (1 - self.DECAY) * (total / count)

    def report(self) -> str:
        rounded = {name: float(f"{1000 * v:.1f}") for name, v in self.context_to_velocity.items()}
        return yaml.dump({"Forces": rounded})


class KernelTimer:
    """Counterpart of the reference's `Timer` (utils/timer.py:10-48): per section an exponential moving average,
    decay 0.9, of its duration - here the sections are the tick's kernels, timed with CUDA events on the stream."""

    DECAY = 0.9

    def __init__(self) -> None:
        self.durations: dict = {}
        self._seen: dict = {}

    def update(self, totals: dict) -> None:
        for name, rec in totals.items():
            launches, ms = self._seen.get(name, (0, 0.0))
            if rec["launches"] > launches:
                dur = (rec["ms"] - ms) / (rec["launches"] - launches) * 1e-3
                self.durations[name] = self.durations.get(name, 0) * self.DECAY + (1 - self.DECAY) * dur
            self._seen[name] = (rec["launches"], rec["ms"])

    def report(self) -> str:
        frame = sum(self.durations.values())
        if frame <= 0:
            return yaml.dump({"Timing": {}, "FPS": "n/a"})
        rows = {k: f"{1e6 * v:.0f} us ({100 * v / frame:.0f}%)" for k, v in self.durations.items()}
        return yaml.dump({"Timing": rows, "FPS": f"{int(1 / frame)} ({1e3 * frame:.3f} ms)"})


class Crate:
    def __init__(self, world_config: WorldConfig, *, precision: str = "f64", noise: str = "reference",
                 device: int = 0, noise_seed: int = 0, capacity: int | None = None, stream: int | None = None,
                 profile: bool = False, monitor: bool = False) -> None:
        np.random.seed(0)  # crate.py:22 - sources and reference-mode noise share this global stream
        self.tick: int = 0
        self.debug_arrows: list = []
        self.debug_prints: str = ""
        self.world_config = world_config
        self.rigid_bodies = build_rigid_bodies(world_config.rigid_bodies)
        self.particle_sources = build_particle_sources(world_config.particle_sources)
        for name in self.editable_coefficients():  # crate.py:55-56: every YAML key becomes a live attribute
            setattr(self, name, world_config.coefficients[name])
        self.gravity = np.array(world_config.coefficients["gravity"])

        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
        if noise not in _NOISES:
            raise ValueError(f"noise must be one of {sorted(_NOISES)}")
        self.precision, self.noise = precision, noise
        self._noise_seed = int(noise_seed)
        self._device, self._stream, self._profile, self._monitor = device, stream, profile, monitor
        self.force_monitor = ForceMonitor()
        self.debug_timer = KernelTimer()
        cap = int(capacity if capacity is not None else max(int(getattr(self, "max_particles", 0) or 0), 1))
        self._ctx = None
        self._open_context(cap)
        self._count = 0
        self._next_uid = 0   # the uid the context gives the next new particle, tracked here so that growing keeps it
        self._cache: dict = {}
        self._kernel_ms: dict = {}

    # ---- context management ----------------------------------------------------------------------------
    def _open_context(self, capacity: int) -> None:
        self._ctx = _lib.Context(capacity, _PRECISIONS[self.precision], self._device, self._stream)
        self._ctx.set_noise(_NOISES[self.noise], self._noise_seed)
        if self._profile:
            self._ctx.profile_enable(True)
        if self._monitor:
            self._ctx.set_monitor(True)

    def _ensure_capacity(self, needed: int) -> None:
        """Moves the scene into a larger context with its identities: counter noise is keyed on uids, so renumbering
        the particles would change the trajectory."""
        if needed <= self._ctx.capacity:
            return
        pos, vel, _ = self._ctx.get_state(want_pressure=False)   # own arrays: they must outlive the old context
        uid = self._ctx.get_uids()
        self._cache = {}
        self._ctx.close()
        self._open_context(max(needed, 2 * self._ctx.capacity))
        self._push_params()
        self._ctx.set_tick(self.tick)
        if len(pos):
            self._ctx.set_state_uids(pos, vel, uid)
        # set_state_uids continues after the largest uid; a clamped emission or a removal can leave a gap above it
        if self._next_uid != (int(uid.max()) + 1 if len(uid) else 0):
            self._ctx.set_next_uid(self._next_uid)

    def close(self) -> None:
        if self._ctx is not None:
            self._cache = {}
            self._ctx.close()
            self._ctx = None

    # ---- reference surface -------------------------------------------------------------------------------
    def editable_coefficients(self) -> list[str]:
        return list(self.world_config.coefficients.keys())

    @property
    def diameter(self) -> float:
        return self.particle_radius * 2

    @property
    def segments(self) -> np.ndarray:
        if not self.rigid_bodies:
            return np.zeros((0, 2, 2))
        return np.vstack([body.segments for body in self.rigid_bodies])

    @property
    def particle_count(self) -> int:
        if self._count is None:  # removal happens on the device (crate.py:149-159); synchronise lazily
            self._count = self._ctx.particle_count()
        return self._count

    def _fetch(self, key: str) -> np.ndarray:
        """One device -> host read per attribute per tick, into page-locked buffers that are refilled in place: like
        the reference's arrays, what `particles` returned last tick is overwritten by this tick's read."""
        if key not in self._cache:
            pos, vel, prs = self._ctx.get_state(want_pos=key == "pos", want_vel=key == "vel",
                                                want_pressure=key == "prs", reuse=True)
            self._cache[key] = {"pos": pos, "vel": vel, "prs": prs}[key]
        return self._cache[key]

    @property
    def particles(self) -> np.ndarray:
        return self._fetch("pos")

    @property
    def particle_velocities(self) -> np.ndarray:
        return self._fetch("vel")

    @property
    def particles_pressure(self) -> np.ndarray:
        return self._fetch("prs")

    def set_particles(self, particles, velocities=None) -> None:
        """Replaces the whole particle set (rows get indices 0..n-1).  Not in the reference (it only grows through
        sources); used by the synthetic scenes and the parity tests."""
        particles = np.ascontiguousarray(particles, dtype=np.float64).reshape(-1, 2)
        velocities = np.zeros_like(particles) if velocities is None else np.ascontiguousarray(
            velocities, dtype=np.float64).reshape(-1, 2)
        self._ensure_capacity(len(particles))
        self._push_params()
        self._ctx.set_state(particles, velocities)
        self._count = len(particles)
        self._next_uid = len(particles)
        self._cache = {}

    # ---- the tick ------------------------------------------------------------------------------------------
    def physics_tick(self) -> None:
        """crate.py:91-129.  Host part: sources, body motion, coefficient push.  Device part: everything else."""
        self.create_new_particles()
        self.debug_arrows = []
        self.apply_bodies_velocity()
        self._push_params()
        self._push_walls()
        self._ctx.set_tick(self.tick)
        if self.noise == "reference":
            # taken even when collider_noise_level == 0: the reference still consumes the stream (crate.py:169)
            n, n_pairs = self._ctx.step_begin()
            # one draw of sum(K_i) x 2 == the reference's per-particle rand(K_i, 2) calls back to back
            self._ctx.step_finish(np.random.rand(n_pairs, 2))
            self._count = n
        else:
            self._ctx.step()      # asynchronous; the live count stays on the device until somebody asks
            self._count = None
        self.apply_gravity_to_free_bodies()
        self._cache = {}
        self.tick += 1
        if self._monitor:
            self.force_monitor.update(*self._ctx.get_monitor())
        if self._profile:
            self.debug_timer.update(self._ctx.profile_read())

    def create_new_particles(self) -> None:  # crate.py:138-147
        if self.noise != "reference":
            return self._emit_on_device()
        for source in self.particle_sources:
            if source.active_ticks <= self.tick:
                continue
            new_pos, new_vel = source.generate_particles(dt=self.dt, max_particles=self.max_particles - self.particle_count)
            if new_pos is not None:
                self._ensure_capacity(self.particle_count + len(new_pos))
                self._push_params()
                self._ctx.append_particles(new_pos, new_vel)
                self._count = self.particle_count + len(new_pos)
                self._next_uid += len(new_pos)
                self._cache = {}

    def _emit_on_device(self) -> None:
        """Production mode: the emission counts come from the counter stream (host arithmetic only), the particles
        are generated, clamped to max_particles and appended by the device - no synchronisation (the reference-stream
        path above has to know the live count, which costs a device round trip per tick while sources are active)."""
        records = counter_records(self.particle_sources, self._noise_seed, self.tick, self.dt)
        if records:
            self._ensure_capacity(int(self.max_particles))   # a no-op after the first call: capacity = max_particles
            self._push_params()
            self._ctx.set_tick(self.tick)
            self._ctx.emit_particles(records, int(self.max_particles))
            self._next_uid += sum(max(int(r[6]), 0) for r in records)   # identities advance by the drawn counts
            self._count = None
            self._cache = {}

    def apply_bodies_velocity(self) -> None:  # crate.py:363-365
        advance_bodies(self.rigid_bodies, self.dt)

    def apply_gravity_to_free_bodies(self) -> None:  # crate.py:311-314 (the particle part runs on the device)
        apply_gravity_to_free_bodies(self.rigid_bodies, self.dt, self.gravity)

    def _push_params(self) -> None:
        g = np.asarray(self.gravity, dtype=np.float64)
        self._ctx.set_params(dt=self.dt, particle_radius=self.particle_radius,
                             wall_collision_decay=self.wall_collision_decay,
                             pressure_amplifier=self.pressure_amplifier, ignored_pressure=self.ignored_pressure,
                             collider_noise_level=self.collider_noise_level, viscosity=self.viscosity,
                             surface_smoothing=self.surface_smoothing, target_pressure=self.target_pressure,
                             gravity_x=g[0], gravity_y=g[1])

    def _push_walls(self) -> None:
        self._ctx.set_walls(*wall_arrays(self.rigid_bodies))

    # ---- overlay text (crate.py:131-136, 367-371) ------------------------------------------------------------
    @property
    def debug_prints(self) -> str:
        """Built on demand so a headless run never synchronises for the overlay."""
        text = f"Tick: {self.tick}\nParticles: {self.particle_count}\n"
        if self._profile:
            text += self.debug_timer.report()
        if self._monitor:
            text += f"\n\n{self.force_monitor.report()}"
        text += f"\n\n{self.get_coefficient_debug()}"
        return text

    @debug_prints.setter
    def debug_prints(self, value: str) -> None:  # the reference assigns it (crate.py:35); accepted and ignored
        pass

    def get_coefficient_debug(self) -> str:
        rows = []
        for name in self.editable_coefficients():
            val = getattr(self, name)
            rows.append({name: val.tolist() if isinstance(val, np.ndarray) else val})
        return yaml.dump(rows)

    # ---- parity taps (not in the reference; used by tests) ---------------------------------------------------
    def last_search(self):
        pos, rows, order = self._ctx.get_search(self.particle_count)
        return pos, rows, order

    def last_neighbors(self):
        counts, idx = self._ctx.get_neighbors(self.particle_count)
        return counts, idx

    def kernel_timings(self) -> dict:
        return self._ctx.profile_read()

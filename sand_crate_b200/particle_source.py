"""Particle sources (reference `src/crate/particle_source.py:9-28`, driven by `Crate.create_new_particles`,
crate.py:138-147), in the two forms the drop-in `Crate` needs:

* **reference stream** (`noise="reference"`): the emission count, positions and velocities are drawn on the host from
  the reference's global NumPy MT19937 stream, in the reference's order (binomial, rand(n, 2), rand(n, 2)), because
  that stream is shared with the step's own per-pair draws (SURVEY.md section 8(c) "noise protocol"); this is what
  makes whole runs bit-identical to the reference.  The rows are handed to the GPU with `sc_append_particles`.
* **counter stream** (`noise="counter"` / `"none"`, production): only the emission COUNT is drawn on the host - from a
  counter-based stream keyed on (seed, tick, source index), no device data needed - and the particles themselves are
  generated, clamped to `max_particles` and appended by the device (`sc_emit_particles`), so a tick with active sources
  costs no host <-> device round trip.  `oracle/oracle.py::emit_counter` restates the device side for the parity tests.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import numpy as np


def binomial_inverse_cdf(u: float, trials: int, p: float) -> int:
    """Smallest k with P(Binomial(trials, p) <= k) >= u, by summing the probability mass upwards from k = 0 (the
    sources of the shipped configs have mean trials * p = 4 and 14)."""
    if trials <= 0 or p <= 0.0:
        return 0
    if p >= 1.0:
        return int(trials)
    q = 1.0 - p
    mass = math.pow(q, trials)
    cdf = mass
    k = 0
    ratio = p / q
    while u > cdf and k < trials:
        k += 1
        mass *= (trials - k + 1) / k * ratio
        cdf += mass
    return k


@dataclass
class ParticleSource:
    radius: float
    position: list
    velocity: list
    flow: float
    active_ticks: int
    noise: float = 0.05

    # ---- reference stream (host) --------------------------------------------------------------------------------
    def generate_particles(self, dt: float, max_particles: int) -> tuple[Optional[np.ndarray], Optional[np.ndarray]]:
        # same draws in the same order as particle_source.py:18-23: binomial, rand(n, 2), rand(n, 2)
        emitted = min(np.round(np.random.binomial(self.flow, dt)), max_particles)
        if emitted == 0:
            return None, None
        jitter = np.random.rand(emitted, 2) - 0.5
        positions = jitter * self.radius + np.array(self.position)
        velocities = np.ones_like(positions) * np.array(self.velocity)[None]
        velocities += (np.random.rand(emitted, 2) - 0.5) * self.noise
        return positions, velocities

    # ---- counter stream (count on the host, particles on the device) -------------------------------------------------
    def counter_count(self, uniform: float, dt: float) -> int:
        """The tick's emission count before the max_particles clamp: Binomial(flow, dt) (particle_source.py:18) through
        its inverse CDF at stream element 0 of this source."""
        return binomial_inverse_cdf(uniform, int(self.flow), dt)

    def emit_record(self, index: int, count: int) -> tuple:
        """The `sc_source` fields of this source."""
        return (float(self.position[0]), float(self.position[1]), float(self.radius), float(self.velocity[0]),
                float(self.velocity[1]), float(self.noise), int(count), int(index))


def counter_records(sources, seed: int, tick: int, dt: float) -> list[tuple]:
    """The `sc_source` records of the sources that emit at `tick` in the counter mode: each count drawn from element 0
    of the source's counter stream (host arithmetic, no device data), so every caller - one context or every rank of a
    strip-decomposed scene - draws the same ones."""
    from . import _lib
    records = []
    for index, source in enumerate(sources):
        if source.active_ticks <= tick:
            continue
        count = source.counter_count(_lib.source_uniform(seed, tick, index, 0), dt)
        if count:
            records.append(source.emit_record(index, count))
    return records


def build_particle_sources(particle_source_configs) -> list[ParticleSource]:
    return [ParticleSource(**cfg) for cfg in (particle_source_configs or [])]

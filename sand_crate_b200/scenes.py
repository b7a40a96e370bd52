"""Synthetic benchmark scenes (SURVEY.md section 8(d), BASELINE.json `configs[2:]`).

The reference's world is hard-wired to the unit square (crate.py:152), so large particle counts mean a small
particle diameter; `dt` is scaled with it so that `v * dt / d` keeps the ratio of the shipped configs.  All scenes:
closed unit box (the four fixed segments of wave_machine.yaml:35-40), no sources, no motored bodies, the
coefficients of wave_machine.yaml:10-22, square lattice at 0.75 * d spacing (the reference's own bulk rest spacing
is 0.67-0.84 * d) with +-5 % uniform jitter from RandomState(42), zero initial velocity, gravity +y (y = 1 is the
floor).
"""
from __future__ import annotations

import math

import numpy as np

from .load_config import WorldConfig

BASE_COEFFICIENTS = {
    "dt": 0.002, "particle_radius": 0.005, "wall_collision_decay": 0.2, "spring_overlap_balance": 0.5,
    "spring_amplifier": 100, "pressure_amplifier": 30, "ignored_pressure": 0.3, "collider_noise_level": 0.1,
    "viscosity": 8, "max_particles": 0, "surface_smoothing": 100, "target_pressure": -2, "gravity": [0, 9.8],
}
UNIT_BOX = {"fixed": {"name": "edge", "segments": [
    [[0.0, 0.0], [0.0, 1.0]], [[0.0, 0.0], [1.0, 0.0]], [[1.0, 0.0], [1.0, 1.0]], [[0.0, 1.0], [1.0, 1.0]]]}}
LATTICE_FRACTION = 0.75


def _world(n: int, diameter: float, **overrides) -> WorldConfig:
    coeffs = dict(BASE_COEFFICIENTS)
    coeffs["particle_radius"] = diameter / 2
    coeffs["dt"] = 0.002 * (diameter / 0.01)
    coeffs["max_particles"] = int(n)
    coeffs.update(overrides)
    return WorldConfig(rigid_bodies=[UNIT_BOX], particle_sources=[], coefficients=coeffs)


def _lattice_chunks(n: int, x0: float, x1: float, y_floor: float, spacing: float, seed: int, chunk: int):
    """The lattice of `_lattice`, produced `chunk` points at a time as (first index, points): the jitter stream is
    drawn in order, so the concatenation is bit-identical to `_lattice` (RandomState.rand fills row-major)."""
    nx = max(int(math.floor((x1 - x0) / spacing)), 1)
    rs = np.random.RandomState(seed)
    for i0 in range(0, n, chunk):
        idx = np.arange(i0, min(i0 + chunk, n), dtype=np.int64)
        ix = (idx % nx).astype(np.float64)
        iy = (idx // nx).astype(np.float64)
        pts = np.stack((x0 + (ix + 0.5) * spacing, y_floor - (iy + 0.5) * spacing), axis=1)
        pts += (rs.rand(len(idx), 2) - 0.5) * (0.1 * spacing)
        yield i0, pts


def _lattice(n: int, x0: float, x1: float, y_floor: float, spacing: float, seed: int) -> np.ndarray:
    """n points on a square lattice filling [x0, x1] row by row upwards from y_floor, jittered by +-5 %."""
    return np.concatenate([p for _, p in _lattice_chunks(n, x0, x1, y_floor, spacing, seed, max(n, 1))]) if n else np.zeros((0, 2))


def _dam_break_geometry(n: int, width: float, height: float):
    spacing = math.sqrt(width * height / n)
    d = spacing / LATTICE_FRACTION
    return d, (n, d, width, 1.0 - d, spacing)


def _box_fill_geometry(n: int):
    spacing = math.sqrt(1.0 / n)
    d = spacing / LATTICE_FRACTION
    return d, (n, d, 1.0 - d, 1.0 - d, spacing * (1.0 - 2 * d))


def dam_break(n: int, seed: int = 42, width: float = 0.4, height: float = 0.8, **overrides):
    """A column of liquid against the left wall that collapses under gravity.
    1M on one GPU: d ~ 7.5e-4, ~1330 cell rows; 64M (`dam_break_64m`): width 0.5, height 1.0 -> d ~ 1.2e-4."""
    d, lat = _dam_break_geometry(n, width, height)
    pts = _lattice(*lat, seed)
    return _world(n, d, **overrides), pts, np.zeros_like(pts)


def box_fill(n: int, seed: int = 42, **overrides):
    """The whole box filled at rest density (uniform load, the multi-GPU strip-decomposition case)."""
    d, lat = _box_fill_geometry(n)
    pts = _lattice(*lat, seed)
    return _world(n, d, **overrides), pts, np.zeros_like(pts)


def dam_break_wide(n: int, seed: int = 42, **overrides):
    """BASELINE.json configs[4] / SURVEY.md section 8(d): the 64M dam break is a column half the box wide and (almost)
    the whole box high (A ~ 0.5; 0.98 keeps the top lattice row below the lid)."""
    return dam_break(n, seed, width=0.5, height=0.98, **overrides)


# wave_machine.yaml's paddle: a thin rectangle against the right wall, rocking about its top corner (placed in the unit box)
WAVE_PADDLE = {"motored": {"name": "moving_wall", "segments": [
    [[0.0, 0.0], [0.0, -1.0]], [[0.0, 0.0], [-1.0, 0.0]], [[-1.0, 0.0], [-1.0, -1.0]], [[0.0, -1.0], [-1.0, -1.0]]],
    "angular_velocity_func": "lambda t: np.cos(t * 8) * 1.5", "scale": [0.02, 0.9], "rotation": -12,
    "position": [1.0, 1.3]}}


def wave_tank(n: int, seed: int = 42, depth: float = 0.4, flow_fraction: float = 1.0, **overrides):
    """An OPEN scene at size (strip decomposition with sources and moving bodies): wave_machine.yaml's paddle in the unit
    box, a liquid bed of n particles filling the bottom `depth` of the box (lattice as dam_break), and one source pouring
    from the upper left.  Scaling as the other scenes: d from the lattice, dt with d, and so the paddle's motion law
    (physical time) moves it by the same number of rows per tick at any n.  The source runs for 0.5 s of physical time
    at `flow_fraction * n` particles per second (Binomial(flow, dt) per tick); max_particles = n + 0.25 * flow, so the
    clamp binds halfway through - override it to move that point."""
    d, lat = _dam_break_geometry(n, 0.98, depth)
    pts = _lattice(*lat, seed)
    world = _world(n, d, **overrides)
    flow = float(flow_fraction * n)
    dt = world.coefficients["dt"]
    world.rigid_bodies = [UNIT_BOX, WAVE_PADDLE]
    world.particle_sources = [{"radius": 0.05, "position": [0.1, 0.1], "velocity": [2.0, 0.0], "flow": flow,
                               "noise": 0.05, "active_ticks": int(round(0.5 / dt))}]
    if "max_particles" not in overrides:
        world.coefficients["max_particles"] = int(n + 0.25 * flow)
    return world, pts, np.zeros_like(pts)


SCENES = {"dam_break": dam_break, "box_fill": box_fill, "dam_break_wide": dam_break_wide}


def scene_chunks(name: str, n: int, seed: int = 42, chunk: int = 4_000_000, **overrides):
    """(world, iterator factory) of a scene WITHOUT materialising it: `chunks()` yields (first row index, positions)
    `chunk` particles at a time, bit-identical to `SCENES[name](n)[1]`.  A rank of a strip-decomposed run keeps only its
    own rows of each chunk, so a 64M scene never costs 2 GB of host memory per rank."""
    if name == "dam_break":
        d, lat = _dam_break_geometry(n, 0.4, 0.8)
    elif name == "dam_break_wide":
        d, lat = _dam_break_geometry(n, 0.5, 0.98)
    elif name == "box_fill":
        d, lat = _box_fill_geometry(n)
    else:
        raise KeyError(name)
    return _world(n, d, **overrides), (lambda: _lattice_chunks(*lat, seed, chunk))

"""Host-side rigid bodies: wall segments and their per-tick kinematics (reference `src/crate/rigid_body.py:18-91`).

O(#segments) work per tick (6-8 segments in the shipped configs), so it is an *input* of the GPU step, not a
kernel: each tick the placed segments and every body's (center_velocity, angular velocity, position) are pushed
through `sc_set_walls`.  Motion laws are Python lambda source strings in the YAML (`velocity_func`,
`angular_velocity_func`, rigid_body.py:80-83) and are evaluated here on the host, never on the device."""
from __future__ import annotations

import copy
import math
from typing import Callable, Optional

import numpy as np


def rotate_vectors_clockwise_90_deg(v: np.ndarray) -> np.ndarray:
    """(x, y) -> (y, -x), geometry_utils.py:176-179."""
    v = np.asarray(v, dtype=np.float64)
    return np.stack((v[..., 1], -v[..., 0]), axis=-1)


def rotate_degrees(x: float, y: float, angle_deg: float) -> tuple[float, float]:
    """What `pygame.Vector2(x, y).rotate(angle_deg)` computes (rigid_body.py:38-39 uses it for placement):
    angle reduced to [0, 360), exact quarter turns special-cased, else cos/sin of `deg * pi / 180`."""
    eps = 1e-6
    a = math.fmod(angle_deg, 360.0)
    if a < 0:
        a += 360.0
    if math.fmod(a + eps, 90.0) < 2 * eps:
        q = int((a + eps) / 90.0) % 4
        return [(x, y), (-y, x), (-x, -y), (y, -x)][q]
    rad = a * math.pi / 180.0
    s, c = math.sin(rad), math.cos(rad)
    return (c * x - s * y, s * x + c * y)


class RigidBody:
    """A "free" body: constant linear/angular velocity unless something (gravity, crate.py:311-314) changes it."""

    kind = "free"

    def __init__(self, segments, name: str = "", center_velocity=None, angular_clockwise_velocity: float = 0.0,
                 scale=None, position=None, rotation: float = 0.0):
        self.segments = np.array(segments, dtype=np.float64).reshape(-1, 2, 2)
        self.name = name
        self.center_velocity = np.array([0.0, 0.0] if center_velocity is None else center_velocity, dtype=np.float64)
        self.angular_clockwise_velocity = angular_clockwise_velocity
        self.scale = [1.0, 1.0] if scale is None else scale
        self.position = [0.0, 0.0] if position is None else position
        self.rotation = rotation

    def __len__(self) -> int:
        return len(self.segments)

    def place_in_world(self) -> None:
        """scale -> rotate -> translate, rigid_body.py:36-40."""
        seg = self.segments * np.array(self.scale, dtype=np.float64)[None]
        for end in (0, 1):
            seg[:, end, :] = np.array([rotate_degrees(px, py, self.rotation) for px, py in seg[:, end, :]])
        self.segments = seg + np.array(self.position, dtype=np.float64)[None]

    def calc_body_points_velocities(self, body_points: np.ndarray) -> np.ndarray:
        """v(point) = center_velocity + rot90cw(point - position) * omega, rigid_body.py:28-34."""
        rel = body_points - self.position
        return self.center_velocity[None] + rotate_vectors_clockwise_90_deg(rel) * self.angular_clockwise_velocity

    def apply_velocity(self, dt: float) -> None:
        """Linearised motion of both endpoints of every segment (rigid_body.py:42-46); `position` is never
        advanced, exactly like the reference."""
        moved = self.segments.copy()
        for end in (0, 1):
            moved[:, end, :] += self.calc_body_points_velocities(self.segments[:, end, :]) * dt
        self.segments = moved

    def kinematics(self) -> list[float]:
        """(vcx, vcy, omega, posx, posy): the row of `body_kin` the C ABI takes."""
        return [float(self.center_velocity[0]), float(self.center_velocity[1]),
                float(self.angular_clockwise_velocity), float(self.position[0]), float(self.position[1])]


class FixedRigidBody(RigidBody):
    kind = "fixed"

    def apply_velocity(self, dt: float) -> None:  # rigid_body.py:53-55
        return None


class MotoredRigidBody(RigidBody):
    kind = "motored"

    def __init__(self, *args, velocity_func: Optional[Callable] = None,
                 angular_velocity_func: Optional[Callable] = None, time_from_start: float = 0.0, **kwargs):
        super().__init__(*args, **kwargs)
        self.velocity_func = velocity_func or (lambda t: np.array([0.0, 0.0]))
        self.angular_velocity_func = angular_velocity_func or (lambda t: 0)
        self.time_from_start = time_from_start

    def apply_velocity(self, dt: float) -> None:  # rigid_body.py:64-68
        self.time_from_start += dt
        self.center_velocity = np.asarray(self.velocity_func(self.time_from_start), dtype=np.float64)
        self.angular_clockwise_velocity = self.angular_velocity_func(self.time_from_start)
        super().apply_velocity(dt)


def advance_bodies(bodies, dt: float) -> None:
    """apply_bodies_velocity (crate.py:363-365): every body's motion law for one tick."""
    for body in bodies:
        body.apply_velocity(dt)


def apply_gravity_to_free_bodies(bodies, dt: float, gravity) -> None:
    """The rigid-body part of crate.py:311-314 (the particle part runs on the device)."""
    for body in bodies:
        if isinstance(body, (FixedRigidBody, MotoredRigidBody)):
            continue
        body.center_velocity = body.center_velocity + dt * np.asarray(gravity, dtype=np.float64)


def wall_arrays(bodies):
    """The `sc_set_walls` arguments of `bodies`: segments S x 2 x 2, segments per body, kinematics nbodies x 5."""
    seg = np.vstack([b.segments for b in bodies]) if bodies else np.zeros((0, 2, 2))
    return seg, [len(b) for b in bodies], np.array([b.kinematics() for b in bodies], dtype=np.float64).reshape(-1, 5)


BODY_TYPE_TO_CLASS = {"motored": MotoredRigidBody, "fixed": FixedRigidBody, "free": RigidBody}


def _compile_law(src):
    # configs are code in the reference too (`eval` with `np` in scope, rigid_body.py:80-83)
    return eval(src, {"np": np, "math": math}) if isinstance(src, str) else src


def build_rigid_bodies(body_configs) -> list[RigidBody]:
    bodies = []
    for entry in copy.deepcopy(body_configs or []):
        body_type, kwargs = next(iter(entry.items()))
        kwargs = dict(kwargs)
        for key in ("velocity_func", "angular_velocity_func"):
            if key in kwargs:
                kwargs[key] = _compile_law(kwargs[key])
        body = BODY_TYPE_TO_CLASS[body_type](**kwargs)
        body.place_in_world()
        bodies.append(body)
    return bodies

"""The wall path checked against the oracle on adversarial geometry (pytest -m gpu for the device tests).

The wall path is W1 / W1b contacts, the W2 hard-wall fix and the cell key (key_particle, in k_prepass and in the force
kernel's tail), F5's virtual rows, B1 bounce and B2 continuous collision (force_tail, fp64 k_force and mixed
k_force_tile), and the host code that builds its culls (refresh_wall_boxes, sc_api.cu).  Every cull claims "never
changes a result, only skips work": seg_box (touch distance x (1 + 1e-6) + 1e-12 scale), pad_box, and the greedy
rectangles safe_contact, safe_ccd and safe_ccd_f32.  The scenes put particles where those claims are tightest: one ulp
either side of the touch distance, at segment ends and corners, on padded-segment ends, moving parallel to padded
segments, and just inside and outside each rectangle.

Each device case takes ONE step from identical inputs and compares with `oracle.step(..., want_all=True)`: in fp64 bit
for bit, and in mixed precision (counter noise and none) with wall counts, search positions, sorted order and lists
bit-exact (the key pass is fp64 in every precision) and vectors, pressures, velocities and positions within the bars of
tests/test_pair_records_gpu.py.  B1 and B2 are continuous across their decisions (the bounce term is -dot h, and
f -> 1 at the crossing limit), so no particle is exempt.  Every scene also asserts that each search position lies in
an interior cell of the grid: the wall fix moves a particle by up to r per contact, and a clamped cell would merge
rows the reference keeps apart.

The NumPy restatements of refresh_wall_boxes and of point_segment run in the CPU suite, and the library's own culls
(`Context.debug_walls`, sc_debug_walls) are checked against them bit for bit on the device.
"""
import math

import numpy as np
import pytest

from conftest import oracle_counter_run, params_from_coeffs, world_from_freerun
from oracle import oracle as O
from sand_crate_b200 import Crate, WorldConfig, _lib
from sand_crate_b200.scenes import UNIT_BOX
from test_pair_records_gpu import PS_PER_PAIR, REL_TOL_F32, U, check_records, coeffs_for, run_step

D = 0.01                          # particle diameter of the scenes (r = 0.005, the shipped configs' radius)
R = D / 2
TOUCH = R * 1.2                   # crate.py:229
MODES = ["f64", "mixed_counter", "mixed_none"]
BOX = np.array(UNIT_BOX["fixed"]["segments"], np.float64).reshape(-1, 4)


# ---- NumPy restatements (checked on the CPU below) ---------------------------------------------------------------
def point_segment_np(p, seg):
    """point_segment (sc_common.cuh) with the kernel's operation order: (nearest [P, S, 2], distance [P, S])."""
    p = np.asarray(p, np.float64).reshape(-1, 2)
    seg = np.asarray(seg, np.float64).reshape(-1, 4)
    px, py = p[:, 0:1], p[:, 1:2]
    ax, ay, bx, by = (seg[None, :, q] for q in range(4))
    abx, aby = bx - ax, by - ay
    apx, apy = px - ax, py - ay
    with np.errstate(invalid="ignore", divide="ignore"):
        rate = (apx * abx + apy * aby) / (abx * abx + aby * aby)
    t = np.where(rate < 0, 0.0, rate)                          # NaN (a zero-length segment) propagates
    t = np.where(t > 1, 1.0, t)
    cx, cy = abx * t + ax, aby * t + ay
    dx, dy = cx - px, cy - py
    return np.stack((cx, cy), -1), np.sqrt(dx * dx + dy * dy)


def grow_box(ax, ay, bx, by, m):
    """refresh_wall_boxes' `grow`: the bounding box grown by m (1 + 1e-6) + 1e-12 scale."""
    xmin, xmax, ymin, ymax = min(ax, bx), max(ax, bx), min(ay, by), max(ay, by)
    scale = max(1.0, max(max(abs(xmin), abs(xmax)), max(abs(ymin), abs(ymax))))
    e = m * (1.0 + 1e-6) + 1e-12 * scale
    return (xmin - e, xmax + e, ymin - e, ymax + e)


def safe_rect(boxes, lo, hi):
    """refresh_wall_boxes' largest-area-greedy rectangle inside [lo, hi]^2 that meets none of the boxes (empty:
    (1, 0, 1, 0))."""
    rect = [lo, hi, lo, hi]
    meets = lambda b: b[0] < rect[1] and b[1] > rect[0] and b[2] < rect[3] and b[3] > rect[2]
    for _ in range(len(boxes) + 1):
        changed = False
        for b in boxes:
            if not meets(b):
                continue
            w_, h_ = rect[1] - rect[0], rect[3] - rect[2]
            area = [(rect[1] - b[1]) * h_, (b[0] - rect[0]) * h_, w_ * (rect[3] - b[3]), w_ * (b[2] - rect[2])]
            best = int(np.argmax(area))                        # first maximum, like the strict > of the C loop
            rect[best] = [b[1], b[0], b[3], b[2]][best]
            changed = True
        if not changed:
            break
    if not (rect[0] < rect[1] and rect[2] < rect[3]) or any(meets(b) for b in boxes):
        rect = [1.0, 0.0, 1.0, 0.0]
    return np.array(rect)


def contact_bound_np(seg_box):
    """contact_bound (sc_api.cu): the most touch boxes sharing a point, at least 1."""
    b = np.asarray(seg_box).reshape(-1, 4)
    if len(b) == 0:
        return 1
    x, y = b[:, 0][:, None, None], b[:, 2][None, :, None]
    inside = (x >= b[:, 0]) & (x <= b[:, 1]) & (y >= b[:, 2]) & (y <= b[:, 3])
    return max(1, int(inside.sum(-1).max()))


def wall_culls(seg, r):
    """refresh_wall_boxes (sc_api.cu) for the walls `seg` and radius r."""
    seg = np.asarray(seg, np.float64).reshape(-1, 4)
    pad = _lib.pad_segments(seg, r).reshape(-1, 4)
    seg_box = np.array([grow_box(*s, r * 1.2) for s in seg]).reshape(-1, 4)
    pad_box = np.array([grow_box(*s, 0.0) for s in pad]).reshape(-1, 4)
    contact = safe_rect(seg_box, -r, 1 + r)
    ccd = safe_rect(pad_box, -r, 1 + r)
    if ccd[0] < ccd[1]:
        f32 = np.array([ccd[0] + 1e-6, ccd[1] - 1e-6, ccd[2] + 1e-6, ccd[3] - 1e-6], np.float32)
    else:
        f32 = np.array([1, 0, 1, 0], np.float32)
    return {"seg_box": seg_box, "pad_box": pad_box, "safe_contact": contact, "safe_ccd": ccd,
            "safe_ccd_f32": f32.astype(np.float64), "pad": pad, "contacts": contact_bound_np(seg_box)}


def touch_flip(seg, a, u, touch=TOUCH):
    """From a point `a` within the touch distance of the segment, along the direction u: the last fp64 point whose
    point_segment distance is <= touch, and the next one, which is not - one ulp apart in the coordinate whose ulp moves
    the distance most (outward normal component x ulp).  None when the ray never leaves the touch zone."""
    dist = lambda x, y: point_segment_np([[x, y]], seg)[1][0, 0]
    lo, hi = 0.0, 4 * touch
    if not dist(a[0] + hi * u[0], a[1] + hi * u[1]) > touch:
        return None
    for _ in range(80):                                        # the zone along a ray is an interval containing 0
        mid = 0.5 * (lo + hi)
        if dist(a[0] + mid * u[0], a[1] + mid * u[1]) <= touch:
            lo = mid
        else:
            hi = mid
    x, y = a[0] + lo * u[0], a[1] + lo * u[1]
    c = point_segment_np([[x, y]], seg)[0][0, 0]
    big_x = abs(x - c[0]) * np.spacing(abs(x)) >= abs(y - c[1]) * np.spacing(abs(y))
    sgn = np.sign(x - c[0] if big_x else y - c[1])
    step = lambda x, y, s: (np.nextafter(x, s * np.inf), y) if big_x else (x, np.nextafter(y, s * np.inf))
    for _ in range(256):
        if dist(x, y) <= touch:
            nx_, ny_ = step(x, y, sgn)
            if not dist(nx_, ny_) <= touch:
                return (x, y), (nx_, ny_)
            x, y = nx_, ny_
        else:
            x, y = step(x, y, -sgn)
    raise AssertionError("no fp64 touch flip found")


def single_body(seg):
    seg = np.asarray(seg, np.float64).reshape(-1, 4)
    return seg, np.array([len(seg)], np.int32), np.zeros((1, 5))


# ---- scenes (deterministic from their seeds) ---------------------------------------------------------------------
def irregular_walls(seed=1):
    """Segments at many angles, lengths from 0.3 d to 0.5, some ending inside the box, one crossing its edge."""
    rs = np.random.RandomState(seed)
    lengths = [0.3 * D, 0.7 * D, 1.3 * D, 3 * D, 0.05, 0.12, 0.25, 0.5]
    seg = []
    for k, L in enumerate(lengths):
        a = np.deg2rad(7 + 23 * k + rs.uniform(-3, 3))
        cx, cy = 0.15 + 0.7 * rs.rand(), 0.15 + 0.7 * rs.rand()
        seg.append([cx - 0.5 * L * np.cos(a), cy - 0.5 * L * np.sin(a), cx + 0.5 * L * np.cos(a), cy + 0.5 * L * np.sin(a)])
    seg.append([0.9, 0.95, 1.1, 1.02])                          # partly outside the box
    return np.concatenate((BOX, np.array(seg)))


def scene_touch_edge(side, seed=2):
    """Particles one ulp inside (side 0) or outside (side 1) the touch distance: perpendicular from interior points of
    every segment, and from both ends of every segment along +-x, +-y and 12 other directions.  Particles closer than
    0.15 d to one already placed are dropped (no near-duplicates without noise).  Returns (pos, vel, place index)."""
    rs = np.random.RandomState(seed)
    seg = irregular_walls()
    pts, place = [], []
    dirs = [(1, 0), (-1, 0), (0, 1), (0, -1)] + [(np.cos(a), np.sin(a)) for a in np.deg2rad(np.arange(12) * 30 + 13)]
    k = 0
    for s in seg:
        ab = np.array([s[2] - s[0], s[3] - s[1]])
        n = np.array([-ab[1], ab[0]]) / np.hypot(*ab)
        starts = [((s[0] + f * ab[0], s[1] + f * ab[1]), tuple(sg * n)) for f in (0.2, 0.5, 0.8) for sg in (1, -1)]
        starts += [((s[q], s[q + 1]), u) for q in (0, 2) for u in dirs]
        for a, u in starts:
            flip = touch_flip(s, a, u)
            k += 1
            if flip is None:
                continue
            pts.append(flip[side])
            place.append(k)
    pts, place = np.array(pts), np.array(place)
    keep = (pts >= -R).all(1) & (pts <= 1 + R).all(1)
    pts, place = pts[keep], place[keep]
    sel = []
    for i, p in enumerate(pts):
        if all(np.hypot(*(p - pts[j])) > 0.15 * D for j in sel):
            sel.append(i)
    pts, place = pts[sel], place[sel]
    return pts, rs.randn(len(pts), 2), place, seg


def fan(hub, angles_deg, length):
    return np.array([[hub[0], hub[1], hub[0] + length * np.cos(np.deg2rad(a)), hub[1] + length * np.sin(np.deg2rad(a))]
                     for a in angles_deg])


def near_points(seg, rs, m, reach=1.4 * TOUCH):
    """m points within `reach` of a random point of the walls, with velocities pointing into them."""
    pts, vel = [], []
    for _ in range(m):
        s = seg[rs.randint(len(seg))]
        f = rs.rand()
        c = np.array([s[0] + f * (s[2] - s[0]), s[1] + f * (s[3] - s[1])])
        a = rs.uniform(0, 2 * np.pi)
        off = reach * np.sqrt(rs.rand()) * np.array([np.cos(a), np.sin(a)])
        pts.append(c + off)
        vel.append(-off / np.hypot(*off) * rs.uniform(0.5, 3) + 0.3 * rs.randn(2))
    return np.array(pts), np.array(vel)


def spaced(pos, vel, min_dist=0.15 * D):
    keep = (pos >= -R).all(1) & (pos <= 1 + R).all(1)
    pos, vel = pos[keep], vel[keep]
    sel = []
    for i, p in enumerate(pos):
        if all(np.hypot(*(p - pos[j])) > min_dist for j in sel):
            sel.append(i)
    return pos[sel], vel[sel]


def scene_multi(kind, seed=3):
    """Multiple contacts.  corners: segment pairs meeting at 10 - 170 degrees, and a segment three times over.  fans:
    3 - 8 segments sharing an end, two of them at the box's edge so that the fix pushes particles out of the box.
    bodies: 4 bodies with distinct kinematics whose segments overlap around common points (the W1b quirk: the body
    order decides which kinematics fill each contact row).  Returns (pos, vel, walls)."""
    rs = np.random.RandomState(seed)
    if kind == "corners":
        seg = [BOX]
        for k, ang in enumerate((10, 30, 60, 90, 120, 150, 170)):
            hub = (0.12 + 0.12 * k, 0.3 + 0.05 * (k % 3))
            a0 = rs.uniform(0, 360)
            seg.append(fan(hub, [a0, a0 + ang], 0.04 + 0.01 * k))
        seg.append(np.repeat([[0.3, 0.75, 0.42, 0.8]], 3, 0))  # duplicated segment
        seg.append(np.array([[0.6, 0.7, 0.6, 0.7]]))          # zero length
        seg = np.concatenate(seg)
        walls = single_body(seg)
    elif kind == "fans":
        seg = np.concatenate((BOX, fan((0.3, 0.4), np.linspace(0, 240, 3), 0.05), fan((0.6, 0.5), np.linspace(10, 350, 8), 0.04),
                              fan((0.5, 1 + R / 2), np.linspace(200, 340, 7), 0.05),
                              fan((-R / 2, 0.7), np.linspace(-60, 60, 6), 0.05)))
        walls = single_body(seg)
    else:
        hubs = [(0.3, 0.3), (0.6, 0.65), (0.75, 0.25)]
        bodies = []
        for b in range(4):
            segs = [fan(h, [20 + 47 * b + 90 * q, 200 + 31 * b + 90 * q], 0.06) for q, h in enumerate(hubs)
                    if (b + q) % 4 != 3]
            bodies.append(np.concatenate(segs))
        bodies[0] = np.concatenate((BOX, bodies[0]))
        kin = np.array([[0.3, -0.2, 1.5, 0.4, 0.4], [-0.5, 0.1, -2.0, 0.6, 0.6], [0.05, 0.6, 0.7, 0.2, 0.7],
                        [-0.2, -0.4, 3.0, 0.8, 0.2]])
        seg = np.concatenate(bodies)
        walls = (seg, np.array([len(b) for b in bodies], np.int32), kin)
    pos, vel = near_points(seg[4:] if kind != "bodies" else np.concatenate(bodies)[4:], rs, 900)
    pos, vel = spaced(pos, vel)
    return pos, vel, walls


def scene_crossings(dt, gy, seed=4):
    """Isolated particles (K = 0; V = 0 where they start clear of the touch distance, so that the velocity B2 sees is
    v0 + dt g exactly) whose movement ends a few ulps before and after a padded segment, passes through padded-segment
    ends, runs parallel to a padded segment (on it and beside it: in contact), crosses two padded segments, or is
    zero.  Returns (pos, vel, walls)."""
    rs = np.random.RandomState(seed)
    seg = np.concatenate((BOX, [[0.2, 0.5, 0.45, 0.5], [0.2, 0.5 + 0.3 * D, 0.45, 0.5 + 0.3 * D],
                                [0.6, 0.2, 0.85, 0.45], [0.55, 0.7, 0.7, 0.9]]))
    pad = _lib.pad_segments(seg, R).reshape(-1, 4)
    pts, ends = [], []
    for q in range(4, len(pad)):
        c, e = pad[q, :2], pad[q, 2:]
        cd = e - c
        n = np.array([cd[1], -cd[0]]) / np.hypot(*cd)          # rot90cw(d - c): a crossing moves against it
        for j, f in enumerate(np.linspace(0.05, 0.95, 14)):
            hit = c + f * cd
            start = hit + n * (2.5 * R + 0.4 * R * rs.rand()) + 0.05 * R * rs.randn(2)
            end = hit + (j % 7 - 3) * 2.0 ** -52 * n           # a few ulps before / after the padded line
            pts.append(start); ends.append(end)
        for corner in (c, e):                                # through the padded segment's ends
            for ang in (30, 100, 160):
                u = np.array([np.cos(np.deg2rad(ang)), np.sin(np.deg2rad(ang))])
                pts.append(corner - 1.5 * R * u); ends.append(corner + 0.5 * R * u)
        u = cd / np.hypot(*cd)                                # parallel: on the padded line and beside it
        for off in (0.0, 1e-3 * R, -1e-3 * R):
            st = c + 0.3 * cd + off * n
            pts.append(st); ends.append(st + 0.8 * R * u)
    for x in np.linspace(0.22, 0.43, 6):                     # down through both upper padded lines at y = 0.5 (+ 0.3 d)
        pts.append(np.array([x, 0.5 + 0.3 * D + 2.6 * R])); ends.append(np.array([x + 0.1 * R, 0.5 - 2.5 * R]))
    for x in np.linspace(0.1, 0.9, 5):                       # zero movement
        pts.append(np.array([x, 0.08])); ends.append(np.array([x, 0.08]))
    pos, end = np.array(pts), np.array(ends)
    v = (end - pos) / dt
    vel = v - np.array([0.0, dt * gy])                        # v0: the velocity after gravity is v
    keep = (pos >= -R).all(1) & (pos <= 1 + R).all(1)        # (the step removes the others first)
    for i in range(len(pos)):                                # isolated: K = 0
        if keep[i]:
            close = np.hypot(*(pos - pos[i]).T) <= 1.01 * D
            close[:i + 1] = False
            keep &= ~close
    return pos[keep], vel[keep], single_body(seg)


def rect_walls():
    """A wall set whose greedy rectangles are small and asymmetric."""
    return np.concatenate((BOX, [[0.3, 0.2, 0.3, 0.75], [0.5, 0.82, 0.9, 0.82], [0.7, 0.1, 0.78, 0.3],
                                 [0.45, 0.3, 0.46, 0.3]]))


def scene_rect_edges(culls, dt, gy, seed=5):
    """Particles a few ulps inside and outside every side of safe_contact, and movements whose box ends a few ulps
    inside and outside every side of safe_ccd and of safe_ccd_f32 (in fp32 ulps for the latter)."""
    rs = np.random.RandomState(seed)
    pts, vel = [], []
    sc, ccd, f32 = culls["safe_contact"], culls["safe_ccd"], culls["safe_ccd_f32"]
    for side in range(4):
        axis = side // 2
        lo, hi = (sc[2], sc[3]) if axis == 0 else (sc[0], sc[1])
        for q, k in enumerate(range(-3, 4)):
            p = [0.0, 0.0]
            v = sc[side]
            for _ in range(abs(k)):
                v = np.nextafter(v, np.inf if k > 0 else -np.inf)
            p[axis], p[1 - axis] = v, lo + (hi - lo) * (0.1 + 0.11 * q)
            pts.append(p); vel.append(0.2 * rs.randn(2))
        for rect, f in ((ccd, np.float64), (f32, np.float32)):
            lo, hi = (rect[2], rect[3]) if axis == 0 else (rect[0], rect[1])
            for q, k in enumerate(range(-3, 4)):
                edge = f(rect[side])
                for _ in range(abs(k)):
                    edge = np.nextafter(edge, f(np.inf if k > 0 else -np.inf))
                along = lo + (hi - lo) * (0.15 + 0.1 * q + (0.05 if f is np.float32 else 0))
                speed = 0.3 * R / dt * (-1 if side in (0, 2) else 1)
                g = dt * gy if axis == 1 else 0.0
                p, v0 = [along, along], [0.0, 0.0]
                p[axis], v0[axis] = float(edge) - speed * dt, speed - g
                pts.append(p); vel.append(v0)
    pos, vel = np.array(pts), np.array(vel)
    keep = (pos >= -R).all(1) & (pos <= 1 + R).all(1)
    for i in range(len(pos)):
        if keep[i]:
            close = np.hypot(*(pos - pos[i]).T) <= 1.01 * D
            close[:i + 1] = False
            keep &= ~close
    return pos[keep], vel[keep]


def scene_limits(seed=6):
    """S = SC_MAX_SEGMENTS over SC_MAX_BODIES bodies with distinct kinematics; particles touching only the last
    segment; one particle exactly on a segment's end (vc = 0: its position becomes NaN in the device and the
    reference alike)."""
    rs = np.random.RandomState(seed)
    S, B = _lib.MAX_SEGMENTS, _lib.MAX_BODIES
    seg = [BOX]
    for k in range(S - 4):
        hub = (0.1 + 0.8 * rs.rand(), 0.1 + 0.8 * rs.rand()) if k % 3 else (0.5, 0.5)
        a = rs.uniform(0, 360)
        seg.append(fan(hub, [a], 0.02 + 0.1 * rs.rand()))
    seg = np.concatenate(seg)
    seg[-1] = [0.05, 0.93, 0.2, 0.93]                         # the last segment, alone in its corner
    body_len = np.full(B, S // B, np.int32)
    kin = np.stack((rs.uniform(-1, 1, B), rs.uniform(-1, 1, B), rs.uniform(-3, 3, B), rs.rand(B), rs.rand(B)), 1)
    pos, vel = near_points(seg[4:], rs, 700)
    last = np.stack((np.linspace(0.07, 0.18, 6), 0.93 + np.array([1, -1, 1, -1, 1, -1]) * 0.9 * TOUCH), 1)
    pos, vel = np.concatenate((last, pos)), np.concatenate((np.tile([[0.0, -1.0]], (6, 1)) * [[1, 1]] * np.sign(
        last[:, 1:2] - 0.93), vel))
    pos, vel = spaced(pos, vel)
    on = np.array([[seg[10, 0], seg[10, 1]]])                 # exactly on a segment's end
    pos = np.concatenate((pos[np.hypot(*(pos - on).T) > 1.5 * D], on))
    vel = np.concatenate((vel[:len(pos) - 1], [[0.5, 0.5]]))
    return pos, vel, (seg, body_len, kin)


def scene_grid_fans(seed=7):
    """Four 8-segment fans whose hubs sit r / 2 outside the middle of each side of the box, fanning into it, with
    particles just outside each hub: the fix sums up to eight pushes of < r and moves them past the rows and columns a
    one-contact grid holds, on the low and the high side, in x and in y.  Plus box particles beside each hub."""
    rs = np.random.RandomState(seed)
    hubs = [((0.5, 1 + R / 2), 200, (0, 1)), ((0.5, -R / 2), 20, (0, -1)), ((1 + R / 2, 0.5), 110, (1, 0)),
            ((-R / 2, 0.5), -70, (-1, 0))]
    seg, pts = [], []
    for hub, a0, out in hubs:
        seg.append(fan(hub, a0 + 140 * np.arange(8) / 7, 0.05))
        along = np.array([out[1], out[0]], float)
        for k in range(8):                                    # just outside the hub, spread along the side
            pts.append(np.array(hub) + np.array(out) * R * (0.01 + 0.1 * (k % 4)) + along * R * (k - 3.5) * 0.003)
        for o, a in ((0.005, 0.0), (0.4, 0.3), (0.25, -0.2), (0.45, 0.5)):   # rows past the old grid, out of x order
            pts.append(np.array(hub) + np.array(out) * R * o + along * R * a)
        for k in range(10):                                   # inside the box, next to the fan
            pts.append(np.array(hub) - np.array(out) * R * (1.5 + 0.4 * rs.rand()) + along * D * (k - 4.5) * 0.9)
    pos = np.array(pts)
    return pos, 0.3 * rs.randn(*pos.shape), single_body(np.concatenate(seg))


# ---- one step on the device and on the oracle, and the checks ----------------------------------------------------
def check_search(ctx, ref, n):
    """Wall counts, search positions, rows and sorted order bit-exact; every search position in an interior cell."""
    assert np.array_equal(ctx.get_wall_counts(n), ref["wall_count"]), "wall counts"
    ps = ref["pos_search"]
    gps, grows, gorder = ctx.get_search(n)
    assert np.array_equal(gps, ps, equal_nan=True), "search positions (hard-wall fix)"
    live = np.isfinite(ps).all(1)          # a NaN row is filed under row 0 by the device; nothing depends on where
    rows_o, order_o, _, _ = O.detect_particle_collisions(ps, 2 * R)
    assert np.array_equal(gorder[live[gorder]], order_o[live[order_o]]), "sorted order"
    assert np.array_equal(grows[live[gorder]], rows_o[live[order_o]]), "sorted rows"
    row_min, col_min, nrows, ncols = ctx.grid()
    rows = np.floor(ps[live, 1] / (2 * R)).astype(np.int64)
    cols = np.floor(ps[live, 0] / (2 * R)).astype(np.int64)
    assert rows.min() >= row_min + 1 and rows.max() <= row_min + nrows - 2, ("rows outside the grid's interior",
                                                                              rows.min(), rows.max(), row_min, nrows)
    assert cols.min() >= col_min + 1 and cols.max() <= col_min + ncols - 2, ("columns outside the grid's interior",
                                                                              cols.min(), cols.max(), col_min, ncols)


def check_state(ctx, ref, cv, mode, vin):
    """check_physics of tests/test_pair_records_gpu.py, with NaN positions compared as equal and left out of the bars."""
    n = len(vin)
    pos, vel, prs = ctx.get_state()
    tens = ctx.get_tension(n)
    assert np.array_equal(np.isnan(pos), np.isnan(ref["pos_out"])) and np.array_equal(np.isnan(vel), np.isnan(ref["vel_out"]))
    if mode == "f64":
        for a, b in ((pos, "pos_out"), (vel, "vel_out"), (prs, "pressure"), (tens, "tension_vec")):
            assert np.array_equal(a, ref[b], equal_nan=True), b
        return
    k = np.isfinite(ref["pos_out"]).all(1) & np.isfinite(ref["vel_out"]).all(1)
    K = ref["nbr_count"]
    bar = PS_PER_PAIR * K + 2 * U * (np.abs(ref["pressure"]) + abs(cv[4]))
    assert (np.abs(prs - ref["pressure"]) <= bar).all(), float((np.abs(prs - ref["pressure"]) / bar).max())
    tbar = PS_PER_PAIR * K + 2 * U * np.abs(ref["tension_vec"]).max(1)
    assert (np.abs(tens - ref["tension_vec"]).max(1) <= tbar).all()
    d = 2 * cv[1]
    v_floor = 0.01 * d / cv[0]
    vr, v, p, pr = ref["vel_out"][k], vel[k], pos[k], ref["pos_out"][k]
    assert np.abs(v - vr).max() <= REL_TOL_F32 * max(np.abs(vr).max(), v_floor), float(np.abs(v - vr).max())
    assert np.abs(p - pr).max() <= REL_TOL_F32 * d, float(np.abs(p - pr).max())
    dv_ref = vr - vin[k]
    if np.abs(dv_ref).max() > 0:
        assert np.abs((v - vin[k]) - dv_ref).max() <= REL_TOL_F32 * np.abs(dv_ref).max()


def check_culls(ctx, walls):
    """The library's culls equal the restatement's bit for bit."""
    got, want = ctx.debug_walls(), wall_culls(walls[0], R)
    for key in ("seg_box", "pad_box", "safe_contact", "safe_ccd", "safe_ccd_f32"):
        assert np.array_equal(got[key], want[key], equal_nan=True), key   # a zero-length segment pads to NaN
    assert got["contacts"] >= want["contacts"]
    return got


def run_walls(pos, vel, mode, walls, seed=17):
    assert ((pos >= -R) & (pos <= 1 + R)).all(), "the step would remove a particle the oracle keeps"
    ctx, ref, cv, vin, tkey, _ = run_step(pos, vel, mode, D, walls, seed)
    n = len(pos)
    check_search(ctx, ref, n)
    check_records(ctx, ref, cv, mode, tkey)
    check_state(ctx, ref, cv, mode, vin)
    check_culls(ctx, walls)
    return ctx, ref, cv, vin


def bodies_touched(pos, walls):
    seg, body_len, _ = walls
    body = np.repeat(np.arange(len(body_len)), body_len)
    touch = point_segment_np(pos, seg)[1] <= TOUCH
    return np.array([len(set(body[t].tolist())) for t in touch])


# ---- CPU: the restatements ---------------------------------------------------------------------------------------
def random_walls(rs):
    """Rotated, very short, zero-length, duplicated and partly outside segments."""
    seg = []
    for k in range(rs.randint(4, _lib.MAX_SEGMENTS - 4)):
        c = rs.uniform(-0.1, 1.1, 2)
        L = [0.0, 1e-9, 0.3 * D, 0.02, 0.3, 0.8][rs.randint(6)]
        a = rs.uniform(0, 2 * np.pi)
        seg.append([c[0], c[1], c[0] + L * np.cos(a), c[1] + L * np.sin(a)])
        if rs.rand() < 0.2:
            seg.append(seg[-1])
    return np.array(seg[:_lib.MAX_SEGMENTS - 4])


def test_point_segment_restatement_matches_oracle():
    rs = np.random.RandomState(11)
    seg = np.concatenate((random_walls(rs), irregular_walls()))
    p = np.concatenate((rs.uniform(-0.1, 1.1, (300, 2)), seg[:, :2], seg[:, 2:], 0.5 * (seg[:, :2] + seg[:, 2:])))
    near, dist = point_segment_np(p, seg)
    o_near, o_dist = O.points_to_segments_distance(p, seg)
    assert np.array_equal(dist, o_dist, equal_nan=True) and np.array_equal(near, o_near, equal_nan=True)


def test_touch_flip_straddles_the_touch_distance():
    seg = irregular_walls()
    n = 0
    for s in seg:
        for u in ((1.0, 0.0), (0.0, -1.0), (np.cos(0.7), np.sin(0.7))):
            flip = touch_flip(s, (s[0], s[1]), u)
            if flip is None:
                continue
            (ix, iy), (ox, oy) = flip
            d_in, d_out = point_segment_np([[ix, iy], [ox, oy]], s)[1][:, 0]
            assert d_in <= TOUCH < d_out
            assert (ix == ox) != (iy == oy) and max(abs(ix - ox), abs(iy - oy)) <= np.spacing(max(abs(ix), abs(iy)))
            n += 1
    assert n >= 2 * len(seg)


def test_wall_culls_on_random_wall_sets():
    """No point within the touch distance of a segment lies outside its seg_box or strictly inside safe_contact; no
    point of a padded segment lies strictly inside safe_ccd; safe_ccd_f32 lies inside safe_ccd; the contact bound
    holds at every sampled point."""
    rs = np.random.RandomState(12)
    checked = 0
    for trial in range(40):
        seg = np.concatenate((BOX, random_walls(rs)))
        c = wall_culls(seg, R)
        pts = []
        for s in seg:                                         # the touch zone: flips, and points inside it
            for u in [(np.cos(a), np.sin(a)) for a in rs.uniform(0, 2 * np.pi, 6)]:
                flip = touch_flip(s, (s[0], s[1]), u)
                if flip is not None:
                    pts.append(flip[0])
            f = rs.rand(8)[:, None]
            a = rs.uniform(0, 2 * np.pi, 8)
            pts += list(s[:2] + f * (s[2:] - s[:2]) + TOUCH * rs.rand(8)[:, None] * np.stack((np.cos(a), np.sin(a)), 1))
        pts = np.array(pts)
        dist = point_segment_np(pts, seg)[1]
        hit = dist <= TOUCH
        b = c["seg_box"]
        inside_box = ((pts[:, None, 0] >= b[:, 0]) & (pts[:, None, 0] <= b[:, 1]) &
                      (pts[:, None, 1] >= b[:, 2]) & (pts[:, None, 1] <= b[:, 3]))
        assert not (hit & ~inside_box).any(), "a contact outside its segment's box"
        assert (hit.sum(1) <= c["contacts"]).all(), "more contacts than the grid has room for"
        sc = c["safe_contact"]
        strictly = ((pts[:, 0] > sc[0]) & (pts[:, 0] < sc[1]) & (pts[:, 1] > sc[2]) & (pts[:, 1] < sc[3]))
        assert not (strictly & hit.any(1)).any(), "a contact strictly inside safe_contact"
        pad = c["pad"]
        f = np.linspace(0, 1, 33)[:, None, None]
        on_pad = (pad[None, :, :2] + f * (pad[None, :, 2:] - pad[None, :, :2])).reshape(-1, 2)
        ccd = c["safe_ccd"]
        assert not ((on_pad[:, 0] > ccd[0]) & (on_pad[:, 0] < ccd[1]) & (on_pad[:, 1] > ccd[2]) &
                    (on_pad[:, 1] < ccd[3])).any(), "a padded segment strictly inside safe_ccd"
        pb = c["pad_box"]
        assert not ((pb[:, 0] < ccd[1]) & (pb[:, 1] > ccd[0]) & (pb[:, 2] < ccd[3]) & (pb[:, 3] > ccd[2])).any()
        f32 = c["safe_ccd_f32"]
        if ccd[0] < ccd[1]:
            assert f32[0] >= ccd[0] and f32[1] <= ccd[1] and f32[2] >= ccd[2] and f32[3] <= ccd[3]
        checked += int(hit.sum())
    assert checked > 5000


def test_contact_bound_restatement():
    assert contact_bound_np(wall_culls(BOX, R)["seg_box"]) == 2              # the box's corners
    seg, _, _ = scene_grid_fans()[2]
    assert contact_bound_np(wall_culls(seg, R)["seg_box"]) == 8
    dup = np.repeat([[0.2, 0.2, 0.4, 0.3]], 5, 0)
    assert contact_bound_np(wall_culls(dup, R)["seg_box"]) == 5
    assert contact_bound_np(np.zeros((0, 4))) == 1


def test_grid_scene_exceeds_a_one_contact_grid():
    """The oracle moves particles of the fan scene past the rows and columns a one-contact grid holds (interior rows
    floor(-2r / d) - 1 .. floor((1 + 2r) / d) + 1), on both sides, in x and y, so that clamping them would change the
    sorted order."""
    pos, vel, walls = scene_grid_fans()
    ref = O.step(coeffs_for(D), pos, vel, *walls, noise_mode=0, want_all=True)
    lo, hi = math.floor(-2 * R / D) - 1, math.floor((1 + 2 * R) / D) + 1
    rc = np.floor(ref["pos_search"] / D).astype(np.int64)
    assert (rc[:, 1] > hi).sum() >= 3 and (rc[:, 1] < lo).sum() >= 3
    assert (rc[:, 0] > hi).sum() >= 3 and (rc[:, 0] < lo).sum() >= 3
    assert ref["wall_count"].max() >= 7
    # a one-contact grid clamps those rows into its last interior one: its cell order (row, column, x) would differ
    # from the reference's (row, x)
    cr, cc = np.clip(rc[:, 1], lo, hi), np.clip(rc[:, 0], lo, hi)
    clamped = np.lexsort((np.arange(len(pos)), ref["pos_search"][:, 0], cc, cr))
    order = O.detect_particle_collisions(ref["pos_search"], D)[1]
    assert (clamped != order).sum() >= 10


def test_scenes_exercise_their_targets():
    """Each scene does what it is for, on the oracle's own outputs."""
    cv = coeffs_for(D)
    dt, gy = cv[0], cv[10]
    # touch edge: V differs between the two sides of a flip in many places
    a_pos, a_vel, a_place, seg = scene_touch_edge(0)
    b_pos, b_vel, b_place, _ = scene_touch_edge(1)
    wa = O.step(cv, a_pos, a_vel, *single_body(seg), want_all=True)["wall_count"]
    wb = O.step(cv, b_pos, b_vel, *single_body(seg), want_all=True)["wall_count"]
    common, ia, ib = np.intersect1d(a_place, b_place, return_indices=True)
    assert (wa[ia] > wb[ib]).sum() >= 150, (wa[ia] > wb[ib]).sum()
    # multiple contacts
    for kind in ("corners", "fans", "bodies"):
        pos, vel, walls = scene_multi(kind)
        ref = O.step(cv, pos, vel, *walls, want_all=True)
        assert (ref["wall_count"] >= 2).sum() >= 30, kind
        if kind != "corners":
            assert (ref["wall_count"] >= 5).sum() >= 5, (kind, np.bincount(ref["wall_count"]))
        if kind == "fans":
            out = (ref["pos_search"] < -R) | (ref["pos_search"] > 1 + R)
            assert out.any(1).sum() >= 3
        if kind == "bodies":
            assert (bodies_touched(pos, walls) >= 2).sum() >= 20
            assert (bodies_touched(pos, walls) >= 3).sum() >= 3
    # crossings
    pos, vel, walls = scene_crossings(dt, gy)
    ref = O.step(cv, pos, vel, *walls, want_all=True)
    assert (ref["nbr_count"] == 0).mean() > 0.9 and (ref["wall_count"] == 0).mean() > 0.7
    f = ref["ccd_factor"]
    assert (f < 1).sum() >= 40 and (f == 1).sum() >= 40
    pad = _lib.pad_segments(walls[0], R).reshape(-1, 4)
    with np.errstate(invalid="ignore", divide="ignore"):
        mv = ref["vel_out"] / f[:, None] * dt                 # the movement B2 tested
    cd = pad[None, :, 2:] - pad[None, :, :2]
    denom = cd[..., 0] * mv[:, None, 1] - cd[..., 1] * mv[:, None, 0]
    assert ((denom == 0) & (np.abs(mv).sum(1) > 0)[:, None]).sum() >= 5, "parallel movements"
    # rectangle edges
    culls = wall_culls(rect_walls(), R)
    sc, ccd = culls["safe_contact"], culls["safe_ccd"]
    assert sc[1] - sc[0] < 0.7 and sc[3] - sc[2] < 0.51 and ccd[3] - ccd[2] < 0.51 and sc[0] != 1 - sc[1]
    pos, vel = scene_rect_edges(culls, dt, gy)
    assert len(pos) >= 60
    # limits
    pos, vel, walls = scene_limits()
    assert len(walls[0]) == _lib.MAX_SEGMENTS and len(walls[1]) == _lib.MAX_BODIES
    ref = O.step(cv, pos, vel, *walls, want_all=True)
    assert np.isnan(ref["pos_search"][-1]).all() and np.isfinite(ref["pos_search"][:-1]).all()
    only_last = (point_segment_np(pos, walls[0])[1] <= TOUCH)
    assert (only_last[:, -1] & (only_last.sum(1) == 1)).sum() >= 3
    assert (bodies_touched(pos, walls) >= 2).sum() >= 10


# ---- GPU: the wall path against the oracle -----------------------------------------------------------------------
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("mode", MODES)
def test_touch_edge(mode, side):
    pos, vel, _, seg = scene_touch_edge(side)
    run_walls(pos, vel, mode, single_body(seg))


@gpu
@pytest.mark.parametrize("kind", ["corners", "fans", "bodies"])
@pytest.mark.parametrize("mode", MODES)
def test_multiple_contacts(mode, kind):
    pos, vel, walls = scene_multi(kind)
    run_walls(pos, vel, mode, walls)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_crossings(mode):
    cv = coeffs_for(D)
    pos, vel, walls = scene_crossings(cv[0], cv[10])
    run_walls(pos, vel, mode, walls)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_rectangle_edges(mode):
    cv = coeffs_for(D)
    walls = single_body(rect_walls())
    culls = wall_culls(walls[0], R)
    pos, vel = scene_rect_edges(culls, cv[0], cv[10])
    pos, vel = np.concatenate((pos, scene_multi("corners")[0][:200])), np.concatenate((vel, np.zeros((200, 2))))
    run_walls(pos, vel, mode, walls)
    if mode == "f64":
        return
    # the bulk fast path (default K5) against the general path (the monitor variant), tick after tick
    ctxs = []
    for monitor in (False, True):
        ctx = _lib.Context(len(pos), _lib.PRECISION_MIXED)
        ctx.set_params(**params_from_coeffs(cv))
        ctx.set_walls(*walls)
        ctx.set_noise(_lib.NOISE_COUNTER if mode == "mixed_counter" else _lib.NOISE_NONE, 21)
        ctx.set_monitor(monitor)
        ctx.set_state(pos, vel)
        ctxs.append(ctx)
    for tick in range(10):
        for ctx in ctxs:
            ctx.set_tick(tick)
            ctx.step()
        a, b = ctxs[0].get_state(want_pressure=False), ctxs[1].get_state(want_pressure=False)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), tick


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_limits(mode):
    pos, vel, walls = scene_limits()
    ctx, ref, _, _ = run_walls(pos, vel, mode, walls)
    assert ctx.debug_walls()["seg_box"].shape == (_lib.MAX_SEGMENTS, 4)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_grid_holds_the_multi_contact_wall_fix(mode):
    pos, vel, walls = scene_grid_fans()
    ctx, ref, _, _ = run_walls(pos, vel, mode, walls)
    assert ctx.debug_walls()["contacts"] >= 8


@gpu
def test_moving_star_body_matches_oracle_over_ticks():
    """A motored star body (six spokes, turning and swaying) in the recorded wave_machine world, pushed with
    set_walls every tick by the Crate; fp64 and counter noise, bit-identical to the oracle loop tick by tick."""
    world, _ = world_from_freerun("wave_machine")
    spokes = [[[0.0, 0.0], [math.cos(a), math.sin(a)]] for a in np.deg2rad(np.arange(6) * 60 + 5)]
    star = {"motored": {"name": "star", "segments": spokes, "scale": [0.12, 0.12], "position": [0.3, 0.85],
                        "angular_velocity_func": "lambda t: 4.0 * np.cos(t * 3)",
                        "velocity_func": "lambda t: np.array([0.4 * np.sin(t * 9), -0.2])"}}
    world = WorldConfig(rigid_bodies=list(world.rigid_bodies) + [star], particle_sources=world.particle_sources,
                        coefficients=world.coefficients)
    crate = Crate(world, precision="f64", noise="counter", noise_seed=5)
    contacts = 0
    for tick, pos, vel, prs in oracle_counter_run(world, 5, 50):
        crate.physics_tick()
        assert np.array_equal(crate.particles, pos) and np.array_equal(crate.particle_velocities, vel), tick
        contacts += int((point_segment_np(pos, crate.segments[-6:].reshape(-1, 4))[1] <= 1.5 * TOUCH).any(1).sum())
    crate.close()
    assert contacts >= 50, "the star must touch the liquid"


@gpu
@pytest.mark.parametrize("precision", [_lib.PRECISION_F64, _lib.PRECISION_MIXED])
def test_keys_from_the_force_kernel_equal_the_pre_pass_on_walls(precision):
    """The fan scene stepped straight (the force kernel keys the next tick) and with a get_state -> set_state_uids
    round trip before every tick (k_prepass keys it): bit-identical for 20 ticks."""
    pos, vel, walls = scene_multi("fans")
    cv = coeffs_for(D)
    ctxs = []
    for _ in range(2):
        ctx = _lib.Context(len(pos), precision)
        ctx.set_params(**params_from_coeffs(cv))
        ctx.set_walls(*walls)
        ctx.set_noise(_lib.NOISE_COUNTER, 3)
        ctx.set_state(pos, vel)
        ctxs.append(ctx)
    straight, tripped = ctxs
    contacts = 0
    for tick in range(20):
        gp, gv, _ = tripped.get_state()
        tripped.set_state_uids(gp, gv, tripped.get_uids())
        for ctx in ctxs:
            ctx.set_walls(*walls)
            ctx.set_tick(tick)
            ctx.step()
        contacts += int((straight.get_wall_counts(straight.particle_count()) >= 2).sum())
        a, b = straight.get_state(), tripped.get_state()
        for x, y in zip(a, b):
            assert np.array_equal(x, y), tick
        assert np.array_equal(straight.get_uids(), tripped.get_uids())
    assert contacts >= 100

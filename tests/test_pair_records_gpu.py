"""The production pair kernels checked on their own outputs (pytest -m gpu for the device tests).

`Context.get_pair_records` (sc_debug_pair_records) returns what the last tick's density kernel handed to its force
kernel: K_i, the neighbors in list order and the unit vectors as the force kernel decodes them.  `get_neighbors` re-runs
the untiled count kernel instead, so only this tap shows the tiled kernel's own lists.  Every case takes ONE step from
identical inputs and compares with `oracle.step(..., want_all=True)`: in fp64, and through the tiled mixed-precision
kernels with counter noise, without noise, and with the reference's noise stream from the host (a split step).

The scenes aim at the places a tiled kernel can be wrong while a random scene still passes: pairs inside the fp32
screen's band around d (the fp64 replay, per range and column offset), cell borders, the 20-trim in each of the four
ranges, and every block shape (staged, staged windows with unstaged cell slices, pass-through; partial blocks).  The
block kinds are predicted by a NumPy restatement of `tile_windows` (sc_tile.cuh) from the oracle's sorted rows.

The last group runs the force kernel with and without the ForceMonitor: the monitor variant always takes the general
fp64 wall / crossing path, so bit-identical results pin the bulk fast path against it.
"""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from conftest import golden, params_from_coeffs, step_goldens, world_from_freerun
from oracle import oracle as O
from sand_crate_b200 import Crate, _lib
from sand_crate_b200.scenes import BASE_COEFFICIENTS, UNIT_BOX, dam_break

MAXN = _lib.MAX_NEIGHBORS
SC_TILE = 256                                   # particles per block of the tiled kernels (sc_common.cuh)
SC_TILE_CAP = 5 * SC_TILE                       # staged particles per block (sc_tile.cuh)
SC_TILE_CELLS = SC_TILE + SC_TILE // 2 + 64     # staged cell boundaries per row slice (sc_tile.cuh)
SC_K5_ROWS = 6                                  # record slots K5 stages in shared memory (sc_tile.cuh)
BAND = 4e-6                                     # the fp32 screen decides alone outside d^2 (1 +- BAND)
U = 2.0 ** -23                                  # fp32 unit roundoff x 2 (one ulp at 1)

# |n_gpu - n_ref| <= VEC_C * U * (1 + d / dist) for the mixed-precision unit vectors, with dist the noised fp64
# distance.  Counted from the operations of density_particle (sc_tile.cuh) and pair_decode (sc_pair.cuh):
#  * rx = fmaf(col_i - col_j, d_f, rel_i.x - rel_j.x): the two fp32 cell-relative coordinates (|rel| < d) carry
#    2^-24 d each, the subtraction 2^-24 d, d_f = fl(d) 2^-24 d, the fma on |rx| <= 2d another 2^-23 d: 3 U d.
#    ry = (rel_i.y - rel_j.y) - (dr * d_f): the same, 3 U d.  Noise fmaf(0.5 - u, amp, rx): 0.5 - u is exact,
#    amp = fl(0.1 d) and the rounding of |rx| <= 1.1 d add 0.6 U d.  So |(drx, dry)| <= sqrt(2) * 3.6 U d = 5.1 U d,
#    which turns the direction by at most 5.1 U d / dist.
#  * length: fmaf(rx, rx, ry * ry) 2 roundings (U relative, half of it under the rsqrt), rsqrt.approx 2 ulp (2 U),
#    rx * inv 0.5 U: 3 U on the encoded (smaller) component m.
#  * decode: big = sqrt.approx(fmaf(-m, m, 1)): the error of m moves big by at most |m| / big <= 1 times it, the fmaf
#    rounding at >= 0.5 gives 0.36 U, sqrt.approx 2 ulp on big <= 1 gives 2 U: big is off by (m's error) + 2.4 U.
#  * both components: sqrt(2) * (5.4 U + direction) <= 7.7 U + 7.3 U d / dist.  VEC_C = 8 bounds both terms.
# fp64 mode stores the exact quotients: bit-exact.
VEC_C = 8.0
# Pressure and surface normal per particle, mixed: each pair's weight w = 1 - clip(dist / d) is off by the distance
# error above (5.1 U relative to d) plus q * inv * inv_d (0.5 + 2 + 0.5 + 0.5 + 0.5 U): <= 9 U; the fp32 sum of K
# weights <= 1 adds <= 10 U per addend (partials <= 20).  The normal's terms (1 - w) w n: |1 - 2 cl| <= 1 times the
# weight error, (1 - w) w <= 1/4 times the vector error (whose d / dist part is cancelled by (1 - w) w <= dist / d),
# roundings: < 17 U per term with the accumulation.  Bar: 20 U per neighbor, plus 2 U of the total for the
# subtraction of `ignored_pressure` and the final rounding.
PS_PER_PAIR = 20 * U
REL_TOL_F32 = 1e-5           # the per-step bars of tests/test_gpu_parity.py (SURVEY.md section 8(c))

MODES = {
    "f64": (_lib.PRECISION_F64, _lib.NOISE_COUNTER, None),
    "mixed_counter": (_lib.PRECISION_MIXED, _lib.NOISE_COUNTER, None),
    "mixed_none": (_lib.PRECISION_MIXED, _lib.NOISE_NONE, None),
    "mixed_level0": (_lib.PRECISION_MIXED, _lib.NOISE_COUNTER, 0.0),   # counter mode with a zero noise level
    "mixed_host": (_lib.PRECISION_MIXED, _lib.NOISE_HOST, None),       # uniforms from the host, split step
}
ORACLE_NOISE = {_lib.NOISE_NONE: 0, _lib.NOISE_COUNTER: 1, _lib.NOISE_HOST: 2}
NO_WALLS = (np.zeros((0, 4)), np.zeros(0, np.int32), np.zeros((0, 5)))
BOX_WALLS = (np.array(UNIT_BOX["fixed"]["segments"], np.float64).reshape(-1, 4), np.array([4], np.int32),
             np.zeros((1, 5)))


# ---- NumPy restatements (checked on the CPU below) ---------------------------------------------------------------
def pair_noise_np(tkey, uid_i, uid_j):
    """pair_noise_bits (sc_common.cuh) -> the two uniforms k / 65536, vectorised."""
    a = np.asarray(uid_i, np.uint32) & np.uint32(0x7FFFFFFF)
    b = np.asarray(uid_j, np.uint32) & np.uint32(0x7FFFFFFF)
    with np.errstate(over="ignore"):
        x = (a * np.uint32(0x9E3779B1)) ^ (b * np.uint32(0x85EBCA77)) ^ np.uint32((tkey ^ (tkey >> 32)) & 0xFFFFFFFF)
        x ^= x >> np.uint32(16); x *= np.uint32(0x7FEB352D)
        x ^= x >> np.uint32(15); x *= np.uint32(0x846CA68B)
        x ^= x >> np.uint32(16)
    return (x >> np.uint32(16)).astype(np.float64) / 65536.0, (x & np.uint32(0xFFFF)).astype(np.float64) / 65536.0


def cell_keys(pos, d, grid):
    """cell_of (sc_common.cuh): clamped (row - row_min) * ncols + (col - col_min)."""
    row_min, col_min, nrows, ncols = grid
    rows = np.floor(pos[:, 1] / d).astype(np.int64)
    cols = np.floor(pos[:, 0] / d).astype(np.int64)
    cr = np.clip(rows - row_min, 1, nrows - 2)
    cc = np.clip(cols - col_min, 1, ncols - 2)
    return cr * ncols + cc


def tile_windows_np(keys_sorted, ncells, ncols):
    """tile_windows (sc_tile.cuh) for every block of SC_TILE sorted particles, from the sorted cell keys: the block
    descriptor k_rank_gather writes, then the staging decision.  Returns a dict of per-block arrays."""
    n = len(keys_sorted)
    cs = np.concatenate(([0], np.cumsum(np.bincount(keys_sorted, minlength=ncells)))).astype(np.int64)
    b0 = np.arange(0, n, SC_TILE)
    c_lo, c_hi = keys_sorted[b0], keys_sorted[np.minimum(b0 + SC_TILE, n) - 1]
    lo = np.stack((cs[c_lo - 1], cs[c_lo + ncols - 1], cs[c_lo - ncols - 1]), 1)
    hi = np.stack((cs[c_hi + 2], cs[c_hi + ncols + 2], cs[c_hi - ncols + 2]), 1)
    base = lo & ~1
    cnt = (hi - base + 1) & ~1
    total = cnt.sum(1)
    ncw = c_hi - c_lo + 4
    staged = total <= SC_TILE_CAP
    off = np.where(staged[:, None], np.concatenate((np.zeros((len(b0), 1), np.int64), np.cumsum(cnt, 1)[:, :2]), 1), base)
    return {"base": base, "cnt": cnt, "off": off, "total": total, "ncw": ncw, "staged": staged,
            "cells_staged": staged & (ncw <= SC_TILE_CELLS)}


def band_pair_count(pos, d, width=3e-6):
    """Unordered pairs whose fp64 squared distance lies within d^2 (1 +- width).  With width 3e-6 < BAND - 1e-6 (the
    fp32 screen's evaluation error is below 1e-6 d^2) every such pair is certainly replayed in fp64 by the kernels."""
    pairs = cKDTree(pos).query_pairs(d * (1 + 2 * width), output_type="ndarray")
    if len(pairs) == 0:
        return 0
    q = ((pos[pairs[:, 0]] - pos[pairs[:, 1]]) ** 2).sum(1) / (d * d)
    return int((np.abs(q - 1) <= width).sum())


def safe_ccd(segments, r):
    """refresh_wall_boxes (sc_api.cu): the largest-area-greedy rectangle no padded segment's box meets."""
    pad = _lib.pad_segments(segments, r).reshape(-1, 4)
    boxes = []
    for ax, ay, bx, by in pad:
        xmin, xmax, ymin, ymax = min(ax, bx), max(ax, bx), min(ay, by), max(ay, by)
        e = 0.0 * (1.0 + 1e-6) + 1e-12 * max(1.0, max(max(abs(xmin), abs(xmax)), max(abs(ymin), abs(ymax))))
        boxes.append((xmin - e, xmax + e, ymin - e, ymax + e))
    rect = [-r, 1 + r, -r, 1 + r]
    meets = lambda b: b[0] < rect[1] and b[1] > rect[0] and b[2] < rect[3] and b[3] > rect[2]
    for _ in range(len(boxes) + 1):
        changed = False
        for b in boxes:
            if not meets(b):
                continue
            w_, h_ = rect[1] - rect[0], rect[3] - rect[2]
            area = [(rect[1] - b[1]) * h_, (b[0] - rect[0]) * h_, w_ * (rect[3] - b[3]), w_ * (b[2] - rect[2])]
            best = int(np.argmax(area))   # first maximum, like the strict > of the C loop
            rect[best] = [b[1], b[0], b[3], b[2]][best]
            changed = True
        if not changed:
            break
    assert rect[0] < rect[1] and rect[2] < rect[3] and not any(meets(b) for b in boxes)
    return np.array(rect)


def safe_ccd_f32(segments, r):
    """The rectangle of the force kernel's bulk fast path: safe_ccd shrunk by 1e-6 and rounded to fp32."""
    rect = safe_ccd(segments, r)
    return np.array([rect[0] + 1e-6, rect[1] - 1e-6, rect[2] + 1e-6, rect[3] - 1e-6], np.float32)


def coeffs_for(d, level=None):
    c = dict(BASE_COEFFICIENTS)
    c["particle_radius"] = d / 2
    c["dt"] = 0.002 * (d / 0.01)
    if level is not None:
        c["collider_noise_level"] = level
    return np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                     c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                     c["target_pressure"], c["gravity"][0], c["gravity"][1]], np.float64)


# ---- scenes (deterministic from their seeds) ---------------------------------------------------------------------
def _fp64_flip(ax, ay, ux, uy, d):
    """The last point B = A + t (ux, uy) (t near d, stepped one ulp at a time in its larger coordinate) with
    sqrt(dx^2 + dy^2) <= d, and the next one, which fails it."""
    big_x = abs(ux) >= abs(uy)
    bx, by = ax + d * ux, ay + d * uy
    ok = lambda x, y: np.sqrt((x - ax) ** 2 + (y - ay) ** 2) <= d
    step = lambda v, s: np.nextafter(v, np.inf if s > 0 else -np.inf)
    sgn = np.sign(ux) if big_x else np.sign(uy)
    for _ in range(64):
        if ok(bx, by):
            nx_, ny_ = (step(bx, sgn), by) if big_x else (bx, step(by, sgn))
            if not ok(nx_, ny_):
                return (bx, by), (nx_, ny_)
            bx, by = nx_, ny_
        else:
            bx, by = (step(bx, -sgn), by) if big_x else (bx, step(by, -sgn))
    raise AssertionError("no fp64 flip found")


def band_pairs(d, rs, slots):
    """Isolated pairs (A, B) at |AB| = d (1 + t), t straddling the fp32 band edges, the fp64 acceptance flip, and the
    reference's x-window quirk (dx = d exactly with dy = 0, which needs a d that A.x + d represents exactly: a power
    of two).  `slots`: centres at least 4 d apart, one pair each.
    Directions cover the same row, the row below and above, column offsets -1, 0, +1."""
    # in d^2 the band edges 1 +- 4e-6 sit at t = +-2e-6; |t| <= 1.5e-6 is certainly replayed in fp64
    ts = [-4e-6, -2.6e-6, -2.1e-6, -1.9e-6, -1.4e-6, -1e-6, -5e-7, -2e-7, 0.0, 2e-7, 5e-7, 1e-6, 1.4e-6, 1.9e-6,
          2.1e-6, 2.6e-6, 4e-6]
    angles = np.deg2rad(np.append(np.arange(0, 180, 7.5), 180 - 1e-4))
    pts, k = [], 0
    for t in ts:
        for a in angles:
            cx, cy = slots[k]; k += 1
            ax, ay = cx + rs.uniform(-0.25, 0.25) * d, cy + rs.uniform(-0.25, 0.25) * d
            pts += [(ax, ay), (ax + d * (1 + t) * np.cos(a), ay + d * (1 + t) * np.sin(a))]
    for a in angles:                                            # one ulp either side of the fp64 acceptance
        for keep in (0, 1):
            cx, cy = slots[k]; k += 1
            ax, ay = cx + rs.uniform(-0.25, 0.25) * d, cy + rs.uniform(-0.25, 0.25) * d
            inside, outside = _fp64_flip(ax, ay, np.cos(a), np.sin(a), d)
            pts += [(ax, ay), inside if keep else outside]
    n_quirk = 0
    while n_quirk < 12:                                         # dx == d exactly, dy == 0
        cx, cy = slots[k]; k += 1
        ax = cx + rs.uniform(-0.25, 0.25) * d
        if (ax + d) - ax == d:
            pts += [(ax, cy), (ax + d, cy)]
            n_quirk += 1
    return np.array(pts), k


def scene_band_staged(d=2.0 ** -10, seed=3):
    rs = np.random.RandomState(seed)
    # slots 3 d apart along a row (pairs of neighboring slots stay > 1.5 d apart), 4 d between rows
    gx, gy = np.arange(0.1, 0.9, 3 * d), np.arange(0.1, 0.9, 4 * d)
    slots = np.stack(np.meshgrid(gx, gy), -1).reshape(-1, 2)
    pts, _ = band_pairs(d, rs, slots)
    return pts


def scene_band_pass_through(d=2.0 ** -10, seed=4):
    """Band pairs in sparse rows directly above a dense row of 1300 particles (windows > SC_TILE_CAP: pass-through
    blocks), kept more than d away from it: pair particles at rel y < 0.3 d, dense particles at rel y > 0.6 d."""
    rs = np.random.RandomState(seed)
    out = []
    for unit in range(4):
        r0 = 200 + 40 * unit                                    # band rows r0 .. r0 + 1, dense row r0 + 2
        for i in range(70):                                     # same-row pairs only (the dense row is one row down)
            ax = 0.1 + i * 0.011 + rs.uniform(0, 0.001)
            ay = (r0 + (i % 2)) * d + rs.uniform(0.02, 0.05) * d
            t = [-3e-6, -1e-6, 0.0, 1e-6, 3e-6][i % 5]
            a = np.deg2rad(rs.uniform(-10, 10))
            out += [(ax, ay), (ax + d * (1 + t) * np.cos(a), ay + d * (1 + t) * np.sin(a))]
        dense_x = 0.1 + (np.arange(1300) + 0.5) * 0.6 * d
        out += list(np.stack((dense_x, (r0 + 2) * d + rs.uniform(0.6, 0.99, 1300) * d), 1))
    return np.array(out)


def scene_cell_borders(d=1e-3, seed=5):
    """Coordinates at k d and the fp64 values around it (where y / d, x / d round across the border), negative
    coordinates in [-r, 0) and rows near 1 + r; no walls (nothing moves them before the search)."""
    rs = np.random.RandomState(seed)
    r = d / 2
    ks = np.concatenate((np.arange(-0, 3), rs.choice(np.arange(3, 998), 60, replace=False), [998, 999, 1000]))
    pts = []
    for j, k in enumerate(ks):
        v = k * d
        for m in (-3, -1, 0, 1, 2):                                   # ulps around k d
            u = v
            for _ in range(abs(m)):
                u = np.nextafter(u, np.inf if m > 0 else -np.inf)
            other = 0.05 + 0.9 * rs.rand()
            pts += [(other, u), (u, other)]
    pts += [(0.3 + 0.7 * d * i, -r + (r * i / 40)) for i in range(40)]            # y in [-r, 0)
    pts += [(-r + (r * i / 40), 0.6 + 0.7 * d * i) for i in range(40)]            # x in [-r, 0)
    pts += [(0.2 + 0.7 * d * i, 1 + r - r * (i % 7) / 7) for i in range(60)]      # top rows
    pts = np.array(pts)
    return pts[(pts >= -r).all(1) & (pts <= 1 + r).all(1)]


def scene_trim_clumps(d=1e-3, seed=6, duplicates=True):
    """Clumps of 25 - 60 particles inside one diameter, centred at varied heights in their cell row, so that the
    20th accept of some particle lands in each of the four ranges; some clumps hold exact duplicates (only with
    noise: without it the reference's unit vector of a coincident pair is 0 / 0)."""
    rs = np.random.RandomState(seed)
    pts = []
    for c in range(48):
        cx, cy = 0.1 + 0.8 * rs.rand(), (100 + 5 * c) * d + [0.02, 0.3, 0.5, 0.7, 0.98][c % 5] * d
        m = rs.randint(25, 61)
        rad = 0.45 * d * np.sqrt(rs.rand(m))
        ang = 2 * np.pi * rs.rand(m)
        clump = np.stack((cx + rad * np.cos(ang), cy + rad * np.sin(ang)), 1)
        if duplicates and c % 4 == 0:
            clump[5:9] = clump[4]                                      # exact duplicates: ties broken by uid
        pts.append(clump)
    return np.concatenate(pts)


def scene_blob(n, d=1e-3, seed=7):
    rs = np.random.RandomState(seed + n)
    side = max(np.sqrt(n) * 0.75 * d, d)
    return 0.5 + (rs.rand(n, 2) - 0.5) * side


def scene_row_wrap(d=1e-3, seed=8):
    """Rows holding particles only at their right end, followed by rows holding particles only at their left end: a
    block that runs from one into the other spans ~ a row of cells (ncw > SC_TILE_CELLS) while its windows stay small
    (staged windows, cell slices from global memory)."""
    rs = np.random.RandomState(seed)
    out = []
    for unit in range(8):
        r0 = 300 + 6 * unit
        out.append(np.stack((0.80 + 0.08 * rs.rand(140), (r0 + rs.rand(140)) * d), 1))
        out.append(np.stack((0.12 + 0.08 * rs.rand(140), (r0 + 1 + rs.rand(140)) * d), 1))
    return np.concatenate(out)


# ---- one step on the device and on the oracle, and the checks ----------------------------------------------------
def run_step(pos, vel, mode, d, walls=NO_WALLS, seed=17, tick=5):
    precision, noise, level = MODES[mode]
    cv = coeffs_for(d, level)
    if precision == _lib.PRECISION_MIXED:
        vel = vel.astype(np.float32).astype(np.float64)          # what the device holds
    ctx = _lib.Context(len(pos), precision)
    ctx.set_params(**params_from_coeffs(cv))
    ctx.set_walls(*walls)
    ctx.set_noise(noise, seed)
    ctx.set_state(pos, vel)
    ctx.set_tick(tick)
    host = None
    if noise == _lib.NOISE_HOST:
        _, n_pairs = ctx.step_begin()
        host = np.random.RandomState(seed).rand(n_pairs, 2)
        ctx.step_finish(host)
    else:
        ctx.step()
    tkey = O.tick_key(seed, tick)
    ref = O.step(cv, pos, vel, *walls, noise_mode=ORACLE_NOISE[noise], noise=host, tkey=tkey, want_all=True)
    return ctx, ref, cv, vel, tkey, host


def ref_vectors(ref, cv, noise_on, tkey=None, host_noise=None):
    """The reference's unit vectors (crate.py:167-174) per list slot, restated from pos_search: nvec[i, k], dist[i, k]."""
    ps, cnt, idx = ref["pos_search"], ref["nbr_count"], ref["nbr_idx_padded"]
    d, level = 2 * cv[1], cv[5]
    i, k = np.nonzero(np.arange(MAXN)[None, :] < cnt[:, None])
    j = idx[i, k]
    qx, qy = ps[j, 0].copy(), ps[j, 1].copy()
    if noise_on:
        if host_noise is not None:
            off = np.concatenate(([0], np.cumsum(cnt)))[i] + k
            u = np.asarray(host_noise).reshape(-1, 2)          # CSR order: particle, slot; x then y
            ux, uy = u[off, 0], u[off, 1]
        else:
            ux, uy = pair_noise_np(tkey, i, j)
        qx = qx + (ux - 0.5) * d * level
        qy = qy + (uy - 0.5) * d * level
    rx, ry = ps[i, 0] - qx, ps[i, 1] - qy
    dist = np.sqrt(rx * rx + ry * ry)
    nv = np.zeros((len(cnt), MAXN, 2))
    dd = np.full((len(cnt), MAXN), np.inf)
    nv[i, k, 0], nv[i, k, 1], dd[i, k] = rx / dist, ry / dist, dist
    return nv, dd


def check_records(ctx, ref, cv, mode, tkey, host_noise=None):
    n = len(ref["nbr_count"])
    counts, rows, nvec = ctx.get_pair_records(n)
    assert np.array_equal(counts, ref["nbr_count"]), "K of the density kernel"
    assert np.array_equal(rows, ref["nbr_idx_padded"]), "lists of the density kernel (order + trim)"
    noise_on = MODES[mode][1] != _lib.NOISE_NONE if mode in MODES else True
    nv, dist = ref_vectors(ref, cv, noise_on, tkey, host_noise)
    d = 2 * cv[1]
    if mode == "f64":
        assert np.array_equal(nvec, nv)
    else:
        err = np.sqrt(((nvec - nv) ** 2).sum(-1))
        bound = VEC_C * U * (1 + d / dist)
        assert (err <= bound).all(), (float((err / bound).max()), np.argwhere(err > bound)[:5])
    return counts


def check_physics(ctx, ref, cv, mode, vel_in):
    n = len(ref["nbr_count"])
    pos, vel, prs = ctx.get_state()
    tens = ctx.get_tension(n)
    if mode == "f64":
        assert np.array_equal(prs, ref["pressure"]) and np.array_equal(tens, ref["tension_vec"])
        assert np.array_equal(vel, ref["vel_out"]) and np.array_equal(pos, ref["pos_out"])
        return
    K = ref["nbr_count"]
    bar = PS_PER_PAIR * K + 2 * U * (np.abs(ref["pressure"]) + abs(cv[4]))
    assert (np.abs(prs - ref["pressure"]) <= bar).all(), float((np.abs(prs - ref["pressure"]) / bar).max())
    tbar = PS_PER_PAIR * K + 2 * U * np.abs(ref["tension_vec"]).max(1)
    assert (np.abs(tens - ref["tension_vec"]).max(1) <= tbar).all()
    d = 2 * cv[1]
    v_floor = 0.01 * d / cv[0]
    assert np.abs(vel - ref["vel_out"]).max() <= REL_TOL_F32 * max(np.abs(ref["vel_out"]).max(), v_floor)
    assert np.abs(pos - ref["pos_out"]).max() <= REL_TOL_F32 * d
    dv_ref = ref["vel_out"] - vel_in
    if np.abs(dv_ref).max() > 0:
        assert np.abs((vel - vel_in) - dv_ref).max() <= REL_TOL_F32 * np.abs(dv_ref).max()


def predicted_blocks(ctx, ref, d):
    """tile_windows restated on the oracle's search; also checks the device's sorted order and rows."""
    n = len(ref["nbr_count"])
    ps = ref["pos_search"]
    rows_o, order_o, _, _ = O.detect_particle_collisions(ps, d)
    gps, grows, gorder = ctx.get_search(n)
    assert np.array_equal(gps, ps) and np.array_equal(gorder, order_o) and np.array_equal(grows, rows_o)
    grid = ctx.grid()
    keys = cell_keys(ps, d, grid)[order_o]
    return tile_windows_np(keys, grid[2] * grid[3], grid[3]), order_o


def run_case(pos, mode, d, walls=NO_WALLS, vel=None, seed=17):
    vel = np.zeros_like(pos) if vel is None else vel
    ctx, ref, cv, vin, tkey, host = run_step(pos, vel, mode, d, walls, seed)
    check_records(ctx, ref, cv, mode, tkey, host)
    return ctx, ref, cv, vin


# ---- CPU: the restatements ---------------------------------------------------------------------------------------
def test_pair_noise_restatement_matches_oracle():
    tkey = O.tick_key(17, 5)
    ui, uj = np.array([0, 1, 7, 123456, 2 ** 31 - 1, 0x80000005]), np.array([3, 0, 7, 99, 5, 12])
    ux, uy = pair_noise_np(tkey, ui, uj)
    for a, b, x, y in zip(ui, uj, ux, uy):
        assert (x, y) == O.pair_noise(tkey, int(a), int(b))


def test_tile_windows_restatement_on_hand_built_layouts():
    ncols, nrows = 1000, 12
    # one particle in cell 2001, two per cell in 2005 .. 2132 (row 2), one per cell in 3005 .. 3105 (row 3)
    keys = np.sort(np.concatenate(([2001], np.repeat(2005 + np.arange(128), 2), 3005 + np.arange(101))))
    w = tile_windows_np(keys, ncols * nrows, ncols)
    # block 0 (cells 2001 .. 2132): W0 = [cs[2000], cs[2134]) = [0, 257), W1 = [257, 358), W2 empty; bases round down
    # to even, counts up to even
    assert w["base"][0].tolist() == [0, 256, 0] and w["cnt"][0].tolist() == [258, 102, 0]
    assert w["off"][0].tolist() == [0, 258, 360] and w["staged"][0] and w["cells_staged"][0]
    # block 1 runs from the end of row 2 into row 3 (cells 2132 .. 3105): windows staged, cell slices not
    assert w["base"][1].tolist() == [252, 358, 0] and w["cnt"][1].tolist() == [106, 0, 206]
    assert w["staged"][1] and not w["cells_staged"][1] and w["ncw"][1] == 3105 - 2132 + 4
    # windows beyond SC_TILE_CAP: pass-through, local index = sorted index
    keys = np.sort(np.concatenate((np.full(200, 2500), np.full(56, 3500), np.full(1500, 4501))))
    w = tile_windows_np(keys, ncols * nrows, ncols)
    assert not w["staged"][0] and w["total"][0] > SC_TILE_CAP and (w["off"][0] == w["base"][0]).all()
    # a partial last block: descriptor from its last live particle
    w = tile_windows_np(np.sort(np.full(300, 5005)), ncols * nrows, ncols)
    assert len(w["staged"]) == 2 and w["ncw"][1] == 4


def test_band_pair_count():
    d = 1e-3
    pts = np.array([[0.5, 0.5], [0.5 + d, 0.5], [0.2, 0.2], [0.2 + 1.01 * d, 0.2], [0.7, 0.7],
                    [0.7 + d * (1 + 1e-6) / np.sqrt(2), 0.7 + d * (1 + 1e-6) / np.sqrt(2)]])
    assert band_pair_count(pts, d) == 2
    assert band_pair_count(scene_band_staged(), 2.0 ** -10) >= 200


def test_safe_rectangle_restatement_is_inside_the_padded_walls():
    seg, r = BOX_WALLS[0], 0.004
    f = safe_ccd_f32(seg, r)
    assert np.float32(r) < f[0] < np.float32(r + 2e-6) and np.float32(1 - r - 2e-6) < f[1] < np.float32(1 - r)
    assert f[2] == f[0] and f[3] == f[1]


# ---- GPU: the tap against the oracle -----------------------------------------------------------------------------
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_band_lattice_staged(mode):
    d = 2.0 ** -10
    pos = scene_band_staged(d)
    assert band_pair_count(pos, d) >= 250, "the fp64 replay must be exercised"
    ctx, ref, cv, vin = run_case(pos, mode, d)
    w, order = predicted_blocks(ctx, ref, d)
    assert w["staged"].all()
    if mode != "f64":
        assert ctx.untiled_blocks() == 0
    # every range and column offset holds a band pair: (dr, dc) of each list entry, forward direction
    row = np.floor(ref["pos_search"][:, 1] / d).astype(np.int64)
    col = np.floor(ref["pos_search"][:, 0] / d).astype(np.int64)
    i = np.repeat(np.arange(len(pos)), ref["nbr_count"])
    j = ref["nbr_idx"]
    seen = {(int(a), int(b)) for a, b in zip(row[j] - row[i], col[j] - col[i])}
    assert {(0, 0), (0, 1), (0, -1), (1, -1), (1, 0), (1, 1), (-1, -1), (-1, 0), (-1, 1)} <= seen, seen
    check_physics(ctx, ref, cv, mode, vin)


@gpu
@pytest.mark.parametrize("mode", ["mixed_counter", "mixed_none", "mixed_host", "f64"])
def test_band_lattice_pass_through(mode):
    d = 2.0 ** -10
    pos = scene_band_pass_through(d)
    ctx, ref, cv, vin = run_case(pos, mode, d)
    w, order = predicted_blocks(ctx, ref, d)
    if mode != "f64":
        assert ctx.untiled_blocks() == int((~w["staged"]).sum()) > 0
    # band particles that sit in pass-through blocks
    blk_of = np.empty(len(pos), np.int64)
    blk_of[order] = np.arange(len(pos)) // SC_TILE
    in_band = np.zeros(len(pos), bool)
    pairs = cKDTree(pos).query_pairs(d * (1 + 6e-6), output_type="ndarray")
    q = ((pos[pairs[:, 0]] - pos[pairs[:, 1]]) ** 2).sum(1) / d ** 2
    in_band[pairs[np.abs(q - 1) <= 3e-6].ravel()] = True
    assert (in_band & ~w["staged"][blk_of]).sum() >= 40
    check_physics(ctx, ref, cv, mode, vin)


@gpu
@pytest.mark.parametrize("mode", ["f64", "mixed_counter", "mixed_none"])
def test_cell_borders(mode):
    d = 1e-3
    pos = scene_cell_borders(d)
    rs = np.random.RandomState(9)
    ctx, ref, cv, vin = run_case(pos, mode, d, vel=rs.randn(*pos.shape) * 0.01)
    predicted_blocks(ctx, ref, d)      # sorted order and rows equal the oracle's
    check_physics(ctx, ref, cv, mode, vin)


@gpu
@pytest.mark.parametrize("mode", ["f64", "mixed_counter", "mixed_none", "mixed_host"])
def test_trim_in_every_range(mode):
    d = 1e-3
    pos = scene_trim_clumps(d, duplicates=MODES[mode][1] != _lib.NOISE_NONE)
    ctx, ref, cv, vin = run_case(pos, mode, d)
    cnt, idx = ref["nbr_count"], ref["nbr_idx_padded"]
    rows_o, order, _, _ = O.detect_particle_collisions(ref["pos_search"], d)
    spos = np.empty(len(pos), np.int64)
    spos[order] = np.arange(len(pos))
    row = np.floor(ref["pos_search"][:, 1] / d).astype(np.int64)
    full = np.nonzero(cnt == MAXN)[0]
    last = idx[full, MAXN - 1]
    dr = row[last] - row[full]
    rng = np.where(dr == 1, 2, np.where(dr == -1, 4, np.where(spos[last] > spos[full], 1, 3)))
    assert set(rng.tolist()) == {1, 2, 3, 4}, np.bincount(rng)
    check_physics(ctx, ref, cv, mode, vin)


@gpu
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 511, 513])
def test_block_shapes_small_n(n):
    d = 1e-3
    pos = scene_blob(n, d)
    for mode in ("f64", "mixed_counter", "mixed_none"):
        ctx, ref, cv, vin = run_case(pos, mode, d)
        check_physics(ctx, ref, cv, mode, vin)
        ctx.close()


@gpu
@pytest.mark.parametrize("mode", ["mixed_counter", "mixed_none", "mixed_level0", "mixed_host", "f64"])
def test_block_kinds_predicted_exactly(mode):
    """One scene with every block kind: staged, staged windows with cell slices from global memory (a block wrapping a
    row end), pass-through; records beyond the staged slots (K > SC_K5_ROWS) and K == 0."""
    d = 1e-3
    pos = np.concatenate((scene_row_wrap(d), scene_band_pass_through(d), scene_blob(3000, d)))
    ctx, ref, cv, vin = run_case(pos, mode, d)
    w, _ = predicted_blocks(ctx, ref, d)
    assert (w["staged"] & w["cells_staged"]).any()
    assert (w["staged"] & ~w["cells_staged"]).any()
    assert (~w["staged"]).any()
    if mode != "f64":
        assert ctx.untiled_blocks() == int((~w["staged"]).sum())
    assert (ref["nbr_count"] > SC_K5_ROWS).any() and (ref["nbr_count"] == 0).any()
    check_physics(ctx, ref, cv, mode, vin)


@gpu
@pytest.mark.parametrize("name", step_goldens()[::3])
def test_golden_steps_tiled_host_noise(name):
    """Host noise through the tiled kernels on the recorded scenes (walls, moving bodies)."""
    g = golden(name)
    ctx = _lib.Context(max(len(g["pos_in"]), 1), _lib.PRECISION_MIXED)
    ctx.set_params(**params_from_coeffs(g["coeffs"]))
    ctx.set_walls(g["segments"], g["body_len"], g["body_kin"])
    ctx.set_noise(_lib.NOISE_HOST, 0)
    ctx.set_state(g["pos_in"], g["vel_in"])
    ctx.step_begin()
    with pytest.raises(_lib.SandCrateError, match="split step"):
        ctx.get_pair_records(len(g["pos_in"]))
    ctx.step_finish(g["noise"])
    n = len(g["pos_search"])
    ref = {"pos_search": g["pos_search"], "nbr_count": g["nbr_count"]}
    idx = np.full((n, MAXN), -1, np.int32)
    off = np.concatenate(([0], np.cumsum(g["nbr_count"])))
    for i in range(n):
        idx[i, :g["nbr_count"][i]] = g["nbr_idx"][off[i]:off[i + 1]]
    ref["nbr_idx_padded"] = idx
    check_records(ctx, ref, g["coeffs"], "mixed_host", None, host_noise=g["noise"])


@gpu
def test_tap_refuses_before_a_step():
    ctx = _lib.Context(4, _lib.PRECISION_MIXED)
    ctx.set_params(**params_from_coeffs(coeffs_for(1e-3)))
    with pytest.raises(_lib.SandCrateError, match="no search state"):
        ctx.get_pair_records(4)


@gpu
@pytest.mark.parametrize("mode", ["f64", "mixed_counter", "mixed_level0", "mixed_host"])
def test_debug_rerun_repeats_the_step_kernels(mode):
    """sc_debug_rerun re-runs the kernels the step ran, with its effective noise mode: state and records are unchanged.
    Under host noise it refuses (-1): the noise offsets need not outlive the step."""
    d = 1e-3
    pos = scene_blob(3000, d)
    ctx, ref, cv, vin, tkey, host = run_step(pos, np.zeros_like(pos), mode, d, BOX_WALLS)
    if mode != "mixed_host":
        ctx.step()                     # this step's force kernel also keys the next tick: the rerun must drop that
    n = len(pos)
    before = ctx.get_state() + ctx.get_pair_records(n)
    rerun = lambda which: ctx._L.sc_debug_rerun(ctx._h, which, 1)
    if mode == "mixed_host":
        assert rerun(4) == -1.0 and rerun(5) == -1.0
    else:
        assert rerun(4) > 0 and rerun(5) > 0
    after = ctx.get_state() + ctx.get_pair_records(n)
    for a, b in zip(before, after):
        assert np.array_equal(a, b)


# ---- the monitor variant against the bulk fast path --------------------------------------------------------------
def edge_particles(d, r, dt, gy):
    """Isolated particles (K = 0, no wall contact at the start) whose movement ends at the fast path's safe rectangle:
    within a few fp32 ulps of each side of the shrunk fp32 rectangle, and - on the two sides near 1, where an fp32
    coordinate is only good to 6e-8 - just beyond the padded wall, from a start whose fp32 rounding is almost half an
    ulp low.  Those movements cross the padded wall in fp64 while their fp32 box ends inside the UNshrunk rectangle:
    only the 1e-6 shrink keeps them off the fast path."""
    f = safe_ccd_f32(BOX_WALLS[0], r)
    exact = safe_ccd(BOX_WALLS[0], r)
    f_dt = np.float32(dt)
    pts, vel = [], []
    for side in range(4):
        ends = []
        for m in range(-4, 5):
            edge = f[side]
            for _ in range(abs(m)):
                edge = np.nextafter(edge, np.float32(np.inf if m > 0 else -np.inf))
            ends.append((float(edge), False))
        if side in (1, 3):
            ends += [(exact[side] + k * 2e-9, True) for k in range(1, 9)]
        for q, (end, low_start) in enumerate(ends):
            # left wall: above the liquid column of dam_break (its top is near y = 0.2); elsewhere clear of it
            along = [0.03, 0.5, 0.55, 0.62][side] + 0.012 * q
            g_t = np.float32(dt * gy) if side >= 2 else np.float32(0)   # x: vx is not changed by the tick (K = V = 0)
            speed = (0.3 * r) / dt * (-1 if side in (0, 2) else 1)
            start = end - speed * dt
            if low_start:
                s32 = np.float32(start)
                start = float(s32) + 0.49 * float(np.spacing(s32))
                speed = (end - start) / dt
            v0 = np.float32(np.float32(speed) - g_t)       # the velocity the fast path tests is v0 + dt * g
            v_t = np.float32(v0 + g_t)
            if not low_start:
                start = end - float(v_t) * float(f_dt)
            p, v = [along, along], [0.0, 0.0]
            p[side // 2], v[side // 2] = start, float(v0)
            pts.append(tuple(p)); vel.append(tuple(v))
    return np.array(pts), np.array(vel)


@gpu
def test_monitor_variant_bit_identical_to_fast_path_and_oracle_monitor():
    n = 100_000
    # The radius is moved by a few 1e-9 from the scene's own so that fl32(1 - r), the fp32 image of the padded floor
    # and right wall, lies ABOVE 1 - r: only then can an fp32 box test without the shrink accept a movement that
    # crosses them (edge_particles).
    r0 = dam_break(n)[0].coefficients["particle_radius"]
    overhang = lambda r: float(np.float32(safe_ccd(BOX_WALLS[0], r)[1])) - (1 - r)
    r = next(r0 + j * 1e-9 for j in range(400) if 2e-8 < overhang(r0 + j * 1e-9) < 2.9e-8)
    world, pos, vel = dam_break(n, particle_radius=r)
    c = world.coefficients
    r, d, dt = c["particle_radius"], 2 * c["particle_radius"], c["dt"]
    ep, ev = edge_particles(d, r, dt, c["gravity"][1])
    # keep the edge particles clear of the liquid column and of each other
    assert cKDTree(pos).query(ep)[0].min() > 2 * d and cKDTree(ep).query(ep, k=2)[0][:, 1].min() > 2 * d
    pos, vel = np.concatenate((pos, ep)), np.concatenate((vel, ev))
    cv = np.array([dt, r, c["wall_collision_decay"], c["pressure_amplifier"], c["ignored_pressure"],
                   c["collider_noise_level"], c["viscosity"], c["surface_smoothing"], c["target_pressure"],
                   c["gravity"][0], c["gravity"][1]])
    ctxs = []
    for monitor in (False, True):
        ctx = _lib.Context(len(pos), _lib.PRECISION_MIXED)
        ctx.set_params(**params_from_coeffs(cv))
        ctx.set_walls(*BOX_WALLS)
        ctx.set_noise(_lib.NOISE_COUNTER, 21)
        ctx.set_monitor(monitor)
        ctx.set_state(pos, vel)
        ctxs.append(ctx)
    vin = vel.astype(np.float32).astype(np.float64)
    for tick in range(20):
        for ctx in ctxs:
            ctx.set_tick(tick)
            ctx.step()
        a, b = ctxs[0].get_state(want_pressure=False), ctxs[1].get_state(want_pressure=False)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), tick
        if tick == 0:
            ref = O.step(cv, pos, vin, *BOX_WALLS, noise_mode=1, tkey=O.tick_key(21, 0), want_all=True)
            assert np.array_equal(ref["nbr_count"][-len(ep):], np.zeros(len(ep)))
            sums, cnt = ctxs[1].get_monitor()
            assert cnt == len(pos)
            # Per particle, every stage velocity of the device is within the per-step increment bar (1e-5 of the
            # tick's largest increment) of the reference's, plus the fp32 rounding of the running velocity (half an
            # ulp per stage, 6 stages); |dv| of a stage takes that from both of its ends, and the mean keeps the bound.
            dv_max = np.abs(ref["vel_out"] - vin).max()
            v_max = max(np.abs(ref["vel_out"]).max(), np.abs(vin).max())
            tol = 2 * (REL_TOL_F32 * dv_max + 6 * 2.0 ** -24 * v_max) + 1e-12
            assert np.abs(sums / cnt - ref["force_monitor"]).max() <= tol, (sums / cnt, ref["force_monitor"], tol)
            check_physics(ctxs[0], ref, cv, "mixed_counter", vin)


@gpu
def test_monitor_on_off_bit_identical_wave_machine():
    """wave_machine's first 150 ticks (sources, the moving paddle) with and without the monitor, no noise."""
    world, _ = world_from_freerun("wave_machine")
    runs = []
    for monitor in (False, True):
        np.random.seed(5)
        crate = Crate(world, precision="mixed", noise="none", monitor=monitor)
        np.random.seed(5)
        states = []
        for _ in range(150):
            crate.physics_tick()
            states.append((crate.particles.copy(), crate.particle_velocities.copy()))
        runs.append(states)
        crate.close()
    assert len(runs[0][-1][0]) > 500
    for t, ((p0, v0), (p1, v1)) in enumerate(zip(*runs)):
        assert np.array_equal(p0, p1) and np.array_equal(v0, v1), t

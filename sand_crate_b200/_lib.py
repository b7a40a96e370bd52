"""ctypes binding of include/sandcrate.h (libsandcrate.so, sm_100a).

This is the only way the Python host side reaches the GPU: there is no CPU fallback.  If the shared library is
missing it is built in-tree with nvcc (sand_crate_b200/build.py); if that fails, or no B200 is visible when a
context is created, the call raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

MAX_NEIGHBORS = 20
MAX_SEGMENTS = 32
MAX_BODIES = 16
PROFILE_SLOTS = 16

PRECISION_F64 = 0
PRECISION_MIXED = 1
NOISE_NONE = 0
NOISE_COUNTER = 1
NOISE_HOST = 2

PARAM_FIELDS = ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier", "ignored_pressure",
                "collider_noise_level", "viscosity", "surface_smoothing", "target_pressure", "gravity_x", "gravity_y")


class ScParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in PARAM_FIELDS]


class ScSource(C.Structure):
    _fields_ = [("position_x", C.c_double), ("position_y", C.c_double), ("radius", C.c_double),
                ("velocity_x", C.c_double), ("velocity_y", C.c_double), ("velocity_noise", C.c_double),
                ("count", C.c_int32), ("index", C.c_uint32)]


class SandCrateError(RuntimeError):
    pass


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)
_up = C.POINTER(C.c_uint32)
_ctx = C.c_void_p

# name -> (restype, argtypes); tests/test_abi.py checks that every function declared in include/sandcrate.h is here
SIGNATURES = {
    "sc_create": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_void_p, C.POINTER(_ctx)]),
    "sc_destroy": (None, [_ctx]),
    "sc_last_error": (C.c_char_p, [_ctx]),
    "sc_version": (C.c_int, []),
    "sc_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "sc_host_free": (C.c_int, [C.c_void_p]),
    "sc_set_params": (C.c_int, [_ctx, C.POINTER(ScParams)]),
    "sc_set_walls": (C.c_int, [_ctx, _dp, C.c_int, _ip, _dp, C.c_int]),
    "sc_set_noise": (C.c_int, [_ctx, C.c_int, C.c_uint64]),
    "sc_set_tick": (C.c_int, [_ctx, C.c_uint64]),
    "sc_set_state": (C.c_int, [_ctx, _dp, _dp, C.c_int64]),
    "sc_append_particles": (C.c_int, [_ctx, _dp, _dp, C.c_int64]),
    "sc_particle_count": (C.c_int, [_ctx, _lp]),
    "sc_emit_particles": (C.c_int, [_ctx, C.POINTER(ScSource), C.c_int, C.c_int64]),
    "sc_source_stream": (C.c_uint64, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, _dp]),
    "sc_get_state": (C.c_int, [_ctx, _dp, _dp, _dp, C.c_int64, _lp]),
    "sc_get_uids": (C.c_int, [_ctx, _up, C.c_int64, _lp]),
    "sc_step": (C.c_int, [_ctx]),
    "sc_step_n": (C.c_int, [_ctx, C.c_int]),
    "sc_step_begin": (C.c_int, [_ctx, _lp, _lp]),
    "sc_step_finish": (C.c_int, [_ctx, _dp]),
    "sc_synchronize": (C.c_int, [_ctx]),
    "sc_get_search": (C.c_int, [_ctx, _dp, _lp, _lp, C.c_int64]),
    "sc_get_neighbors": (C.c_int, [_ctx, _ip, _ip, C.c_int64]),
    "sc_get_tension": (C.c_int, [_ctx, _dp, C.c_int64]),
    "sc_get_wall_counts": (C.c_int, [_ctx, _ip, C.c_int64]),
    "sc_detect_particle_collisions": (C.c_int, [_ctx, _dp, C.c_int64, C.c_double, _lp, _lp, _ip, _ip]),
    "sc_points_to_segments_distance": (C.c_int, [_ctx, _dp, C.c_int64, _dp, C.c_int, _dp, _dp]),
    "sc_pad_segments": (C.c_int, [_dp, C.c_int, C.c_double, _dp]),
    "sc_dist_wire_bytes": (C.c_int64, [C.c_int64]),
    "sc_dist_configure": (C.c_int, [_ctx, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int64]),
    "sc_dist_pack": (C.c_int, [_ctx, C.c_void_p, C.c_void_p]),
    "sc_dist_unpack": (C.c_int, [_ctx, C.c_void_p, C.c_void_p]),
    "sc_dist_unpack_flagged": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "sc_dist_pack_push": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]),
    "sc_dist_get_owned": (C.c_int, [_ctx, _dp, _dp, _up, C.c_int64, _lp]),
    "sc_dist_status": (C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), _lp]),
    "sc_dist_row_histogram": (C.c_int, [_ctx, C.c_int64, C.c_int64, C.POINTER(C.c_uint64)]),
    "sc_dist_set_rows": (C.c_int, [_ctx, C.c_int64, C.c_int64]),
    "sc_dist_set_reach": (C.c_int, [_ctx, C.c_int64, C.c_int64]),
    "sc_set_state_uids": (C.c_int, [_ctx, _dp, _dp, _up, C.c_int64]),
    "sc_set_next_uid": (C.c_int, [_ctx, C.c_uint32]),
    "sc_dist_halo_rows": (C.c_int, [_dp, C.c_int, C.c_double]),
    "sc_dist_owned_count": (C.c_int, [_ctx, C.c_void_p]),
    "sc_dist_emit_particles": (C.c_int, [_ctx, C.POINTER(ScSource), C.c_int, C.c_int64, C.c_uint32, C.c_void_p]),
    "sc_set_monitor": (C.c_int, [_ctx, C.c_int]),
    "sc_get_monitor": (C.c_int, [_ctx, _dp, _lp]),
    "sc_profile_enable": (C.c_int, [_ctx, C.c_int]),
    "sc_profile_read": (C.c_int, [_ctx, _lp, _dp, C.c_int]),
    "sc_profile_name": (C.c_char_p, [C.c_int]),
    "sc_launch_count": (C.c_int64, [_ctx]),
    "sc_sync_count": (C.c_int64, [_ctx]),
    "sc_last_pair_count": (C.c_int, [_ctx, _lp]),
    "sc_debug_rerun": (C.c_double, [_ctx, C.c_int, C.c_int]),
    "sc_debug_untiled_blocks": (C.c_int64, [_ctx]),
    "sc_debug_pair_records": (C.c_int, [_ctx, _ip, _ip, _dp, C.c_int64]),
    "sc_debug_grid": (C.c_int, [_ctx, _lp]),
    "sc_debug_walls": (C.c_int, [_ctx, _dp, _dp, _dp, _ip]),
    "sc_ens_configure": (C.c_int, [_ctx, C.c_int, C.c_int]),
    "sc_ens_set_params": (C.c_int, [_ctx, C.POINTER(ScParams), C.POINTER(C.c_uint64)]),
    "sc_ens_set_state": (C.c_int, [_ctx, _dp, _dp, _lp, _up, _up]),
    "sc_ens_emit_particles": (C.c_int, [_ctx, C.POINTER(ScSource), C.c_int, _ip, _lp]),
    "sc_ens_member_counts": (C.c_int, [_ctx, _lp, C.c_void_p]),
    "sc_ens_get_state": (C.c_int, [_ctx, _dp, _dp, _dp, C.c_int64, _lp]),
}

_lib = None


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """dlopen libsandcrate.so (building it first if the sources are newer).  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and _build.needs_build():
        _build.build()
    if not os.path.exists(_build.LIB):
        raise SandCrateError(f"{_build.LIB} is missing and could not be built; there is no CPU fallback")
    L = C.CDLL(_build.LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _f64(a, shape_last=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape_last is not None:
        a = a.reshape(-1, shape_last)
    return a


def _ptr(a, typ):
    return a.ctypes.data_as(typ) if a is not None else None


class _PinnedBlock:
    """One cudaHostAlloc allocation; freed when the last reference to it goes."""

    def __init__(self, L, nbytes):
        self._L = L
        self._p = C.c_void_p()
        if L.sc_host_alloc(max(nbytes, 1), C.byref(self._p)):
            raise SandCrateError(L.sc_last_error(None).decode())

    def __del__(self):
        try:
            if self._p.value:
                self._L.sc_host_free(self._p)
                self._p = C.c_void_p()
        except Exception:
            pass


class PinnedArray:
    """A NumPy array over page-locked host memory (sc_host_alloc).  The memory belongs to the ARRAY: every view of it
    keeps the allocation alive (NumPy base chain -> ctypes buffer -> block), so an array handed out by `Crate.particles`
    stays valid for as long as somebody holds it - like the reference's own arrays - even after the context that filled
    it is closed or has grown a larger buffer.  `close()` only drops this object's reference."""

    def __init__(self, shape, dtype=np.float64):
        self.shape = tuple(int(x) for x in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        block = _PinnedBlock(load(), nbytes)
        raw = (C.c_byte * max(nbytes, 1)).from_address(block._p.value)
        raw._block = block   # the ctypes buffer (which NumPy keeps as the array's base) owns the allocation
        self.array = np.frombuffer(raw, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def close(self):
        self.array = None


class Context:
    """Owns one `sc_ctx`.  Thin: every method is one C-ABI call plus NumPy buffer management."""

    def __init__(self, capacity: int, precision: int = PRECISION_F64, device: int = 0, stream: int | None = None):
        self._L = load()
        self._h = _ctx()
        rc = self._L.sc_create(int(device), int(precision), int(capacity), C.c_void_p(stream) if stream else None,
                               C.byref(self._h))
        if rc:
            raise SandCrateError(self._L.sc_last_error(None).decode())
        self.capacity = int(capacity)
        self.precision = int(precision)
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value is not None:
            self._L.sc_destroy(self._h)
            self._h = _ctx()
        for b in getattr(self, "_pinned", {}).values():
            b.close()
        self._pinned = {}

    def _pinned_rows(self, name: str, rows: int, shape_tail=(), dtype=np.float64):
        """A reusable page-locked readback buffer with room for `rows` rows (grown by doubling)."""
        bufs = self.__dict__.setdefault("_pinned", {})
        b = bufs.get(name)
        if b is None or b.shape[0] < rows:
            b = bufs[name] = PinnedArray((max(rows, self.capacity),) + tuple(shape_tail), dtype)
        return b.array

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise SandCrateError(self._L.sc_last_error(self._h).decode())

    # ---- configuration ----
    def set_params(self, **kw):
        p = ScParams(*[float(kw[n]) for n in PARAM_FIELDS])
        self._ck(self._L.sc_set_params(self._h, C.byref(p)))

    def set_walls(self, segments, body_len, body_kin):
        seg = _f64(segments, 4)
        bl = np.ascontiguousarray(body_len, dtype=np.int32)
        bk = _f64(body_kin, 5)
        self._ck(self._L.sc_set_walls(self._h, _ptr(seg, _dp), seg.shape[0], _ptr(bl, _ip), _ptr(bk, _dp), bl.shape[0]))

    def set_noise(self, mode: int, seed: int = 0):
        self._ck(self._L.sc_set_noise(self._h, int(mode), C.c_uint64(seed)))

    def set_tick(self, tick: int):
        self._ck(self._L.sc_set_tick(self._h, C.c_uint64(tick)))

    # ---- state ----
    def set_state(self, pos, vel):
        pos, vel = _f64(pos, 2), _f64(vel, 2)
        assert pos.shape == vel.shape
        self._ck(self._L.sc_set_state(self._h, _ptr(pos, _dp), _ptr(vel, _dp), pos.shape[0]))

    def append_particles(self, pos, vel):
        pos, vel = _f64(pos, 2), _f64(vel, 2)
        assert pos.shape == vel.shape
        self._ck(self._L.sc_append_particles(self._h, _ptr(pos, _dp), _ptr(vel, _dp), pos.shape[0]))

    def emit_particles(self, records, max_particles: int):
        """records: `ParticleSource.emit_record` tuples of the sources that emit this tick (device-side sources)."""
        arr = (ScSource * len(records))(*[ScSource(*r) for r in records])
        self._ck(self._L.sc_emit_particles(self._h, arr, len(records), int(max_particles)))

    def particle_count(self) -> int:
        n = C.c_int64()
        self._ck(self._L.sc_particle_count(self._h, C.byref(n)))
        return n.value

    def get_state(self, want_vel=True, want_pressure=True, reuse=False, want_pos=True):
        """reuse=True: the arrays are views of this context's page-locked readback buffers - valid until the next
        reuse=True call or close() (the reference's own `particles` array is updated in place just the same)."""
        n = self.particle_count()
        if not want_pos:
            pos = None
        elif reuse:
            pos = self._pinned_rows("pos", n, (2,))[:n]
        if reuse:
            vel = self._pinned_rows("vel", n, (2,))[:n] if want_vel else None
            prs = self._pinned_rows("prs", n)[:n] if want_pressure else None
        else:
            pos = np.empty((n, 2)) if want_pos else None
            vel = np.empty((n, 2)) if want_vel else None
            prs = np.empty(n) if want_pressure else None
        m = C.c_int64()
        self._ck(self._L.sc_get_state(self._h, _ptr(pos, _dp), _ptr(vel, _dp), _ptr(prs, _dp), n, C.byref(m)))
        assert m.value == n
        return pos, vel, prs

    def get_uids(self):
        n = self.particle_count()
        uid = np.empty(n, np.uint32)
        m = C.c_int64()
        self._ck(self._L.sc_get_uids(self._h, _ptr(uid, _up), n, C.byref(m)))
        return uid

    # ---- step ----
    def step(self, n: int = 1):
        self._ck(self._L.sc_step_n(self._h, int(n)) if n != 1 else self._L.sc_step(self._h))

    def step_begin(self):
        n, k = C.c_int64(), C.c_int64()
        self._ck(self._L.sc_step_begin(self._h, C.byref(n), C.byref(k)))
        return n.value, k.value

    def step_finish(self, noise=None):
        if noise is not None:
            noise = _f64(noise)
        self._ck(self._L.sc_step_finish(self._h, _ptr(noise, _dp)))

    def synchronize(self):
        self._ck(self._L.sc_synchronize(self._h))

    # ---- taps ----
    def get_search(self, n: int):
        pos = np.empty((n, 2))
        rows = np.empty(n, np.int64)
        order = np.empty(n, np.int64)
        self._ck(self._L.sc_get_search(self._h, _ptr(pos, _dp), _ptr(rows, _lp), _ptr(order, _lp), n))
        return pos, rows, order

    def get_neighbors(self, n: int):
        counts = np.empty(n, np.int32)
        idx = np.empty((n, MAX_NEIGHBORS), np.int32)
        self._ck(self._L.sc_get_neighbors(self._h, _ptr(counts, _ip), _ptr(idx, _ip), n))
        return counts, idx

    def get_tension(self, n: int):
        t = np.empty((n, 2))
        self._ck(self._L.sc_get_tension(self._h, _ptr(t, _dp), n))
        return t

    def get_wall_counts(self, n: int):
        c = np.empty(n, np.int32)
        self._ck(self._L.sc_get_wall_counts(self._h, _ptr(c, _ip), n))
        return c

    # ---- standalone layer-2 ops ----
    def detect_particle_collisions(self, particles, diameter):
        pts = _f64(particles, 2)
        P = pts.shape[0]
        rows = np.empty(P, np.int64)
        order = np.empty(P, np.int64)
        counts = np.empty(P, np.int32)
        idx = np.empty((P, MAX_NEIGHBORS), np.int32)
        self._ck(self._L.sc_detect_particle_collisions(self._h, _ptr(pts, _dp), P, float(diameter), _ptr(rows, _lp),
                                                       _ptr(order, _lp), _ptr(counts, _ip), _ptr(idx, _ip)))
        return rows, order, counts, idx

    def points_to_segments_distance(self, p, segments):
        p = _f64(p, 2)
        seg = _f64(segments, 4)
        near = np.empty((p.shape[0], seg.shape[0], 2))
        dist = np.empty((p.shape[0], seg.shape[0]))
        self._ck(self._L.sc_points_to_segments_distance(self._h, _ptr(p, _dp), p.shape[0], _ptr(seg, _dp), seg.shape[0],
                                                        _ptr(near, _dp), _ptr(dist, _dp)))
        return near, dist

    # ---- strip decomposition (device pointers are plain ints, e.g. torch.Tensor.data_ptr()) ----
    def set_state_uids(self, pos, vel, uid):
        pos, vel = _f64(pos, 2), _f64(vel, 2)
        uid = np.ascontiguousarray(uid, dtype=np.uint32)
        assert pos.shape == vel.shape and uid.shape[0] == pos.shape[0]
        self._ck(self._L.sc_set_state_uids(self._h, _ptr(pos, _dp), _ptr(vel, _dp), _ptr(uid, _up), pos.shape[0]))

    def set_next_uid(self, next_uid: int):
        """The uid the next appended or emitted particle gets (sc_set_next_uid)."""
        self._ck(self._L.sc_set_next_uid(self._h, C.c_uint32(next_uid)))

    def dist_configure(self, rank, nranks, row_lo, row_hi, halo_rows, wire_capacity):
        self._ck(self._L.sc_dist_configure(self._h, int(rank), int(nranks), int(row_lo), int(row_hi), int(halo_rows),
                                           int(wire_capacity)))

    @staticmethod
    def _devptr(buf):
        """None, an integer device address, or anything with data_ptr() (a torch tensor on this GPU)."""
        if buf is None:
            return C.c_void_p(None)
        return C.c_void_p(int(buf.data_ptr()) if hasattr(buf, "data_ptr") else int(buf))

    def dist_pack(self, send_lo, send_hi):
        self._ck(self._L.sc_dist_pack(self._h, self._devptr(send_lo), self._devptr(send_hi)))

    def dist_unpack(self, recv_lo, recv_hi):
        self._ck(self._L.sc_dist_unpack(self._h, self._devptr(recv_lo), self._devptr(recv_hi)))

    def dist_pack_push(self, lo, hi, value):
        """pack with the records written straight into the neighbors' receive buffers.  lo / hi: None or (send buffer,
        peer receive address, peer flag address)."""
        lo, hi = lo or (None, None, None), hi or (None, None, None)
        self._ck(self._L.sc_dist_pack_push(self._h, *[self._devptr(x) for x in lo], *[self._devptr(x) for x in hi],
                                           C.c_uint32(value)))

    def dist_unpack_flagged(self, lo, hi, value):
        """lo / hi: None or (receive address, flag address)."""
        lo, hi = lo or (None, None), hi or (None, None)
        self._ck(self._L.sc_dist_unpack_flagged(self._h, *[self._devptr(x) for x in lo],
                                                *[self._devptr(x) for x in hi], C.c_uint32(value)))

    def dist_row_histogram(self, row0: int, nrows: int):
        hist = np.zeros(nrows, np.uint64)
        self._ck(self._L.sc_dist_row_histogram(self._h, int(row0), int(nrows), hist.ctypes.data_as(C.POINTER(C.c_uint64))))
        return hist

    def dist_set_rows(self, row_lo: int, row_hi: int):
        self._ck(self._L.sc_dist_set_rows(self._h, int(row_lo), int(row_hi)))

    def dist_set_reach(self, far_lo: int, far_hi: int):
        self._ck(self._L.sc_dist_set_reach(self._h, int(far_lo), int(far_hi)))

    def dist_owned_count(self, count_dev):
        """Enqueue: this rank's live non-ghost particle count -> the 4-byte device word `count_dev` (no host wait)."""
        self._ck(self._L.sc_dist_owned_count(self._h, self._devptr(count_dev)))

    def dist_emit_particles(self, records, max_particles: int, first_uid: int, scene_count_dev=None):
        """Device-side sources on a strip: `records` as for emit_particles, the same on every rank; `scene_count_dev`:
        a device word holding the scene's particle count, or None where the clamp cannot bind."""
        arr = (ScSource * len(records))(*[ScSource(*r) for r in records])
        self._ck(self._L.sc_dist_emit_particles(self._h, arr, len(records), int(max_particles), C.c_uint32(first_uid),
                                                self._devptr(scene_count_dev)))

    def dist_get_owned(self, want_vel=True, want_uid=True, reuse=False):
        """(pos, vel, uid) of the owned particles.  reuse=True: views of page-locked buffers, valid until the next
        reuse=True call; parts not asked for come back as None."""
        cap = self.capacity
        n = C.c_int64()
        if reuse:
            pos = self._pinned_rows("own_pos", cap, (2,))
            vel = self._pinned_rows("own_vel", cap, (2,)) if want_vel else None
            uid = self._pinned_rows("own_uid", cap, (), np.uint32) if want_uid else None
        else:
            pos = np.empty((cap, 2))
            vel = np.empty((cap, 2)) if want_vel else None
            uid = np.empty(cap, np.uint32) if want_uid else None
        self._ck(self._L.sc_dist_get_owned(self._h, _ptr(pos, _dp), _ptr(vel, _dp), _ptr(uid, _up), cap, C.byref(n)))
        m = n.value
        if reuse:
            return pos[:m], None if vel is None else vel[:m], None if uid is None else uid[:m]
        return pos[:m].copy(), None if vel is None else vel[:m].copy(), None if uid is None else uid[:m].copy()

    def dist_status(self, send_lo=None, send_hi=None):
        ov, far, n = C.c_int(), C.c_int(), C.c_int64()
        self._ck(self._L.sc_dist_status(self._h, self._devptr(send_lo), self._devptr(send_hi),
                                        C.byref(ov), C.byref(far), C.byref(n)))
        return {"overflow": bool(ov.value), "too_far": bool(far.value), "n_local": n.value}

    # ---- ForceMonitor ----
    def set_monitor(self, on: bool = True):
        self._ck(self._L.sc_set_monitor(self._h, int(on)))

    def get_monitor(self):
        """(sum over particles of |dv| for the six force sections, particle count) of the last tick."""
        sums = np.zeros(6)
        n = C.c_int64()
        self._ck(self._L.sc_get_monitor(self._h, _ptr(sums, _dp), C.byref(n)))
        return sums, n.value

    # ---- measurement ----
    def profile_enable(self, on: bool = True):
        self._ck(self._L.sc_profile_enable(self._h, int(on)))

    def profile_read(self):
        launches = np.zeros(PROFILE_SLOTS, np.int64)
        ms = np.zeros(PROFILE_SLOTS)
        self._ck(self._L.sc_profile_read(self._h, _ptr(launches, _lp), _ptr(ms, _dp), PROFILE_SLOTS))
        out = {}
        for i in range(PROFILE_SLOTS):
            name = self._L.sc_profile_name(i).decode()
            if name and launches[i]:
                out[name] = {"launches": int(launches[i]), "ms": float(ms[i])}
        return out

    def launch_count(self) -> int:
        return int(self._L.sc_launch_count(self._h))

    def sync_count(self) -> int:
        return int(self._L.sc_sync_count(self._h))

    def last_pair_count(self) -> int:
        n = C.c_int64()
        self._ck(self._L.sc_last_pair_count(self._h, C.byref(n)))
        return n.value

    def untiled_blocks(self) -> int:
        return int(self._L.sc_debug_untiled_blocks(self._h))

    def get_pair_records(self, n: int):
        """(counts, neighbor rows, unit vectors) of the pair records the last tick's density kernel handed to its
        force kernel, in original index order (sc_debug_pair_records)."""
        counts = np.empty(n, np.int32)
        rows = np.empty((n, MAX_NEIGHBORS), np.int32)
        nvec = np.empty((n, MAX_NEIGHBORS, 2))
        self._ck(self._L.sc_debug_pair_records(self._h, _ptr(counts, _ip), _ptr(rows, _ip), _ptr(nvec, _dp), n))
        return counts, rows, nvec

    def grid(self):
        """(row_min, col_min, nrows, ncols) of the cell grid (sc_debug_grid)."""
        g = np.zeros(4, np.int64)
        self._ck(self._L.sc_debug_grid(self._h, _ptr(g, _lp)))
        return tuple(int(x) for x in g)

    def debug_walls(self):
        """The wall culls of the current walls (sc_debug_walls): a dict of safe_contact, safe_ccd, safe_ccd_f32 (4 each),
        seg_box (S x 4), pad_box (2S x 4), each as (xmin, xmax, ymin, ymax), and `contacts`, the wall contacts per
        particle the cell grid has room for."""
        rects = np.empty(12)
        seg_box, pad_box = np.empty((MAX_SEGMENTS, 4)), np.empty((2 * MAX_SEGMENTS, 4))
        counts = np.zeros(2, np.int32)
        self._ck(self._L.sc_debug_walls(self._h, _ptr(rects, _dp), _ptr(seg_box, _dp), _ptr(pad_box, _dp),
                                        _ptr(counts, _ip)))
        S = int(counts[0])
        return {"safe_contact": rects[0:4], "safe_ccd": rects[4:8], "safe_ccd_f32": rects[8:12],
                "seg_box": seg_box[:S].copy(), "pad_box": pad_box[:2 * S].copy(), "contacts": int(counts[1])}


    # ---- ensembles (include/sandcrate.h "ensembles") ----
    def ens_configure(self, members: int, uid_bits: int):
        self._ck(self._L.sc_ens_configure(self._h, int(members), int(uid_bits)))
        self.members = int(members)

    def ens_set_params(self, params, seeds):
        """params: one keyword dict of PARAM_FIELDS per member; seeds: one noise seed per member."""
        arr = (ScParams * len(params))(*[ScParams(*[float(p[n]) for n in PARAM_FIELDS]) for p in params])
        sd = np.ascontiguousarray(seeds, dtype=np.uint64)
        self._ck(self._L.sc_ens_set_params(self._h, arr, sd.ctypes.data_as(C.POINTER(C.c_uint64))))

    def ens_set_state(self, pos, vel, counts, uid=None, next_local=None):
        """Member-major rows, counts[m] of member m; uid (global) and next_local (per member) default to a fresh
        numbering (sc_ens_set_state)."""
        pos, vel = _f64(pos, 2), _f64(vel, 2)
        counts = np.ascontiguousarray(counts, dtype=np.int64)
        assert pos.shape == vel.shape and counts.sum() == pos.shape[0]
        uid = None if uid is None else np.ascontiguousarray(uid, dtype=np.uint32)
        nxt = None if next_local is None else np.ascontiguousarray(next_local, dtype=np.uint32)
        self._ck(self._L.sc_ens_set_state(self._h, _ptr(pos, _dp), _ptr(vel, _dp), _ptr(counts, _lp), _ptr(uid, _up),
                                          _ptr(nxt, _up)))

    def ens_emit_particles(self, records, counts, max_particles):
        """records: `ParticleSource.emit_record` tuples (their count is ignored); counts: members x len(records) drawn
        counts; max_particles: one per member."""
        arr = (ScSource * len(records))(*[ScSource(*r) for r in records])
        cnt = np.ascontiguousarray(counts, dtype=np.int32).reshape(-1)
        mx = np.ascontiguousarray(max_particles, dtype=np.int64)
        self._ck(self._L.sc_ens_emit_particles(self._h, arr, len(records), _ptr(cnt, _ip), _ptr(mx, _lp)))

    def ens_member_counts(self, counts_dev=None, want_host=True):
        """Per-member live counts (synchronises) and/or, enqueued without a host wait, into the uint32 device words
        `counts_dev`."""
        counts = np.zeros(self.members, np.int64) if want_host else None
        self._ck(self._L.sc_ens_member_counts(self._h, _ptr(counts, _lp), self._devptr(counts_dev)))
        return counts

    def ens_get_state(self, want_pressure=True):
        """(pos, vel, pressure, offsets) of all members, member-major; member m's rows are offsets[m]:offsets[m + 1]."""
        n = self.particle_count()
        pos, vel = np.empty((n, 2)), np.empty((n, 2))
        prs = np.empty(n) if want_pressure else None
        off = np.zeros(self.members + 1, np.int64)
        self._ck(self._L.sc_ens_get_state(self._h, _ptr(pos, _dp), _ptr(vel, _dp), _ptr(prs, _dp), n, _ptr(off, _lp)))
        return pos, vel, prs, off


def source_uniform(seed: int, tick: int, source_index: int, j: int) -> float:
    """Element j of a source's counter stream (host arithmetic of the library, no GPU needed)."""
    u = C.c_double()
    load().sc_source_stream(C.c_uint64(seed), C.c_uint64(tick), C.c_uint32(source_index), C.c_uint64(j), C.byref(u))
    return u.value


def wire_bytes(wire_capacity: int) -> int:
    return int(load().sc_dist_wire_bytes(int(wire_capacity)))


def dist_halo_rows(segments, particle_radius: float) -> int:
    """The halo rows a strip needs under these walls (sc_dist_halo_rows; host arithmetic, no GPU needed)."""
    seg = _f64(segments, 4)
    h = int(load().sc_dist_halo_rows(_ptr(seg, _dp), seg.shape[0], float(particle_radius)))
    if h < 0:
        raise SandCrateError("sc_dist_halo_rows: bad arguments")
    return h


def pad_segments(segments, pad):
    """geometry_utils.py:146-172 through the C ABI (host arithmetic, no GPU needed)."""
    seg = _f64(segments, 4)
    out = np.empty((2 * seg.shape[0], 2, 2))
    load().sc_pad_segments(_ptr(seg, _dp), seg.shape[0], float(pad), _ptr(out, _dp))
    return out

"""Test double: a `Context` look-alike that runs the step through the CPU oracle (oracle/step_oracle.c).

It exists so the HOST logic of `sand_crate_b200.Crate` (RNG protocol, particle sources, rigid-body motion, lazy
counts, capacity growth) can be tested on a machine without a GPU.  It lives under tests/ because only tests may
touch oracle/; the product never sees it."""
import numpy as np

from oracle import oracle as O
from sand_crate_b200._lib import SandCrateError


class OracleContext:
    def __init__(self, capacity, precision=0, device=0, stream=None):
        self.capacity, self.precision, self.device = int(capacity), precision, device
        self.pos = np.zeros((0, 2))
        self.vel = np.zeros((0, 2))
        self.prs = np.zeros(0)
        self.uid = np.zeros(0, np.uint32)
        self.next_uid = 0
        self.params = None
        self.walls = None
        self.noise_mode, self.seed, self.tick = 0, 0, 0
        self._pending = None

    def close(self):
        pass

    def set_params(self, **kw):
        self.params = kw

    def set_walls(self, segments, body_len, body_kin):
        self.walls = (np.array(segments, dtype=np.float64).reshape(-1, 4), np.array(body_len, np.int32),
                      np.array(body_kin, dtype=np.float64).reshape(-1, 5))

    def set_noise(self, mode, seed=0):
        self.noise_mode, self.seed = mode, seed

    def set_tick(self, tick):
        self.tick = tick

    def profile_enable(self, on=True):
        pass

    def set_monitor(self, on=True):
        self.monitor = None

    def get_monitor(self):
        return self.monitor * len(self.prs), len(self.prs)

    def profile_read(self):
        return {}

    def set_state(self, pos, vel):
        self.pos, self.vel = np.array(pos, dtype=np.float64), np.array(vel, dtype=np.float64)
        self.uid = np.arange(len(self.pos), dtype=np.uint32)
        self.next_uid = len(self.pos)
        self.prs = np.zeros(len(self.pos))
        self.pair_cnt = None

    def append_particles(self, pos, vel):
        assert len(self.pos) + len(pos) <= self.capacity
        self.pos = np.vstack((self.pos, pos))
        self.vel = np.vstack((self.vel, vel))
        self.uid = np.concatenate((self.uid, np.arange(self.next_uid, self.next_uid + len(pos), dtype=np.uint32)))
        self.next_uid += len(pos)
        self.prs = np.zeros(len(self.pos))

    def emit_particles(self, records, max_particles):
        """sc_emit_particles: the oracle's restatement of the device-side sources.  Identities advance by the DRAWN
        counts (a clamp leaves a gap), like the library's."""
        if not records:
            return
        src = np.array([r[:6] for r in records], dtype=np.float64)
        cnt = np.array([r[6] for r in records], dtype=np.int32)
        idx = np.array([r[7] for r in records], dtype=np.uint32)
        import ctypes as C
        pos = np.zeros((int(cnt.sum()), 2))
        vel = np.zeros((int(cnt.sum()), 2))
        P = len(self.pos)
        m = O.lib().oc_emit_counter(C.c_uint64(O.tick_key(self.seed, self.tick)), len(records), O._dp(src), O._ip(cnt),
                                    idx.ctypes.data_as(C.POINTER(C.c_uint32)), P, int(max_particles), O._dp(pos), O._dp(vel))
        uids, base, room = [], self.next_uid, max(int(max_particles) - P, 0)
        for n in cnt:
            a = min(int(n), room)
            uids.append(np.arange(base, base + a, dtype=np.uint32))
            base += int(n)
            room -= a
        self.next_uid = base
        self.pos = np.vstack((self.pos, pos[:m]))
        self.vel = np.vstack((self.vel, vel[:m]))
        self.uid = np.concatenate([self.uid] + uids)
        self.prs = np.zeros(len(self.pos))

    def particle_count(self):
        return len(self.pos)

    def get_state(self, want_vel=True, want_pressure=True, reuse=False, want_pos=True):
        return self.pos.copy(), self.vel.copy(), self.prs.copy()

    def _coeffs(self):
        p = self.params
        return np.array([p[k] for k in ("dt", "particle_radius", "wall_collision_decay", "pressure_amplifier",
                                        "ignored_pressure", "collider_noise_level", "viscosity",
                                        "surface_smoothing", "target_pressure", "gravity_x", "gravity_y")])

    def _remove(self):
        pos, vel, mask = O.remove_particles(self.pos, self.vel, self.params["particle_radius"])
        self.uid = self.uid[~mask]
        self.pos, self.vel = pos, vel

    def _sort_by_identity(self):
        """The oracle breaks exact x ties by array index (= uid order in a single domain, like np.lexsort's
        stability in the reference); a strip's local arrays are in arrival order, so restore uid order first."""
        order = np.argsort(self.uid & np.uint32(0x7FFFFFFF), kind="stable")
        self.pos, self.vel, self.uid = self.pos[order], self.vel[order], self.uid[order]

    def step_begin(self):
        self._sort_by_identity()
        self._remove()
        seg, bl, bk = self.walls
        probe = O.step(self._coeffs(), self.pos, self.vel, seg, bl, bk, noise_mode=0)
        self._pending = True
        return len(self.pos), int(probe["nbr_count"].sum())

    def step_finish(self, noise=None):
        seg, bl, bk = self.walls
        mode = self.noise_mode if self.params["collider_noise_level"] != 0 else 0
        out = O.step(self._coeffs(), self.pos, self.vel, seg, bl, bk, noise_mode=mode, noise=noise,
                     tkey=O.tick_key(self.seed, self.tick), uid=self.uid & np.uint32(0x7FFFFFFF))
        self.pos, self.vel, self.prs = out["pos_out"], out["vel_out"], out["pressure"]
        self.pair_cnt = np.asarray(out["nbr_count"], dtype=np.int64)   # K_i of this tick, in the order of self.pos
        self.monitor = out["force_monitor"]
        self.tick += 1
        self._pending = None

    def step(self, n=1):
        for _ in range(n):
            self.step_begin()
            self.step_finish(None)

    # ---- strip decomposition: the same protocol as sc_dist_* (csrc/sc_dist.cuh), in NumPy -----------------------
    WIRE_REC = np.dtype([("px", "f8"), ("py", "f8"), ("vx", "f8"), ("vy", "f8"), ("uid", "u4"), ("kind", "u4")])
    GHOST = np.uint32(0x80000000)

    def set_state_uids(self, pos, vel, uid):
        self.set_state(pos, vel)
        self.uid = np.array(uid, dtype=np.uint32)
        self.next_uid = int(self.uid.max()) + 1 if len(self.uid) else 0

    def set_next_uid(self, next_uid):
        """sc_set_next_uid: refused below the current next uid and at or above 2^31."""
        if not self.next_uid <= next_uid < 2 ** 31:
            raise SandCrateError(f"sc_set_next_uid: {next_uid} out of range")
        self.next_uid = int(next_uid)

    def dist_configure(self, rank, nranks, row_lo, row_hi, halo_rows, wire_capacity):
        self.dist = dict(lo=row_lo, hi=row_hi, halo=halo_rows, has_lo=rank > 0, has_hi=rank < nranks - 1,
                         cap=wire_capacity)
        self.flags = {"overflow": False, "too_far": False}

    def _write_wire(self, tensor, recs):
        raw = tensor.numpy()
        assert len(recs) <= self.dist["cap"], "wire overflow"
        raw[:16].view(np.uint32)[:] = [len(recs), 0, 0, 0]
        raw[16:16 + 40 * len(recs)].view(self.WIRE_REC)[:] = recs

    def _read_wire(self, tensor):
        raw = tensor.numpy()
        n = int(raw[:16].view(np.uint32)[0])
        return raw[16:16 + 40 * n].view(self.WIRE_REC).copy()

    def _records(self, mask, kind):
        r = np.zeros(int(mask.sum()), self.WIRE_REC)
        r["px"], r["py"] = self.pos[mask, 0], self.pos[mask, 1]
        r["vx"], r["vy"] = self.vel[mask, 0], self.vel[mask, 1]
        r["uid"], r["kind"] = self.uid[mask], kind
        return r

    def dist_pack(self, send_lo, send_hi):
        D = self.dist
        self.pair_cnt = None   # the arrays change below: the last tick's pair counts no longer line up (rows_valid)
        keep = (self.uid & self.GHOST) == 0
        self.pos, self.vel, self.uid = self.pos[keep], self.vel[keep], self.uid[keep]
        d = 2 * self.params["particle_radius"]
        rows = np.floor(self.pos[:, 1] / d).astype(np.int64)
        below = (rows < D["lo"]) & D["has_lo"]
        above = (rows >= D["hi"]) & D["has_hi"]
        owned = ~(below | above)
        if (below & (rows < D["lo"] - D["halo"])).any() or (above & (rows >= D["hi"] + D["halo"])).any():
            self.flags["too_far"] = True
        if D["has_lo"]:
            self._write_wire(send_lo, np.concatenate([self._records(below, 0),
                                                      self._records(owned & (rows < D["lo"] + D["halo"]), 1)]))
        if D["has_hi"]:
            self._write_wire(send_hi, np.concatenate([self._records(above, 0),
                                                      self._records(owned & (rows >= D["hi"] - D["halo"]), 1)]))
        self.uid = np.where(owned, self.uid, self.uid | self.GHOST).astype(np.uint32)
        self.prs = np.zeros(len(self.pos))

    def dist_unpack(self, recv_lo, recv_hi):
        for has, buf in ((self.dist["has_lo"], recv_lo), (self.dist["has_hi"], recv_hi)):
            if not has:
                continue
            r = self._read_wire(buf)
            self.pos = np.vstack((self.pos, np.stack((r["px"], r["py"]), 1)))
            self.vel = np.vstack((self.vel, np.stack((r["vx"], r["vy"]), 1)))
            self.uid = np.concatenate((self.uid, np.where(r["kind"] == 1, r["uid"] | self.GHOST, r["uid"]))).astype(np.uint32)
        assert len(self.pos) <= self.capacity, "particle capacity overflow"
        self.prs = np.zeros(len(self.pos))

    WORK_BASE = 2   # sc_api.cu work_base(): a particle weighs 2 + its pair count of the last tick

    def dist_row_histogram(self, row0, nrows):
        """k_dist_row_hist restated: summed weight of the owned particles per cell row, outliers clamped to the ends;
        equal weights while there is no tick whose pair counts match the arrays."""
        own = (self.uid & self.GHOST) == 0
        d = 2 * self.params["particle_radius"]
        rows = np.clip(np.floor(self.pos[own, 1] / d).astype(np.int64) - row0, 0, nrows - 1)
        k = getattr(self, "pair_cnt", None)
        w = np.full(int(own.sum()), self.WORK_BASE, dtype=np.int64)
        if k is not None and len(k) == len(self.pos):
            w = w + k[own]
        return np.bincount(rows, weights=w, minlength=nrows).astype(np.uint64)

    def dist_set_rows(self, row_lo, row_hi):
        self.dist["lo"], self.dist["hi"] = row_lo, row_hi

    def dist_get_owned(self, want_vel=True, want_uid=True, reuse=False):
        own = (self.uid & self.GHOST) == 0
        return self.pos[own].copy(), self.vel[own].copy(), self.uid[own].copy()

    def dist_status(self, send_lo=None, send_hi=None):
        return dict(self.flags, n_local=len(self.pos))

    def get_uids(self):
        return self.uid.copy()

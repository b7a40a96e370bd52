"""Test double for open scenes on strips: OracleContext (tests/oracle_backend.py) plus the two entry points that
particle sources on a strip need, restated in NumPy from sc_dist.cuh (k_dist_owned_count, k_dist_emit)."""
import ctypes as C

import numpy as np

from oracle import oracle as O
from oracle_backend import OracleContext


class OpenOracleContext(OracleContext):
    def dist_owned_count(self, count_dev):
        """This rank's live particles that are not ghosts, into the caller's one-element tensor."""
        count_dev[0] = int(((self.uid & self.GHOST) == 0).sum())

    def dist_emit_particles(self, records, max_particles, first_uid, scene_count_dev=None):
        """sc_emit_particles' clamp with particle_count = the scene's count (None: no clamp), identities from the
        scene-wide `first_uid`, and only the rows this strip owns appended, in (source, k) order."""
        if not records:
            return
        src = np.array([r[:6] for r in records], dtype=np.float64)
        cnt = np.array([r[6] for r in records], dtype=np.int32)
        idx = np.array([r[7] for r in records], dtype=np.uint32)
        total = int(cnt.sum())
        P, cap = (int(scene_count_dev[0]), int(max_particles)) if scene_count_dev is not None else (0, total)
        pos, vel = np.zeros((total, 2)), np.zeros((total, 2))
        m = O.lib().oc_emit_counter(C.c_uint64(O.tick_key(self.seed, self.tick)), len(records), O._dp(src), O._ip(cnt),
                                    idx.ctypes.data_as(C.POINTER(C.c_uint32)), P, cap, O._dp(pos), O._dp(vel))
        uids, base, room = [], int(first_uid), max(cap - P, 0)
        for n in cnt:
            a = min(int(n), room)
            uids.append(np.arange(base, base + a, dtype=np.uint32))
            base += int(n)
            room -= a
        pos, vel, uid = pos[:m], vel[:m], np.concatenate(uids)
        rows = np.floor(pos[:, 1] / (2 * self.params["particle_radius"])).astype(np.int64)
        mine = (rows >= self.dist["lo"]) & (rows < self.dist["hi"])
        self.pos = np.vstack((self.pos, pos[mine]))
        self.vel = np.vstack((self.vel, vel[mine]))
        self.uid = np.concatenate((self.uid, uid[mine])).astype(np.uint32)
        self.next_uid = max(self.next_uid, base)
        self.prs = np.zeros(len(self.pos))
        assert len(self.pos) <= self.capacity, "particle capacity overflow"

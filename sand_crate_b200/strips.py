"""Strip decomposition of one scene across the GPUs of a box: one process per GPU, `torch.distributed` for the
plumbing (NCCL over NVLink on GPUs; gloo in the CPU tests), the C ABI's `sc_dist_*` entry points for the device work.

The reference's neighbor search is already a 1-D strip decomposition in y with strip height one diameter
(collision_detector.py:10-31, 124-128).  The same cell rows are the partition unit here: rank k owns the rows
`cuts[k] <= floor(y / d) < cuts[k + 1]`, chosen so that every rank starts with the same number of particles.

Per tick (SURVEY.md section 8(e)):

    pack      device: migrants (row left the strip) + halo copies (within `halo_rows` of a cut) -> two wire buffers
    exchange  isend / irecv of the fixed-size buffers with rank - 1 and rank + 1 only (open chain: walls at y = 0, 1)
    unpack    device: migrants become owned particles, halos become ghosts
    step      the ordinary single-GPU tick on owned + ghosts; the next pack throws the ghosts away

There is no collective on the data path and no host synchronisation: the buffers have a fixed capacity and carry
their own record count, particle counts stay on the device.
"""
from __future__ import annotations

import time

import numpy as np

from . import _lib

HALO_ROWS = 4  # see DESIGN.md section 6: 1 row of neighbors + 1 row for their pressures/normals + 2 for wall-fix shifts
INT64_MIN, INT64_MAX = -(2 ** 62), 2 ** 62


def bind_to_gpu_numa_node(device: int) -> dict:
    """Pin this process (and with it the pages of whatever it allocates next: page-locked staging buffers are placed on the
    node of the thread that touches them first) to the CPU cores NVML lists as local to GPU `device`.  `torchrun` starts
    all ranks with the same affinity, so on a two-socket box every rank's host buffers land on one socket and the ranks
    on the other socket's GPUs copy across the inter-socket link: round 1 measured 14 GB/s per GPU of PCIe at 8 ranks
    against 41 GB/s alone.  Call before allocating host buffers.  Returns what was done (never raises)."""
    import os
    out = {"device": int(device), "bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        # honour CUDA_VISIBLE_DEVICES: NVML enumerates physical devices
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[device]) if visible and all(v.strip().isdigit() for v in visible.split(",")) else device
        handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            out.update(bound=True, cpus=len(cpus), first_cpu=min(cpus))
        else:
            out.update(cpus=len(cpus), note="NVML's local cores are all the allowed cores (one NUMA node, or a restricted cpuset)")
        try:
            out["numa_node"] = int(pynvml.nvmlDeviceGetNumaNodeId(handle))
        except Exception:
            pass
    except Exception as e:  # no NVML, no permission: run unbound
        out["error"] = f"{type(e).__name__}: {e}"
    return out


def rows_of(pos: np.ndarray, diameter: float) -> np.ndarray:
    """floor(y / d), the reference's strip index (collision_detector.py:126)."""
    return np.floor(np.asarray(pos)[:, 1] / diameter).astype(np.int64)


def partition_rows(rows: np.ndarray, nranks: int, halo_rows: int = HALO_ROWS) -> list[int]:
    """Row cuts [c_0 = -inf, c_1, ..., c_n = +inf] giving every rank about len(rows) / nranks particles, strips at
    least 2 * halo_rows high."""
    if nranks == 1:
        return [INT64_MIN, INT64_MAX]
    lo = int(rows.min())
    return partition_histogram(np.bincount(rows - lo), lo, nranks, halo_rows)


def cuts_from_histogram(hist: np.ndarray, row0: int, nranks: int, halo_rows: int = HALO_ROWS) -> list[int]:
    """Equal-weight cuts from a per-row histogram (`hist[k]` = weight of row `row0 + k`): cut k is the row after the
    one where the cumulative weight reaches k / nranks of the total, and at least 2 * halo_rows above the previous cut.
    The first cut's floor is `row0 + 2 * halo_rows`, so the histogram is used as given: trimming its empty end rows
    would move that floor."""
    if nranks == 1:
        return [INT64_MIN, INT64_MAX]
    cum = np.cumsum(hist.astype(np.int64))
    cuts = [INT64_MIN]
    prev = row0
    for k in range(1, nranks):
        r = row0 + int(np.searchsorted(cum, cum[-1] * k / nranks, side="left")) + 1
        r = max(r, prev + 2 * halo_rows)
        cuts.append(r)
        prev = r
    cuts.append(INT64_MAX)
    return cuts


def partition_histogram(hist: np.ndarray, row0: int, nranks: int, halo_rows: int = HALO_ROWS) -> list[int]:
    """`cuts_from_histogram` over the occupied rows of `hist` (`hist[k]` = particles in row `row0 + k`); raises if
    they are too few for nranks strips of at least 2 * halo_rows rows."""
    nz = np.nonzero(hist)[0]
    lo, hi = row0 + int(nz[0]), row0 + int(nz[-1])
    cuts = cuts_from_histogram(hist[nz[0]:nz[-1] + 1], lo, nranks, halo_rows)
    if nranks > 1 and cuts[-2] + 2 * halo_rows > hi + 1:
        raise ValueError(f"scene has too few cell rows ({hi - lo + 1}) for {nranks} strips of >= {2 * halo_rows} rows")
    return cuts


def world_rows(particle_radius: float) -> tuple[int, int]:
    """(first row, number of rows) covering every position a live particle can have (crate.py:152: -r <= y <= 1 + r,
    plus the wall fix's shift of < r)."""
    d = 2 * particle_radius
    row0 = int(np.floor(-2 * particle_radius / d)) - 1
    return row0, int(np.floor((1 + 2 * particle_radius) / d)) + 2 - row0


def next_rebalance_interval(every: int, shift: int, first: int, floor: int = 1) -> int:
    """The re-cut interval after a re-cut that asked the cuts to move by at most `shift` rows: halved (not below
    min(25, first)) when the partition was found far off (> 8 rows), doubled when it was found in place (<= 2 rows);
    then raised to `floor` - the interval at which the measured idle time of a re-cut is 2 % of the ticks between two
    re-cuts - and capped at max(1000, first), `first` being the interval the caller started with."""
    hi = max(1000, first)
    if shift > 8:
        new = max(every // 2, min(25, first))
    elif shift <= 2:
        new = min(every * 2, hi)
    else:
        new = every
    return min(max(new, floor), hi)


class StripDomain:
    """One rank's share of a strip-decomposed scene.

    `world` is a WorldConfig (closed scenes: no particle sources).  The initial scene comes either as `pos` / `vel`
    (the WHOLE scene, every rank generates it from the same seed and keeps its rows) or as `chunks` (a callable returning
    an iterator of (first row index, positions): `scenes.scene_chunks`; velocities zero) - the form the 16M / 64M scenes
    use, so that no rank ever holds the whole scene.  uids are the global row indices of the scene.

    Restrictions of the strip mode (they hold for the synthetic multi-GPU configs): closed scenes, fixed walls,
    counter or no noise."""

    def __init__(self, world, pos=None, vel=None, *, rank: int, world_size: int, precision: str = "mixed",
                 noise: str = "counter", noise_seed: int = 0, device: int = 0, stream: int | None = None,
                 halo_rows: int = HALO_ROWS, slack: float = 1.3, wire_capacity: int | None = None,
                 context_factory=None, tensor_device=None, comm=None, transport: str = "nccl",
                 rebalance_every: int = 0, cuts: list | None = None, chunks=None, check_every: int = 256,
                 adaptive_rebalance: bool = True):
        import torch

        if world.particle_sources:
            raise ValueError("strip decomposition supports closed scenes only (no particle sources)")
        if noise == "reference":
            raise ValueError("the reference-RNG noise mode is single-GPU only")
        self.rank, self.world_size = rank, world_size
        self.world = world
        self.halo_rows = halo_rows
        c = world.coefficients
        self.diameter = 2 * c["particle_radius"]
        self._row0, self._nrows = world_rows(c["particle_radius"])
        if chunks is None:
            whole_pos, whole_vel = np.asarray(pos, dtype=np.float64), np.asarray(vel, dtype=np.float64)
            chunks = lambda: iter([(0, whole_pos)])  # noqa: E731
        else:
            whole_vel = None
        # pass 1: per-row histogram of the whole scene -> equal-count cuts, capacities
        hist = np.zeros(self._nrows, np.int64)
        n_total = 0
        for _, p in chunks():
            r = np.clip(rows_of(p, self.diameter) - self._row0, 0, self._nrows - 1)
            hist += np.bincount(r, minlength=self._nrows)
            n_total += len(p)
        self.cuts = list(cuts) if cuts is not None else partition_histogram(hist, self._row0, world_size, halo_rows)
        assert len(self.cuts) == world_size + 1
        self.row_lo, self.row_hi = self.cuts[rank], self.cuts[rank + 1]
        # pass 2: this rank's rows
        keep_uid, keep_pos, keep_vel = [], [], []
        for i0, p in chunks():
            r = rows_of(p, self.diameter)
            m = np.nonzero((r >= self.row_lo) & (r < self.row_hi))[0]
            keep_uid.append((m + i0).astype(np.uint32))
            keep_pos.append(p[m])
            keep_vel.append(whole_vel[m + i0] if whole_vel is not None else np.zeros((len(m), 2)))
        mine = np.concatenate(keep_uid)
        pos_mine, vel_mine = np.concatenate(keep_pos), np.concatenate(keep_vel)
        del keep_uid, keep_pos, keep_vel
        self.n_total = n_total
        per_row = max(int(hist.max()), 1)
        self.wire_capacity = int(wire_capacity or max(4 * (halo_rows + 2) * per_row, 1024))
        # room for this rank's share after re-balancing as well as for an unbalanced start
        capacity = int(max(len(mine), -(-n_total // world_size)) * slack) + 2 * self.wire_capacity + 1024
        self.wire_capacity = min(self.wire_capacity, capacity)
        self._torch_stream = None
        if context_factory is None:
            # The context launches on ONE stream and everything torch does for this domain (wire-buffer allocation,
            # NCCL send / recv, the re-cut all-reduce) must be ordered against it.  So the domain owns the choice: a
            # caller's stream handle is wrapped, otherwise a torch stream is created; exchange() runs under it.
            # (Handle 0 / None used to make the library open a private stream that NCCL never saw: stale halos.)
            if stream:
                self._torch_stream = torch.cuda.ExternalStream(int(stream), device=torch.device("cuda", device))
            else:
                self._torch_stream = torch.cuda.Stream(device=torch.device("cuda", device))
                stream = self._torch_stream.cuda_stream
            if not stream:
                raise ValueError("strip decomposition needs a non-default CUDA stream")
        factory = context_factory or _lib.Context
        prec = {"f64": _lib.PRECISION_F64, "mixed": _lib.PRECISION_MIXED}[precision]
        self.ctx = factory(capacity, prec, device, stream)
        self.ctx.set_params(dt=c["dt"], particle_radius=c["particle_radius"],
                            wall_collision_decay=c["wall_collision_decay"],
                            pressure_amplifier=c["pressure_amplifier"], ignored_pressure=c["ignored_pressure"],
                            collider_noise_level=c["collider_noise_level"], viscosity=c["viscosity"],
                            surface_smoothing=c["surface_smoothing"], target_pressure=c["target_pressure"],
                            gravity_x=c["gravity"][0], gravity_y=c["gravity"][1])
        from .rigid_body import build_rigid_bodies
        bodies = build_rigid_bodies(world.rigid_bodies)
        if any(b.kind != "fixed" for b in bodies):
            raise ValueError("strip decomposition supports fixed walls only")
        seg = np.vstack([b.segments for b in bodies]) if bodies else np.zeros((0, 2, 2))
        self.ctx.set_walls(seg, [len(b) for b in bodies], np.array([b.kinematics() for b in bodies]).reshape(-1, 5))
        self.ctx.set_noise({"counter": _lib.NOISE_COUNTER, "none": _lib.NOISE_NONE}[noise], noise_seed)
        self.ctx.set_state_uids(pos_mine, vel_mine, mine)
        del pos_mine, vel_mine, mine
        self.ctx.dist_configure(rank, world_size, self.row_lo, self.row_hi, halo_rows, self.wire_capacity)
        self._push_reach()
        self.tick = 0
        # re-balancing: every `rebalance_every` ticks the per-row histogram is summed over the ranks (the scheme's
        # only collective) and the cuts then SLIDE towards the new equal-count positions by at most halo - 2 rows per
        # tick, so the rows a cut hands over travel as ordinary migrants (DESIGN.md section 6)
        self.rebalance_every = int(rebalance_every)
        self.adaptive_rebalance = bool(adaptive_rebalance)   # False: re-cut every `rebalance_every` ticks exactly
        self.rebalance_log: list = []          # (tick, largest cut shift asked for, interval chosen) per re-cut
        self._next_rebalance = self._rebalance_first = self.rebalance_every
        self._recut_tick, self._recut_end, self._recut_idle_us = 0, time.perf_counter(), 0.0
        self.check_every = int(check_every)   # poll the device's overflow / too_far flags this often (synchronises)
        self.target_cuts = list(self.cuts)
        self.max_cut_shift = max(halo_rows - 2, 1)
        self._tensor_device = tensor_device

        nbytes = _lib.wire_bytes(self.wire_capacity) if context_factory is None else 16 + 40 * self.wire_capacity
        dev = tensor_device if tensor_device is not None else torch.device("cuda", device)
        self.has_lo, self.has_hi = rank > 0, rank < world_size - 1
        with self._on_stream():
            mk = lambda: torch.zeros(nbytes, dtype=torch.uint8, device=dev)  # noqa: E731
            self.send_lo, self.recv_lo = (mk(), mk()) if self.has_lo else (None, None)
            self.send_hi, self.recv_hi = (mk(), mk()) if self.has_hi else (None, None)
        self._comm = comm  # torch.distributed module or a test double with batch_isend_irecv / P2POp / isend / irecv
        if transport not in ("nccl", "p2p", "auto"):
            raise ValueError("transport must be 'nccl', 'p2p' or 'auto'")
        self.transport = transport
        self._symm = None
        if transport in ("p2p", "auto") and world_size > 1 and context_factory is None:
            try:
                with self._on_stream():
                    self._setup_p2p(nbytes, dev)
                ok = 1
            except Exception:  # no peer access / no symmetric memory on this box
                if transport == "p2p":
                    raise
                ok = 0
            if transport == "auto":  # every rank must take the same path
                import torch.distributed as dist
                flag = torch.tensor([ok], device=dev, dtype=torch.int32)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if int(flag.item()) == 0:
                    self._symm = None
                self.transport = "p2p" if self._symm is not None else "nccl"
        elif transport == "auto":
            self.transport = "nccl"

    def _push_reach(self) -> None:
        """A migrant is handed to the adjacent rank only: tell the device where that rank's strip ends."""
        if hasattr(self.ctx, "dist_set_reach") and self.world_size > 1:
            self.ctx.dist_set_reach(self.cuts[max(self.rank - 1, 0)], self.cuts[min(self.rank + 2, self.world_size)])

    def _on_stream(self):
        """Context manager: torch work issued inside is ordered on the context's launch stream."""
        import contextlib
        import torch
        if self._torch_stream is None:
            return contextlib.nullcontext()
        return torch.cuda.stream(self._torch_stream)

    # ---- direct NVLink transport (torch symmetric memory): peer stores + stream signals, no NCCL call per tick ----
    def _setup_p2p(self, nbytes: int, dev) -> None:
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        slot = (nbytes + 255) // 256 * 256
        # layout: 256 bytes of flags, then [parity 0: from-lo | from-hi][parity 1: from-lo | from-hi]; double buffered
        # so that a neighbor one tick ahead never overwrites records this rank has not unpacked yet.
        # flag word (parity, side) at byte 64 * (2 * parity + side): last tick whose records have fully arrived.
        self._symm_buf = symm_mem.empty(256 + 4 * slot, dtype=torch.uint8, device=dev)
        self._symm_buf.zero_()
        self._symm = symm_mem.rendezvous(self._symm_buf, dist.group.WORLD.group_name)
        self._slot = slot
        self._peer = [int(p) for p in self._symm.buffer_ptrs]
        torch.cuda.synchronize()
        self._symm.barrier(channel=0)

    def _exchange_p2p(self) -> None:
        par = self.tick & 1
        data = 256 + 2 * par * self._slot
        value = self.tick + 1
        lo = hi = None
        # my lower neighbor receives "from hi" (side 1), my upper neighbor receives "from lo" (side 0)
        if self.has_lo:
            peer = self._peer[self.rank - 1]
            lo = (self.send_lo, peer + data + self._slot, peer + 64 * (2 * par + 1))
        if self.has_hi:
            peer = self._peer[self.rank + 1]
            hi = (self.send_hi, peer + data, peer + 64 * (2 * par))
        self.ctx.dist_pack_push(lo, hi, value)   # pack and NVLink transfer are one kernel
        mine = self._peer[self.rank]
        self.ctx.dist_unpack_flagged((mine + data, mine + 64 * (2 * par)) if self.has_lo else None,
                                     (mine + data + self._slot, mine + 64 * (2 * par + 1)) if self.has_hi else None,
                                     value)

    # ---- one tick ----------------------------------------------------------------------------------------------
    def exchange(self) -> None:
        """The only communication of a tick: the two wire buffers, whole, to and from the y-neighbors."""
        if self.world_size == 1:
            return
        import torch.distributed as dist
        d = self._comm or dist
        ops = []
        if self.has_lo:
            ops.append(d.P2POp(d.isend, self.send_lo, self.rank - 1))
            ops.append(d.P2POp(d.irecv, self.recv_lo, self.rank - 1))
        if self.has_hi:
            ops.append(d.P2POp(d.isend, self.send_hi, self.rank + 1))
            ops.append(d.P2POp(d.irecv, self.recv_hi, self.rank + 1))
        with self._on_stream():  # NCCL orders against torch's CURRENT stream: make that the context's launch stream
            for req in d.batch_isend_irecv(ops):
                req.wait()  # NCCL: the launch stream waits, the host does not

    # ---- re-balancing -------------------------------------------------------------------------------------------
    def rebalance(self) -> None:
        """Collective (every rank, same tick): new equal-WORK target cuts from the global row histogram, and a new
        re-cut interval.  How often to re-cut depends on how fast the scene's work distribution moves: a settled box
        needs it almost never, the collapsing 64M column every few dozen ticks (its dense bottom layer thickens, and
        the strip above it overloads within a couple of hundred ticks) - and on what a re-cut costs: it drains the
        stream, so the device idles while the host reduces the histogram.  The interval therefore adapts
        (next_rebalance_interval): halved when the new targets are more than 8 rows from the current cuts, doubled when
        they are within 2, and never shorter than what keeps the measured idle time of a re-cut under 2 % of the
        measured tick time.  The two measurements ride in the same all-reduce as the histogram (as rank means), so every
        rank takes the same decision."""
        import time
        import torch
        import torch.distributed as dist
        hist = self.ctx.dist_row_histogram(self._row0, self._nrows).astype(np.int64)
        t_drained = time.perf_counter()          # the stream is empty here: every tick since the last re-cut has run
        ticks = self.tick - self._recut_tick
        tick_us = (t_drained - self._recut_end) / max(ticks, 1) * 1e6
        dev = self._tensor_device if self._tensor_device is not None else torch.device("cuda", self.ctx.device)
        with self._on_stream():
            t = torch.from_numpy(np.concatenate([hist, [int(self._recut_idle_us), int(tick_us)]]).astype(np.int64)).to(dev)
            dist.all_reduce(t)
            t = t.cpu().numpy()
        idle_us, tick_us = t[-2] / self.world_size, t[-1] / self.world_size
        self.target_cuts = cuts_from_histogram(t[:-2], self._row0, self.world_size, self.halo_rows)
        shift = max((abs(a - b) for a, b in zip(self.target_cuts[1:-1], self.cuts[1:-1])), default=0)
        if self.adaptive_rebalance:
            floor = int(np.ceil(idle_us / (0.02 * tick_us))) if tick_us > 0 else 1
            self.rebalance_every = next_rebalance_interval(self.rebalance_every, shift, self._rebalance_first, floor)
        self._next_rebalance = self.tick + self.rebalance_every
        self._recut_tick, self._recut_end = self.tick, time.perf_counter()
        self._recut_idle_us = (self._recut_end - t_drained) * 1e6
        self.rebalance_log.append((self.tick, int(shift), int(self.rebalance_every), round(self._recut_idle_us),
                                   round(float(tick_us), 1)))

    def _slide_cuts(self) -> None:
        """Every rank holds the whole cut list and moves it identically; no communication."""
        new = list(self.cuts)
        for k in range(1, self.world_size):
            delta = self.target_cuts[k] - new[k]
            new[k] += max(-self.max_cut_shift, min(self.max_cut_shift, delta))
        for k in range(1, self.world_size):  # never squeeze an interior strip below two halos
            if k >= 2 and new[k] - new[k - 1] < 2 * self.halo_rows:
                new[k] = new[k - 1] + 2 * self.halo_rows
        if new != self.cuts:
            self.cuts = new
            self.row_lo, self.row_hi = new[self.rank], new[self.rank + 1]
            self.ctx.dist_set_rows(self.row_lo, self.row_hi)
            self._push_reach()

    def physics_tick(self) -> None:
        self.ctx.set_tick(self.tick)
        if self.world_size > 1:
            if self.rebalance_every and self.tick and self.tick >= self._next_rebalance:
                self.rebalance()
            if self.cuts != self.target_cuts:
                self._slide_cuts()
            if self._symm is not None:
                self._exchange_p2p()
            else:
                self.ctx.dist_pack(self.send_lo, self.send_hi)
                self.exchange()
                self.ctx.dist_unpack(self.recv_lo, self.recv_hi)
        self.ctx.step()
        self.tick += 1
        if self.check_every and self.world_size > 1 and self.tick % self.check_every == 0:
            self._check_flags()

    def _check_flags(self) -> None:
        """Raise if the device has flagged a capacity overflow or a particle that outran the halo (results after such
        a tick are wrong; the arrays themselves stay in bounds: the live count is clamped to the capacity)."""
        st = self.status()
        if st["overflow"] or st["too_far"]:
            raise _lib.SandCrateError(f"strip {self.rank}: device flags {st} at tick {self.tick} (raise `slack` / "
                                      f"`wire_capacity`, or `halo_rows` if particles move more than a halo per tick)")

    def step(self, n: int = 1) -> None:
        for _ in range(n):
            self.physics_tick()

    # ---- readback ----------------------------------------------------------------------------------------------
    def owned(self):
        """(uid, pos, vel) of this rank's particles, sorted by uid."""
        if self.world_size == 1:
            pos, vel, _ = self.ctx.get_state(want_pressure=False)
            return self.ctx.get_uids(), pos, vel
        pos, vel, uid = self.ctx.dist_get_owned()
        order = np.argsort(uid, kind="stable")
        return uid[order], pos[order], vel[order]

    def status(self) -> dict:
        if self.world_size == 1:
            return {"overflow": False, "too_far": False, "n_local": self.ctx.particle_count()}
        return self.ctx.dist_status(self.send_lo, self.send_hi)

    def gather(self):
        """All ranks' particles on every rank, sorted by uid: the global state in the reference's row order."""
        uid, pos, vel = self.owned()
        if self.world_size == 1:
            return uid, pos, vel
        import torch.distributed as dist
        parts = [None] * self.world_size
        dist.all_gather_object(parts, (uid, pos, vel))
        uid = np.concatenate([p[0] for p in parts])
        pos = np.concatenate([p[1] for p in parts])
        vel = np.concatenate([p[2] for p in parts])
        order = np.argsort(uid, kind="stable")
        return uid[order], pos[order], vel[order]

    def close(self) -> None:
        self.ctx.close()

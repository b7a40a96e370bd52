"""Strip decomposition on ONE GPU: N strips of a scene as N contexts in one process, stepped in lockstep on one stream.

tests/test_strips.py proves the per-tick protocol on the CPU (gloo, the oracle-backed context); the multi-GPU checks
need two or more GPUs.  Here the device side runs on any GPU machine: the pack kernel (k_dist_pack, both transports),
the unpacking pre-pass (k_prepass<true, true>), the owned readback, the re-cut histogram and sc_dist_set_rows, over
many ticks, against a single context of the whole scene and against the oracle.  The pack kernel's records are also
compared with a NumPy restatement of its rule (sc_dist.cuh), and the wire buffers' overflow / too_far flags are driven
on a raw context.

The lockstep driver runs the phases of StripDomain.physics_tick, each over every rank before the next.  All contexts
launch on the SAME stream, so the program order of the host calls is the device order: the exchange is a plain copy
between two ranks' buffers (or, for the direct transport, the pack kernel's own stores into the neighbor's receive
slot), with nothing to wait for across streams.  The driver itself is first run on the oracle-backed context on the
CPU, so a failure on the GPU is in the library, not in the driver."""
import functools

import numpy as np
import pytest
import torch

from oracle import oracle as O
from oracle_backend import OracleContext
from sand_crate_b200 import _lib
from sand_crate_b200.scenes import box_fill, dam_break
from sand_crate_b200.strips import HALO_ROWS, StripDomain, cuts_from_histogram, partition_rows, rows_of

SEED = 5            # counter-noise seed of every run here (tests/mgpu_check.py's)
MIGRANT, HALO = 0, 1  # WireRec.kind (SC_WIRE_MIGRANT, SC_WIRE_HALO)
REC = np.dtype([("px", "f8"), ("py", "f8"), ("vx", "f8"), ("vy", "f8"), ("uid", "u4"), ("kind", "u4")])


# ---- scenes ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _scene(maker, n):
    """A scene with a fast random velocity of 0.3 diameters per tick added, so that rows change hands every tick."""
    world, pos, vel = maker(n)
    c = world.coefficients
    d = 2 * c["particle_radius"]
    vel = vel + np.random.RandomState(3).randn(*vel.shape) * (d / c["dt"]) * 0.3
    return world, pos, vel


def _wrong_cuts(world, pos, nranks):
    """The equal-count cuts of ANOTHER scene (the column 0.1 lower): far from balanced here, the re-cutter must move
    them (tests/mgpu_check.py, case 3)."""
    shifted = pos.copy()
    shifted[:, 1] -= 0.1
    return partition_rows(rows_of(shifted, 2 * world.coefficients["particle_radius"]), nranks)


def _coeff_vec(c):
    return np.array([c["dt"], c["particle_radius"], c["wall_collision_decay"], c["pressure_amplifier"],
                     c["ignored_pressure"], c["collider_noise_level"], c["viscosity"], c["surface_smoothing"],
                     c["target_pressure"], c["gravity"][0], c["gravity"][1]], dtype=np.float64)


def _oracle_run(world, pos, vel, ticks):
    """The same ticks on the whole scene in the oracle: (uid, pos, vel) in uid order."""
    c = world.coefficients
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    cv = _coeff_vec(c)
    uid = np.arange(len(pos), dtype=np.uint32)
    for tick in range(ticks):
        pos, vel, mask = O.remove_particles(pos, vel, c["particle_radius"])
        uid = uid[~mask]
        out = O.step(cv, pos, vel, seg, [len(seg)], np.zeros((1, 5)), noise_mode=1, tkey=O.tick_key(SEED, tick),
                     uid=uid, want_all=False)
        pos, vel = out["pos_out"], out["vel_out"]
    return uid, pos, vel


@functools.lru_cache(maxsize=None)
def _oracle_cached(maker, n, ticks):
    return _oracle_run(*_scene(maker, n), ticks)


@functools.lru_cache(maxsize=None)
def _single_context(maker, n, ticks, precision):
    """The same ticks on the whole scene in ONE context on this GPU (world_size 1): (uid, pos, vel) in uid order."""
    world, pos, vel = _scene(maker, n)
    stream = torch.cuda.Stream()
    dom = StripDomain(world, pos, vel, rank=0, world_size=1, precision=precision, noise="counter", noise_seed=SEED,
                      stream=stream.cuda_stream)
    try:
        dom.step(ticks)
        uid, p, v = dom.owned()
    finally:
        dom.close()
    order = np.argsort(uid, kind="stable")
    return uid[order], p[order], v[order]


# ---- the lockstep driver --------------------------------------------------------------------------------------------
class Lockstep:
    """N StripDomains of one scene in one process.  One tick = the phases of StripDomain.physics_tick, each over every
    rank before the next: set_tick, re-cut (the rank histograms summed here instead of all-reduced), slide the cuts,
    pack, exchange, unpack, step.  Only where the communication happens differs from physics_tick.

    GPU: every context launches on one torch stream, and the exchange copies are issued on it (`_on_stream`).
    `direct=True`: the direct transport - each rank has a receive buffer with two slots (from the lower / upper
    neighbor) and two flag words; the pack kernel writes its records into the neighbor's slot and raises the flag, the
    unpacking pre-pass waits for it.  Before any step is enqueued the driver synchronises and checks every flag on the
    host, so a pack that failed to raise one fails the test instead of leaving a pre-pass spinning.
    `oracle=True`: OracleContext on CPU tensors (copy exchange only)."""

    def __init__(self, world, pos, vel, nranks, *, precision="f64", direct=False, rebalance_every=0, cuts=None,
                 oracle=False):
        if oracle:
            assert not direct
            kw = dict(context_factory=OracleContext, tensor_device=torch.device("cpu"))
            self.stream = None
        else:
            self.stream = torch.cuda.Stream()
            kw = dict(stream=self.stream.cuda_stream)
        self.n, self.t, self.every = nranks, 0, rebalance_every
        self.doms = []
        for k in range(nranks):
            self.doms.append(StripDomain(world, pos, vel, rank=k, world_size=nranks, precision=precision,
                                         noise="counter", noise_seed=SEED, rebalance_every=rebalance_every, cuts=cuts,
                                         adaptive_rebalance=False, check_every=0, **kw))
        self.cap = self.doms[0].wire_capacity
        assert all(d.wire_capacity == self.cap for d in self.doms), "the ranks' wire buffers must have one size"
        self.recuts = 0
        self.direct = direct
        if direct:
            self.slot = (_lib.wire_bytes(self.cap) + 15) // 16 * 16
            with self._on_stream():
                self.inbox = [torch.zeros(2 * self.slot + 16, dtype=torch.uint8, device="cuda") for _ in self.doms]

    def _on_stream(self):
        return self.doms[0]._on_stream()   # one stream for all of them

    # direct transport: rank k's receive slot / flag word for records from its lower (side 0) or upper (side 1) neighbor
    def _slot(self, k, side):
        return self.inbox[k].data_ptr() + side * self.slot

    def _flag(self, k, side):
        return self.inbox[k].data_ptr() + 2 * self.slot + 8 * side

    # ---- the phases of one tick ----
    def begin(self):
        t = self.t
        for d in self.doms:
            d.ctx.set_tick(t)
        if self.every and t and t % self.every == 0:   # StripDomain.rebalance without the all-reduce
            d0 = self.doms[0]
            hist = sum(d.ctx.dist_row_histogram(d._row0, d._nrows).astype(np.int64) for d in self.doms)
            target = cuts_from_histogram(hist, d0._row0, self.n, d0.halo_rows)
            for d in self.doms:
                d.target_cuts = list(target)
            self.recuts += 1
        for d in self.doms:
            if d.cuts != d.target_cuts:
                d._slide_cuts()
        assert all(d.cuts == self.doms[0].cuts for d in self.doms)

    def pack(self):
        if not self.direct:
            for d in self.doms:
                d.ctx.dist_pack(d.send_lo, d.send_hi)
            return
        value = self.t + 1
        for k, d in enumerate(self.doms):
            lo = (d.send_lo, self._slot(k - 1, 1), self._flag(k - 1, 1)) if d.has_lo else None
            hi = (d.send_hi, self._slot(k + 1, 0), self._flag(k + 1, 0)) if d.has_hi else None
            d.ctx.dist_pack_push(lo, hi, value=value)

    def exchange(self):
        if self.direct:   # the records are already there: check every flag before anything waits on one
            self.stream.synchronize()
            for k, d in enumerate(self.doms):
                with self._on_stream():
                    words = self.inbox[k][2 * self.slot:].cpu().numpy().view(np.uint32)
                flags = [int(words[0]) if d.has_lo else None, int(words[2]) if d.has_hi else None]
                want = [self.t + 1 if d.has_lo else None, self.t + 1 if d.has_hi else None]
                assert flags == want, f"tick {self.t}: rank {k}'s receive flags are {flags}, expected {want}"
            return
        with self._on_stream():
            for k in range(self.n - 1):
                a, b = self.doms[k], self.doms[k + 1]
                b.recv_lo.copy_(a.send_hi)
                a.recv_hi.copy_(b.send_lo)

    def unpack(self):
        for k, d in enumerate(self.doms):
            if self.direct:
                d.ctx.dist_unpack_flagged((self._slot(k, 0), self._flag(k, 0)) if d.has_lo else None,
                                          (self._slot(k, 1), self._flag(k, 1)) if d.has_hi else None, self.t + 1)
            else:
                d.ctx.dist_unpack(d.recv_lo, d.recv_hi)

    def step(self):
        for d in self.doms:
            d.ctx.step()
            d.tick += 1
        self.t += 1

    def tick(self):
        self.begin()
        self.pack()
        self.exchange()
        self.unpack()
        self.step()

    def run(self, ticks):
        for _ in range(ticks):
            self.tick()

    # ---- readback ----
    def gather(self):
        """(uid, pos, vel, owner rank) of every rank's owned particles in uid order; no uid may be owned twice."""
        parts = [d.owned() for d in self.doms]
        uid = np.concatenate([p[0] for p in parts])
        pos = np.concatenate([p[1] for p in parts])
        vel = np.concatenate([p[2] for p in parts])
        owner = np.concatenate([np.full(len(p[0]), k) for k, p in enumerate(parts)])
        order = np.argsort(uid, kind="stable")
        uid, pos, vel, owner = uid[order], pos[order], vel[order], owner[order]
        dup = uid[1:][uid[1:] == uid[:-1]]
        assert len(dup) == 0, f"{len(dup)} uids owned twice, e.g. {dup[:5].tolist()}"
        return uid, pos, vel, owner

    def status(self):
        return [d.status() for d in self.doms]

    def close(self):
        for d in self.doms:
            d.close()


def _assert_same_particles(got_uid, got_pos, got_vel, uid, pos, vel, what, bitwise=True):
    missing, extra = np.setdiff1d(uid, got_uid), np.setdiff1d(got_uid, uid)
    assert len(missing) == 0 and len(extra) == 0, \
        f"{what}: {len(missing)} uids missing (e.g. {missing[:5].tolist()}), {len(extra)} extra"
    assert np.array_equal(got_uid, uid)
    if bitwise:   # the same kernels on the same inputs: the same bits, signed zeros included
        same_p = got_pos.view(np.uint64) == pos.view(np.uint64)
        same_v = got_vel.view(np.uint64) == vel.view(np.uint64)
    else:
        same_p, same_v = got_pos == pos, got_vel == vel
    bad = np.nonzero(~(same_p.all(1) & same_v.all(1)))[0]
    assert len(bad) == 0, (f"{what}: {len(bad)} of {len(uid)} particles differ, e.g. uid {uid[bad[:5]].tolist()}, "
                           f"max |dpos| {np.abs(got_pos - pos).max():.3e}, max |dvel| {np.abs(got_vel - vel).max():.3e}")


def _assert_exchange_happened(start_owner, uid, owner, nranks, both_ways=True):
    """Some uid changed owner; with 3+ strips and fixed cuts an interior rank gained particles from BOTH neighbors
    (while cuts slide, the rows they hand over travel one way and may outweigh the rest)."""
    before = start_owner[uid]
    assert (before != owner).any(), "no particle changed owner: the run did not exercise migration"
    if nranks >= 3 and both_ways:
        both = [k for k in range(1, nranks - 1)
                if ((owner == k) & (before == k - 1)).any() and ((owner == k) & (before == k + 1)).any()]
        assert both, "no interior rank received migrants from both of its neighbors"


def _owner_map(ls, n_total):
    owner = np.full(n_total, -1, np.int64)
    for k, d in enumerate(ls.doms):
        owner[d.owned()[0]] = k
    assert (owner >= 0).all()
    return owner


# ---- 1. the driver, proved on the CPU (oracle-backed contexts, no GPU) ----------------------------------------------
@pytest.mark.parametrize("nranks,recut", [(2, 0), (3, 0), (3, 3)])
def test_lockstep_driver_on_the_oracle_matches_one_domain(nranks, recut):
    """The lockstep driver with OracleContext: 2 and 3 strips with fixed cuts, and 3 strips started from wrong cuts and
    re-cut every 3 ticks.  The gathered state must be the single-domain oracle run's, bit for bit."""
    n, ticks = 6000, 7
    world, pos, vel = _scene(dam_break, n)
    cuts = _wrong_cuts(world, pos, nranks) if recut else None
    ls = Lockstep(world, pos, vel, nranks, rebalance_every=recut, cuts=cuts, oracle=True)
    start = _owner_map(ls, n)
    cuts0 = list(ls.doms[0].cuts)
    ls.run(ticks)
    uid, p, v, owner = ls.gather()
    st = ls.status()
    ls.close()
    _assert_same_particles(uid, p, v, *_oracle_run(world, pos, vel, ticks), "lockstep oracle strips vs one domain")
    assert not any(s["too_far"] for s in st)
    _assert_exchange_happened(start, uid, owner, nranks, both_ways=not recut)
    if recut:
        assert ls.recuts == 2 and ls.doms[0].cuts != cuts0, "the cuts must have moved"


# ---- 2. whole-run parity on the device ------------------------------------------------------------------------------
CASES = [  # maker, n, ticks, strips, precision, transport, re-cut interval
    pytest.param(dam_break, 200_000, 12, 2, "f64", "copy", 0, id="dam_break-2-f64-copy"),
    pytest.param(dam_break, 200_000, 12, 3, "f64", "copy", 0, id="dam_break-3-f64-copy"),
    pytest.param(box_fill, 300_000, 8, 4, "f64", "copy", 0, id="box_fill-4-f64-copy"),
    pytest.param(dam_break, 200_000, 12, 3, "mixed", "copy", 0, id="dam_break-3-mixed-copy"),
    pytest.param(dam_break, 200_000, 16, 3, "f64", "copy", 3, id="dam_break-3-f64-copy-recut3"),
    pytest.param(dam_break, 200_000, 12, 3, "f64", "direct", 0, id="dam_break-3-f64-direct"),
    pytest.param(dam_break, 200_000, 12, 3, "mixed", "direct", 0, id="dam_break-3-mixed-direct"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("maker,n,ticks,nranks,precision,transport,recut", CASES)
def test_lockstep_strips_bit_identical_to_one_context(maker, n, ticks, nranks, precision, transport, recut):
    """N strips on one GPU against one context of the whole scene: the same uids, positions and velocities, bit for
    bit; the fp64 dam break without re-cuts also against the oracle.  No rank may flag an overflow or a particle that
    outran the halo, and particles must actually have changed hands."""
    world, pos, vel = _scene(maker, n)
    cuts = _wrong_cuts(world, pos, nranks) if recut else None
    ls = Lockstep(world, pos, vel, nranks, precision=precision, direct=transport == "direct",
                  rebalance_every=recut, cuts=cuts)
    try:
        start = _owner_map(ls, n)
        cuts0 = list(ls.doms[0].cuts)
        ls.run(ticks)
        uid, p, v, owner = ls.gather()
        st = ls.status()
        cuts1 = list(ls.doms[0].cuts)
    finally:
        ls.close()
    flagged = [(k, s) for k, s in enumerate(st) if s["overflow"] or s["too_far"]]
    assert not flagged, f"device flags raised: {flagged}"
    _assert_exchange_happened(start, uid, owner, nranks, both_ways=not recut)
    if recut:
        assert ls.recuts == (ticks - 1) // recut and cuts1 != cuts0, "the cuts must have moved"
    _assert_same_particles(uid, p, v, *_single_context(maker, n, ticks, precision),
                           f"{nranks} strips ({transport}) vs one context")
    if precision == "f64" and maker is dam_break and not recut:
        _assert_same_particles(uid, p, v, *_oracle_cached(maker, n, ticks), f"{nranks} strips vs the oracle",
                               bitwise=False)


# ---- 3. the pack kernel against a NumPy restatement of its rule -----------------------------------------------------
def _read_wire(buf, cap):
    """(header words [count, overflow, too_far, pad], the records stored) of a wire buffer on the device."""
    raw = buf.cpu().numpy()
    hdr = raw[:16].view(np.uint32).copy()
    stored = min(int(hdr[0]), cap)
    return hdr, raw[16:16 + REC.itemsize * stored].view(REC).copy()


def _records(pos, vel, uid, mask, kind):
    r = np.zeros(int(mask.sum()), REC)
    r["px"], r["py"], r["vx"], r["vy"] = pos[mask, 0], pos[mask, 1], vel[mask, 0], vel[mask, 1]
    r["uid"], r["kind"] = uid[mask], kind
    return r


def _predict_pack(pos, vel, uid, d, row_lo, row_hi, halo, has_lo, has_hi):
    """The records k_dist_pack must write for these owned particles (sc_dist.cuh): a particle whose row left the strip
    is a MIGRANT for that side's neighbor; an owned one within `halo` rows of a cut a HALO for that neighbor (both, in
    a strip two halos high)."""
    rows = rows_of(pos, d)
    below, above = (rows < row_lo) & has_lo, (rows >= row_hi) & has_hi
    own = ~(below | above)
    lo = np.concatenate([_records(pos, vel, uid, below, MIGRANT),
                         _records(pos, vel, uid, own & (rows < row_lo + halo), HALO)]) if has_lo else None
    hi = np.concatenate([_records(pos, vel, uid, above, MIGRANT),
                         _records(pos, vel, uid, own & (rows >= row_hi - halo), HALO)]) if has_hi else None
    return lo, hi


def _by_uid_kind(r):
    return r[np.lexsort((r["kind"], r["uid"]))]


def _assert_records(got_hdr, got, want, what):
    assert int(got_hdr[0]) == len(want), f"{what}: count {int(got_hdr[0])}, predicted {len(want)}"
    assert int(got_hdr[1]) == 0 and int(got_hdr[2]) == 0, f"{what}: overflow / too_far raised: {got_hdr.tolist()}"
    got, want = _by_uid_kind(got), _by_uid_kind(want)
    assert np.array_equal(got["uid"], want["uid"]) and np.array_equal(got["kind"], want["kind"]), \
        f"{what}: (uid, kind) differ: {len(np.setdiff1d(want['uid'], got['uid']))} predicted uids missing, " \
        f"{len(np.setdiff1d(got['uid'], want['uid']))} unexpected"
    assert got.tobytes() == want.tobytes(), f"{what}: positions / velocities differ from the owned state"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "mixed"])
def test_pack_records_follow_the_rule(precision):
    """3 strips in lockstep.  Before the pack of tick 0 (a pass over the whole arrays: no search state yet) and of
    tick 4 (only the two boundary zones of the last sort order), each rank's owned state is read back and the records
    its send buffers must hold are predicted from row = floor(y / d): count, flags and every record bit for bit.  After
    the step that follows, a rank no longer owns the migrants it sent - the neighbor does."""
    world, pos, vel = _scene(dam_break, 200_000)
    d = 2 * world.coefficients["particle_radius"]
    ls = Lockstep(world, pos, vel, 3, precision=precision)
    try:
        migrated = {}
        for t in range(6):
            ls.begin()
            check = t in (0, 4)
            if check:
                want = []
                for dom in ls.doms:
                    p, v, u = dom.ctx.dist_get_owned()
                    want.append(_predict_pack(p, v, u, d, dom.row_lo, dom.row_hi, dom.halo_rows, dom.has_lo,
                                              dom.has_hi))
            ls.pack()
            if check:
                sent = {}
                with ls._on_stream():
                    for k, dom in enumerate(ls.doms):
                        for side, buf, w in (("lo", dom.send_lo, want[k][0]), ("hi", dom.send_hi, want[k][1])):
                            if buf is None:
                                continue
                            hdr, got = _read_wire(buf, ls.cap)
                            _assert_records(hdr, got, w, f"tick {t}, rank {k}, {side} buffer")
                            sent[k, side] = got["uid"][got["kind"] == MIGRANT]
                # tick 0 starts from the strip's own rows: halos only.  Later the interior rank sends both ways.
                assert (sum(len(m) for m in sent.values()) == 0) == (t == 0)
                if t:
                    assert len(sent[1, "lo"]) and len(sent[1, "hi"]), "the interior rank must send migrants both ways"
            ls.exchange()
            ls.unpack()
            ls.step()
            if check:
                owned = [set(dom.ctx.dist_get_owned()[2].tolist()) for dom in ls.doms]
                for (k, side), m in sent.items():
                    to = k - 1 if side == "lo" else k + 1
                    m = set(m.tolist())
                    assert not (m & owned[k]), f"tick {t}: rank {k} still owns {len(m & owned[k])} of its migrants"
                    assert m <= owned[to], f"tick {t}: rank {to} does not own {len(m - owned[to])} migrants sent to it"
                    migrated[t] = migrated.get(t, 0) + len(m)
        assert migrated.get(4, 0) > 0
    finally:
        ls.close()


# ---- 4. the wire flags, on a raw context ----------------------------------------------------------------------------
def _strip_world():
    world, _, _ = dam_break(4000)
    return world, 2 * world.coefficients["particle_radius"]


def _raw_strip(world, pos, uid, wire_cap, row_lo, row_hi, rank=1, nranks=3):
    """A context holding `pos` (at rest) as strip `rank` of `nranks`, owning rows [row_lo, row_hi), default reach."""
    c = world.coefficients
    ctx = _lib.Context(len(pos) + 1024, _lib.PRECISION_F64)
    ctx.set_params(**{k: float(c[k]) for k in _lib.PARAM_FIELDS[:9]},
                   gravity_x=float(c["gravity"][0]), gravity_y=float(c["gravity"][1]))
    seg = np.array(world.rigid_bodies[0]["fixed"]["segments"], dtype=np.float64)
    ctx.set_walls(seg, [len(seg)], np.zeros((1, 5)))
    ctx.set_noise(_lib.NOISE_COUNTER, 3)
    ctx.set_state_uids(pos, np.zeros_like(pos), np.asarray(uid, np.uint32))
    ctx.dist_configure(rank, nranks, row_lo, row_hi, HALO_ROWS, wire_cap)
    return ctx


def _wire_pair(wire_cap, tail=0):
    """Two send buffers of `wire_cap` records, each followed by `tail` guard bytes of 0xA5."""
    bufs = []
    for _ in range(2):
        b = torch.full((_lib.wire_bytes(wire_cap) + tail,), 0xA5, dtype=torch.uint8, device="cuda")
        bufs.append(b)
    torch.cuda.synchronize()   # written on torch's stream, used on the context's
    return bufs


@pytest.mark.gpu
@pytest.mark.parametrize("side", ["lo", "hi"])
def test_pack_flags_a_migrant_beyond_the_reach(side):
    """The default reach of a strip is `halo` rows past each cut: a particle that left the strip by more than that
    would need a second hop, so the pack raises too_far.  Row row_hi + halo (row_lo - halo - 1) is the first row out of
    reach and must be flagged; row row_hi + halo - 1 (row_lo - halo), the last row in reach, must not."""
    world, d = _strip_world()
    row_lo, row_hi, h = 30, 50, HALO_ROWS
    far, near = (row_hi + h, row_hi + h - 1) if side == "hi" else (row_lo - h - 1, row_lo - h)
    for rows, too_far in (([far, near], True), ([near], False)):   # the second in a fresh context: the flag is sticky
        pos = np.array([[0.3 + 0.1 * i, (r + 0.5) * d] for i, r in enumerate(rows)])
        assert np.array_equal(rows_of(pos, d), rows)
        ctx = _raw_strip(world, pos, np.arange(len(rows)), 64, row_lo, row_hi)
        try:
            send_lo, send_hi = _wire_pair(64)
            ctx.dist_pack(send_lo, send_hi)
            st = ctx.dist_status(send_lo, send_hi)
            assert st["too_far"] == too_far, (rows, st)
            assert not st["overflow"]
            hdr_lo, recs_lo = _read_wire(send_lo, 64)
            hdr_hi, recs_hi = _read_wire(send_hi, 64)
            hdr, recs, other = (hdr_hi, recs_hi, hdr_lo) if side == "hi" else (hdr_lo, recs_lo, hdr_hi)
            assert int(hdr[2]) == int(too_far) and int(other[2]) == 0, (hdr.tolist(), other.tolist())
            # out of reach or not, a particle that left the strip is still handed over as a migrant
            assert int(hdr[0]) == len(rows) and int(other[0]) == 0
            assert sorted(recs["uid"].tolist()) == list(range(len(rows))) and (recs["kind"] == MIGRANT).all()
        finally:
            ctx.close()


@pytest.mark.gpu
def test_pack_wire_overflow_is_flagged_and_stays_in_bounds():
    """50 particles in the upper halo rows of an interior strip, wire capacity 8: the header counts all 50 and raises
    overflow, the 8 records stored are 8 of the 50 predicted ones, nothing is written past the buffer, and
    sc_dist_status reports the overflow.  (The pack stores a record only below the capacity; the unpacking pre-pass
    clamps a received count to it.  No step is taken with the overflowing buffers.)"""
    world, d = _strip_world()
    row_lo, row_hi, h, cap, n = 30, 50, HALO_ROWS, 8, 50
    rng = np.random.RandomState(1)
    rows = rng.randint(row_hi - h, row_hi, n)
    pos = np.stack([0.05 + 0.9 * rng.rand(n), (rows + 0.1 + 0.8 * rng.rand(n)) * d], 1)
    uid = np.arange(100, 100 + n)
    ctx = _raw_strip(world, pos, uid, cap, row_lo, row_hi)
    try:
        assert np.array_equal(rows_of(pos, d), rows)
        tail = 4 * REC.itemsize
        send_lo, send_hi = _wire_pair(cap, tail)
        ctx.dist_pack(send_lo, send_hi)
        ctx.synchronize()
        _, want_hi = _predict_pack(pos, np.zeros_like(pos), uid.astype(np.uint32), d, row_lo, row_hi, h, True, True)
        assert len(want_hi) == n and (want_hi["kind"] == HALO).all()
        hdr, got = _read_wire(send_hi, cap)
        assert int(hdr[0]) == n and int(hdr[1]) == 1 and int(hdr[2]) == 0, hdr.tolist()
        assert len(got) == cap and len(set(got["uid"].tolist())) == cap
        want_by_uid = {int(r["uid"]): r.tobytes() for r in want_hi}
        assert all(want_by_uid.get(int(r["uid"])) == r.tobytes() for r in got), "a stored record is not a predicted one"
        hdr_lo, _ = _read_wire(send_lo, cap)
        assert hdr_lo.tolist() == [0, 0, 0, 0]
        for b in (send_lo, send_hi):
            assert (b[_lib.wire_bytes(cap):].cpu().numpy() == 0xA5).all(), "the pack wrote past the wire buffer"
        st = ctx.dist_status(send_lo, send_hi)
        assert st["overflow"] and not st["too_far"]
    finally:
        ctx.close()

"""CPU tests of `bench.py --dump-outputs`: which rows are written, in what order, and that the files stay within the
64 MB the option promises (headers included) for the benchmark's own layouts."""
import os

import numpy as np
import pytest

import bench


def state(uid):
    """Per-particle arrays whose values encode the uid, in the layout of the one-GPU dump."""
    u = uid.astype(np.float64)
    return {"positions": np.stack((u, -u), 1), "velocities": np.stack((2 * u, u + 0.5), 1), "pressure": 3 * u}


def dumped_bytes(path):
    return sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def test_full_dump_in_ascending_uid_when_it_fits(tmp_path):
    uid = np.random.RandomState(1).permutation(1000).astype(np.uint32)
    cols = state(uid)
    assert bench.dump_sample(len(uid), cols) is None
    bench.write_dump(tmp_path, *bench.select_rows(uid, cols, None))
    assert np.array_equal(np.load(tmp_path / "uid.npy"), np.arange(1000.0))
    for name, v in state(np.arange(1000)).items():
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, v), name


@pytest.mark.parametrize("n_total,pressure", [(1_000_000, True), (2_000_000, True), (16_000_000, False),
                                               (64_000_000, False)])
def test_dump_is_seeded_and_within_64_mb(tmp_path, n_total, pressure):
    """1M on one GPU fits whole; 2M on one GPU and the 16M / 64M strip runs (no pressure) are sampled.  The files
    hold the sampled rows only, so they are built from the sample directly."""
    layout = {k: v for k, v in state(np.arange(2)).items() if pressure or k != "pressure"}
    sample = bench.dump_sample(n_total, layout)
    if n_total == 1_000_000:
        assert sample is None
        sample = np.arange(n_total)
    else:
        again = bench.dump_sample(n_total, layout)
        assert np.array_equal(sample, again) and np.all(np.diff(sample) > 0) and sample[-1] < n_total
    uid = sample.astype(np.uint32)
    cols = {k: v for k, v in state(uid).items() if k in layout}
    bench.write_dump(tmp_path, *bench.select_rows(uid, cols, None))
    size = dumped_bytes(tmp_path)
    assert size <= bench.DUMP_BYTES == 64_000_000, size
    if n_total > 1_000_000:
        assert size > 0.99 * bench.DUMP_BYTES, size   # the sample uses the budget


def test_rank_parts_merge_to_the_single_process_dump():
    """Strips: every rank samples its own rows, rank 0 merges them; the result equals the dump of the whole state."""
    n = 50_000
    rs = np.random.RandomState(2)
    uid = rs.permutation(n).astype(np.uint32)
    cols = state(uid)
    sample = bench.dump_sample(n, cols, budget=200_000)
    assert sample is not None and len(sample) < n
    want_uid, want = bench.select_rows(uid, cols, sample)
    assert np.array_equal(want_uid, sample)
    rank_of = rs.randint(0, 3, n)
    parts = [bench.select_rows(uid[rank_of == r], {k: v[rank_of == r] for k, v in cols.items()}, sample)
             for r in (2, 0, 1)]
    got_uid, got = bench.merge_rows(parts)
    assert np.array_equal(got_uid, want_uid)
    for k in cols:
        assert np.array_equal(got[k], want[k]), k

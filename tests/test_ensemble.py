"""Ensembles on the host: sweep expansion, uid packing, identity bits, per-member emission records, the model's
refusals, and the runner's --sweep / --replicas handling up to the point where a device is needed."""
import json
import os

import numpy as np
import pytest
import yaml

from conftest import world_from_freerun
from sand_crate_b200 import SandCrateError, run as runner
from sand_crate_b200.ensemble import (default_uid_bits, member_coefficients, member_emission, pack_uid, sweep_members,
                                      unpack_uid)
from sand_crate_b200.particle_source import build_particle_sources, counter_records


def test_sweep_is_cartesian_product_in_mapping_order_replicas_innermost():
    overrides, seeds = sweep_members({"viscosity": [4, 8, 16], "gravity": [[0, 9.8], [0, 5]]}, replicas=2)
    assert len(overrides) == 12 and seeds == [0, 1] * 6
    assert overrides[0] == {"viscosity": 4, "gravity": [0, 9.8]} == overrides[1]
    assert overrides[2] == {"viscosity": 4, "gravity": [0, 5]}
    assert overrides[4] == {"viscosity": 8, "gravity": [0, 9.8]}
    assert overrides[-1] == {"viscosity": 16, "gravity": [0, 5]}
    assert sweep_members(None, 3) == ([{}, {}, {}], [0, 1, 2])
    with pytest.raises(ValueError, match="non-empty list"):
        sweep_members({"viscosity": 4})
    with pytest.raises(ValueError, match="replicas"):
        sweep_members({}, 0)


def test_uid_packing_and_default_bits():
    uid = pack_uid(5, np.arange(4), 12)
    assert uid.dtype == np.uint32 and list(uid) == [5 * 4096 + k for k in range(4)]
    m, local = unpack_uid(uid, 12)
    assert list(m) == [5] * 4 and list(local) == [0, 1, 2, 3]
    # 16 x max_particles identities, at least 2^10
    assert default_uid_bits([4000], 1) == 16 and default_uid_bits([600, 100], 8) == 14 and default_uid_bits([3], 1) == 10
    # M members of B bits must stay below 2^31 (bit 31 is not an identity bit)
    assert default_uid_bits([4000], 1 << 15) == 16
    with pytest.raises(ValueError, match="member_uid_bits"):
        default_uid_bits([4000], (1 << 15) + 1)


def test_member_emission_equals_counter_records_of_each_seed():
    world, _ = world_from_freerun("wave_machine")
    sources = build_particle_sources(world.particle_sources)
    seeds = [0, 1, 2, 77]
    for tick in (0, 1, 250, 499):
        records, counts = member_emission(sources, seeds, tick, 0.002)
        for m, s in enumerate(seeds):
            own = counter_records(sources, s, tick, 0.002)
            got = [r[:6] + (int(counts[m, k]), r[7]) for k, r in enumerate(records) if counts[m, k]]
            assert got == own, (tick, m)
    assert member_emission(sources, seeds, 500, 0.002) == (None, None)   # the source is active for 500 ticks


def test_refusal_logic_names_the_cause():
    world, _ = world_from_freerun("wave_machine")
    assert len(member_coefficients(world, 3)) == 3
    assert member_coefficients(world, [{"viscosity": 2}])[0]["viscosity"] == 2
    with pytest.raises(ValueError, match="dt differs between member 0 and member 1"):
        member_coefficients(world, [{}, {"dt": 0.001}])
    with pytest.raises(ValueError, match="particle_radius differs"):
        member_coefficients(world, [{}, {}, {"particle_radius": 0.01}])
    with pytest.raises(ValueError, match="not a coefficient"):
        member_coefficients(world, [{"viscosty": 2}])
    # a motored paddle does not fall: gravity may differ
    assert member_coefficients(world, [{}, {"gravity": [0, 1.0]}])[1]["gravity"] == [0, 1.0]
    free, _ = world_from_freerun("free_body")
    with pytest.raises(ValueError, match="free body"):
        member_coefficients(free, [{}, {"gravity": [0, 1.0]}])
    with pytest.raises(ValueError, match="at least one member"):
        member_coefficients(world, [])


def _config_file(tmp_path, name):
    world, _ = world_from_freerun(name)
    raw = {"world": {"coefficients": world.coefficients, "particle_sources": world.particle_sources,
                     "rigid_bodies": world.rigid_bodies}, "playback": {"ticks_to_record": 20}}
    p = tmp_path / f"{name}.yaml"
    p.write_text(yaml.safe_dump(raw))
    return str(p)


def test_runner_sweep_arguments_and_members_json(tmp_path, monkeypatch):
    cfg = _config_file(tmp_path, "stirring_cup")
    sweep = tmp_path / "sweep.yaml"
    sweep.write_text(yaml.safe_dump({"viscosity": [4, 8], "pressure_amplifier": [20, 30, 40]}))
    out = tmp_path / "out"
    seen = {}

    def fake_run_ensemble(config_path, sweep, replicas, ticks, every, out, precision, noise, device):
        seen.update(sweep=sweep, replicas=replicas, noise=noise, precision=precision)
    monkeypatch.setattr(runner, "run_ensemble", fake_run_ensemble)
    runner.main([cfg, "--sweep", str(sweep), "--replicas", "3", "--out", str(out)])
    assert seen == {"sweep": {"viscosity": [4, 8], "pressure_amplifier": [20, 30, 40]}, "replicas": 3,
                    "noise": "counter", "precision": "f64"}
    runner.main([cfg, "--replicas", "2", "--noise", "none", "--precision", "mixed"])
    assert seen == {"sweep": None, "replicas": 2, "noise": "none", "precision": "mixed"}
    with pytest.raises(SystemExit):
        runner.main([cfg, "--replicas", "2", "--noise", "reference"])
    monkeypatch.undo()
    # members.json is written before the device is needed (this machine may have none: the Ensemble then raises)
    try:
        runner.run_ensemble(cfg, {"viscosity": [4, 8]}, 2, 3, 1, str(out), "mixed", "counter", 0, quiet=True)
    except SandCrateError:
        pass
    members = json.loads((out / "members.json").read_text())
    assert members == [{"member": 0, "overrides": {"viscosity": 4}, "seed": 0},
                       {"member": 1, "overrides": {"viscosity": 4}, "seed": 1},
                       {"member": 2, "overrides": {"viscosity": 8}, "seed": 0},
                       {"member": 3, "overrides": {"viscosity": 8}, "seed": 1}]


def test_member_recording_layout_reads_with_load_recording(tmp_path):
    cfg = _config_file(tmp_path, "wave_machine")
    rng = np.random.default_rng(0)
    counts = [3, 0, 5]
    pos = [rng.random((c, 2)) for c in counts]
    prs = [rng.random(c) for c in counts]
    segs = [rng.random((8, 2, 2)) for _ in counts]
    path = os.path.join(tmp_path, "member_0.npz")
    runner.save_recording(path, cfg, [10, 20, 30], counts, pos, prs, segs, {"member": 0})
    frames = list(runner.load_recording(path))
    assert [f[0] for f in frames] == [10, 20, 30]
    for k, (tick, p, q, s) in enumerate(frames):
        assert np.array_equal(p, pos[k]) and np.array_equal(q, prs[k]) and np.array_equal(s, segs[k])

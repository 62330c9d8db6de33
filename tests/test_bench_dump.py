"""bench.py --dump-outputs on the CPU: the dumped arrays split back into every sampled path's outputs, the sample shrinks
to the size budget, and the reference arm writes the summary rows of its last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_result(oracle_mod, packed):
    """A ProfileResult on CPU tensors, filled from the oracle, with unused tails poisoned."""
    import torch
    from vexautonomousplanner_b200.engine import OUT_NAMES, ProfileResult
    refs = [oracle_mod.full(packed.node_attr[b], packed.node_flags[b], packed.ap_attr[b, :packed.n_ap[b]],
                            packed.ap_flags[b, :packed.n_ap[b]], packed.cons[b]) for b in range(packed.B)]
    B, T, D = packed.B, max(r["T"] for r in refs) + 5, max(r["D"] for r in refs) + 5
    out = torch.full((len(OUT_NAMES), B, T), np.nan, dtype=torch.float64)
    vel = torch.full((B, D), np.nan, dtype=torch.float64)
    nodes_map = torch.full((B, packed.node_attr.shape[1] + 1), 99, dtype=torch.int32)
    actions_map = torch.full((B, packed.ap_attr.shape[1]), 99, dtype=torch.int32)
    n_maps = torch.zeros((B, 2), dtype=torch.int32)
    for b, r in enumerate(refs):
        for i, name in enumerate(OUT_NAMES):
            out[i, b, :r["T"]] = torch.from_numpy(r[name])
        vel[b, :r["D"]] = torch.from_numpy(r["vel"])
        nodes_map[b, :len(r["nodes_map"])] = torch.from_numpy(r["nodes_map"].astype(np.int32))
        actions_map[b, :len(r["actions_map"])] = torch.from_numpy(r["actions_map"].astype(np.int32))
        n_maps[b] = torch.tensor([len(r["nodes_map"]), len(r["actions_map"])])
    res = ProfileResult(B, T, out, torch.tensor([r["T"] for r in refs], dtype=torch.int32), nodes_map, actions_map, n_maps,
                        torch.zeros(B, dtype=torch.int32), torch.from_numpy(np.stack([r["summary"] for r in refs])), vel,
                        torch.tensor([r["D"] for r in refs], dtype=torch.int32))
    return res, refs


def test_profile_dump_round_trip_and_budget(oracle_mod, tmp_path, monkeypatch):
    pytest.importorskip("torch")
    import bench
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import OUT_NAMES
    res, refs = _oracle_result(oracle_mod, synth.mixed_paths(24, 6, seed=5))
    full = bench.profile_dump(res, max_paths=8)
    monkeypatch.setattr(bench, "DUMP_BYTES", sum(a.nbytes for a in bench.profile_dump(res, max_paths=2).values()))
    for d, k in ((full, 8), (bench.profile_dump(res, max_paths=8), 2)):
        paths = d["paths"].astype(int)
        assert len(paths) == k and np.all(np.diff(paths) > 0)
        assert np.array_equal(d["summary"], res.summary.numpy()) and np.array_equal(d["n_samples"], res.n_samples.numpy())
        off = np.concatenate([[0], np.cumsum(d["summary"][paths, 0].astype(int))])
        voff = np.concatenate([[0], np.cumsum(d["n_samples"][paths].astype(int))])
        for j, b in enumerate(paths):
            r = refs[b]
            for name in OUT_NAMES:
                assert np.array_equal(d[name][off[j]:off[j + 1]], r[name]), (b, name)
            assert np.array_equal(d["vel"][voff[j]:voff[j + 1]], r["vel"])
            for name in ("nodes_map", "actions_map"):
                n = len(r[name])
                assert d[name][j, :n].tolist() == r[name].tolist() and (d[name][j, n:] == -1).all(), (b, name)
    assert set(d["paths"]) <= set(full["paths"])                # a smaller budget keeps part of the same sample
    bench.write_dump(str(tmp_path / "d"), d)
    assert sorted(os.listdir(tmp_path / "d")) == sorted(f"{k}.npy" for k in d)
    assert all(np.load(tmp_path / "d" / f"{k}.npy").dtype == np.float64 for k in d)
    with pytest.raises(ValueError):
        bench.write_dump(str(tmp_path / "e"), full)


def test_reference_arm_dumps_its_last_step(oracle_mod, tmp_path):
    from vexautonomousplanner_b200 import synth
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "0", "--no-pyref", "--ref-sample", "16", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, check=True).stdout
    assert json.loads(out.strip().splitlines()[-1])["steps"] == 2
    p = synth.random_paths(4096, 8, seed=0).slice(0, 16)
    assert os.listdir(tmp_path) == ["summary.npy"]
    assert np.array_equal(np.load(tmp_path / "summary.npy"), oracle_mod.full_batch(p.node_attr, p.node_flags, p.cons))

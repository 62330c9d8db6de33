"""Bulk save: every path's trajectory .txt body assembled on the device (export.save_text_batch, vap_splice_plan /
vap_splice_actions) and the save_routes command that re-saves a folder of routes."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _insert_rows(lines, nodes_map, node_actions, actions_map, ap_actions):
    """The reference's splice (gui_manager.py:297-310) on a list of text lines, with Python's own list.insert."""
    from vexautonomousplanner_b200.export import format_rows
    lines = list(lines)
    for i in range(len(nodes_map)):
        lines.insert(int(nodes_map[i]) + i, format_rows([[1] + list(node_actions[i])]))
    for j in range(len(actions_map)):
        lines.insert(int(actions_map[j]) + j, format_rows([[1] + list(ap_actions[j])]))
    return "".join(lines)


# ------------------------------------------------------------------------------------------------------------- CPU
def test_action_row_text_cpu():
    """Host text of the action rows: format_rows([[1, *v]]) for every row, whatever the value types (ints, bools, floats,
    numpy scalars, -0.0 next to 0.0, 1 next to 1.0 and True), laid out path by path, node rows first."""
    from vexautonomousplanner_b200 import export as ex
    node_actions = [[[0, 0], [0, 0], [True, 0], [1, 0], [1.0, 0], [0.0], [-0.0], []],
                    [],
                    [[np.float64(0.1), np.int64(3)], [0, 0], (2, "x")]]
    ap_actions = [[[0, 0], [False]], [[5, 5, 5]], [[0.30000000000000004, 1e22], [[1, 2]]]]
    text, off, first, rows = ex.pack_action_rows(node_actions, ap_actions)
    assert rows.tolist() == [[8, 2], [0, 1], [3, 2]] and first.tolist() == [0, 10, 11]
    flat = [v for b in range(3) for v in list(node_actions[b]) + list(ap_actions[b])]
    assert len(off) == len(flat) + 1 and off[0] == 0 and off[-1] == len(text)
    got = [bytes(text[off[i]:off[i + 1]]).decode() for i in range(len(flat))]
    assert got == [ex.format_rows([[1, *v]]) for v in flat]
    assert got[2] == "1 True 0 \n" and got[4] == "1 1.0 0 \n" and got[6] == "1 -0.0 \n" and got[7] == "1 \n"
    assert got[-1] == "1 [1, 2] \n"
    e_text, e_off, e_first, e_rows = ex.pack_action_rows([[]], [[]])
    assert e_text.size == 0 and e_off.tolist() == [0] and e_first.tolist() == [0] and e_rows.tolist() == [[0, 0]]
    with pytest.raises(ValueError):
        ex.pack_action_rows([[]], [])


def test_save_routes_reads_folder_and_config_cpu(tmp_path):
    """The command's host side: which files of a folder are routes, which are listed and skipped, and the constraints
    from the factory defaults, from a config.yaml in the GUI's layout and from flags."""
    from vexautonomousplanner_b200 import save_routes as sr
    from vexautonomousplanner_b200.synth import FACTORY
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "gui_reference.json")))
    d = tmp_path / "routes"
    d.mkdir()
    (d / "a_cfg1.txt").write_text(ref["cfg1"]["built"]["json"])
    (d / "b_turns.txt").write_text(ref["turn_reverse_wait"]["built"]["json"])
    (d / "c_notes.txt").write_text("not json at all\n")
    (d / "d_dict.txt").write_text('{"nodes": []}')
    nodes, aps = json.loads(ref["cfg1"]["built"]["json"])
    no_end = [n[:3] + [0] + n[4:] for n in nodes]
    (d / "e_no_end.txt").write_text(json.dumps([no_end, aps]))
    (d / "f_two_nodes.txt").write_text(json.dumps([[nodes[0], nodes[-1]], []]))
    (d / "g_other.json").write_text(ref["cfg1"]["built"]["json"])          # not a .txt: not a route file
    routes, skipped = sr.read_routes(str(d))
    assert [r[0] for r in routes] == ["a_cfg1.txt", "b_turns.txt"]
    assert [s[0] for s in skipped] == ["c_notes.txt", "d_dict.txt", "e_no_end.txt", "f_two_nodes.txt"]
    assert "not route JSON" in skipped[0][1] and "not route JSON" in skipped[1][1]
    assert "end node missing" in skipped[2][1] and "2 nodes" in skipped[3][1]
    name, pts, rnodes, raps = routes[1]
    assert pts.shape == (len(rnodes), 2) and len(raps) == len(ref["turn_reverse_wait"]["built"]["action_points"])

    assert sr.constraints(sr.parse_args(["r", "o"])) == FACTORY
    cfg = tmp_path / "config.yaml"
    cfg.write_text("robot:\n  width: 15\n  track_width: 11.5\nmotion:\n  max_velocity: 5.5\n  max_acceleration: 12.0\n"
                   "files:\n  routes_folder: x\n")
    c = sr.constraints(sr.parse_args(["r", "o", "--config", str(cfg)]))
    assert c == (5.5, 12.0, 12.0, 0.8, FACTORY[4], 11.5 / 12)                 # max_jerk missing: the factory value
    c = sr.constraints(sr.parse_args(["r", "o", "--config", str(cfg), "--max-jerk", "43", "--track-width-in", "12"]))
    assert c == (5.5, 12.0, 12.0, 0.8, 43.0, 1.0)
    c = sr.constraints(sr.parse_args(["r", "o", "--max-velocity", "3", "--max-acceleration", "6"]))
    assert c == (3.0, 6.0, 6.0, 0.8, FACTORY[4], FACTORY[5])


# ------------------------------------------------------------------------------------------------------------- GPU
def _route_batch(ref, names):
    from test_next_rows import _route_objects
    from vexautonomousplanner_b200 import export as ex
    paths, node_actions, ap_actions = [], [], []
    for name in names:
        st = ref[name]["built"]
        nodes, aps = _route_objects(st)
        paths.append((ex.px_points_to_ft(st["ordered_px"]), nodes, aps))
        node_actions.append([n.action_values for n in nodes])
        ap_actions.append([a.action_values for a in aps])
    return paths, node_actions, ap_actions


@pytest.mark.gpu
def test_batch_save_against_the_reference_save_path():
    """Two routes the reference saved itself (tests/golden/save_txt_*.txt.gz) with a failing path between them: every ok
    body matches the reference's file under the token rule of test_trajectory_txt_against_the_reference_save_path and
    equals trajectory_text byte for byte; the failing path (a turn on its last node, IndexError) has zero bytes."""
    import torch
    from golden_util import GOLDEN_DIR
    from test_next_rows import _gui_ref
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.packing import pack_paths
    from vexautonomousplanner_b200.synth import FACTORY
    ref = _gui_ref()
    paths, node_actions, ap_actions = _route_batch(ref, ["turn_reverse_wait", "node0_wait", "node0_wait"])
    paths[1][1][-1].turn = 90                       # the middle path: a turn on the last node
    eng = Engine("cuda:0")
    db = eng.upload(pack_paths(paths, FACTORY))
    res = eng.profile(db)
    assert res.status.cpu().tolist() == [0, -2, 0]
    text, offs, ok = ex.save_text_batch(eng, res, db, node_actions, ap_actions)
    assert ok.tolist() == [True, False, True] and offs[1] == offs[2] and offs[-1] == len(text)
    for b, name in ((0, "turn_reverse_wait"), (2, "node0_wait")):
        got = bytes(text[offs[b]:offs[b + 1]]).decode()
        assert got == ex.trajectory_text(eng, res, b, node_actions[b], ap_actions[b], db=db), name
        want = gzip.open(os.path.join(GOLDEN_DIR, f"save_txt_{name}.txt.gz"), "rt").read()
        gl, wl = got.splitlines(), want.splitlines()
        assert len(gl) == len(wl), name
        n_int = 0
        for r, (g, w) in enumerate(zip(gl, wl)):
            gt, wt = g.split(" "), w.split(" ")
            assert len(gt) == len(wt), (name, r, g, w)
            for c, (x, y) in enumerate(zip(gt, wt)):
                is_int = y.lstrip("-").isdigit()
                if is_int or y == "":
                    assert x == y, (name, r, c, g, w)
                    n_int += is_int
                else:
                    assert not x.lstrip("-").isdigit(), (name, r, c, g, w)
                    tol = dict(rtol=1e-9, atol=1e-9) if c in (2, 3, 4) else dict(rtol=1e-6, atol=1e-6)
                    np.testing.assert_allclose(float(x), float(y), err_msg=f"{name} row {r} col {c}", **tol)
        assert n_int > len(wl)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_batch_save_mixed_batch_equals_host_splice():
    """4096 mixed paths (turns, waits, reverses, stops, action points) with random int action tuples of length 0-3: every
    body equals the device trajectory lines spliced on the host with list.insert, byte for byte."""
    from vexautonomousplanner_b200 import export as ex, synth
    from vexautonomousplanner_b200.engine import Engine
    packed = synth.mixed_paths(4096, 8, seed=17)
    rng = np.random.default_rng(4)

    def tuples(n):
        return [tuple(int(x) for x in rng.integers(-3, 12, rng.integers(0, 4))) for _ in range(n)]
    node_actions = [tuples(int(n)) for n in packed.n_nodes]
    ap_actions = [tuples(int(a)) for a in packed.n_ap]
    eng = Engine("cuda:0")
    db = eng.upload(packed)
    res = eng.profile(db)
    text, offs, ok = ex.save_text_batch(eng, res, db, node_actions, ap_actions)
    assert offs[-1] == len(text) and offs[0] == 0
    dtext, droff, dpoff_d = ex.export_text_device(eng, res, db)
    kinds = ex.row_kinds(eng, res, db, offsets=dpoff_d, n_rows=int(dpoff_d[-1]))
    dtext, droff, dpoff = bytes(dtext.cpu().numpy()), droff.cpu().numpy(), dpoff_d.cpu().numpy()
    status, n_maps = res.status.cpu().numpy(), res.n_maps.cpu().numpy()
    nmap, amap = res.nodes_map.cpu().numpy(), res.actions_map.cpu().numpy()
    assert (ok == (status == 0)).all() and ok.sum() > res.B // 2
    for b in range(res.B):
        body = bytes(text[offs[b]:offs[b + 1]]).decode()
        if not ok[b]:
            assert body == ""
            continue
        lines = dtext[droff[dpoff[b]]:droff[dpoff[b + 1]]].decode().splitlines(keepends=True)
        want = _insert_rows(lines, nmap[b, :n_maps[b, 0]], node_actions[b], amap[b, :n_maps[b, 1]], ap_actions[b])
        assert body == want, b
    assert (n_maps[status == 0, 1] > 0).sum() > 100                                     # action-point rows
    assert ((kinds.cpu().numpy() & ex.RK_INSERTED) != 0).sum() > 1000                   # inserted turn / wait rows
    assert sum(len(t) == 0 for a in node_actions for t in a) > 1000                     # empty action tuples: "1 \n"


def _hand_batch(eng, n_lines, status, node_maps, ap_maps, seed=0):
    """Device inputs of splice_bodies for hand-made paths: random export rows formatted by vap_format_rows, maps as given."""
    import torch
    from vexautonomousplanner_b200 import export as ex
    rng = np.random.default_rng(seed)
    B = len(n_lines)
    row_off = np.zeros(B + 1, dtype=np.int64)
    row_off[1:] = np.cumsum(n_lines)
    rows = rng.uniform(-50, 50, (int(row_off[-1]), 7))
    rows[:, 0] = 0
    dev = eng.device
    slots, lens, line_off = ex._format_slots(eng, torch.tensor(rows, device=dev), None)
    N_max = max(len(m) for m in node_maps)
    A = max([len(m) for m in ap_maps] + [1])
    nm = np.zeros((B, N_max), dtype=np.int32)
    am = np.zeros((B, A), dtype=np.int32)
    cnt = np.zeros((B, 2), dtype=np.int32)
    for b in range(B):
        nm[b, :len(node_maps[b])] = node_maps[b]
        am[b, :len(ap_maps[b])] = ap_maps[b]
        cnt[b] = len(node_maps[b]), len(ap_maps[b])
    t = lambda a: torch.tensor(a, device=dev)
    args = (slots, lens, line_off, t(row_off), t(np.asarray(status, dtype=np.int32)), t(nm), t(am), t(cnt))
    lines = [[ex.format_rows([[0, *map(float, r[1:])]]) for r in rows[row_off[b]:row_off[b + 1]]] for b in range(B)]
    return args, lines


HAND = dict(                      # lines, status, nodes_map, actions_map
    n_lines=[4, 0, 3, 0, 0, 2, 5],
    status=[0, -2, 0, 0, -5, 0, 0],
    node_maps=[[0, 2, 2, 4], [], [0, 10, -1], [0, 0], [], [1, 2], [0, 2, 5]],
    ap_maps=[[3, 3], [], [-5, 100], [], [], [0], [-1, 2, 2]],
)


@pytest.mark.gpu
def test_splice_insert_rules_on_hand_made_paths():
    """Python's list.insert rules through vap_splice_plan / vap_splice_actions: equal node indices, duplicate action
    indices, an action index equal to a node row's, indices past the end (append), negative indices (from the end,
    clamped at 0), a path with node rows but no trajectory lines, failing paths between ok ones."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    args, lines = _hand_batch(eng, **HAND)
    B = len(HAND["status"])
    node_actions = [[(b, i) for i in range(len(HAND["node_maps"][b]))] for b in range(B)]
    ap_actions = [[(b, -j, True, 0.5) for j in range(len(HAND["ap_maps"][b]))] for b in range(B)]
    node_actions[6].append(("unused",))             # more rows than the maps use: the extra row is in no body
    text, offs, ok = ex.splice_bodies(eng, *args, node_actions, ap_actions)
    assert ok.tolist() == [s == 0 for s in HAND["status"]] and offs[-1] == len(text)
    for b in range(B):
        body = bytes(text[offs[b]:offs[b + 1]]).decode()
        if HAND["status"][b]:
            assert body == "", b
        else:
            assert body == _insert_rows(lines[b], HAND["node_maps"][b], node_actions[b], HAND["ap_maps"][b], ap_actions[b]), b
    assert bytes(text[offs[3]:offs[4]]).decode() == "1 3 0 \n1 3 1 \n"
    assert "unused" not in bytes(text).decode()


@pytest.mark.gpu
def test_splice_too_few_action_rows_raises():
    """A path whose maps need more node or action-point rows than were passed raises ValueError (the reference raises
    IndexError); the short path is the last one, so its rows would lie past the end of the row buffers.  The same batch
    with enough rows assembles afterwards."""
    import torch
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    args, lines = _hand_batch(eng, **HAND)
    B = len(HAND["status"])
    full_n = [[(i,) for i in range(len(HAND["node_maps"][b]))] for b in range(B)]
    full_a = [[(7, j) for j in range(len(HAND["ap_maps"][b]))] for b in range(B)]
    for short_n, short_a in ((full_n[:-1] + [full_n[-1][:2]], full_a), (full_n, full_a[:-1] + [full_a[-1][:1]]),
                             (full_n[:-1] + [[]], full_a[:-1] + [[]])):
        with pytest.raises(ValueError, match="more action rows"):
            ex.splice_bodies(eng, *args, short_n, short_a)
    torch.cuda.synchronize()
    text, offs, ok = ex.splice_bodies(eng, *args, full_n, full_a)
    assert bytes(text[offs[6]:offs[7]]).decode() == _insert_rows(lines[6], HAND["node_maps"][6], full_n[6],
                                                                 HAND["ap_maps"][6], full_a[6])


@pytest.mark.gpu
def test_save_routes_command(tmp_path):
    """python -m vexautonomousplanner_b200.save_routes over a folder of every built route of gui_reference.json, one
    non-route file and one route without an end node, two routes per tile: each written file equals trajectory_text of
    the same loaded route, the two bad inputs are listed and not written, the exit status is 1; a run with
    OUT_DIR == ROUTES_DIR refuses."""
    from test_next_rows import _gui_ref
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.packing import pack_paths
    from vexautonomousplanner_b200.synth import FACTORY
    ref = _gui_ref()
    rdir, odir = tmp_path / "routes", tmp_path / "out"
    rdir.mkdir()
    names = [n for n, r in ref.items() if "built" in r]
    assert len(names) >= 5
    for n in names:
        (rdir / f"{n}.txt").write_text(ref[n]["built"]["json"])
    (rdir / "readme.txt").write_text("these are our routes\n")
    nodes, aps = json.loads(ref["cfg1"]["built"]["json"])
    (rdir / "no_end.txt").write_text(json.dumps([[n[:3] + [0] + n[4:] for n in nodes], aps]))
    before = {p.name: p.read_bytes() for p in rdir.iterdir()}
    cmd = [sys.executable, "-m", "vexautonomousplanner_b200.save_routes", str(rdir), str(odir), "--tile-paths", "2"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 1, r.stdout + r.stderr
    assert "not written: readme.txt: not route JSON" in r.stdout and "not written: no_end.txt:" in r.stdout, r.stdout
    eng = Engine("cuda:0")
    written = []
    for n in names:
        pts, rnodes, raps, _ = ex.load_nodes(ref[n]["built"]["json"])
        db = eng.upload(pack_paths([(ex.px_points_to_ft(pts), rnodes, raps)], FACTORY))
        res = eng.profile(db)
        out = odir / f"{n}.txt"
        if int(res.status[0]) != 0:
            assert not out.exists() and f"not written: {n}.txt: profile failed" in r.stdout, n
            continue
        want = ex.trajectory_text(eng, res, 0, [x.action_values for x in rnodes], [a.action_values for a in raps], db=db)
        assert out.read_bytes().decode() == want, n
        written.append(out.name)
    assert len(written) >= 4
    assert sorted(p.name for p in odir.iterdir()) == sorted(written)          # nothing for readme.txt / no_end.txt
    same = subprocess.run(cmd[:4] + [str(rdir)], cwd=ROOT, capture_output=True, text=True)
    assert same.returncode == 2 and "refusing" in same.stderr
    assert {p.name: p.read_bytes() for p in rdir.iterdir()} == before

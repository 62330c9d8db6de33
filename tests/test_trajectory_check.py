"""Reading saved trajectory .txt files back on the device (export.parse_doubles_device / parse_text_batch /
compare_text_batch, csrc/vap_parse.cuh) and the save_routes --check mode built on them."""
import gzip
import json
import os
import struct

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MALFORMED = ["", "-", "1.", ".5", "1e", "1e+", "--1", "1.2.3", "abc", "0x10", "1e5x", "+1", " 1", "1 ", "in", "infinity",
             "nan0", "1_000", "0,5", "1e-", "-.5", "e5", "1.0e5.0", "1\t"]


def _tokens(n, seed=0):
    """repr() of random bit patterns (every exponent), subnormals, +-0, +-inf, nan and the int 0; %.17g, %.25e and
    30-digit fixed forms of the same values; exact midpoints between neighbouring doubles and decimals just off them.
    Returns (tokens, number of repr tokens at the front)."""
    from decimal import Decimal, getcontext
    getcontext().prec = 800
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2 ** 63, n, dtype=np.int64).view(np.uint64) | (rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63))
    sub = rng.integers(0, 2 ** 52, n // 8, dtype=np.int64).view(np.float64)
    xs = np.concatenate([bits.view(np.float64), sub, [0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, 2.2250738585072014e-308,
                                                      1.7976931348623157e308]]).tolist()
    toks = [repr(x) for x in xs] + ["0", "-0"]
    n_repr = len(toks)
    fin = [x for x in xs if np.isfinite(x)]
    for x in fin[: n // 2]:
        toks += ["%.17g" % x, "%.25e" % x, np.format_float_positional(x, precision=30, unique=False, fractional=False, trim="0")]
    for x in fin[: n // 16]:
        x = abs(x)
        if x == 0 or x >= 1.7e308:
            continue
        nx = float(np.nextafter(x, np.inf))
        mid, eps = (Decimal(x) + Decimal(nx)) / 2, Decimal(nx - x) / 10 ** 30
        toks += [format(mid, "e"), format(mid + eps, "e"), format(mid - eps, "e")]
    return toks, n_repr


def _bits(x):
    return struct.unpack("<q", struct.pack("<d", x))[0]


# ------------------------------------------------------------------------------------------------------------- CPU
def test_check_arguments_and_refusal_cpu(tmp_path):
    """--check is a flag of the save_routes command; with OUT_DIR == ROUTES_DIR it refuses (exit 2) before anything
    runs, and writes nothing."""
    from vexautonomousplanner_b200 import save_routes as sr
    assert sr.parse_args(["r", "o", "--check"]).check and not sr.parse_args(["r", "o"]).check
    a = sr.parse_args(["r", "o", "--check", "--max-velocity", "2", "--tile-paths", "3"])
    assert a.max_velocity == 2.0 and a.tile_paths == 3
    d = tmp_path / "routes"
    d.mkdir()
    (d / "x.txt").write_text("[[], []]")
    assert sr.main([str(d), str(d) + "/", "--check"]) == 2
    assert [p.name for p in d.iterdir()] == ["x.txt"]
    with pytest.raises(SystemExit):
        sr.parse_args(["r", "o", "--check", "--tile-paths", "0"])


def _stub(diff=-1, line=0, rows=(10, 10), err=(0, 0), t=(1.5, 1.25), d=(0.0,) * 6, act=0):
    from vexautonomousplanner_b200.export import CMP_F, CMP_I
    ints = np.array([diff, line, rows[0], rows[1], act, err[0], err[1]], dtype=np.int64)
    floats = np.array([t[0], t[1], *d], dtype=np.float64)
    assert len(ints) == len(CMP_I) and len(floats) == len(CMP_F)
    return ints, floats


def test_check_report_lines_and_exit_codes_cpu(tmp_path, monkeypatch, capsys):
    """The report line of each state from a stubbed comparison, and the exit status of the command: 0 only when every
    route is up to date; skipped routes are listed."""
    from vexautonomousplanner_b200 import save_routes as sr
    assert sr.check_line("a.txt", *_stub()) == ("up to date", "up to date: a.txt")
    state, line = sr.check_line("b.txt", *_stub(diff=40, line=3, err=(3, 5)))
    assert state == "unreadable" and line == "unreadable: b.txt: line 3: token 2 (t) is not a number"
    assert sr.check_line("b.txt", *_stub(diff=0, line=1, err=(1, 2)))[1] == \
        "unreadable: b.txt: line 1: the first token is neither 0 nor 1"
    assert sr.check_line("b.txt", *_stub(diff=0, line=1, err=(7, 3)))[1].endswith("line 7: a trajectory row without 7 tokens")
    state, line = sr.check_line("c.txt", *_stub(diff=100, line=2, rows=(1430, 1388), t=(5.7, 5.55),
                                               d=(0.1, 0.0123, 0.25, 0.001, 1.5, 0.3), act=2))
    assert state == "stale"
    assert line == ("stale: c.txt: first difference on line 2; rows 1430 -> 1388; duration 5.7 -> 5.55 s; max |dx| 0.0123 in, "
                    "|dy| 0.25 in, |dv| 1.5 in/s, |dheading| 0.001; 2 action rows differ")

    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "gui_reference.json")))
    d = tmp_path / "routes"
    d.mkdir()
    (d / "a.txt").write_text(ref["cfg1"]["built"]["json"])
    (d / "b.txt").write_text(ref["turn_reverse_wait"]["built"]["json"])
    results = {}
    monkeypatch.setattr(sr, "check_routes", lambda routes, out_dir, cons, tile, dev: [(n, *results[n]) for n, *_ in routes])
    results.update({"a.txt": ("up to date", "up to date: a.txt"), "b.txt": ("up to date", "up to date: b.txt")})
    assert sr.main([str(d), str(tmp_path / "out"), "--check"]) == 0
    out = capsys.readouterr().out
    assert "up to date: a.txt" in out and "2 of 2 files up to date" in out
    assert not (tmp_path / "out").exists()                                   # --check writes nothing, not even OUT_DIR
    for other in ("missing", "stale", "unreadable", "not checked"):
        results["b.txt"] = (other, f"{other}: b.txt")
        assert sr.main([str(d), str(tmp_path / "out"), "--check"]) == 1, other
        assert "1 of 2 files up to date" in capsys.readouterr().out
    results["b.txt"] = ("up to date", "up to date: b.txt")
    (d / "notes.txt").write_text("not a route")
    assert sr.main([str(d), str(tmp_path / "out"), "--check"]) == 1
    assert "not checked: notes.txt: not route JSON" in capsys.readouterr().out


def test_host_fallback_finishes_flagged_tokens_cpu():
    """Tokens the device leaves undecided are finished with float() into their slots; the others stay as they are."""
    import torch
    from vexautonomousplanner_b200 import export as ex
    rows = torch.full((3, 7), float("nan"), dtype=torch.float64)
    toks = [b"2.2250738585072011e-308", b"9007199254740993", b"0.1000000000000000055511151231257827021181583404541015625",
            b"-inf"]
    ex._host_finish(rows, [1 * 7 + 2, 0 * 7 + 6, 2 * 7 + 1, 2 * 7 + 3], toks)
    want = {(1, 2): float(toks[0]), (0, 6): float(toks[1]), (2, 1): float(toks[2]), (2, 3): float("-inf")}
    for r in range(3):
        for c in range(7):
            v = float(rows[r, c])
            if (r, c) in want:
                assert _bits(v) == _bits(want[(r, c)]), (r, c)
            else:
                assert v != v
    ex._host_finish(rows, [], [])
    assert ex.line_error_text(4 + 6) == "token 7 (omega) is not a number"


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_parse_doubles_bit_equal_to_float():
    """parse_doubles_device(s) == float(s) bit for bit (nan by class) on more than 5e5 tokens: repr of random bit patterns,
    non-shortest forms, exact midpoints; malformed tokens are flagged.  No repr token needs the host."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    toks, n_repr = _tokens(200_000)
    assert len(toks) >= 500_000
    eng = Engine("cuda:0")
    x, flags = ex.parse_doubles_device(eng, toks + MALFORMED)
    got = x.cpu().numpy()
    n = len(toks)
    assert (flags[n:] == 2).all(), [t for t, f in zip(MALFORMED, flags[n:]) if f != 2]
    assert (flags[:n] != 2).all(), [toks[i] for i in np.flatnonzero(flags[:n] == 2)[:5]]
    want = np.array([float(t) for t in toks])
    nan = np.isnan(want)
    assert (np.isnan(got[:n]) == nan).all()
    bad = np.flatnonzero(~nan & (got[:n].view(np.int64) != want.view(np.int64)))
    assert bad.size == 0, [(toks[i], got[i], want[i]) for i in bad[:5]]
    n_host = int((flags[:n] == 1).sum())
    print(f"\n{n} tokens, {n_host} finished on the host ({int((flags[:n_repr] == 1).sum())} of {n_repr} repr tokens)")
    assert (flags[:n_repr] == 0).all()


def _mixed_batch(B, seed):
    """synth.mixed_paths with node and action rows as profiles/tools/save_speed.py builds them."""
    from vexautonomousplanner_b200 import synth
    packed = synth.mixed_paths(B, 8, seed=seed)
    rng = np.random.default_rng(5)
    tup = lambda: [int(v) for v in rng.integers(0, 10, rng.integers(0, 4))]
    return packed, [[tup() for _ in range(int(n))] for n in packed.n_nodes], [[tup() for _ in range(int(a))] for a in packed.n_ap]


@pytest.mark.gpu
def test_round_trip_mixed_batch():
    """parse_text_batch(save_text_batch(...)) on 2048 mixed paths: the trajectory rows are bit-equal to export_rows (a
    column the reference writes as the int 0 reads back as +0.0), and the action rows sit where list.insert put them."""
    import torch
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    packed, na, aa = _mixed_batch(2048, 3)
    eng = Engine("cuda:0")
    db = eng.upload(packed)
    res = eng.profile(db)
    text, offs, ok = ex.save_text_batch(eng, res, db, na, aa)
    rows, row_off = ex.export_rows(eng, res)
    p = ex.parse_text_batch(eng, text, offs)
    assert p.n_host == 0 and int((p.line_errors != 0).sum()) == 0
    assert torch.equal(p.row_offsets, row_off)
    same = (p.rows.view(torch.int64) == rows.view(torch.int64)) | ((p.rows == 0) & (rows == 0))
    assert bool(same.all()), torch.nonzero(~same)[:5].tolist()
    kinds, pl = p.line_kinds.cpu().numpy(), p.path_line_offsets.cpu().numpy()
    ro, n_maps = row_off.cpu().numpy(), res.n_maps.cpu().numpy()
    nmap, amap = res.nodes_map.cpu().numpy(), res.actions_map.cpu().numpy()
    assert (p.act_offsets.cpu().numpy()[1:] - p.act_offsets.cpu().numpy()[:-1] == np.where(ok, n_maps.sum(axis=1), 0)).all()
    n_act = 0
    for b in range(res.B):
        if not ok[b]:
            assert pl[b] == pl[b + 1]
            continue
        lines = ["T"] * int(ro[b + 1] - ro[b])
        for i in range(n_maps[b, 0]):
            lines.insert(int(nmap[b, i]) + i, "A")
        for j in range(n_maps[b, 1]):
            lines.insert(int(amap[b, j]) + j, "A")
        want = np.array([ex.LINE_ACTION if s == "A" else ex.LINE_TRAJ for s in lines], dtype=np.uint8)
        assert np.array_equal(kinds[pl[b]:pl[b + 1]], want), b
        n_act += n_maps[b, 1]
    assert n_act > 100


@pytest.mark.gpu
def test_reference_saved_files_parse():
    """The two files the reference saved itself: every token of a trajectory row parses to float() of the token, the
    line kinds follow the first token, and nothing is flagged."""
    from golden_util import GOLDEN_DIR
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    bodies = [gzip.open(os.path.join(GOLDEN_DIR, f"save_txt_{n}.txt.gz"), "rb").read()
              for n in ("turn_reverse_wait", "node0_wait")]
    offs = np.cumsum([0] + [len(b) for b in bodies])
    eng = Engine("cuda:0")
    p = ex.parse_text_batch(eng, b"".join(bodies), offs)
    assert p.n_host == 0 and int((p.line_errors != 0).sum()) == 0
    rows, kinds = p.rows.cpu().numpy(), p.line_kinds.cpu().numpy()
    want_rows, want_kinds = [], []
    for body in bodies:
        for line in body.decode().splitlines():
            t = line.split()
            want_kinds.append(ex.LINE_TRAJ if t[0] == "0" else ex.LINE_ACTION)
            if t[0] == "0":
                assert len(t) == 7
                want_rows.append([float(v) for v in t])
    assert kinds.tolist() == want_kinds and ex.LINE_ACTION in want_kinds
    assert rows.shape == (len(want_rows), 7)
    assert np.array_equal(rows.view(np.int64), np.array(want_rows).view(np.int64))
    assert p.path_line_offsets.cpu().tolist() == [0, bodies[0].count(b"\n"), len(want_kinds)]


def _route_folder(eng, rdir, half):
    """Write to rdir the GUI reference routes that the save accepts and that profile at the factory constraints and
    at `half`; returns {file name: [t_end at the factory constraints, t_end at half]}."""
    from test_next_rows import _gui_ref
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.packing import pack_paths
    from vexautonomousplanner_b200.synth import FACTORY
    rdir.mkdir()
    t_end = {}
    for n, r in _gui_ref().items():
        if "built" not in r:
            continue
        pts, nodes, aps, _ = ex.load_nodes(r["built"]["json"])
        if not (len(nodes) > 2 and any(x.is_start_node for x in nodes) and any(x.is_end_node for x in nodes)):
            continue
        res = [eng.profile(eng.upload(pack_paths([(ex.px_points_to_ft(pts), nodes, aps)], c))) for c in (FACTORY, half)]
        if all(int(x.status[0]) == 0 for x in res):
            (rdir / f"{n}.txt").write_text(r["built"]["json"])
            t_end[f"{n}.txt"] = [float(x.summary[0, 2]) for x in res]
    return t_end


def _reader_lines(names, odir, fresh_dir):
    """{name: the report line of the reader's comparison of odir/name with fresh_dir/name}."""
    from test_check_vs_reference import ref_body, ref_compare
    from vexautonomousplanner_b200 import save_routes as sr
    out = {}
    for n in names:
        new = (fresh_dir / n).read_bytes()
        out[n] = sr.check_line(n, *ref_compare((odir / n).read_bytes(), new, ref_body(new)[0]))[1]
    return out


@pytest.mark.gpu
def test_check_command_on_a_folder(tmp_path, capsys):
    """save, then --check: every route up to date (exit 0); with --max-velocity halved every route is stale, with the
    fresh profile's t_end as the new duration and the first run's as the old one; a deleted file is missing, a
    corrupted token unreadable with its line (exit 1).  Every stale and unreadable line is the one the Python reader
    of test_check_vs_reference gives for the saved file and the fresh body."""
    from vexautonomousplanner_b200 import save_routes as sr
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.synth import FACTORY
    eng = Engine("cuda:0")
    half = (FACTORY[0] / 2,) + tuple(FACTORY[1:])
    rdir, odir, hdir = tmp_path / "routes", tmp_path / "out", tmp_path / "half"
    t_end = _route_folder(eng, rdir, half)
    names = sorted(t_end)
    assert len(names) >= 4
    assert all(t[1] > t[0] for t in t_end.values())
    base = [str(rdir), str(odir), "--tile-paths", "3"]
    assert sr.main(base) == 0
    assert sr.main([str(rdir), str(hdir), "--tile-paths", "3", "--max-velocity", str(half[0])]) == 0
    capsys.readouterr()
    assert sr.main(base + ["--check"]) == 0
    out = capsys.readouterr().out
    assert all(f"up to date: {n}" in out for n in names), out

    assert sr.main(base + ["--check", "--max-velocity", str(half[0])]) == 1
    out = capsys.readouterr().out.splitlines()
    stale = [line for line in out if line.startswith("stale: ")]
    assert len(stale) == len(names), out
    want = _reader_lines(names, odir, hdir)
    for line in stale:
        name = line.split(": ")[1]
        assert line == want[name]
        dur = line.split("; duration ")[1].split(" s;")[0].split(" -> ")
        assert [float(v) for v in dur] == t_end[name], line

    gone = names[0]
    (odir / gone).unlink()
    bad = names[1]
    fresh = tmp_path / "fresh"
    fresh.mkdir()
    (fresh / bad).write_bytes((odir / bad).read_bytes())
    lines = (odir / bad).read_text().splitlines(keepends=True)
    k = next(i for i, l in enumerate(lines) if l.startswith("0 ") and i > 5)
    tok = lines[k].split(" ")
    tok[3] = tok[3] + "x"
    lines[k] = " ".join(tok)
    (odir / bad).write_text("".join(lines))
    before = {p.name: p.read_bytes() for p in odir.iterdir()}
    assert sr.main(base + ["--check"]) == 1
    out = capsys.readouterr().out
    assert f"missing: {gone}" in out
    assert f"unreadable: {bad}: line {k + 1}: token 4 (y) is not a number" in out, out
    assert _reader_lines([bad], odir, fresh)[bad] in out.splitlines()
    assert all(f"up to date: {n}" in out for n in names[2:]), out
    assert {p.name: p.read_bytes() for p in odir.iterdir()} == before

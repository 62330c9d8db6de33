"""Two robots running two routes at the same time: export.pair_check (csrc/vap_pairs.cuh) against a plain numpy
reference, and the pair_check command built on it."""
import math
import os

import numpy as np
import pytest

EPS = 1e-9          # inches: how far the device's values may be from the reference's


# ----------------------------------------------------------------------------------------------- numpy reference
def _seg_d2(px, py, ax, ay, bx, by):
    """Squared distance from points (px, py) to segments a-b (broadcast)."""
    ex, ey = bx - ax, by - ay
    wx, wy = px - ax, py - ay
    t = np.clip((wx * ex + wy * ey) / (ex * ex + ey * ey), 0.0, 1.0)
    dx, dy = wx - t * ex, wy - t * ey
    return dx * dx + dy * dy


def ref_corners(x, y, h, hl, hw):
    """Corners [n, 4] in polygon order: (x + a cos h - b sin h, y + a sin h + b cos h)."""
    c, s = np.cos(h)[:, None], np.sin(h)[:, None]
    a = np.array([hl, hl, -hl, -hl])[None]
    b = np.array([hw, -hw, -hw, hw])[None]
    return x[:, None] + a * c - b * s, y[:, None] + a * s + b * c


def ref_distance(pa, pb, ha, hb):
    """Signed distance of robot A at poses pa = (x, y, h) arrays (half-sizes ha = (hl, hw)) and robot B at pb: with
    overlap on all four separating axes minus the smallest overlap, else the minimum over vertex-edge pairs both ways."""
    ax, ay = ref_corners(*pa, *ha)
    bx, by = ref_corners(*pb, *hb)
    over = []
    for h in (pa[2], pb[2]):
        c, s = np.cos(h)[:, None], np.sin(h)[:, None]
        for ux, uy in ((c, s), (-s, c)):
            qa, qb = ax * ux + ay * uy, bx * ux + by * uy
            over.append(np.minimum(qa.max(axis=1), qb.max(axis=1)) - np.maximum(qa.min(axis=1), qb.min(axis=1)))
    over = np.stack(over, axis=1)
    inside = (over > 0).all(axis=1)
    d2 = np.full(ax.shape[0], np.inf)
    for e in range(4):
        f = (e + 1) % 4
        for (px, py), (qx, qy) in (((ax, ay), (bx, by)), ((bx, by), (ax, ay))):
            d2 = np.minimum(d2, _seg_d2(px, py, qx[:, e:e + 1], qy[:, e:e + 1], qx[:, f:f + 1], qy[:, f:f + 1]).min(axis=1))
    return np.where(inside, -over.min(axis=1), np.sqrt(d2))


def ref_bad(rows):
    """(row, reason) of a route: (-1, 0) valid, (-1, 1) no rows, (r, 2) first non-finite row, (r, 3) t decreases."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 7)
    if rows.shape[0] == 0:
        return -1, 1
    nonfin = ~np.isfinite(rows[:, 1:5]).all(axis=1)
    dec = np.zeros(rows.shape[0], dtype=bool)
    dec[1:] = rows[1:, 1] < rows[:-1, 1]
    bad = nonfin | dec
    if not bad.any():
        return -1, 0
    r = int(np.argmax(bad))
    return r, 2 if nonfin[r] else 3


def ref_step(rows, hl, hw):
    if rows.shape[0] < 2:
        return 0.0
    cx, cy = ref_corners(rows[:, 2], rows[:, 3], rows[:, 4], hl, hw)
    return float(np.sqrt((cx[1:] - cx[:-1]) ** 2 + (cy[1:] - cy[:-1]) ** 2).max())


def ref_pair(ra, rb, ha, hb, gap):
    """One pair's (ints by PC_I, floats by PC_F, per-event data): events are the rows of either route, the other
    robot held at np.searchsorted(t_other, t, side="right") - 1, clamped to its first row."""
    ra, rb = np.asarray(ra, dtype=np.float64).reshape(-1, 7), np.asarray(rb, dtype=np.float64).reshape(-1, 7)
    ba, bb = ref_bad(ra), ref_bad(rb)
    if ba[1] or bb[1]:
        st = 1 if ba[1] else 2
        return [st, 0, -1, -1, 0, -1, -1], [np.nan, np.inf, np.nan, np.nan, np.nan, 0.0], None
    ta, tb = ra[:, 1], rb[:, 1]
    ja = np.maximum(np.searchsorted(tb, ta, side="right") - 1, 0)       # B's held row at A's events
    jb = np.maximum(np.searchsorted(ta, tb, side="right") - 1, 0)
    pose = lambda r, idx: (r[idx, 2], r[idx, 3], r[idx, 4])
    ia, ib = np.arange(ra.shape[0]), np.arange(rb.shape[0])
    d = np.concatenate([ref_distance(pose(ra, ia), pose(rb, ja), ha, hb), ref_distance(pose(ra, jb), pose(rb, ib), ha, hb)])
    t = np.concatenate([ta, tb])
    side = np.concatenate([np.zeros(ra.shape[0], dtype=np.int64), np.ones(rb.shape[0], dtype=np.int64)])
    row = np.concatenate([ia, ib])
    order = np.lexsort((row, side, t))                                  # by (t, side, row)
    contact = d < gap
    first = next((int(k) for k in order if contact[k]), -1)
    near = int(order[np.argmin(d[order])])                             # the smallest key among equal minima
    ints = [0, len(t), int(side[first]) if first >= 0 else -1, int(row[first]) if first >= 0 else -1,
            int(contact.sum()), int(side[near]), int(row[near])]
    floats = [t[first] if first >= 0 else np.nan, d[near], t[near], ta[-1], tb[-1],
              max(ref_step(ra, *ha), ref_step(rb, *hb))]
    return ints, floats, dict(d=d, t=t, side=side, row=row)


def assert_matches(gi, gf, ref, gap, where=""):
    """Device result of one pair against ref_pair's: integers exactly, except where an event's distance is within EPS of
    min_gap (then the device's first contact must be one of the undecided or decided contacts, with no decided contact
    keyed before it); floats within EPS."""
    ri, rf, e = ref
    assert gi[0] == ri[0], (where, gi, ri)
    if e is None:
        assert list(gi) == ri and np.isnan(gf[[0, 2, 3, 4]]).all() and gf[1] == np.inf and gf[5] == 0.0, (where, gi, gf)
        return
    assert gi[1] == ri[1], where
    d, t, side, row = e["d"], e["t"], e["side"], e["row"]
    idx = {(int(s), int(r)): k for k, (s, r) in enumerate(zip(side, row))}
    undecided = np.abs(d - gap) <= EPS
    assert abs(gi[4] - ri[4]) <= undecided.sum(), (where, gi, ri)
    if not undecided.any():
        assert gi[2:5].tolist() == ri[2:5], (where, gi, ri)
    elif gi[3] != ri[3] or gi[2] != ri[2]:
        k = idx[(int(gi[2]), int(gi[3]))]
        assert d[k] < gap + EPS, (where, gi, ri)
        decided = (d < gap) & ~undecided
        before = (t < t[k]) | ((t == t[k]) & ((side < side[k]) | ((side == side[k]) & (row < row[k]))))
        assert not (decided & before).any(), (where, gi, ri)
    if gi[2] >= 0:
        assert gf[0] == t[idx[(int(gi[2]), int(gi[3]))]], where
    else:
        assert np.isnan(gf[0]), where
    k = idx[(int(gi[5]), int(gi[6]))]
    assert d[k] <= rf[1] + EPS and abs(gf[1] - rf[1]) <= EPS and gf[2] == t[k], (where, gi, gf, ri, rf)
    assert gf[3] == rf[3] and gf[4] == rf[4], where
    assert abs(gf[5] - rf[5]) <= EPS, (where, gf[5], rf[5])


# ------------------------------------------------------------------------------------------------------------- CPU
def _line(x0, vx, y0, vy, h, n, dt=1 / 16):
    """n rows of a robot driving at a constant velocity from (x0, y0) at heading h, from t = 0."""
    r = np.zeros((n, 7))
    k = np.arange(n)
    r[:, 1] = k * dt
    r[:, 2] = x0 + vx * k * dt
    r[:, 3] = y0 + vy * k * dt
    r[:, 4] = h
    return r


def test_reference_head_on_cpu():
    """Two 12 x 12 robots driving head-on along y = 0 at 32 and 16 in/s from x = -60 and x = 60 (a row every 1/16 s,
    all exact): their faces touch when the centres are 12 in apart, at t = (120 - 12) / 48 = 2.25 s, which is not a
    contact; the next rows overlap.  With a 2 in gap the contact starts at the first row under 14 in, 2.25 s."""
    a = _line(-60.0, 32.0, 0.0, 0.0, 0.0, 81)
    b = _line(60.0, -16.0, 0.0, 0.0, 0.0, 81)        # driving backwards: heading 0 is the same rectangle as pi
    ints, floats, e = ref_pair(a, b, (6.0, 6.0), (6.0, 6.0), 0.0)
    assert ints[:4] == [0, 162, 0, 37] and floats[0] == 37 / 16
    k = np.where((e["side"] == 0) & (e["row"] == 36))[0][0]
    assert e["d"][k] == 0.0 and e["t"][k] == 2.25
    ints, floats, _ = ref_pair(a, b, (6.0, 6.0), (6.0, 6.0), 2.0)
    assert ints[:4] == [0, 162, 0, 36] and floats[0] == 2.25
    assert floats[5] == 2.0                                           # A's corners move 2 in per row
    assert floats[1] == -12.0 and ints[5:] == [0, 40]                 # both centred on x = 20 at row 40


def test_reference_same_pose_and_diamond_cpu():
    """Aligned robots at one pose: penetration 2 min(hl_a, hl_b, hw_a, hw_b); a diamond against a square: the
    corner-to-edge distance; swapping the robots gives the same distance."""
    z = np.zeros(1)
    p = (z, z, z)
    d = ref_distance(p, p, (9.0, 7.5), (6.0, 8.0))
    assert abs(d[0] + 2 * 6.0) < 1e-12
    diamond = (z, z, z + math.pi / 4)                                  # 2 x 2 at 45 degrees: corner at sqrt 2
    square = (z + 4.0, z, z)                                           # 2 x 2 centred at x = 4: edge at x = 3
    r2 = math.sqrt(2.0)
    assert abs(ref_distance(diamond, square, (1.0, 1.0), (1.0, 1.0))[0] - (3.0 - r2)) < 1e-12
    assert abs(ref_distance(square, diamond, (1.0, 1.0), (1.0, 1.0))[0] - (3.0 - r2)) < 1e-12
    assert ref_bad(np.zeros((0, 7))) == (-1, 1)
    r = _line(0.0, 1.0, 0.0, 0.0, 0.0, 5)
    assert ref_bad(r) == (-1, 0)
    r[3, 4] = np.nan
    assert ref_bad(r) == (3, 2)
    r[3, 4], r[2, 1] = 0.0, -1.0
    assert ref_bad(r) == (2, 3)


def test_cabi_argument_errors_cpu():
    """Argument errors come back < 0 with text before anything touches the device."""
    import ctypes as C
    import vexautonomousplanner_b200 as vap
    from vexautonomousplanner_b200 import _lib
    vap.build()
    L = _lib.lib()
    pairs = (C.c_int64 * 2)(0, 0)

    def call(P=1, pairs=pairs, hl_a=1.0, hw_a=1.0, hl_b=1.0, hw_b=1.0, gap=0.0, B_a=1, B_b=1):
        return L.vap_pair_check(C.c_int64(P), pairs, C.c_int64(B_a), None, C.c_int64(0), None, None, C.c_double(hl_a),
                                C.c_double(hw_a), C.c_int64(B_b), None, C.c_int64(0), None, None, C.c_double(hl_b),
                                C.c_double(hw_b), C.c_double(gap), None, None, None)
    for kw, text in ((dict(P=-1), "P >= 0"), (dict(B_b=-2), "B_b >= 0"), (dict(pairs=None), "pairs is NULL"),
                     (dict(hl_a=0.0), "half-length"), (dict(hw_a=-1.0), "half-length"), (dict(hl_b=float("inf")), "half"),
                     (dict(hw_b=float("nan")), "half"), (dict(gap=float("nan")), "min_gap"), (dict(gap=float("-inf")), "min_gap")):
        rc = call(**kw)
        assert rc < 0, kw
        assert text in L.vap_last_error().decode(), (kw, L.vap_last_error())
    assert call(P=0, pairs=None) == 0                                  # nothing to do, nothing launched
    assert L.vap_pose_planes(C.c_int64(-1), None, None, C.c_int64(0), None, None, None) < 0
    assert "B >= 0" in L.vap_last_error().decode()
    assert L.vap_pose_planes(C.c_int64(0), None, None, C.c_int64(0), None, None, None) == 0


def test_pair_check_arguments_cpu(tmp_path, capsys):
    """L,W parsing and its errors, B's size defaulting to A's, unordered pairs for one folder, exit 2."""
    from vexautonomousplanner_b200 import pair_check as pc
    a = pc.parse_args(["x", "y", "--robot-a-in", "18,15"])
    assert a.size_a == (18.0, 15.0) and a.size_b == (18.0, 15.0) and a.min_gap == 0.0
    a = pc.parse_args(["x", "y", "--robot-a-in", "18,15", "--robot-b-in", "1.5e1,12", "--min-gap-in", "2"])
    assert a.size_b == (15.0, 12.0) and a.min_gap == 2.0
    for bad in ("18", "18,15,3", "a,b", "0,15", "18,-1", "inf,3", "nan,3", ""):
        with pytest.raises(SystemExit) as e:
            pc.parse_args(["x", "y", "--robot-a-in", bad])
        assert e.value.code == 2, bad
    for bad in ([], ["--robot-a-in", "18,15", "--min-gap-in", "inf"], ["--robot-a-in", "18,15", "--robot-b-in", "3"]):
        with pytest.raises(SystemExit) as e:
            pc.parse_args(["x", "y"] + bad)
        assert e.value.code == 2, bad
    assert pc.pairs_of(3, 3, True) == [(0, 1), (0, 2), (1, 2)]
    assert pc.pairs_of(2, 3, False) == [(0, 0), (0, 1), (0, 2), (1, 0), (1, 1), (1, 2)]
    assert pc.pairs_of(1, 1, True) == []
    capsys.readouterr()
    empty, full = tmp_path / "empty", tmp_path / "full"
    empty.mkdir(), full.mkdir()
    (empty / "notes.md").write_text("x")
    (full / "r.txt").write_text("0 0 0 0 0 0 0\n")
    assert pc.main([str(empty), str(full), "--robot-a-in", "18,15"]) == 2
    assert "no trajectory .txt files" in capsys.readouterr().err
    assert pc.main([str(full), str(tmp_path / "missing"), "--robot-a-in", "18,15"]) == 2


def _arrays(status=0, events=600, fs=-1, fr=-1, n=0, ns=1, nr=40, ft=float("nan"), nd=7.25, nt=1.2, la=2.5, lb=3.0,
            step=0.45):
    from vexautonomousplanner_b200.export import PC_F, PC_I
    ints = np.array([status, events, fs, fr, n, ns, nr], dtype=np.int64)
    floats = np.array([ft, nd, nt, la, lb, step])
    assert len(ints) == len(PC_I) and len(floats) == len(PC_F)
    return ints, floats


def test_pair_check_report_lines_cpu():
    """The report line of each state from given arrays."""
    from vexautonomousplanner_b200.pair_check import report_line
    ok = (-1, 0)
    assert report_line("a.txt", "b.txt", *_arrays(), ok, ok) == (
        "clear", "clear: a.txt x b.txt: closest 7.250 in at t 1.200 s; A ends at 2.500 s, B at 3.000 s; "
                 "sampling step <= 0.450 in")
    assert report_line("a.txt", "b.txt", *_arrays(fs=1, fr=17, n=9, ft=0.85, nd=-1.5, ns=0, nt=1.0), ok, ok) == (
        "contact", "contact: a.txt x b.txt: first at t 0.850 s (B row 17); closest -1.500 in at t 1.000 s; 9 of 600 events")
    assert report_line("a.txt", "b.txt", *_arrays(fs=0, fr=3, n=1, ft=0.03, nd=1.0), ok, ok)[1].startswith(
        "contact: a.txt x b.txt: first at t 0.030 s (A row 3); closest 1.000 in")
    bad = dict(status=1, events=0, ns=-1, nr=-1, nd=np.inf, nt=np.nan, la=np.nan, lb=np.nan, step=0.0)
    assert report_line("a.txt", "b.txt", *_arrays(**bad), (4, 2), ok) == (
        "not checked", "not checked: a.txt x b.txt: a.txt: row 4 is not finite")
    assert report_line("a.txt", "b.txt", *_arrays(**{**bad, "status": 2}), ok, (7, 3))[1] == (
        "not checked: a.txt x b.txt: b.txt: t decreases at row 7")
    assert report_line("a.txt", "b.txt", *_arrays(**bad), (-1, 1), ok)[1] == (
        "not checked: a.txt x b.txt: a.txt: no trajectory rows")


# ------------------------------------------------------------------------------------------------------------- GPU
def _random_rows(rng, B, box=40.0):
    """B routes with strictly increasing t: random walks within +-box in, every fourth much shorter than the rest so
    that the parked pose matters; headings turning, some runs in place."""
    rows, off = [], [0]
    for b in range(B):
        n = int(rng.integers(1, 40)) if b % 4 == 0 else int(rng.integers(200, 1500))
        t = np.cumsum(rng.uniform(0.005, 0.02, n)) - 0.005
        x = rng.uniform(-box, box) + np.cumsum(rng.normal(0, 0.3, n))
        y = rng.uniform(-box, box) + np.cumsum(rng.normal(0, 0.3, n))
        h = rng.uniform(-4, 4) + np.cumsum(rng.normal(0, 0.03, n))
        if n > 30:
            k = int(rng.integers(0, n - 20))
            x[k:k + 20], y[k:k + 20] = x[k], y[k]
        r = np.zeros((n, 7))
        r[:, 1], r[:, 2], r[:, 3], r[:, 4] = t, x, y, h
        r[:, 5] = rng.uniform(0, 50, n)
        rows.append(r)
        off.append(off[-1] + n)
    return np.concatenate(rows), np.array(off, dtype=np.int64)


def _route(rows, off, b):
    return rows[off[b]:off[b + 1]]


@pytest.mark.gpu
def test_random_cross_products_match_numpy():
    """24 x 20 random routes, unequal robots, min_gap 0 and 2, against numpy; swapping the sides swaps only the labels;
    two runs are bit-identical; the same set on both sides builds its planes once and matches."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rng = np.random.default_rng(17)
    ra, oa = _random_rows(rng, 24)
    rb, ob = _random_rows(rng, 20)
    pairs = np.array([(i, j) for i in range(24) for j in range(20)], dtype=np.int64)
    sa, sb = (18.0, 15.0), (18.0, 18.0)
    contacts = 0
    for gap in (0.0, 2.0):
        gi, gf, ba, bb = ex.pair_check(eng, ra, oa, sa, rb, ob, sb, pairs, gap)
        assert (ba == [-1, 0]).all() and (bb == [-1, 0]).all() and ba.shape == (24, 2) and bb.shape == (20, 2)
        for k, (i, j) in enumerate(pairs):
            ref = ref_pair(_route(ra, oa, i), _route(rb, ob, j), (9.0, 7.5), (9.0, 9.0), gap)
            assert_matches(gi[k], gf[k], ref, gap, where=(gap, i, j))
        contacts += int((gi[:, 2] >= 0).sum())
        gi2, gf2, _, _ = ex.pair_check(eng, ra, oa, sa, rb, ob, sb, pairs, gap)
        assert np.array_equal(gi, gi2) and np.array_equal(gf.view(np.int64), gf2.view(np.int64))
        si, sf, _, _ = ex.pair_check(eng, rb, ob, sb, ra, oa, sa, pairs[:, ::-1], gap)
        assert np.array_equal(si[:, [0, 1, 4]], gi[:, [0, 1, 4]])
        for c in (0, 1, 2, 5):
            assert np.array_equal(sf[:, c].view(np.int64), gf[:, c].view(np.int64)), c
        assert np.array_equal(sf[:, 3], gf[:, 4]) and np.array_equal(sf[:, 4], gf[:, 3])
        hit = gi[:, 2] >= 0
        assert np.array_equal(si[hit, 2], 1 - gi[hit, 2]) and np.array_equal(si[hit, 3], gi[hit, 3])
        same = np.array([(i, j) for i in range(24) for j in range(i + 1, 24)], dtype=np.int64)
        mi, mf, ma, mb = ex.pair_check(eng, ra, oa, sa, ra, oa, sa, same, gap)
        assert ma is mb
        for k in range(0, len(same), 7):
            i, j = same[k]
            assert_matches(mi[k], mf[k], ref_pair(_route(ra, oa, i), _route(ra, oa, j), (9.0, 7.5), (9.0, 7.5), gap),
                           gap, where=("same", gap, i, j))
    assert 50 < contacts < 2 * len(pairs) - 50, contacts


@pytest.mark.gpu
def test_one_row_set_with_two_offset_arrays():
    """The first routes of one row set as side A and the rest as side B (the same rows object, two offset arrays): the
    results equal those of two separate row sets bit for bit and match numpy; B's routes and their validity come from
    B's offsets."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rng = np.random.default_rng(23)
    ra, oa = _random_rows(rng, 12)
    rb, ob = _random_rows(rng, 9)
    rows = np.concatenate([ra, rb])
    off = np.concatenate([oa, ob[1:] + oa[-1]])
    pairs = np.array([(i, j) for i in range(12) for j in range(9)], dtype=np.int64)
    gi, gf, ba, bb = ex.pair_check(eng, ra, oa, (18.0, 15.0), rb, ob, (18.0, 18.0), pairs, 2.0)
    si, sf, sa, sb = ex.pair_check(eng, rows, off[:13], (18.0, 15.0), rows, off[12:], (18.0, 18.0), pairs, 2.0)
    assert (gi[:, 0] == 0).all() and sa.shape == (12, 2) and sb.shape == (9, 2) and (sb == [-1, 0]).all()
    assert np.array_equal(si, gi) and np.array_equal(sf.view(np.int64), gf.view(np.int64))
    for k in range(0, len(pairs), 5):
        i, j = pairs[k]
        assert_matches(si[k], sf[k], ref_pair(_route(ra, oa, i), _route(rb, ob, j), (9.0, 7.5), (9.0, 9.0), 2.0), 2.0,
                       where=(i, j))


@pytest.mark.gpu
def test_parked_robot_is_hit_after_its_last_row():
    """A finishes at 1.125 s, parked at the origin across B's path; B drives up through it from y = -80.5 at 32 in/s
    and first overlaps at its row 35 (y = -10.5), at 2.1875 s."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    a = _line(-18.0, 16.0, 0.0, 0.0, 0.0, 19)
    b = _line(0.0, 0.0, -80.5, 32.0, math.pi / 2, 81)
    rows = np.concatenate([a, b])
    gi, gf, _, _ = ex.pair_check(eng, rows, [0, 19, 100], (12.0, 12.0), rows, [0, 19, 100], (12.0, 12.0), [(0, 1)])
    assert_matches(gi[0], gf[0], ref_pair(a, b, (6.0, 6.0), (6.0, 6.0), 0.0), 0.0)
    assert gi[0, 2:4].tolist() == [1, 35] and gf[0, 0] == 35 / 16 and gf[0, 3] == 1.125
    assert abs(gf[0, 1] + 11.5) < 1e-9                               # deepest at y = -0.5 (row 40): 12 - 0.5


@pytest.mark.gpu
def test_invalid_routes_and_empty_launches():
    """A NaN heading, a decreasing t, an empty route and an index out of range give their status and reason; the other
    pairs of the launch are unaffected.  P = 0 and empty row sets return empty arrays."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    good = _line(-40.0, 10.0, 0.0, 0.0, 0.0, 128)
    nanh = _line(0.0, 0.0, -40.0, 10.0, math.pi / 2, 200)
    nanh[57, 4] = np.nan
    dec = _line(0.0, 0.0, -40.0, 10.0, math.pi / 2, 200)
    dec[120, 1] = dec[118, 1]
    other = _line(0.0, 0.0, -40.0, 10.0, math.pi / 2, 200)
    ra, oa = good, np.array([0, 128])
    rb = np.concatenate([nanh, dec, other])
    ob = np.array([0, 200, 400, 400, 600])                              # route 2 is empty
    pairs = [(0, 0), (0, 1), (0, 2), (0, 3), (0, 4), (1, 3), (-1, 3)]
    gi, gf, ba, bb = ex.pair_check(eng, ra, oa, (12.0, 12.0), rb, ob, (12.0, 12.0), pairs)
    assert ba.tolist() == [[-1, 0]] and bb.tolist() == [[57, 2], [120, 3], [-1, 1], [-1, 0]]
    assert gi[:, 0].tolist() == [2, 2, 2, 0, 3, 3, 3]
    for k in (0, 1, 2, 4, 5, 6):
        assert gi[k, 1:].tolist() == [0, -1, -1, 0, -1, -1] and gf[k, 1] == np.inf and np.isnan(gf[k, [0, 2, 3, 4]]).all()
    assert_matches(gi[3], gf[3], ref_pair(good, other, (6.0, 6.0), (6.0, 6.0), 0.0), 0.0)
    assert gi[3, 2] >= 0
    assert [ex.pair_reason_text(*r) for r in bb] == ["row 57 is not finite", "t decreases at row 120",
                                                     "no trajectory rows", "valid"]
    gi, gf, ba, bb = ex.pair_check(eng, rb, ob, (12.0, 12.0), ra, oa, (12.0, 12.0), [(1, 0)])
    assert gi[0, 0] == 1
    # finite coordinates whose differences overflow: the distance is garbage but never NaN, so the nearest event is set
    far = _line(1.5e308, 0.0, -1.5e308, 0.0, 0.75, 4)
    near = _line(-1.5e308, 0.0, 1.5e308, 0.0, 0.75, 3)
    gi, gf, _, _ = ex.pair_check(eng, far, [0, 4], (12.0, 12.0), near, [0, 3], (12.0, 12.0), [(0, 0)])
    assert gi[0, 0] == 0 and gi[0, 1] == 7 and gi[0, 5] in (0, 1) and 0 <= gi[0, 6] < 4 and not np.isnan(gf[0, 1])
    gi, gf, ba, bb = ex.pair_check(eng, ra, oa, (12.0, 12.0), rb, ob, (12.0, 12.0), np.zeros((0, 2), dtype=np.int64))
    assert gi.shape == (0, 7) and gf.shape == (0, 6) and ba.shape == (1, 2) and bb.shape == (4, 2)
    gi, gf, ba, bb = ex.pair_check(eng, np.zeros((0, 7)), [0, 0], (12.0, 12.0), np.zeros((0, 7)), [0, 0, 0], (9.0, 9.0),
                                   [(0, 1)])
    assert gi[:, 0].tolist() == [1] and ba.tolist() == [[-1, 1]] and bb.tolist() == [[-1, 1], [-1, 1]]
    gi, gf, ba, bb = ex.pair_check(eng, np.zeros((0, 7)), [0], (12.0, 12.0), np.zeros((0, 7)), [0], (9.0, 9.0), [])
    assert gi.shape == (0, 7) and ba.shape == (0, 2) and bb.shape == (0, 2)
    from vexautonomousplanner_b200._lib import VapError
    for kw, text in ((dict(size_a=(0.0, 12.0)), "half-length"), (dict(size_b=(12.0, float("inf"))), "half"),
                     (dict(min_gap_in=float("nan")), "min_gap")):
        args = dict(size_a=(12.0, 12.0), size_b=(12.0, 12.0), min_gap_in=0.0)
        args.update(kw)
        with pytest.raises(VapError, match=text):
            ex.pair_check(eng, ra, oa, args["size_a"], rb, ob, args["size_b"], [(0, 3)], args["min_gap_in"])


@pytest.mark.gpu
def test_fresh_and_saved_rows_match():
    """64 x 64 of synth.mixed_paths through export_rows against numpy, and the same batch through save_text_batch ->
    parse_text_batch gives bit-identical outputs."""
    from test_trajectory_check import _mixed_batch
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    packed, na, aa = _mixed_batch(128, 3)
    db = eng.upload(packed)
    res = eng.profile(db)
    rows, off = ex.export_rows(eng, res)
    pairs = np.array([(i, 64 + j) for i in range(64) for j in range(64)], dtype=np.int64)
    gi, gf, ba, bb = ex.pair_check(eng, rows, off, (18.0, 15.0), rows, off, (18.0, 18.0), pairs, 1.0)
    assert ba is bb
    r, o = rows.cpu().numpy(), off.cpu().numpy()
    for k in range(0, len(pairs), 13):
        i, j = pairs[k]
        assert_matches(gi[k], gf[k], ref_pair(_route(r, o, i), _route(r, o, j), (9.0, 7.5), (9.0, 9.0), 1.0), 1.0,
                       where=(i, j))
    ok = res.status.cpu().numpy() == 0
    assert ((gi[:, 0] == 0) == (ok[pairs[:, 0]] & ok[pairs[:, 1]])).all()
    assert int((gi[:, 2] >= 0).sum()) > 20
    text, offs, _ = ex.save_text_batch(eng, res, db, na, aa)
    p = ex.parse_text_batch(eng, text, offs)
    pi, pf, pa, pb = ex.pair_check(eng, p.rows, p.row_offsets, (18.0, 15.0), p.rows, p.row_offsets, (18.0, 18.0), pairs, 1.0)
    assert np.array_equal(pi, gi) and np.array_equal(pf.view(np.int64), gf.view(np.int64)) and np.array_equal(pa, ba)


def _route_json(points_txt_in, wait0=0.0):
    """Node JSON of a route through the given .txt-frame points (JSON y is the negated .txt y), waiting wait0 s at
    its first node."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.export import RouteNode
    nodes = []
    for i in range(len(points_txt_in)):
        n = RouteNode()
        n.is_start_node, n.is_end_node = i == 0, i == len(points_txt_in) - 1
        n.wait_time = wait0 if i == 0 else 0
        nodes.append(n)
    return ex.nodes_to_json([(ex.in_to_px(x), ex.in_to_px(-y)) for x, y in points_txt_in], nodes)


A_PTS = [(-66.0, 0.0), (-30.0, 0.0), (0.0, 0.0), (30.0, 0.0)]          # along +x through the origin
B_PTS = [(0.0, -18.0), (0.0, 20.0), (0.0, 66.0)]                      # along +y through the origin


def _profile_rows(eng, *routes):
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.packing import pack_paths
    from vexautonomousplanner_b200.synth import FACTORY
    loaded = [ex.load_nodes(r) for r in routes]
    res = eng.profile(eng.upload(pack_paths([(ex.px_points_to_ft(pts), nodes, aps) for pts, nodes, aps, _ in loaded],
                                            FACTORY)))
    assert (res.status.cpu().numpy() == 0).all()
    rows, off = ex.export_rows(eng, res)
    return rows.cpu().numpy(), off.cpu().numpy()


def _band_entry(r, col, half):
    """First row time at which the centre coordinate col is within half of 0."""
    return r[np.argmax(np.abs(r[:, col]) < half), 1]


@pytest.mark.gpu
def test_crossing_routes_clear_as_saved_and_contact_with_a_wait():
    """Two 12 x 12 robots on straight routes crossing at right angles.  As profiled, B passes the crossing before A
    reaches it: clear, although a keep-out box around B's path would flag A.  A wait at B's first node that brings B to
    the crossing while A is in it: contact, first when both are in the band, within the sampling step."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rows, off = _profile_rows(eng, _route_json(A_PTS), _route_json(B_PTS))
    a, b = _route(rows, off, 0), _route(rows, off, 1)
    gi, gf, _, _ = ex.pair_check(eng, a, [0, len(a)], (12.0, 12.0), b, [0, len(b)], (12.0, 12.0), [(0, 0)])
    assert_matches(gi[0], gf[0], ref_pair(a, b, (6.0, 6.0), (6.0, 6.0), 0.0), 0.0)
    assert gi[0, 0] == 0 and gi[0, 2] == -1 and gf[0, 1] > 0, (gi, gf)
    box = [(-6.0, -18.0, 6.0, 66.0)]                                    # B's swept path as a static keep-out box
    fi, _ = ex.footprint_check(eng, a, [0, len(a)], 12.0, 12.0, keep_out=box)
    assert fi[0, 1] >= 0 and fi[0, 2] == ex.FP_KIND_BOX
    ta_in, tb_in = _band_entry(a, 2, 12.0), _band_entry(b, 3, 12.0)
    assert tb_in + 0.3 < ta_in
    wait = round(ta_in - tb_in + 0.2, 2)
    rows, off = _profile_rows(eng, _route_json(A_PTS), _route_json(B_PTS, wait0=wait))
    a, b = _route(rows, off, 0), _route(rows, off, 1)
    gi, gf, _, _ = ex.pair_check(eng, a, [0, len(a)], (12.0, 12.0), b, [0, len(b)], (12.0, 12.0), [(0, 0)])
    assert_matches(gi[0], gf[0], ref_pair(a, b, (6.0, 6.0), (6.0, 6.0), 0.0), 0.0)
    assert gi[0, 2] >= 0 and gf[0, 1] < 0, (gi, gf)
    window = max(_band_entry(a, 2, 12.0), _band_entry(b, 3, 12.0))    # the first row with both centres in the band
    assert abs(gf[0, 0] - window) <= 0.02, (gf[0, 0], window)


def _folders(tmp_path):
    """routes A (one route) and B (clear, contact, and one file made unreadable after saving), saved by save_routes."""
    from vexautonomousplanner_b200 import save_routes as sr
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rows, off = _profile_rows(eng, _route_json(A_PTS), _route_json(B_PTS))
    wait = round(_band_entry(_route(rows, off, 0), 2, 12.0) - _band_entry(_route(rows, off, 1), 3, 12.0) + 0.2, 2)
    ra, rb, sa, sb = (tmp_path / n for n in ("ra", "rb", "a", "b"))
    for d in (ra, rb):
        d.mkdir()
    (ra / "across.txt").write_text(_route_json(A_PTS))
    (rb / "early.txt").write_text(_route_json(B_PTS))
    (rb / "late.txt").write_text(_route_json(B_PTS, wait0=wait))
    (rb / "broken.txt").write_text(_route_json(B_PTS))
    assert sr.main([str(ra), str(sa)]) == 0 and sr.main([str(rb), str(sb)]) == 0
    body = (sb / "broken.txt").read_text()
    (sb / "broken.txt").write_text(body.replace("\n", "\nx\n", 1))
    return sa, sb


@pytest.mark.gpu
def test_pair_check_command_on_folders(tmp_path, capsys):
    """Clear, contact, unreadable and same-folder cases, the exit codes and the count line."""
    from vexautonomousplanner_b200 import pair_check as pc
    sa, sb = _folders(tmp_path)
    capsys.readouterr()
    assert pc.main([str(sa), str(sb), "--robot-a-in", "12,12"]) == 1
    out = capsys.readouterr().out.splitlines()
    assert len(out) == 4
    assert out[0] == "not checked: across.txt x broken.txt: broken.txt: line 2: the first token is neither 0 nor 1"
    assert out[1].startswith("clear: across.txt x early.txt: closest ") and "; A ends at " in out[1]
    assert "sampling step <= " in out[1]
    assert out[2].startswith("contact: across.txt x late.txt: first at t ") and " events" in out[2]
    assert out[3] == f"1 of 3 pairs clear (A {sa}, robot 12 x 12 in; B {sb}, robot 12 x 12 in; min gap 0 in)"
    assert pc.main([str(sb), str(sb) + os.sep, "--robot-a-in", "12,12", "--robot-b-in", "10,10"]) == 1
    out = capsys.readouterr().out.splitlines()
    assert [l.split(": ")[1] for l in out[:-1]] == ["broken.txt x early.txt", "broken.txt x late.txt", "early.txt x late.txt"]
    assert out[0].startswith("not checked: ") and out[1].startswith("not checked: ")
    assert out[2].startswith("contact: early.txt x late.txt: first at t 0.000 s (A row 0)")
    assert out[-1].startswith("0 of 3 pairs clear")
    (sb / "broken.txt").unlink()
    (sb / "late.txt").unlink()
    assert pc.main([str(sa), str(sb), "--robot-a-in", "12,12"]) == 0
    assert capsys.readouterr().out.splitlines()[-1].startswith("1 of 1 pairs clear")
    assert pc.main([str(sa), str(sb), "--robot-a-in", "12,12", "--min-gap-in", "100"]) == 1
    assert capsys.readouterr().out.startswith("contact: across.txt x early.txt: first at t 0.000 s (A row 0)")

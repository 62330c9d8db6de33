"""The robot's footprint along every route: export.footprint_check (csrc/vap_footprint.cuh) against a plain numpy
reference of the geometry, and the field_check command built on it."""
import json
import math
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-9          # inches: how far the device's values may be from the reference's


# ----------------------------------------------------------------------------------------------- numpy reference
def _seg_d2(px, py, ax, ay, bx, by):
    """Squared distance from points (px, py) to segments a-b (broadcast)."""
    ex, ey = bx - ax, by - ay
    wx, wy = px - ax, py - ay
    t = np.clip((wx * ex + wy * ey) / (ex * ex + ey * ey), 0.0, 1.0)
    dx, dy = wx - t * ex, wy - t * ey
    return dx * dx + dy * dy


def ref_rows(rows, hl, hw, field, boxes):
    """Per row: (finite[R], wall margin[R], box distance[R, K], corners cx[R, 4], cy[R, 4]) of the geometry in the
    header of vap_footprint.cuh, literally: corners (x + a cos h - b sin h, y + a sin h + b cos h), SAT on the four
    axes, else the minimum over vertex-edge pairs both ways."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 7)
    x, y, h = rows[:, 2], rows[:, 3], rows[:, 4]
    fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(h)
    x, y, h = np.where(fin, x, 0.0), np.where(fin, y, 0.0), np.where(fin, h, 0.0)
    c, s = np.cos(h)[:, None], np.sin(h)[:, None]
    a = np.array([hl, hl, -hl, -hl])[None]               # polygon order
    b = np.array([hw, -hw, -hw, hw])[None]
    cx = x[:, None] + a * c - b * s
    cy = y[:, None] + a * s + b * c
    xmin, xmax, ymin, ymax = field
    wall = np.maximum.reduce([xmin - cx, cx - xmax, ymin - cy, cy - ymax]).max(axis=1)
    dist = np.full((rows.shape[0], len(boxes)), np.inf)
    for k, (x0, y0, x1, y1) in enumerate(boxes):
        bxs, bys = np.array([x0, x1, x1, x0]), np.array([y0, y0, y1, y1])
        over = []
        for ax, ay in ((1.0, 0.0), (0.0, 1.0), (c, s), (-s, c)):
            pr = cx * ax + cy * ay
            pb = bxs[None] * ax + bys[None] * ay
            over.append(np.minimum(pr.max(axis=1), pb.max(axis=1)) - np.maximum(pr.min(axis=1), pb.min(axis=1)))
        over = np.stack(over, axis=1)
        inside = (over > 0).all(axis=1)
        d2 = np.inf
        for e in range(4):                                   # robot corners -> box edges, box corners -> robot edges
            f = (e + 1) % 4
            d2 = np.minimum(d2, _seg_d2(cx, cy, bxs[e], bys[e], bxs[f], bys[f]).min(axis=1))
            d2 = np.minimum(d2, _seg_d2(bxs[None], bys[None], cx[:, e:e + 1], cy[:, e:e + 1], cx[:, f:f + 1],
                                        cy[:, f:f + 1]).min(axis=1))
        dist[:, k] = np.where(inside, -over.min(axis=1), np.sqrt(d2))
    return fin, wall, dist, cx, cy


def ref_path(rows, hl, hw, field, boxes, tol):
    """One path's (ints by FP_I, floats by FP_F, per-row data for the tie checks)."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 7)
    n = rows.shape[0]
    fin, wall, dist, cx, cy = ref_rows(rows, hl, hw, field, boxes)
    K = len(boxes)
    kind = np.full(n, -1)
    boxviol = (dist < -tol) if K else np.zeros((n, 0), dtype=bool)
    if K:
        anybox = fin & boxviol.any(axis=1)
        kind[anybox] = 2 + np.argmax(boxviol, axis=1)[anybox]
    kind[fin & (wall > tol)] = 0
    kind[~fin] = 1
    viol = kind >= 0
    first = int(np.argmax(viol)) if viol.any() else -1
    wf = np.where(fin, wall, -np.inf)
    wr = int(np.argmax(wf)) if fin.any() else -1
    if K and fin.any():
        dd = np.where(fin[:, None], dist, np.inf)
        flat = int(np.argmin(dd))                            # row-major: lowest row, then lowest box
        nr, nk, nd = flat // K, flat % K, float(dd.flat[flat])
    else:
        nr, nk, nd = -1, -1, np.inf
    pair = fin[1:] & fin[:-1]
    step = np.sqrt((cx[1:] - cx[:-1]) ** 2 + (cy[1:] - cy[:-1]) ** 2).max(axis=1)[pair] if n > 1 else np.zeros(0)
    t = rows[:, 1]
    ints = [n, first, int(kind[first]) if first >= 0 else -1, int(viol.sum()), wr, nr, nk]
    floats = [t[first] if first >= 0 else np.nan, wf[wr] if wr >= 0 else -np.inf, t[wr] if wr >= 0 else np.nan, nd,
              t[nr] if nr >= 0 else np.nan, float(step.max()) if step.size else 0.0]
    return ints, floats, dict(fin=fin, wall=wall, dist=dist, viol=viol, kind=kind, t=t)


def ref_batch(rows, row_off, hl, hw, field, boxes, tol):
    rows = np.asarray(rows).reshape(-1, 7)
    out = [ref_path(rows[row_off[b]:row_off[b + 1]], hl, hw, field, boxes, tol) for b in range(len(row_off) - 1)]
    return out


def assert_matches(gi, gf, ref, tol, where=""):
    """Device result of one path against ref_path's: integers exactly, except where the reference's decisive margin
    is within EPS of tol (then the device's row must be one of the tied candidates); floats within EPS."""
    ri, rf, d = ref
    fin, wall, dist, viol = d["fin"], d["wall"], d["dist"], d["viol"]
    near = fin & ((np.abs(wall - tol) <= EPS) | (np.abs(dist + tol) <= EPS).any(axis=1))   # undecided rows
    assert gi[0] == ri[0], where
    assert abs(gi[3] - ri[3]) <= near.sum(), (where, gi[3], ri[3])
    if not near.any():
        assert gi[3] == ri[3] and gi[1] == ri[1] and gi[2] == ri[2], (where, gi, ri)
    elif gi[1] != ri[1]:
        g = gi[1]
        assert g >= 0 and (viol[g] or near[g]), (where, gi, ri)
        assert not (viol[:g] & ~near[:g]).any(), (where, gi, ri)
    # worst wall row: any row within EPS of the reference maximum
    assert (gi[4] < 0) == (ri[4] < 0), where
    if ri[4] >= 0:
        assert fin[gi[4]] and wall[gi[4]] >= rf[1] - EPS, (where, gi, ri)
        assert abs(gf[1] - rf[1]) <= EPS and gf[2] == d["t"][gi[4]], (where, gf, rf)
    else:
        assert gf[1] == -np.inf and np.isnan(gf[2])
    assert (gi[5] < 0) == (ri[5] < 0), where
    if ri[5] >= 0:
        g, k = gi[5], gi[6]
        assert fin[g] and dist[g, k] <= rf[3] + EPS, (where, gi, ri)
        assert abs(gf[3] - rf[3]) <= EPS and gf[4] == d["t"][g], (where, gf, rf)
    else:
        assert gi[6] == -1 and gf[3] == np.inf and np.isnan(gf[4])
    if gi[1] >= 0:
        assert gf[0] == d["t"][gi[1]]
    else:
        assert np.isnan(gf[0])
    assert abs(gf[5] - rf[5]) <= EPS, (where, gf[5], rf[5])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_reference_wall_margin_hand_cases_cpu():
    """A robot parallel to a wall at a known gap, and the same robot turned 90 degrees."""
    field = (-50.0, 50.0, -50.0, 50.0)
    rows = np.array([[0, 0.0, 0.0, 40.0, 0.0, 0, 0],               # 12 x 8 along x, 10 in from the top wall
                     [0, 0.1, 0.0, 40.0, math.pi / 2, 0, 0],       # turned: the half-length points at the wall
                     [0, 0.2, 0.0, 40.0, -math.pi, 0, 0],          # reversed: the same rectangle as heading 0
                     [0, 0.3, 45.0, 0.0, 0.0, 0, 0]])              # 1 in over the right wall
    fin, wall, dist, _, _ = ref_rows(rows, 6.0, 4.0, field, [])
    assert fin.all() and dist.shape == (4, 0)
    np.testing.assert_allclose(wall, [-6.0, -4.0, -6.0, 1.0], atol=1e-12)


def test_reference_box_distance_hand_cases_cpu():
    """Separation corner-to-edge and edge-to-corner, and the penetration depth of an overlap."""
    diamond = np.array([[0, 0.0, 0.0, 0.0, math.pi / 4, 0, 0]])   # 2 x 2 square at 45 degrees: corners at +-sqrt 2
    field = (-100.0, 100.0, -100.0, 100.0)
    r2 = math.sqrt(2.0)
    _, _, d, _, _ = ref_rows(diamond, 1.0, 1.0, field, [(3.0, -1.0, 5.0, 1.0)])        # robot corner -> box edge
    assert abs(d[0, 0] - (3.0 - r2)) < 1e-12
    _, _, d, _, _ = ref_rows(diamond, 1.0, 1.0, field, [(1.5, 1.5, 3.0, 3.0)])         # box corner -> robot edge
    assert abs(d[0, 0] - (3.0 - r2) / r2) < 1e-12
    flat = np.array([[0, 0.0, 0.0, 0.0, 0.0, 0, 0]])                                    # 4 x 2 along x
    _, _, d, _, _ = ref_rows(flat, 2.0, 1.0, field, [(1.5, -5.0, 5.0, 5.0), (2.0, 1.0, 3.0, 2.0), (-9.0, -3.0, 9.0, -2.0)])
    np.testing.assert_allclose(d[0], [-0.5, 0.0, 1.0], atol=1e-12)                      # penetration, touching, gap
    ints, floats, _ = ref_path(np.concatenate([flat, flat]), 2.0, 1.0, field, [(-9.0, -3.0, 9.0, -2.0), (1.5, -5.0, 5.0, 5.0)], 0.0)
    assert ints == [2, 0, 3, 2, 0, 0, 1] and floats[3] == -0.5 and floats[5] == 0.0


def test_cabi_argument_errors_cpu():
    """Argument errors come back < 0 with text before anything touches the device."""
    import ctypes as C
    import vexautonomousplanner_b200 as vap
    from vexautonomousplanner_b200 import _lib
    vap.build()
    L = _lib.lib()
    box = (C.c_double * 8)(0, 0, 1, 1, 2, 2, 1, 3)

    def call(hl=1.0, hw=1.0, field=(-1.0, 1.0, -1.0, 1.0), K=0, boxes=None, tol=0.0):
        return L.vap_footprint_check(C.c_int64(4), None, None, C.c_double(hl), C.c_double(hw), *map(C.c_double, field),
                                     C.c_int(K), boxes, C.c_double(tol), None, None, None)
    for kw, text in ((dict(hl=0.0), "half-length"), (dict(hw=-1.0), "half-length"), (dict(hw=float("nan")), "half"),
                     (dict(field=(1.0, 1.0, -1.0, 1.0)), "empty field"), (dict(field=(-1.0, 1.0, 2.0, 1.0)), "empty field"),
                     (dict(K=65, boxes=box), "K <= 64"), (dict(K=-1), "K <= 64"), (dict(K=2, boxes=box), "keep-out box 1"),
                     (dict(K=1), "NULL"), (dict(tol=float("inf")), "tolerance")):
        rc = call(**kw)
        assert rc < 0, kw
        assert text in L.vap_last_error().decode(), (kw, L.vap_last_error())


def test_field_check_arguments_cpu(tmp_path, capsys):
    """--keep-out parsing, the robot size from the flags or robot.length / robot.width of --config, exit 2 without it."""
    from vexautonomousplanner_b200 import field_check as fc
    a = fc.parse_args(["d", "--keep-out", "1,2,3,4", "--keep-out=-5.5,-1e1,0,0", "--robot-length-in", "18",
                       "--robot-width-in", "15", "--tolerance-in", "0.25", "--field-half-in", "70", "--max-velocity", "3"])
    assert a.keep_out == [(1.0, 2.0, 3.0, 4.0), (-5.5, -10.0, 0.0, 0.0)] and a.tol_in == 0.25 and a.max_velocity == 3.0
    assert fc.robot_size(a) == (18.0, 15.0) and not a.trajectories
    for bad in ("1,2,3", "1,2,3,4,5", "a,b,c,d", "1,2,1,4", "1,4,3,2", "1,2,inf,4", ""):
        with pytest.raises(SystemExit) as e:
            fc.parse_args(["d", "--keep-out", bad])
        assert e.value.code == 2, bad
    for bad in (["--field-half-in", "0"], ["--tile-paths", "0"], ["--keep-out", "0,0,1,1"] * 65, ["--tolerance-in", "nan"]):
        with pytest.raises(SystemExit) as e:
            fc.parse_args(["d"] + bad)
        assert e.value.code == 2, bad
    capsys.readouterr()
    d = tmp_path / "routes"
    d.mkdir()
    assert fc.main([str(d)]) == 2
    assert "robot's size is unknown" in capsys.readouterr().err
    assert fc.main([str(d), "--robot-length-in", "18"]) == 2
    cfg = tmp_path / "config.yaml"
    cfg.write_text("motion:\n  max_velocity: 3\nrobot:\n  track_width: 11.5\n  length: 17.5\n  width: 14\n")
    assert fc.read_robot_size(str(cfg)) == (17.5, 14.0)
    assert fc.robot_size(fc.parse_args(["d", "--config", str(cfg)])) == (17.5, 14.0)
    assert fc.robot_size(fc.parse_args(["d", "--config", str(cfg), "--robot-width-in", "12"])) == (17.5, 12.0)
    half = tmp_path / "half.yaml"
    half.write_text("robot:\n  length: 17.5\n")
    assert fc.read_robot_size(str(half)) == (17.5, None)
    assert fc.main([str(d), "--config", str(half)]) == 2
    assert fc.main([str(d), "--robot-length-in", "-1", "--robot-width-in", "3"]) == 2
    from vexautonomousplanner_b200.save_routes import read_config
    assert read_config(str(cfg))["track_width_in"] == 11.5          # read_config's result is unchanged
    assert "length" not in read_config(str(cfg))


def _arrays(rows=100, first=-1, kind=-1, n_viol=0, wr=5, nr=7, nk=1, t_first=float("nan"), worst=-3.25, wt=0.05,
            nd=12.5, nt=0.07, step=0.4):
    from vexautonomousplanner_b200.export import FP_F, FP_I
    ints = np.array([rows, first, kind, n_viol, wr, nr, nk], dtype=np.int64)
    floats = np.array([t_first, worst, wt, nd, nt, step])
    assert len(ints) == len(FP_I) and len(floats) == len(FP_F)
    return ints, floats


def test_field_check_report_lines_cpu():
    """The report line of each state from given arrays."""
    from vexautonomousplanner_b200.field_check import report_line
    assert report_line("a.txt", *_arrays(), 2) == (
        "clear", "clear: a.txt: wall clearance 3.250 in at t 0.050 s; nearest keep-out box 1 at 12.500 in, t 0.070 s; "
                 "sampling step <= 0.400 in")
    assert report_line("a.txt", *_arrays(nr=-1, nk=-1, nd=np.inf, nt=np.nan), 0)[1] == (
        "clear: a.txt: wall clearance 3.250 in at t 0.050 s; no keep-out boxes; sampling step <= 0.400 in")
    assert report_line("b.txt", *_arrays(first=40, kind=0, n_viol=12, wr=44, worst=2.5, wt=0.44, t_first=0.4), 0) == (
        "hits", "hits: b.txt: first at t 0.400 s (row 40): wall; worst wall overhang 2.500 in at t 0.440 s; "
                "no keep-out boxes; 12 of 100 rows")
    assert report_line("c.txt", *_arrays(first=3, kind=4, n_viol=9, t_first=0.03, nr=5, nk=2, nd=-1.25, nt=0.05), 3)[1] == (
        "hits: c.txt: first at t 0.030 s (row 3): keep-out box 2; worst wall overhang -3.250 in at t 0.050 s; "
        "nearest keep-out box 2 at -1.250 in, t 0.050 s; 9 of 100 rows")
    assert report_line("d.txt", *_arrays(first=0, kind=1, n_viol=1, t_first=0.0), 1)[1].startswith(
        "hits: d.txt: first at t 0.000 s (row 0): non-finite row;")
    assert report_line("e.txt", *_arrays(rows=0, wr=-1, nr=-1), 1) == ("not checked", "not checked: e.txt: no trajectory rows")


# ------------------------------------------------------------------------------------------------------------- GPU
def _random_rows(rng, B, field):
    """B paths of 0-3000 rows: random walks that start anywhere in the field, a third of them within 10 in of a wall,
    with repeated rows (waits) and turn-in-place runs (same x, y, heading moving)."""
    xmin, xmax, ymin, ymax = field
    rows, off = [], [0]
    for b in range(B):
        n = int(rng.integers(0, 3001)) if b % 7 else int(rng.integers(0, 3))
        if rng.random() < 0.35:
            x0 = rng.choice([xmin, xmax]) + rng.uniform(-10, 10)
            y0 = rng.uniform(ymin, ymax)
        else:
            x0, y0 = rng.uniform(xmin, xmax), rng.uniform(ymin, ymax)
        step = rng.uniform(0.01, 0.6)
        dx = np.cumsum(rng.normal(0, step, n))
        dy = np.cumsum(rng.normal(0, step, n))
        h = rng.uniform(-4, 4) + np.cumsum(rng.normal(0, 0.05, n))
        if n > 20:
            a = int(rng.integers(0, n - 10))
            dx[a:a + 10], dy[a:a + 10] = dx[a], dy[a]             # in place, heading turning
            w = int(rng.integers(0, n - 5))
            dx[w:w + 5], dy[w:w + 5], h[w:w + 5] = dx[w], dy[w], h[w]   # a wait: identical rows
        r = np.zeros((n, 7))
        r[:, 1] = np.arange(n) * 0.01
        r[:, 2], r[:, 3], r[:, 4] = x0 + dx, y0 + dy, h
        r[:, 5] = rng.uniform(0, 50, n)
        rows.append(r)
        off.append(off[-1] + n)
    return np.concatenate(rows), np.array(off, dtype=np.int64)


def _random_boxes(rng, K, field):
    xmin, xmax, ymin, ymax = field
    out = []
    for _ in range(K):
        x0, y0 = rng.uniform(xmin, xmax), rng.uniform(ymin, ymax)
        out.append((x0, y0, x0 + rng.uniform(0.5, 30), y0 + rng.uniform(0.5, 30)))
    return out


@pytest.mark.gpu
def test_random_rows_match_numpy():
    """~2000 random paths of 0-3000 rows in six batches (K = 0..5 random boxes, random robot sizes, fields and
    tolerances) against the numpy reference; permuting the paths permutes the outputs; two runs are bit-identical."""
    import torch
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rng = np.random.default_rng(11)
    checked = hits = 0
    for K in range(6):
        field = ex.default_field() if K % 2 else tuple(np.array([-1, 1, -1, 1]) * rng.uniform(40, 80))
        rows, off = _random_rows(rng, 340, field)
        boxes = _random_boxes(rng, K, field)
        length, width, tol = rng.uniform(5, 30), rng.uniform(5, 30), [0.0, 0.5, 0.0][K % 3]
        gi, gf = ex.footprint_check(eng, torch.from_numpy(rows).cuda(), torch.from_numpy(off).cuda(), length, width,
                                    field=field, keep_out=boxes, tol_in=tol)
        ref = ref_batch(rows, off, length / 2, width / 2, field, boxes, tol)
        for b in range(len(off) - 1):
            assert_matches(gi[b], gf[b], ref[b], tol, where=(K, b))
        checked += len(off) - 1
        hits += int((gi[:, 1] >= 0).sum())
        gi2, gf2 = ex.footprint_check(eng, rows, off, length, width, field=field, keep_out=boxes, tol_in=tol)
        assert np.array_equal(gi, gi2) and np.array_equal(gf.view(np.int64), gf2.view(np.int64))
        perm = rng.permutation(len(off) - 1)
        prow = np.concatenate([rows[off[p]:off[p + 1]] for p in perm])
        poff = np.concatenate([[0], np.cumsum(np.diff(off)[perm])])
        pi, pf = ex.footprint_check(eng, prow, poff, length, width, field=field, keep_out=boxes, tol_in=tol)
        assert np.array_equal(pi, gi[perm]) and np.array_equal(pf.view(np.int64), gf[perm].view(np.int64))
    assert checked > 2000 and 0.05 * checked < hits < checked, (checked, hits)


def _boxes_for(field):
    xmin, xmax, ymin, ymax = field
    return [(-10.0, -10.0, 10.0, 10.0), (xmin + 5, ymin + 5, xmin + 25, ymin + 15), (30.0, -60.0, 45.0, 60.0)]


@pytest.mark.gpu
def test_fresh_profiles_and_saved_files_match():
    """synth.mixed_paths(1024) and synth.long_path() through export_rows against numpy; the mixed batch through
    save_text_batch -> parse_text_batch gives bit-identical outputs."""
    from test_trajectory_check import _mixed_batch
    from vexautonomousplanner_b200 import export as ex, synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    field = ex.default_field()
    boxes = _boxes_for(field)
    packed, na, aa = _mixed_batch(1024, 3)
    db = eng.upload(packed)
    res = eng.profile(db)
    rows, off = ex.export_rows(eng, res)
    gi, gf = ex.footprint_check(eng, rows, off, 18.0, 15.0, keep_out=boxes, tol_in=0.25)
    ref = ref_batch(rows.cpu().numpy(), off.cpu().numpy(), 9.0, 7.5, field, boxes, 0.25)
    status = res.status.cpu().numpy()
    for b in range(res.B):
        assert_matches(gi[b], gf[b], ref[b], 0.25, where=b)
        if status[b] != 0:
            assert gi[b].tolist() == [0, -1, -1, 0, -1, -1, -1] and np.isnan(gf[b, [0, 2, 4]]).all()
    assert int((gi[:, 1] >= 0).sum()) > 50
    assert set(gi[gi[:, 1] >= 0, 2].tolist()) >= {0, 2}
    text, offs, ok = ex.save_text_batch(eng, res, db, na, aa)
    p = ex.parse_text_batch(eng, text, offs)
    pi, pf = ex.footprint_check(eng, p.rows, p.row_offsets, 18.0, 15.0, keep_out=boxes, tol_in=0.25)
    assert np.array_equal(pi, gi) and np.array_equal(pf.view(np.int64), gf.view(np.int64))

    res = eng.profile(eng.upload(synth.long_path()))
    rows, off = ex.export_rows(eng, res)
    assert int(off[1]) > 100_000
    for L, W in ((18.0, 15.0), (40.0, 30.0)):
        gi, gf = ex.footprint_check(eng, rows, off, L, W, keep_out=boxes)
        ref = ref_batch(rows.cpu().numpy(), off.cpu().numpy(), L / 2, W / 2, field, boxes, 0.0)
        assert_matches(gi[0], gf[0], ref[0], 0.0, where=("long", L))


@pytest.mark.gpu
def test_nan_rows_and_empty_paths():
    """A NaN row reports kind 1 (the rows around it still count); paths without rows report 0 rows and -1."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rows = np.zeros((6, 7))
    rows[:, 1] = np.arange(6) * 0.01
    rows[:, 2] = np.arange(6) * 1.0
    rows[3, 3] = np.nan
    rows[5, 4] = np.inf
    gi, gf = ex.footprint_check(eng, rows, [0, 0, 6, 6, 6], 10.0, 10.0, keep_out=[(50.0, 50.0, 60.0, 60.0)])
    assert gi[1].tolist()[:4] == [6, 3, 1, 2] and gf[1, 0] == rows[3, 1]
    for b in (0, 2, 3):
        assert gi[b].tolist() == [0, -1, -1, 0, -1, -1, -1]
        assert np.isnan(gf[b, 0]) and gf[b, 1] == -np.inf and gf[b, 3] == np.inf and gf[b, 5] == 0.0
    ref = ref_batch(rows, [0, 6], 5.0, 5.0, ex.default_field(), [(50.0, 50.0, 60.0, 60.0)], 0.0)[0]
    assert_matches(gi[1], gf[1], ref, 0.0)
    gi, gf = ex.footprint_check(eng, np.zeros((0, 7)), [0], 10.0, 10.0)
    assert gi.shape == (0, 7) and gf.shape == (0, 6)


@pytest.mark.gpu
def test_argument_errors_raise_with_text():
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200._lib import VapError
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    rows = np.zeros((2, 7))
    for kw, text in ((dict(length_in=0.0), "half-length"), (dict(field=(0, 0, -1, 1)), "empty field"),
                     (dict(keep_out=[(0, 0, 1, 1)] * 65), "K <= 64"), (dict(keep_out=[(0, 0, 1, 1), (2, 0, 1, 1)]), "box 1")):
        args = dict(length_in=10.0, width_in=10.0)
        args.update(kw)
        with pytest.raises(VapError, match=text):
            ex.footprint_check(eng, rows, [0, 2], **args)


def _node(start=False, end=False, turn=0):
    from vexautonomousplanner_b200.export import RouteNode
    n = RouteNode()
    n.is_start_node, n.is_end_node, n.turn = start, end, turn
    return n


def _route_json(xs_in, y_txt_in, turn_at=None, turn=90):
    """Node JSON of a straight route through x = xs_in at .txt-frame height y_txt_in (JSON y is the negated .txt y)."""
    from vexautonomousplanner_b200 import export as ex
    n = len(xs_in)
    nodes = [_node(i == 0, i == n - 1, turn if i == turn_at else 0) for i in range(n)]
    return ex.nodes_to_json([(ex.in_to_px(x), ex.in_to_px(-y_txt_in)) for x in xs_in], nodes)


@pytest.mark.gpu
def test_turn_in_place_corners_leave_the_field():
    """A 24 x 8 in robot on a straight route 8 in below the top wall clears the wall by 4 in while it drives; the 90
    degree turn in place at its middle node swings its half-length past the wall.  The first violating row lies inside
    that node's inserted turn rows (which hold the position with v = 0)."""
    from vexautonomousplanner_b200 import export as ex
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.packing import pack_paths
    from vexautonomousplanner_b200.synth import FACTORY
    top = ex.default_field()[3]
    eng = Engine("cuda:0")
    pts, nodes, aps, _ = ex.load_nodes(_route_json([-36.0, -15.0, 0.0, 15.0, 36.0], top - 8.0, turn_at=2))
    res = eng.profile(eng.upload(pack_paths([(ex.px_points_to_ft(pts), nodes, aps)], FACTORY)))
    assert int(res.status[0]) == 0
    rows, off = ex.export_rows(eng, res)
    r = rows.cpu().numpy()
    k0 = int(res.nodes_map[0, 2])                                           # node 2's turn rows start here
    assert np.abs(r[:k0, 3] - (top - 8.0)).max() < 1e-6                    # up to the turn: 8 in from the wall
    gi, gf = ex.footprint_check(eng, rows, off, 24.0, 8.0)
    assert gi[0, 2] == ex.FP_KIND_WALL, gi
    first = int(gi[0, 1])
    assert k0 <= first
    held = r[k0:first + 1]
    assert (held[:, 2] == r[k0 - 1, 2]).all() and (held[:, 3] == r[k0 - 1, 3]).all() and (held[:, 5] == 0).all()
    assert gf[0, 1] > 3.9                                                   # 12 - 8 in once the turn is done
    gi, gf = ex.footprint_check(eng, rows, off, 8.0, 4.0)                   # small enough to swing inside
    assert gi[0, 1] == -1 and gf[0, 1] < 0, (gi, gf)


def _folder(tmp_path):
    from vexautonomousplanner_b200 import export as ex
    field = ex.default_field()
    d = tmp_path / "routes"
    d.mkdir()
    xs = [-40.0, -15.0, 10.0, 40.0]
    (d / "clear.txt").write_text(_route_json(xs, -20.0))
    (d / "hug.txt").write_text(_route_json(xs, field[2] + 3.0))            # 3 in from the bottom wall, half-width 6
    (d / "box.txt").write_text(_route_json(xs, 35.0))                       # through the keep-out box
    (d / "notes.txt").write_text("not a route")
    return d


@pytest.mark.gpu
def test_field_check_command_on_a_folder(tmp_path, capsys):
    """A clear route, one hugging a wall, one through a keep-out box and a file that is not route JSON: the right lines
    and exit 1; --trajectories on the folder save_routes wrote gives the same verdicts."""
    from vexautonomousplanner_b200 import field_check as fc, save_routes as sr
    d = _folder(tmp_path)
    args = ["--robot-length-in", "18", "--robot-width-in", "12", "--keep-out=-5,30,5,40"]
    assert fc.main([str(d)] + args) == 1
    out = capsys.readouterr().out.splitlines()
    lines = {l.split(": ")[1]: l for l in out if ": " in l}
    assert lines["clear.txt"].startswith("clear: clear.txt: wall clearance ")
    assert "nearest keep-out box 0 at " in lines["clear.txt"] and "sampling step <= " in lines["clear.txt"]
    assert lines["hug.txt"].startswith("hits: hug.txt: first at t ") and "(row 0): wall;" in lines["hug.txt"]
    overhang = float(lines["hug.txt"].split("worst wall overhang ")[1].split(" in")[0])
    assert abs(overhang - 3.0) < 0.05
    assert lines["box.txt"].startswith("hits: box.txt: first at t ") and "): keep-out box 0;" in lines["box.txt"]
    assert lines["notes.txt"].startswith("not checked: notes.txt: not route JSON")
    assert out[-1].startswith("1 of 4 files clear in ")
    odir = tmp_path / "saved"
    assert sr.main([str(d), str(odir)]) == 1                               # notes.txt is not written
    capsys.readouterr()
    assert fc.main([str(odir), "--trajectories"] + args) == 1
    out2 = capsys.readouterr().out.splitlines()
    lines2 = {l.split(": ")[1]: l for l in out2 if ": " in l}
    assert sorted(lines2) == ["box.txt", "clear.txt", "hug.txt"] and out2[-1].startswith("1 of 3 files clear in ")
    for n in lines2:
        assert lines2[n] == lines[n]
    (odir / "hug.txt").write_text((odir / "hug.txt").read_text().replace("\n", "\nx\n", 1))
    assert fc.main([str(odir), "--trajectories"] + args) == 1
    assert "unreadable: hug.txt: line 2: the first token is neither 0 nor 1" in capsys.readouterr().out
    assert fc.main([str(odir), "--trajectories", "--robot-length-in", "18", "--robot-width-in", "12",
                    "--field-half-in", "200"]) == 1
    out3 = capsys.readouterr().out
    assert "clear: box.txt" in out3 and "clear: clear.txt" in out3 and "unreadable: hug.txt" in out3

"""Graph and pipelined replays fed batches that the captured batch did not size, against the CPU oracle.

A captured step (GraphedProfile, PipelinedProfiler) keeps every capacity of the batch it was captured on: the distance
samples (D_cap), the time rows (T_cap) and the distance table's row width, samples * max_splines, where max_splines is
1 + the number of interior turn / reverse nodes and so depends on the data.  A later batch copied into the static inputs
may need more of any of them.  Such paths must come back as ST_CAPACITY (never as a short "ok" profile), run() must redo
them exactly, and the slots of a pipeline must flag exactly the paths that do not fit.  Every batch is built from seeds;
each test asserts the property of its batches it relies on, so that a change of seed cannot quietly remove its point.
Oracle comparisons use the north-star tolerances of tests/test_gpu_parity.py with integer outputs exact.
"""
import ctypes as C
from dataclasses import replace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

B, N, TILES = 203, 10, 4           # B is not a multiple of the tile count; n_nodes is ragged (2 .. N)
ST_CAPACITY = -4
TURNS = (30.0, -45.0, 90.0, -135.0, 45.0, -30.0)
STREAM_TOL = {"times": (1e-6, 1e-12), "positions": (1e-9, 1e-12), "linear_vels": (1e-6, 1e-9),
              "accelerations": (1e-6, 1e-6), "headings": (1e-9, 1e-10), "angular_vels": (1e-6, 1e-9),
              "x": (1e-9, 1e-10), "y": (1e-9, 1e-10)}
FAIL = 1                           # the heavy batch's failing path: a turn at node 0 (the reference raises IndexError)


@pytest.fixture(scope="module")
def ora(oracle_mod):
    oracle_mod.set_sq_mode(1)
    yield oracle_mod
    oracle_mod.set_sq_mode(0)


# ------------------------------------------------------------------------------------------------ batches
def _rotations(p):
    from vexautonomousplanner_b200.packing import rotation_table
    p.node_attr[:, :, 10], p.node_attr[:, :, 11] = rotation_table(p.node_attr[:, :, 2], (p.node_flags & 1) != 0)
    return p


def _split_nodes(p):
    idx = np.arange(p.N_max)[None, :]
    interior = (idx >= 1) & (idx < p.n_nodes[:, None] - 1)
    return (((p.node_flags & 1) != 0) | (p.node_attr[:, :, 2] != 0)) & interior


def _clear_splits(p, mask):
    p.node_attr[:, :, 2][mask] = 0.0
    p.node_flags[mask] &= ~1


def light_batch(seed, scale=1.0):
    """Mixed paths (turns, waits, stops, reverses, action points, per-path constraints) with at most one interior split
    node per path: max_splines = 2.  scale < 1 shrinks the paths towards the centre of the field."""
    from vexautonomousplanner_b200 import synth
    p = synth.mixed_paths(B, N, seed=seed)
    p.node_attr[:, :, 0:2] *= scale
    split = _split_nodes(p)
    _clear_splits(p, split & (np.cumsum(split, axis=1) > 1))
    return _rotations(p)


def heavy_batch(seed, s):
    """Mixed paths with ragged n_nodes (every 5th path: 2 .. N-1 nodes), a turn on every interior node of every 7th path
    (N-1 splines), exactly s interior splits on others (s+1 splines), and one path with a turn at node 0."""
    from vexautonomousplanner_b200 import synth
    p = synth.mixed_paths(B, N, seed=seed)
    rng = np.random.default_rng(seed)
    rows = np.arange(B)
    ragged = rows % 5 == 4
    p.n_nodes[ragged] = 2 + (rows[ragged] // 5) % (N - 2)
    n = p.n_nodes.astype(np.int64)
    p.ap_attr[:, :, 0] *= ((n - 1) / (N - 1))[:, None]          # action points stay on the shortened paths
    idx = np.arange(N)[None, :]
    tail = idx >= n[:, None] - 1                                  # a turn / reverse at the last node crashes the reference
    _clear_splits(p, tail)
    interior = (idx >= 1) & (idx < n[:, None] - 1)
    every = (rows % 7 == 0) & (n == N)
    _clear_splits(p, every[:, None] & interior)
    p.node_attr[every, 1:N - 1, 2] = rng.choice(TURNS, (int(every.sum()), N - 2))
    one_more = (rows % 7 == 3) & (n - 2 >= s)
    for b in np.nonzero(one_more)[0]:
        _clear_splits(p, (rows == b)[:, None] & interior)
        at = 1 + rng.choice(int(n[b]) - 2, s, replace=False)
        p.node_attr[b, at, 2] = rng.choice(TURNS, s)
    _clear_splits(p, (rows == FAIL)[:, None] & interior)
    p.node_attr[FAIL, 0, 2] = 30.0
    return _rotations(p)


def zigzag_and_waits(light):
    """The light batch with path 0 replaced by a zig-zag from one corner of the field to the other (about 110 ft: more
    distance samples than any path of a light batch shrunk to half size) and path 1 waiting 5 s on every node it leaves
    from (more time rows)."""
    from vexautonomousplanner_b200.packing import px_to_ft
    p = type(light)(*(a.copy() for a in (light.node_attr, light.node_flags, light.n_nodes, light.ap_attr, light.ap_flags,
                                         light.n_ap, light.cons)))
    px = np.stack([np.where(np.arange(N) % 2 == 0, 15.0, 1985.0), np.linspace(15.0, 1985.0, N)], axis=1)
    p.node_attr[0] = 0.0
    p.node_attr[0, :, 0:2] = px_to_ft(px)
    p.node_flags[0] = 0
    p.n_nodes[0] = N
    p.n_ap[0] = 0
    p.node_attr[1, : int(p.n_nodes[1]) - 1, 3] = 5.0
    return _rotations(p)


_REFS = {}


def oracle_refs(ora, name, p):
    """Per path: the oracle's full result (status 0) or its status, and its spline count S."""
    if name not in _REFS:
        refs = []
        for b in range(p.B):
            n, A = int(p.n_nodes[b]), int(p.n_ap[b])
            na, nf = p.node_attr[b, :n], p.node_flags[b, :n]
            try:
                r = ora.full(na, nf, p.ap_attr[b, :A] if A else None, p.ap_flags[b, :A] if A else None, p.cons[b])
                r["status"] = 0
            except ora.OracleError as e:
                r = dict(status=e.code)
            r["S"] = ora.Geometry(na, nf).S
            refs.append(r)
        _REFS[name] = refs
    return _REFS[name]


# ------------------------------------------------------------------------------------------------ checks
def snapshot(r):
    from vexautonomousplanner_b200.engine import ProfileResult
    return ProfileResult(r.B, r.T_cap, r.out.clone(), r.n_out.clone(), r.nodes_map.clone(), r.actions_map.clone(),
                         r.n_maps.clone(), r.status.clone(), r.summary.clone(), r.vel.clone(), r.n_samples.clone())


def check_vs_oracle(refs, res, rows, streams):
    """Status, counts, maps and summary row of every path in `rows`; also the streams of the paths in `streams`."""
    status, n_out, n_samples = (t.cpu().numpy() for t in (res.status, res.n_out, res.n_samples))
    n_maps, nodes_map, actions_map = (t.cpu().numpy() for t in (res.n_maps, res.nodes_map, res.actions_map))
    summ = res.summary.cpu().numpy()
    for b in rows:
        r = refs[b]
        assert status[b] == r["status"] and summ[b, 4] == r["status"], (b, status[b], r["status"])
        if r["status"] != 0:
            assert n_out[b] == 0, b
            continue
        assert n_out[b] == r["T"] and n_samples[b] == r["D"], (b, n_out[b], r["T"], n_samples[b], r["D"])
        assert nodes_map[b, : n_maps[b, 0]].tolist() == r["nodes_map"].tolist(), b
        assert actions_map[b, : n_maps[b, 1]].tolist() == r["actions_map"].tolist(), b
        assert summ[b, 0] == r["T"], b
        np.testing.assert_allclose(summ[b, 1], r["summary"][1], rtol=1e-12, err_msg=f"path {b} total length")
        np.testing.assert_allclose(summ[b, 2:4], r["summary"][2:4], rtol=1e-6, err_msg=f"path {b} t_end, max |v|")
        if b in streams:
            got = res.path(b)
            np.testing.assert_allclose(got["vel"], r["vel"], rtol=1e-6, atol=1e-12, err_msg=f"path {b} vel")
            for k, (rtol, atol) in STREAM_TOL.items():
                np.testing.assert_allclose(got[k], r[k], rtol=rtol, atol=atol, err_msg=f"path {b} {k}")


def same_bits(ref, got, rows=None):
    """Every output of the paths in `rows` (default: all) bit for bit."""
    sel = torch.ones(ref.B, dtype=torch.bool, device=ref.status.device)
    if rows is not None:
        sel = torch.zeros_like(sel)
        sel[torch.as_tensor(np.asarray(rows), dtype=torch.long, device=sel.device)] = True
    for name in ("status", "n_out", "n_samples", "n_maps"):
        assert torch.equal(getattr(ref, name)[sel], getattr(got, name)[sel]), name
    assert torch.equal(ref.summary[sel].view(torch.int64), got.summary[sel].view(torch.int64))
    n = torch.where(sel, ref.n_out, 0).long()
    Tm = min(ref.T_cap, got.T_cap)
    assert int(n.max()) <= Tm
    mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
    for i in range(8):
        assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), i
    D = torch.where(sel, ref.n_samples, 0).long()
    Dm = min(ref.vel.shape[1], got.vel.shape[1])
    md = torch.arange(Dm, device=D.device)[None, :] < D[:, None]
    assert torch.equal(ref.vel[:, :Dm][md].view(torch.int64), got.vel[:, :Dm][md].view(torch.int64))
    nm = torch.arange(ref.nodes_map.shape[1], device=D.device)[None, :] < torch.where(sel, ref.n_maps[:, 0], 0)[:, None]
    assert torch.equal(ref.nodes_map[nm], got.nodes_map[nm])
    am = torch.arange(ref.actions_map.shape[1], device=D.device)[None, :] < torch.where(sel, ref.n_maps[:, 1], 0)[:, None]
    assert torch.equal(ref.actions_map[am], got.actions_map[am])


def eager(packed):
    from vexautonomousplanner_b200.engine import Engine
    e = Engine("cuda:0")
    return e.profile(e.upload(packed))


def heavy_preconditions(heavy, refs, s):
    S = np.array([r["S"] for r in refs])
    assert S.max() == N - 1 and (S == s + 1).any() and int((S > s).sum()) >= 20, np.bincount(S)
    assert sorted(set(heavy.n_nodes.tolist())) == list(range(2, N + 1))
    assert refs[FAIL]["status"] == -2 and S[FAIL] <= s
    assert B % TILES != 0
    return S


# ------------------------------------------------------------------------------------------------ tests
def test_graph_replay_with_more_splines_than_captured(ora):
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    light = light_batch(61)
    g = eng.capture(eng.upload(light), tiles=TILES)
    s = g.db.max_splines
    assert s == light.max_splines() == 2
    heavy = heavy_batch(62, s)
    refs = oracle_refs(ora, "heavy62", heavy)
    S = heavy_preconditions(heavy, refs, s)
    assert heavy.max_splines() > s
    got = g.run(eng.upload(heavy))
    torch.cuda.synchronize()
    assert g.db.max_splines == s                           # the redo never touches the graph's static batch
    streams = {b for b in range(B) if S[b] > s or b % 9 == 0}
    check_vs_oracle(refs, got, range(B), streams)
    same_bits(eager(heavy), got)
    # and the graph still replays the light batch exactly afterwards
    again = g.run(eng.upload(light))
    torch.cuda.synchronize()
    same_bits(eager(light), again)


def test_pipelined_replays_flag_exactly_the_paths_that_do_not_fit(ora):
    from vexautonomousplanner_b200.engine import Engine, PipelinedProfiler
    eng = Engine("cuda:0")
    light_a, light_b = light_batch(61), light_batch(63)
    db_a = eng.upload(light_a)
    pipe = PipelinedProfiler(eng, db_a, depth=2)
    s = pipe.graphs[0].db.max_splines
    heavy = heavy_batch(62, s)
    heavy_db = eng.upload(heavy)
    snaps = []

    def consume(res):
        snaps.append(snapshot(res))

    # light, heavy, light through submit(new_db); the last light batch is the one the pipeline was built from, after
    # another batch went through its slot
    order = [("light63", light_b), ("heavy62", heavy), ("light61", light_a), ("heavy62", heavy)]
    slots, inputs = [], []                 # inputs stay alive until drain(): the slots' streams copy from them
    for name, p in order[:3]:
        slots.append(pipe.graphs[pipe.n % 2])
        inputs.append(eng.upload(p) if p is not light_a else db_a)
        pipe.submit(inputs[-1], consume)
    # the way bench.py feeds a slot: inputs copied straight into its static buffers on its stream, then submit(None)
    main = torch.cuda.current_stream()
    slot, st = pipe.graphs[pipe.n % 2], pipe.streams[pipe.n % 2]
    st.wait_stream(main)
    with torch.cuda.stream(st):
        slot.db.copy_(heavy_db)
    slots.append(slot)
    pipe.submit(None, consume)
    pipe.drain()
    torch.cuda.synchronize()
    assert len(snaps) == 4
    fresh = eng.upload(light_a)
    for name, a, b in zip(db_a.FIELDS, db_a.tensors(), fresh.tensors()):
        assert torch.equal(a, b), name                      # the caller's batch is not a slot's input
    flagged_any = []
    for (name, p), slot, res in zip(order, slots, snaps):
        refs = oracle_refs(ora, name, p)
        want = eager(p)
        torch.cuda.synchronize()
        S = np.array([r["S"] for r in refs])
        D = want.n_samples.cpu().numpy()
        T = np.array([r.get("T", 0) for r in refs])
        ok = np.array([r["status"] == 0 for r in refs])
        need = (S > slot.db.max_splines) | (D > slot.D_cap) | (ok & (T > slot.T_cap))
        flagged = res.status.cpu().numpy() == ST_CAPACITY
        assert np.array_equal(flagged, need), (name, np.nonzero(flagged != need)[0][:10].tolist())
        flagged_any.append(bool(flagged.any()))
        rows = np.nonzero(~need)[0]
        check_vs_oracle(refs, res, rows, {b for b in rows if b % 9 == 0})
        same_bits(want, res, rows)
        if flagged.any():
            # the documented caller redo
            redo = eng.profile(eng.upload(p))
            torch.cuda.synchronize()
            check_vs_oracle(refs, redo, range(B), {b for b in range(B) if need[b] or b % 9 == 0})
    assert flagged_any[1] and flagged_any[3] and not flagged_any[2], flagged_any


def test_replay_redoes_distance_and_time_overflows(ora):
    from vexautonomousplanner_b200 import _lib
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    light = light_batch(61, scale=0.5)
    g = eng.capture(eng.upload(light), tiles=TILES, to_host=True)
    big = zigzag_and_waits(light)
    refs = oracle_refs(ora, "zigzag61", big)
    assert refs[0]["status"] == 0 and refs[0]["D"] > g.D_cap, (refs[0].get("D"), g.D_cap)
    assert refs[1]["status"] == 0 and refs[1]["T"] > g.T_cap, (refs[1].get("T"), g.T_cap)
    assert max(r["S"] for r in refs) <= g.db.max_splines
    got = g.run(eng.upload(big))
    torch.cuda.synchronize()
    check_vs_oracle(refs, got, range(B), {b for b in range(B) if b < 2 or b % 9 == 0})
    same_bits(eager(big), got)
    # the host-out replay cannot redo inside the graph: it raises, as documented
    with pytest.raises(_lib.VapError):
        g.run_host(big)
    heavy = heavy_batch(62, g.db.max_splines)
    heavy_preconditions(heavy, oracle_refs(ora, "heavy62", heavy), g.db.max_splines)
    with pytest.raises(_lib.VapError):
        g.run_host(heavy)
    h = g.run_host(light)
    want = eager(light)
    torch.cuda.synchronize()
    assert h.status.tolist() == want.status.cpu().tolist() and h.n_out.tolist() == want.n_out.cpu().tolist()
    assert np.array_equal(h.summary.numpy(), want.summary.cpu().numpy())


def test_replay_rejects_other_batch_shapes():
    """B, N_max or A_max of another size raise ValueError before anything is copied (a size-1 dimension would otherwise
    broadcast silently); the captured batch is then still reproduced bit for bit."""
    from vexautonomousplanner_b200.engine import Engine, PipelinedProfiler
    eng = Engine("cuda:0")
    light = light_batch(61)
    db = eng.upload(light)
    g = eng.capture(eng.upload(light), tiles=TILES)
    pipe = PipelinedProfiler(eng, db, depth=2)
    first = snapshot(g.run())
    z = lambda *shape, dt=torch.float64: torch.zeros(shape, dtype=dt, device=db.node_attr.device)     # noqa: E731
    bad = {
        "B=1": db.rows(0, 1),
        "B-1": db.rows(0, B - 1),
        "N_max-1": replace(db, node_attr=db.node_attr[:, : N - 1], node_flags=db.node_flags[:, : N - 1]),
        "N_max=1": replace(db, node_attr=db.node_attr[:, :1], node_flags=db.node_flags[:, :1]),
        "A_max+1": replace(db, ap_attr=z(B, db.A_max + 1, 4), ap_flags=z(B, db.A_max + 1, dt=torch.int32)),
        "A_max=1": replace(db, ap_attr=db.ap_attr[:, :1], ap_flags=db.ap_flags[:, :1]),
    }
    for what, new in bad.items():
        with pytest.raises(ValueError):
            g.run(new)
        with pytest.raises(ValueError):
            pipe.submit(new)
        assert pipe.n == 0, what
    again = g.run()
    res = pipe.submit(None)
    pipe.drain()
    torch.cuda.synchronize()
    same_bits(first, again)
    same_bits(eager(light), res)


def test_pipeline_capacities_do_not_compound():
    """Every slot of a pipeline gets the margin once: the same (D_cap, T_cap) as plan_capacities(db, margin) of a fresh
    engine, and the engine's plan stays the exact one."""
    from vexautonomousplanner_b200.engine import Engine, PipelinedProfiler
    light = light_batch(61)
    eng = Engine("cuda:0")
    db = eng.upload(light)
    pipe = PipelinedProfiler(eng, db, depth=3, margin=1.3)
    fresh = Engine("cuda:0")
    fdb = fresh.upload(light)
    want = fresh.plan_capacities(fdb, 1.3)
    key = (db.B, db.N_max, db.A_max, db.max_splines)
    exact = fresh._plan[key]
    assert want[0] > exact[0] and want[1] > exact[1]
    assert [(gr.D_cap, gr.T_cap) for gr in pipe.graphs] == [want] * 3
    assert eng._plan[key] == exact
    ref = eager(light)
    results = []
    for _ in range(3):
        pipe.submit(None, lambda r: results.append(snapshot(r)))
    pipe.drain()
    torch.cuda.synchronize()
    for r in results:
        same_bits(ref, r)


def test_understated_max_splines_is_redone_exactly(ora):
    """A DeviceBatch whose max_splines is below the batch's own count (here 1): Engine.profile and Engine.profile_batch
    find the true count from the geometry kernel and redo; every path equals the oracle and the exact-count run."""
    from vexautonomousplanner_b200.engine import Engine
    heavy = heavy_batch(62, 2)
    refs = oracle_refs(ora, "heavy62", heavy)
    S = heavy_preconditions(heavy, refs, 2)
    eng = Engine("cuda:0")
    exact = eng.upload(heavy)
    assert exact.max_splines == N - 1
    low = replace(exact, max_splines=1)
    want = eng.profile(exact)
    streams = {b for b in range(B) if S[b] > 1 and b % 3 == 0 or b % 9 == 0}
    for got in (Engine("cuda:0").profile(low), Engine("cuda:0").profile_batch(low)):
        torch.cuda.synchronize()
        assert low.max_splines == 1
        check_vs_oracle(refs, got, range(B), streams)
        same_bits(want, got)


def test_profile_batch_raw_ctypes_flags_paths_with_more_splines(ora):
    """vap_profile_batch called directly with max_splines below the batch's count: VAP_ERR_CAPACITY on exactly the paths
    with more splines, every other path bit for bit what the call with the exact count returns."""
    from vexautonomousplanner_b200 import _lib
    from vexautonomousplanner_b200.engine import Engine
    heavy = heavy_batch(62, 2)
    refs = oracle_refs(ora, "heavy62", heavy)
    S = heavy_preconditions(heavy, refs, 2)
    eng = Engine("cuda:0")
    db = eng.upload(heavy)
    D_cap, T_cap = eng.plan_capacities(db)
    L = _lib.lib()

    def run(max_splines):
        Bn, Nn, An = db.B, db.N_max, db.A_max
        grid, rden = eng.dgrid(D_cap + 2), eng.lerp_recip(D_cap + 2)
        nbytes = L.vap_workspace_bytes(C.c_int64(Bn), Nn, An, max_splines, 1000, 1000, C.c_int64(D_cap), C.c_int64(T_cap), 32)
        assert nbytes > 0
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=db.node_attr.device)
        z = lambda *shape, dt=torch.int32: torch.zeros(shape, dtype=dt, device=ws.device)     # noqa: E731
        o = dict(out=z(8, Bn, T_cap, dt=torch.float64), n_out=z(Bn), nodes_map=z(Bn, Nn + 1), actions_map=z(Bn, max(An, 1)),
                 n_maps=z(Bn, 2), status=z(Bn), summary=z(Bn, 5, dt=torch.float64), vel=z(Bn, D_cap, dt=torch.float64),
                 n_samples=z(Bn), need=z(3, dt=torch.int64))
        p = lambda t: C.c_void_p(t.data_ptr())     # noqa: E731
        rc = L.vap_profile_batch(
            C.c_int64(Bn), Nn, An, max_splines, p(db.node_attr), p(db.node_flags), p(db.n_nodes), p(db.ap_attr),
            p(db.ap_flags), p(db.n_ap), p(db.cons), C.c_double(0.01), C.c_double(0.005), C.c_double(0.01), C.c_double(0.01),
            1000, 1000, C.c_int64(D_cap), C.c_int64(T_cap), 32, p(grid), C.c_int64(grid.numel()), p(rden),
            C.c_int64(rden.numel()), C.c_void_p((ws.data_ptr() + 255) // 256 * 256), C.c_int64(nbytes), p(o["out"]),
            C.c_int64(0), p(o["n_out"]), p(o["nodes_map"]), p(o["actions_map"]), p(o["n_maps"]), p(o["status"]),
            p(o["summary"]), p(o["vel"]), p(o["n_samples"]), p(o["need"]),
            C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, L.vap_last_error()
        torch.cuda.synchronize()
        from vexautonomousplanner_b200.engine import ProfileResult
        return ProfileResult(Bn, T_cap, o["out"], o["n_out"], o["nodes_map"], o["actions_map"], o["n_maps"], o["status"],
                             o["summary"], o["vel"], o["n_samples"])

    full = run(N - 1)
    assert not bool((full.status == ST_CAPACITY).any())
    check_vs_oracle(refs, full, range(B), set(range(0, B, 9)))
    for small in (1, 2, 5):
        got = run(small)
        over = S > small
        assert over.any() and not over.all()
        assert np.array_equal(got.status.cpu().numpy() == ST_CAPACITY, over), small
        assert (got.n_out.cpu().numpy()[over] == 0).all() and (got.n_samples.cpu().numpy()[over] == 0).all()
        same_bits(full, got, np.nonzero(~over)[0])

"""GPU parity tests: the CUDA engine (through the C ABI) against the CPU oracle and the reference goldens.

Stage-wise checks feed the oracle the engine's own upstream tables, so every stage that is pure IEEE
arithmetic must agree BIT FOR BIT (the oracle runs with x**2 == x*x, the one place where the engine
deliberately uses the correctly rounded product instead of libm pow; see DESIGN.md).  End-to-end checks
against the reference's golden outputs use the north-star tolerances (1e-9 relative for positions, 1e-6 for
velocities and times) with exact integer outputs; coordinates and headings cross zero, so their relative
tolerance is paired with atol = 1e-10 (1e-11 of the 12.1 ft field).
"""
import numpy as np
import pytest

from golden_util import bit_equal, case_names, load_case, ulp_diff

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["fast", "serial"])
def eng(request):
    """Both implementations go through every parity test: the fast path (chunk-speculative velocity passes, split
    time loop) and the reference-shaped one-thread-per-path kernels."""
    from vexautonomousplanner_b200.engine import Engine
    if request.param == "fast":
        return Engine("cuda:0", velocity_impl="chunked", time_impl="split")
    return Engine("cuda:0", velocity_impl="serial", time_impl="serial")


@pytest.fixture(scope="module")
def ora(oracle_mod):
    oracle_mod.set_sq_mode(1)
    yield oracle_mod
    oracle_mod.set_sq_mode(0)


def _bits(a, b, what):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if not bit_equal(a, b):
        u = ulp_diff(a, b)
        raise AssertionError(f"{what}: {int((u > 0).sum())}/{u.size} differ, max {int(u.max())} ulp")


def golden_batch():
    """All golden cases as ONE ragged batch (N from 2 to 16, 0..3 action points)."""
    from vexautonomousplanner_b200.packing import PackedPaths
    cases = [load_case(n) for n in case_names()]
    B = len(cases)
    N = max(c["n"] for c in cases)
    A = max(max(len(c["ap_t"]) for c in cases), 1)
    na = np.zeros((B, N, 12)); nf = np.zeros((B, N), dtype=np.int32); nn = np.zeros(B, dtype=np.int32)
    apa = np.zeros((B, A, 4)); apf = np.zeros((B, A), dtype=np.int32); nap = np.zeros(B, dtype=np.int32)
    cons = np.zeros((B, 6))
    for b, c in enumerate(cases):
        n, a = c["n"], len(c["ap_t"])
        na[b, :n] = c["node_attr"]; nf[b, :n] = c["node_flags"]; nn[b] = n
        apa[b, :a] = c["ap_attr"]; apf[b, :a] = c["ap_flags"]; nap[b] = a
        cons[b] = c["constraints"]
    return cases, PackedPaths(na, nf, nn, apa, apf, nap, cons)


def stagewise_check(ora, packed, res, b, n_api=0):
    """Oracle re-run of every stage on the engine's own upstream data; bit-exact comparisons."""
    n = int(packed.n_nodes[b]); A = int(packed.n_ap[b])
    na, nf = packed.node_attr[b, :n], packed.node_flags[b, :n]
    apa, apf = packed.ap_attr[b, :A], packed.ap_flags[b, :A]
    cons = packed.cons[b]
    g, t, ex = res.geometry, res.tables, res.extra
    geo = ora.Geometry(na, nf)
    S = geo.S
    assert int(g.n_splines[b]) == S
    assert g.first_node[b, : S + 1].cpu().numpy().tolist() == geo.first_node.tolist()
    _bits(g.seg[b, : n - 1].cpu().numpy(), geo.seg, "segments")
    _bits(g.param_end[b, :S].cpu().numpy(), geo.param_end, "param_end")
    _bits(g.seglen[b, : n - 1].cpu().numpy(), geo.seglen, "segment lengths")
    ld, lt, total = geo.build_lut()
    _bits(t.lut_d[b, : 1000 * S].cpu().numpy(), ld, "lut distances")
    _bits(t.lut_t[b, : 1000 * S].cpu().numpy(), lt, "lut parameters")
    _bits(t.total_len[b].cpu().numpy(), total, "total length")
    K = np.ascontiguousarray(t.prop_k[b, : 1000 * n].cpu().numpy())
    H = np.ascontiguousarray(t.prop_h[b, : 1000 * n].cpu().numpy())
    ko, ho = geo.build_props()
    assert ulp_diff(K, ko).max() <= 8, "curvature table"
    assert ulp_diff(H, ho).max() <= 8, "heading table"
    ds = ora.dist_sample(geo, apa, apf, cons, 0.005, ld, lt, total, K, H)
    D = int(res.n_samples[b])
    assert D == ds["D"]
    _bits(ex["t"][b, :D].cpu().numpy(), ds["t"], "t_i")
    _bits(ex["kap"][b, :D].cpu().numpy(), ds["kap"], "kappa_i")
    _bits(ex["th"][b, :D].cpu().numpy(), ds["th"], "theta_i")
    n_acc, n_b = (int(v) for v in ex["n_ev"][b])
    _bits(ex["max_accels"][b, :n_acc].cpu().numpy(), ds["max_accels"], "max_accels")
    assert ex["bidx"][b, :n_b].cpu().numpy().tolist() == ds["bidx"].tolist()
    assert ex["bval"][b, :n_b].cpu().numpy().tolist() == ds["bval"].tolist()
    v = ora.fwd_bwd(ds["kap"], ds["th"], ds["v0"], cons, 0.005, ds["max_accels"], ds["bidx"], ds["bval"])
    vel = res.vel[b, :D].cpu().numpy()
    _bits(vel, v, "velocities")
    pr = ora.profile(geo, apa, apf, cons, 0.01, 0.005, ld, lt, total, K, H, v)
    got = res.path(b)
    assert got["status"] == 0
    assert len(got["times"]) == pr["T"]
    for k in ("times", "positions", "linear_vels", "accelerations", "headings", "angular_vels", "x", "y"):
        _bits(got[k], pr[k], k)
    assert got["nodes_map"].tolist() == pr["nodes_map"].tolist()
    assert got["actions_map"].tolist() == pr["actions_map"].tolist()
    return got


def test_golden_batch_stagewise_and_end_to_end(eng, ora):
    cases, packed = golden_batch()
    res = eng.profile(eng.upload(packed), keep=True)
    torch.cuda.synchronize()
    assert res.status.cpu().numpy().tolist() == [0] * len(cases)
    for b, c in enumerate(cases):
        got = stagewise_check(ora, packed, res, b)
        # ---- against the reference's own outputs
        n = c["n"]
        seg = res.geometry.seg[b, : n - 1].cpu().numpy()
        assert ulp_diff(seg, c["seg"]).max() <= 1               # rows 4,5: L*L vs libm pow(L,2)
        _bits(seg[:, :4], c["seg"][:, :4], "segment rows 0-3 vs reference")
        S = len(c["spline_param_end"])
        np.testing.assert_allclose(res.tables.lut_d[b, : 1000 * S].cpu().numpy(), c["lut_d"], rtol=1e-13)
        np.testing.assert_allclose(res.tables.lut_t[b, : 1000 * S].cpu().numpy(), c["lut_t"], rtol=0, atol=0)
        assert ulp_diff(res.tables.prop_k[b, : 1000 * n].cpu().numpy(), c["prop_k"]).max() <= 8
        assert ulp_diff(res.tables.prop_h[b, : 1000 * n].cpu().numpy(), c["prop_h"]).max() <= 8
        D = len(c["vel"])
        assert int(res.n_samples[b]) == D
        np.testing.assert_allclose(res.extra["t"][b, :D].cpu().numpy(), c["t"], rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(got["vel"], c["vel"], rtol=1e-6, atol=1e-12)
        assert len(got["times"]) == len(c["times"])
        assert got["nodes_map"].tolist() == c["nodes_map"].tolist()
        assert got["actions_map"].tolist() == c["actions_map"].tolist()
        np.testing.assert_allclose(got["x"], c["coords"][:, 0], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["y"], c["coords"][:, 1], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["positions"], c["positions"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(got["times"], c["times"], rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(got["linear_vels"], c["linear_vels"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got["angular_vels"], c["angular_vels"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got["accelerations"], c["accelerations"], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(got["headings"], c["headings"], rtol=1e-9, atol=1e-10)


@pytest.mark.parametrize("kind", ["cfg2", "cfg5"])
def test_random_batch_vs_oracle(eng, ora, kind):
    from vexautonomousplanner_b200 import synth
    B = 192
    packed = synth.random_paths(B, 8, seed=0) if kind == "cfg2" else synth.mixed_paths(B, 8, seed=3)
    res = eng.profile(eng.upload(packed), keep=True)
    torch.cuda.synchronize()
    assert (res.status == 0).all()
    for b in range(0, B, 7):
        stagewise_check(ora, packed, res, b)
    # every path end to end against the oracle with its own libm tables
    summ = res.summary.cpu().numpy()
    for b in range(B):
        A = int(packed.n_ap[b])
        ref = ora.full(packed.node_attr[b], packed.node_flags[b], packed.ap_attr[b, :A], packed.ap_flags[b, :A],
                       packed.cons[b])
        got = res.path(b)
        assert len(got["times"]) == ref["T"], b
        assert int(res.n_samples[b]) == ref["D"], b
        assert got["nodes_map"].tolist() == ref["nodes_map"].tolist()
        assert got["actions_map"].tolist() == ref["actions_map"].tolist()
        np.testing.assert_allclose(got["vel"], ref["vel"], rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(got["x"], ref["x"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["y"], ref["y"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["times"], ref["times"], rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(got["linear_vels"], ref["linear_vels"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got["angular_vels"], ref["angular_vels"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got["headings"], ref["headings"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(summ[b, :4], ref["summary"][:4], rtol=1e-6)


def test_cfg3_16_node_sample(eng, ora):
    from vexautonomousplanner_b200 import synth
    packed = synth.random_paths(24, 16, seed=1)
    res = eng.profile(eng.upload(packed), keep=True)
    torch.cuda.synchronize()
    for b in range(0, 24, 5):
        stagewise_check(ora, packed, res, b)


def test_error_conventions(eng):
    """F7: inputs that crash the reference come back as per-path status codes, the rest of the batch is fine."""
    from vexautonomousplanner_b200 import synth
    packed = synth.random_paths(6, 6, seed=11)
    packed.node_flags[1, 5] |= 1                      # reverse at the last node -> IndexError
    packed.node_attr[2, 0, 2] = 30.0                  # turn at node 0 -> IndexError in the profile
    packed.node_attr[3, 5, 2] = 45.0                  # turn at the last node -> IndexError
    packed.n_nodes[4] = 1                             # fewer than 2 points -> False
    from vexautonomousplanner_b200.packing import rotation_table
    packed.node_attr[:, :, 10], packed.node_attr[:, :, 11] = rotation_table(packed.node_attr[:, :, 2],
                                                                             (packed.node_flags & 1) != 0)
    res = eng.profile(eng.upload(packed))
    torch.cuda.synchronize()
    assert res.status.cpu().numpy().tolist() == [0, -2, -2, -2, -1, 0]
    assert res.n_out.cpu().numpy()[[1, 2, 3, 4]].tolist() == [0, 0, 0, 0]
    assert int(res.n_out[0]) > 100 and int(res.n_out[5]) > 100


def test_cfg2_full_size_properties(eng, ora):
    """4096 x 8-node batch (BASELINE configs[1]): size-independent properties, run-to-run determinism, and a
    strided sample of paths against the oracle.

    (Mirror symmetry is NOT a property of the reference: delta_theta in the velocity passes sees the atan2 branch
    cut, motion_profile_generator.py:202,268, so a mirrored path gets a slightly different profile -- the golden
    pair mixed8_0 / mixed8_0_mirror already differs in nodes_map.)"""
    from vexautonomousplanner_b200 import synth
    packed = synth.random_paths(4096, 8, seed=0)
    db = eng.upload(packed)
    res = eng.profile(db)
    res2 = eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    assert (res.status == 0).all()
    n = res.n_out.long()
    T = res.T_cap
    mask = torch.arange(T, device=n.device)[None, :] < n[:, None]
    # determinism: same bits on a second run (different capacities are allowed, valid regions must agree)
    assert torch.equal(res.n_out, res2.n_out)
    Tm = min(T, res2.T_cap)
    m2 = mask[:, :Tm]
    for i in range(8):
        assert torch.equal(res.out[i][:, :Tm][m2], res2.out[i][:, :Tm][m2])
    # time advances by dt, velocity within the constraint, position is non-decreasing and ends just past L
    tm = res.stream("times")
    d = (tm[:, 1:] - tm[:, :-1])[mask[:, 1:]]
    assert torch.allclose(d, torch.full_like(d, 0.01), rtol=0, atol=1e-9)
    v = res.stream("linear_vels")[mask]
    assert float(v.max()) <= 4.0 + 1e-12 and float(v.min()) >= 0.0
    pos = res.stream("positions")
    assert bool(((pos[:, 1:] - pos[:, :-1])[mask[:, 1:]] > 0).all())
    last = pos.gather(1, (n - 1).clamp(min=0)[:, None])[:, 0]
    assert torch.all(last >= res.summary[:, 1])
    assert torch.all(last <= res.summary[:, 1] + 0.05)
    summ = res.summary.cpu().numpy()
    for b in range(0, 4096, 97):
        ref = ora.full(packed.node_attr[b], packed.node_flags[b], None, None, packed.cons[b])
        assert int(res.n_out[b]) == ref["T"] and int(res.n_samples[b]) == ref["D"]
        np.testing.assert_allclose(summ[b, :4], ref["summary"][:4], rtol=1e-6)
        got = res.path(b)
        np.testing.assert_allclose(got["x"], ref["x"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["linear_vels"], ref["linear_vels"], rtol=1e-6, atol=1e-9)


def test_chunked_equals_serial_bitwise():
    """The chunk-speculative velocity passes must reproduce the serial recurrences bit for bit, for every chunk count,
    including ragged batches, node actions, max_acceleration overrides (the pre-pass's override fix-up) and a path long
    enough to need many fix-up sweeps.  The sampling outputs (t / kappa / theta, max_accels, the boundary map) of the
    fused sampling + pre-pass kernel must equal the serial ones bit for bit as well."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    ser = Engine("cuda:0", velocity_impl="serial", time_impl="serial")
    overrides = synth.mixed_paths(320, 8, seed=9)
    batches = [synth.random_paths(512, 8, seed=5), synth.mixed_paths(512, 8, seed=6), overrides, golden_batch()[1],
               synth.random_paths(3, 120, seed=8)]
    for packed in batches:
        db = ser.upload(packed)
        ref = ser.profile(db, keep=True)
        D = ref.n_samples.long()
        m = torch.arange(ref.vel.shape[1], device=D.device)[None, :] < D[:, None]
        ne = ref.extra["n_ev"].long()
        em = torch.arange(ref.extra["max_accels"].shape[1], device=D.device)[None, :]
        m_acc, m_map = em < ne[:, 0:1], em < ne[:, 1:2]
        if packed is overrides:
            assert bool((ref.status == 0).all())
            A0 = db.cons[:, 1:2]
            assert bool((m_acc & (ref.extra["max_accels"] != A0)).any()), "the batch has no max_acceleration overrides"
        for chunks in (8, 16, 32, 64, 256):
            chk = Engine("cuda:0", velocity_impl="chunked", chunks=chunks, time_impl="split")
            got = chk.profile(db, keep=True)
            torch.cuda.synchronize()
            assert torch.equal(ref.n_samples, got.n_samples)
            for key in ("t", "kap", "th"):
                assert torch.equal(ref.extra[key][m].view(torch.int64), got.extra[key][m].view(torch.int64)), (key, chunks)
            assert torch.equal(ref.vel[m].view(torch.int64), got.vel[m].view(torch.int64)), f"chunks={chunks}"
            assert torch.equal(ref.extra["n_ev"], got.extra["n_ev"])
            ma_ref, ma_got = ref.extra["max_accels"][m_acc], got.extra["max_accels"][m_acc]
            assert torch.equal(ma_ref.view(torch.int64), ma_got.view(torch.int64)), f"chunks={chunks}"
            assert torch.equal(ref.extra["bidx"][m_map], got.extra["bidx"][m_map])
            assert torch.equal(ref.extra["bval"][m_map], got.extra["bval"][m_map])
            assert torch.equal(ref.n_out, got.n_out)
            n = ref.n_out.long()
            Tm = min(ref.T_cap, got.T_cap)
            mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
            for i in range(8):
                assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64))
            assert int(got.extra["rounds"].max()) < chunks
            assert torch.equal(ref.n_maps, got.n_maps)
            nmm = torch.arange(ref.nodes_map.shape[1], device=D.device)[None, :] < ref.n_maps[:, 0:1]
            assert torch.equal(ref.nodes_map[nmm], got.nodes_map[nmm])
            am = torch.arange(ref.actions_map.shape[1], device=D.device)[None, :] < ref.n_maps[:, 1:2]
            assert torch.equal(ref.actions_map[am], got.actions_map[am])
            assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))


def test_time_loop_lane_counts_and_failed_paths_bitwise(monkeypatch):
    """The time loop's warps leave their fast run on a vote, and the paths of a warp are served in turns: the result must not
    depend on how many paths share a warp (1 ... 32, ragged last warp), on failed paths sitting in a live warp (they only
    vote), or on a capacity so small that most steps land in the overflow slot -- all bit for bit against the
    reference-shaped serial kernel (k_resample)."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.packing import rotation_table
    packed = synth.mixed_paths(77, 8, seed=21)
    packed.node_flags[5, packed.n_nodes[5] - 1] |= 1          # reverse at the last node: status -2 inside a live warp
    packed.n_nodes[33] = 1                                    # fewer than two points: status -1
    packed.node_attr[:, :, 10], packed.node_attr[:, :, 11] = rotation_table(packed.node_attr[:, :, 2],
                                                                             (packed.node_flags & 1) != 0)
    ser = Engine("cuda:0", velocity_impl="serial", time_impl="serial")
    db = ser.upload(packed)
    ref = ser.profile(db)
    torch.cuda.synchronize()
    assert int(ref.status[5]) == -2 and int(ref.status[33]) == -1 and int((ref.status == 0).sum()) == 75
    n = ref.n_out.long()
    for lanes, blk in (("1", "128"), ("3", "64"), ("7", "128"), ("7", "64"), ("10", "64"), ("32", "128"), ("32", "64")):
        monkeypatch.setenv("VAP_STATE_LANES", lanes)
        monkeypatch.setenv("VAP_STATE_BLK", blk)          # samples per staged ring block (64 is what large batches use)
        got = Engine("cuda:0").profile(db)
        torch.cuda.synchronize()
        assert torch.equal(ref.status, got.status), lanes
        assert torch.equal(ref.n_out, got.n_out), lanes
        Tm = min(ref.T_cap, got.T_cap)
        mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
        for i in range(8):
            assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), (lanes, i)
        assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64)), lanes
    monkeypatch.delenv("VAP_STATE_LANES")
    monkeypatch.delenv("VAP_STATE_BLK")
    # an undersized row capacity: the paths come back as ST_CAPACITY with their true needs, and the redo is exact
    eng = Engine("cuda:0")
    D_cap, _ = eng.plan_capacities(db)
    small = eng.profile_batch(db, D_cap, 256)
    torch.cuda.synchronize()
    assert torch.equal(ref.n_out, small.n_out)
    Tm = min(ref.T_cap, small.T_cap)
    mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
    for i in range(8):
        assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), small.out[i][:, :Tm][mt].view(torch.int64)), i


def test_oscillating_positions_are_redone_serially():
    """30-node mixed paths, dt = 0.02, dd = 0.0025 and max_dec up to 160: near stops the position moves back and forth across
    action points and node boundaries more often than the parallel event detection has candidate slots for (27 of these
    2048 paths).  The time stage redoes exactly those paths with the reference-shaped serial kernel: same status (OK), same
    bits as the all-serial run, nothing left as VAP_ERR_EVENTS."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    rng = np.random.default_rng(1001)
    rng.choice([3, 5, 8, 12, 20, 30]); rng.choice([97, 640, 2048, 5000])     # the draws of the stress run that found the case
    packed = synth.mixed_paths(2048, 30, seed=201)
    B = packed.cons.shape[0]
    packed.cons[:, 0] = rng.uniform(0.3, 14.0, B)
    packed.cons[:, 1] = 10.0 ** rng.uniform(-0.7, 1.6, B)
    packed.cons[:, 2] = 10.0 ** rng.uniform(-0.7, 2.2, B)
    packed.cons[:, 5] = rng.uniform(0.4, 2.5, B)
    ser = Engine("cuda:0", dt=0.02, dd=0.0025, time_impl="serial")
    fast = Engine("cuda:0", dt=0.02, dd=0.0025)
    ref = ser.profile(ser.upload(packed))
    db = fast.upload(packed)
    for got in (fast.profile(db), fast.profile_batch(db)):          # staged entry points and the single C call
        torch.cuda.synchronize()
        assert int((got.status == -6).sum()) == 0
        assert torch.equal(ref.status, got.status)
        assert torch.equal(ref.n_out, got.n_out)
        n = ref.n_out.long()
        Tm = min(ref.T_cap, got.T_cap)
        mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
        for i in range(8):
            assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), i
        assert torch.equal(ref.n_maps, got.n_maps)
        nmm = torch.arange(ref.nodes_map.shape[1], device=n.device)[None, :] < ref.n_maps[:, 0:1]
        assert torch.equal(ref.nodes_map[nmm], got.nodes_map[nmm])
        am = torch.arange(ref.actions_map.shape[1], device=n.device)[None, :] < ref.n_maps[:, 1:2]
        assert torch.equal(ref.actions_map[am], got.actions_map[am])
        assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))


@pytest.mark.parametrize("dt,dd", [(0.01, 0.005), (0.025, 0.01), (0.004, 0.02)])
def test_time_loop_fuzz_constraints_bitwise(dt, dd):
    """The fast time loop against the reference-shaped serial kernel on constraints far from the factory values -- crawling
    and very fast robots, max_dec large enough for the position to move BACKWARDS in a step (delta_pos < 0 when
    max_dec > 0.2 / dt), steps that jump over many distance samples or stay inside one -- bit for bit, status included."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    rng = np.random.default_rng(int(dt * 1e4) + 7)
    packed = synth.mixed_paths(640, 8, seed=31)
    B = packed.cons.shape[0]
    packed.cons[:, 0] = rng.uniform(0.3, 14.0, B)            # max_vel
    packed.cons[:, 1] = 10.0 ** rng.uniform(-0.7, 1.6, B)    # max_acc 0.2 ... 40
    packed.cons[:, 2] = 10.0 ** rng.uniform(-0.7, 2.2, B)    # max_dec 0.2 ... 160
    packed.cons[:, 5] = rng.uniform(0.4, 2.5, B)             # track width
    ser = Engine("cuda:0", dt=dt, dd=dd, time_impl="serial")
    fast = Engine("cuda:0", dt=dt, dd=dd)
    ref = ser.profile(ser.upload(packed))
    got = fast.profile(fast.upload(packed), keep=True)
    torch.cuda.synchronize()
    assert torch.equal(ref.status, got.status)
    assert int((ref.status == 0).sum()) > B // 2
    bad = (ref.n_out != got.n_out).nonzero().flatten().tolist()
    assert not bad, [(b, int(ref.n_out[b]), int(got.n_out[b]), int(got.extra["n_main"][b])) for b in bad[:6]]
    n = ref.n_out.long()
    Tm = min(ref.T_cap, got.T_cap)
    mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
    for i in range(8):
        assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), i
    assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))


def test_short_paths_and_chunk_edges():
    """Paths far shorter than the chunk count (one step per chunk, idle chunks), lengths around multiples of the chunk
    count, a stop node (exact reset of the forward pass) and every warm-up length: fast == serial bit for bit."""
    import os
    import vexautonomousplanner_b200 as vap
    from vexautonomousplanner_b200.engine import Engine
    cons = [4.0, 8.0, 8.0, 0.8, 16.0, 12.5 / 12]
    paths = []
    for L in (0.012, 0.05, 0.155, 0.16, 0.165, 0.32, 0.645, 1.0, 1.285, 2.0):       # 3 .. 400 distance samples
        paths.append(np.array([[1.0, 1.0], [1.0 + L, 1.0 + 0.3 * L]]))
    paths.append(np.array([[0.0, 0.0], [0.4, 0.1], [0.7, -0.2]]))
    N = max(len(p) for p in paths)
    pts = np.zeros((len(paths), N, 2)); nn = np.zeros(len(paths), dtype=np.int32)
    for b, p in enumerate(paths):
        pts[b, :len(p)] = p; pts[b, len(p):] = p[-1] + np.arange(1, N - len(p) + 1)[:, None] * 0.5; nn[b] = len(p)
    stop = np.zeros((len(paths), N), dtype=bool); stop[-1, 1] = True
    packed = vap.pack_arrays(pts, cons, n_nodes=nn, stop=stop)
    ser = Engine("cuda:0", velocity_impl="serial", time_impl="serial")
    ref = ser.profile(ser.upload(packed), keep=True)
    assert bool((ref.status == 0).all())
    old = os.environ.get("VAP_CHUNK_WARM")
    try:
        for warm in ("0", "1", "7", "96", "1000"):
            os.environ["VAP_CHUNK_WARM"] = warm
            for chunks in (8, 16, 32, 128):
                got = Engine("cuda:0", chunks=chunks).profile(ser.upload(packed), keep=True)
                torch.cuda.synchronize()
                assert torch.equal(ref.n_samples, got.n_samples) and torch.equal(ref.n_out, got.n_out)
                D = ref.n_samples.long()
                m = torch.arange(ref.vel.shape[1], device=D.device)[None, :] < D[:, None]
                assert torch.equal(ref.vel[m].view(torch.int64), got.vel[m].view(torch.int64)), (warm, chunks)
                n = ref.n_out.long()
                Tm = min(ref.T_cap, got.T_cap)
                mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
                for i in range(8):
                    assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), (warm, chunks, i)
    finally:
        if old is None:
            os.environ.pop("VAP_CHUNK_WARM", None)
        else:
            os.environ["VAP_CHUNK_WARM"] = old


def _same_valid_bits(ref, got):
    assert torch.equal(ref.status, got.status) and torch.equal(ref.n_out, got.n_out)
    assert torch.equal(ref.n_samples, got.n_samples)
    n = ref.n_out.long()
    Tm = min(ref.T_cap, got.T_cap)
    mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
    for i in range(8):
        assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), i
    D = ref.n_samples.long()
    md = torch.arange(min(ref.vel.shape[1], got.vel.shape[1]), device=n.device)[None, :] < D[:, None]
    assert torch.equal(ref.vel[:, :md.shape[1]][md].view(torch.int64), got.vel[:, :md.shape[1]][md].view(torch.int64))
    assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))


def test_capacity_retry():
    """A deliberately undersized plan (through vap_profile_batch) and an undersized row estimate of the staged run must
    be detected on the device and redone exactly."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    packed = synth.mixed_paths(64, 8, seed=9)
    e1 = Engine("cuda:0")
    db = e1.upload(packed)
    ref = e1.profile(db)
    torch.cuda.synchronize()
    assert bool((ref.status == 0).all())
    e2 = Engine("cuda:0")
    key = (db.B, db.N_max, db.A_max, db.max_splines)
    for plan in ((int(ref.n_samples.max()) + 8, 300),            # T_cap far too small
                 (1000, ref.T_cap)):                              # D_cap far too small
        e2._plan[key] = plan
        got = e2.profile(db, reuse_plan=True)
        torch.cuda.synchronize()
        assert "need" in got.extra                                # the planned step is vap_profile_batch
        _same_valid_bits(ref, got)
        assert e2._plan[key] == (got.vel.shape[1], got.T_cap)
    # the staged run: its T_cap estimate (Engine._plan_rows) replaced by one far too small; the time stage is redone with
    # T_cap = max(n_main + ceil(ins_est)) + 8
    e3 = Engine("cuda:0")
    forced = []

    def small(est, status):
        forced.append(Engine._plan_rows(e3, est, status) // 5)
        return forced[-1]

    e3._plan_rows = small
    got = e3.profile(db)
    torch.cuda.synchronize()
    assert len(forced) == 1 and int(ref.n_out.max()) > forced[0]      # the rows overflowed once
    _same_valid_bits(ref, got)
    assert e3._plan[key] == (got.vel.shape[1], got.T_cap)


def test_split_time_stage_needs_the_chunked_velocity_stage():
    """The split time stage redoes an overflow with the chunked velocity stage's bound of the inserted rows, which the
    serial velocity stage does not compute: that combination is refused."""
    from vexautonomousplanner_b200.engine import Engine
    with pytest.raises(ValueError):
        Engine("cuda:0", velocity_impl="serial", time_impl="split")


def test_const_division_is_ieee():
    """The hoisted-reciprocal division by dt inside the time loop must equal the IEEE quotient for every numerator."""
    import ctypes as C
    from vexautonomousplanner_b200 import _lib
    L = _lib.lib()
    bad = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for seed, b in ((1, 0.01), (2, 0.01), (3, 0.005), (4, 0.025), (5, 0.02), (6, 1.0 / 3.0)):
        _lib.check(L.vap_test_div_const(C.c_int64(1 << 26), C.c_uint64(seed), C.c_double(b), C.c_void_p(bad.data_ptr()), st))
    torch.cuda.synchronize()
    assert int(bad.item()) == 0


def test_recip_division_is_ieee():
    """The velocity passes divide by 2|dtheta| with the reciprocal made by the pre-pass and two fused residual corrections;
    2^30 random (numerator, denominator) pairs, incl. zero denominators / numerators and all-ones significands, must give
    the IEEE quotient bit for bit."""
    import ctypes as C
    from vexautonomousplanner_b200 import _lib
    L = _lib.lib()
    bad = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for seed in range(4):
        _lib.check(L.vap_test_div_recip(C.c_int64(1 << 28), C.c_uint64(seed * 7919 + 1), C.c_void_p(bad.data_ptr()), st))
    torch.cuda.synchronize()
    assert int(bad.item()) == 0


def test_accelerators_do_not_change_bits():
    """The inverse LUT index (seeded searchsorted) and the tabulated lerp reciprocals are pure accelerators: with NULL passed
    for both, the kernels fall back to the binary search / the plain divisions and must produce the same bits."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    fast = Engine("cuda:0")
    plain = Engine("cuda:0", accelerators=False)
    for packed in (synth.random_paths(300, 8, seed=31), synth.mixed_paths(200, 8, seed=32), synth.random_paths(40, 16, seed=33)):
        a = fast.profile(fast.upload(packed), keep=True)
        b = plain.profile(plain.upload(packed), keep=True)
        torch.cuda.synchronize()
        assert torch.equal(a.n_out, b.n_out) and torch.equal(a.status, b.status) and torch.equal(a.n_samples, b.n_samples)
        D = a.n_samples.long()
        md = torch.arange(a.vel.shape[1], device=D.device)[None, :] < D[:, None]
        for name in ("t", "kap", "th"):
            assert torch.equal(a.extra[name][md].view(torch.int64), b.extra[name][md].view(torch.int64)), name
        assert torch.equal(a.vel[md].view(torch.int64), b.vel[md].view(torch.int64))
        n = a.n_out.long()
        Tm = min(a.T_cap, b.T_cap)
        mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
        for i in range(8):
            assert torch.equal(a.out[i][:, :Tm][mt].view(torch.int64), b.out[i][:, :Tm][mt].view(torch.int64)), i
        assert torch.equal(a.summary.view(torch.int64), b.summary.view(torch.int64))


def test_tiled_multistream_equals_untiled():
    """Row tiles on separate CUDA streams must give the same bits as one pass over the batch."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    for packed in (synth.random_paths(700, 8, seed=21), synth.mixed_paths(300, 8, seed=22)):
        db = eng.upload(packed)
        ref = eng.profile(db)
        for tiles in (2, 4, 7):
            got = eng.profile(db, reuse_plan=True, tiles=tiles)
            torch.cuda.synchronize()
            assert torch.equal(ref.n_out, got.n_out) and torch.equal(ref.status, got.status)
            assert torch.equal(ref.n_samples, got.n_samples)
            n = ref.n_out.long()
            Tm = min(ref.T_cap, got.T_cap)
            mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
            for i in range(8):
                assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64))
            assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))
            nmm = torch.arange(ref.nodes_map.shape[1], device=n.device)[None, :] < ref.n_maps[:, 0:1]
            assert torch.equal(ref.nodes_map[nmm], got.nodes_map[nmm])


def test_cuda_graph_replay_equals_eager():
    """The captured step (tiles forked over streams inside one CUDA graph) reproduces the eager results bit for bit,
    also after new inputs are copied into the static buffers."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    a, b = synth.mixed_paths(512, 8, seed=31), synth.mixed_paths(512, 8, seed=32)
    ref_a, ref_b = eng.profile(eng.upload(a)), eng.profile(eng.upload(b))
    g = eng.capture(eng.upload(a), tiles=4)
    for ref, new in ((ref_a, None), (ref_b, eng.upload(b)), (ref_a, eng.upload(a))):
        got = g.run(new)
        torch.cuda.synchronize()
        assert torch.equal(ref.n_out, got.n_out) and torch.equal(ref.status, got.status)
        n = ref.n_out.long()
        Tm = min(ref.T_cap, got.T_cap)
        mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
        for i in range(8):
            assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64))


def test_host_in_host_out_packing():
    """run_host: numpy in, pinned host buffers out (dense rows written by the pack kernels) == device results."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    packed = synth.mixed_paths(400, 8, seed=41)
    packed.node_attr[7, 0, 2] = 30.0            # one failing path (turn at node 0): packs to zero rows
    ref = eng.profile(eng.upload(packed))
    g = eng.capture(eng.upload(packed), tiles=3, to_host=True)
    state = None
    for it in range(4):
        if it < 2:
            h = g.run_host(packed)                              # pack kernels write pinned host memory (CUDA graph)
        else:
            h = eng.profile_to_host(packed, tiles=5, state=state)   # dense device rows + copy engine
            state = h.state
        assert h.status.tolist() == ref.status.cpu().tolist()
        assert h.n_out.tolist() == ref.n_out.cpu().tolist()
        for b in (0, 7, 133, 134, 266, 399):
            got, want = h.path(b), ref.path(b)
            for k in ("times", "positions", "linear_vels", "accelerations", "headings", "angular_vels", "x", "y"):
                assert np.array_equal(got[k], want[k]), (b, k)
            assert got["nodes_map"].tolist() == want["nodes_map"].tolist()
        assert np.array_equal(h.summary.numpy(), ref.summary.cpu().numpy())
        assert h.bytes_per_step() < 8 * 8 * 400 * g.T_cap


def test_cfg4_single_long_path(ora):
    """BASELINE configs[3]: one very long path (N = 801 nodes, about 10^6 distance samples) -- the case that needs the
    intra-path chunked passes (256 chunks).  Every stage bit-exact against the oracle fed with the engine's tables."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    packed = synth.long_path(801, seed=2)
    res = eng.profile(eng.upload(packed), keep=True)
    torch.cuda.synchronize()
    assert int(res.status[0]) == 0
    assert int(res.n_samples[0]) > 900_000
    got = stagewise_check(ora, packed, res, 0)
    assert len(got["times"]) > 100_000
    assert int(res.extra["rounds"].max()) < 256


def test_late_acceleration_override_on_long_path(ora):
    """A 300-node path whose nodes all carry max_acceleration = the path's own value except node 280: more regimes than
    one pre-pass CTA has threads, and the only real override sits past the 256th.  Every stage bit-exact against the oracle."""
    import numpy as np
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.packing import pack_arrays
    from vexautonomousplanner_b200.engine import Engine
    rng = np.random.default_rng(11)
    N = 300
    cons = np.array(synth.FACTORY, dtype=np.float64)
    ma = np.full((1, N), cons[1])
    ma[0, 280] = 0.5 * cons[1]
    packed = pack_arrays(synth.px_to_ft(synth.random_pixels(rng, 1, N)), cons, max_acceleration=ma)
    eng = Engine("cuda:0")
    res = eng.profile(eng.upload(packed), keep=True)
    torch.cuda.synchronize()
    assert int(res.status[0]) == 0
    stagewise_check(ora, packed, res, 0)
    plain = pack_arrays(synth.px_to_ft(synth.random_pixels(np.random.default_rng(11), 1, N)), cons)
    res2 = eng.profile(eng.upload(plain), keep=True)
    torch.cuda.synchronize()
    assert int(res.n_out[0]) != int(res2.n_out[0])          # the override took effect


def test_cfg3_tiled_job_summaries(ora):
    """BASELINE configs[2] in miniature: a job bigger than one call is tiled by profile_many; summaries match the oracle."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    packed = synth.random_paths(700, 16, seed=1)
    seen = []
    summ = eng.profile_many(packed, tile_paths=256, sink=lambda lo, hi, r: seen.append((lo, hi, int(r.n_out.sum())))).cpu().numpy()
    assert [s[:2] for s in seen] == [(0, 256), (256, 512), (512, 700)]
    assert summ.shape == (700, 5) and (summ[:, 4] == 0).all()
    assert sum(s[2] for s in seen) == int(summ[:, 0].sum())
    for b in range(0, 700, 41):
        ref = ora.full(packed.node_attr[b], packed.node_flags[b], None, None, packed.cons[b])
        assert int(summ[b, 0]) == ref["T"]
        np.testing.assert_allclose(summ[b, :4], ref["summary"][:4], rtol=1e-6)


def test_stream_to_host_pipeline():
    """Bulk streaming API: results of a pipelined stream equal the one-batch-at-a-time results, in order."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    batches = [synth.mixed_paths(256, 8, seed=50 + i) for i in range(5)]
    refs = [eng.profile(eng.upload(p)) for p in batches]
    n = 0
    for h, ref in zip(eng.stream_to_host(batches, tiles=3), refs):
        assert h.n_out.tolist() == ref.n_out.cpu().tolist()
        for b in (0, 100, 255):
            got, want = h.path(b), ref.path(b)
            for k in ("times", "x", "linear_vels", "headings"):
                assert np.array_equal(got[k], want[k])
        n += 1
    assert n == 5


@pytest.mark.parametrize("kind,nn", [("cfg5", 8), ("cfg2", 8), ("cfg3", 16)])
def test_fuzz_summaries_against_oracle(eng, ora, kind, nn):
    """Thousands of random paths: sample counts exact, summary values within tolerance, for every path of the batch
    (the oracle's OpenMP batch driver computes the reference summaries in a few seconds)."""
    from vexautonomousplanner_b200 import synth
    B = 3000 if nn == 8 else 600
    packed = synth.mixed_paths(B, nn, seed=77) if kind == "cfg5" else synth.random_paths(B, nn, seed=78)
    res = eng.profile(eng.upload(packed))
    torch.cuda.synchronize()
    got = res.summary.cpu().numpy()
    want = ora.full_batch(packed.node_attr, packed.node_flags, packed.cons, n_ap=packed.n_ap, ap_attr=packed.ap_attr,
                          ap_flags=packed.ap_flags, cap_d=80000, cap_t=60000)
    assert (got[:, 4] == 0).all() and (want[:, 4] == 0).all()
    bad = np.nonzero(got[:, 0] != want[:, 0])[0]
    assert bad.size == 0, f"time-sample counts differ for paths {bad[:10].tolist()}"
    np.testing.assert_allclose(got[:, 1], want[:, 1], rtol=1e-12)        # total length
    np.testing.assert_allclose(got[:, 2], want[:, 2], rtol=1e-6)         # t_end
    np.testing.assert_allclose(got[:, 3], want[:, 3], rtol=1e-6)         # max |v|


@pytest.mark.parametrize("dt,dd", [(0.01, 0.005), (0.02, 0.0025)])
def test_fuzz_extreme_constraints_against_oracle(ora, dt, dd):
    """Mixed paths with constraints far from the factory values (crawling and very fast robots, max_acc 0.2 ... 40, wide and
    narrow track widths; max_dec below 0.2 / dt so that no step moves backwards -- the oscillating regime is chaotic in the
    last bits of the tables and has its own bitwise and reference-pinned tests) and a second dt / dd pair, against the
    oracle: status and time-sample count exact for every path, summary values within the north-star tolerances."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    rng = np.random.default_rng(int(dd * 1e5) + 3)
    packed = synth.mixed_paths(600, 8, seed=91)
    B = packed.cons.shape[0]
    packed.cons[:, 0] = rng.uniform(0.3, 14.0, B)
    packed.cons[:, 1] = 10.0 ** rng.uniform(-0.7, 1.6, B)
    packed.cons[:, 2] = 10.0 ** rng.uniform(-0.7, np.log10(0.18 / dt), B)
    packed.cons[:, 5] = rng.uniform(0.4, 2.5, B)
    eng = Engine("cuda:0", dt=dt, dd=dd)
    res = eng.profile(eng.upload(packed))
    torch.cuda.synchronize()
    got = res.summary.cpu().numpy()
    want = ora.full_batch(packed.node_attr, packed.node_flags, packed.cons, n_ap=packed.n_ap, ap_attr=packed.ap_attr,
                          ap_flags=packed.ap_flags, dt=dt, dd=dd, cap_d=400000, cap_t=400000)
    assert (got[:, 4] == want[:, 4]).all(), np.nonzero(got[:, 4] != want[:, 4])[0][:10].tolist()
    ok = want[:, 4] == 0
    assert ok.sum() > B // 2
    bad = np.nonzero((got[:, 0] != want[:, 0]) & ok)[0]
    assert bad.size == 0, f"time-sample counts differ for paths {bad[:10].tolist()}"
    np.testing.assert_allclose(got[ok, 1], want[ok, 1], rtol=1e-12)        # total length
    np.testing.assert_allclose(got[ok, 2], want[ok, 2], rtol=1e-6)         # t_end
    np.testing.assert_allclose(got[ok, 3], want[ok, 3], rtol=1e-6)         # max |v|


def test_degenerate_inputs_never_hang(eng):
    """Inputs for which the reference would loop forever or blow up come back with a status instead of hanging the GPU:
    a deceleration limit so large that a step moves backwards, an absurd wait, an absurdly slow turn profile."""
    from vexautonomousplanner_b200 import synth
    packed = synth.random_paths(6, 6, seed=91)
    packed.cons[1, 1] = packed.cons[1, 2] = 250.0           # dpos = 0.1*dt - 0.5*250*dt^2 < 0 near a stop: never reaches L
    packed.node_flags[1, 2] |= 2                             # a stop node, so the profile really brakes
    packed.node_attr[2, 2, 3] = 1e12                         # wait of 1e12 s = 1e14 rows
    packed.node_attr[3, 2, 2] = 90.0; packed.cons[3, 1] = packed.cons[3, 2] = 1e-14   # turn profile with 1e9+ samples
    from vexautonomousplanner_b200.packing import rotation_table
    packed.node_attr[:, :, 10], packed.node_attr[:, :, 11] = rotation_table(packed.node_attr[:, :, 2], (packed.node_flags & 1) != 0)
    res = eng.profile(eng.upload(packed))
    torch.cuda.synchronize()
    st = res.status.cpu().numpy().tolist()
    assert st[0] == 0 and st[4] == 0 and st[5] == 0
    assert st[2] == -5 and st[3] in (-5, -4, 0) and st[1] in (-5, 0)
    assert int(res.n_out[2]) == 0


def test_gl_arclength_and_inverse_batched_bit_exact(ora):
    """Row a4: Gauss-Legendre arc length and its bisection inverse (quintic_hermite_spline.py:592-717), BATCHED --
    every spline of every golden case in one launch, > 10^4 queries per launch, path[q] / spl[q] indirection -- bit for
    bit against the oracle (which tests/test_oracle_golden.py pins bit for bit to the reference's own values), and
    directly against the reference's fixture values wherever the segment table of the spline is bit-identical to the
    reference's (the x*x vs pow(x, 2) ulp of DESIGN.md 3.5 can touch rows 4-5 of a segment)."""
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    cases, packed = golden_batch()
    db = eng.upload(packed)
    g = eng.build_geometry(db)
    torch.cuda.synchronize()
    assert g.status.cpu().numpy().tolist() == [0] * len(cases)
    pts, wts = np.polynomial.legendre.leggauss(20)
    rng = np.random.default_rng(11)
    qa = dict(path=[], spl=[], a=[], b=[], fix=[])      # arc-length queries
    qi = dict(path=[], spl=[], a=[], fix=[])            # inverse queries
    geos = []
    for bi, c in enumerate(cases):
        n = c["n"]
        geo = ora.Geometry(packed.node_attr[bi, :n], packed.node_flags[bi, :n])
        _bits(g.seg[bi, : n - 1].cpu().numpy(), geo.seg, "segments")
        geos.append(geo)
        same_seg = bit_equal(geo.seg, c["seg"])
        for k, t0, t1, want in zip(c["gl_spline"], c["gl_t0"], c["gl_t1"], c["gl_len"]):
            qa["path"].append(bi); qa["spl"].append(int(k)); qa["a"].append(t0); qa["b"].append(t1)
            qa["fix"].append((want, same_seg))
        for k, s, want in zip(c["inv_spline"], c["inv_s"], c["inv_t"]):
            qi["path"].append(bi); qi["spl"].append(int(k)); qi["a"].append(s); qi["fix"].append((want, same_seg))
        for k in range(geo.S):
            pe = float(geo.param_end[k])
            tot = geo.gl_arclen(k, 0.0, pe, pts, wts)
            lo = rng.uniform(0, pe, 130); hi = rng.uniform(0, pe, 130)
            t0, t1 = np.minimum(lo, hi), np.maximum(lo, hi)
            t0[0], t1[0] = 0.0, pe                                   # whole spline
            t0[1], t1[1] = 0.0, np.nextafter(0.0, 1.0)               # degenerate but legal range
            for x, y in zip(t0, t1):
                if x < y:
                    qa["path"].append(bi); qa["spl"].append(k); qa["a"].append(x); qa["b"].append(y); qa["fix"].append(None)
            ss = np.concatenate([rng.uniform(0, tot, 127), [0.0, tot, np.nextafter(tot, 0.0)]])
            for s in ss:
                qi["path"].append(bi); qi["spl"].append(k); qi["a"].append(s); qi["fix"].append(None)
    # pad both launches beyond 10^4 queries by repeating random picks (different threads, same answers)
    for q in (qa, qi):
        m = len(q["a"])
        extra = rng.integers(0, m, max(0, 12000 - m))
        for key in q:
            q[key] = list(q[key]) + [q[key][j] for j in extra]
    va, sa = eng.gl_queries(g, qa["path"], qa["spl"], qa["a"], qa["b"], mode=0)
    vi, si = eng.gl_queries(g, qi["path"], qi["spl"], qi["a"], 1e-6, mode=1)
    assert len(qa["a"]) >= 10000 and len(qi["a"]) >= 10000
    assert int(sa.abs().max()) == 0 and int(si.abs().max()) == 0
    va, vi = va.cpu().numpy(), vi.cpu().numpy()
    want_a = np.array([geos[p].gl_arclen(k, x, y, pts, wts) for p, k, x, y in zip(qa["path"], qa["spl"], qa["a"], qa["b"])])
    _bits(va, want_a, "batched GL arc length vs oracle")
    want_i = np.array([geos[p].gl_inverse(k, s, pts, wts) for p, k, s in zip(qi["path"], qi["spl"], qi["a"])])
    _bits(vi, want_i, "batched GL inverse vs oracle")
    n_exact = 0
    for got, fix in list(zip(va, qa["fix"])) + list(zip(vi, qi["fix"])):
        if fix is None:
            continue
        want, same = fix
        if same:
            assert np.float64(got).view(np.int64) == np.float64(want).view(np.int64)     # the reference's own value
            n_exact += 1
        else:
            np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-15)
    assert n_exact > 500
    # error convention: t_start >= t_end, out of range, negative / too large arc length -> the reference raises ValueError
    bad, sb = eng.gl_queries(g, [0, 0, 0], [0, 0, 0], [1.0, -0.5, 0.0], [1.0, 1.0, 99.0], mode=0)
    assert sb.cpu().numpy().tolist() == [-3, -3, -3]
    bad, sb = eng.gl_queries(g, [0, 0], [0, 0], [-1.0, 1e9], 1e-6, mode=1)
    assert sb.cpu().numpy().tolist() == [-3, -3]


def test_bad_lengths_do_not_break_the_batch():
    """Sizing is per batch, status is per path: a NaN coordinate (the reference's loops then simply do not run), an
    absurdly long path (5e8 distance samples: the reference would run out of memory) and a path with an infinite length
    neither raise during sizing nor size the buffers of the healthy paths; repeated calls (plan reuse) keep working."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    packed = synth.random_paths(6, 6, seed=92)
    packed.node_attr[1, 2, 0] = np.nan
    packed.node_attr[2, 3, 0:2] = [2.5e6, -2.5e6]          # > 5e7 samples at dd = 0.005
    packed.node_attr[3, 1, 1] = np.inf
    db = eng.upload(packed)
    ref = eng.profile(eng.upload(synth.random_paths(6, 6, seed=92)))
    for reuse in (False, True, True):
        res = eng.profile(db, reuse_plan=reuse)
        torch.cuda.synchronize()
        st = res.status.cpu().numpy().tolist()
        assert st[0] == 0 and st[4] == 0 and st[5] == 0, st
        assert st[2] == -5, st
        assert st[1] != -4 and st[3] != -4, st              # never a capacity retry loop
        assert int(res.n_out[1]) == 0 and int(res.n_out[2]) == 0 and int(res.n_out[3]) == 0
        for b in (0, 4, 5):
            assert int(res.n_out[b]) == int(ref.n_out[b])
            assert torch.equal(res.out[:, b, : int(res.n_out[b])], ref.out[:, b, : int(ref.n_out[b])])
        assert res.vel.shape[1] < 40000                     # the outliers did not size the distance-domain rows


@pytest.mark.gpu
def test_profile_batch_single_c_entry_raw_ctypes(ora):
    """The drop-in boundary as a C caller sees it (include/vap.h, SURVEY.md 8b): the whole hot path through the ONE symbol
    vap_profile_batch, on buffers from cudaMalloc, with no Engine, no torch tensors and no Python orchestration.  Checked
    against the oracle on every path of a mixed batch, against Engine.profile bit for bit, and for the device-side
    capacity protocol (VAP_ERR_CAPACITY + need[] -> retry)."""
    import ctypes as C
    from vexautonomousplanner_b200 import _lib, synth
    from vexautonomousplanner_b200.engine import Engine
    torch.zeros(1, device="cuda")                             # the CUDA runtime is loaded (and its context created) by torch
    L = _lib.lib()
    rt = C.CDLL([ln.split()[-1] for ln in open("/proc/self/maps") if "libcudart" in ln][0])
    rt.cudaMalloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    rt.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    rt.cudaFree.argtypes = [C.c_void_p]
    H2D, D2H = 1, 2
    bufs = []

    def dev(nbytes):
        p = C.c_void_p()
        assert rt.cudaMalloc(C.byref(p), max(int(nbytes), 256)) == 0
        bufs.append(p)
        return p

    def up(a):
        a = np.ascontiguousarray(a)
        p = dev(a.nbytes)
        assert rt.cudaMemcpy(p, a.ctypes.data_as(C.c_void_p), a.nbytes, H2D) == 0
        return p

    def down(p, shape, dtype):
        a = np.empty(shape, dtype=dtype)
        assert rt.cudaMemcpy(a.ctypes.data_as(C.c_void_p), p, a.nbytes, D2H) == 0
        return a

    packed = synth.mixed_paths(48, 8, seed=11)
    B, N, A = packed.B, packed.N_max, packed.A_max
    S = packed.max_splines()
    dt, dd, samples, spn, chunks = 0.01, 0.005, 1000, 1000, 32
    d_in = [up(x) for x in (packed.node_attr, packed.node_flags, packed.n_nodes, packed.ap_attr, packed.ap_flags, packed.n_ap,
                            packed.cons)]

    def run(D_cap, T_cap):
        n_grid = D_cap + 2
        dgrid, rden = dev(8 * n_grid), dev(8 * n_grid)
        assert L.vap_build_dgrid(C.c_int64(n_grid), C.c_double(dd), dgrid, None) == 0
        assert L.vap_build_lerp_recip(C.c_int64(n_grid), C.c_double(dd), rden, None) == 0
        nbytes = L.vap_workspace_bytes(C.c_int64(B), N, A, S, samples, spn, C.c_int64(D_cap), C.c_int64(T_cap), chunks)
        assert nbytes > 0
        ws = dev(nbytes)
        o = dict(out=dev(8 * 8 * B * T_cap), n_out=dev(4 * B), nodes_map=dev(4 * B * (N + 1)), actions_map=dev(4 * B * max(A, 1)),
                 n_maps=dev(8 * B), status=dev(4 * B), summary=dev(40 * B), vel=dev(8 * B * D_cap), n_samples=dev(4 * B),
                 need=dev(24))
        rc = L.vap_profile_batch(C.c_int64(B), N, A, S, *d_in, C.c_double(dt), C.c_double(dd), C.c_double(0.01), C.c_double(0.01),
                                 samples, spn, C.c_int64(D_cap), C.c_int64(T_cap), chunks, dgrid, C.c_int64(n_grid), rden,
                                 C.c_int64(n_grid), ws, C.c_int64(nbytes), o["out"], C.c_int64(0), o["n_out"], o["nodes_map"],
                                 o["actions_map"], o["n_maps"], o["status"], o["summary"], o["vel"], o["n_samples"], o["need"], None)
        assert rc == 0, L.vap_last_error()
        assert rt.cudaDeviceSynchronize() == 0
        return dict(out=down(o["out"], (8, B, T_cap), np.float64), n_out=down(o["n_out"], (B,), np.int32),
                    nodes_map=down(o["nodes_map"], (B, N + 1), np.int32), actions_map=down(o["actions_map"], (B, max(A, 1)), np.int32),
                    n_maps=down(o["n_maps"], (B, 2), np.int32), status=down(o["status"], (B,), np.int32),
                    summary=down(o["summary"], (B, 5), np.float64), vel=down(o["vel"], (B, D_cap), np.float64),
                    n_samples=down(o["n_samples"], (B,), np.int32), need=down(o["need"], (3,), np.int64))

    try:
        # 1. undersized on purpose: every path reports VAP_ERR_CAPACITY or fits; need[] says what the batch wants
        small = run(1024, 256)
        assert (small["status"] == -4).any()
        d_need, t_est, _ = (int(v) for v in small["need"])
        assert d_need > 1024
        # 2. the retry a C caller would make
        D_cap = (d_need + 8 + 127) // 128 * 128
        got = run(D_cap, int(t_est * 1.10) + 64)
        if (got["status"] == -4).any():                       # the time estimate is only an estimate: one more exact retry
            got = run(D_cap, int(max(got["need"][1], got["need"][2])) + 64)
        assert (got["status"] == 0).all(), (got["status"], got["need"], got["n_samples"], got["n_out"], D_cap)
        # 3. every path against the oracle (engine arithmetic: mode 1), integers exact
        for b in range(B):
            na_ = int(packed.n_ap[b])
            ref = ora.full(packed.node_attr[b], packed.node_flags[b], packed.ap_attr[b, :na_] if na_ else None,
                           packed.ap_flags[b, :na_] if na_ else None, packed.cons[b])
            T = int(got["n_out"][b])
            assert T == ref["T"] and int(got["n_samples"][b]) == ref["D"]
            nm, am = (int(v) for v in got["n_maps"][b])
            assert got["nodes_map"][b, :nm].tolist() == ref["nodes_map"].tolist()
            assert got["actions_map"][b, :am].tolist() == ref["actions_map"].tolist()
            np.testing.assert_allclose(got["vel"][b, :ref["D"]], ref["vel"], rtol=1e-6, atol=1e-12)
            tols = dict(times=(1e-6, 1e-12), linear_vels=(1e-6, 1e-9), angular_vels=(1e-6, 1e-9), headings=(1e-9, 1e-10),
                        x=(1e-9, 1e-10), y=(1e-9, 1e-10))
            for i, nm_ in enumerate(("times", "positions", "linear_vels", "accelerations", "headings", "angular_vels", "x", "y")):
                if nm_ in tols:
                    np.testing.assert_allclose(got["out"][i, b, :T], ref[nm_], rtol=tols[nm_][0], atol=tols[nm_][1],
                                               err_msg=f"path {b} {nm_}")
        # 4. bit for bit what the staged Python orchestration (Engine.profile) returns
        eng = Engine("cuda:0")
        res = eng.profile(eng.upload(packed))
        torch.cuda.synchronize()
        assert np.array_equal(res.n_out.cpu().numpy(), got["n_out"])
        for b in range(B):
            T = int(got["n_out"][b])
            assert np.array_equal(res.out[:, b, :T].cpu().numpy(), got["out"][:, b, :T])
            assert np.array_equal(res.vel[b, :int(got["n_samples"][b])].cpu().numpy(), got["vel"][b, :int(got["n_samples"][b])])
        np.testing.assert_array_equal(res.summary.cpu().numpy(), got["summary"])
        # 5. the Engine's thin wrapper over the same symbol
        rb = eng.profile_batch(eng.upload(packed))
        torch.cuda.synchronize()
        assert np.array_equal(rb.n_out.cpu().numpy(), got["n_out"]) and bool((rb.status == 0).all())
        for b in range(0, B, 7):
            T = int(got["n_out"][b])
            assert np.array_equal(rb.out[:, b, :T].cpu().numpy(), got["out"][:, b, :T])
    finally:
        for p in bufs:
            rt.cudaFree(p)


@pytest.mark.gpu
def test_cfg3_full_tile_against_oracle(ora):
    """BASELINE configs[2] at full tile size: ONE 16 384-path tile of the 2**20-path job (seed 1, 16 nodes) in one call;
    a strided sample of its paths against oracle.full_batch (integers exact, summaries within the north-star tolerances),
    plus size-independent properties over all of it (status, monotone times, bounded velocities, determinism)."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    B = 16384
    packed = synth.random_paths(B, 16, seed=1)
    eng = Engine("cuda:0")
    db = eng.upload(packed)
    res = eng.profile(db)
    torch.cuda.synchronize()
    assert bool((res.status == 0).all().item())
    summ = res.summary.cpu().numpy()
    sel = np.arange(0, B, 257)
    ref = ora.full_batch(packed.node_attr[sel], packed.node_flags[sel], packed.cons[sel])
    assert (ref[:, 4] == 0).all()
    assert np.array_equal(summ[sel, 0], ref[:, 0])                          # T: bit-exact sample indexing
    np.testing.assert_allclose(summ[sel, 1], ref[:, 1], rtol=1e-12)         # total length
    np.testing.assert_allclose(summ[sel, 2], ref[:, 2], rtol=1e-6)          # t_end
    np.testing.assert_allclose(summ[sel, 3], ref[:, 3], rtol=1e-6)          # max |v|
    for b in (0, 4097, B - 1):                                              # three whole trajectories
        r1 = ora.full(packed.node_attr[b], packed.node_flags[b], None, None, packed.cons[b])
        got = res.path(b)
        assert len(got["times"]) == r1["T"] and int(res.n_samples[b]) == r1["D"]
        assert got["nodes_map"].tolist() == r1["nodes_map"].tolist()
        np.testing.assert_allclose(got["x"], r1["x"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["y"], r1["y"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(got["linear_vels"], r1["linear_vels"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(got["times"], r1["times"], rtol=1e-6, atol=1e-12)
    # properties over the whole tile
    T = res.n_out.long()
    idx = torch.arange(res.T_cap, device=T.device)[None, :]
    valid = idx < T[:, None]
    times = res.stream("times")
    dtm = times[:, 1:] - times[:, :-1]
    assert bool((dtm[valid[:, 1:]] > 0).all().item())
    v = res.stream("linear_vels")
    assert bool((v[valid].abs() <= 4.0 * (1 + 1e-12)).all().item())
    assert torch.equal(res.summary[:, 0].long(), T)
    # determinism: the same tile through the single C entry point gives the same bits
    rb = eng.profile_batch(db)
    torch.cuda.synchronize()
    assert torch.equal(rb.n_out, res.n_out)
    m = min(rb.T_cap, res.T_cap)
    vb = torch.arange(m, device=T.device)[None, :] < T[:, None]
    for i in range(8):
        assert torch.equal(rb.out[i, :, :m][vb], res.out[i, :, :m][vb])


@pytest.mark.gpu
def test_repeated_runs_are_bitwise_identical():
    """Race detector of last resort (compute-sanitizer's racecheck is closed on the GPU pool): the TMA rings, the mbarrier
    hand-overs and the shared-memory state exchange of the speculative chunks are timing dependent if they are wrong, the
    results are not.  Twelve runs of a mixed batch (fast path, eager and through the one-call entry) must agree bit for bit."""
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    packed = synth.mixed_paths(768, 8, seed=5)
    eng = Engine("cuda:0")
    db = eng.upload(packed)
    ref = eng.profile(db)
    torch.cuda.synchronize()
    T = ref.n_out.long()
    valid = torch.arange(ref.T_cap, device=T.device)[None, :] < T[:, None]
    D = ref.n_samples.long()
    dvalid = torch.arange(ref.vel.shape[1], device=T.device)[None, :] < D[:, None]
    for k in range(12):
        got = eng.profile(db, reuse_plan=True) if k % 2 == 0 else eng.profile_batch(db)
        torch.cuda.synchronize()
        assert torch.equal(got.n_out, ref.n_out) and torch.equal(got.status, ref.status)
        m = min(got.T_cap, ref.T_cap)
        for i in range(8):
            assert torch.equal(got.out[i, :, :m][valid[:, :m]], ref.out[i, :, :m][valid[:, :m]]), (k, i)
        dm = min(got.vel.shape[1], ref.vel.shape[1])
        assert torch.equal(got.vel[:, :dm][dvalid[:, :dm]], ref.vel[:, :dm][dvalid[:, :dm]]), k

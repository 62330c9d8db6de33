"""The tiled, graphed, pipelined and host-streamed steps are vap_profile_batch calls: they flag absurd paths as eager
Engine.profile does, return its bits on every healthy path, and redo a capacity overflow once with the sizes the device
reported."""
from dataclasses import replace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

B, N, TILES = 7, 6, 3              # B is not a multiple of the tile count
BAD = (1, 2, 3)                    # NaN coordinate, 2.5e6 ft (> 5e7 distance samples), infinite coordinate
GOOD = [b for b in range(B) if b not in BAD]


def bad_batch():
    from vexautonomousplanner_b200 import synth
    p = synth.random_paths(B, N, seed=92)
    p.node_attr[1, 2, 0] = np.nan
    p.node_attr[2, 3, 0:2] = [2.5e6, -2.5e6]
    p.node_attr[3, 1, 1] = np.inf
    return p


def scaled(p, s):
    from vexautonomousplanner_b200.packing import PackedPaths
    q = PackedPaths(*(a.copy() for a in (p.node_attr, p.node_flags, p.n_nodes, p.ap_attr, p.ap_flags, p.n_ap, p.cons)))
    q.node_attr[:, :, 0:2] *= s
    return q


def same_bits(ref, got, rows):
    """Status and counts of every path; every output of the paths in `rows` bit for bit."""
    for name in ("status", "n_out", "n_samples"):
        assert getattr(ref, name).tolist() == getattr(got, name).tolist(), name
    for b in rows:
        T, D = int(ref.n_out[b]), int(ref.n_samples[b])
        assert T > 0 and D > 0, b
        assert torch.equal(ref.out[:, b, :T].view(torch.int64), got.out[:, b, :T].view(torch.int64)), b
        assert torch.equal(ref.vel[b, :D].view(torch.int64), got.vel[b, :D].view(torch.int64)), b
        assert torch.equal(ref.summary[b].view(torch.int64), got.summary[b].view(torch.int64)), b
        nm, am = (int(v) for v in ref.n_maps[b])
        assert ref.n_maps[b].tolist() == got.n_maps[b].tolist(), b
        assert ref.nodes_map[b, :nm].tolist() == got.nodes_map[b, :nm].tolist(), b
        assert ref.actions_map[b, :am].tolist() == got.actions_map[b, :am].tolist(), b


def test_every_step_flags_absurd_paths_as_eager_profile():
    from vexautonomousplanner_b200.engine import ST_CAPACITY, ST_DIVERGED, Engine, PipelinedProfiler
    eng = Engine("cuda:0")
    packed = bad_batch()
    db = eng.upload(packed)
    ref = eng.profile(db)
    torch.cuda.synchronize()
    assert int(ref.status[2]) == ST_DIVERGED and not bool((ref.status == ST_CAPACITY).any())
    assert all(int(ref.status[b]) == 0 for b in GOOD)
    tiled = eng.profile(db, reuse_plan=True, tiles=TILES)
    graph = eng.capture(db.clone(), tiles=TILES)
    replay = graph.run(check=False)
    pipe = PipelinedProfiler(eng, db, depth=2)
    piped = [pipe.submit(db), pipe.submit(None)]
    pipe.drain()
    torch.cuda.synchronize()
    for got in [tiled, replay] + piped:
        same_bits(ref, got, GOOD)
    host = eng.profile_to_host(packed, tiles=TILES)
    assert host.status.tolist() == ref.status.tolist() and host.n_out.tolist() == ref.n_out.tolist()
    assert np.array_equal(host.summary.numpy().view(np.int64), ref.summary.cpu().numpy().view(np.int64))
    for b in GOOD:
        want, got = ref.path(b), host.path(b)
        for name in ("times", "x", "y", "linear_vels", "headings", "nodes_map"):
            assert np.array_equal(want[name], got[name]), (b, name)


def test_tiled_run_that_outgrows_its_plan_is_redone_once():
    """A batch of the planned shape with longer paths (more distance samples and time rows) overflows the tiled call;
    the redo is exact, becomes the plan, and an identical second call runs the tiles only.  A graph fed the same batch
    redoes it without writing to its static inputs."""
    from vexautonomousplanner_b200.engine import PROFILE_BATCH_KERNELS, Engine
    from vexautonomousplanner_b200 import synth
    small, big = scaled(synth.random_paths(B, N, seed=93), 0.4), synth.random_paths(B, N, seed=93)
    ref_eng = Engine("cuda:0")
    want = ref_eng.profile(ref_eng.upload(big))
    eng = Engine("cuda:0")
    sdb, bdb = eng.upload(small), eng.upload(big)
    assert sdb.max_splines == bdb.max_splines
    planned = eng.profile(sdb)
    torch.cuda.synchronize()
    assert int(want.n_out.max()) > planned.T_cap and int(want.n_samples.max()) > planned.vel.shape[1]
    l0 = eng.launches
    first = eng.profile(bdb, reuse_plan=True, tiles=TILES)
    torch.cuda.synchronize()
    assert eng.launches - l0 > TILES * PROFILE_BATCH_KERNELS            # the tiles, then the redo
    same_bits(want, first, range(B))
    l0 = eng.launches
    again = eng.profile(bdb, reuse_plan=True, tiles=TILES)
    torch.cuda.synchronize()
    assert eng.launches - l0 == TILES * PROFILE_BATCH_KERNELS
    same_bits(want, again, range(B))

    fresh = Engine("cuda:0")                 # sized from the small batch only
    g = fresh.capture(fresh.upload(small), tiles=TILES)
    s = g.db.max_splines
    assert int(want.n_samples.max()) > g.D_cap
    redo = g.run(bdb)
    torch.cuda.synchronize()
    same_bits(want, redo, range(B))
    assert g.db.max_splines == s
    for mine, src in zip(g.db.tensors(), bdb.tensors()):
        assert torch.equal(mine, src)


def test_tiled_batch_with_one_node_column_raises():
    """N_max = 1: the staged path (vap_build_path) and the tiled one (vap_profile_batch) both reject the batch with
    VapError; neither returns rows."""
    from vexautonomousplanner_b200 import _lib, synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    db = eng.upload(synth.random_paths(B, 2, seed=94))
    one = replace(db, node_attr=db.node_attr[:, :1].contiguous(), node_flags=db.node_flags[:, :1].contiguous(),
                  n_nodes=db.n_nodes.clamp(max=1), max_splines=1)
    with pytest.raises(_lib.VapError, match="N_max"):
        eng.profile(one)
    eng._plan[(one.B, one.N_max, one.A_max, one.max_splines)] = (128, 64)      # a plan, so that tiles > 1 takes the tiled path
    with pytest.raises(_lib.VapError, match="bad sizes"):
        eng.profile(one, reuse_plan=True, tiles=TILES)

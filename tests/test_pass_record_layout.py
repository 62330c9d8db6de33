"""The velocity passes stream four record planes per sample ({|kappa|, G, stat, gh}, 32 bytes) and make the reciprocal of
the wheel-acceleration denominator gh themselves with recip_for_pass.  Every branch of that function that geometry can
reach must give the serial recurrences' bits, and the workspace must be exactly one plane of B x RS doubles smaller than
with the 40-byte records that carried the reciprocal as a fifth plane."""
import ctypes as C

import numpy as np
import pytest

CONS = [4.0, 8.0, 8.0, 0.8, 16.0, 12.5 / 12]

# (B, N_max, A_max, max_splines, lut_samples, samples_per_node, D_cap, T_cap, chunks) and vap_workspace_bytes of the
# 40-byte-record layout for it
WORKSPACE_40B = [((4096, 8, 0, 7, 1000, 1000, 18432, 4096, 32), 6481330432),
                 ((320, 8, 3, 7, 1000, 1000, 12800, 4096, 8), 402055936),
                 ((3, 120, 0, 119, 1000, 1000, 1048576, 8192, 256), 191079936)]


def test_workspace_is_one_plane_smaller():
    from vexautonomousplanner_b200 import _lib
    L = _lib.lib()
    for (B, N, A, S, ls, spn, D_cap, T_cap, chunks), old in WORKSPACE_40B:
        RS = int(L.vap_pass_row_slots(C.c_int64(D_cap), C.c_int(chunks)))
        new = int(L.vap_workspace_bytes(C.c_int64(B), C.c_int(N), C.c_int(A), C.c_int(S), C.c_int(ls), C.c_int(spn),
                                        C.c_int64(D_cap), C.c_int64(T_cap), C.c_int(chunks)))
        assert new == old - 8 * B * RS, (B, N, chunks, new, old)


def straight_paths():
    """Collinear nodes: axis-parallel lines (heading and curvature exactly 0), a diagonal line, and a path whose middle
    segment is straight between two curved ones."""
    import vexautonomousplanner_b200 as vap
    paths = [np.array([[1.0, 2.0], [3.0, 2.0], [6.0, 2.0], [9.0, 2.0]]),
             np.array([[2.0, 1.0], [2.0, 4.0], [2.0, 8.0]]),
             np.array([[1.0, 1.0], [2.5, 2.5], [4.0, 4.0], [7.0, 7.0]]),
             np.array([[1.0, 1.0], [4.0, 1.0], [7.0, 1.0], [9.0, 4.0], [9.5, 8.0]]),
             np.array([[0.5, 3.0], [2.0, 5.0], [4.0, 5.0], [6.0, 5.0], [8.0, 2.0]])]
    N = max(len(p) for p in paths)
    pts = np.zeros((len(paths), N, 2))
    nn = np.zeros(len(paths), dtype=np.int32)
    for b, p in enumerate(paths):
        pts[b, :len(p)] = p
        pts[b, len(p):] = p[-1] + np.arange(1, N - len(p) + 1)[:, None] * 0.5
        nn[b] = len(p)
    return vap.pack_arrays(pts, CONS, n_nodes=nn)


def denominator_kinds(ref):
    """Counts of the cases of recip_for_pass the passes meet on this batch, from the serial run's heading / curvature per
    distance sample: gh = 2|theta[e+1] - theta[e]| with |kappa| >= 1e-6 at the sample that multiplies it (the wheel term
    of a straight sample never uses the reciprocal)."""
    import torch
    th = ref.extra["th"].double()
    kap = ref.extra["kap"].double()
    D = ref.n_samples.long()
    e = torch.arange(th.shape[1] - 1, device=D.device)[None, :]
    m = e < (D[:, None] - 1)
    gh = 2 * (th[:, 1:] - th[:, :-1]).abs()
    # forward step e multiplies by |kappa_e|, backward step e+1 by |kappa_{e+1}|: a denominator is used when either is curved
    curved = (kap[:, :-1].abs() >= 1e-6) | (kap[:, 1:].abs() >= 1e-6)
    bits = gh.view(torch.int64)
    all_ones = (bits & 0x000FFFFFFFFFFFFF) == 0x000FFFFFFFFFFFFF
    safe = (gh >= 2.2250738585072014e-308) & (gh < 1e300) & ~all_ones
    return dict(zero=int((m & curved & (gh == 0)).sum()), safe=int((m & curved & safe).sum()),
                other=int((m & curved & ~safe & (gh != 0)).sum()),
                straight=int((m & ~curved).sum()), exactly_straight=int((m & (kap[:, :-1] == 0)).sum()))


@pytest.mark.gpu
def test_pass_reciprocal_branches_equal_serial_bitwise():
    """gh == 0 (two samples snapped to the same heading entry: the reciprocal is +inf), gh a normal number (RN(1/gh)),
    straight samples (the reciprocal is not used) and max_acceleration overrides (the backward limit from statB), at 8
    and 256 chunks: velocities, sampling outputs and time-domain outputs bit for bit equal to the serial kernels.
    The third branch of recip_for_pass (-1: gh subnormal, NaN or with an all-ones significand, sent to the generic
    division) cannot be produced through real geometry: gh is twice the difference of two heading-table entries, which
    is subnormal only for headings below 2^-969 rad, and an all-ones significand is one value in 2^52 of a binade.  That
    branch is checked directly against '/' by tests/test_gpu_parity.py::test_recip_division_is_ieee."""
    import torch
    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine
    ser = Engine("cuda:0", velocity_impl="serial", time_impl="serial")
    overrides = synth.mixed_paths(128, 8, seed=9)
    seen = dict(zero=0, safe=0, other=0, straight=0, exactly_straight=0)
    for packed in (straight_paths(), overrides, synth.random_paths(128, 8, seed=11)):
        db = ser.upload(packed)
        ref = ser.profile(db, keep=True)
        torch.cuda.synchronize()
        assert bool((ref.status == 0).all())
        for k, v in denominator_kinds(ref).items():
            seen[k] += v
        D = ref.n_samples.long()
        m = torch.arange(ref.vel.shape[1], device=D.device)[None, :] < D[:, None]
        if packed is overrides:
            ne = ref.extra["n_ev"].long()
            em = torch.arange(ref.extra["max_accels"].shape[1], device=D.device)[None, :]
            assert bool(((em < ne[:, 0:1]) & (ref.extra["max_accels"] != db.cons[:, 1:2])).any()), "no overrides"
        for chunks in (8, 256):
            got = Engine("cuda:0", velocity_impl="chunked", chunks=chunks, time_impl="split").profile(db, keep=True)
            torch.cuda.synchronize()
            assert torch.equal(ref.n_samples, got.n_samples)
            for key in ("t", "kap", "th"):
                assert torch.equal(ref.extra[key][m].view(torch.int64), got.extra[key][m].view(torch.int64)), (key, chunks)
            assert torch.equal(ref.vel[m].view(torch.int64), got.vel[m].view(torch.int64)), f"chunks={chunks}"
            assert torch.equal(ref.n_out, got.n_out)
            n = ref.n_out.long()
            Tm = min(ref.T_cap, got.T_cap)
            mt = torch.arange(Tm, device=n.device)[None, :] < n[:, None]
            for i in range(8):
                assert torch.equal(ref.out[i][:, :Tm][mt].view(torch.int64), got.out[i][:, :Tm][mt].view(torch.int64)), (chunks, i)
            assert torch.equal(ref.summary.view(torch.int64), got.summary.view(torch.int64))
    assert seen["zero"] > 0 and seen["safe"] > 0, seen
    assert seen["straight"] > 0 and seen["exactly_straight"] > 0, seen

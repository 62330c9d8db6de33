"""Drop-in tests: the mirrors of the reference classes (same names / signatures / error behaviour) against the
reference's golden outputs.  These read like the reference's own usage: build a manager from duck-typed nodes,
call generate_motion_profile, compare with what the reference returned for the same inputs."""
import numpy as np
import pytest

from golden_util import GOLDEN_DIR, bit_equal, case_names, load_case, ulp_diff

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


class Node:            # attribute names of gui/node.py:17-51
    def __init__(self, **kw):
        self.is_reverse_node = False; self.turn = 0; self.wait_time = 0; self.stop = False; self.tangent = None
        self.incoming_magnitude = None; self.outgoing_magnitude = None; self.max_velocity = 0; self.max_acceleration = 0
        self.__dict__.update(kw)


class ActionPoint:     # gui/action_point.py:16-41
    def __init__(self, t, **kw):
        self.t = t; self.stop = False; self.wait_time = 0; self.max_velocity = 0; self.max_acceleration = 0
        self.__dict__.update(kw)


def objects_from_case(g):
    nodes = []
    for i in range(g["n"]):
        kw = dict(is_reverse_node=bool(g["n_reverse"][i]), turn=float(g["n_turn"][i]) if g["n_turn"][i] != int(g["n_turn"][i]) else int(g["n_turn"][i]),
                  wait_time=float(g["n_wait"][i]), stop=bool(g["n_stop"][i]), max_velocity=float(g["n_maxvel"][i]),
                  max_acceleration=float(g["n_maxacc"][i]))
        if g["n_has_tangent"][i]:
            kw.update(tangent=np.array(g["n_tangent"][i]), incoming_magnitude=float(g["n_inmag"][i]),
                      outgoing_magnitude=float(g["n_outmag"][i]))
        nodes.append(Node(**kw))
    aps = [ActionPoint(float(t), stop=bool(s), wait_time=float(w), max_velocity=float(v), max_acceleration=float(a))
           for t, s, w, v, a in zip(g["ap_t"], g["ap_stop"], g["ap_wait"], g["ap_maxvel"], g["ap_maxacc"])]
    return nodes, aps


CASES = ["cfg1_factory", "cfg1_reporoot", "actions", "tangents", "multi_split", "two_nodes", "mixed8_0", "node0_wait_rev"]


@pytest.mark.parametrize("name", CASES)
def test_manager_and_profile_match_reference(name):
    from vexautonomousplanner_b200.motion_profiling_v2 import motion_profile_generator as mpg
    from vexautonomousplanner_b200.splines.spline_manager import QuinticHermiteSplineManager
    g = load_case(name)
    nodes, aps = objects_from_case(g)
    sm = QuinticHermiteSplineManager()
    assert sm.build_path(g["points_ft"], nodes, aps) is True
    # ---- geometry attributes
    assert len(sm.splines) == len(g["spline_param_end"])
    seg = np.concatenate([np.stack(sp.segments) for sp in sm.splines])
    assert ulp_diff(seg, g["seg"]).max() <= 1
    params = np.concatenate([sp.parameters for sp in sm.splines])
    assert bit_equal(params, g["spline_params_concat"])
    assert bit_equal(np.array([float(v) for sp in sm.splines for v in sp.segment_lengths]), g["spline_seglen"])
    # ---- point queries
    for key, fn in (("api_point", sm.get_point_at_parameter), ("api_d1", sm.get_derivative_at_parameter),
                    ("api_d2", sm.get_second_derivative_at_parameter)):
        got = np.array([fn(t) for t in g["api_t"][:12]])
        np.testing.assert_allclose(got, g[key][:12], rtol=1e-13, atol=1e-13)
    got = sm.get_point_at_parameter(0.5)
    assert isinstance(got, np.ndarray) and got.shape == (2,)
    np.testing.assert_allclose([sm._get_heading(t) for t in g["api_t"][:6]], g["api_heading_exact"][:6], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose([sm._get_curvature(t) for t in g["api_t"][:6]], g["api_curv_exact"][:6], rtol=1e-12, atol=1e-14)
    # ---- tables
    sm.rebuild_tables()
    np.testing.assert_allclose(sm.lookup_table.distances, g["lut_d"], rtol=1e-13)
    np.testing.assert_allclose(sm.lookup_table.parameters, g["lut_t"], rtol=1e-15)
    assert abs(sm.get_total_arc_length() - float(g["total_length"])) <= 1e-12
    assert ulp_diff(sm._precomputed_properties["curvatures"], g["prop_k"]).max() <= 8
    assert ulp_diff(sm._precomputed_properties["headings"], g["prop_h"]).max() <= 8
    assert bit_equal(sm._precomputed_properties["parameters"], np.linspace(0, g["n"] - 1, 1000 * g["n"]))
    np.testing.assert_allclose([sm.get_heading(t) for t in g["api_t"][:8]], g["api_heading_snap"][:8], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose([sm.get_curvature(t) for t in g["api_t"][:8]], g["api_curv_snap"][:8], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose([float(sm.distance_to_time(d)) for d in g["api_dist"][:8]], g["api_dist_t"][:8], rtol=1e-12, atol=1e-13)
    assert sm.distance_to_time(-1.0) == 0 and sm.distance_to_time(1e9) == g["n"] - 1
    # ---- velocity passes and the full profile
    c = mpg.Constraints(*g["constraints"])
    vel = mpg.forward_backward_pass(sm, c, 0.005)
    assert isinstance(vel, list) and len(vel) == len(g["vel"])
    np.testing.assert_allclose(vel, g["vel"], rtol=1e-6, atol=1e-12)
    assert (c.max_acc, c.max_dec) == (g["constraints"][1], g["constraints"][2])
    times, positions, lin, acc, head, ang, nodes_map, actions_map, coords = mpg.generate_motion_profile(sm, c)
    assert len(times) == len(g["times"])
    assert nodes_map + [len(times)] == g["nodes_map"].tolist()          # the caller appends len(times), path.py:342
    assert actions_map == g["actions_map"].tolist()
    np.testing.assert_allclose(times, g["times"], rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(positions, g["positions"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(lin, g["linear_vels"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(acc, g["accelerations"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(head, g["headings"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(ang, g["angular_vels"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(np.array(coords), g["coords"], rtol=1e-9, atol=1e-10)
    assert isinstance(coords[0], np.ndarray) and coords[0].shape == (2,)


def test_standalone_spline_api():
    """QuinticHermiteSpline used directly: fit conventions, evaluation, Gauss-Legendre arc length and its inverse."""
    from vexautonomousplanner_b200.splines.quintic_hermite_spline import QuinticHermiteSpline
    g = load_case("cfg1_factory")
    x, y = g["points_ft"][:, 0], g["points_ft"][:, 1]
    sp = QuinticHermiteSpline()
    with pytest.raises(ValueError):
        sp.get_point(0.5)
    assert sp.fit(x, y) is False                      # no set_all_tangents -> the reference's fit() fails (F7)
    assert sp.fit(x, y[:-1]) is False and sp.fit(x[:1], y[:1]) is False
    sp = QuinticHermiteSpline()
    sp.set_all_tangents([[None, None]] * len(x))
    assert sp.fit(x, y) is True
    assert ulp_diff(np.stack(sp.segments), g["seg"]).max() <= 1
    assert bit_equal(sp.parameters, g["spline_params_concat"])
    t = g["api_t"][:10]
    np.testing.assert_allclose([sp.get_point(v) for v in t], g["api_point"][:10], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose([sp.get_heading(v) for v in t], g["api_heading_exact"][:10], rtol=1e-13, atol=1e-14)
    np.testing.assert_allclose([sp.get_curvature(v) for v in t], g["api_curv_exact"][:10], rtol=1e-12, atol=1e-14)
    got = [sp.get_arc_length(a, b) for a, b in zip(g["gl_t0"], g["gl_t1"])]
    np.testing.assert_allclose(got, g["gl_len"], rtol=1e-13)
    assert abs(sp.get_total_arc_length() - g["gl_total"][0]) <= 1e-12
    inv = [sp.get_parameter_by_arc_length(s) for s in g["inv_s"]]
    np.testing.assert_allclose(inv, g["inv_t"], rtol=1e-12, atol=1e-13)
    with pytest.raises(ValueError):
        sp.get_arc_length(2.0, 1.0)
    with pytest.raises(ValueError):
        sp.get_arc_length(-0.1, 1.0)
    with pytest.raises(ValueError):
        sp.get_parameter_by_arc_length(-1.0)
    with pytest.raises(ValueError):
        sp.get_parameter_by_arc_length(1e9)
    assert sp.get_end_parameter() == sp.parameters[-1]
    assert sp.set_starting_tangent([1.0, 0.0]) is False
    assert sp.set_ending_tangent(np.array([1.0, 2.0])) is True
    assert sp.segments[-1][3].tolist() == [1.0, 2.0]
    d = sp.get_derivative(len(x) - 1)
    np.testing.assert_allclose(d, [1.0, 2.0], rtol=1e-12)


def test_error_conventions():
    from vexautonomousplanner_b200.motion_profiling_v2 import motion_profile_generator as mpg
    from vexautonomousplanner_b200.splines.spline_manager import QuinticHermiteSplineManager
    g = load_case("cfg1_factory")
    sm = QuinticHermiteSplineManager()
    with pytest.raises(ValueError):
        sm.get_point_at_parameter(0.0)
    with pytest.raises(ValueError):
        sm.build_lookup_table()
    nodes, _ = objects_from_case(g)
    assert sm.build_path(g["points_ft"][:3], nodes, []) is False
    assert sm.build_path(g["points_ft"][:1], nodes[:1], []) is False
    nodes[-1].is_reverse_node = True
    with pytest.raises(IndexError):
        sm.build_path(g["points_ft"], nodes, [])
    nodes, _ = objects_from_case(g)
    nodes[0].turn = 30
    assert sm.build_path(g["points_ft"], nodes, []) is True
    with pytest.raises(IndexError):
        mpg.generate_motion_profile(sm, mpg.Constraints(*g["constraints"]))


def test_forward_backward_pass_refuses_an_absurd_length():
    """A 2.5e6 ft path needs more distance samples than the engine accepts (the reference's sampling loop would not fit in
    memory): forward_backward_pass raises with status -5 instead of sizing its buffers on it."""
    from vexautonomousplanner_b200.motion_profiling_v2 import motion_profile_generator as mpg
    from vexautonomousplanner_b200.splines.spline_manager import QuinticHermiteSplineManager
    sm = QuinticHermiteSplineManager()
    assert sm.build_path(np.array([[0.0, 0.0], [2.5e6, -2.5e6]]), [Node(), Node()], []) is True
    with pytest.raises(RuntimeError, match="status -5"):
        mpg.forward_backward_pass(sm, mpg.Constraints(4.0, 8.0, 8.0, 0.8, 16.0, 12.5 / 12), 0.005)


def test_misc_api_matches_reference():
    from vexautonomousplanner_b200.motion_profiling_v2 import motion_profile_generator as mpg
    from vexautonomousplanner_b200.motion_profiling_v2.one_dim_mp_generator import generate_trapezoidal_profile
    m = dict(np.load(f"{GOLDEN_DIR}/misc_api.npz"))
    off = 0
    for V, A, w, deg, rad, K in m["angle_meta"]:
        K = int(K)
        h, om = mpg.motion_profile_angle(rad, mpg.Constraints(V, A, A, 0.8, 16.0, w), 0.01)
        assert len(h) == K and len(om) == K
        np.testing.assert_allclose(h, m["angle_headings"][off:off + K], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(om, m["angle_omegas"][off:off + K], rtol=1e-9, atol=1e-12)
        off += K
    off = 0
    for V, A, dist, K in m["trap_meta"]:
        K = int(K)
        v = generate_trapezoidal_profile(V, A, dist)
        assert isinstance(v, np.ndarray) and len(v) == K
        np.testing.assert_allclose(v, m["trap_v"][off:off + K], rtol=1e-12, atol=1e-15)
        off += K
    xs = tuple(i * 0.005 for i in range(400))
    got = [mpg.lerp(x, xs, tuple(m["lerp_ys"])) for x in m["lerp_q"][:40]]
    assert bit_equal(np.array(got), m["lerp_out"][:40])
    l, r = mpg.get_wheel_trajectory(list(m["wheel_lin"]), list(m["wheel_ang"]), 12.5 / 12)
    assert bit_equal(np.array(l), m["wheel_l"]) and bit_equal(np.array(r), m["wheel_r"])
    c = mpg.Constraints(4.0, 8.0, 8.0, 0.8, 16.0, 12.5 / 12)
    assert c.max_speed_at_curvature(0.0) == 4.0 and c.max_accels_at_turn(1.0) == 8.0 - 12.5 / 12 / 2

"""Mirror of src/motion_profiling_v2/motion_profile_generator.py on the CUDA engine.

  forward_backward_pass     -> S0..S5 through Engine (motion_profile_generator.py:70-316)
  generate_motion_profile   -> Engine.profile        (:389-628)
  motion_profile_angle      -> vap_turn_profile      (:319-346)
  lerp                      -> vap_lerp              (:349-386)
  get_wheel_trajectory      -> vap_wheel_trajectory  (:631-646)
`spline_manager` may be this package's QuinticHermiteSplineManager or the reference's own manager object: only the
control points of its splines, `.nodes` and `.action_points` are read.
"""
from __future__ import annotations

import logging
import math
from dataclasses import dataclass
from typing import List, Tuple

import numpy as np
import torch

from ..packing import pack_paths
from ..runtime import C, Keep, _p, check, dev, get_engine, stream
from . import one_dim_mp_generator

logger = logging.getLogger(__name__)


@dataclass
class Constraints:
    """motion_profile_generator.py:14-67.  The scalar helper methods are plain host arithmetic (they are not on the
    batched path; the kernels carry their own copies of these formulas)."""
    max_vel: float
    max_acc: float
    max_dec: float
    friction_coef: float
    max_jerk: float
    track_width: float

    def max_speed_at_curvature(self, curvature: float) -> float:
        if abs(curvature) < 1e-6:
            return self.max_vel
        max_turn_speed = ((2 * self.max_vel / self.track_width) * self.max_vel) / (
            abs(curvature) * self.max_vel + (2 * self.max_vel / self.track_width))
        return min(max_turn_speed, self.max_vel)

    def set_max_vel(self, max_vel):
        self.max_vel = max_vel

    def set_max_acc(self, max_acc):
        self.max_acc = max_acc

    def limit_velocity_by_ang_accel(self, dkappads: float, max_angular_accel: float) -> float:
        if abs(dkappads) < 1e-9:
            return self.max_vel
        max_v_sq = max_angular_accel / abs(dkappads)
        if max_v_sq < 0:
            return 0.0
        return min(math.sqrt(max_v_sq), self.max_vel)

    def max_accels_at_turn(self, angular_accel: float):
        left_lin_ac = self.max_acc + angular_accel * self.track_width / 2
        right_lin_ac = self.max_acc - angular_accel * self.track_width / 2
        return left_lin_ac if abs(left_lin_ac) < abs(right_lin_ac) else right_lin_ac

    def get_wheel_speeds(self, linear_vel: float, angular_vel: float) -> Tuple[float, float]:
        return (linear_vel - (angular_vel * self.track_width / 2), linear_vel + (angular_vel * self.track_width / 2))


def _points_of(spline_manager) -> np.ndarray:
    pts = getattr(spline_manager, "_points", None)
    if pts is not None:
        return np.asarray(pts, dtype=np.float64)
    rows = []
    for k, sp in enumerate(spline_manager.splines):      # the reference's manager: stitch the control points back
        cp = np.asarray(sp.control_points, dtype=np.float64)
        rows.append(cp if k == 0 else cp[1:])
    return np.concatenate(rows, axis=0)


def _pack(spline_manager, constraints):
    pts = _points_of(spline_manager)
    return pack_paths([(pts, spline_manager.nodes, spline_manager.action_points)], constraints)


def _raise_for(status: int):
    if status == -2:
        raise IndexError("list index out of range")
    if status == -1:
        raise ValueError("No splines have been initialized")
    if status != 0:
        raise RuntimeError(f"engine status {status}")


def forward_backward_pass(spline_manager, constraints: Constraints, delta_dist: float, start_vel: float = 0.01,
                          end_vel: float = 0.01) -> List[float]:
    """Forward-backward velocity smoothing over distance samples (motion_profile_generator.py:70-316)."""
    from ..engine import Engine
    base = get_engine()
    eng = base if (delta_dist == base.dd and start_vel == base.start_vel and end_vel == base.end_vel) else \
        Engine(base.device, dt=base.dt, dd=delta_dist, start_vel=start_vel, end_vel=end_vel)
    db = eng.upload(_pack(spline_manager, constraints))
    g = eng.build_geometry(db)
    t = eng.build_lut(db, g)
    eng.build_props(db, g, t)
    _raise_for(int(g.status.item()))
    status = g.status.clone()
    D_cap = eng._plan_distance(t, status)                   # an absurd length is status -5, not a buffer of its size
    n_samples, vel, _, _, _ = eng.velocity_chunked(db, g, t, status, D_cap)
    _raise_for(int(status.item()))
    return [np.float64(v) for v in vel[0, : int(n_samples.item())].cpu().numpy()]


def motion_profile_angle(angle, constraints: Constraints, dt: float = 0.01):
    """Turn-in-place profile: (headings, angular_velocities) (motion_profile_generator.py:319-346)."""
    h, w = one_dim_mp_generator._turn_profile(angle, constraints.max_vel, constraints.max_acc, constraints.track_width,
                                              dt, mode=0)
    return [np.float64(x) for x in h], [0] + [np.float64(x) for x in w[1:]]


def lerp(x, x_array, y_array, cache=None):
    """Linear interpolation on a sorted table (motion_profile_generator.py:349-386)."""
    eng = get_engine()
    xs = dev(np.asarray(x_array, dtype=np.float64)); ys = dev(np.asarray(y_array, dtype=np.float64))
    out = eng._empty((1,))
    k = Keep()
    check(eng.lib.vap_lerp(C.c_int64(1), k([float(x)]), C.c_int64(xs.numel()), _p(xs), _p(ys), _p(out), stream()),
          "vap_lerp")
    if cache is not None:
        idx = int(np.searchsorted(np.asarray(x_array), x, side="right") - 1)
        if 0 <= idx < len(x_array) - 1:
            cache["last_idx"] = idx
    return np.float64(out.item())


def generate_motion_profile(spline_manager, constraints: Constraints, dt: float = 0.01, dd: float = 0.005):
    """Complete motion profile (motion_profile_generator.py:389-628).  Returns the reference's 9-tuple
    (times, positions, linear_vels, accelerations, headings, angular_vels, nodes_map, actions_map, coords)."""
    from ..engine import Engine
    base = get_engine()
    eng = base if (dt == base.dt and dd == base.dd) else Engine(base.device, dt=dt, dd=dd)
    logger.info("Generating motion profile")
    if hasattr(spline_manager, "rebuild_tables") and hasattr(spline_manager, "_db"):
        spline_manager.rebuild_tables()                      # same side effect as the reference (:402)
    from ..export import RK_INSERTED, RK_OMEGA_INT, RK_POS_INT, RK_TIME_INT, row_kinds
    db = eng.upload(_pack(spline_manager, constraints))
    res = eng.profile(db)
    _raise_for(int(res.status.item()))
    p = res.path(0)
    T = len(p["times"])
    # the entries the reference appends as Python ints: current_time starts as the int 0 (:425); inserted turn / wait rows
    # extend the lists with the int 0 (:448-453, 500-503, 511-515) and the first angular velocity of a turn is 0 (:343)
    kinds = row_kinds(eng, res, db)[0, :T].cpu().numpy()

    def col(name, bit):
        return [0 if (k & bit) else np.float64(v) for v, k in zip(p[name], kinds)]

    coords = [np.array([x, y]) for x, y in zip(p["x"], p["y"])]
    logger.info(f"Generated {T} points")
    return (col("times", RK_TIME_INT), col("positions", RK_POS_INT), col("linear_vels", RK_INSERTED),
            col("accelerations", RK_INSERTED), [np.float64(v) for v in p["headings"]], col("angular_vels", RK_OMEGA_INT),
            [int(v) for v in p["nodes_map"][:-1]], [int(v) for v in p["actions_map"]], coords)


def get_wheel_trajectory(linear_vels: List[float], angular_vels: List[float], track_width: float):
    """Left / right wheel velocities (motion_profile_generator.py:631-646)."""
    eng = get_engine()
    n = min(len(linear_vels), len(angular_vels))
    if n == 0:
        return [], []
    lin = dev(np.asarray(linear_vels[:n], dtype=np.float64)); ang = dev(np.asarray(angular_vels[:n], dtype=np.float64))
    left = eng._empty((n,)); right = eng._empty((n,))
    check(eng.lib.vap_wheel_trajectory(C.c_int64(n), _p(lin), _p(ang), C.c_double(track_width), _p(left), _p(right),
                                       stream()), "vap_wheel_trajectory")
    return [np.float64(v) for v in left.cpu().numpy()], [np.float64(v) for v in right.cpu().numpy()]

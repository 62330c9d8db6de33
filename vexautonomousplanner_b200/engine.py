"""Batched spline -> motion-profile engine: Python driver of libvap.so (include/vap.h).

PyTorch is plumbing only: device memory, streams, a few reductions for sizing.  All arithmetic of the
hot path happens in the hand-written sm_100a kernels of csrc/vap_kernels.cu; there is no CPU fallback.

Stages (SURVEY.md 2.2): S0 build_path -> S1 distance LUT -> S2 curvature/heading tables -> S3 distance
sampling -> S3 events + S4 forward + S5 backward -> S6 time-domain resampling (+ S7 summary rows).
"""
from __future__ import annotations

import ctypes as C
import os
from contextlib import contextmanager
from dataclasses import dataclass, field, replace
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .packing import PackedPaths

OUT_NAMES = ("times", "positions", "linear_vels", "accelerations", "headings", "angular_vels", "x", "y")
ST_OK, ST_FALSE, ST_INDEX, ST_VALUE, ST_CAPACITY, ST_DIVERGED, ST_EVENTS = 0, -1, -2, -3, -4, -5, -6
ROW_LIMIT = 1.0e7      # more time samples than this per path: treated as a non-terminating profile (status -5)
DIST_LIMIT = 5.0e7     # more distance samples than this per path (L / dd; an infinite length too): status -5
_POISON = bool(int(os.environ.get("VAP_POISON", "0")))
MAX_RETRIES = 2        # exact re-runs after a capacity overflow; a status that survives them is returned as it is
PROFILE_BATCH_KERNELS = 18   # kernels of one vap_profile_batch call (besides one memset and one 24-byte device copy)


def _p(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


@dataclass
class DeviceBatch:
    """PackedPaths resident on the device."""
    FIELDS = ("node_attr", "node_flags", "n_nodes", "ap_attr", "ap_flags", "n_ap", "cons")   # the input tensors, in order
    node_attr: torch.Tensor
    node_flags: torch.Tensor
    n_nodes: torch.Tensor
    ap_attr: torch.Tensor
    ap_flags: torch.Tensor
    n_ap: torch.Tensor
    cons: torch.Tensor
    max_splines: int

    @property
    def B(self):
        return self.node_attr.shape[0]

    @property
    def N_max(self):
        return self.node_attr.shape[1]

    @property
    def A_max(self):
        return self.ap_attr.shape[1]

    def tensors(self) -> list:
        return [getattr(self, name) for name in self.FIELDS]

    @staticmethod
    def from_packed(p: PackedPaths, device, non_blocking: bool = True) -> "DeviceBatch":
        return DeviceBatch(*(torch.from_numpy(getattr(p, name)).to(device, non_blocking=non_blocking)
                             for name in DeviceBatch.FIELDS), p.max_splines())

    def rows(self, lo: int, hi: int) -> "DeviceBatch":
        """Paths lo..hi as views of these tensors."""
        return DeviceBatch(*(t[lo:hi] for t in self.tensors()), self.max_splines)

    def clone(self) -> "DeviceBatch":
        return DeviceBatch(*(t.clone() for t in self.tensors()), self.max_splines)

    def copy_(self, other, non_blocking: bool = True) -> None:
        """Copy the inputs of `other` (a DeviceBatch of the same shape) into these tensors, on the current stream."""
        for dst, src in zip(self.tensors(), other.tensors()):
            dst.copy_(src, non_blocking=non_blocking)

    def pinned(self) -> "DeviceBatch":
        """Pinned host buffers of this batch's shape, for upload_()."""
        return DeviceBatch(*(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in self.tensors()), self.max_splines)

    def upload_(self, p: PackedPaths, pin: "DeviceBatch") -> None:
        """Copy the host batch `p` into these tensors through the pinned buffers `pin` (from pinned())."""
        for name, buf in zip(self.FIELDS, pin.tensors()):
            buf.copy_(torch.from_numpy(getattr(p, name)))
        self.copy_(pin)


@dataclass
class Geometry:
    seg: torch.Tensor          # [B, N_max-1, 6, 2]
    first_node: torch.Tensor   # [B, N_max+1] i32
    param_end: torch.Tensor    # [B, N_max]
    seglen: torch.Tensor       # [B, N_max]
    n_splines: torch.Tensor    # [B] i32
    status: torch.Tensor       # [B] i32
    params: Optional[torch.Tensor] = None   # [B, 2*N_max] concatenated spline.parameters (only when requested)
    derivs: Optional[torch.Tensor] = None   # [B, 2*N_max, 4] first / second derivatives of the control points


@dataclass
class Tables:
    samples: int
    spn: int
    Q_cap: int
    P_cap: int
    lut_d: torch.Tensor        # [B, Q_cap]
    lut_t: torch.Tensor
    total_len: torch.Tensor    # [B]
    prop_k: Optional[torch.Tensor] = None   # [B, P_cap]
    prop_h: Optional[torch.Tensor] = None
    lut_inv: Optional[torch.Tensor] = None  # [B, vap_lut_index_row_ints(Q_cap)] i32 inverse index of lut_d


@dataclass
class ProfileResult:
    """Device-resident result of one batch.  Row b of every [B, cap] array is valid up to its count."""
    B: int
    T_cap: int
    out: torch.Tensor            # [8, B, T_cap]: times, positions, linear_vels, accelerations, headings, angular_vels, x, y
    n_out: torch.Tensor          # [B] i32  number of time samples
    nodes_map: torch.Tensor      # [B, N_max+1] i32
    actions_map: torch.Tensor    # [B, A_max] i32
    n_maps: torch.Tensor         # [B, 2] i32 (len(nodes_map), len(actions_map))
    status: torch.Tensor         # [B] i32
    summary: torch.Tensor        # [B, 5]: n_out, total_length, t_end, max|v|, status
    vel: torch.Tensor            # [B, D_cap] velocities of forward_backward_pass
    n_samples: torch.Tensor      # [B] i32 (= D)
    geometry: Optional[Geometry] = None
    tables: Optional[Tables] = None
    extra: Dict[str, torch.Tensor] = field(default_factory=dict)

    def stream(self, name: str) -> torch.Tensor:
        return self.out[OUT_NAMES.index(name)]

    def path(self, b: int) -> Dict[str, np.ndarray]:
        """Copy path b to the host as numpy arrays trimmed to their true lengths."""
        T = int(self.n_out[b])
        res = {nm: self.out[i, b, :T].cpu().numpy() for i, nm in enumerate(OUT_NAMES)}
        nm_, am_ = (int(v) for v in self.n_maps[b])
        res["nodes_map"] = self.nodes_map[b, :nm_].cpu().numpy()
        res["actions_map"] = self.actions_map[b, :am_].cpu().numpy()
        res["vel"] = self.vel[b, : int(self.n_samples[b])].cpu().numpy()
        res["status"] = int(self.status[b])
        return res


class Engine:
    """One engine per device/stream user.  Holds only the cached accumulated-distance grid and the last plan."""

    def __init__(self, device="cuda:0", dt: float = 0.01, dd: float = 0.005, lut_samples: int = 1000,
                 samples_per_node: int = 1000, start_vel: float = 0.01, end_vel: float = 0.01,
                 velocity_impl: str = "chunked", chunks: int = 32, time_impl: str = "split", accelerators: bool = True):
        if not torch.cuda.is_available():
            raise _lib.VapError("no CUDA device: vexautonomousplanner_b200 has no CPU fallback")
        self.lib = _lib.lib()
        self.device = torch.device(device)
        self.dt, self.dd = float(dt), float(dd)
        self.samples, self.spn = int(lut_samples), int(samples_per_node)
        self.start_vel, self.end_vel = float(start_vel), float(end_vel)
        if velocity_impl not in ("chunked", "serial"):
            raise ValueError("velocity_impl must be 'chunked' or 'serial'")
        self.velocity_impl, self.chunks = velocity_impl, int(chunks)
        if time_impl not in ("split", "serial"):
            raise ValueError("time_impl must be 'split' or 'serial'")
        if (velocity_impl, time_impl) == ("serial", "split"):
            # the split time stage sizes its row redo from the chunked velocity stage's bound of the inserted rows
            raise ValueError("time_impl='split' needs velocity_impl='chunked'")
        self.time_impl = time_impl
        # accelerators=False passes NULL for the inverse LUT index and the lerp reciprocals (binary search / plain division
        # instead: same bits, slower); tests use it to pin the equivalence
        self.accelerators = bool(accelerators)
        self._dgrid: Optional[torch.Tensor] = None
        self._rden: Optional[torch.Tensor] = None
        self._retired: list = []                # outgrown path-independent tables, kept alive for captured graphs
        self._plan: Dict[tuple, tuple] = {}
        self._streams: list = []
        self._host_slots: Dict[int, list] = {}
        self.launches = 0      # kernels launched by this engine (bench.py reports it)
        self.stage_events = None   # set to a list to record (stage, start_event, end_event) per stage call

    @contextmanager
    def _stage(self, name: str):
        if self.stage_events is None:
            yield
            return
        s = torch.cuda.Event(enable_timing=True)
        e = torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.stage_events.append((name, s, e))

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _empty(self, shape, dtype=torch.float64):
        t = torch.empty(shape, dtype=dtype, device=self.device)
        if _POISON:                  # debugging aid (VAP_POISON=1): scratch starts as NaN / a large odd integer, never as zeros
            t.fill_(float("nan") if dtype.is_floating_point else (1 if dtype == torch.uint8 else 0x5a5a5a5))
        return t

    def upload(self, p: PackedPaths) -> DeviceBatch:
        return DeviceBatch.from_packed(p, self.device)

    def _with_true_splines(self, db: DeviceBatch, n_splines: Optional[torch.Tensor] = None) -> DeviceBatch:
        """db, or a DeviceBatch over the same tensors that carries the batch's true spline count when db.max_splines
        understates it (e.g. a captured graph's static inputs with another batch copied in).  The count is the geometry
        kernel's own n_splines (0 for failed paths); without them, one vap_build_path runs here (retry path only)."""
        if n_splines is None:
            n_splines = self.build_geometry(db).n_splines
        S = int(n_splines.max().item()) if n_splines.numel() else 0
        return replace(db, max_splines=S) if S > db.max_splines else db

    def dgrid(self, n: int) -> torch.Tensor:
        """Accumulated distance grid d_{i+1} = fl(d_i + dd), cached and grown geometrically."""
        if self._dgrid is None or self._dgrid.numel() < n:
            m = max(int(n * 1.5), 1 << 14)
            g = self._empty((m,))
            _lib.check(self.lib.vap_build_dgrid(C.c_int64(m), C.c_double(self.dd), _p(g), self._stream()), "vap_build_dgrid")
            self.launches += 1
            if self._dgrid is not None:
                self._retired.append(self._dgrid)      # captured graphs may still read the smaller table
            self._dgrid = g
        return self._dgrid

    def lerp_recip(self, n: int) -> torch.Tensor:
        """1 / (xs[i+1] - xs[i]) on xs[i] = fl(i*dd) (the time loop's lerp denominators), cached and grown geometrically."""
        if self._rden is None or self._rden.numel() < n:
            m = max(int(n * 1.5), 1 << 14)
            r = self._empty((m,))
            _lib.check(self.lib.vap_build_lerp_recip(C.c_int64(m), C.c_double(self.dd), _p(r), self._stream()), "vap_build_lerp_recip")
            self.launches += 1
            if self._rden is not None:
                self._retired.append(self._rden)
            self._rden = r
        return self._rden

    # ------------------------------------------------------------------ stages
    def build_geometry(self, db: DeviceBatch, with_params: bool = False) -> Geometry:
        B, N = db.B, db.N_max
        g = Geometry(self._empty((B, max(N - 1, 1), 6, 2)), self._empty((B, N + 1), torch.int32), self._empty((B, N)),
                     self._empty((B, N)), self._empty((B,), torch.int32), self._empty((B,), torch.int32))
        scratch = self._empty((B, N, 9))
        if with_params:
            g.params = torch.zeros((B, 2 * N), dtype=torch.float64, device=self.device)
            g.derivs = torch.zeros((B, 2 * N, 4), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.vap_build_path(C.c_int64(B), C.c_int(N), _p(db.node_attr), _p(db.node_flags), _p(db.n_nodes),
                                           _p(g.seg), _p(g.first_node), _p(g.param_end), _p(g.seglen), _p(g.n_splines),
                                           _p(g.status), _p(scratch), _p(g.params), _p(g.derivs), self._stream()),
                   "vap_build_path")
        self.launches += 1
        return g

    def build_lut(self, db: DeviceBatch, g: Geometry, samples: Optional[int] = None) -> Tables:
        samples = samples or self.samples
        B = db.B
        Q_cap = samples * max(db.max_splines, 1)
        t = Tables(samples, self.spn, Q_cap, 0, self._empty((B, Q_cap)), self._empty((B, Q_cap)), self._empty((B,)))
        _lib.check(self.lib.vap_build_lut(C.c_int64(B), C.c_int(db.N_max), _p(g.seg), _p(g.first_node), _p(g.param_end),
                                          _p(g.n_splines), _p(g.status), C.c_int(samples), C.c_int64(Q_cap), _p(t.lut_d),
                                          _p(t.lut_t), _p(t.total_len), self._stream()), "vap_build_lut")
        self.launches += 1
        # inverse index of the distance table: seeds every later distance_to_time lookup (same results, ~10x fewer loads)
        t.lut_inv = self._empty((B, int(self.lib.vap_lut_index_row_ints(C.c_int64(Q_cap)))), torch.int32)
        _lib.check(self.lib.vap_build_lut_index(C.c_int64(B), _p(g.n_splines), _p(g.status), C.c_int(samples), C.c_int64(Q_cap),
                                                _p(t.lut_d), _p(t.total_len), _p(t.lut_inv), self._stream()), "vap_build_lut_index")
        self.launches += 1
        return t

    def build_props(self, db: DeviceBatch, g: Geometry, t: Tables, spn: Optional[int] = None) -> Tables:
        spn = spn or self.spn
        B = db.B
        t.spn = spn
        t.P_cap = spn * db.N_max
        t.prop_k = self._empty((B, t.P_cap))
        t.prop_h = self._empty((B, t.P_cap))
        _lib.check(self.lib.vap_build_props(C.c_int64(B), C.c_int(db.N_max), _p(db.n_nodes), _p(g.seg), _p(g.first_node),
                                            _p(g.param_end), _p(g.n_splines), _p(g.status), C.c_int(spn), C.c_int64(t.P_cap),
                                            _p(t.prop_k), _p(t.prop_h), self._stream()), "vap_build_props")
        self.launches += 1
        return t

    def gl_queries(self, g: Geometry, path, spl, a, b, mode: int = 0, num_points: int = 20, max_iter: int = 50):
        """Batched Gauss-Legendre arc length (mode 0: a, b = t_start, t_end) or its bisection inverse (mode 1: a = arc
        length, b = tolerance) on spline spl[q] of path path[q] (quintic_hermite_spline.py:592-717): one thread per
        query.  Returns (values[n] f64, qstatus[n] i32: 0 ok, -3 where the reference raises ValueError)."""
        path = torch.as_tensor(path, dtype=torch.int32).to(self.device)
        spl = torch.as_tensor(spl, dtype=torch.int32).to(self.device)
        a = torch.as_tensor(a, dtype=torch.float64).to(self.device)
        b = torch.as_tensor(b, dtype=torch.float64).to(self.device).expand_as(a).contiguous()
        n = int(a.numel())
        pts, wts = np.polynomial.legendre.leggauss(num_points)     # the reference's own nodes / weights (:628)
        dp, dw = torch.from_numpy(pts).to(self.device), torch.from_numpy(wts).to(self.device)
        out = self._empty((n,)); qst = self._empty((n,), torch.int32)
        N_max = g.param_end.shape[1]
        _lib.check(self.lib.vap_gl(C.c_int64(n), _p(path), _p(spl), _p(a), _p(b), C.c_int(mode), C.c_int(max_iter),
                                   C.c_int(num_points), _p(dp), _p(dw), C.c_int(N_max), _p(g.seg), _p(g.first_node),
                                   _p(g.param_end), _p(out), _p(qst), self._stream()), "vap_gl")
        self.launches += 1
        torch.cuda.current_stream(self.device).synchronize()     # dp / dw / the converted inputs die with this frame
        return out, qst

    def dist_sample(self, db: DeviceBatch, g: Geometry, t: Tables, status: torch.Tensor, D_cap: int):
        B = db.B
        grid = self.dgrid(D_cap + 2)
        n_samples = self._empty((B,), torch.int32)
        tq, kap, th = self._empty((B, D_cap)), self._empty((B, D_cap)), self._empty((B, D_cap))
        _lib.check(self.lib.vap_dist_sample(C.c_int64(B), _p(db.n_nodes), _p(g.n_splines), _p(status), C.c_int64(grid.numel()),
                                            _p(grid), C.c_int(t.samples), C.c_int64(t.Q_cap), _p(t.lut_d), _p(t.lut_t),
                                            _p(t.total_len), C.c_int(t.spn), C.c_int64(t.P_cap), _p(t.prop_k), _p(t.prop_h),
                                            C.c_int64(D_cap), _p(n_samples), _p(tq), _p(kap), _p(th), self._stream()),
                   "vap_dist_sample")
        self.launches += 2
        return n_samples, tq, kap, th

    def fwd_bwd(self, db: DeviceBatch, status, D_cap, n_samples, tq, kap, th, mode: int = 0):
        B = db.B
        E_cap = db.N_max + db.A_max + 2
        vel = self._empty((B, D_cap))
        ma = self._empty((B, E_cap))
        bidx = self._empty((B, E_cap), torch.int32)
        bval = self._empty((B, E_cap), torch.int32)
        n_ev = self._empty((B, 2), torch.int32)
        t_est = self._empty((B,))
        _lib.check(self.lib.vap_fwd_bwd(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), _p(db.node_attr),
                                        _p(db.node_flags), _p(db.n_nodes), _p(db.ap_attr), _p(db.ap_flags), _p(db.n_ap),
                                        _p(db.cons), _p(status), C.c_double(self.dd), C.c_double(self.dt),
                                        C.c_double(self.start_vel), C.c_double(self.end_vel), C.c_int64(D_cap),
                                        _p(n_samples), _p(tq), _p(kap), _p(th), _p(vel), C.c_int(E_cap), _p(ma), _p(bidx),
                                        _p(bval), _p(n_ev), _p(t_est), C.c_int(mode), self._stream()), "vap_fwd_bwd")
        self.launches += 1
        return vel, ma, bidx, bval, n_ev, t_est

    def velocity_chunked(self, db: DeviceBatch, g: Geometry, t: Tables, status: torch.Tensor, D_cap: int, mode: int = 0,
                         want_t: bool = True):
        """S3 + events + S4 + S5, fast path: sampling fused with the hoisted pre-pass (vap_velocity_profile), sample-parallel
        events, chunk-speculative passes.  want_t: also write t / kappa / theta per distance sample (inspection outputs).
        Returns n_samples, vel, t_est (time samples of the main loop), ins_est (bound of the rows that waits and turns
        insert) and the intermediates."""
        B = db.B
        E_cap = db.N_max + db.A_max + 2
        grid = self.dgrid(D_cap + 2)
        n_samples = self._empty((B,), torch.int32)
        tq = self._empty((B, D_cap)) if want_t else None      # t / kappa / theta per distance sample: inspection outputs
        kap = self._empty((B, D_cap)) if want_t else None
        th = self._empty((B, D_cap)) if want_t else None
        ma = self._empty((B, E_cap)); bidx = self._empty((B, E_cap), torch.int32); bval = self._empty((B, E_cap), torch.int32)
        n_ev = self._empty((B, 2), torch.int32)
        vr_idx = self._empty((B, E_cap), torch.int32); vr_val = self._empty((B, E_cap))
        st_idx = self._empty((B, E_cap), torch.int32); n_vr = self._empty((B, 2), torch.int32)
        ins_est = self._empty((B,), torch.float32)
        nscr = int(self.lib.vap_event_scratch_ints(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max)))
        scr = self._empty((nscr,), torch.int32)
        chunks = self.chunks if D_cap <= 65536 else 256
        RS = int(self.lib.vap_pass_row_slots(C.c_int64(D_cap), C.c_int(chunks)))     # chunk-interleaved rows of the pass arrays
        rec = self._empty((B, RS, 4)); statB = self._empty((B, RS))
        vel_f = self._empty((B, RS)); vel = self._empty((B, D_cap))
        t_est = self._empty((B,), torch.float32)
        rounds = torch.zeros((B, 2), dtype=torch.int32, device=self.device)
        inv = t.lut_inv if self.accelerators else None
        with self._stage("S345_velocity"):
            _lib.check(self.lib.vap_velocity_profile(
                C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), _p(db.node_attr), _p(db.node_flags), _p(db.n_nodes),
                _p(db.ap_attr), _p(db.ap_flags), _p(db.n_ap), _p(db.cons), _p(g.n_splines), _p(status),
                C.c_int64(grid.numel()), _p(grid), C.c_int(t.samples), C.c_int64(t.Q_cap), _p(t.lut_d), _p(t.lut_t),
                _p(t.total_len), C.c_int(t.spn), C.c_int64(t.P_cap), _p(t.prop_k), _p(t.prop_h), _p(inv),
                C.c_double(self.dd), C.c_double(self.dt), C.c_double(self.start_vel), C.c_double(self.end_vel),
                C.c_int64(D_cap), _p(n_samples), _p(tq), _p(kap), _p(th), C.c_int(E_cap), _p(ma), _p(bidx), _p(bval),
                _p(n_ev), _p(vr_idx), _p(vr_val), _p(st_idx), _p(n_vr), _p(ins_est), _p(scr), _p(rec), _p(statB),
                _p(vel_f), _p(vel), _p(t_est), _p(rounds), C.c_int(chunks), C.c_int(mode), self._stream()),
                "vap_velocity_profile")
            self.launches += 6
        extra = dict(t=tq, kap=kap, th=th, max_accels=ma, bidx=bidx, bval=bval, n_ev=n_ev, vel_f=vel_f, rounds=rounds,
                     vr_idx=vr_idx, vr_val=vr_val, st_idx=st_idx, n_vr=n_vr)
        return n_samples, vel, t_est, ins_est, extra

    def velocity_serial(self, db: DeviceBatch, g: Geometry, t: Tables, status: torch.Tensor, D_cap: int, mode: int = 0):
        """S3 + events + S4 + S5, reference-shaped variant: one thread walks each path (kept as a cross-check).  Returns
        what velocity_chunked does, except that t_est already counts the inserted rows and ins_est is None."""
        with self._stage("S3_dist_sample"):
            n_samples, tq, kap, th = self.dist_sample(db, g, t, status, D_cap)
        with self._stage("S45_fwd_bwd"):
            vel, ma, bidx, bval, n_ev, t_est = self.fwd_bwd(db, status, D_cap, n_samples, tq, kap, th, mode)
        extra = dict(t=tq, kap=kap, th=th, max_accels=ma, bidx=bidx, bval=bval, n_ev=n_ev)
        return n_samples, vel, t_est, None, extra

    def resample(self, db: DeviceBatch, g: Geometry, t: Tables, status, D_cap, n_samples, vel, T_cap):
        """S6 + S7, reference-shaped variant: returns what time_profile does, with None for n_main (not counted)."""
        B = db.B
        out = self._empty((8, B, T_cap))
        nodes_map = self._empty((B, db.N_max + 1), torch.int32)
        actions_map = self._empty((B, max(db.A_max, 1)), torch.int32)
        n_maps = self._empty((B, 2), torch.int32)
        n_out = self._empty((B,), torch.int32)
        summary = self._empty((B, 5))
        _lib.check(self.lib.vap_resample(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), _p(db.node_attr),
                                         _p(db.node_flags), _p(db.n_nodes), _p(db.ap_attr), _p(db.ap_flags), _p(db.n_ap),
                                         _p(db.cons), _p(status), C.c_double(self.dt), C.c_double(self.dd), _p(g.seg),
                                         _p(g.first_node), _p(g.param_end), _p(g.n_splines), C.c_int(t.samples),
                                         C.c_int64(t.Q_cap), _p(t.lut_d), _p(t.lut_t), _p(t.total_len), C.c_int(t.spn),
                                         C.c_int64(t.P_cap), _p(t.prop_k), _p(t.prop_h), C.c_int64(D_cap), _p(n_samples),
                                         _p(vel), C.c_int64(T_cap), _p(out), _p(nodes_map), _p(actions_map), _p(n_maps),
                                         _p(n_out), _p(summary), self._stream()), "vap_resample")
        self.launches += 1
        return out, nodes_map, actions_map, n_maps, n_out, summary, None

    def time_profile(self, db: DeviceBatch, g: Geometry, t: Tables, status, D_cap, n_samples, vel, T_cap):
        """S6 + S7, fast path (vap_time_profile): state recurrence / parallel lookups / event replay / scatter.  n_main, the
        last output, counts each path's main-loop rows (exact also when the rows did not fit)."""
        B = db.B
        E_cap = db.N_max + db.A_max + 2
        out = self._empty((8, B, T_cap))
        nodes_map = self._empty((B, db.N_max + 1), torch.int32)
        actions_map = self._empty((B, max(db.A_max, 1)), torch.int32)
        n_maps = self._empty((B, 2), torch.int32)
        n_out = self._empty((B,), torch.int32)
        summary = self._empty((B, 5))
        n_main = self._empty((B,), torch.int32)
        rden = self.lerp_recip(D_cap + 2)
        stage = self._empty((8, B, T_cap + 1))
        seg_tab = self._empty((3 * B * E_cap + B,), torch.int32)
        nscr = int(self.lib.vap_event_scratch_ints(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max)))
        scr = self._empty((nscr,), torch.int32)
        _lib.check(self.lib.vap_time_profile(
            C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), _p(db.node_attr), _p(db.node_flags), _p(db.n_nodes),
            _p(db.ap_attr), _p(db.ap_flags), _p(db.n_ap), _p(db.cons), _p(status), C.c_double(self.dt), C.c_double(self.dd),
            _p(g.seg), _p(g.first_node), _p(g.param_end), _p(g.n_splines), C.c_int(t.samples), C.c_int64(t.Q_cap),
            _p(t.lut_d), _p(t.lut_t), _p(t.total_len), C.c_int(t.spn), C.c_int64(t.P_cap), _p(t.prop_k), _p(t.prop_h),
            C.c_int64(D_cap), _p(n_samples), _p(vel), C.c_int64(T_cap), _p(out), _p(nodes_map), _p(actions_map), _p(n_maps),
            _p(n_out), _p(summary), _p(n_main), _p(stage), C.c_int(E_cap), _p(seg_tab), _p(scr), C.c_int64(0),
            _p(t.lut_inv if self.accelerators else None), _p(rden if self.accelerators else None), C.c_int64(rden.numel()),
            self._stream()), "vap_time_profile")
        self.launches += 5
        return out, nodes_map, actions_map, n_maps, n_out, summary, n_main

    # ------------------------------------------------------------------ tiled, multi-stream execution
    def _profile_tiled(self, db: DeviceBatch, D_cap: int, T_cap: int, tiles: int, host: "Optional[HostResult]" = None,
                       dense: Optional[torch.Tensor] = None, events: Optional[list] = None) -> ProfileResult:
        """vap_profile_batch over `tiles` row slices of the batch, each on its own CUDA stream.

        The serial chains (time loop, chunked velocity passes) are latency-bound and leave most issue slots idle,
        while the table / sampling / pre-pass kernels are throughput-bound; running tiles on separate streams lets the
        block scheduler co-schedule one tile's chains with another tile's sample-parallel kernels.  Tiles write straight
        into their rows of the batch-wide outputs (out_plane_stride); row k of res.extra["need"] is tile k's `need`.
        Capacities come from the cached plan.  Like every vap_profile_batch call this uses the inverse LUT index also
        when the engine was built with accelerators=False (the same bits).
        """
        B = db.B
        main = torch.cuda.current_stream(self.device)
        res = self._batch_result(db, D_cap, T_cap, tiles)
        self.dgrid(D_cap + 2)                      # make sure the shared tables exist before the side streams read them
        self.lerp_recip(D_cap + 2)
        while len(self._streams) < tiles:
            # earlier tiles get higher stream priority, so that they finish (and start streaming their rows to the host)
            # while later tiles still compute, instead of all tiles finishing together
            k = len(self._streams)
            self._streams.append(torch.cuda.Stream(device=self.device, priority=max(-5, -(5 - min(k, 5)))))
        bounds = [(B * k // tiles, B * (k + 1) // tiles) for k in range(tiles)]
        for k, (lo, hi) in enumerate(bounds):
            if hi <= lo:
                continue
            s = self._streams[k]
            s.wait_stream(main)
            with torch.cuda.stream(s):
                self._profile_rows(db, res, lo, hi, k)
                if host is not None:
                    # dense rows straight into pinned host memory (the kernel streams them over PCIe), then the small
                    # per-path arrays with ordinary async copies; all of it overlaps the other tiles' kernels
                    offs = host.dev_offsets[lo + k: hi + k + 1]
                    # dst: pinned host memory (the kernel streams over PCIe itself) or a dense device buffer that the
                    # copy engine moves afterwards, once the host knows the tile's row count
                    base = host.packed if dense is None else dense
                    dst = C.c_void_p(base.data_ptr() + 8 * 8 * lo * T_cap)
                    _lib.check(self.lib.vap_pack_rows(C.c_int64(hi - lo), C.c_int64(T_cap), C.c_int64(B * T_cap),
                                                      _p(res.out[:, lo:hi]), _p(res.n_out[lo:hi]), _p(res.status[lo:hi]),
                                                      _p(offs), dst, self._stream()), "vap_pack_rows")
                    self.launches += 2
                    host.offsets[lo + k: hi + k + 1].copy_(offs, non_blocking=True)
                    for name in ("n_out", "status", "nodes_map", "actions_map", "n_maps", "summary"):
                        getattr(host, name)[lo:hi].copy_(getattr(res, name)[lo:hi], non_blocking=True)
                    if events is not None:
                        events[k].record(s)
        for k in range(tiles):
            main.wait_stream(self._streams[k])
        return res

    def profile_many(self, packed: PackedPaths, tile_paths: int = 16384, sink=None) -> torch.Tensor:
        """Jobs larger than one call (e.g. 2**20 16-node paths: 190 GB of trajectories): profile `tile_paths` paths at a
        time, hand every tile's device-resident ProfileResult to `sink(lo, hi, result)` (export, reduction, D2H ...) and
        return the [B, 5] summary rows of the whole job.  Capacities are planned once per tile shape and reused."""
        B = packed.B
        rows = []
        for lo in range(0, B, tile_paths):
            hi = min(B, lo + tile_paths)
            res = self.profile(self.upload(packed.slice(lo, hi)), reuse_plan=True)
            if sink is not None:
                sink(lo, hi, res)
            rows.append(res.summary)
        return torch.cat(rows, dim=0) if rows else self._empty((0, 5))

    def _host_state(self, packed: PackedPaths, tiles: int, state: Optional[dict]) -> dict:
        """Reusable buffers of the host-in / host-out path for one batch shape (device inputs, dense device rows, pinned
        inputs and results, per-tile events, a copy stream)."""
        B = packed.B
        key = (B, packed.N_max, packed.A_max, packed.max_splines())
        st = state or {}
        if st.get("key") == key:
            return st
        db = self.upload(packed)
        self.profile(db, reuse_plan=True)                       # plan (D_cap, T_cap) for this shape
        D_cap, T_cap = self._plan[(B, db.N_max, db.A_max, db.max_splines)]
        tiles = max(1, min(tiles, B))
        return dict(key=key, db=db, D_cap=D_cap, T_cap=T_cap, tiles=tiles,
                    host=HostResult(self, B, db.N_max, db.A_max, T_cap, tiles),
                    dense=self._empty((8 * B * T_cap,)), events=[torch.cuda.Event() for _ in range(tiles)],
                    copy_stream=torch.cuda.Stream(device=self.device), pin=db.pinned())

    def _host_submit(self, packed: PackedPaths, st: dict) -> None:
        """Enqueue one batch: inputs host -> device, every tile's kernels, dense packing, small result arrays."""
        st["db"].upload_(packed, st["pin"])
        self._profile_tiled(st["db"], st["D_cap"], st["T_cap"], st["tiles"], host=st["host"], dense=st["dense"],
                            events=st["events"])

    def _host_issue_d2h(self, st: dict) -> None:
        """As each tile's row count reaches the host, queue the copy of exactly those bytes on the copy stream (the copy
        engine is the bottleneck of the host-out path: nothing else may delay these enqueues)."""
        host, T_cap, cs = st["host"], st["T_cap"], st["copy_stream"]
        for k, (lo, hi) in enumerate(host.bounds):
            if hi <= lo:
                continue
            st["events"][k].synchronize()                          # tile k packed; its counts are in pinned memory
            total = int(host.offsets[hi + k])
            a = 8 * lo * T_cap
            with torch.cuda.stream(cs):
                host.packed[a: a + 8 * total].copy_(st["dense"][a: a + 8 * total], non_blocking=True)
        if st.get("d2h_done") is None:
            st["d2h_done"] = torch.cuda.Event()
        st["d2h_done"].record(cs)

    def _host_wait(self, st: dict) -> "HostResult":
        st["d2h_done"].synchronize()
        host = st["host"]
        host.state = st
        return host

    def _host_collect(self, st: dict) -> "HostResult":
        self._host_issue_d2h(st)
        return self._host_wait(st)

    def profile_to_host(self, packed: PackedPaths, tiles: int = 8, state: Optional[dict] = None,
                        _retry: int = 0) -> "HostResult":
        """Host buffers in, host buffers out: every tile packs its valid rows densely on the device; as soon as a tile's
        row count has reached the host, the copy engine moves exactly those bytes into pinned memory while later tiles
        are still computing.  `state` (returned in HostResult.state) carries the reusable buffers."""
        st = self._host_state(packed, tiles, state)
        self._host_submit(packed, st)
        host = self._host_collect(st)
        torch.cuda.current_stream(self.device).synchronize()
        if bool((host.status == ST_CAPACITY).any()) and _retry < MAX_RETRIES:
            self._plan.pop((packed.B, st["db"].N_max, st["db"].A_max, st["db"].max_splines), None)
            st["key"] = None
            return self.profile_to_host(packed, tiles, st, _retry=_retry + 1)
        return host

    def stream_to_host(self, batches, tiles: int = 4, depth: int = 3):
        """Bulk jobs: a generator over HostResults for an iterable of same-shape PackedPaths batches, software-pipelined
        three deep: while batch n's rows cross PCIe, batch n+1's kernels run and batch n+2 is being enqueued.  The copy
        engine is the bottleneck, so the order per step is: enqueue the next batch's kernels, queue the device -> host copy
        of the batch that just finished computing, and only then wait for the copy before it -- the copy stream never runs
        dry behind host-side launch work.  A yielded HostResult is valid until the generator is advanced."""
        depth = max(int(depth), 3)
        slots = self._host_slots.setdefault(depth, [None] * depth)   # pinned buffers are expensive: kept across calls
        submitted, copying = [], []                              # (slot index, batch): kernels in flight / copy in flight
        n = 0
        for packed in batches:
            k = n % depth
            slots[k] = self._host_state(packed, tiles, slots[k])
            self._host_submit(packed, slots[k])
            submitted.append((k, packed))
            n += 1
            while len(submitted) > 1:
                ks, pk = submitted.pop(0)
                self._host_issue_d2h(slots[ks])
                copying.append((ks, pk))
            while len(copying) > 1:
                ks, pk = copying.pop(0)
                yield self._finish_streamed(slots, ks, pk, tiles)
        while submitted:
            ks, pk = submitted.pop(0)
            self._host_issue_d2h(slots[ks])
            copying.append((ks, pk))
        while copying:
            ks, pk = copying.pop(0)
            yield self._finish_streamed(slots, ks, pk, tiles)

    def _finish_streamed(self, slots, k, packed, tiles):
        host = self._host_wait(slots[k])
        if bool((host.status == ST_CAPACITY).any()):             # rare: plan too small -> exact, unpipelined redo
            host = self.profile_to_host(packed, tiles, None)
        return host

    def capture(self, db: DeviceBatch, tiles: int = 4, to_host: bool = False, margin: float = 1.0) -> "GraphedProfile":
        """Capture the tiled fast path for this batch shape into a CUDA graph (one launch per step afterwards).
        to_host=True adds the pack kernels that stream the dense result rows into pinned host memory.
        margin > 1 enlarges the capacities planned from `db`, for graphs that will be fed OTHER batches of the same shape
        (run(new_db)); a batch that still does not fit is detected on the device and redone exactly, outside the graph."""
        return GraphedProfile(self, db, tiles, to_host=to_host, margin=margin)

    # ------------------------------------------------------------------ whole path, one C call
    def plan_capacities(self, db: DeviceBatch, margin: float = 1.0):
        """(D_cap, T_cap) for this batch shape: the cached plan, or one exact profile() that measures them."""
        key = (db.B, db.N_max, db.A_max, db.max_splines)
        if key not in self._plan:
            self.profile(db, reuse_plan=False)
        if key not in self._plan:
            # db understates its spline count: profile() redid (and planned) the batch under its true count
            key = key[:3] + (self._with_true_splines(db).max_splines,)
        D_cap, T_cap = self._plan[key]
        if margin > 1.0:
            D_cap, T_cap = (int(D_cap * margin) + 127) // 128 * 128, int(T_cap * margin) + 64
        return D_cap, T_cap

    def profile_batch(self, db: DeviceBatch, D_cap: Optional[int] = None, T_cap: Optional[int] = None,
                      _retry: int = 0) -> ProfileResult:
        """The whole hot path through the single C entry point vap_profile_batch (include/vap.h): S0 -> S7 out of ONE
        workspace, capacities checked on the device.  Without capacities the cached plan (or one exact profile()) sizes
        the call; a path that outgrows them comes back as ST_CAPACITY and the call is redone with the sizes the device
        reported in `need` (bounded retries)."""
        if D_cap is None or T_cap is None:
            D_cap, T_cap = self.plan_capacities(db)
        res = self._batch_result(db, (int(D_cap) + 127) // 128 * 128, int(T_cap), 1)
        self._profile_rows(db, res, 0, db.B, 0)
        return self._redo_overflow(db, res, _retry)

    def _batch_result(self, db: DeviceBatch, D_cap: int, T_cap: int, parts: int) -> ProfileResult:
        """Outputs of vap_profile_batch for the whole batch, filled by `parts` calls on row slices (_profile_rows)."""
        B = db.B
        res = ProfileResult(B, T_cap, self._empty((8, B, T_cap)), self._empty((B,), torch.int32),
                            self._empty((B, db.N_max + 1), torch.int32), self._empty((B, max(db.A_max, 1)), torch.int32),
                            self._empty((B, 2), torch.int32), self._empty((B,), torch.int32), self._empty((B, 5)),
                            self._empty((B, D_cap)), self._empty((B,), torch.int32))
        res.extra = dict(need=self._empty((parts, 3), torch.int64), workspace=[])
        return res

    def _profile_rows(self, db: DeviceBatch, res: ProfileResult, lo: int, hi: int, part: int) -> None:
        """One vap_profile_batch call on paths lo..hi of `db`, on the current stream, into the same rows of `res`, with
        res.extra["need"][part] as its `need`.  Its workspace stays alive with `res` (a captured graph replays into it).
        The inverse LUT index is always used; the lerp reciprocals only with accelerators (both give the same bits)."""
        B, D_cap, T_cap = hi - lo, res.vel.shape[1], res.T_cap
        S = max(db.max_splines, 1)
        chunks = self.chunks if D_cap <= 65536 else 256
        grid, rden = self.dgrid(D_cap + 2), self.lerp_recip(D_cap + 2)
        nbytes = int(self.lib.vap_workspace_bytes(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), C.c_int(S),
                                                  C.c_int(self.samples), C.c_int(self.spn), C.c_int64(D_cap), C.c_int64(T_cap),
                                                  C.c_int(chunks)))
        if nbytes < 0:
            raise _lib.VapError("vap_workspace_bytes: " + self.lib.vap_last_error().decode())
        ws = torch.empty((nbytes + 255,), dtype=torch.uint8, device=self.device)
        res.extra["workspace"].append(ws)
        sub = db.rows(lo, hi)
        _lib.check(self.lib.vap_profile_batch(
            C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), C.c_int(S), *(_p(t) for t in sub.tensors()),
            C.c_double(self.dt), C.c_double(self.dd), C.c_double(self.start_vel), C.c_double(self.end_vel),
            C.c_int(self.samples), C.c_int(self.spn), C.c_int64(D_cap), C.c_int64(T_cap), C.c_int(chunks), _p(grid),
            C.c_int64(grid.numel()), _p(rden if self.accelerators else None), C.c_int64(rden.numel()),
            C.c_void_p((ws.data_ptr() + 255) // 256 * 256), C.c_int64(nbytes), C.c_void_p(res.out.data_ptr() + 8 * lo * T_cap),
            C.c_int64(res.B * T_cap), _p(res.n_out[lo:hi]), _p(res.nodes_map[lo:hi]), _p(res.actions_map[lo:hi]),
            _p(res.n_maps[lo:hi]), _p(res.status[lo:hi]), _p(res.summary[lo:hi]), _p(res.vel[lo:hi]),
            _p(res.n_samples[lo:hi]), _p(res.extra["need"][part]), self._stream()), "vap_profile_batch")
        self.launches += PROFILE_BATCH_KERNELS

    def _redo_overflow(self, db: DeviceBatch, res: ProfileResult, retry: int = 0) -> ProfileResult:
        """`res` (from vap_profile_batch calls on db), or, when a path outgrew the capacities (ST_CAPACITY), its redo through
        profile_batch with the sizes the device reported in res.extra["need"] (the maximum over its calls); bounded by
        MAX_RETRIES.  db is only read: a redo runs on a new DeviceBatch over the same tensors."""
        if retry >= MAX_RETRIES or not bool((res.status == ST_CAPACITY).any().item()):
            return res
        d_need, t_est, t_exact = (int(v) for v in res.extra["need"].max(dim=0).values.tolist())
        # need[] does not cover paths with more splines than db.max_splines (they were stopped before sampling): the
        # redo carries the true count, which can only be short once, so that redo does not use up a retry
        exact = self._with_true_splines(db)
        return self.profile_batch(exact, max(res.vel.shape[1], d_need + 8),
                                  max(res.T_cap, int(max(t_est, t_exact) * 1.10) + 64), retry + (1 if exact is db else 0))

    # ------------------------------------------------------------------ whole path
    def _plan_distance(self, t: Tables, status: torch.Tensor) -> int:
        """D_cap from the longest healthy path.  Paths whose length is infinite or absurd (the reference's sampling loop
        `while d < total_length` would never end / never fit in memory) are flagged ST_DIVERGED here, so that neither they
        nor a NaN length (for which the reference's loops simply do not run: empty result lists) size the buffers."""
        L = t.total_len
        absurd = (L / self.dd > DIST_LIMIT) & (status == ST_OK)          # false for NaN
        status[absurd] = ST_DIVERGED
        ok_len = torch.where((status == ST_OK) & torch.isfinite(L), L, torch.zeros_like(L))
        Lmax = float(ok_len.max().item()) if ok_len.numel() else 0.0
        D_cap = (int(Lmax / self.dd) + 8 + 127) // 128 * 128             # rows padded to whole 128-sample blocks
        need = 12 * 8 * D_cap * max(int(L.numel()), 1)                   # ~12 [B, D_cap] fp64 arrays live at the peak
        free, _ = torch.cuda.mem_get_info(self.device)
        reusable = torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if need > free + reusable:
            raise _lib.VapError(f"batch needs about {need / 2**30:.1f} GiB of distance-domain scratch (longest path: {Lmax:.1f} ft = "
                                f"{D_cap} samples x {L.numel()} paths) but only {(free + reusable) / 2**30:.1f} GiB are free: "
                                "tile the batch (Engine.profile_many) or bucket the paths by length")
        return D_cap

    def _plan_rows(self, est: torch.Tensor, status: torch.Tensor) -> int:
        """T_cap from the estimated time samples of every path (inserted rows included).  Paths whose profile would need an
        absurd number of rows (the reference would effectively never return) are flagged ST_DIVERGED here, so that they
        neither size the buffers nor spin in the time loop."""
        absurd = ~(est < ROW_LIMIT)
        status[absurd & (status == ST_OK)] = ST_DIVERGED
        return int(float(torch.where(absurd, torch.zeros_like(est), est).max().item()) * 1.10) + 64

    def profile(self, db: DeviceBatch, keep: bool = False, reuse_plan: bool = False, tiles: int = 1,
                _retry: int = 0) -> ProfileResult:
        """build_path + generate_motion_profile for every path of the batch.

        reuse_plan, with a plan for this batch shape (and the fast implementations, keep=False, no stage_events): the
        planned step, vap_profile_batch sized by the plan -- one call on the current stream (tiles == 1) or `tiles` row
        slices on their own streams (_profile_tiled).  Capacity overflows are detected on the device and redone
        (_redo_overflow); the capacities that ran become the plan of this shape.
        Every other call is the staged run, one C entry per stage: it measures D_cap / T_cap from the data (two
        read-backs), records per-stage timings when stage_events is a list, and plans this batch shape.
        keep: also return geometry / tables / distance-domain intermediates.
        """
        B = db.B
        key = (B, db.N_max, db.A_max, db.max_splines)
        if (reuse_plan and not keep and key in self._plan and self.stage_events is None
                and self.velocity_impl == "chunked" and self.time_impl == "split"):
            D_cap, T_cap = self._plan[key]
            tiles = min(tiles, B)
            if tiles > 1:
                res = self._redo_overflow(db, self._profile_tiled(db, D_cap, T_cap, tiles), _retry)
            else:
                res = self.profile_batch(db, D_cap, T_cap, _retry)
            self._plan[key] = (res.vel.shape[1], res.T_cap)
            return res
        with self._stage("S0_build_path"):
            g = self.build_geometry(db)
        with self._stage("S1_lut"):
            t = self.build_lut(db, g)
        with self._stage("S2_props"):
            self.build_props(db, g, t)
        status = g.status.clone()
        D_cap = self._plan_distance(t, status)
        if self.velocity_impl == "chunked":
            n_samples, vel, t_est, ins_est, extra = self.velocity_chunked(db, g, t, status, D_cap, want_t=keep)
            t_est = t_est + ins_est
        else:
            n_samples, vel, t_est, ins_est, extra = self.velocity_serial(db, g, t, status, D_cap)
        T_cap = self._plan_rows(t_est, status)
        status_pre = status.clone()
        tfun = self.time_profile if self.time_impl == "split" else self.resample
        with self._stage("S6_resample"):
            out, nodes_map, actions_map, n_maps, n_out, summary, n_main = tfun(db, g, t, status, D_cap, n_samples, vel, T_cap)
        # capacity check (one small read-back; also what a caller needs to trim the rows)
        if bool((status == ST_CAPACITY).any().item()):
            if bool((status_pre == ST_CAPACITY).any().item()) and _retry < MAX_RETRIES:
                # D_cap is measured, so only an understated db.max_splines (it sizes the distance table) overflows it:
                # redo with the geometry's true spline count (bounded: a status that survives the re-runs is reported)
                return self.profile(self._with_true_splines(db, g.n_splines), keep=keep, _retry=_retry + 1)
            if self.time_impl == "split":
                # k_need_rows' rule: n_main is exact even on overflow, the inserted rows are bounded by ins_est
                live = (status == ST_OK) | (status == ST_CAPACITY)
                rows = n_main.clamp(min=0).long() + ins_est.ceil().long()
                T_cap = int(torch.where(live, rows, torch.zeros_like(rows)).max().item()) + 8
            else:
                T_cap = int(n_out.max().item()) + 8
            status = status_pre.clone()
            out, nodes_map, actions_map, n_maps, n_out, summary, n_main = tfun(db, g, t, status, D_cap, n_samples, vel, T_cap)
        self._plan[key] = (D_cap, T_cap)
        res = ProfileResult(B, T_cap, out, n_out, nodes_map, actions_map, n_maps, status, summary, vel, n_samples)
        if keep:
            res.geometry, res.tables = g, t
            res.extra = dict(extra, t_est=t_est, n_main=n_main)
        return res


class HostResult:
    """Pinned host buffers for one batch shape: results packed densely per path (no padding crosses PCIe).

    packed: for tile k (paths lo..hi) the block starts at element 8*lo*T_cap; inside it path b's eight streams are stored
    back to back at 8*offsets[b] .. 8*(offsets[b] + n_out[b]) in the order of engine.OUT_NAMES.
    """

    def __init__(self, eng: "Engine", B: int, N_max: int, A_max: int, T_cap: int, tiles: int):
        self.B, self.T_cap, self.tiles = B, T_cap, tiles
        self.bounds = [(B * k // tiles, B * (k + 1) // tiles) for k in range(tiles)]
        pin = dict(pin_memory=True)
        self.packed = torch.empty(8 * B * T_cap, dtype=torch.float64, **pin)
        self.offsets = torch.zeros(B + tiles, dtype=torch.int64, **pin)         # tile k owns offsets[lo+k : hi+k+1]
        self.dev_offsets = torch.zeros(B + tiles, dtype=torch.int64, device=eng.device)
        self.n_out = torch.zeros(B, dtype=torch.int32, **pin)
        self.status = torch.zeros(B, dtype=torch.int32, **pin)
        self.nodes_map = torch.zeros((B, N_max + 1), dtype=torch.int32, **pin)
        self.actions_map = torch.zeros((B, max(A_max, 1)), dtype=torch.int32, **pin)
        self.n_maps = torch.zeros((B, 2), dtype=torch.int32, **pin)
        self.summary = torch.zeros((B, 5), dtype=torch.float64, **pin)

    def bytes_per_step(self) -> int:
        """Bytes that crossed PCIe towards the host for the last batch."""
        rows = int(sum(int(self.offsets[hi + k]) for k, (lo, hi) in enumerate(self.bounds)))
        small = sum(t.numel() * t.element_size() for t in (self.offsets, self.n_out, self.status, self.nodes_map,
                                                          self.actions_map, self.n_maps, self.summary))
        return rows * 8 * 8 + small

    def path(self, b: int) -> Dict[str, np.ndarray]:
        k = next(i for i, (lo, hi) in enumerate(self.bounds) if lo <= b < hi)
        lo, _ = self.bounds[k]
        n = int(self.n_out[b])
        off = 8 * lo * self.T_cap + 8 * int(self.offsets[b + k])
        blk = self.packed[off: off + 8 * n].numpy().reshape(8, n)
        res = {nm: blk[i] for i, nm in enumerate(OUT_NAMES)}
        nm_, am_ = (int(v) for v in self.n_maps[b])
        res["nodes_map"] = self.nodes_map[b, :nm_].numpy()
        res["actions_map"] = self.actions_map[b, :am_].numpy()
        res["status"] = int(self.status[b])
        return res


class GraphedProfile:
    """The whole hot path for one batch shape as a CUDA graph: every kernel of every tile, forked over the engine's
    streams and joined again, replayed with a single launch.  The serial chains are latency-bound, so what limits a
    small batch is how quickly independent tiles can be put in flight; a graph removes the per-launch host cost.

    Inputs live in static device tensors (`self.db`); `run(new_batch)` copies a new batch of the same shape into them.
    An undersized plan is detected after the replay and the step is redone through Engine.profile_batch, with the sizes
    the device reported; the static inputs are only read by the redo.
    """

    def __init__(self, eng: Engine, db: DeviceBatch, tiles: int = 4, to_host: bool = False, margin: float = 1.0):
        if eng.velocity_impl != "chunked" or eng.time_impl != "split":
            raise ValueError("graph capture needs the fast path (velocity_impl='chunked', time_impl='split')")
        self.eng, self.db, self.tiles = eng, db, max(1, min(tiles, db.B))
        self.host: Optional[HostResult] = None
        warm = eng.profile(db, reuse_plan=True)                # sizes the plan, builds the distance grid
        # the engine's plan stays the exact one: later captures of the same shape apply the margin once, not again
        self.D_cap, self.T_cap = eng.plan_capacities(db, margin)
        if to_host:
            self.host = HostResult(eng, db.B, db.N_max, db.A_max, self.T_cap, self.tiles)
            self.host_in = db.pinned()
        l0 = eng.launches
        eng._profile_tiled(db, self.D_cap, self.T_cap, self.tiles, host=self.host)   # warm the per-stream allocator pools
        self._launches_warm = eng.launches - l0                # kernels of one step (what a replay launches)
        torch.cuda.synchronize(eng.device)
        del warm
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.res = eng._profile_tiled(db, self.D_cap, self.T_cap, self.tiles, host=self.host)
        self.launches_per_run = self._launches_warm

    def check_shape(self, new) -> None:
        """Raise ValueError unless `new` (a DeviceBatch or PackedPaths) has this graph's B, N_max and A_max.  There is no
        max_splines check: more splines than captured are flagged on the device (ST_CAPACITY), also for inputs copied
        straight into the static buffers."""
        got, want = (new.B, new.N_max, new.A_max), (self.db.B, self.db.N_max, self.db.A_max)
        if got != want:
            raise ValueError(f"batch shape (B, N_max, A_max) = {got} differs from the captured {want}: capture a graph for it")

    def run(self, new_db: Optional[DeviceBatch] = None, check: bool = True) -> ProfileResult:
        if new_db is not None:
            self.check_shape(new_db)
            self.db.copy_(new_db)
        self.graph.replay()
        self.eng.launches += self.launches_per_run
        return self.eng._redo_overflow(self.db, self.res) if check else self.res

    def run_host(self, packed: PackedPaths) -> HostResult:
        """Host buffers in, host buffers out: copy the packed inputs to the device, replay the graph (whose pack kernels
        stream the dense rows into pinned host memory while other tiles still compute), wait, return the host view."""
        if self.host is None:
            raise ValueError("capture(..., to_host=True) first")
        self.check_shape(packed)
        self.db.upload_(packed, self.host_in)
        self.graph.replay()
        self.eng.launches += self.launches_per_run
        torch.cuda.current_stream(self.eng.device).synchronize()
        if bool((self.host.status == ST_CAPACITY).any()):
            raise _lib.VapError("capacity plan too small for this batch: re-capture (Engine.capture) with the new batch")
        return self.host

    def h2d_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.host_in.tensors())


class PipelinedProfiler:
    """Independent batches of one shape, software-pipelined on the device: `depth` CUDA graphs (each with its own static
    inputs, scratch and outputs) are replayed round-robin on `depth` streams, so that the latency-bound tails of batch n
    (the per-path time loop runs one warp per scheduler and uses ~6 % of the warp slots, the event replays a few threads)
    overlap the bandwidth-bound front of batch n+1 instead of leaving the GPU idle.  Every batch still runs every kernel.

    submit(new_db, consume): enqueue one batch -- copy `new_db` (None: the slot keeps its inputs; otherwise B, N_max and
    A_max must be the constructor's) into the slot's static inputs (every slot starts with its own copy of `db`), replay, then call consume(result) with the slot's stream current, so that whatever it enqueues (a copy of the
    summary rows, an export kernel, a device->host copy ...) is ordered before the slot is reused.  drain() joins all
    streams back into the caller's stream.  Capacity overflows are reported in the status / summary rows as usual
    (ST_CAPACITY); the caller redoes those batches through Engine.profile.
    """

    def __init__(self, eng: Engine, db: DeviceBatch, depth: int = 2, margin: float = 1.0):
        self.eng, self.depth = eng, max(1, int(depth))
        # every slot owns its static inputs: none aliases the caller's `db`, which submit(new_db) would overwrite
        self.graphs = [eng.capture(db.clone(), tiles=1, margin=margin) for _ in range(self.depth)]
        self.streams = [torch.cuda.Stream(device=eng.device) for _ in range(self.depth)]
        self.n = 0

    def submit(self, new_db: Optional[DeviceBatch] = None, consume=None) -> ProfileResult:
        k = self.n % self.depth
        g, st = self.graphs[k], self.streams[k]
        if new_db is not None:
            g.check_shape(new_db)
        st.wait_stream(torch.cuda.current_stream(self.eng.device))          # inputs prepared on the caller's stream
        with torch.cuda.stream(st):
            if new_db is not None:
                g.db.copy_(new_db)
            g.graph.replay()
            if consume is not None:
                consume(g.res)
        self.eng.launches += g.launches_per_run
        self.n += 1
        return g.res

    def drain(self) -> None:
        main = torch.cuda.current_stream(self.eng.device)
        for st in self.streams:
            main.wait_stream(st)
        self.n = 0

"""'Next' rows f1 + f2 of SURVEY.md section 8: what runs right after / right before the profiled path.

f1  trajectory export (gui_manager.py:220-230, 284-316): rows [0, t, x*12, -y*12, heading, v*12, omega] per time sample
    (built on the device, vap_export_rows), action rows [1, *action_values] spliced at nodes_map[i] + i and
    actions_map[i] + i, text written as f"{v} " per value -- the same formatting expression as the reference, so the
    text is identical for identical numbers.  trajectory_text builds one path's .txt body, save_text_batch every
    path's at once on the device (the command save_routes re-saves a folder of routes with it).
f2  node JSON codec (gui_manager.py:388-427, gui/path.py:590-644): [[x_in, y_in, start, end, reverse, stop, turn, wait,
    tangent, in_mag, out_mag, *actions], ...], [[x_in, y_in, t, stop, wait, *actions], ...] with the inch <-> pixel <->
    foot conversions of the GUI (145.308474301 in, 12.1090395251 ft per 2000 px).
"""
from __future__ import annotations

import ctypes as C
import json
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .engine import Engine, ProfileResult, _p
from .packing import PX_TO_FT

PX_TO_IN = 145.308474301          # gui/node.py:39-40


def export_rows(eng: Engine, res: ProfileResult):
    """Device-built numeric export rows for every path: returns (rows[sum_T, 7] tensor, offsets[B+1] tensor)."""
    B, T_cap = res.B, res.T_cap
    offsets = torch.zeros(B + 1, dtype=torch.int64, device=eng.device)
    total_cap = int(res.n_out.clamp(min=0).sum().item())
    rows = torch.empty((max(total_cap, 1), 7), dtype=torch.float64, device=eng.device)
    _lib.check(eng.lib.vap_export_rows(C.c_int64(B), C.c_int64(T_cap), C.c_int64(res.out.shape[1] * T_cap), _p(res.out),
                                       _p(res.n_out), _p(res.status), _p(offsets), _p(rows), eng._stream()),
               "vap_export_rows")
    eng.launches += 2
    return rows[:total_cap], offsets


def format_rows_device(eng: Engine, rows: torch.Tensor, int_time: Optional[torch.Tensor] = None):
    """Text of export rows on the device (repr(float)-exact, vap_format_rows + vap_compact_rows); int_time: the u8 row
    kinds of row_kinds() (bit 1 alone = "the time prints as the int 0").
    Returns (text uint8[total], row_offsets int64[R+1]); line r is text[row_offsets[r]:row_offsets[r+1]]."""
    R = rows.shape[0]
    slots, lens, offsets = _format_slots(eng, rows, int_time)
    total = int(offsets[R].item())
    text = torch.empty(max(total, 1), dtype=torch.uint8, device=eng.device)
    _lib.check(eng.lib.vap_compact_rows(C.c_int64(R), _p(slots), _p(lens), _p(offsets), _p(text), eng._stream()),
               "vap_compact_rows")
    eng.launches += 1
    return text[:total], offsets


def _format_slots(eng: Engine, rows: torch.Tensor, kinds: Optional[torch.Tensor]):
    """vap_format_rows: (slots[R, stride], lens[R], offsets[R+1] = exclusive scan of lens), nothing read back."""
    R = rows.shape[0]
    stride = int(eng.lib.vap_row_text_stride())
    slots = torch.empty((max(R, 1), stride), dtype=torch.uint8, device=eng.device)
    lens = torch.zeros(max(R, 1), dtype=torch.int32, device=eng.device)
    _lib.check(eng.lib.vap_format_rows(C.c_int64(R), _p(rows), _p(kinds), _p(slots), _p(lens), eng._stream()),
               "vap_format_rows")
    eng.launches += 1
    offsets = torch.zeros(R + 1, dtype=torch.int64, device=eng.device)
    torch.cumsum(lens[:R], dim=0, out=offsets[1:])                 # plumbing: exclusive scan of the line lengths
    return slots, lens, offsets


RK_TIME_INT, RK_INSERTED, RK_OMEGA_INT, RK_POS_INT = 1, 2, 4, 8


def row_kinds(eng: Engine, res: ProfileResult, db, offsets: Optional[torch.Tensor] = None, n_rows: Optional[int] = None):
    """Which entries of the reference's result lists are Python ints (vap_row_kinds): u8 bit set per result row --
    RK_TIME_INT times[r], RK_INSERTED linear_vels / accelerations, RK_OMEGA_INT angular_vels, RK_POS_INT positions.
    With `offsets` (from export_rows) the rows are the dense export rows, else a [B, T_cap] array."""
    B, T_cap = res.B, res.T_cap
    n = int(n_rows) if offsets is not None else B * T_cap
    kinds = torch.empty(max(n, 1), dtype=torch.uint8, device=eng.device)
    _lib.check(eng.lib.vap_row_kinds(C.c_int64(B), C.c_int(db.N_max), C.c_int(db.A_max), _p(db.node_attr), _p(db.n_nodes),
                                     _p(db.ap_attr), _p(db.n_ap), _p(db.cons), _p(res.status), C.c_double(eng.dt),
                                     _p(res.nodes_map), _p(res.actions_map), _p(res.n_maps), _p(res.n_out), C.c_int64(T_cap),
                                     _p(offsets), C.c_int64(n), _p(kinds), eng._stream()), "vap_row_kinds")
    eng.launches += 1
    return kinds if offsets is not None else kinds.view(B, T_cap)


def export_text_device(eng: Engine, res: ProfileResult, db=None):
    """Trajectory lines of every path of the batch, formatted on the device.
    Returns (text, row_offsets, path_row_offsets): path b owns rows path_row_offsets[b] .. path_row_offsets[b+1].
    db: the DeviceBatch the result was profiled from.  It tells which columns hold a Python int in the reference and
    print as "0" (times[0] without a prologue; v*12 and omega on inserted turn / wait rows,
    motion_profile_generator.py:425,448-453,500-515); None = plain paths without waits / turns (only times[0] is an int)."""
    rows, poff = export_rows(eng, res)
    R = rows.shape[0]
    if db is not None:
        kinds = row_kinds(eng, res, db, offsets=poff, n_rows=R)
    else:
        kinds = torch.zeros(max(R, 1), dtype=torch.uint8, device=eng.device)
        if R:
            kinds[poff[:-1][res.n_out.clamp(min=0) > 0]] = RK_TIME_INT
    text, roff = format_rows_device(eng, rows, kinds)
    return text, roff, poff


def format_doubles_device(eng: Engine, x: torch.Tensor) -> List[str]:
    """repr() of every element of a device fp64 tensor (test / utility entry point of the formatter)."""
    n = x.numel()
    out = torch.zeros((max(n, 1), 32), dtype=torch.uint8, device=eng.device)
    lens = torch.zeros(max(n, 1), dtype=torch.int32, device=eng.device)
    _lib.check(eng.lib.vap_format_doubles(C.c_int64(n), _p(x.contiguous()), _p(out), _p(lens), eng._stream()),
               "vap_format_doubles")
    eng.launches += 1
    o, l = out.cpu().numpy(), lens.cpu().numpy()
    return [bytes(o[i, : l[i]]).decode() for i in range(n)]


def _host_finish(out: torch.Tensor, flat_idx: Sequence[int], tokens: Sequence) -> None:
    """out.view(-1)[flat_idx[k]] = float(tokens[k]): the tokens the device left undecided, finished by Python."""
    if len(flat_idx):
        vals = torch.tensor([float(t) for t in tokens], dtype=torch.float64)
        out.view(-1)[torch.tensor(list(flat_idx), dtype=torch.int64).to(out.device)] = vals.to(out.device)


def parse_doubles_device(eng: Engine, strings: Sequence[str]):
    """float() of every string, parsed on the device (vap_parse_doubles): the inverse of format_doubles_device.
    Returns (x, flags): x fp64 device tensor, bit-equal to float(s) for every token of the grammar [-]digits[.digits]
    [e[+|-]digits], [-]inf, [-]nan; flags int8 host array: 0 parsed on the device, 1 finished on the host with float()
    (the device could not decide it), 2 not a token of the grammar (x is NaN)."""
    enc = [s.encode() for s in strings]
    n = len(enc)
    tok_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, enc), dtype=np.int64, count=n), out=tok_off[1:])
    text = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)
    text_d = torch.from_numpy(text.copy()).to(eng.device)
    off_d = torch.from_numpy(tok_off).to(eng.device)
    out = torch.empty(max(n, 1), dtype=torch.float64, device=eng.device)
    flags = torch.empty(max(n, 1), dtype=torch.int8, device=eng.device)
    _lib.check(eng.lib.vap_parse_doubles(C.c_int64(n), _p(text_d), _p(off_d), _p(out), _p(flags), eng._stream()),
               "vap_parse_doubles")
    eng.launches += 1
    fl = flags[:n].cpu().numpy()
    host = np.flatnonzero(fl == 1)
    _host_finish(out, host.tolist(), [strings[i] for i in host])
    return out[:n], fl


LINE_TRAJ, LINE_ACTION, LINE_OTHER = 0, 1, 2
LINE_ERRORS = {1: "blank line", 2: "the first token is neither 0 nor 1", 3: "a trajectory row without 7 tokens"}
ROW_COLUMNS = ("kind", "t", "x", "y", "heading", "v", "omega")


def line_error_text(code: int) -> str:
    """What a line error code of parse_text_batch means."""
    if code >= 4:
        c = code - 4
        return f"token {c + 1} ({ROW_COLUMNS[c] if c < 7 else '?'}) is not a number"
    return LINE_ERRORS.get(code, f"error {code}")


@dataclass
class ParsedText:
    """Bodies read back on the device (parse_text_batch).  Body b owns lines path_line_offsets[b] .. [b+1], trajectory
    rows row_offsets[b] .. [b+1] and action rows act_offsets[b] .. [b+1]; line l is text[line_offsets[l] ..
    line_offsets[l+1]).  All tensors are on the device."""
    text: torch.Tensor                # uint8[n_bytes], the uploaded bodies
    path_offsets: torch.Tensor        # int64[B+1]
    rows: torch.Tensor                # fp64[R, 7] {0, t, x, y, heading, v, omega} as written
    row_offsets: torch.Tensor         # int64[B+1]
    line_offsets: torch.Tensor        # int64[L+1]
    path_line_offsets: torch.Tensor   # int64[B+1]
    line_kinds: torch.Tensor          # uint8[L]: LINE_TRAJ, LINE_ACTION, LINE_OTHER
    line_errors: torch.Tensor         # int32[L]: 0, or a code line_error_text explains
    act_lines: torch.Tensor           # int64[A]: the line of every action row
    act_offsets: torch.Tensor         # int64[B+1]
    n_host: int                       # tokens finished on the host with float()


def _as_u8(text) -> np.ndarray:
    if isinstance(text, torch.Tensor):
        return text.numpy()
    if isinstance(text, (bytes, bytearray, memoryview)):
        return np.frombuffer(text, dtype=np.uint8)
    return np.asarray(text, dtype=np.uint8)


def _pinned_text(text) -> torch.Tensor:
    if isinstance(text, torch.Tensor) and text.is_pinned():
        return text
    a = _as_u8(text)
    t = torch.empty(max(a.size, 1), dtype=torch.uint8, pin_memory=True)
    t[:a.size].numpy()[:] = a
    return t[:a.size]


MAX_READ_BYTES = 2 ** 31 - 1     # bytes one parse_text_batch / compare_text_batch call reads: the line scan is int32


def _read_bodies(eng: Engine, text, path_offsets, parse_paths: int) -> ParsedText:
    """parse_text_batch, with the trajectory rows parsed for the first parse_paths bodies only (the lines, kinds,
    first-token errors and action rows of every body)."""
    poff = np.ascontiguousarray(path_offsets, dtype=np.int64)
    B, N = poff.shape[0] - 1, int(poff[-1])
    host = _pinned_text(text)
    if host.numel() < N or poff[0] != 0 or (np.diff(poff) < 0).any():
        raise ValueError("path_offsets must start at 0, never decrease and end within the text")
    if N > MAX_READ_BYTES:
        raise ValueError(f"{N} bytes: at most {MAX_READ_BYTES} bytes per call (tile the batch)")
    dev, st, L_ = eng.device, eng._stream(), eng.lib
    with eng._stage("read_upload"):
        text_d = host[:max(N, 1)].to(dev, non_blocking=True) if N else torch.zeros(1, dtype=torch.uint8, device=dev)
    poff_d = torch.from_numpy(poff).to(dev)
    with eng._stage("read_lines"):
        starts = torch.empty(max(N, 1), dtype=torch.uint8, device=dev)
        _lib.check(L_.vap_line_starts(C.c_int64(B), C.c_int64(N), _p(text_d), _p(poff_d), _p(starts), st), "vap_line_starts")
        scan = torch.cumsum(starts[:N], 0, dtype=torch.int32) if N else torch.zeros(1, dtype=torch.int32, device=dev)
        L = int(scan[-1].item()) if N else 0                               # read-back 1: the number of lines
        line_off = torch.empty(L + 1, dtype=torch.int64, device=dev)
        pl = torch.empty(B + 1, dtype=torch.int64, device=dev)
        _lib.check(L_.vap_line_offsets(C.c_int64(B), C.c_int64(N), _p(starts), _p(scan), _p(poff_d), _p(line_off), _p(pl), st),
                   "vap_line_offsets")
        del starts, scan
        Lc = max(L, 1)
        kinds = torch.empty(Lc, dtype=torch.uint8, device=dev)
        errors = torch.zeros(Lc, dtype=torch.int32, device=dev)
        counts = torch.empty(Lc, dtype=torch.int64, device=dev)
        _lib.check(L_.vap_line_kinds(C.c_int64(L), _p(text_d), _p(line_off), _p(kinds), _p(errors), _p(counts), st),
                   "vap_line_kinds")
        cscan = torch.cumsum(counts[:L], 0) if L else torch.zeros(1, dtype=torch.int64, device=dev)   # rows + 2^32 actions
        del counts
    with eng._stage("read_parse"):
        row_off = torch.empty(B + 1, dtype=torch.int64, device=dev)
        act_off = torch.empty(B + 1, dtype=torch.int64, device=dev)
        act_line = torch.empty(Lc, dtype=torch.int64, device=dev)
        rows = torch.empty((Lc, 7), dtype=torch.float64, device=dev)
        host_mask = torch.empty(Lc, dtype=torch.uint8, device=dev)
        _lib.check(L_.vap_parse_rows(C.c_int64(B), C.c_int64(L), _p(text_d), _p(line_off), _p(kinds), _p(cscan), _p(pl),
                                     C.c_int64(parse_paths), _p(row_off), _p(act_off), _p(act_line), _p(rows),
                                     _p(host_mask), _p(errors), st), "vap_parse_rows")
    eng.launches += 8
    flagged = host_mask[:L] != 0
    head = torch.stack([row_off[parse_paths], act_off[B], flagged.sum()]).cpu().tolist()   # read-back 2
    R, A, n_flag = head
    n_host = 0
    if n_flag:                                                              # read-back 3: the lines left for float()
        idx = torch.nonzero_static(flagged, size=n_flag).flatten()
        info = torch.stack([host_mask[idx].long(), line_off[idx], line_off[idx + 1], (cscan[idx] & 0xffffffff) - 1]).cpu().numpy()
        hb = host.numpy()
        flat, toks = [], []
        for mask, s, e, r in info.T:
            # the device's tokens: runs of ' ' separate them, '\n' ends the line; any other byte ('\t', '\r') is part
            # of a token, so bytes.split() would number the columns differently
            words = [w for w in bytes(hb[s:e]).rstrip(b"\n").split(b" ") if w]
            for c in range(1, 7):
                if mask >> c & 1:
                    flat.append(int(r) * 7 + c)
                    toks.append(words[c])
        _host_finish(rows, flat, toks)
        n_host = len(flat)
    return ParsedText(text_d, poff_d, rows[:R], row_off, line_off, pl, kinds[:L], errors[:L], act_line[:A], act_off, n_host)


def parse_text_batch(eng: Engine, text, path_offsets) -> ParsedText:
    """Read saved .txt bodies back on the device: text holds B bodies back to back (bytes, a uint8 array, or a pinned
    uint8 CPU tensor), body b is text[path_offsets[b] .. path_offsets[b+1]).  Returns a ParsedText: the trajectory rows
    [R, 7] as written (bit-equal to float() of every token), per-body row, line and action-row offsets, line kinds and
    per-line errors; tokens the device could not decide are already finished with float() (their count: n_host).
    The text goes to the device in one copy from pinned memory; the call reads back from the device at most three
    times, whatever B is."""
    return _read_bodies(eng, text, path_offsets, len(path_offsets) - 1)


CMP_I = ("diff_byte", "diff_line", "old_rows", "new_rows", "action_rows_differ", "error_line", "error_code")
CMP_F = ("old_t", "new_t", "max_dt", "max_dx", "max_dy", "max_dheading", "max_dv", "max_domega")


def compare_text_batch(eng: Engine, old_text, old_offsets, new_text, new_offsets, new_rows: torch.Tensor,
                       new_row_offsets: torch.Tensor):
    """Saved bodies against fresh ones, path by path, on the device (vap_compare_bodies).  old_text / old_offsets: the
    saved bodies as parse_text_batch takes them (old_text may be a pinned tensor with room for the fresh text behind
    old_offsets[-1]: the fresh text then goes there and both travel in one copy); new_text / new_offsets: the fresh
    bodies (save_text_batch); new_rows / new_row_offsets: their numeric rows (export_rows).
    Returns (ints int64[B, 7] named by CMP_I, floats fp64[B, 8] named by CMP_F, n_host), host arrays: first differing
    byte (-1 equal) and its line in the saved body, saved and fresh row counts, differing action rows, first saved line
    with an error and its code (line_error_text), last saved and fresh t, max |saved - fresh| of t, x, y, heading, v,
    omega over the common rows (as written: inches and inch/s)."""
    oo = np.ascontiguousarray(old_offsets, dtype=np.int64)
    no = np.ascontiguousarray(new_offsets, dtype=np.int64)
    B, n_old, n_new = oo.shape[0] - 1, int(oo[-1]), int(no[-1])
    if no.shape[0] != B + 1:
        raise ValueError(f"{B} saved bodies but {no.shape[0] - 1} fresh ones")
    if isinstance(old_text, torch.Tensor) and old_text.is_pinned() and old_text.numel() >= n_old + n_new:
        buf = old_text
    else:
        buf = torch.empty(max(n_old + n_new, 1), dtype=torch.uint8, pin_memory=True)
        buf[:n_old].numpy()[:] = _as_u8(old_text)[:n_old]
    buf[n_old:n_old + n_new].numpy()[:] = _as_u8(new_text)[:n_new]
    poff = np.concatenate([oo, n_old + no[1:]])
    p = _read_bodies(eng, buf[:n_old + n_new], poff, B)
    out_i = torch.empty((max(B, 1), len(CMP_I)), dtype=torch.int64, device=eng.device)
    out_f = torch.empty((max(B, 1), len(CMP_F)), dtype=torch.float64, device=eng.device)
    with eng._stage("read_compare"):
        _lib.check(eng.lib.vap_compare_bodies(C.c_int64(B), _p(p.text), _p(p.path_offsets), _p(p.path_offsets[B:]),
                                              _p(p.line_offsets), _p(p.line_errors), _p(p.path_line_offsets), _p(p.act_lines),
                                              _p(p.act_offsets), _p(p.act_offsets[B:]), _p(p.rows), _p(p.row_offsets),
                                              _p(new_rows), _p(new_row_offsets), _p(out_i), _p(out_f), eng._stream()),
                   "vap_compare_bodies")
    eng.launches += 1
    return out_i[:B].cpu().numpy(), out_f[:B].cpu().numpy(), p.n_host                # read-back 4


FP_I = ("rows", "first_row", "first_kind", "violating_rows", "worst_wall_row", "nearest_box_row", "nearest_box")
FP_F = ("first_t", "worst_wall_in", "worst_wall_t", "nearest_box_in", "nearest_box_t", "max_corner_step_in")
FP_KIND_WALL, FP_KIND_NONFINITE, FP_KIND_BOX = 0, 1, 2
FP_MAX_BOXES = 64


def default_field():
    """(xmin, xmax, ymin, ymax) in inches: the GUI's 2000-px canvas, which it clamps nodes into."""
    lo, hi = px_to_in(0), px_to_in(2000)
    return lo, hi, lo, hi


def footprint_check(eng: Engine, rows, row_offsets, length_in: float, width_in: float, field=None, keep_out=(),
                    tol_in: float = 0.0):
    """Does a robot length_in long (along the heading) and width_in wide, centred on every export row, stay on the field
    and clear the keep-out boxes?  Per path, on the device (vap_footprint_check).
    rows / row_offsets: rows[R, 7] fp64 {0, t, x, y, heading, v, omega} in the .txt frame (inches, heading CCW from +x)
    and int64[B+1] offsets, path b owning rows row_offsets[b] .. [b+1] -- export_rows(eng, res) gives them for fresh
    profiles, parse_text_batch(...).rows / .row_offsets for saved files.  field: (xmin, xmax, ymin, ymax) in inches,
    None = default_field(); keep_out: up to 64 boxes (x0, y0, x1, y1) in inches in the same frame; tol_in: overhangs
    and penetrations up to tol_in inches do not count.
    Returns (ints int64[B, 7] named by FP_I, floats fp64[B, 6] named by FP_F), host arrays, with one read-back:
    rows, first violating row (-1 none) and its kind (-1, FP_KIND_WALL, FP_KIND_NONFINITE, FP_KIND_BOX + k for box k),
    violating rows, row of the largest wall margin, row and index of the nearest box; t of the first violation, largest
    wall margin (positive: overhang, negative: clearance) and its t, nearest box distance (negative: penetration
    depth; +inf without boxes) and its t, and the largest corner displacement between consecutive rows (the sampling
    resolution: an excursion shorter than this between two rows is not seen).  Rows count from 0 within the path.
    Raises VapError for a non-positive size, an empty field or box, or more than 64 boxes."""
    rows = torch.as_tensor(rows, dtype=torch.float64, device=eng.device).contiguous()
    roff = torch.as_tensor(row_offsets, dtype=torch.int64, device=eng.device).contiguous()
    B = roff.shape[0] - 1
    xmin, xmax, ymin, ymax = default_field() if field is None else (float(v) for v in field)
    boxes = np.ascontiguousarray(np.asarray(keep_out, dtype=np.float64).reshape(-1, 4))
    K = boxes.shape[0]
    buf = torch.empty(max(B, 1) * (len(FP_I) + len(FP_F)), dtype=torch.int64, device=eng.device)
    out_f = buf[max(B, 1) * len(FP_I):].view(torch.float64)
    _lib.check(eng.lib.vap_footprint_check(C.c_int64(B), _p(rows), _p(roff), C.c_double(length_in / 2),
                                           C.c_double(width_in / 2), C.c_double(xmin), C.c_double(xmax), C.c_double(ymin),
                                           C.c_double(ymax), C.c_int(K), boxes.ctypes.data_as(C.c_void_p),
                                           C.c_double(tol_in), _p(buf), _p(out_f), eng._stream()), "vap_footprint_check")
    eng.launches += 1
    host = buf.cpu().numpy()                                                             # the one read-back
    n_i = max(B, 1) * len(FP_I)
    return host[:n_i].reshape(-1, len(FP_I))[:B], host[n_i:].view(np.float64).reshape(-1, len(FP_F))[:B]


PC_I = ("status", "events", "first_side", "first_row", "contacts", "nearest_side", "nearest_row")
PC_F = ("first_t", "nearest_in", "nearest_t", "last_t_a", "last_t_b", "max_corner_step_in")
PC_OK, PC_A_INVALID, PC_B_INVALID, PC_BAD_INDEX = 0, 1, 2, 3                 # status
PC_BAD_NONE, PC_BAD_EMPTY, PC_BAD_NONFINITE, PC_BAD_DECREASING = 0, 1, 2, 3  # reason of bad[b] = (row, reason)


def pair_reason_text(row: int, reason: int) -> str:
    """What bad[b] = (row, reason) of pair_check says about a route."""
    if reason == PC_BAD_EMPTY:
        return "no trajectory rows"
    if reason == PC_BAD_NONFINITE:
        return f"row {row} is not finite"
    if reason == PC_BAD_DECREASING:
        return f"t decreases at row {row}"
    return "valid" if reason == PC_BAD_NONE else f"reason {reason}"


def _pose_planes(eng: Engine, rows, roff: torch.Tensor, bad: torch.Tensor):
    """vap_pose_planes: planes fp64[5 * R] of rows, bad[b] = (row, reason) written into bad (int64[B, 2])."""
    rows = torch.as_tensor(rows, dtype=torch.float64, device=eng.device).reshape(-1, 7).contiguous()
    R = int(rows.shape[0])
    planes = torch.empty(5 * max(R, 1), dtype=torch.float64, device=eng.device)
    _lib.check(eng.lib.vap_pose_planes(C.c_int64(roff.shape[0] - 1), _p(rows), _p(roff), C.c_int64(R), _p(planes), _p(bad),
                                       eng._stream()), "vap_pose_planes")
    eng.launches += 1
    return planes, R


def pair_check(eng: Engine, rows_a, off_a, size_a, rows_b, off_b, size_b, pairs, min_gap_in: float = 0.0):
    """Two robots driving two routes at the same time: where do their rectangles first come closer than min_gap_in?
    On the device (vap_pose_planes, vap_pair_check).
    rows_a / off_a: row set A, rows[R, 7] fp64 {0, t, x, y, heading, v, omega} in the .txt frame (inches, heading CCW
    from +x) and int64[B_a+1] offsets -- export_rows(eng, res) for fresh profiles, parse_text_batch(...).rows /
    .row_offsets for saved files; rows_b / off_b likewise.  When rows_b is rows_a and off_b is off_a (one route set on
    both sides) the planes and the per-route checks are built once; other offsets into the same rows get their own,
    since whether t decreases depends on where each route begins.  size_a, size_b: (length_in, width_in) of each
    robot, length along the heading.  pairs: int64[P, 2] of (route of A, route of B).
    Every row of either route is an event; at it the other robot holds its last row with t <= the event's t (its first
    row before it starts, its last row once it has finished).  An event is a contact when the signed distance of the
    rectangles (negative: penetration depth) is < min_gap_in; events are ordered by (t, side, row), side A = 0.
    Returns host arrays (ints int64[P, 7] named by PC_I, floats fp64[P, 6] named by PC_F, bad_a int64[B_a, 2],
    bad_b int64[B_b, 2]) with one read-back: per pair the status (PC_OK, PC_A_INVALID, PC_B_INVALID, PC_BAD_INDEX),
    events, first contact's side and row (-1 none) and t (NaN), contact events, the nearest event's side, row, distance
    and t, both routes' last t, and the largest corner move between consecutive rows of either route (the check's
    resolution); per route (row, reason) of its first invalid row (pair_reason_text explains it).
    Raises VapError for a size that is not positive and finite or a min_gap_in that is not finite."""
    (la, wa), (lb, wb) = ((float(v) for v in size_a), (float(v) for v in size_b))
    same = rows_b is rows_a and off_b is off_a
    roff_a = torch.as_tensor(off_a, dtype=torch.int64, device=eng.device).contiguous()
    roff_b = roff_a if same else torch.as_tensor(off_b, dtype=torch.int64, device=eng.device).contiguous()
    B_a, B_b = roff_a.shape[0] - 1, roff_b.shape[0] - 1
    pr = torch.from_numpy(np.ascontiguousarray(np.asarray(pairs, dtype=np.int64).reshape(-1, 2))).to(eng.device)
    P = int(pr.shape[0])
    n_i, n_f, n_a = max(P, 1) * len(PC_I), max(P, 1) * len(PC_F), 2 * max(B_a, 1)
    buf = torch.empty(n_i + n_f + n_a + 2 * max(B_b, 1), dtype=torch.int64, device=eng.device)
    out_f = buf[n_i:n_i + n_f].view(torch.float64)
    bad_a, bad_b = buf[n_i + n_f:n_i + n_f + n_a], buf[n_i + n_f + n_a:]
    pa, R_a = _pose_planes(eng, rows_a, roff_a, bad_a)
    pb, R_b = (pa, R_a) if same else _pose_planes(eng, rows_b, roff_b, bad_b)
    _lib.check(eng.lib.vap_pair_check(
        C.c_int64(P), _p(pr), C.c_int64(B_a), _p(pa), C.c_int64(R_a), _p(roff_a), _p(bad_a), C.c_double(la / 2),
        C.c_double(wa / 2), C.c_int64(B_b), _p(pb), C.c_int64(R_b), _p(roff_b), _p(bad_a if same else bad_b),
        C.c_double(lb / 2), C.c_double(wb / 2), C.c_double(min_gap_in), _p(buf), _p(out_f), eng._stream()),
        "vap_pair_check")
    eng.launches += 1
    host = buf.cpu().numpy()                                                             # the one read-back
    o = n_i + n_f
    ha = host[o:o + 2 * B_a].reshape(-1, 2)
    hb = ha if same else host[o + n_a:o + n_a + 2 * B_b].reshape(-1, 2)
    return host[:n_i].reshape(-1, len(PC_I))[:P], host[n_i:o].view(np.float64).reshape(-1, len(PC_F))[:P], ha, hb


def splice_action_rows(traj_rows: Sequence[Sequence[float]], nodes_map: Sequence[int], node_actions: Sequence[Sequence],
                       actions_map: Sequence[int] = (), action_rows: Sequence[Sequence] = ()) -> List[list]:
    """gui_manager.py:284-310: trajectory rows with the node / action-point rows inserted at map[i] + i."""
    data = [[0] + [v for v in r[1:]] for r in traj_rows]
    for i in range(len(nodes_map)):
        data.insert(int(nodes_map[i] / 1) + i, [1] + list(node_actions[i]))
    for i in range(len(actions_map)):
        data.insert(int(actions_map[i] / 1) + i, [1] + list(action_rows[i]))
    return data


def format_rows(nodes_data: Sequence[Sequence]) -> str:
    """fill_txt_file (gui_manager.py:220-230): every value followed by a blank, one row per line."""
    res = ""
    for data in nodes_data:
        for v in data:
            res += f"{v} "
        res += "\n"
    return res


def trajectory_text(eng: Engine, res: ProfileResult, b: int, node_actions: Sequence[Sequence],
                    action_rows: Sequence[Sequence] = (), db=None, device_text=None) -> str:
    """The .txt body the reference writes for path b (nodes_map includes the trailing len(times), gui/path.py:342).
    The trajectory lines come from the device formatter; only the handful of action rows is formatted and spliced here.
    device_text: result of export_text_device (reuse it when writing many paths of one batch)."""
    text, roff, poff = device_text if device_text is not None else export_text_device(eng, res, db)
    r0, r1 = int(poff[b]), int(poff[b + 1])
    lines = bytes(text[int(roff[r0]): int(roff[r1])].cpu().numpy()).decode().splitlines(keepends=True)
    nm = res.nodes_map[b, : int(res.n_maps[b, 0])].cpu().numpy()
    am = res.actions_map[b, : int(res.n_maps[b, 1])].cpu().numpy()
    for i in range(len(nm)):
        lines.insert(int(nm[i] / 1) + i, format_rows([[1] + list(node_actions[i])]))
    for i in range(len(am)):
        lines.insert(int(am[i] / 1) + i, format_rows([[1] + list(action_rows[i])]))
    return "".join(lines)


_CACHED_TYPES = (int, bool, str)      # f"{v}" of these depends on the value alone (unlike 0.0 == -0.0, 1 == 1.0 == True)


def pack_action_rows(node_actions: Sequence[Sequence[Sequence]], ap_actions: Sequence[Sequence[Sequence]]):
    """Text of every action row [1, *action_values] of a batch as format_rows writes it, laid out for vap_splice_plan.
    node_actions[b][i] / ap_actions[b][j]: the action_values of path b's nodes / action points.
    Returns (text uint8[n], act_off int64[rows+1], act_first int64[B], act_rows int32[B, 2]); the rows of path b start at
    act_first[b], its node rows first.  A row of plain ints / bools / strings is formatted once per batch."""
    B = len(node_actions)
    if len(ap_actions) != B:
        raise ValueError(f"node_actions has {B} paths, ap_actions {len(ap_actions)}")
    cache, pieces = {}, []
    act_rows = np.zeros((B, 2), dtype=np.int32)
    for b in range(B):
        na, aa = node_actions[b], ap_actions[b]
        act_rows[b] = len(na), len(aa)
        for v in (*na, *aa):
            vals = tuple(v)
            try:
                key = (tuple(map(type, vals)), vals)
                s = cache.get(key)
            except TypeError:                              # unhashable values: format every time
                key, s = None, None
            if s is None:
                s = format_rows([(1, *vals)]).encode()
                if key is not None and all(t in _CACHED_TYPES for t in key[0]):
                    cache[key] = s
            pieces.append(s)
    act_off = np.zeros(len(pieces) + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, pieces), dtype=np.int64, count=len(pieces)), out=act_off[1:])
    act_first = np.zeros(B, dtype=np.int64)
    np.cumsum(act_rows.sum(axis=1, dtype=np.int64)[:-1], out=act_first[1:])
    return np.frombuffer(bytearray(b"".join(pieces)), dtype=np.uint8), act_off, act_first, act_rows


def splice_bodies(eng: Engine, slots: torch.Tensor, lens: torch.Tensor, line_off: torch.Tensor, row_off: torch.Tensor,
                  status: torch.Tensor, nodes_map: torch.Tensor, actions_map: torch.Tensor, n_maps: torch.Tensor,
                  node_actions: Sequence[Sequence[Sequence]], ap_actions: Sequence[Sequence[Sequence]]):
    """The .txt bodies of B paths from their formatted trajectory lines (vap_format_rows: slots, lens, line_off = exclusive
    scan of lens; path b owns lines row_off[b] .. row_off[b+1]) and the maps of the time stage: vap_splice_plan,
    vap_compact_rows onto the gapped line positions, vap_splice_actions, one copy to pinned host memory.
    Returns (text uint8[total] host, path_offsets int64[B+1] host, ok bool[B] host).  Raises ValueError when a path's maps
    need more action rows than node_actions / ap_actions give it."""
    B, R = status.shape[0], line_off.shape[0] - 1
    dev = eng.device
    text_h, act_off_h, act_first_h, act_rows_h = pack_action_rows(node_actions, ap_actions)
    n_act = act_off_h.shape[0] - 1

    def up(a):
        return torch.from_numpy(a if a.size else np.zeros(1, dtype=a.dtype)).to(dev, non_blocking=True)
    act_text, act_off, act_first, act_rows = up(text_h), up(act_off_h), up(act_first_h), up(act_rows_h)
    path_off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    line_dst = torch.empty(max(R, 1), dtype=torch.int64, device=dev)
    act_dst = torch.empty(max(n_act, 1), dtype=torch.int64, device=dev)
    flags = torch.zeros(max(B, 1), dtype=torch.int32, device=dev)
    N_max, A_stride = nodes_map.shape[1] - 1, actions_map.shape[1]
    with eng._stage("text_splice_plan"):
        _lib.check(eng.lib.vap_splice_plan(C.c_int64(B), C.c_int(N_max), C.c_int(A_stride), _p(status), _p(nodes_map),
                                           _p(actions_map), _p(n_maps), _p(row_off), _p(line_off), _p(act_first),
                                           _p(act_rows), C.c_int64(n_act), _p(act_off), _p(path_off), _p(line_dst),
                                           _p(act_dst), _p(flags), eng._stream()), "vap_splice_plan")
    eng.launches += 2
    flags = flags[:B]
    head = torch.stack([path_off[B], (flags == 2).sum()]).cpu()          # the one read-back: size of the text
    if int(head[1]):
        bad = torch.nonzero(flags == 2).flatten()[:8].tolist()
        raise ValueError(f"{int(head[1])} path(s) need more action rows than were passed (first: {bad}); node_actions[b] "
                         "must cover n_maps[b, 0] rows and ap_actions[b] n_maps[b, 1]")
    total = int(head[0])
    text = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
    with eng._stage("text_splice_copy"):
        _lib.check(eng.lib.vap_compact_rows(C.c_int64(R), _p(slots), _p(lens), _p(line_dst), _p(text), eng._stream()),
                   "vap_compact_rows")
        _lib.check(eng.lib.vap_splice_actions(C.c_int64(n_act), _p(act_text), _p(act_off), _p(act_dst), _p(text),
                                              eng._stream()), "vap_splice_actions")
    eng.launches += 2
    host = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=True)
    offs = torch.empty(B + 1, dtype=torch.int64, pin_memory=True)
    ok = torch.empty(max(B, 1), dtype=torch.bool, pin_memory=True)
    with eng._stage("text_d2h"):
        host.copy_(text, non_blocking=True)
    offs.copy_(path_off, non_blocking=True)
    ok[:B].copy_(flags == 0, non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    return host.numpy()[:total], offs.numpy(), ok.numpy()[:B]


def save_text_batch(eng: Engine, res: ProfileResult, db, node_actions: Sequence[Sequence[Sequence]],
                    ap_actions: Sequence[Sequence[Sequence]]):
    """The .txt body save_nodes_to_file writes (gui_manager.py:232-316) for every path of a batch, assembled on the device.
    node_actions[b][i] / ap_actions[b][j]: the action_values of path b's nodes (widget list order) and action points, as
    trajectory_text takes them for one path.  db: the DeviceBatch res was profiled from.
    Returns (text, path_offsets, ok), all on the host: path b's body is text[path_offsets[b]:path_offsets[b+1]] (bytes,
    equal to trajectory_text's for that path); ok[b] is False for a path with status != 0, whose body is empty.
    Reads back from the device a fixed number of times, whatever B is.  Raises ValueError when a path's maps need more
    action rows than were passed (the reference raises IndexError there)."""
    if len(node_actions) != res.B or len(ap_actions) != res.B:
        raise ValueError(f"{res.B} paths, but {len(node_actions)} node_actions and {len(ap_actions)} ap_actions")
    with eng._stage("text_format"):
        rows, poff = export_rows(eng, res)
        kinds = row_kinds(eng, res, db, offsets=poff, n_rows=rows.shape[0])
        slots, lens, line_off = _format_slots(eng, rows, kinds)
    return splice_bodies(eng, slots, lens, line_off, poff, res.status, res.nodes_map, res.actions_map, res.n_maps,
                         node_actions, ap_actions)


ROUTES_DECL = "std::vector<std::vector<double>> "
ROUTES_SKELETON = ("#ifndef ROUTES_H\n", "#define ROUTES_H\n", "#include <vector>\n", "\n", None, "\n", "#endif\n")


def routes_header_entry(name: str, nodes_data: Sequence[Sequence]) -> str:
    """The one-line C++ initialiser the legacy routes.h export holds per route (fill_template, gui_manager.py:442-454):
    rows of more than two values as "{a, b, c}", shorter rows as "{row[0], row[1]}", values printed like f"{v}"."""
    rows = []
    for row in nodes_data:
        vals = row if len(row) > 2 else (row[0], row[1])
        rows.append("{" + ", ".join(f"{v}" for v in vals) + "}")
    return f"{ROUTES_DECL}{name} = {{{', '.join(rows)}}};\n"


def update_routes_header(lines: Optional[Sequence[str]], name: str, nodes_data: Sequence[Sequence]) -> List[str]:
    """New content of routes.h (gui_manager.py:456-500).  lines: the current file as readlines() gives it, None when
    the file does not exist, empty when it is empty.  An existing declaration of `name` is replaced in place; otherwise
    the entry goes in front of the "#endif" line (and, like the reference, nowhere if there is none); a missing or
    empty file becomes the include-guard skeleton around the entry."""
    entry = routes_header_entry(name, nodes_data)
    if not lines:
        return [entry if x is None else x for x in ROUTES_SKELETON]
    out = list(lines)
    head = f"{ROUTES_DECL}{name} ="
    for i, line in enumerate(out):
        if line.strip().startswith(head):
            out[i] = entry
            return out
    for i, line in enumerate(out):
        if line.strip() == "#endif":
            out.insert(i, entry)
            break
    return out


def write_routes_header(path: str, name: str, nodes_data: Sequence[Sequence]) -> None:
    """fill_template's file handling: read, update, write back (a zero-length file counts as missing, :488-491)."""
    import os
    lines = None
    if os.path.exists(path) and os.stat(path).st_size > 0:
        with open(path, "r") as f:
            lines = f.readlines()
    with open(path, "w") as f:
        f.writelines(update_routes_header(lines, name, nodes_data))


# ---------------------------------------------------------------------------------------------------- f2: JSON codec
def px_to_in(px: float) -> float:
    return ((px / 2000) - 0.5) * PX_TO_IN          # Node.get_abs_x (gui/node.py:53-55)


def in_to_px(v: float) -> float:
    return (v / PX_TO_IN + 0.5) * 2000             # PathWidget.convert_point (gui/path.py:590-594)


def nodes_to_json(points_px, nodes, action_points=(), action_points_px=(), as_list: bool = False):
    """convert_nodes (gui_manager.py:388-427).  Node objects are duck-typed (attributes of gui/node.py)."""
    nodes_data = []
    for (x, y), nd in zip(points_px, nodes):
        tan = getattr(nd, "tangent", None)
        nodes_data.append([px_to_in(x), px_to_in(y), int(getattr(nd, "is_start_node", False)),
                           int(getattr(nd, "is_end_node", False)), int(nd.is_reverse_node), int(nd.stop), nd.turn,
                           nd.wait_time, None if tan is None else [float(tan[0]), float(tan[1])],
                           nd.incoming_magnitude, nd.outgoing_magnitude] + list(getattr(nd, "action_values", [])))
    action_data = []
    for (x, y), ap in zip(action_points_px, action_points):
        action_data.append([px_to_in(x), px_to_in(y), ap.t, int(ap.stop), ap.wait_time]
                           + list(getattr(ap, "action_values", [])))
    if as_list:
        return [nodes_data, action_data]
    return json.dumps([nodes_data, action_data], separators=(",", ":"))


class RouteNode:
    """Plain stand-in for gui.node.Node with the attributes the hot path reads."""

    def __init__(self):
        self.is_start_node = False; self.is_end_node = False; self.is_reverse_node = False; self.stop = False
        self.turn = 0; self.wait_time = 0; self.tangent = None; self.incoming_magnitude = None
        self.outgoing_magnitude = None; self.max_velocity = 0; self.max_acceleration = 0; self.action_values = []
        self.px = None


class RouteActionPoint:
    def __init__(self, t):
        self.t = t; self.stop = False; self.wait_time = 0; self.max_velocity = 0; self.max_acceleration = 0
        self.action_values = []; self.px = None


def load_nodes(node_str: str):
    """load_nodes (gui/path.py:602-644) without Qt: returns (points_px[N,2], nodes, action_points, action_px[A,2]).

    `nodes` is the widget's node LIST, built with add_node's insertion rule (path.py:439-446: once an end node exists,
    every further node goes in front of the last list element); `points_px` is the point order
    _execute_update_path hands to build_path together with that list (path.py:403-413: the start node, every node that
    is flagged neither start nor end, the end node) -- empty unless a start node, an end node and two nodes exist.
    Each node also carries its own pixel position as `.px`.  Action points are kept sorted by t (path.py:459-471)."""
    data = json.loads(node_str)
    nodes_data, action_data = (data[0], data[1]) if len(data) == 2 else (data, [])
    nodes, start_node, end_node = [], None, None
    for nd in nodes_data:
        if len(nd) > 4:
            n = RouteNode()
            n.px = [in_to_px(nd[0]), in_to_px(nd[1])]
            if end_node is not None:
                nodes.insert(len(nodes) - 1, n)
            else:
                nodes.append(n)
            start_node = n if bool(nd[2]) else start_node
            n.is_start_node = bool(nd[2])
            end_node = n if bool(nd[3]) else end_node
            n.is_end_node = bool(nd[3])
            n.is_reverse_node, n.stop = bool(nd[4]), bool(nd[5])
            n.turn, n.wait_time = nd[6], nd[7]
            n.tangent = None if nd[8] is None else np.array(nd[8])
            n.incoming_magnitude, n.outgoing_magnitude = nd[9], nd[10]
            n.action_values = list(nd[11:])
    aps = []
    for ad in action_data:
        a = RouteActionPoint(ad[2])
        a.px = [in_to_px(ad[0]), in_to_px(ad[1])]
        a.stop, a.wait_time = ad[3], ad[4]
        a.action_values = list(ad[5:])
        k = next((i for i, o in enumerate(aps) if o.t > a.t), len(aps))
        aps.insert(k, a)
    pts = []
    if start_node is not None and end_node is not None and len(nodes) > 1:
        pts = [start_node.px] + [n.px for n in nodes if not (n.is_end_node or n.is_start_node)] + [end_node.px]
    return (np.array(pts, dtype=np.float64).reshape(-1, 2), nodes, aps,
            np.array([a.px for a in aps], dtype=np.float64).reshape(-1, 2))


def px_points_to_ft(points_px) -> np.ndarray:
    """PathWidget.update_spline (gui/path.py:365-367)."""
    p = np.asarray(points_px, dtype=np.float64)
    return (p / 2000 - 0.5) * PX_TO_FT

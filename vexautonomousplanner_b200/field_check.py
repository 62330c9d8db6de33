"""python -m vexautonomousplanner_b200.field_check DIR [options]

Checks on the device that a robot's rectangular footprint stays on the field and clear of keep-out boxes for the whole
run of every route of a folder (export.footprint_check).  The GUI's robot preview shows the footprint at one point at a
time; the corners of a robot turning in place at a node near a wall can leave the field while the path's centre line
stays inside.

DIR is a routes folder (node-JSON *.txt, the GUI's routes folder): the routes are read, packed and profiled as
save_routes does (the same --config and constraint flags, --tile-paths).  With --trajectories, DIR holds saved
trajectory .txt files (what save_routes writes), read back on the device with export.parse_text_batch.

All coordinates are inches in the trajectory .txt frame: x as in the GUI, y = -12 * y_ft (the GUI's y axis flipped),
heading counter-clockwise from +x.  The field defaults to the GUI's 2000-px canvas (+-72.654 in on both axes).

One line per file:
  clear: NAME: wall clearance C in at t T s; nearest keep-out box k at D in, t T s; sampling step <= S in
  hits: NAME: first at t T s (row r): wall | keep-out box k | non-finite row; worst wall overhang W in at t T s;
        nearest keep-out box k at D in, t T s (a negative D is a penetration depth); N of M rows
  unreadable: NAME: line L: reason
  not checked: NAME: reason
and a final count.  Rows count from 0 within the route's trajectory rows.  The sampling step is the largest move of a
corner between consecutive rows: the check sees the footprint at the rows only, so an excursion shorter than that
between two rows can be missed.  Exit status 0 only when every file is clear, 1 otherwise, 2 for argument errors.
"""
from __future__ import annotations

import argparse
import math
import os
import sys
from typing import List, Optional, Sequence, Tuple

from .save_routes import STATUS_NAMES, add_constraint_flags, byte_groups, constraints, read_routes


def read_robot_size(path: str) -> Tuple[Optional[float], Optional[float]]:
    """(robot.length, robot.width) of a config.yaml in the GUI's layout, None where a key is missing.  Taken in
    inches, like robot.track_width."""
    import yaml
    with open(path) as f:
        cfg = yaml.safe_load(f) or {}
    robot = cfg.get("robot") or {}
    return tuple(None if robot.get(k) is None else float(robot[k]) for k in ("length", "width"))


def keep_out_box(text: str) -> Tuple[float, float, float, float]:
    """argparse type of --keep-out: "X0,Y0,X1,Y1" with X0 < X1 and Y0 < Y1, all finite."""
    parts = text.split(",")
    try:
        box = tuple(float(v) for v in parts)
    except ValueError:
        box = ()
    if len(box) != 4 or not all(math.isfinite(v) for v in box):
        raise argparse.ArgumentTypeError(f"{text!r} is not X0,Y0,X1,Y1 (four finite numbers, inches)")
    if not (box[0] < box[2] and box[1] < box[3]):
        raise argparse.ArgumentTypeError(f"{text!r} is empty: X0 < X1 and Y0 < Y1 required")
    return box


def parse_args(argv: Optional[List[str]] = None) -> argparse.Namespace:
    from .export import FP_MAX_BOXES
    p = argparse.ArgumentParser(prog="python -m vexautonomousplanner_b200.field_check",
                                description="Check that the robot's footprint stays on the field and clear of keep-out "
                                            "boxes along every route of a folder.")
    p.add_argument("dir", help="folder of node-JSON routes (*.txt), or with --trajectories of saved trajectory .txt files")
    p.add_argument("--trajectories", action="store_true", help="DIR holds saved trajectory .txt files, not routes")
    p.add_argument("--config", help="config.yaml in the GUI's layout: motion.*, robot.track_width, and robot.length / "
                                    "robot.width for the footprint")
    add_constraint_flags(p)
    p.add_argument("--robot-length-in", type=float, dest="length_in",
                   help="robot length along its heading, inches (default: robot.length of --config, read as inches like "
                        "robot.track_width -- an assumption: the GUI's config does not state that unit)")
    p.add_argument("--robot-width-in", type=float, dest="width_in",
                   help="robot width across its heading, inches (default: robot.width of --config, read as inches)")
    p.add_argument("--field-half-in", type=float, dest="field_half_in",
                   help="the field is -H .. H inches on both axes (default: the GUI's canvas, +-72.654 in)")
    p.add_argument("--keep-out", type=keep_out_box, action="append", default=[], metavar="X0,Y0,X1,Y1",
                   help="an axis-aligned keep-out box in inches in the trajectory .txt frame (y = -12 * y_ft); repeatable; "
                        "write --keep-out=X0,... when X0 is negative")
    p.add_argument("--tolerance-in", type=float, default=0.0, dest="tol_in",
                   help="overhangs and penetrations up to this many inches do not count (default 0)")
    p.add_argument("--tile-paths", type=int, default=8192, help="routes profiled per batch (default 8192)")
    p.add_argument("--device", default="cuda:0")
    args = p.parse_args(argv)
    if args.tile_paths < 1:
        p.error("--tile-paths must be at least 1")
    if len(args.keep_out) > FP_MAX_BOXES:
        p.error(f"at most {FP_MAX_BOXES} --keep-out boxes")
    if args.field_half_in is not None and not (args.field_half_in > 0 and math.isfinite(args.field_half_in)):
        p.error("--field-half-in must be positive")
    if not math.isfinite(args.tol_in):
        p.error("--tolerance-in must be finite")
    return args


def robot_size(args: argparse.Namespace) -> Optional[Tuple[float, float]]:
    """(length, width) in inches from the flags, else from --config; None when either is unknown or not positive."""
    length, width = args.length_in, args.width_in
    if args.config and (length is None or width is None):
        cl, cw = read_robot_size(args.config)
        length = cl if length is None else length
        width = cw if width is None else width
    if length is None or width is None or not (length > 0 and width > 0) or not math.isfinite(length + width):
        return None
    return length, width


def report_line(name: str, ints, floats, n_boxes: int) -> Tuple[str, str]:
    """(state, report line) of one file from its footprint_check result (ints named by FP_I, floats by FP_F)."""
    from .export import FP_F, FP_I, FP_KIND_BOX, FP_KIND_WALL
    i = dict(zip(FP_I, (int(v) for v in ints)))
    f = dict(zip(FP_F, (float(v) for v in floats)))
    if i["rows"] == 0:
        return "not checked", f"not checked: {name}: no trajectory rows"
    box = (f"nearest keep-out box {i['nearest_box']} at {f['nearest_box_in']:.3f} in, t {f['nearest_box_t']:.3f} s"
           if n_boxes and i["nearest_box_row"] >= 0 else "no keep-out boxes")
    if i["first_row"] < 0:
        return "clear", (f"clear: {name}: wall clearance {-f['worst_wall_in']:.3f} in at t {f['worst_wall_t']:.3f} s; "
                         f"{box}; sampling step <= {f['max_corner_step_in']:.3f} in")
    k = i["first_kind"]
    what = "wall" if k == FP_KIND_WALL else f"keep-out box {k - FP_KIND_BOX}" if k >= FP_KIND_BOX else "non-finite row"
    wall = (f"worst wall overhang {f['worst_wall_in']:.3f} in at t {f['worst_wall_t']:.3f} s"
            if i["worst_wall_row"] >= 0 else "no finite row")
    return "hits", (f"hits: {name}: first at t {f['first_t']:.3f} s (row {i['first_row']}): {what}; {wall}; {box}; "
                    f"{i['violating_rows']} of {i['rows']} rows")


def check_routes(routes: Sequence, cons, size, field, boxes, tol_in: float, tile_paths: int = 8192,
                 device: str = "cuda:0"):
    """Profile every route (tile_paths at a time) and check its footprint.  Returns [(name, state, report line)]."""
    from . import export
    from .engine import Engine
    from .packing import pack_paths
    eng = Engine(device)
    out = []
    for lo in range(0, len(routes), tile_paths):
        tile = routes[lo: lo + tile_paths]
        res = eng.profile(eng.upload(pack_paths([(pts, nodes, aps) for _, pts, nodes, aps in tile], cons)))
        rows, row_off = export.export_rows(eng, res)
        ints, floats = export.footprint_check(eng, rows, row_off, *size, field=field, keep_out=boxes, tol_in=tol_in)
        status = res.status.cpu().tolist()
        for b, (name, _, _, _) in enumerate(tile):
            s = int(status[b])
            if s != 0:
                out.append((name, "not checked", f"not checked: {name}: profile failed, status {s} "
                                                 f"({STATUS_NAMES.get(s, 'unknown')})"))
            else:
                out.append((name, *report_line(name, ints[b], floats[b], len(boxes))))
    return out


def check_trajectories(folder: str, size, field, boxes, tol_in: float, device: str = "cuda:0"):
    """Read every *.txt of folder back on the device (groups of at most export.MAX_READ_BYTES) and check its
    footprint.  Returns [(name, state, report line)]."""
    import numpy as np
    import torch
    from . import export
    from .engine import Engine
    names = sorted(n for n in os.listdir(folder) if n.endswith(".txt") and os.path.isfile(os.path.join(folder, n)))
    sizes = [os.path.getsize(os.path.join(folder, n)) for n in names]
    eng = Engine(device)
    out = []
    for g0, g1 in byte_groups(sizes, export.MAX_READ_BYTES):
        if sizes[g0] > export.MAX_READ_BYTES:
            out.append((names[g0], "not checked", f"not checked: {names[g0]}: more than {export.MAX_READ_BYTES} bytes"))
            continue
        offs = np.zeros(g1 - g0 + 1, dtype=np.int64)
        np.cumsum(sizes[g0:g1], out=offs[1:])
        buf = torch.empty(max(int(offs[-1]), 1), dtype=torch.uint8, pin_memory=True)
        view = memoryview(buf.numpy())
        for n, a, z in zip(names[g0:g1], offs[:-1], offs[1:]):
            with open(os.path.join(folder, n), "rb") as f:
                f.readinto(view[a:z])
        p = export.parse_text_batch(eng, buf[:int(offs[-1])], offs)
        ints, floats = export.footprint_check(eng, p.rows, p.row_offsets, *size, field=field, keep_out=boxes,
                                              tol_in=tol_in)
        bad = torch.nonzero(p.line_errors).flatten()
        first_err = {}
        if bad.numel():
            codes = p.line_errors[bad].cpu().numpy()
            lines, pl = bad.cpu().numpy(), p.path_line_offsets.cpu().numpy()
            for line, code, b in zip(lines, codes, np.searchsorted(pl, lines, side="right") - 1):
                first_err.setdefault(int(b), (int(line - pl[b]) + 1, int(code)))
        for b, name in enumerate(names[g0:g1]):
            if b in first_err:
                line, code = first_err[b]
                out.append((name, "unreadable", f"unreadable: {name}: line {line}: {export.line_error_text(code)}"))
            else:
                out.append((name, *report_line(name, ints[b], floats[b], len(boxes))))
    return out


def main(argv: Optional[List[str]] = None) -> int:
    args = parse_args(argv)
    size = robot_size(args)
    if size is None:
        print("the robot's size is unknown: pass --robot-length-in and --robot-width-in (positive inches), or a --config "
              "with robot.length and robot.width", file=sys.stderr)
        return 2
    from .export import default_field
    h = args.field_half_in
    field = default_field() if h is None else (-h, h, -h, h)
    if args.trajectories:
        skipped = []
        checked = check_trajectories(args.dir, size, field, args.keep_out, args.tol_in, args.device)
    else:
        routes, skipped = read_routes(args.dir)
        checked = (check_routes(routes, constraints(args), size, field, args.keep_out, args.tol_in, args.tile_paths,
                                args.device) if routes else [])
    for name, why in skipped:
        print(f"not checked: {name}: {why}")
    for _, _, line in checked:
        print(line)
    n_clear = sum(state == "clear" for _, state, _ in checked)
    total = len(checked) + len(skipped)
    print(f"{n_clear} of {total} files clear in {args.dir} (robot {size[0]:g} x {size[1]:g} in, field x {field[0]:g} .. "
          f"{field[1]:g}, y {field[2]:g} .. {field[3]:g} in, {len(args.keep_out)} keep-out boxes, tolerance {args.tol_in:g} in)")
    return 0 if n_clear == total else 1


if __name__ == "__main__":
    sys.exit(main())

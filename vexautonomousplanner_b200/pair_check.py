"""python -m vexautonomousplanner_b200.pair_check DIR_A DIR_B --robot-a-in L,W [--robot-b-in L,W] [--min-gap-in G]

Checks on the device where two robots running two routes at the same time first touch (export.pair_check): every
saved trajectory .txt of DIR_A against every one of DIR_B.  In autonomous both robots of an alliance drive at once; a
keep-out box drawn around the partner's path (field_check) flags every crossing, including those the two robots pass
at different times.

Both folders hold saved trajectory files (what save_routes writes), read back on the device with
export.parse_text_batch; each side's constraints are baked into its own files.  When both arguments name the same
folder, every unordered pair of its files is checked once and no file is paired with itself.  Both robots start at
t = 0 of their own rows; a robot that has finished stays parked at its last row.  Sizes are inches, length along the
heading; --robot-b-in defaults to A's size.

One line per pair:
  clear: A x B: closest D in at t T s; A ends at T s, B at T s; sampling step <= S in
  contact: A x B: first at t T s (A row r | B row r); closest D in at t T s; N of M events
  not checked: A x B: NAME: line L: reason | row r is not finite | t decreases at row r | no trajectory rows
and a final count.  A negative D is a penetration depth.  Rows count from 0 within the route's trajectory rows.  The
sampling step is the largest move of a robot's corner between consecutive rows of its own route: the check sees the
robots at the rows only.  Exit status 0 only when every pair is clear, 1 otherwise, 2 for argument errors.
"""
from __future__ import annotations

import argparse
import math
import os
import sys
from typing import List, Optional, Tuple


def robot_size(text: str) -> Tuple[float, float]:
    """argparse type of --robot-a-in / --robot-b-in: "L,W", two positive finite inches (length along the heading)."""
    parts = text.split(",")
    try:
        size = tuple(float(v) for v in parts)
    except ValueError:
        size = ()
    if len(size) != 2 or not all(v > 0 and math.isfinite(v) for v in size):
        raise argparse.ArgumentTypeError(f"{text!r} is not L,W (two positive finite numbers, inches)")
    return size


def parse_args(argv: Optional[List[str]] = None) -> argparse.Namespace:
    p = argparse.ArgumentParser(prog="python -m vexautonomousplanner_b200.pair_check",
                                description="Check where two robots running saved routes at the same time first touch: "
                                            "every trajectory .txt of DIR_A against every one of DIR_B.")
    p.add_argument("dir_a", help="folder of saved trajectory .txt files (robot A)")
    p.add_argument("dir_b", help="folder of saved trajectory .txt files (robot B); the same folder checks its unordered pairs")
    p.add_argument("--robot-a-in", type=robot_size, required=True, dest="size_a", metavar="L,W",
                   help="robot A's length along its heading and width, inches")
    p.add_argument("--robot-b-in", type=robot_size, dest="size_b", metavar="L,W", help="robot B's size (default: A's)")
    p.add_argument("--min-gap-in", type=float, default=0.0, dest="min_gap",
                   help="a gap smaller than this many inches is a contact (default 0: only an overlap is)")
    p.add_argument("--device", default="cuda:0")
    args = p.parse_args(argv)
    if not math.isfinite(args.min_gap):
        p.error("--min-gap-in must be finite")
    if args.size_b is None:
        args.size_b = args.size_a
    return args


def pairs_of(n_a: int, n_b: int, same: bool) -> List[Tuple[int, int]]:
    """Every (i, j) of A's and B's files; for one folder on both sides, i < j only."""
    return [(i, j) for i in range(n_a) for j in range(i + 1 if same else 0, n_b)]


def read_folder(eng, folder: str):
    """(names, rows, row_offsets, errors) of every *.txt of folder read back on the device: rows[R, 7] and offsets[B+1]
    of all groups of field_check.trajectory_groups concatenated; errors maps a file's index to why it is unreadable."""
    import torch
    from . import export
    from .field_check import trajectory_groups
    names, rows, offs, errors, total = [], [], [torch.zeros(1, dtype=torch.int64, device=eng.device)], {}, 0
    for gnames, p, gerr in trajectory_groups(eng, folder):
        base = len(names)
        names += gnames
        if p is None:
            errors[base] = f"more than {export.MAX_READ_BYTES} bytes"
            offs.append(torch.full((len(gnames),), total, dtype=torch.int64, device=eng.device))
            continue
        errors.update({base + b: f"line {line}: {why}" for b, (line, why) in gerr.items()})
        rows.append(p.rows)
        offs.append(p.row_offsets[1:] + total)
        total += int(p.rows.shape[0])
    rows = torch.cat(rows) if rows else torch.zeros((0, 7), dtype=torch.float64, device=eng.device)
    return names, rows, torch.cat(offs), errors


def report_line(name_a: str, name_b: str, ints, floats, bad_a, bad_b) -> Tuple[str, str]:
    """(state, report line) of one pair from its pair_check result (ints named by PC_I, floats by PC_F) and the
    (row, reason) of both routes."""
    from .export import PC_A_INVALID, PC_B_INVALID, PC_F, PC_I, PC_OK, pair_reason_text
    i = dict(zip(PC_I, (int(v) for v in ints)))
    f = dict(zip(PC_F, (float(v) for v in floats)))
    head = f"{name_a} x {name_b}"
    if i["status"] != PC_OK:
        if i["status"] == PC_A_INVALID:
            why = f"{name_a}: {pair_reason_text(int(bad_a[0]), int(bad_a[1]))}"
        elif i["status"] == PC_B_INVALID:
            why = f"{name_b}: {pair_reason_text(int(bad_b[0]), int(bad_b[1]))}"
        else:
            why = "a route index out of range"
        return "not checked", f"not checked: {head}: {why}"
    closest = f"closest {f['nearest_in']:.3f} in at t {f['nearest_t']:.3f} s"
    if i["first_row"] < 0:
        return "clear", (f"clear: {head}: {closest}; A ends at {f['last_t_a']:.3f} s, B at {f['last_t_b']:.3f} s; "
                         f"sampling step <= {f['max_corner_step_in']:.3f} in")
    side = "AB"[i["first_side"]]
    return "contact", (f"contact: {head}: first at t {f['first_t']:.3f} s ({side} row {i['first_row']}); {closest}; "
                       f"{i['contacts']} of {i['events']} events")


def check_folders(dir_a: str, dir_b: str, size_a, size_b, min_gap: float = 0.0, device: str = "cuda:0"):
    """Every file of dir_a against every file of dir_b (unordered pairs when both are the same folder).
    Returns [(state, report line)] in pair order."""
    import numpy as np
    from . import export
    from .engine import Engine
    eng = Engine(device)
    same = os.path.realpath(dir_a) == os.path.realpath(dir_b)
    names_a, rows_a, off_a, err_a = read_folder(eng, dir_a)
    names_b, rows_b, off_b, err_b = (names_a, rows_a, off_a, err_a) if same else read_folder(eng, dir_b)
    pairs = pairs_of(len(names_a), len(names_b), same)
    run = [(i, j) for i, j in pairs if i not in err_a and j not in err_b]
    if run:
        ints, floats, bad_a, bad_b = export.pair_check(eng, rows_a, off_a, size_a, rows_b, off_b, size_b,
                                                       np.array(run, dtype=np.int64), min_gap)
        res = {ij: k for k, ij in enumerate(run)}
    out = []
    for i, j in pairs:
        head = f"{names_a[i]} x {names_b[j]}"
        if i in err_a:
            out.append(("not checked", f"not checked: {head}: {names_a[i]}: {err_a[i]}"))
        elif j in err_b:
            out.append(("not checked", f"not checked: {head}: {names_b[j]}: {err_b[j]}"))
        else:
            k = res[(i, j)]
            out.append(report_line(names_a[i], names_b[j], ints[k], floats[k], bad_a[i], bad_b[j]))
    return out


def main(argv: Optional[List[str]] = None) -> int:
    from .field_check import trajectory_files
    args = parse_args(argv)
    for d in (args.dir_a, args.dir_b):
        if not os.path.isdir(d) or not trajectory_files(d):
            print(f"{d}: no trajectory .txt files", file=sys.stderr)
            return 2
    checked = check_folders(args.dir_a, args.dir_b, args.size_a, args.size_b, args.min_gap, args.device)
    for _, line in checked:
        print(line)
    n_clear = sum(state == "clear" for state, _ in checked)
    (la, wa), (lb, wb) = args.size_a, args.size_b
    print(f"{n_clear} of {len(checked)} pairs clear (A {args.dir_a}, robot {la:g} x {wa:g} in; B {args.dir_b}, robot "
          f"{lb:g} x {wb:g} in; min gap {args.min_gap:g} in)")
    return 0 if n_clear == len(checked) else 1


if __name__ == "__main__":
    sys.exit(main())

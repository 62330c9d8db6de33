"""python -m vexautonomousplanner_b200.save_routes ROUTES_DIR OUT_DIR [options]

Re-saves a folder of routes the way the GUI's save does (save_nodes_to_file, gui_manager.py:232-316), for every route at
once: each ROUTES_DIR/*.txt is a node-JSON route (what the GUI writes to its routes folder); its trajectory .txt body goes
to OUT_DIR/<same name>.txt.  Typical use: a robot constant changed and every route has to be saved again.

Constraints are built as the GUI builds them (path.py:314-321): max_dec = max_acc, friction 0.8, track_width in feet =
track width in inches / 12.  They come from --config (a config.yaml in the GUI's layout: motion.max_velocity,
motion.max_acceleration, motion.max_jerk, robot.track_width in inches; missing keys take the factory values, as
ConfigManager does), and the explicit flags override them; without either, the factory set (synth.FACTORY).

Files that are not route JSON and routes the GUI's save refuses (it needs more than two nodes, a start node and an end
node, gui_manager.py:263-267) are listed and not written; so are routes whose profile fails (status != 0).  The exit
status is 0 only when every route was written.

With --check nothing is written: every route's fresh body is compared with OUT_DIR/<name>.txt on the device (the saved
file is read back with export.compare_text_batch) and one line per route says "up to date" (the bytes are equal),
"stale" (the first differing line, old -> new trajectory rows, old -> new duration, the largest moves of x, y, v and
heading over the common rows, the action rows that differ), "missing" or "unreadable" (the line and the reason).  The
exit status is 0 only when every route is up to date.  Use it in CI to see that committed trajectory files are current,
or after a constant changed to see what the change does to each route.
"""
from __future__ import annotations

import argparse
import os
import sys
from typing import List, Optional, Sequence, Tuple

from .export import load_nodes, px_points_to_ft
from .synth import FACTORY

DEFAULTS = dict(max_velocity=FACTORY[0], max_acceleration=FACTORY[1], max_jerk=FACTORY[4], track_width_in=12.5)
STATUS_NAMES = {-1: "build_path returns False", -2: "IndexError", -3: "ValueError", -4: "capacity",
                -5: "profile does not terminate", -6: "event tables full"}


def read_config(path: str) -> dict:
    """The constraint values of a config.yaml in the GUI's layout (PyYAML is imported only here)."""
    import yaml
    with open(path) as f:
        cfg = yaml.safe_load(f) or {}
    motion, robot = cfg.get("motion") or {}, cfg.get("robot") or {}
    out = dict(DEFAULTS)
    for key in ("max_velocity", "max_acceleration", "max_jerk"):
        if motion.get(key) is not None:
            out[key] = float(motion[key])
    if robot.get("track_width") is not None:
        out["track_width_in"] = float(robot["track_width"])
    return out


def constraints(args: argparse.Namespace) -> Tuple[float, ...]:
    """(max_vel, max_acc, max_dec, friction, max_jerk, track_width_ft) as path.py:314-321 builds them."""
    vals = read_config(args.config) if args.config else dict(DEFAULTS)
    for key in DEFAULTS:
        if getattr(args, key) is not None:
            vals[key] = float(getattr(args, key))
    a = vals["max_acceleration"]
    return (vals["max_velocity"], a, a, 0.8, vals["max_jerk"], vals["track_width_in"] / 12)


def read_routes(routes_dir: str):
    """Parse every *.txt of routes_dir.  Returns (routes, skipped): routes = [(name, points_ft, nodes, action_points)],
    skipped = [(name, reason)] for files that are not route JSON and routes the GUI's save refuses."""
    routes, skipped = [], []
    for name in sorted(os.listdir(routes_dir)):
        path = os.path.join(routes_dir, name)
        if not name.endswith(".txt") or not os.path.isfile(path):
            continue
        try:
            with open(path, encoding="utf-8") as f:
                pts_px, nodes, aps, _ = load_nodes(f.read())
        except (ValueError, TypeError, IndexError, KeyError, AttributeError) as e:
            skipped.append((name, f"not route JSON ({type(e).__name__}: {e})"))
            continue
        has_start = any(n.is_start_node for n in nodes)
        has_end = any(n.is_end_node for n in nodes)
        if not (len(nodes) > 2 and has_start and has_end):
            skipped.append((name, f"the GUI's save refuses it: {len(nodes)} nodes, start node {'present' if has_start else 'missing'}, "
                                  f"end node {'present' if has_end else 'missing'} (it needs more than two nodes and both)"))
            continue
        routes.append((name, px_points_to_ft(pts_px), nodes, aps))
    return routes, skipped


def save_routes(routes: Sequence, out_dir: str, cons, tile_paths: int = 8192, device: str = "cuda:0"):
    """Profile and write every route, tile_paths at a time.  Returns [(name, reason)] of the routes not written."""
    from .engine import Engine
    from .export import save_text_batch
    from .packing import pack_paths
    eng = Engine(device)
    failed = []
    for lo in range(0, len(routes), tile_paths):
        tile = routes[lo: lo + tile_paths]
        db = eng.upload(pack_paths([(pts, nodes, aps) for _, pts, nodes, aps in tile], cons))
        res = eng.profile(db)
        text, offs, ok = save_text_batch(eng, res, db, [[n.action_values for n in nodes] for _, _, nodes, _ in tile],
                                         [[a.action_values for a in aps] for _, _, _, aps in tile])
        status = res.status.cpu().tolist() if not ok.all() else None
        for b, (name, _, _, _) in enumerate(tile):
            if not ok[b]:
                s = int(status[b])
                failed.append((name, f"status {s} ({STATUS_NAMES.get(s, 'unknown')})"))
                continue
            with open(os.path.join(out_dir, name), "wb") as f:
                f.write(text[offs[b]: offs[b + 1]].tobytes())
    return failed


def check_line(name: str, ints, floats) -> Tuple[str, str]:
    """(state, report line) of one route from its compare_text_batch result (ints named by CMP_I, floats by CMP_F)."""
    from .export import CMP_F, CMP_I, line_error_text
    i = dict(zip(CMP_I, (int(v) for v in ints)))
    f = dict(zip(CMP_F, (float(v) for v in floats)))
    if i["diff_byte"] < 0:
        return "up to date", f"up to date: {name}"
    if i["error_line"] > 0:
        return "unreadable", f"unreadable: {name}: line {i['error_line']}: {line_error_text(i['error_code'])}"
    return "stale", (f"stale: {name}: first difference on line {i['diff_line']}; rows {i['old_rows']} -> {i['new_rows']}; "
                     f"duration {f['old_t']!r} -> {f['new_t']!r} s; max |dx| {f['max_dx']:.6g} in, |dy| {f['max_dy']:.6g} in, "
                     f"|dv| {f['max_dv']:.6g} in/s, |dheading| {f['max_dheading']:.6g}; "
                     f"{i['action_rows_differ']} action rows differ")


def byte_groups(sizes: Sequence[int], limit: int) -> List[Tuple[int, int]]:
    """Consecutive groups [g0, g1) of items whose sizes add up to at most limit each; an item larger than limit on its
    own is a group of one."""
    groups, g0, total = [], 0, 0
    for b, s in enumerate(sizes):
        if b > g0 and total + s > limit:
            groups.append((g0, b))
            g0, total = b, 0
        total += s
    if g0 < len(sizes):
        groups.append((g0, len(sizes)))
    return groups


def check_batch(eng, db, node_actions, ap_actions, files: Sequence[str]):
    """One batch of --check: profile db, assemble the fresh bodies, read the saved files[b] (missing ones as empty
    bodies) into one pinned buffer and compare on the device, in groups of routes whose saved and fresh bodies together
    fit one read (export.MAX_READ_BYTES).  Returns (res, ok, present, ints, floats) with ints / floats as
    export.compare_text_batch gives them."""
    import numpy as np
    import torch
    from . import export
    res = eng.profile(db)
    text, offs, ok = export.save_text_batch(eng, res, db, node_actions, ap_actions)
    rows, row_off = export.export_rows(eng, res)
    present = [os.path.isfile(p) for p in files]
    sizes = np.array([os.path.getsize(p) if there else 0 for p, there in zip(files, present)], dtype=np.int64)
    groups = byte_groups((sizes + np.diff(offs)).tolist(), export.MAX_READ_BYTES)
    # group by group: the saved files, then room for the fresh bodies (compare_text_batch puts them there)
    buf = torch.empty(max(int(sizes.sum() + offs[-1]), 1), dtype=torch.uint8, pin_memory=True)
    view = memoryview(buf.numpy())
    ints, floats, base = [], [], 0
    for g0, g1 in groups:
        old_off = np.zeros(g1 - g0 + 1, dtype=np.int64)
        np.cumsum(sizes[g0:g1], out=old_off[1:])
        for p, there, a, z in zip(files[g0:g1], present[g0:g1], base + old_off[:-1], base + old_off[1:]):
            if there:
                with open(p, "rb") as f:
                    f.readinto(view[a:z])
        n = int(old_off[-1] + offs[g1] - offs[g0])
        # row_off[g0:g1 + 1] still indexes the whole batch's rows
        gi, gf, _ = export.compare_text_batch(eng, buf[base:base + n], old_off, text[offs[g0]:offs[g1]],
                                              offs[g0:g1 + 1] - offs[g0], rows, row_off[g0:g1 + 1])
        ints.append(gi)
        floats.append(gf)
        base += n
    return res, ok, present, np.concatenate(ints), np.concatenate(floats)


def check_routes(routes: Sequence, out_dir: str, cons, tile_paths: int = 8192, device: str = "cuda:0"):
    """Compare every route's fresh body with out_dir/<name>, tile_paths routes at a time; writes nothing.
    Returns [(name, state, report line)], state one of "up to date", "stale", "missing", "unreadable", "not checked"."""
    from .engine import Engine
    from .packing import pack_paths
    eng = Engine(device)
    out = []
    for lo in range(0, len(routes), tile_paths):
        tile = routes[lo: lo + tile_paths]
        db = eng.upload(pack_paths([(pts, nodes, aps) for _, pts, nodes, aps in tile], cons))
        res, ok, present, ints, floats = check_batch(eng, db, [[n.action_values for n in nodes] for _, _, nodes, _ in tile],
                                                     [[a.action_values for a in aps] for _, _, _, aps in tile],
                                                     [os.path.join(out_dir, name) for name, _, _, _ in tile])
        status = res.status.cpu().tolist() if not ok.all() else None
        for b, (name, _, _, _) in enumerate(tile):
            if not ok[b]:
                s = int(status[b])
                out.append((name, "not checked", f"not checked: {name}: profile failed, status {s} "
                                                 f"({STATUS_NAMES.get(s, 'unknown')})"))
            elif not present[b]:
                out.append((name, "missing", f"missing: {name}"))
            else:
                out.append((name, *check_line(name, ints[b], floats[b])))
    return out


def parse_args(argv: Optional[List[str]] = None) -> argparse.Namespace:
    p = argparse.ArgumentParser(prog="python -m vexautonomousplanner_b200.save_routes",
                                description="Re-save every route of a folder: write each route's trajectory .txt.")
    p.add_argument("routes_dir", help="folder of node-JSON routes (*.txt), the GUI's routes folder")
    p.add_argument("out_dir", help="folder for the trajectory files (must differ from routes_dir)")
    p.add_argument("--config", help="config.yaml in the GUI's layout (motion.*, robot.track_width in inches)")
    p.add_argument("--max-velocity", type=float, dest="max_velocity", help=f"ft/s (factory {DEFAULTS['max_velocity']})")
    p.add_argument("--max-acceleration", type=float, dest="max_acceleration",
                   help=f"ft/s^2, also the deceleration (factory {DEFAULTS['max_acceleration']})")
    p.add_argument("--max-jerk", type=float, dest="max_jerk", help=f"ft/s^3 (factory {DEFAULTS['max_jerk']})")
    p.add_argument("--track-width-in", type=float, dest="track_width_in",
                   help=f"track width in inches (factory {DEFAULTS['track_width_in']})")
    p.add_argument("--tile-paths", type=int, default=8192, help="routes profiled per batch (default 8192)")
    p.add_argument("--device", default="cuda:0")
    p.add_argument("--check", action="store_true",
                   help="write nothing: report which files of OUT_DIR are up to date, stale, missing or unreadable")
    args = p.parse_args(argv)
    if args.tile_paths < 1:
        p.error("--tile-paths must be at least 1")
    return args


def main(argv: Optional[List[str]] = None) -> int:
    args = parse_args(argv)
    if os.path.realpath(args.out_dir) == os.path.realpath(args.routes_dir):
        print(f"refusing to write into the routes folder itself ({args.routes_dir}): the trajectory files would "
              "overwrite the routes; choose another OUT_DIR", file=sys.stderr)
        return 2
    cons = constraints(args)
    routes, skipped = read_routes(args.routes_dir)
    cons_text = (f"max_velocity {cons[0]}, max_acceleration {cons[1]}, max_jerk {cons[4]}, track_width {cons[5]} ft")
    if args.check:
        checked = check_routes(routes, args.out_dir, cons, args.tile_paths, args.device) if routes else []
        for name, why in skipped:
            print(f"not checked: {name}: {why}")
        for _, _, line in checked:
            print(line)
        n_up = sum(state == "up to date" for _, state, _ in checked)
        print(f"{n_up} of {len(routes) + len(skipped)} files up to date in {args.out_dir} ({cons_text})")
        return 0 if n_up == len(routes) + len(skipped) else 1
    os.makedirs(args.out_dir, exist_ok=True)
    failed = save_routes(routes, args.out_dir, cons, args.tile_paths, args.device) if routes else []
    for name, why in skipped:
        print(f"not written: {name}: {why}")
    for name, why in failed:
        print(f"not written: {name}: profile failed, {why}")
    n_written = len(routes) - len(failed)
    print(f"wrote {n_written} of {len(routes) + len(skipped)} files to {args.out_dir} ({cons_text})")
    return 0 if not skipped and not failed else 1


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""Cost of growing streaming trajectories during the run and of reading them mid-run (ftkb_get_live_curveset,
ftkb_group_get_live_curveset), on the two workloads a streaming user runs on several devices:

    c3_slabs      a streaming z-slab group over the C3 shape: 512^3 moving extremum (bench.py's c3 generator), 32 steps
    woven_chunks  a streaming time-chunk group (8 timesteps per chunk) over the woven 4096^2 x 32 field of scripts/stream_timing.py

Every step is push (generated on the device) + advance_timestep; the series ends with update_timestep.  ms_per_step is the wall
clock of that loop over the steps, ms_finalize the group's (or tracker's) finalize after it -- together the time to trajectories.
The same workloads on one tracker, with a live query after every step (--live-queries) and without, give the cost of the query.

    python scripts/live_stream_timing.py [--tree DIR] [--label NAME] [--devices 0 1 ...] [--live-queries] > out.jsonl

--tree runs the ftk_b200 package of another checkout (built there), so that one session can alternate two versions;
--live-queries needs a tree that has them.  One JSON line per run.
"""
import argparse
import json
import os
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--label", default="this")
ap.add_argument("--devices", type=int, nargs="+", default=None, help="group device list (default: every visible GPU, at least two entries)")
ap.add_argument("--live-queries", action="store_true", help="also time one tracker with and without a live query after every step")
ap.add_argument("--steps", type=int, default=32)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.tree))

from ftk_b200 import _lib as L  # noqa: E402
from ftk_b200 import tracker as T  # noqa: E402
from ftk_b200.group import GroupTracker  # noqa: E402

C3_DIMS, C3_PARAMS = [512, 512, 512], [256.3, 255.7, 256.1, 0.1, 0.11, 0.1]
WOVEN_DIMS = [4096, 4096]
WORKLOADS = {
    "c3_slabs": dict(dims=C3_DIMS, kind=L.SYN_MOVING_EXTREMUM, params=C3_PARAMS, chunk=0, time=lambda k, n: float(k)),
    "woven_chunks": dict(dims=WOVEN_DIMS, kind=L.SYN_WOVEN, params=[], chunk=8, time=lambda k, n: k / (n - 1)),
}


def series(tr, w, steps, after_step=None):
    t0 = time.perf_counter()
    for k in range(steps):
        tr.push_synthetic_snapshot(w["kind"], w["params"], w["time"](k, steps))
        if k != 0:
            tr.advance_timestep()
        if k == steps - 1:
            tr.update_timestep()
        if after_step:
            after_step(tr)
    return t0


def query(tr):
    _, cs = tr.live_curveset()
    cs.close()


def run_group(name, ids, steps):
    w = WORKLOADS[name]
    g = GroupTracker(w["dims"], ids, field="scalar", chunk=w["chunk"], streaming=True)
    t0 = series(g, w, steps)
    t1 = time.perf_counter()
    root = g.finalize()
    t2 = time.perf_counter()
    out = {"label": args.label, "workload": name, "tracker": "group", "devices": ids, "steps": steps,
           "ms_per_step": (t1 - t0) * 1e3 / steps, "ms_finalize": (t2 - t1) * 1e3, "ms_to_trajectories": (t2 - t0) * 1e3,
           "points": len(root.get_discrete_critical_points()), "trajectories": len(root.get_trajectory_index())}
    g.close()
    return out


def run_one(name, steps, live):
    w = WORKLOADS[name]
    tr = T.make_tracker(w["dims"], field="scalar", streaming=True)
    t0 = series(tr, w, steps, query if live else None)
    tr.synchronize()
    t1 = time.perf_counter()
    tr.finalize()
    t2 = time.perf_counter()
    out = {"label": args.label, "workload": name, "tracker": "one", "live_query_every_step": live, "steps": steps,
           "ms_per_step": (t1 - t0) * 1e3 / steps, "ms_finalize": (t2 - t1) * 1e3, "ms_to_trajectories": (t2 - t0) * 1e3,
           "points": int(tr.stats()["points"]), "trajectories": len(tr.get_trajectory_index())}
    tr.close()
    return out


if __name__ == "__main__":
    ndev = L.lib().ftkb_device_count()
    if ndev < 1:
        sys.exit("no B200 visible: nothing measured")
    ids = args.devices or (list(range(ndev)) if ndev >= 2 else [0, 0])
    for name in WORKLOADS:
        run_group(name, ids, 4)                   # warm-up: contexts, module load, buffers
        print(json.dumps(run_group(name, ids, args.steps)), flush=True)
        if args.live_queries:
            for live in (False, True, False, True):
                print(json.dumps(run_one(name, args.steps, live)), flush=True)

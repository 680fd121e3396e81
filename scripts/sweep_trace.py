#!/usr/bin/env python
"""sweep_trace.py -- what the sweeps of a build run, case by case, for comparing two builds of the host code.

    python scripts/sweep_trace.py [--root TREE] [--out FILE] [--only SUBSTRING]

One JSON line per case: the kernels the case launched (torch.profiler with CUDA activities, in start order per stream), every
integer field of ftkb_stats plus the factor and the resolution, whether ms_derive > 0, and a hash of the points and the ordered
trajectories.  Timing fields are left out, so two builds that choose the same scans with the same parameters write identical
lines.  --root imports ftk_b200 (and the test field builders) from another tree, e.g. a build of the parent commit.

Cases: every (field, scan path) of tests/test_scan_boundaries.py MATRIX; FTKB_DEFER=0 and FTKB_WL_CAP=64 runs; last_layer_resolution()
on an aligned 2D scalar layer, a borrowed 2D layer at +8 bytes, a 3D scalar layer and vector layers (poisoned ones included); a
3-slab group on a 3D scalar field.
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

INT_STATS = ["simplices_tested", "cells_scanned", "cells_refined", "points", "kernel_launches", "h2d_bytes", "d2h_bytes",
             "scan_launches", "sweeps_repeated"]


class Env:
    """the setenv / delenv half of pytest's monkeypatch that test_scan_boundaries.make uses"""
    def setenv(self, k, v):
        os.environ[k] = v

    def delenv(self, k):
        os.environ.pop(k, None)


def result_hash(tr):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(tr.get_discrete_critical_points()).tobytes())
    for idx, loop in tr.get_trajectory_index():
        h.update(np.asarray(idx, np.int64).tobytes())
        h.update(b"L" if loop else b"O")
    return h.hexdigest()[:24]


def kernels(prof):
    """kernel names in start order, per stream (streams renumbered in the order of their raw ids)"""
    import torch
    evs = [e for e in prof.profiler.kineto_results.events() if e.device_type() == torch.autograd.DeviceType.CUDA]
    evs = [e for e in evs if not e.name().startswith(("Memcpy", "Memset"))]
    streams = sorted({e.device_resource_id() for e in evs})
    out = {}
    for e in sorted(evs, key=lambda e: e.start_ns()):
        out.setdefault(str(streams.index(e.device_resource_id())), []).append(e.name())
    return out


def traced(name, fn):
    """run fn() under the profiler; fn returns (stats dict, hash or None, extra dict)"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        st, h, extra = fn()
        torch.cuda.synchronize()
    rec = {"case": name, "kernels": kernels(prof)}
    rec.update({k: int(st[k]) for k in INT_STATS})
    rec["scaling_factor"] = float(st["scaling_factor"])
    rec["resolution"] = float(st["resolution"]).hex()
    rec["ms_derive_positive"] = bool(st["ms_derive"] > 0)
    rec["hash"] = h
    rec.update(extra)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    root = os.path.abspath(a.root)
    sys.path[:0] = [root, os.path.join(root, "tests")]
    import torch
    import ftk_b200
    import test_scan_boundaries as B
    from oracle import cp_oracle as O
    from ftk_b200.group import track_on_devices
    assert ftk_b200.__file__.startswith(root), ftk_b200.__file__
    env = Env()
    out = open(a.out, "w") if a.out else sys.stdout

    def emit(name, fn):
        if a.only and a.only not in name:
            return
        rec = traced(name, fn)
        out.write(json.dumps(rec, sort_keys=True) + "\n")
        out.flush()

    def finish(tr, extra=None):
        st, h = tr.stats(), result_hash(tr)
        tr.close()
        return st, h, extra or {}

    # every field through every scan path of the boundary tests
    for name, path in B.MATRIX:
        emit(f"matrix/{name}/{path}", lambda n=name, p=path: finish(B.run(ftk_b200, p, n, env)))

    # synchronous steps, and a worklist that overflows (deferred replays and synchronous regrowth)
    for var, val in (("FTKB_DEFER", "0"), ("FTKB_WL_CAP", "64")):
        for gen, dims, T in (("woven", [256, 192], 8), ("moving_extremum", [40, 36, 34], 5)):
            def fn(var=var, val=val, gen=gen, dims=dims, T=T):
                os.environ[var] = val
                try:
                    tr = ftk_b200.track(list(O.synthetic_series(gen, dims, T, None)), dims, field="scalar")
                finally:
                    os.environ.pop(var)
                return finish(tr)
            emit(f"env/{var}={val}/{gen}", fn)

    # last_layer_resolution() on a layer no sweep has streamed yet
    rng = np.random.default_rng(5)

    def resolution_case(dims, field, snaps, borrow=False):
        def fn():
            tr = B.make(ftk_b200, "reg_borrow8" if borrow else ("vcells" if field == "vector" else "keys"), dims, field, env)
            res = []
            for k, s in enumerate(snaps):
                B.push(tr, field, s)
                res.append(float(tr.last_layer_resolution()).hex())
                if k:
                    tr.advance_timestep()
            tr.update_timestep()
            tr.finalize()
            return finish(tr, {"layer_resolutions": res})
        return fn

    def series(dims, nv=1, T=3):     # arrays are (D,) H, W (, components), x fastest
        shape = tuple(reversed(dims)) + ((nv,) if nv > 1 else ())
        return [rng.standard_normal(shape) for _ in range(T)]
    s2, s3, v2, v3 = series([96, 80]), series([34, 30, 28]), series([96, 80], 2), series([34, 30, 28], 3)
    v2p = [v.copy() for v in v2]
    v2p[1][40, 30, 0] = 1.5 * 2.0 ** 1000
    s3p = [s.copy() for s in s3]
    s3p[1][14, 15, 17] = 1.5 * 2.0 ** 1000
    for name, dims, field, snaps, borrow in (("2d_scalar", [96, 80], "scalar", s2, False), ("2d_scalar_borrow8", [96, 80], "scalar", s2, True),
                                             ("3d_scalar", [34, 30, 28], "scalar", s3, False), ("3d_scalar_poison", [34, 30, 28], "scalar", s3p, False),
                                             ("2d_vector", [96, 80], "vector", v2, False), ("2d_vector_poison", [96, 80], "vector", v2p, False),
                                             ("3d_vector", [34, 30, 28], "vector", v3, False)):
        emit(f"resolution/{name}", resolution_case(dims, field, snaps, borrow))

    # z-slabs: every slab context resolves its first layer outside a sweep
    def slabs():
        dims = [36, 30, 26]
        snaps = series(dims, T=4)
        g, root = track_on_devices(snaps, dims, [0, 0, 0], field="scalar", chunk=0)
        st, h = g.stats(), result_hash(root)
        g.close()
        return st, h, {}
    emit("group/zslabs3/3d_scalar", slabs)
    torch.cuda.synchronize()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Device-resident snapshots on several devices (ftkb_group_push_snapshot_device, DESIGN.md 7.1): ms per step of the C3 shape
(512^3 moving extremum, synthetic.hh:332-354 with C3's x0 / dir) when a producer on device 0 writes every snapshot with torch on a
side stream (named as the producer stream, no host synchronise) and the tracker reads it
  - on one context: copied device to device, and borrowed in place (FTKB_MEM_DEVICE_BORROW, a ring of buffers);
  - on groups of 2, 4 and 8 devices, as z-slabs and as time chunks of 8: every device copies what it needs from device 0
    (cudaMemcpyPeerAsync, NVLink).  With fewer GPUs visible the device ids repeat (ids i mod N, recorded in every row): the
    contexts then share the GPUs and the copies stay on one device;
  - on the same groups through page-locked host memory: the producer copies the snapshot to the host (its D2H is inside the
    timed window: a producer on a GPU pays it), then ftkb_group_push_snapshot sends it to every device over PCIe.
Every row times the same series: a host clock around K timed steps plus finalize, ended by a synchronise of every device,
after W warm-up steps.  The points of every row must equal those of the first row (host and device input give the same
result).  The card's name and power limit are read in the same run.
    python scripts/group_device_input_timing.py [--dims 512 512 512] [--steps 60] [--warmup 4] [--out FILE.jsonl]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ftk_b200  # noqa: E402
from ftk_b200 import _lib as L  # noqa: E402
from ftk_b200.group import GroupTracker  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--dims", type=int, nargs=3, default=[512, 512, 512])
ap.add_argument("--steps", type=int, default=60)
ap.add_argument("--warmup", type=int, default=4)
ap.add_argument("--chunk", type=int, default=8)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_group_device_input.jsonl"))
args = ap.parse_args()
dims, K, W = args.dims, args.steps, args.warmup
T = W + K
ndev = torch.cuda.device_count()
if ndev == 0:
    sys.exit("no CUDA device: this script measures on the GPU only")
x0 = [dims[0] / 2 + 0.3, dims[1] / 2 - 0.3, dims[2] / 2 + 0.1]      # C3: [256.3, 255.7, 256.1] at 512^3
d = [0.1, 0.11, 0.1]
shape = tuple(reversed(dims))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpus_visible": ndev, "nvidia_smi": [l.strip() for l in q.stdout.strip().splitlines()], "torch_name": torch.cuda.get_device_name(0)}


# ---- the producer: torch on device 0, on a side stream -------------------------------------------------------------------------
dev0 = torch.device("cuda:0")
prod = torch.cuda.Stream(device=dev0)
with torch.cuda.device(0), torch.cuda.stream(prod):
    zs, ys, xs = [torch.arange(n, dtype=torch.float64, device=dev0) for n in shape]
    plane = torch.empty(shape[1:], dtype=torch.float64, device=dev0)


def produce(k, out):
    """snapshot k of the moving extremum into `out`, enqueued on the producer stream"""
    with torch.cuda.device(0), torch.cuda.stream(prod):
        torch.add(((xs - (x0[0] + d[0] * k)) ** 2)[None, :], ((ys - (x0[1] + d[1] * k)) ** 2)[:, None], out=plane)
        torch.add(plane[None], ((zs - (x0[2] + d[2] * k)) ** 2)[:, None, None], out=out)


def sync_all():
    for i in range(ndev):
        torch.cuda.synchronize(i)


def pinned(n):
    p = C.c_void_p()
    assert L.lib().ftkb_host_alloc(n * 8, C.byref(p)) == 0
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(n,)).reshape(shape), p


def run(ids, chunk, source, ring):
    """source: "device" (tensor on device 0), "borrow" (one context, in place) or "host" (D2H into pinned memory, host push)"""
    one = len(ids) == 1
    tr = ftk_b200.make_tracker(dims, field="scalar", device=ids[0]) if one else GroupTracker(dims, ids, field="scalar", chunk=chunk)
    bufs = ring[:5] if source == "borrow" else ring[:1]       # a borrowed layer is read until three advances after its push
    d2h = 0.0

    def step(k):
        nonlocal d2h
        buf = bufs[k % len(bufs)]
        produce(k, buf)
        if source == "host":
            t = time.perf_counter()
            with torch.cuda.device(0), torch.cuda.stream(prod):
                host_t.copy_(buf, non_blocking=True)
            prod.synchronize()
            d2h += time.perf_counter() - t
            tr.push_scalar_field_snapshot(host_a)
        else:
            with torch.cuda.device(0), torch.cuda.stream(prod):      # torch's current stream = the producer stream
                if one:
                    tr.push_field_data_snapshot(scalar=buf, borrow=source == "borrow")
                else:
                    tr.push_scalar_field_snapshot(buf)
        if k:
            tr.advance_timestep()
        if k == T - 1:
            tr.update_timestep()

    for k in range(W):
        step(k)
    if one:
        tr.synchronize()
    sync_all()
    d2h = 0.0
    t0 = time.perf_counter()
    for k in range(W, T):
        step(k)
    root = tr.finalize() if not one else (tr.finalize() or tr)
    sync_all()
    dt = time.perf_counter() - t0
    pts = root.get_discrete_critical_points().copy()
    tr.close()
    row = {"devices": ids, "mode": "one context" if one else ("z-slabs" if chunk == 0 else f"time chunks of {chunk}"), "input": source,
           "dims": dims, "steps": K, "warmup": W, "ms_per_step": 1e3 * dt / K, "punctured_simplices": int(len(pts))}
    if source == "host":
        row["d2h_ms_per_step"] = 1e3 * d2h / K
    return row, pts


host_a, host_p = pinned(int(np.prod(shape)))
host_t = torch.from_numpy(host_a)
ring = [torch.empty(shape, dtype=torch.float64, device=dev0) for _ in range(5)]
info = card()
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as f:
    def emit(row):
        line = json.dumps(row)
        print(line, flush=True)
        f.write(line + "\n")
        f.flush()

    emit({"card": info, "timing": "host perf_counter around K steps (produce + push + advance) and finalize, ended by "
          "torch.cuda.synchronize on every device; W warm-up steps before", "torch": torch.__version__})
    first = None
    layouts = [([0], 0, "device"), ([0], 0, "borrow")]
    for n in (2, 4, 8):
        ids = [i % ndev for i in range(n)]           # fewer GPUs than n: ids repeat, and the row says so
        for chunk in (0, args.chunk):
            layouts += [(ids, chunk, "device"), (ids, chunk, "host")]
    for ids, chunk, source in layouts:
        row, pts = run(ids, chunk, source, ring)
        if first is None:
            first = pts
        row["points_equal_first_row"] = bool(len(pts) == len(first) and pts.tobytes() == first.tobytes())
        emit(row)
L.lib().ftkb_host_free(host_p)

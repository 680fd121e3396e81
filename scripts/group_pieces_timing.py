#!/usr/bin/env python
"""Snapshots in pieces on several devices (ftkb_group_push_pieces_device, DESIGN.md 7.1): ms per step of the C3 shape (512^3
moving extremum, synthetic.hh:332-354 with C3's x0 / dir) on one device group, fed three ways from torch producers that write
every snapshot on a producer stream (no host synchronise):
  - pieces: the producer is decomposed like the group -- piece s holds the planes slab s owns (ftkb_group_get_slab of a z-slab
    group on the same device list, also for time chunks) and is written on device_ids[s]; every context copies the planes it
    needs from the pieces that hold them;
  - device: the whole snapshot is written on device 0 and every context copies its planes from there;
  - host: the snapshot is written on device 0 and copied to page-locked host memory (that D2H is inside the timed window: a
    producer on a GPU pays it), then ftkb_group_push_snapshot sends it over PCIe.
The group runs as z-slabs and as time chunks of 8.  With fewer GPUs than --devices the ids repeat (ids i mod N, recorded in
every row): the contexts then share the GPUs, and copies between "devices" stay on one GPU.  The three feeds alternate,
--rounds times, in the same run, in reverse order in odd rounds.  Every row times the same series: a host clock around K timed steps plus finalize, ended by a
synchronise of every device, after W warm-up steps; the points of every row must equal those of the first row.  Bytes copied
across devices (different device ids) and within a device (same id) per timed step are counted on the host from the copy
plan the library follows.  The card's name and power limit are read in the same run.
    python scripts/group_pieces_timing.py [--dims 512 512 512] [--devices 8] [--steps 60] [--warmup 4] [--out FILE.jsonl]"""
import argparse
import contextlib
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
from ftk_b200 import _lib as L  # noqa: E402
from ftk_b200.group import GroupTracker  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--dims", type=int, nargs=3, default=[512, 512, 512])
ap.add_argument("--devices", type=int, default=8)
ap.add_argument("--steps", type=int, default=60)
ap.add_argument("--warmup", type=int, default=4)
ap.add_argument("--chunk", type=int, default=8)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_group_pieces.jsonl"))
args = ap.parse_args()
dims, K, W, B = args.dims, args.steps, args.warmup, args.chunk
T = W + K
ndev = torch.cuda.device_count()
if ndev == 0:
    sys.exit("no CUDA device: this script measures on the GPU only")
ids = [i % ndev for i in range(args.devices)]
x0 = [dims[0] / 2 + 0.3, dims[1] / 2 - 0.3, dims[2] / 2 + 0.1]      # C3: [256.3, 255.7, 256.1] at 512^3
d = [0.1, 0.11, 0.1]
shape = tuple(reversed(dims))
D, plane_bytes = dims[2], 8 * dims[0] * dims[1]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpus_visible": ndev, "nvidia_smi": [l.strip() for l in q.stdout.strip().splitlines()], "torch_name": torch.cuda.get_device_name(0)}


# ---- the producers: torch on every physical device, each on a producer stream of its own ----------------------------------------
prod, axes = {}, {}
for dev in sorted(set(ids)):
    prod[dev] = torch.cuda.Stream(device=dev)
    with torch.cuda.device(dev), torch.cuda.stream(prod[dev]):
        axes[dev] = [torch.arange(n, dtype=torch.float64, device=f"cuda:{dev}") for n in shape]


def produce(k, outs):
    """snapshot k of the moving extremum into outs = [(tensor, device, first plane)], enqueued on each device's producer
    stream.  Every device computes the separable terms once per snapshot, then one add per output writes its planes, so the
    whole-array producer and the decomposed one do the same arithmetic"""
    terms = {}
    for out, dev, z0 in outs:
        with torch.cuda.device(dev), torch.cuda.stream(prod[dev]):
            if dev not in terms:
                zs, ys, xs = axes[dev]
                terms[dev] = (((xs - (x0[0] + d[0] * k)) ** 2)[None, :] + ((ys - (x0[1] + d[1] * k)) ** 2)[:, None],
                              (zs - (x0[2] + d[2] * k)) ** 2)
            p, zt = terms[dev]
            torch.add(p[None], zt[z0:z0 + out.shape[0], None, None], out=out)


@contextlib.contextmanager
def producer_streams():
    """torch's current stream on every device is its producer stream (the group orders its copies after it)"""
    with contextlib.ExitStack() as st:
        for dev, s in prod.items():
            st.enter_context(torch.cuda.device(dev))
            st.enter_context(torch.cuda.stream(s))
        yield


def sync_all():
    for i in range(ndev):
        torch.cuda.synchronize(i)


def slab_cuts():
    g = GroupTracker(dims, ids, field="scalar", chunk=0)
    slabs = [g.slab(s) for s in range(len(ids))]
    g.close()
    return [0] + [sl[0] for sl in slabs[1:]] + [D], slabs


CUTS, SLABS = slab_cuts()
PIECES = [(CUTS[s], CUTS[s + 1], ids[s]) for s in range(len(ids))]      # (first, end, device)


def plan_bytes(chunk, feed):
    """bytes per timed step copied (across devices, within a device, host to device), from the plan the library follows"""
    src = PIECES if feed == "pieces" else [(0, D, ids[0] if feed == "device" else -1)]
    across = within = h2d = 0

    def copy(lo, hi, dst):
        nonlocal across, within, h2d
        for a, b, dev in src:
            n = max(0, min(hi, b) - max(lo, a)) * plane_bytes
            if dev < 0:
                h2d += n
            elif dev == dst:
                within += n
            else:
                across += n
    for k in range(W, T):
        if chunk == 0:
            for s, (_, _, a0, a1) in enumerate(SLABS):
                copy(a0, a1 + 1, ids[s])
            continue
        c = k // chunk
        copy(0, D, ids[c % len(ids)])                  # the chunk's context, or the staging buffers of a new chunk
        if k % chunk == 0 and k > 0:
            copy(0, D, ids[(c - 1) % len(ids)])        # the halo layer of the chunk before
            within += D * plane_bytes                  # staged layer -> the new chunk's context
    return {"bytes_across_devices_per_step": across / K, "bytes_within_device_per_step": within / K, "bytes_h2d_per_step": h2d / K}


def run(chunk, feed):
    g = GroupTracker(dims, ids, field="scalar", chunk=chunk)
    d2h = 0.0
    push = {}                  # timed step -> seconds inside the push call

    def step(k):
        nonlocal d2h
        if feed == "pieces":
            produce(k, [(buf, dev, a) for (a, b, dev), buf in zip(PIECES, piece_bufs)])
            t = time.perf_counter()
            with producer_streams():
                g.push_field_data_snapshot_pieces(scalar=piece_bufs)
        else:
            produce(k, [(whole_buf, ids[0], 0)])
            if feed == "host":
                t = time.perf_counter()
                with torch.cuda.device(ids[0]), torch.cuda.stream(prod[ids[0]]):
                    host_t.copy_(whole_buf, non_blocking=True)
                prod[ids[0]].synchronize()
                d2h += time.perf_counter() - t
                t = time.perf_counter()
                g.push_scalar_field_snapshot(host_a)
            else:
                t = time.perf_counter()
                with producer_streams():
                    g.push_scalar_field_snapshot(whole_buf)
        push[k] = time.perf_counter() - t
        if k:
            g.advance_timestep()
        if k == T - 1:
            g.update_timestep()

    for k in range(W):
        step(k)
    sync_all()
    d2h = 0.0
    push.clear()
    t0 = time.perf_counter()
    for k in range(W, T):
        step(k)
    root = g.finalize()
    sync_all()
    dt = time.perf_counter() - t0
    pts = root.get_discrete_critical_points().copy()
    g.close()
    row = {"devices": ids, "gpus_visible": ndev, "mode": "z-slabs" if chunk == 0 else f"time chunks of {chunk}", "input": feed,
           "dims": dims, "steps": K, "warmup": W, "ms_per_step": 1e3 * dt / K, "push_call_ms_per_step": 1e3 * sum(push.values()) / K, "punctured_simplices": int(len(pts))}
    # where the push time goes: time chunks stage the first layer of every chunk (k % chunk == 0), the other steps do not
    ms = {k: 1e3 * v for k, v in push.items()}
    first_of_chunk = [v for k, v in ms.items() if chunk and k % chunk == 0]
    other = [v for k, v in ms.items() if not (chunk and k % chunk == 0)]
    row["push_ms_median_other_steps"] = float(np.median(other))
    row["push_ms_max_other_steps"] = max(other)
    if first_of_chunk:
        row["push_ms_median_first_layer_of_chunk"] = float(np.median(first_of_chunk))
        row["push_ms_max_first_layer_of_chunk"] = max(first_of_chunk)
    row["push_steps_over_4x_median"] = sum(v > 4 * row["push_ms_median_other_steps"] for v in ms.values())
    if feed == "pieces":
        row["pieces"] = [list(p) for p in PIECES]
    if feed == "host":
        row["d2h_ms_per_step"] = 1e3 * d2h / K
    row.update(plan_bytes(chunk, feed))
    return row, pts


def pinned(n):
    p = C.c_void_p()
    assert L.lib().ftkb_host_alloc(n * 8, C.byref(p)) == 0
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(n,)).reshape(shape), p


host_a, host_p = pinned(int(np.prod(shape)))
host_t = torch.from_numpy(host_a)
whole_buf = torch.empty(shape, dtype=torch.float64, device=f"cuda:{ids[0]}")
piece_bufs = [torch.empty((b - a,) + shape[1:], dtype=torch.float64, device=f"cuda:{dev}") for a, b, dev in PIECES]
info = card()
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
with open(args.out, "w") as f:
    def emit(row):
        line = json.dumps(row)
        print(line, flush=True)
        f.write(line + "\n")
        f.flush()

    emit({"card": info, "timing": "host perf_counter around K steps (produce + push + advance) and finalize, ended by "
          "torch.cuda.synchronize on every device; W warm-up steps before; feeds alternate within each round, in reverse order in odd rounds", "torch": torch.__version__,
          "multi_gpu": "measured" if ndev > 1 else "not measured: one GPU visible, device ids repeat, no copy crosses devices"})
    first = None
    for rnd in range(args.rounds):
        for chunk in (0, B):
            for feed in ("pieces", "device", "host")[::1 if rnd % 2 == 0 else -1]:
                row, pts = run(chunk, feed)
                if first is None:
                    first = pts
                row["round"] = rnd
                row["points_equal_first_row"] = bool(len(pts) == len(first) and pts.tobytes() == first.tobytes())
                emit(row)
L.lib().ftkb_host_free(host_p)

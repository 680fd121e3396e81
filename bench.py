#!/usr/bin/env python
"""bench.py -- space-time simplices tested per second (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5|woven] [--impl reference] [--dump-outputs DIR]

One "step" = one advance_timestep of the tracker on one new snapshot: field derivation (gradient +
min non-zero |v|), quantisation factor, ordinal sweep at t and interval sweep over [t, t+1]
(scan + per-simplex test kernels), i.e. 12 (2D) / 60 (3D) enumerated simplices per domain corner.

Default workload = BASELINE.json configs[1]: moving-extremum 2D scalar field 8192 x 8192, 64 distinct
timesteps resident in HBM (the sweep ping-pongs through them when K > 63).  `value` is measured
with the snapshots already resident in HBM (borrowed in place through the C ABI); `e2e` repeats the
measurement through the same C-ABI calls with pinned HOST buffers (H2D of every snapshot inside
the timed region).

N > 1: one process per GPU, each rank owns a contiguous time slab of K steps (weak scaling).  The
slab's last sweep reads the first layer of the next slab in place through NVLink peer memory (range
cells + the sparse vertices around surviving cubes; FTKB_HALO=nccl copies the layer with
ncclSend/ncclRecv inside the timed region instead).  The timed region is the K sweeps of every rank
between two barriers (device time, max over ranks); the once-per-slab epilogue -- one packed
all_gather of the slab minima of min non-zero |v|, checked against the running quantisation factor --
runs right after the stopwatch and is reported as `slab_epilogue_ms`.  Finalize (union-find + trace
ordering) is reported separately.

Every default line also carries `scaling_c4` / `scaling_c3` (BASELINE configs[3] and [2]: the
1024^3 vector field and the 512^3 scalar field at the same N, fewer steps) and `dense_woven` (a
feature-dense 2D field), so that one driver run records the scaling curve of the configurations
north_star names.  --only-main skips them.

--impl reference times the unmodified reference CPU tracker (oracle/_ref/ftk_ref_oracle, built from
/root/reference by oracle/build_ref.sh) on a bounded sample of the same workload.

--dump-outputs DIR writes what a caller of the timed path receives after its last step: the punctured simplices the
tracker of the main workload holds then (DIR/points_<field>.npy, float64, one file per field of the point record).  The
inputs are generated without randomness, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (workload label, dims, generator params x0+dir, distinct timesteps resident)
    "c2": ("moving_extremum_2d_scalar_8192x8192x64", [8192, 8192], [4096.3, 4095.7, 0.1, 0.1], 64),
    "c3": ("moving_extremum_3d_scalar_512x512x512x32", [512, 512, 512], [256.3, 255.7, 256.1, 0.1, 0.11, 0.1], 32),
    "c2s": ("moving_extremum_2d_scalar_2048x2048x16", [2048, 2048], [1024.3, 1023.7, 0.1, 0.1], 16),
    # vector input (field GIVEN, Jacobian derived at punctured simplices): BASELINE configs[3] and configs[4]
    "c4": ("unsteady_abc_3d_vector_1024x1024x1024x64", [1024, 1024, 1024], None, 4),      # 25.8 GB per layer: 4 distinct layers resident
    "c5": ("double_gyre_2d_vector_16384x8192x256", [16384, 8192], None, 32),
    "c4s": ("unsteady_abc_3d_vector_256x256x256x64", [256, 256, 256], None, 8),
    # feature-dense scalar field (thousands of critical points per layer): the scan's cold path and the test kernel carry weight
    "woven": ("spiral_woven_2d_scalar_8192x8192x16", [8192, 8192], None, 16),
    "wovens": ("spiral_woven_2d_scalar_1024x1024x8", [1024, 1024], None, 8),
}
VECTOR_CONFIGS = ("c4", "c5", "c4s")
WOVEN_CONFIGS = ("woven", "wovens")
METRIC = "space_time_simplices_tested_per_sec"
UNIT = "simplices/s"
# --dump-outputs: a point is 14 float64 values (112 bytes); counting 128 bytes a point leaves room for the .npy headers
# and keeps a dump under 64 MB
DUMP_POINTS_MAX = (64 << 20) // 128


def tri(g, period):
    """ping-pong index 0..period-1..0 so that the field keeps moving continuously"""
    m = 2 * (period - 1)
    g = g % m
    return g if g < period else m - g


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons of one GPU through NVML while the timed region runs"""

    def __init__(self, index, enabled=True):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.nv = None
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ---------------------------------------------------------------------------------------------------
# the reference's CPU tracker (oracle/_ref, unmodified headers) on a bounded sample of a workload
# ---------------------------------------------------------------------------------------------------
def _ref_sample_cmd(config, scale):
    """(command line of oracle/_ref/ftk_ref_oracle, simplices it enumerates, description) for a reduced extent of `config`"""
    label, dims, params, _ = CONFIGS[config]
    nd = len(dims)
    cores = os.cpu_count() or 1
    binary = os.path.join(ROOT, "oracle", "_ref", "ftk_ref_oracle")
    vector = config in VECTOR_CONFIGS
    T = scale["T"]
    sdims = scale["dims2"] if nd == 2 else scale["dims3"]
    if config == "c5":
        sdims = [2 * sdims[0], sdims[1]]
    margin = 2 if vector else 3
    ncore = 1
    for d in sdims:
        ncore *= d - margin
    simplices = ncore * ((12 * (T - 1) + 2) if nd == 2 else (60 * (T - 1) + 6))
    cmd = [binary, "--nd", str(nd), "--nv", str(nd if vector else 1), "--dims"] + [str(d) for d in sdims] + ["--nt", str(T)]
    if config in WOVEN_CONFIGS:
        cmd += ["--gen", "woven"]
        gen = "woven"
    elif config == "c5":
        cmd += ["--gen", "double_gyre"]
        gen = "double_gyre"
    elif vector:
        cmd += ["--gen", "abc"]
        gen = "abc (unsteady amplitude)"
    else:
        sp = [d / 2 + 0.3 for d in sdims] + list(params[nd:])
        cmd += ["--gen", "moving_extremum", "--p"] + [repr(float(v)) for v in sp]
        gen = "moving_extremum"
    cmd += ["--no-trace", "--quiet", "--nthreads", str(cores)]
    sample = f"{gen} {'x'.join(map(str, sdims))}x{T} timesteps, {cores} threads"
    return cmd, simplices, sample, cores, os.path.exists(binary)


def _run_ref(cmd, timeout=900):
    out = subprocess.run(cmd, check=True, capture_output=True, timeout=timeout).stdout.decode().strip().splitlines()[-1]
    return json.loads(out)


def reference_arm(args, rank):
    """the unmodified reference CPU tracker on a bounded sample of the workload (rank 0 only)"""
    if rank != 0:
        return
    label = CONFIGS[args.config][0]
    # one step = the reference's tracker loop over 2 snapshots of a reduced extent of the same generator
    cmd, simplices, sample, cores, have = _ref_sample_cmd(args.config, {"T": 2, "dims2": [512, 512], "dims3": [48, 48, 48]})
    kind = "reference" if have else "port"

    def one_step():
        t0 = time.perf_counter()
        if have:
            st = _run_ref(cmd)
            t_path = st["t_push"] + st["t_sweep"]            # derive + sweep: the hot path
            assert int(st["simplices"]) == simplices, (st["simplices"], simplices)
        else:
            from oracle import cp_oracle as O               # plain-C port of the reference path
            _, dims, params, _ = CONFIGS["c2"]
            sdims = [512, 512]
            sp = [d / 2 + 0.3 for d in sdims] + list(params[2:])
            snaps = [O.gen_moving_extremum(sdims, sp[:2], sp[2:], float(k)) for k in range(2)]
            t1 = time.perf_counter()
            O.track(snaps, sdims, field="scalar", trace=False)
            t_path = time.perf_counter() - t1
        return t_path, time.perf_counter() - t0

    for _ in range(args.warmup):
        one_step()
    tot = wall = 0.0
    for _ in range(args.steps):
        a, b = one_step()
        tot += a
        wall += b
    value = simplices * args.steps / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64+int64", "data": "synthetic",
        "config": {"workload": label, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_ms_per_step": 1e3 * wall / args.steps,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(config):
    """bounded sample (about 10-30 s of CPU work) of the reference CPU tracker on this box's host cores"""
    # sized for about 10 s of wall clock on 16 host threads (the earlier 1536^2 / 96^3 sample took 3.8 s)
    cmd, simplices, sample, cores, have = _ref_sample_cmd(config, {"T": 3, "dims2": [2560, 2560], "dims3": [128, 128, 128]} if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ftk_ref_oracle"))
                                                          else {"T": 3, "dims2": [1536, 1536], "dims3": [96, 96, 96]})
    try:
        if have:
            st = _run_ref(cmd)
            return {"value": st["simplices"] / (st["t_push"] + st["t_sweep"]), "unit": UNIT, "cores": cores, "kind": "reference",
                    "sample": sample, "t_derive_s": st["t_push"], "t_sweep_s": st["t_sweep"]}
        if config in VECTOR_CONFIGS or config in WOVEN_CONFIGS:
            return {"value": None, "unit": UNIT, "cores": cores, "kind": "unavailable", "sample": "oracle/_ref missing"}
        from oracle import cp_oracle as O
        _, dims, params, _ = CONFIGS[config]
        nd = len(dims)
        sdims = [1536, 1536] if nd == 2 else [96, 96, 96]
        sp = [d / 2 + 0.3 for d in sdims] + list(params[nd:])
        snaps = [O.gen_moving_extremum(sdims, sp[:nd], sp[nd:], float(k)) for k in range(3)]
        t0 = time.perf_counter()
        O.track(snaps, sdims, field="scalar", trace=False)
        dt = time.perf_counter() - t0
        return {"value": simplices / dt, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}
    except Exception as e:  # the baseline is reported, never required
        return {"value": None, "unit": UNIT, "cores": cores, "kind": "unavailable", "sample": f"failed: {e}"}


# ---------------------------------------------------------------------------------------------------
# one workload on this rank's GPU
# ---------------------------------------------------------------------------------------------------
class Env:
    pass


def generate_layers(env, config):
    import torch
    label, dims, params, NL = CONFIGS[config]
    nd = len(dims)
    dev = env.dev
    vector = config in VECTOR_CONFIGS
    x0, dirv = (params[:nd], params[nd:]) if params else (None, None)

    def gen_layer(j):
        """synthetic_moving_extremum at time j (ref: synthetic.hh:332-354), memory order ([D,]H,W)"""
        axes = [torch.arange(d, dtype=torch.float64, device=dev) for d in dims]
        e = [(axes[q] - (x0[q] + dirv[q] * float(j))) ** 2 for q in range(nd)]
        if nd == 2:
            s = e[0][None, :] + e[1][:, None]
        else:
            s = (e[0][None, None, :] + e[1][None, :, None]) + e[2][:, None, None]
        return s.contiguous()

    def gen_woven(j):
        """synthetic_woven (synthetic.hh:32-48, scaling factor 15), t = j / (NL - 1) + 1e-4 (synthetic.hh:90-109)"""
        t = j / (NL - 1) + 1e-4
        x = ((torch.arange(dims[0], dtype=torch.float64, device=dev) / (dims[0] - 1)) - 0.5) * 15
        y = ((torch.arange(dims[1], dtype=torch.float64, device=dev) / (dims[1] - 1)) - 0.5) * 15
        a = x[None, :] * math.cos(t) - y[:, None] * math.sin(t)
        b = x[None, :] * math.sin(t) + y[:, None] * math.cos(t)
        return (torch.cos(a) * torch.sin(b)).contiguous()

    def gen_vector_layer(j):
        """C5: synthetic_double_gyre(time = 0.1 j) (synthetic.hh:130-150,193-217); C4: synthetic_abc_flow (synthetic.hh:239-260)
        with A(j) = sqrt(3) + 0.5 (j/64) sin(pi j/64) (SURVEY.md 8d: the time dependence is ours); memory order ([D,]H,W,n)"""
        out = torch.empty(tuple(reversed(dims)) + (nd,), dtype=torch.float64, device=dev)
        ax = [torch.arange(d, dtype=torch.float64, device=dev) / (d - 1) for d in dims]
        if nd == 2:
            A, omega, eps, t = 0.1, 2 * math.pi, 0.25, 0.1 * j
            x, y = ax[0] * 2, ax[1]
            a, b = eps * math.sin(omega * t), 1 - 2 * eps * math.sin(omega * t)
            f, dfdx = a * x * x + b * x, 2 * a * x + b
            out[..., 0] = (-math.pi * A * torch.sin(math.pi * f))[None, :] * torch.cos(math.pi * y)[:, None]
            out[..., 1] = (math.pi * A * torch.cos(math.pi * f) * dfdx)[None, :] * torch.sin(math.pi * y)[:, None]
        else:
            A, B, Cc = math.sqrt(3.0) + 0.5 * (j / 64.0) * math.sin(math.pi * j / 64.0), math.sqrt(2.0), 1.0
            x, y, z = (a * 2 * math.pi for a in ax)
            for k0 in range(0, dims[2], 64):       # slabs of 64 planes keep the temporaries small next to 25.8 GB layers
                zs = z[k0:k0 + 64]
                o = out[k0:k0 + 64]
                o[..., 0] = (A * torch.sin(zs))[:, None, None] + (Cc * torch.cos(y))[None, :, None]
                o[..., 1] = (B * torch.sin(x))[None, None, :] + (A * torch.cos(zs))[:, None, None]
                o[..., 2] = (Cc * torch.sin(y))[None, :, None] + (B * torch.cos(x))[None, None, :]
        return out

    g = gen_vector_layer if vector else (gen_woven if config in WOVEN_CONFIGS else gen_layer)
    layers = [g(j) for j in range(NL)]
    torch.cuda.synchronize()
    return layers


def dump_points(out_dir, pts):
    """the punctured simplices in the element order the library returns them, one float64 array per field of the point
    record; above DUMP_POINTS_MAX a fixed, seeded sample of them, still in that order"""
    import numpy as np
    if len(pts) > DUMP_POINTS_MAX:
        pts = pts[np.sort(np.random.default_rng(0).choice(len(pts), DUMP_POINTS_MAX, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for field in pts.dtype.names:
        np.save(os.path.join(out_dir, f"points_{field}.npy"), pts[field].astype(np.float64))


def run_config(env, config, K, W, e2e_steps, sample_clocks, dump_dir=None):
    """time K sweeps of `config` on this rank (after W warm-up sweeps); returns the rank-0 record.  dump_dir: write the
    punctured simplices the tracker holds after its last timed sweep there (dump_points)"""
    import numpy as np
    import torch
    import ftk_b200
    from ftk_b200 import _lib
    dist, rank, world, local, dev = env.dist, env.rank, env.world, env.local, env.dev
    label, dims, params, NL = CONFIGS[config]
    nd = len(dims)
    vector = config in VECTOR_CONFIGS
    ncore = 1
    for d in dims:
        ncore *= d - (2 if vector else 3)      # json_interface.hh:639-654: [1, D-2] for vector input, [2, D-2] for scalar input
    per_step = ncore * (12 if nd == 2 else 60)
    nvert = int(np.prod(dims))
    layers = generate_layers(env, config)
    g0 = rank * (W + K)
    fld = "vector" if vector else "scalar"

    def make():
        return ftk_b200.make_tracker(dims, field=fld, device=local, start_timestep=g0)

    def push_ptr(t, ptr):
        if vector:
            t.push_device_pointers(vector=ptr)
        else:
            t.push_device_pointers(scalar=ptr)

    # ---- device-resident measurement -------------------------------------------------------------
    tr = make()
    ptrs = [int(l.data_ptr()) for l in layers]     # resident layers are borrowed in place through the C ABI
    push_ptr(tr, ptrs[tri(g0, NL)])
    # N > 1, halo through NVLink peer memory (default; FTKB_HALO=nccl copies the layer with ncclSend/Recv instead): the slab
    # below needs this rank's first layer only for its last sweep, and of it only the 16-byte range cells and the vertices
    # around the surviving cubes -- the owner exports IPC handles of the layer and of its cells, the neighbour maps them and
    # pushes the layer as a remote snapshot (ftkb_push_snapshot_remote): nothing is copied.  Handle exchange and mapping are
    # set-up (once per run), like NCCL's channel set-up; they stay outside the timed region.
    peer = None
    first_done = False
    if dist and os.environ.get("FTKB_HALO", "peer") == "peer":
        mine = None
        try:
            push_ptr(tr, ptrs[tri(g0 + 1, NL)])
            tr.update_timestep()                         # the sweep that builds the cells of this rank's first layer
            cptr, cbytes, cres = tr.export_layer_cells(0)
            mine = (_lib.ipc_export(ptrs[tri(g0, NL)]), _lib.ipc_export(cptr), cres)
        except _lib.FTKBError:
            mine = None
        tr.advance_timestep()                            # warm-up step 0 completes (repeated sweep from the cells, layer popped)
        first_done = True
        allh = [None] * world
        dist.all_gather_object(allh, mine)
        if all(h is not None for h in allh):
            try:
                if rank < world - 1:
                    lh, ch, cres = allh[rank + 1]
                    peer = (_lib.ipc_import(lh, local), _lib.ipc_import(ch, local), cres)
                else:
                    peer = ()
            except _lib.FTKBError:
                peer = None
        oks = [None] * world
        dist.all_gather_object(oks, peer is not None)
        if not all(oks):
            peer = None          # some rank could not export / map: every rank copies the halo with NCCL instead
    use_peer = peer is not None
    for i in range(1 if first_done else 0, W):
        push_ptr(tr, ptrs[tri(g0 + i + 1, NL)])
        tr.advance_timestep()
    halo = None
    sampler = ClockSampler(physical_gpu_index(local), enabled=sample_clocks and rank == 0)
    torch.cuda.synchronize()
    tr.synchronize()
    warm = tr.stats()                                    # running minimum / factor after the warm-up sweeps (confirms them all)

    def exchange_halo():
        """one-layer halo: the first layer of the next slab (ncclSend/ncclRecv over NVLink), one batched P2P group"""
        ops = []
        if rank > 0:
            ops.append(dist.P2POp(dist.isend, layers[tri(g0, NL)], rank - 1))
        if rank < world - 1:
            ops.append(dist.P2POp(dist.irecv, halo, rank + 1))
        return dist.batch_isend_irecv(ops) if ops else []

    packed = None
    if dist:
        # untimed: NCCL sets its peer-to-peer channels up lazily on first use (hundreds of ms); the timed exchange
        # below then moves the halo over warm channels, as every exchange after the first would in a long run
        if not use_peer:
            if rank < world - 1:
                halo = torch.empty_like(layers[0])
            for r in exchange_halo():
                r.wait()
        packed = torch.zeros(world * 2, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(packed, torch.zeros(2, dtype=torch.float64, device=dev))
        tmax = torch.zeros(1, dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        torch.cuda.synchronize()
        dist.barrier()
    tr.reset_stats()
    sampler.start()
    tr.timer_start()
    reqs = exchange_halo() if (dist and not use_peer) else []     # inside the timed region
    for i in range(W, W + K):
        nxt = ptrs[tri(g0 + i + 1, NL)]
        if use_peer and peer and i == W + K - 1:
            # the slab's last sweep: the next slab's first layer stays where it is, in the neighbour GPU's memory
            if vector:
                tr.push_remote_snapshot(vector=peer[0], cells=peer[1], resolution=peer[2])
            else:
                tr.push_remote_snapshot(scalar=peer[0], cells=peer[1], resolution=peer[2])
            tr.advance_timestep()
            continue
        if halo is not None and i == W + K - 1:
            for r in reqs:
                r.wait()
            torch.cuda.current_stream().synchronize()
            nxt = int(halo.data_ptr())
        push_ptr(tr, nxt)
        tr.advance_timestep()
    for r in reqs:
        r.wait()
    ms = tr.timer_stop()                                 # device time of this rank's K sweeps (both streams of the context)
    sampler.stop_flag = True
    t_epi = time.perf_counter()
    st = tr.stats()
    redo = 0
    if dist:
        # once per slab, right after the sweeps: the slab minima of min non-zero |v| in ONE packed all_gather and one D2H copy.
        # The reference's factor is a running quantity; a slab swept optimistically with its own minimum: had the exclusive
        # prefix over the earlier slabs changed the factor of any of its sweeps, the slab would be swept again with
        # resolution_init = prefix (moving-extremum / ABC / double-gyre slabs never differ).
        mine = torch.tensor([st["resolution"], ms], dtype=torch.float64).to(dev)
        dist.all_gather_into_tensor(packed, mine)
        host = packed.cpu().numpy().reshape(world, 2)
        ms = float(host[:, 1].max())                     # max over ranks
        prefix = min([float(v) for v in host[:rank, 0]] + [float("inf")])

        def nbits(res):
            return max(8, min(int(math.ceil(math.log2(1.0 / res))), 21)) if res > 0 and math.isfinite(res) else 8
        if prefix < float("inf") and nbits(prefix) > nbits(warm["resolution"]):
            redo = K                                     # (upper bound: sweeps whose running minimum was still above the prefix)
        dist.barrier()
    epilogue_ms = 1e3 * (time.perf_counter() - t_epi)
    torch.cuda.synchronize()
    sampler.join(timeout=1.0) if sampler.is_alive() else None

    # ---- finalize (not part of a step; reported separately) --------------------------------------
    t0 = time.perf_counter()
    pts = tr.get_discrete_critical_points()
    if dist:
        gathered = [None] * world
        dist.all_gather_object(gathered, pts.tobytes())
        if rank == 0:
            for b in gathered[1:]:
                tr.import_points(np.frombuffer(b, dtype=_lib.POINT_DTYPE))
    ntraj = npts_total = None
    fin = {}
    if rank == 0:
        before = tr.stats()
        tr.finalize()
        ntraj = len(tr.get_trajectory_index())
        npts_total = len(tr.get_discrete_critical_points())
        after = tr.stats()
        fin = {"device": after["ms_finalize_device"] - before["ms_finalize_device"], "host": after["ms_finalize_host"] - before["ms_finalize_host"],
               # wall clock inside the library: sort + dedup + copy of the punctured simplices, then neighbour search + union-find + ordering
               "library": after["ms_sort_wall"] + after["ms_trace_wall"]}
    finalize_ms = 1e3 * (time.perf_counter() - t0)
    tr.close()
    if dump_dir and rank == 0:
        dump_points(dump_dir, pts)

    # ---- end-to-end measurement: host buffers through the same C-ABI calls ------------------------
    ms2, E, st2 = None, 0, None
    if e2e_steps > 0:
        E = max(1, min(e2e_steps, K))
        NH = min(8, NL) if layers[0].numel() * 8 < (4 << 30) else 2      # pinned host copies: two are enough for 25.8 GB layers
        E = E if NH > 2 else min(E, 2)
        host = [torch.empty(tuple(layers[0].shape), dtype=torch.float64).pin_memory() for _ in range(NH)]
        for j in range(NH):
            host[j].copy_(layers[j])
        torch.cuda.synchronize()
        if NH == 2:       # 25.8 GB layers: the context's own copies need the room the resident series occupied
            layers = []
            ptrs = []
            torch.cuda.empty_cache()
        tr2 = make()

        def push_host(t, a):
            if vector:
                t.push_vector_field_snapshot(a)
            else:
                t.push_scalar_field_snapshot(a)

        push_host(tr2, host[0].numpy())
        for i in range(3):
            push_host(tr2, host[tri(i + 1, NH)].numpy())
            tr2.advance_timestep()
        tr2.synchronize()
        if dist:
            dist.barrier()
        tr2.reset_stats()
        tr2.timer_start()
        for i in range(3, 3 + E):
            push_host(tr2, host[tri(i + 1, NH)].numpy())   # H2D inside the timed region
            tr2.advance_timestep()                                         # counters + resolution read back every step
        ms2 = tr2.timer_stop()
        if dist:
            t = torch.tensor([ms2], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms2 = float(t.item())
        st2 = tr2.stats()
        tr2.close()
        del host
    del layers
    torch.cuda.empty_cache()

    if rank != 0:
        return None
    peak, peak_src = measured_peaks()
    nscan = max(int(st["scan_launches"]), 1)
    scan_ms = st["ms_scan"] / nscan
    fused = (not vector) and st["ms_derive"] == 0.0   # scalar input: gradient fused into the scan, the vector field is never materialised
    # the default scans stream ONE layer per step and read / write 16-byte range cells for the other (DESIGN.md 4.2);
    # FTKB_SCAN2D / FTKB_SCAN3D / FTKB_VSCAN = twolayer select the kernels that re-read both layers
    twolayer = os.environ.get("FTKB_VSCAN" if vector else ("FTKB_SCAN2D" if nd == 2 else "FTKB_SCAN3D"), "") in ("twolayer", "plain") \
        or os.environ.get("FTKB_SCAN", "tile") != "tile"
    layer_bytes = nvert * (nd if vector or not fused else 1) * 8
    cell_bytes = nvert * (2.1 if nd == 3 else (1.04 if not vector else 1.03))
    hit_bytes = 72 * (st["points"] / max(K, 1))
    # algorithmic bytes of one scan launch as THIS design moves them: the new layer once, its cells written, the current
    # layer's cells read (two-layer kernels: both layers); the measured DRAM traffic (ncu) is reported next to it
    alg_bytes = (2 * layer_bytes if twolayer else layer_bytes + 2 * cell_bytes) + hit_bytes
    achieved = alg_bytes / (scan_ms * 1e-3) / 1e9
    # the streaming-operator contract of SURVEY.md 8(d): two materialised fp64 vector layers per step (2.667 B/simplex in 2D, 0.8 in 3D)
    survey_bytes = (32.0 / 12.0 if nd == 2 else 48.0 / 60.0) * per_step
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "scan_traffic.json")) as f:
            traffic = json.load(f).get(config)
    except Exception:
        pass
    if twolayer:
        traffic = None
    if vector:
        kname = ("scan2d_kernel<true>" if nd == 2 else "scan3d_kernel<true>") if twolayer else \
                ("vscan2d_build_kernel<1,true>" if nd == 2 else "vscan3d_build_kernel<1,true>")
    elif nd == 2:
        kname = "scan2d_tile_kernel<true>" if twolayer else \
                ("scan2d_build_kernel<1,true>" if os.environ.get("FTKB_SCAN2D", "") == "f32" else "scan2d_keys_build_kernel<1,true>")
    else:
        kname = ("scan3d_fused_kernel<true>" if fused else "scan3d_kernel<true>") if twolayer else "scan3d_build_kernel<1,true>"
    line = {
        "metric": METRIC, "value": per_step * K * world / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64+int64", "data": "synthetic",
        "config": {"workload": label, "simplices_per_step_per_gpu": per_step, "layers_resident": NL,
                   "l2": "inputs larger than L2 (each fp64 layer >= 0.5 GB; no flush needed)",
                   "parallelism": f"time-slab x{world}" if world > 1 else "single GPU",
                   "halo": (("nvlink peer memory: the next slab's first layer is read in place (range cells + sparse vertices), nothing copied"
                             if use_peer else "ncclSend/ncclRecv of the next slab's first layer, inside the timed region") if world > 1 else None),
                   "step": "one advance_timestep: gradient + min|v| + range cells + exact sign early-out (fused scan kernel) + per-simplex test kernel" if fused else
                           "one advance_timestep: min|v| + range cells + exact sign early-out (scan kernel) + per-simplex test kernel",
                   "steps_enqueued_ahead": os.environ.get("FTKB_DEFER", "1") != "0"},
        "roofline": {"bound": "hbm", "kernel": kname,
                     # frac = bytes this launch really moves / launch time / measured copy bandwidth.  `achieved` counts the
                     # design's own algorithmic bytes (one layer + cells in and out); `traffic` is ncu's dram bytes per launch
                     # of the same kernel (profiles/scan_traffic.json) -- the two agree within a few per cent.
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_gbs": (traffic / (scan_ms * 1e-3) / 1e9) if traffic else None,
                     "traffic_frac": (traffic / (scan_ms * 1e-3) / 1e9 / peak) if traffic else None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": scan_ms,
                     "launches_timed": nscan, "sweeps_repeated": int(st["sweeps_repeated"]),
                     "survey_8d_contract": {"bytes_per_launch": survey_bytes, "gbs": survey_bytes / (scan_ms * 1e-3) / 1e9,
                                            "frac": survey_bytes / (scan_ms * 1e-3) / 1e9 / peak,
                                            "note": "SURVEY.md 8(d) counts two materialised fp64 vector layers per step; this design reads one "
                                                    "layer (the scalar itself for scalar input) + 16-byte range cells, so the contract figure can exceed 1"},
                     "note": "rank 0; tensor cores unused by design (no dense contraction on this path)"},
        "kernel_ms_per_step": {"derive": st["ms_derive"] / K, "scan": scan_ms, "test": st["ms_test"] / K,
                               "step_minus_scan": ms / K - scan_ms},
        "e2e": ({"value": per_step * E * world / (ms2 * 1e-3), "unit": UNIT, "steps": E, "ms_per_step": ms2 / E,
                 "h2d_bytes_per_step": st2["h2d_bytes"] / E, "d2h_bytes_per_step": st2["d2h_bytes"] / E,
                 "api": "ftkb_push_snapshot(host) + ftkb_advance_timestep"} if E else None),
        "gpu_launches": int(st["kernel_launches"]),
        "clocks": sampler.result() if sample_clocks else None,
        "finalize_ms": finalize_ms, "finalize_ms_library": fin.get("library"), "finalize_ms_device": fin.get("device"), "finalize_ms_host": fin.get("host"),
        "trajectories": ntraj, "punctured_simplices": int(npts_total),
        "cells_refined_per_step": st["cells_refined"] / K, "slab_refactor_steps": redo,
        "slab_epilogue_ms": epilogue_ms if world > 1 else None,
    }
    return line


def sub_record(line):
    """what a scaling sub-record keeps of a full line"""
    keep = ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "trajectories", "punctured_simplices", "finalize_ms", "finalize_ms_library",
            "slab_epilogue_ms", "slab_refactor_steps", "cells_refined_per_step")
    out = {k: line[k] for k in keep}
    out["workload"] = line["config"]["workload"]
    out["halo"] = line["config"]["halo"]
    out["scan_kernel"] = line["roofline"]["kernel"]
    out["scan_ms"] = line["roofline"]["avg_launch_ms"]
    out["frac"] = line["roofline"]["frac"]
    out["test_ms"] = line["kernel_ms_per_step"]["test"]
    return out


def self_check(env):
    """untimed, N > 1: the time-sharded run of a reduced configuration (halo through peer memory, merge on rank 0) must equal
    the one-GPU run of the same series -- punctured simplices bit for bit, the same ordered trajectories"""
    import numpy as np
    import torch
    import ftk_b200
    from ftk_b200 import distributed as D
    dims, T = [384, 320], 4 * env.world
    x0, dirv = [190.3, 161.7], [0.9, 0.7]
    ax = [torch.arange(d, dtype=torch.float64, device=env.dev) for d in dims]

    def layer(k):
        mov = ((ax[0] - (x0[0] + dirv[0] * k)) ** 2)[None, :] + ((ax[1] - (x0[1] + dirv[1] * k)) ** 2)[:, None]
        wav = torch.cos(ax[0] * 0.21 + 0.05 * k)[None, :] * torch.sin(ax[1] * 0.17 - 0.03 * k)[:, None]
        return (1e-3 * mov + wav).contiguous()

    tr, info = D.track_time_sharded(layer, dims, T, field="scalar", halo="peer", device=env.local)
    ok, detail = True, {}
    if env.rank == 0:
        one = ftk_b200.track([layer(k) for k in range(T)], dims, field="scalar", device=env.local)
        a, b = tr.get_discrete_critical_points(), one.get_discrete_critical_points()
        ta = sorted((tuple(int(i) for i in idx), bool(lp)) for idx, lp in tr.get_trajectory_index())
        tb = sorted((tuple(int(i) for i in idx), bool(lp)) for idx, lp in one.get_trajectory_index())
        ok = len(a) == len(b) and a.tobytes() == b.tobytes() and ta == tb
        detail = {"workload": f"moving extremum + waves 2D scalar {dims[0]}x{dims[1]}x{T}", "punctured_simplices": int(len(b)),
                  "trajectories": len(tb), "halo": info["halo"], "slab_repeated": bool(info["slab_repeated"])}
        one.close()
    tr.close()
    env.dist.barrier()
    return {"ok": bool(ok), **detail}


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 252; 20 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only-main", action="store_true", help="skip the scaling_c4 / scaling_c3 / dense_woven sub-records and the N > 1 self-check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the punctured simplices of the main workload after its last timed step as DIR/points_<field>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the CUDA path computed; --impl reference has no such output")
        if args.steps is None:
            args.steps = 20   # default sized so the whole run ends within a few minutes
        reference_arm(args, rank)
        return
    if args.steps is None:
        args.steps = 252
    if args.warmup < 3:
        args.warmup = 3
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    from ftk_b200 import _lib
    _lib.lib()   # fail loudly if the CUDA library is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local)
    # one rank per GPU: run on the CPUs next to it, so the pinned host snapshots of the e2e leg live in that socket's memory
    numa_cpus = _lib.lib().ftkb_bind_thread_to_device(local)
    env = Env()
    env.rank, env.world, env.local = rank, world, local
    env.dev = torch.device("cuda", local)
    env.dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=env.dev)
        env.dist = dist

    t_all = time.perf_counter()
    line = run_config(env, args.config, args.steps, args.warmup, args.e2e_steps, sample_clocks=True, dump_dir=args.dump_outputs)
    if line is not None:
        line["config"]["host_cpus_bound_per_rank"] = int(numa_cpus)     # CPUs next to the rank's GPU (0: affinity left alone)
    extras = {}
    if args.config == "c2" and not args.only_main:
        # the configurations north_star quotes its scaling targets on, at the same N, in the same driver-run line
        def budget_ok():
            # one decision for all ranks (rank 0's clock): a rank that skipped on its own would leave the others in a collective
            ok = time.perf_counter() - t_all < 420.0
            if env.dist:
                flag = [ok]
                env.dist.broadcast_object_list(flag, src=0)
                ok = bool(flag[0])
            return ok
        for key, cfg, k in (("scaling_c4", "c4", 8), ("scaling_c3", "c3", 12), ("dense_woven", "woven", 12)):
            if not budget_ok():
                extras[key] = {"skipped": "time budget of the default run"}
                continue
            try:
                rec = run_config(env, cfg, k, 3, 0, sample_clocks=False)
                if rank == 0:
                    extras[key] = sub_record(rec)
            except Exception as e:      # a sub-record never takes the headline down with it
                extras[key] = {"failed": f"{type(e).__name__}: {e}"}
        if world > 1 and budget_ok():
            try:
                extras["selfcheck"] = self_check(env)
            except Exception as e:
                extras["selfcheck"] = {"ok": False, "failed": f"{type(e).__name__}: {e}"}
    if rank == 0:
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_sample(args.config)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if env.dist:
        env.dist.barrier()
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Streaming trajectories read while the series is still running (ftkb_get_live_curveset, ftkb_group_get_live_curveset,
include/ftkb200.h): the reference's traced_critical_points, which trace_critical_points_online keeps current after every
interval sweep (critical_point_tracker.hh:522-641).

The expected state after every step comes from oracle/cp_online.py's OnlineTracer (checked against the reference's stream
fixtures in test_streaming.py), grown one timestep at a time.  A group -- time chunks or z-slabs -- must answer, call for call,
exactly what one tracker fed the same series answers."""
import ctypes as C
import functools
import os
import subprocess

import numpy as np
import pytest

import _parity as P
from test_group_options import STREAM_3D, STREAM_NAMES, _skip_if_too_thin
from test_streaming import load_stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNKS = [(1, [0, 0]), (3, [0, 0, 0])]           # (timesteps per chunk, device list)
SLABS = [[0, 0], [0, 0, 0]]


def _ndev():
    from ftk_b200 import _lib
    return _lib.lib().ftkb_device_count()


def _field(meta):
    return "scalar" if meta["nv"] == 1 else "vector"


def _kw(meta):
    return {} if meta.get("symmetric") is None else {"jacobian_symmetric": bool(meta["symmetric"])}


@functools.lru_cache(maxsize=None)
def _oracle_states(name):
    """trajectories [(elements, loop, complete)] after the grow step of timestep j, for j = 0 .. T-2"""
    from oracle import cp_online
    meta, gold, _ = P.load_golden(name)
    p = gold["points"]
    elems = [tuple(int(v) for v in c) + (int(ty),) for c, ty in zip(p["corner"], p["simplex_type"])]
    tr = cp_online.OnlineTracer(meta["nd"])
    states = []
    for j in range(meta["T"] - 1):
        tr.grow(e for e, ts in zip(elems, p["timestep"]) if int(ts) == j)
        states.append([(list(t["elements"]), bool(t["loop"]), bool(t["complete"])) for t in tr.trajectories])
    return states


def _expected(name, grown_through):
    return [] if grown_through < 0 else _oracle_states(name)[grown_through]


def _live(obj):
    """(grown_through, curve infos, curve points) of a tracker's or a group's live curve set"""
    t, cs = obj.live_curveset()
    infos, pts = cs.arrays()
    cs.close()
    return t, infos, pts


def _elements(infos, pts):
    assert infos["id"].tolist() == list(range(len(infos)))          # id order
    out = []
    for inf in infos:
        q = pts[int(inf["first"]):int(inf["first"] + inf["count"])]["p"]
        out.append(([tuple(int(v) for v in c) + (int(ty),) for c, ty in zip(q["corner"], q["simplex_type"])], bool(inf["loop"]), bool(inf["complete"])))
    return out


def _check_step(name, live, grown_through, what):
    t, infos, pts = live
    assert t == grown_through, f"{what}: grown_through {t}, expected {grown_through}"
    assert _elements(infos, pts) == _expected(name, grown_through), what


def _same_live(a, b, what):
    assert a[0] == b[0], f"{what}: grown_through {a[0]} != {b[0]}"
    assert a[1].tobytes() == b[1].tobytes() and a[2].tobytes() == b[2].tobytes(), what


def _push(tr, field, s):
    (tr.push_scalar_field_snapshot if field == "scalar" else tr.push_vector_field_snapshot)(s)


def _run(name, oracle, group=None, after_step=None):
    """the reference's front-end loop over a fixture on one tracker (and, in lockstep, a group), both streaming; after every
    push / advance / final update, after_step(k, tracker, group) -- k the snapshot index, the timesteps grown through k - 1"""
    from ftk_b200 import tracker as T
    meta, gold, inp = P.load_golden(name)
    field = _field(meta)
    snaps = P.golden_snapshots(meta, inp, oracle)
    tr = T.make_tracker(meta["dims"], field=field, streaming=True, **_kw(meta))
    for k, s in enumerate(snaps):
        _push(tr, field, s)
        if group is not None:
            group.push(k, s)
        if k != 0:
            tr.advance_timestep()
            if group is not None:
                group.g.advance_timestep()
        if k == len(snaps) - 1:
            tr.update_timestep()
            if group is not None:
                group.g.update_timestep()
        if after_step:
            after_step(k, tr, group.g if group is not None else None)
    return meta, gold, tr


class _Group:
    """a streaming group over a fixture, fed from the host or, with `pieces`, from device memory in pieces along z"""

    def __init__(self, meta, ids, chunk, pieces=None):
        from ftk_b200.group import GroupTracker
        self.field = _field(meta)
        self.g = GroupTracker(meta["dims"], ids, field=self.field, chunk=chunk, streaming=True, **_kw(meta))
        self.pieces = pieces

    def push(self, k, s):
        if self.pieces is None:
            _push(self.g, self.field, s)
            return
        import torch
        t = torch.from_numpy(np.ascontiguousarray(s))
        parts = [t[self.pieces[i]:self.pieces[i + 1]].to("cuda:0") for i in range(len(self.pieces) - 1)]
        if self.field == "scalar":
            self.g.push_field_data_snapshot_pieces(scalar=parts)
        else:
            self.g.push_field_data_snapshot_pieces(vector=parts)
        torch.cuda.synchronize()


def _final_checks(name, gold, tr, live_before_finalize=None):
    from ftk_b200.curves import CurveSet
    tr.finalize()
    after = _live(tr)
    cs = CurveSet.from_tracker(tr)
    infos, pts = cs.arrays()
    cs.close()
    _same_live(after, (after[0], infos, pts), f"{name}: live set after finalize != get_curveset")
    pts_sorted = tr.get_discrete_critical_points()
    assert np.array_equal(pts_sorted["corner"], gold["points"]["corner"])
    complete = tr.get_trajectory_complete()
    got = [(idx.tolist(), loop, bool(complete[i])) for i, (idx, loop) in enumerate(tr.get_trajectory_index())]
    assert got == load_stream(name)
    if live_before_finalize is not None:
        _same_live(after, live_before_finalize, f"{name}: finalize changed the grown trajectories")


# ---- one context ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", STREAM_NAMES)
def test_live_curveset_one_context_every_step(name, oracle):
    """after every push, advance and the final update: the trajectories grown so far, ids, element sequences, loop and complete
    flags and grown_through as the oracle has them after the same grow steps; after finalize the live set is get_curveset's"""
    last = {}

    def step(k, tr, _):
        live = _live(tr)
        _check_step(name, live, k - 1 if k > 0 else -1, f"{name} k={k}")
        last["live"] = live

    meta, gold, tr = _run(name, oracle, after_step=step)
    assert last["live"][0] == meta["T"] - 2
    _final_checks(name, gold, tr, last["live"])
    tr.close()


@pytest.mark.gpu
def test_live_slice_of_grown_timestep(oracle):
    """CurveSet.slice(t) holds the ordinal points of timestep t as soon as t has been grown (a moving extremum: one point)"""
    seen = []

    def step(k, tr, _):
        t, cs = tr.live_curveset()
        if t >= 0:
            s = cs.slice(t)
            assert len(s) == 1 and s["p"]["timestep"][0] == t and s["p"]["ordinal"][0] == 1
            seen.append(t)
        cs.close()

    meta, _, tr = _run("mx2d_21x21x32", oracle, after_step=step)
    assert seen[-1] == meta["T"] - 2
    tr.close()


# ---- groups -----------------------------------------------------------------------------------------------------------------------
def _group_case(name, oracle, ids, chunk, pieces=False):
    meta = P.load_golden(name)[0]
    cuts = None
    if pieces:
        D = meta["dims"][2]
        cuts = [0, D // 3, D // 3 + 1, D]           # a one-plane piece in the middle
    grp = _Group(meta, ids, chunk, cuts)
    last = {}

    def step(k, tr, g):
        one, many = _live(tr), _live(g)
        _check_step(name, one, k - 1 if k > 0 else -1, f"{name} k={k}")
        _same_live(many, one, f"{name} ids={ids} chunk={chunk} k={k}: group != one device")
        last["live"] = many

    _, gold, tr = _run(name, oracle, group=grp, after_step=step)
    root = grp.g.finalize()
    after = _live(grp.g)
    _same_live(after, last["live"], f"{name}: group finalize changed the grown trajectories")
    complete = root.get_trajectory_complete()
    got = [(idx.tolist(), loop, bool(complete[i])) for i, (idx, loop) in enumerate(root.get_trajectory_index())]
    assert got == load_stream(name)
    grp.g.close()
    tr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk,ids", CHUNKS)
@pytest.mark.parametrize("name", STREAM_NAMES)
def test_live_curveset_time_chunks_equal_one_device(name, chunk, ids, oracle):
    _group_case(name, oracle, ids, chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("ids", SLABS)
@pytest.mark.parametrize("name", STREAM_3D)
def test_live_curveset_z_slabs_equal_one_device(name, ids, oracle):
    _skip_if_too_thin(P.load_golden(name)[0], ids)
    _group_case(name, oracle, ids, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", STREAM_3D)
def test_live_curveset_z_slabs_fed_in_pieces(name, oracle):
    """a z-slab group fed from device memory in pieces (ftkb_group_push_pieces_device)"""
    _skip_if_too_thin(P.load_golden(name)[0], [0, 0])
    _group_case(name, oracle, [0, 0], 0, pieces=True)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["chunks", "slabs"])
def test_live_curveset_on_real_device_list(mode, oracle):
    """the same on two GPUs: peer copies of every step's points to the merged context"""
    if _ndev() < 2:
        pytest.skip("needs 2 GPUs")
    if mode == "chunks":
        _group_case("woven_128x128x10", oracle, [0, 1], 2)
        _group_case("mx2d_21x21x32", oracle, [1, 0], 3)
    else:
        _group_case("mx3d_21x21x21x10", oracle, [0, 1], 0)
        _group_case("mx3d_21x21x21x10", oracle, [0, 1], 0, pieces=True)


# ---- queries do not perturb -------------------------------------------------------------------------------------------------------
def _outcome(tr):
    pts = tr.get_discrete_critical_points().copy()
    complete = tr.get_trajectory_complete()
    trajs = [(idx.tolist(), loop, bool(complete[i])) for i, (idx, loop) in enumerate(tr.get_trajectory_index())]
    return pts, trajs


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["woven_128x128x10", "rand2d_vector_normal_sym", "mx3d_21x21x21x10", "rand3d_scalar_normal"])
def test_live_queries_do_not_perturb(name, oracle):
    """a run queried at every step -- its live sets post-processed -- gives the points and trajectories of a run never queried"""
    def step(k, tr, _):
        t, cs = tr.live_curveset()
        cs.post_process("legacy")
        cs.slice(max(t, 0))
        cs.close()

    _, _, quiet = _run(name, oracle)
    quiet.finalize()
    _, _, busy = _run(name, oracle, after_step=step)
    busy.finalize()
    a, b = _outcome(quiet), _outcome(busy)
    assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1]
    quiet.close()
    busy.close()


@pytest.mark.gpu
def test_live_queries_do_not_perturb_groups(oracle):
    from ftk_b200.group import track_on_devices
    for name, chunk, ids in [("woven_128x128x10", 2, [0, 0]), ("mx3d_21x21x21x10", 0, [0, 0, 0])]:
        meta, _, inp = P.load_golden(name)
        snaps = P.golden_snapshots(meta, inp, oracle)
        g0, r0 = track_on_devices(snaps, meta["dims"], ids, field=_field(meta), chunk=chunk, streaming=True, **_kw(meta))
        a = _outcome(r0)
        grp = _Group(meta, ids, chunk)
        for k, s in enumerate(snaps):
            grp.push(k, s)
            if k != 0:
                grp.g.advance_timestep()
            if k == len(snaps) - 1:
                grp.g.update_timestep()
            t, cs = grp.g.live_curveset()
            cs.post_process("legacy")
            cs.close()
        b = _outcome(grp.g.finalize())
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1], name
        g0.close()
        grp.g.close()


# ---- refusals ---------------------------------------------------------------------------------------------------------------------
def test_live_curveset_exported_and_null_arguments():
    """both calls are declared, exported and refuse a NULL tracker or group with FTKB_ERR_INVALID"""
    from ftk_b200 import _lib
    header = open(os.path.join(ROOT, "include", "ftkb200.h")).read()
    L = _lib.lib()
    t, h = C.c_int32(), C.c_void_p()
    for fn in ("ftkb_get_live_curveset", "ftkb_group_get_live_curveset"):
        assert fn in _lib.EXPORTS and f"int {fn}(" in header
        assert getattr(L, fn)(None, C.byref(t), C.byref(h)) == 1 and not h.value


@pytest.mark.gpu
def test_live_curveset_refusals():
    from ftk_b200 import _lib
    from ftk_b200 import tracker as T
    from ftk_b200.group import GroupTracker
    L = _lib.lib()
    t, h = C.c_int32(), C.c_void_p()
    off = T.make_tracker([21, 21])
    assert L.ftkb_get_live_curveset(off._h, C.byref(t), C.byref(h)) == 1 and not h.value
    assert "streaming" in L.ftkb_last_error(off._h).decode()
    on = T.make_tracker([21, 21], streaming=True)
    assert L.ftkb_get_live_curveset(on._h, None, C.byref(h)) == 1 and "null" in L.ftkb_last_error(on._h).decode()
    assert L.ftkb_get_live_curveset(on._h, C.byref(t), None) == 1
    assert L.ftkb_get_live_curveset(on._h, C.byref(t), C.byref(h)) == 0 and t.value == -1   # nothing grown yet
    L.ftkb_curveset_destroy(h)
    for g, streaming in ((GroupTracker([21, 21], [0, 0], chunk=2), False), (GroupTracker([21, 21], [0, 0], chunk=2, streaming=True), True)):
        h = C.c_void_p()
        if not streaming:
            assert L.ftkb_group_get_live_curveset(g._g, C.byref(t), C.byref(h)) == 1
            assert "streaming" in L.ftkb_group_last_error(g._g).decode()
        assert L.ftkb_group_get_live_curveset(g._g, None, C.byref(h)) == 1
        assert "null" in L.ftkb_group_last_error(g._g).decode()
        g.close()
    off.close()
    on.close()


# ---- C++ shim ---------------------------------------------------------------------------------------------------------------------
SHIM_PROGRAM = r'''
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "ftk_b200/critical_point_tracker_regular.hh"
// argv: W H T file-of-doubles; prints the traced set after every advance and after the final update
int main(int argc, char **argv) {
  const size_t W = std::atoi(argv[1]), H = std::atoi(argv[2]), T = std::atoi(argv[3]);
  std::vector<double> data(W * H * T);
  FILE *f = std::fopen(argv[4], "rb");
  if (!f || std::fread(data.data(), sizeof(double), data.size(), f) != data.size()) return 2;
  std::fclose(f);
  ftk_b200::critical_point_tracker_2d_regular tracker;
  tracker.set_domain(ftk_b200::lattice({2, 2}, {(int)W - 3, (int)H - 3}));
  tracker.set_array_domain(ftk_b200::lattice({0, 0}, {(int)W, (int)H}));
  tracker.set_scalar_field_source(ftk_b200::SOURCE_GIVEN);
  tracker.set_vector_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_symmetric(true);
  tracker.set_enable_streaming_trajectories(true);
  tracker.initialize();
  for (size_t k = 0; k < T; k++) {
    tracker.push_scalar_field_snapshot(ftk_b200::ndarray<double>::wrap(data.data() + k * W * H, {W, H}));
    if (k != 0) tracker.advance_timestep();
    if (k == T - 1) tracker.update_timestep();
    if (k == 0) continue;
    std::printf("step %zu\n", k);
    for (const auto &kv : tracker.get_traced_critical_points()) {
      std::printf("curve %d %d %d", (int)kv.first, (int)kv.second.loop, (int)kv.second.complete);
      for (const auto &p : kv.second) std::printf(" %d,%d,%d,%d,%d", p.corner[0], p.corner[1], p.corner[2], p.corner[3], p.simplex_type);
      std::printf("\n");
    }
  }
  return 0;
}
'''


@pytest.mark.gpu
def test_cpp_shim_traced_set_is_live(tmp_path, oracle):
    """the shim's get_traced_critical_points() after every advance: the trajectories the oracle has grown by then"""
    from ftk_b200 import build
    build.build()
    name = "mx2d_21x21x32"
    meta, _, inp = P.load_golden(name)
    snaps = P.golden_snapshots(meta, inp, oracle)
    W, H = meta["dims"]
    path = tmp_path / "series.bin"
    np.concatenate([np.ascontiguousarray(s, np.float64).ravel() for s in snaps]).tofile(path)
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    src = tmp_path / "shim_live.cpp"
    src.write_text(SHIM_PROGRAM)
    exe = tmp_path / "shim_live"
    lib = os.path.join(ROOT, "ftk_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           str(src), "-o", str(exe), "-L" + lib, "-lftkb200", "-Wl,-rpath," + lib])
    r = subprocess.run([str(exe), str(W), str(H), str(meta["T"]), str(path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    steps = {}
    for line in r.stdout.splitlines():
        if line.startswith("step"):
            cur = steps.setdefault(int(line.split()[1]), [])
        else:
            w = line.split()
            assert int(w[1]) == len(cur)
            cur.append(([tuple(int(v) for v in e.split(",")) for e in w[4:]], w[2] == "1", w[3] == "1"))
    assert sorted(steps) == list(range(1, meta["T"]))
    for k, got in steps.items():
        assert got == _expected(name, k - 1), f"step {k}"

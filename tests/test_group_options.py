"""Tracker options on several devices (ftkb_group_set_streaming_trajectories / ftkb_group_set_coords, include/ftkb200.h):
streaming trajectories and physical coordinates through time chunks and z-slabs give what one device gives -- the reference's
stream fixtures (trajectory index lists, loop and complete flags, order included) and coordinate fixtures (punctured set and
types exact, x / t / scalar within TOL).  Device lists repeat id 0, so every case runs on one GPU."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np
import pytest

import _parity as P
from test_coords import check as check_coords, load as load_coords, snapshots as coords_snapshots
from test_streaming import load_stream

STREAM_NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(P.GOLDEN_DIR, "stream", "*.npz")))
COORDS_NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(P.GOLDEN_DIR, "coords", "*.npz")))
STREAM_3D = [n for n in STREAM_NAMES if P.load_golden(n)[0]["nd"] == 3]
COORDS_3D = [n for n in COORDS_NAMES if load_coords(n)[0]["nd"] == 3]

CHUNKS = [(1, [0, 0]), (3, [0, 0, 0])]           # (timesteps per chunk, device list)
SLABS = [[0, 0], [0, 0, 0]]


def _field(meta):
    return "scalar" if meta["nv"] == 1 else "vector"


def _skip_if_too_thin(meta, ids):
    """ftkb_group_create needs at least two corner planes per slab"""
    margin = 2 if meta["nv"] == 1 else 1
    nplanes = (meta["dims"][2] - 2) - margin + 1
    if nplanes < 2 * len(ids):
        pytest.skip(f"{nplanes} corner planes cannot be cut into {len(ids)} slabs")


def _streamed(root):
    complete = root.get_trajectory_complete()
    return [(idx.tolist(), loop, bool(complete[i])) for i, (idx, loop) in enumerate(root.get_trajectory_index())]


def _stream_case(name, oracle, ids, chunk):
    from ftk_b200.group import track_on_devices
    meta, gold, inp = P.load_golden(name)
    kw = {} if meta.get("symmetric") is None else {"jacobian_symmetric": bool(meta["symmetric"])}
    g, root = track_on_devices(P.golden_snapshots(meta, inp, oracle), meta["dims"], ids, field=_field(meta), chunk=chunk, streaming=True, **kw)
    pts = root.get_discrete_critical_points()
    assert np.array_equal(pts["corner"], gold["points"]["corner"]) and np.array_equal(pts["simplex_type"], gold["points"]["simplex_type"])
    assert _streamed(root) == load_stream(name)
    g.close()


# ---- 1. streaming, time chunks ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk,ids", CHUNKS)
@pytest.mark.parametrize("name", STREAM_NAMES)
def test_streaming_time_chunks_match_reference(name, chunk, ids, oracle):
    _stream_case(name, oracle, ids, chunk)


# ---- 2. streaming, z-slabs -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ids", SLABS)
@pytest.mark.parametrize("name", STREAM_3D)
def test_streaming_z_slabs_match_reference(name, ids, oracle):
    _skip_if_too_thin(P.load_golden(name)[0], ids)
    _stream_case(name, oracle, ids, 0)


# ---- 3. physical coordinates -----------------------------------------------------------------------------------------------------
def _coords_layouts():
    out = []
    for name in COORDS_NAMES:
        out += [(name, chunk, ids) for chunk, ids in CHUNKS]
        if name in COORDS_3D:
            out += [(name, 0, ids) for ids in SLABS]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,chunk,ids", _coords_layouts())
def test_coords_match_reference(name, chunk, ids, oracle):
    from ftk_b200.group import track_on_devices
    meta, z = load_coords(name)
    if chunk == 0:
        _skip_if_too_thin(meta, ids)
    g, root = track_on_devices(coords_snapshots(meta, z, oracle), meta["dims"], ids, field=_field(meta), chunk=chunk,
                               coords=(meta["coords_mode"], z["coords"]))
    check_coords(root.get_discrete_critical_points(), z, f"{name} chunk {chunk} on {ids}")
    g.close()


# ---- 4. both options at once ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk,ids", [(0, [0, 0, 0]), (2, [0, 0])])
def test_streaming_with_bounds_equals_one_device(chunk, ids, oracle):
    """a moving extremum that crosses every cut of three z-slabs (3.7 planes per step), bounds coordinates and streaming on"""
    import ftk_b200
    from ftk_b200.group import track_on_devices
    dims, T = [32, 28, 40], 6
    x0, d = [15.3, 13.7, 10.1], [0.2, 0.1, 3.7]
    snaps = [oracle.gen_moving_extremum(dims, x0, d, float(k)) for k in range(T)]
    coords = ("bounds", [-1.0, 2.0, 0.5, 3.5, 10.0, 50.0])
    one = ftk_b200.track(snaps, dims, field="scalar", streaming=True, coords=coords)
    want = {"points": one.get_discrete_critical_points(), "trajectories": one.get_trajectory_index()}
    assert len(want["trajectories"]) >= 1 and sum(len(i) for i, _ in want["trajectories"]) > T
    assert np.abs(want["points"]["x"][:, 2] - want["points"]["corner"][:, 2]).max() > 1.0     # not grid units
    g, root = track_on_devices(snaps, dims, ids, field="scalar", chunk=chunk, streaming=True, coords=coords)
    got = {"points": root.get_discrete_critical_points(), "trajectories": root.get_trajectory_index()}
    P.assert_same_result(got, want, tol=0.0, what=f"chunk {chunk} on {ids}")
    assert [(i.tolist(), l) for i, l in got["trajectories"]] == [(i.tolist(), l) for i, l in want["trajectories"]]
    assert root.get_trajectory_complete().tolist() == one.get_trajectory_complete().tolist()
    g.close()
    one.close()


# ---- 5. CLI --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("args,lists", [
    (["--synthetic", "woven", "--width", "31", "--height", "37", "--timesteps", "32"], ["0", "0,0"]),
    (["--synthetic", "moving_extremum_3d", "--width", "24", "--height", "22", "--depth", "30", "--timesteps", "6",
      "--x0", "11.3,10.7,6.1", "--dir", "0.2,0.1,3.7", "--time-chunk", "0"], ["0", "0,0", "0,0,0"]),
], ids=["woven-time-chunks", "moving-extremum-z-slabs"])
def test_cli_stream_on_device_list(args, lists, tmp_path):
    """`ftkb200 -f cp --stream --device 0,0` writes the same traced file as `--device 0`"""
    from ftk_b200 import build
    cli = build.build_cli()
    outs = []
    for k, ids in enumerate(lists):
        out = tmp_path / f"traced_{k}.txt"
        r = subprocess.run([cli, "-f", "cp"] + args + ["--stream", "--device", ids, "-o", str(out)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append(out.read_bytes())
    assert outs[0].startswith(b"#trajectories=") and not outs[0].startswith(b"#trajectories=0\n")
    for o in outs[1:]:
        assert o == outs[0]


# ---- 6. argument checks --------------------------------------------------------------------------------------------------------
def test_group_options_reject_null_group():
    from ftk_b200 import _lib
    data = np.zeros(4)
    assert _lib.lib().ftkb_group_set_coords(None, _lib.COORDS_BOUNDS, data.ctypes.data, 4) == 1        # FTKB_ERR_INVALID
    assert _lib.lib().ftkb_group_set_streaming_trajectories(None, 1) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 2])
def test_group_set_coords_checks_whole_array_sizes(chunk):
    from ftk_b200 import _lib
    from ftk_b200.group import GroupTracker
    W, H, D = 20, 18, 24
    g = GroupTracker([W, H, D], [0, 0], field="scalar", chunk=chunk)
    lib = _lib.lib()

    def rc(mode, n):
        a = np.linspace(0.0, 1.0, max(n, 1))
        return lib.ftkb_group_set_coords(g._g, mode, a.ctypes.data, n)

    assert rc(7, 6) == 1
    assert rc(-1, 6) == 1
    assert rc(_lib.COORDS_BOUNDS, 4) == 1 and rc(_lib.COORDS_BOUNDS, 6) == 0
    assert rc(_lib.COORDS_RECTILINEAR, W + H + D // 2 + 2) == 1            # a slab's own depth is not the array's
    assert rc(_lib.COORDS_RECTILINEAR, W + H + D) == 0
    assert rc(_lib.COORDS_EXPLICIT, 2 * W * H) == 1 and rc(_lib.COORDS_EXPLICIT, 3 * W * H + 1) == 1
    assert rc(_lib.COORDS_EXPLICIT, 3 * W * H) == 0
    assert lib.ftkb_group_set_coords(g._g, _lib.COORDS_RECTILINEAR, None, W + H + D) == 1
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 2])
def test_group_options_refused_after_first_push(chunk, oracle):
    from ftk_b200 import _lib
    from ftk_b200.group import GroupTracker
    dims = [20, 18, 24]
    g = GroupTracker(dims, [0, 0], field="scalar", chunk=chunk)
    lib = _lib.lib()
    b = np.array([0.0, 1.0, 0.0, 1.0, 0.0, 1.0])
    assert lib.ftkb_group_set_streaming_trajectories(g._g, 1) == 0 and lib.ftkb_group_set_coords(g._g, _lib.COORDS_BOUNDS, b.ctypes.data, 6) == 0
    g.push_scalar_field_snapshot(oracle.gen_moving_extremum(dims, [9.3, 8.7, 11.1], [0.1, 0.1, 0.5], 0.0))
    assert lib.ftkb_group_set_streaming_trajectories(g._g, 0) == 1
    assert lib.ftkb_group_set_coords(g._g, _lib.COORDS_BOUNDS, b.ctypes.data, 6) == 1
    assert b"first push" in lib.ftkb_group_last_error(g._g)
    g.close()


@pytest.mark.gpu
def test_streaming_context_that_swept_refuses_imports_merged_one_accepts(oracle):
    """ftkb_import_points on a streaming context: refused once it holds snapshots, accepted while it has swept nothing"""
    from ftk_b200 import _lib, tracker as T
    snaps = list(oracle.synthetic_series("woven", [31, 37], 4, None))
    tr = T.make_tracker([31, 37], streaming=True)
    tr.push_scalar_field_snapshot(snaps[0])
    pts = np.zeros(1, _lib.POINT_DTYPE)
    assert _lib.lib().ftkb_import_points(tr._h, pts.ctypes.data, 1) == 1
    tr.close()
    full = T.track(snaps, [31, 37])
    pts = full.get_discrete_critical_points()
    full.close()
    fresh = T.make_tracker([31, 37], streaming=True)
    assert _lib.lib().ftkb_import_points(fresh._h, pts.ctypes.data, len(pts)) == 0
    fresh.finalize()          # nothing grown: every point is there, no trajectory
    assert len(fresh.get_discrete_critical_points()) == len(pts) and fresh.get_trajectory_index() == []
    fresh.close()

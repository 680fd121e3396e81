"""Snapshots in pieces on several devices (ftkb_group_push_pieces_device, include/ftkb200.h): a tracker spread over a device
list takes a snapshot as contiguous ranges of planes along its slowest axis (z in 3D, y in 2D), each in device memory, and
gives, bit for bit and in the same order, what the one-device tracker and the same group fed from the host give.  Device lists
repeat id 0, so every case runs on one GPU; with 2 or 4 GPUs visible the same cases also run with the group and the pieces
spread over them."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _parity as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ndev():
    from ftk_b200 import _lib
    return _lib.lib().ftkb_device_count()


def _layouts(lists):
    """(group device list, devices the pieces go to in turn)"""
    n = _ndev()
    out = [(ids, [0]) for ids in lists]
    if n >= 2:
        out.append(([0, 1], [0, 1]))
    if n >= 4:
        out.append(([0, 1, 2, 3], [0, 1, 2, 3]))
    return out


def _result(tr):
    return {"points": tr.get_discrete_critical_points().copy(), "trajectories": tr.get_trajectory_index()}


def _same(got, want, what):
    P.assert_same_result(got, want, tol=0.0, what=what)
    assert [(i.tolist(), l) for i, l in got["trajectories"]] == [(i.tolist(), l) for i, l in want["trajectories"]], what


def _pieces(a, cuts, devices):
    """host array `a` cut along its leading axis at `cuts` (0 = cuts[0] < ... < cuts[-1] = extent), piece i on devices[i mod len]"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    return [t[cuts[i]:cuts[i + 1]].to(f"cuda:{devices[i % len(devices)]}") for i in range(len(cuts) - 1)]


def _slab_cuts(g, nslabs, extent):
    """pieces that end where the slabs' corner planes do: slab s's producer owns [c0, c1] (the first and last also the
    array's end planes)"""
    return [0] + [g.slab(s)[0] for s in range(1, nslabs)] + [extent]


def _edge_cuts(g, nslabs, extent):
    """cuts at every slab's a0, c0, c1 + 1 and a1 + 1, each +-1: ghost planes come from the neighbour's piece and from the
    neighbour's neighbour's, and many pieces hold a plane or two"""
    cuts = {0, extent}
    for s in range(nslabs):
        c0, c1, a0, a1 = g.slab(s)
        cuts |= {x + d for x in (a0, c0, c1 + 1, a1 + 1) for d in (-1, 0, 1) if 0 < x + d < extent}
    return sorted(cuts)


def _plan_group(dims, nslabs):
    from ftk_b200.group import GroupTracker
    return GroupTracker(dims, [0] * nslabs, field="scalar", chunk=0)


def _edge_cuts_of(dims, nslabs):
    """_edge_cuts of an nslabs-device z-slab group over `dims` (for any group over those dims)"""
    plan = _plan_group(dims, nslabs)
    cuts = _edge_cuts(plan, nslabs, dims[2])
    plan.close()
    return cuts


def _push_series(g, series, names, cuts, devices):
    """series: per timestep a tuple of host arrays, one per name"""
    for k, arrays in enumerate(series):
        g.push_field_data_snapshot_pieces(**{n: _pieces(a, cuts, devices) for n, a in zip(names, arrays)})
        if k:
            g.advance_timestep()
        if k == len(series) - 1:
            g.update_timestep()
    return _result(g.finalize())


def _check(snaps, dims, field, chunk, lists, cuts_of, **kw):
    """fed from pieces, the group equals the one-device host run and its own host run; cuts_of(group, ids) gives the cuts"""
    import ftk_b200
    from ftk_b200.group import GroupTracker, track_on_devices
    one = ftk_b200.track(snaps, dims, field=field, **kw)
    want = _result(one)
    one.close()
    assert len(want["points"]) > 0
    for ids, devices in _layouts(lists):
        g, root = track_on_devices(snaps, dims, ids, field=field, chunk=chunk, **kw)
        host = _result(root)
        g.close()
        g = GroupTracker(dims, ids, field=field, chunk=chunk, **kw)
        cuts = cuts_of(g, ids)
        what = f"{field} chunk {chunk} on {ids}, pieces {cuts} on {devices}"
        got = _push_series(g, [(s,) for s in snaps], [field], cuts, devices)
        g.close()
        _same(got, want, what + " vs one device")
        _same(got, host, what + " vs host-fed group")


# ---- 1. 2D, time chunks: row pieces ---------------------------------------------------------------------------------------------
ROWS = {"one": lambda H: [0, H], "two": lambda H: [0, H // 2, H], "uneven": lambda H: [0, 1, 2, H // 2 - 1, H - 1, H]}


@pytest.mark.gpu
@pytest.mark.parametrize("cut", sorted(ROWS))
@pytest.mark.parametrize("chunk", [1, 3])
def test_pieces_2d_scalar_time_chunks(chunk, cut, oracle):
    dims = [96, 80]
    _check(list(oracle.synthetic_series("woven", dims, 11, None)), dims, "scalar", chunk, [[0, 0], [0, 0, 0]], lambda g, ids: ROWS[cut](dims[1]))


@pytest.mark.gpu
@pytest.mark.parametrize("cut", sorted(ROWS))
@pytest.mark.parametrize("chunk", [1, 3])
def test_pieces_2d_vector_time_chunks(chunk, cut, oracle):
    dims = [64, 32]
    _check(list(oracle.synthetic_series("double_gyre", dims, 10, None)), dims, "vector", chunk, [[0, 0], [0, 0, 0]], lambda g, ids: ROWS[cut](dims[1]))


# ---- 2. 3D scalar, z-slabs and time chunks --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cut", ["slabs", "edges", "fewer"])
@pytest.mark.parametrize("kind", ["smooth", "int"])
@pytest.mark.parametrize("chunk,nslabs", [(0, 2), (0, 3), (2, 3)])
def test_pieces_3d_scalar(chunk, nslabs, kind, cut):
    """integer values: the quantisation factor never saturates, so the slabs combine their minima before every sweep.  The
    cuts follow the slabs of an nslabs-device z-slab group (for time chunks too): at the slabs' own cuts, at every edge of
    their corner and array ranges +-1, or fewer pieces than devices"""
    from test_gpu_parity import _rand_series
    dims = [36, 30, 26]
    D = dims[2]
    snaps = _rand_series(np.random.default_rng(91), dims, 4 if chunk == 0 else 6, 1, kind)
    plan = _plan_group(dims, nslabs)
    cuts = {"slabs": _slab_cuts(plan, nslabs, D), "edges": _edge_cuts(plan, nslabs, D), "fewer": [0, plan.slab(1)[2] + 1, D] if nslabs == 3 else [0, D]}[cut]
    plan.close()
    if cut == "edges":
        assert len(cuts) - 1 > 3 * nslabs and min(np.diff(cuts)) == 1
    _check(snaps, dims, "scalar", chunk, [[0] * nslabs], lambda g, ids: cuts)


# ---- 3. 3D vector on z-slabs ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cut", ["slabs", "edges"])
def test_pieces_3d_vector_z_slabs(cut, oracle):
    dims = [20, 18, 16]
    f = _slab_cuts if cut == "slabs" else _edge_cuts
    _check(list(oracle.synthetic_series("abc", dims, 5, None)), dims, "vector", 0, [[0, 0], [0, 0, 0]], lambda g, ids: f(g, len(ids), dims[2]))


# ---- 4. a GIVEN Jacobian -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dims,chunk,ids", [([13, 11], 2, [0, 0]), ([14, 12, 12], 0, [0, 0, 0])])
def test_pieces_given_jacobian(dims, chunk, ids):
    import ftk_b200
    from ftk_b200.group import GroupTracker
    rng = np.random.default_rng(5)
    nd, T = len(dims), 5
    shape = tuple(reversed(dims))
    series = [(rng.standard_normal(shape), rng.standard_normal(shape + (nd,)), rng.standard_normal(shape + (nd, nd))) for _ in range(T)]
    kw = dict(field="vector", scalar_source=1, vector_source=1, jacobian_source=1, jacobian_symmetric=False)
    one = ftk_b200.make_tracker(dims, **kw)
    host = GroupTracker(dims, ids, chunk=chunk, **kw)
    for k, (s, v, j) in enumerate(series):
        for tr in (one, host):
            tr.push_field_data_snapshot(scalar=s, vector=v, jacobian=j)
            if k:
                tr.advance_timestep()
            if k == T - 1:
                tr.update_timestep()
    one.finalize()
    want = _result(one)
    assert len(want["points"]) > 0
    host_r = _result(host.finalize())
    for ids_, devices in _layouts([ids]):
        g = GroupTracker(dims, ids_, chunk=chunk, **kw)
        extent = dims[-1]
        cuts = _edge_cuts(g, len(ids_), extent) if chunk == 0 else [0, 1, extent // 2, extent - 1, extent]
        got = _push_series(g, series, ["scalar", "vector", "jacobian"], cuts, devices)
        _same(got, want, f"given jacobian on {ids_}, pieces {cuts}")
        _same(got, host_r, f"given jacobian on {ids_}, pieces {cuts} vs host-fed group")
        g.close()
    host.close()
    one.close()


# ---- 5. options compose: streaming trajectories with bounds coordinates -------------------------------------------------------
@pytest.mark.gpu
def test_pieces_streaming_with_bounds_z_slabs(oracle):
    import ftk_b200
    from ftk_b200.group import GroupTracker
    dims, T = [32, 28, 40], 6
    snaps = [oracle.gen_moving_extremum(dims, [15.3, 13.7, 10.1], [0.2, 0.1, 3.7], float(k)) for k in range(T)]
    coords = ("bounds", [-1.0, 2.0, 0.5, 3.5, 10.0, 50.0])
    one = ftk_b200.track(snaps, dims, field="scalar", streaming=True, coords=coords)
    want = _result(one)
    assert len(want["trajectories"]) >= 1 and sum(len(i) for i, _ in want["trajectories"]) > T
    for ids, devices in _layouts([[0, 0, 0]]):
        g = GroupTracker(dims, ids, field="scalar", chunk=0, streaming=True, coords=coords)
        got = _push_series(g, [(s,) for s in snaps], ["scalar"], _edge_cuts(g, len(ids), dims[2]), devices)
        _same(got, want, f"streaming with bounds on {ids}")
        assert g._root.get_trajectory_complete().tolist() == one.get_trajectory_complete().tolist()
        g.close()
    one.close()


# ---- 6. ordering and lifetime -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 2])
def test_pieces_ordered_after_their_streams_and_copied_before_return(chunk, oracle):
    """Every piece is rewritten for every snapshot on a torch stream of its own that first idles for a while, and the push
    follows without a host synchronise: each piece's copies must wait for its stream.  Right after the push every piece is
    filled with NaN on its stream: the copies must be complete when the push returns."""
    import torch
    import ftk_b200
    from ftk_b200.group import GroupTracker
    dims, T = [32, 28, 40], 6
    snaps = [oracle.gen_moving_extremum(dims, [15.3, 13.7, 10.1], [0.2, 0.1, 3.7], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    for ids, devices in _layouts([[0, 0, 0]]):
        g = GroupTracker(dims, ids, field="scalar", chunk=chunk)
        cuts = _edge_cuts_of(dims, 3)
        src = [_pieces(s, cuts, devices) for s in snaps]
        for d in set(devices):
            torch.cuda.synchronize(d)
        bufs = [torch.empty_like(p) for p in src[0]]
        streams = [torch.cuda.Stream(device=b.device) for b in bufs]
        for k in range(T):
            for b, s, p in zip(bufs, streams, src[k]):
                with torch.cuda.device(b.device), torch.cuda.stream(s):
                    torch.cuda._sleep(1 << 20)
                    b.copy_(p)
            # (pieces on one device written by different streams: GroupTracker would name torch's current stream for all)
            _push_on_streams(g, bufs, streams)
            for b, s in zip(bufs, streams):
                with torch.cuda.device(b.device), torch.cuda.stream(s):
                    b.fill_(float("nan"))
            if k:
                g.advance_timestep()
            if k == T - 1:
                g.update_timestep()
        _same(_result(g.finalize()), want, f"chunk {chunk} on {ids}, pieces {cuts} on {devices}")
        for d in set(devices):
            torch.cuda.synchronize(d)
        g.close()


def _push_on_streams(g, bufs, streams):
    """push `bufs` as scalar pieces, each ordered after its own stream (ftkb_piece.stream)"""
    from ftk_b200 import _lib
    pieces = (_lib.Piece * len(bufs))()
    first = 0
    for p, b, s in zip(pieces, bufs, streams):
        p.scalar, p.first, p.count = b.data_ptr(), first, b.shape[0]
        p.stream, p.has_stream = int(s.cuda_stream), 1
        first += b.shape[0]
    g._check(_lib.lib().ftkb_group_push_pieces_device(g._g, pieces, len(bufs)))


@pytest.mark.gpu
@pytest.mark.skipif("_ndev() < 2")
@pytest.mark.parametrize("chunk", [0, 2])
def test_producer_stream_on_another_device_than_the_arrays(chunk, oracle):
    """Arrays on device 1, written by a stream of device 1 that first idles, and the stream the group is told to wait for on
    device 0 (made to wait for device 1's stream): the copies must still read the arrays from device 1, for a whole-device
    push (ftkb_group_set_producer_stream) and for a piece push (ftkb_piece.stream)"""
    import torch
    import ftk_b200
    from ftk_b200 import _lib
    from ftk_b200.group import GroupTracker
    dims, T = [32, 28, 40], 6
    snaps = [oracle.gen_moving_extremum(dims, [15.3, 13.7, 10.1], [0.2, 0.1, 3.7], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    src = _on_device(snaps, 1)
    writer, named = torch.cuda.Stream(device=1), torch.cuda.Stream(device=0)
    for pieces in (False, True):
        g = GroupTracker(dims, [0, 0], field="scalar", chunk=chunk)
        buf = torch.empty_like(src[0])
        if not pieces:
            g._check(_lib.lib().ftkb_group_set_producer_stream(g._g, C.c_void_p(int(named.cuda_stream)), 1))
        for k in range(T):
            with torch.cuda.device(1), torch.cuda.stream(writer):
                torch.cuda._sleep(1 << 20)
                buf.copy_(src[k])
            named.wait_stream(writer)
            if pieces:
                _push_on_streams(g, [buf[:17], buf[17:]], [named, named])
            else:
                g._check(_lib.lib().ftkb_group_push_snapshot_device(g._g, buf.data_ptr(), None, None))
            if k:
                g.advance_timestep()
            if k == T - 1:
                g.update_timestep()
        _same(_result(g.finalize()), want, f"arrays on device 1, stream on device 0, pieces={pieces}, chunk {chunk}")
        torch.cuda.synchronize(1)
        g.close()


def _on_device(snaps, device):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(s)).to(f"cuda:{device}") for s in snaps]


# ---- 7. host, whole-device and piece pushes in one series ----------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 3])
def test_host_device_and_piece_pushes_alternate(chunk, oracle):
    import torch
    import ftk_b200
    from ftk_b200.group import GroupTracker
    dims, T = [24, 22, 30], 9
    snaps = [oracle.gen_moving_extremum(dims, [11.3, 10.7, 6.1], [0.2, 0.1, 2.3], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    g = GroupTracker(dims, [0, 0, 0], field="scalar", chunk=chunk)
    cuts = _edge_cuts_of(dims, 3)
    for k, s in enumerate(snaps):
        if k % 3 == 0:
            g.push_scalar_field_snapshot(s)
        elif k % 3 == 1:
            g.push_scalar_field_snapshot(torch.from_numpy(s).to("cuda:0"))
        else:
            g.push_field_data_snapshot_pieces(scalar=_pieces(s, cuts, [0]))
        if k:
            g.advance_timestep()
        if k == T - 1:
            g.update_timestep()
    _same(_result(g.finalize()), want, f"alternating pushes, chunk {chunk}")
    g.close()


# ---- 8. refusals ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 2])
def test_piece_push_refusals_leave_the_group_usable(chunk, oracle):
    """every malformed push is refused with FTKB_ERR_INVALID and a message naming the piece; no refused push hands the library
    a pointer it would read out of bounds; the same group then takes the valid series and gives the right result"""
    import torch
    import ftk_b200
    from ftk_b200 import _lib
    from ftk_b200.group import GroupTracker
    lib = _lib.lib()
    dims, T = [20, 18, 24], 4
    D, plane = dims[2], dims[0] * dims[1]
    snaps = [oracle.gen_moving_extremum(dims, [9.3, 8.7, 11.1], [0.1, 0.1, 0.5], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    g = GroupTracker(dims, [0, 0], field="scalar", chunk=chunk)
    whole = torch.zeros(2 * D * plane, dtype=torch.float64, device="cuda:0")       # every offset below stays inside it
    host = np.zeros(D * plane)

    def at(z):
        return whole.data_ptr() + 8 * plane * z

    def rejected(spec, words, n=None):
        pieces = (_lib.Piece * max(len(spec), 1))()
        for p, (ptr, first, count) in zip(pieces, spec):
            p.scalar, p.first, p.count = ptr, first, count
        assert lib.ftkb_group_push_pieces_device(g._g, pieces, len(spec) if n is None else n) == _lib.ERR_INVALID, spec
        msg = lib.ftkb_group_last_error(g._g).decode()
        assert all(w in msg for w in words), msg

    assert lib.ftkb_group_push_pieces_device(None, None, 1) == _lib.ERR_INVALID
    rejected([(at(0), 0, D)], ["no pieces", "n = 0"], n=0)
    rejected([(at(0), 0, D)], ["no pieces", "n = -1"], n=-1)
    rejected([(at(0), 0, 10), (at(11), 11, D - 11)], ["piece 1", "a gap"])
    rejected([(at(0), 0, 10), (at(9), 9, D - 9)], ["piece 1", "an overlap"])
    rejected([(at(10), 10, D - 10), (at(0), 0, 10)], ["piece 0", "starts at z plane 10"])
    rejected([(at(0), 0, 10), (at(10), 10, D - 11)], ["piece 1", f"end at z plane {D - 1}"])
    rejected([(at(0), 0, 10), (at(10), 10, D - 9)], ["piece 1", "past the array"])
    rejected([(at(0), 0, 0), (at(0), 0, D)], ["piece 0", "count is 0"])
    rejected([(at(0), 0, 10), (at(10), 10, 0), (at(10), 10, D - 10)], ["piece 1", "count is 0"])
    rejected([(at(0), 0, 10), (host.ctypes.data + 8 * plane * 10, 10, D - 10)], ["piece 1", "scalar", "not CUDA device memory"])
    pinned = torch.zeros(D * plane, dtype=torch.float64).pin_memory()
    rejected([(pinned.data_ptr(), 0, 10), (at(10), 10, D - 10)], ["piece 0", "scalar", "not CUDA device memory"])
    rejected([(at(0), 0, 10), (at(10) + 4, 10, D - 10)], ["piece 1", "scalar", "aligned"])
    rejected([(at(0), 0, 10), (None, 10, D - 10)], ["piece 1", "lacks the scalar array"])
    rejected([(None, 0, 10), (None, 10, D - 10)], ["piece 0", "no array"])
    # a piece that passes an array the others lack, through the Python front end
    vec = torch.zeros((D, dims[1], dims[0], 3), dtype=torch.float64, device="cuda:0")
    with pytest.raises(_lib.FTKBError, match="piece 1: passes a vector array"):
        g.push_field_data_snapshot_pieces(scalar=[whole[:10 * plane].view(10, dims[1], dims[0]), whole[10 * plane:D * plane].view(D - 10, dims[1], dims[0])],
                                          vector=[None, vec[10:]])
    if _ndev() >= 2:
        pieces = (_lib.Piece * 2)()
        vec1 = torch.zeros(3 * D * plane, dtype=torch.float64, device="cuda:1")
        pieces[0].scalar, pieces[0].vector, pieces[0].first, pieces[0].count = at(0), vec1.data_ptr(), 0, 10
        pieces[1].scalar, pieces[1].vector, pieces[1].first, pieces[1].count = at(10), vec1.data_ptr(), 10, D - 10
        assert lib.ftkb_group_push_pieces_device(g._g, pieces, 2) == _lib.ERR_INVALID
        msg = lib.ftkb_group_last_error(g._g).decode()
        assert "piece 0" in msg and "vector" in msg and "another device" in msg, msg
    with pytest.raises(ValueError):
        g.push_field_data_snapshot_pieces(scalar=[whole[:D * plane].view(D, dims[1], dims[0]).float()])
    with pytest.raises(ValueError):
        g.push_field_data_snapshot_pieces(scalar=[whole[:D * plane].view(D, dims[0], dims[1])])
    planes = (C.c_int32 * 4)()
    for s in (2, -1):
        assert lib.ftkb_group_get_slab(g._g, s, planes) == _lib.ERR_INVALID
        msg = lib.ftkb_group_last_error(g._g).decode()
        assert ("runs time chunks" if chunk else f"slab {s} does not exist") in msg, msg
    if chunk:
        assert lib.ftkb_group_get_slab(g._g, 0, planes) == _lib.ERR_INVALID
        with pytest.raises(_lib.FTKBError, match="get_slab: the group runs time chunks"):
            g.slab(0)
    else:
        with pytest.raises(_lib.FTKBError, match="get_slab: slab 5 does not exist"):
            g.slab(5)
        c0, c1, a0, a1 = g.slab(1)
        assert g.slab(0)[1] + 1 == c0 and a0 == c0 - 2 and a1 == D - 1 and c1 == dims[2] - 2
    # the group still takes the valid series
    cuts = [0, 7, 13, D]
    _same(_push_series(g, [(s,) for s in snaps], ["scalar"], cuts, [0]), want, f"after refused pushes, chunk {chunk}")
    g.close()


# ---- 9. the C++ shim -----------------------------------------------------------------------------------------------------------
SHIM_PROGRAM = r'''
#include <cmath>
#include <cstdio>
#include <iostream>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "ftk_b200/critical_point_tracker_regular.hh"
int main(int argc, char **argv) {
  const bool pieces = std::string(argv[1]) == "pieces";
  const int W = 24, H = 22, D = 26, T = 6;
  const std::vector<int> first = {0, 1, 9, 10, 17, 25};       // pieces of 1, 8, 1, 7, 8 and 1 planes
  ftk_b200::critical_point_tracker_3d_regular tracker;
  tracker.set_device_ids({0, 0, 0});
  tracker.set_time_chunk(0);
  tracker.set_domain(ftk_b200::lattice({2, 2, 2}, {W - 4, H - 4, D - 4}));
  tracker.set_array_domain(ftk_b200::lattice({0, 0, 0}, {W, H, D}));
  tracker.set_scalar_field_source(ftk_b200::SOURCE_GIVEN);
  tracker.set_vector_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_symmetric(true);
  tracker.initialize();
  const size_t plane = (size_t)W * H;
  std::vector<double> h(plane * D);
  std::vector<double *> d(first.size(), nullptr);
  for (size_t i = 0; i < first.size(); i++) {
    const int count = (i + 1 < first.size() ? first[i + 1] : D) - first[i];
    if (cudaMalloc(&d[i], plane * count * sizeof(double)) != cudaSuccess) return 3;
  }
  for (int k = 0; k < T; k++) {
    for (int z = 0; z < D; z++)
      for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++)
          h[x + W * (y + H * (size_t)z)] = std::cos(0.31 * x + 0.05 * k) * std::sin(0.27 * y - 0.07 * k) * std::cos(0.23 * z + 0.04 * k) + 0.01 * x;
    if (pieces) {
      std::vector<ftk_b200::ndarray<double>> views;
      for (size_t i = 0; i < first.size(); i++) {
        const int count = (i + 1 < first.size() ? first[i + 1] : D) - first[i];
        if (cudaMemcpy(d[i], h.data() + plane * first[i], plane * count * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) return 3;
        views.push_back(ftk_b200::ndarray<double>::wrap(d[i], {(size_t)W, (size_t)H, (size_t)count}, true));
      }
      tracker.push_field_data_snapshot_pieces(first, views);
    } else {
      tracker.push_scalar_field_snapshot(ftk_b200::ndarray<double>::wrap(h.data(), {(size_t)W, (size_t)H, (size_t)D}));
    }
    if (k) tracker.advance_timestep();
    if (k == T - 1) tracker.update_timestep();
  }
  tracker.finalize();
  tracker.write_traced_critical_points_text(std::cout);
  std::printf("points=%zu\n", tracker.get_critical_points().size());
  ftk_b200::critical_point_tracker_3d_regular one;
  one.set_domain(ftk_b200::lattice({2, 2, 2}, {W - 4, H - 4, D - 4}));
  one.set_array_domain(ftk_b200::lattice({0, 0, 0}, {W, H, D}));
  one.set_scalar_field_source(ftk_b200::SOURCE_GIVEN);
  one.initialize();
  try {
    one.push_field_data_snapshot_pieces({0}, {ftk_b200::ndarray<double>::wrap(d[0], {(size_t)W, (size_t)H, (size_t)D}, true)});
    std::printf("single device took pieces\n");
  } catch (const std::runtime_error &e) {
    std::printf("single device: %s\n", e.what());
  }
  for (double *p : d) cudaFree(p);
  return 0;
}
'''


@pytest.mark.gpu
def test_cpp_shim_pieces_on_device_list(tmp_path):
    from ftk_b200 import build
    build.build()
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    src = tmp_path / "shim_pieces.cpp"
    src.write_text(SHIM_PROGRAM)
    exe = tmp_path / "shim_pieces"
    lib = os.path.join(ROOT, "ftk_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           str(src), "-o", str(exe), "-L" + lib, "-lftkb200", "-Wl,-rpath," + lib,
                           "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(cuda, "lib64")])
    outs = {}
    for mode in ("host", "pieces"):
        r = subprocess.run([str(exe), mode], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs[mode] = r.stdout
    assert "points=0" not in outs["host"] and len(outs["host"]) > 100
    assert "single device: ftk_b200: snapshot pieces need a tracker on several devices" in outs["host"]
    assert outs["pieces"] == outs["host"]


# ---- CPU: the ctypes mirror of ftkb_piece ---------------------------------------------------------------------------------------
def test_piece_struct_layout_matches_header(tmp_path):
    from ftk_b200 import _lib
    src = tmp_path / "piece.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ftkb200.h"\nint main(void){printf("%zu %zu %zu %zu %zu\\n", '
                   'sizeof(ftkb_piece), offsetof(ftkb_piece, first), offsetof(ftkb_piece, count), offsetof(ftkb_piece, stream), '
                   'offsetof(ftkb_piece, has_stream));return 0;}\n')
    exe = tmp_path / "piece"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    P_ = _lib.Piece
    assert got == [C.sizeof(P_), P_.first.offset, P_.count.offset, P_.stream.offset, P_.has_stream.offset]

"""Device-resident snapshots on several devices (ftkb_group_push_snapshot_device, include/ftkb200.h): a tracker spread over a
device list takes torch CUDA tensors on any visible device and gives, bit for bit and in the same order, what the one-device
tracker and the same group give when fed from the host.  Device lists repeat id 0, so every case runs on one GPU; with more
GPUs visible the same cases run across them, fed from a device of the group or from one outside it."""
import os
import subprocess

import numpy as np
import pytest

import _parity as P

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ndev():
    from ftk_b200 import _lib
    return _lib.lib().ftkb_device_count()


def _layouts(lists):
    """(device list, source device): the group's first device feeds every list; a two-device group is also fed from its
    second device and from a device outside it"""
    n = _ndev()
    out = [(ids, 0) for ids in lists]
    if n >= 2:
        out += [([0, 1], 0), ([0, 1], 1)]
    if n >= 3:
        out.append(([0, 1], 2))
    if n >= 4:
        out.append(([0, 1, 2, 3], 0))
    return out


def _result(tr):
    return {"points": tr.get_discrete_critical_points().copy(), "trajectories": tr.get_trajectory_index()}


def _same(got, want, what):
    P.assert_same_result(got, want, tol=0.0, what=what)
    assert [(i.tolist(), l) for i, l in got["trajectories"]] == [(i.tolist(), l) for i, l in want["trajectories"]], what


def _on(snaps, device):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(s)).to(f"cuda:{device}") for s in snaps]


def _check_layouts(snaps, dims, field, chunk, lists, **kw):
    """the group fed from device tensors equals the one-device host run and the group's own host run"""
    import ftk_b200
    from ftk_b200.group import track_on_devices
    one = ftk_b200.track(snaps, dims, field=field, **kw)
    want = _result(one)
    one.close()
    assert len(want["points"]) > 0
    for ids, src in _layouts(lists):
        what = f"{field} chunk {chunk} on {ids} from device {src}"
        g, root = track_on_devices(snaps, dims, ids, field=field, chunk=chunk, **kw)
        host = _result(root)
        g.close()
        g, root = track_on_devices(_on(snaps, src), dims, ids, field=field, chunk=chunk, **kw)
        got = _result(root)
        g.close()
        _same(got, want, what + " vs one device")
        _same(got, host, what + " vs host-fed group")


# ---- 1. 2D, time chunks --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [1, 3])
def test_device_input_2d_scalar_time_chunks(chunk, oracle):
    dims = [96, 80]
    _check_layouts(list(oracle.synthetic_series("woven", dims, 11, None)), dims, "scalar", chunk, [[0, 0], [0, 0, 0]])


def test_device_input_2d_vector_time_chunks(oracle):
    dims = [64, 32]
    _check_layouts(list(oracle.synthetic_series("double_gyre", dims, 10, None)), dims, "vector", 3, [[0, 0], [0, 0, 0]])


# ---- 2. 3D, z-slabs and time chunks --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["smooth", "int"])
@pytest.mark.parametrize("chunk", [0, 2])
def test_device_input_3d_scalar(chunk, kind):
    """integer values: the quantisation factor never saturates, so slabs combine their minima before every sweep and chunks
    inherit the running minimum one after another"""
    from test_gpu_parity import _rand_series
    dims = [36, 30, 26]
    snaps = _rand_series(np.random.default_rng(91), dims, 4 if chunk == 0 else 6, 1, kind)
    _check_layouts(snaps, dims, "scalar", chunk, [[0, 0], [0, 0, 0]])


def test_device_input_3d_vector_z_slabs(oracle):
    dims = [20, 18, 16]
    _check_layouts(list(oracle.synthetic_series("abc", dims, 5, None)), dims, "vector", 0, [[0, 0], [0, 0, 0]])


# ---- 3. a GIVEN Jacobian -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims,chunk", [([13, 11], 2), ([14, 12, 12], 0)])
def test_device_input_given_jacobian(dims, chunk):
    import ftk_b200
    from ftk_b200.group import GroupTracker
    rng = np.random.default_rng(5)
    nd, T = len(dims), 5
    shape = tuple(reversed(dims))
    series = [(rng.standard_normal(shape), rng.standard_normal(shape + (nd,)), rng.standard_normal(shape + (nd, nd))) for _ in range(T)]
    kw = dict(field="vector", scalar_source=1, vector_source=1, jacobian_source=1, jacobian_symmetric=False)
    one = ftk_b200.make_tracker(dims, **kw)
    trackers = [(one, None)] + [(GroupTracker(dims, ids, chunk=chunk, **kw), src) for ids, src in _layouts([[0, 0]])]
    for k, (s, v, j) in enumerate(series):
        for tr, src in trackers:
            if src is None:
                tr.push_field_data_snapshot(scalar=s, vector=v, jacobian=j)
            else:
                tr.push_field_data_snapshot(*_on((s, v, j), src))
            if k:
                tr.advance_timestep()
            if k == T - 1:
                tr.update_timestep()
    one.finalize()
    want = _result(one)
    assert len(want["points"]) > 0
    if nd == 2:
        assert len(set(want["points"]["cp_type"])) > 2       # foci / centres appear with a full Jacobian
    for tr, src in trackers[1:]:
        _same(_result(tr.finalize()), want, f"given jacobian from device {src}")
        tr.close()
    one.close()


# ---- 4. / 5. copies are done on return; copies wait for the producer stream -------------------------------------------------
@pytest.mark.parametrize("chunk", [0, 2])
def test_device_input_copied_before_return_and_ordered_after_producer(chunk, oracle):
    """One buffer on the source device is rewritten for every snapshot on a side stream that first idles for a while, and the
    push follows without a host synchronise: the copies must wait for that stream.  After the push the buffer is filled with
    NaN on the same stream: the copies must be complete when the push returns."""
    import torch
    import ftk_b200
    from ftk_b200.group import GroupTracker
    dims, T = [32, 28, 40], 6
    snaps = [oracle.gen_moving_extremum(dims, [15.3, 13.7, 10.1], [0.2, 0.1, 3.7], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    for ids, src in _layouts([[0, 0], [0, 0, 0]]):
        dev = _on(snaps, src)
        torch.cuda.synchronize(src)
        buf = torch.empty_like(dev[0])
        side = torch.cuda.Stream(device=src)
        g = GroupTracker(dims, ids, field="scalar", chunk=chunk)
        for k in range(T):
            with torch.cuda.device(src), torch.cuda.stream(side):
                torch.cuda._sleep(1 << 21)
                buf.copy_(dev[k])
                g.push_scalar_field_snapshot(buf)
                buf.fill_(float("nan"))
            if k:
                g.advance_timestep()
            if k == T - 1:
                g.update_timestep()
        _same(_result(g.finalize()), want, f"chunk {chunk} on {ids} from device {src}")
        torch.cuda.synchronize(src)
        g.close()


# ---- 6. with streaming trajectories and physical coordinates -----------------------------------------------------------------
@pytest.mark.parametrize("chunk,ids", [(0, [0, 0, 0]), (2, [0, 0])])
def test_device_input_streaming_with_bounds(chunk, ids, oracle):
    import ftk_b200
    from ftk_b200.group import track_on_devices
    dims, T = [32, 28, 40], 6
    snaps = [oracle.gen_moving_extremum(dims, [15.3, 13.7, 10.1], [0.2, 0.1, 3.7], float(k)) for k in range(T)]
    coords = ("bounds", [-1.0, 2.0, 0.5, 3.5, 10.0, 50.0])
    one = ftk_b200.track(snaps, dims, field="scalar", streaming=True, coords=coords)
    want = _result(one)
    assert len(want["trajectories"]) >= 1 and sum(len(i) for i, _ in want["trajectories"]) > T
    g, root = track_on_devices(_on(snaps, 0), dims, ids, field="scalar", chunk=chunk, streaming=True, coords=coords)
    _same(_result(root), want, f"streaming chunk {chunk} on {ids}")
    assert root.get_trajectory_complete().tolist() == one.get_trajectory_complete().tolist()
    g.close()
    one.close()


# ---- 7. host and device pushes in one series ----------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [0, 3])
def test_host_and_device_pushes_alternate(chunk, oracle):
    import ftk_b200
    from ftk_b200.group import track_on_devices
    dims, T = [24, 22, 30], 8
    snaps = [oracle.gen_moving_extremum(dims, [11.3, 10.7, 6.1], [0.2, 0.1, 2.3], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    dev = _on(snaps, 0)
    mixed = [dev[k] if k % 2 else snaps[k] for k in range(T)]
    g, root = track_on_devices(mixed, dims, [0, 0, 0], field="scalar", chunk=chunk)
    _same(_result(root), want, f"alternating pushes, chunk {chunk}")
    g.close()


# ---- 8. argument checks -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk", [0, 2])
def test_device_push_rejects_bad_pointers(chunk, oracle):
    import torch
    import ftk_b200
    from ftk_b200 import _lib
    from ftk_b200.group import GroupTracker
    lib = _lib.lib()
    assert lib.ftkb_group_push_snapshot_device(None, None, None, None) == _lib.ERR_INVALID
    assert lib.ftkb_group_set_producer_stream(None, None, 1) == _lib.ERR_INVALID
    dims, T = [20, 18, 24], 4
    snaps = [oracle.gen_moving_extremum(dims, [9.3, 8.7, 11.1], [0.1, 0.1, 0.5], float(k)) for k in range(T)]
    want = _result(ftk_b200.track(snaps, dims, field="scalar"))
    g = GroupTracker(dims, [0, 0], field="scalar", chunk=chunk)

    def rejected(s, v, words):
        assert lib.ftkb_group_push_snapshot_device(g._g, s, v, None) == _lib.ERR_INVALID
        msg = lib.ftkb_group_last_error(g._g).decode()
        assert all(w in msg for w in words), msg

    host = np.ascontiguousarray(snaps[0])
    rejected(host.ctypes.data, None, ["scalar", "not CUDA device memory"])
    pinned = torch.from_numpy(host).pin_memory()
    rejected(pinned.data_ptr(), None, ["scalar", "not CUDA device memory"])
    dev = _on(snaps, 0)
    raw = torch.zeros(dev[0].numel() + 1, dtype=torch.float64, device="cuda:0")
    rejected(raw.data_ptr() + 4, None, ["scalar", "aligned"])
    vec = torch.zeros(dev[0].numel() * 3, dtype=torch.float64, device="cuda:0")
    rejected(dev[0].data_ptr(), pinned.data_ptr(), ["vector", "not CUDA device memory"])
    if _ndev() >= 2:
        vec1 = vec.to("cuda:1")
        rejected(dev[0].data_ptr(), vec1.data_ptr(), ["vector", "another device"])
    with pytest.raises(ValueError):
        g.push_scalar_field_snapshot(dev[0].float())
    with pytest.raises(ValueError):
        g.push_scalar_field_snapshot(dev[0][:, :, :-1])
    # the group still takes the valid series
    for k in range(T):
        g.push_scalar_field_snapshot(dev[k])
        if k:
            g.advance_timestep()
        if k == T - 1:
            g.update_timestep()
    _same(_result(g.finalize()), want, f"after rejected pushes, chunk {chunk}")
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
  const bool device = std::string(argv[1]) == "device";
  const int W = 48, H = 40, T = 9;
  ftk_b200::critical_point_tracker_2d_regular tracker;
  tracker.set_device_ids({0, 0});
  tracker.set_time_chunk(3);
  tracker.set_domain(ftk_b200::lattice({2, 2}, {W - 4, H - 4}));
  tracker.set_array_domain(ftk_b200::lattice({0, 0}, {W, H}));
  tracker.set_scalar_field_source(ftk_b200::SOURCE_GIVEN);
  tracker.set_vector_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_field_source(ftk_b200::SOURCE_DERIVED);
  tracker.set_jacobian_symmetric(true);
  tracker.initialize();
  std::vector<double> h((size_t)W * H);
  double *d = nullptr;
  if (cudaMalloc(&d, h.size() * sizeof(double)) != cudaSuccess) return 3;
  for (int k = 0; k < T; k++) {
    for (int y = 0; y < H; y++)
      for (int x = 0; x < W; x++) h[x + W * y] = std::cos(0.31 * x + 0.05 * k) * std::sin(0.27 * y - 0.07 * k) + 0.01 * x;
    if (device) {
      if (cudaMemcpy(d, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) return 3;
      tracker.push_scalar_field_snapshot(ftk_b200::ndarray<double>::wrap(d, {(size_t)W, (size_t)H}, true));
    } else {
      tracker.push_scalar_field_snapshot(ftk_b200::ndarray<double>::wrap(h.data(), {(size_t)W, (size_t)H}));
    }
    if (k) tracker.advance_timestep();
    if (k == T - 1) tracker.update_timestep();
  }
  tracker.finalize();
  tracker.write_traced_critical_points_text(std::cout);
  std::printf("points=%zu\n", tracker.get_critical_points().size());
  cudaFree(d);
  return 0;
}
'''


def test_cpp_shim_device_ndarray_on_device_list(tmp_path):
    from ftk_b200 import build
    build.build()
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    src = tmp_path / "shim_device.cpp"
    src.write_text(SHIM_PROGRAM)
    exe = tmp_path / "shim_device"
    lib = os.path.join(ROOT, "ftk_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           str(src), "-o", str(exe), "-L" + lib, "-lftkb200", "-Wl,-rpath," + lib,
                           "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(cuda, "lib64")])
    outs = {}
    for mode in ("host", "device"):
        r = subprocess.run([str(exe), mode], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs[mode] = r.stdout
    assert "points=0" not in outs["host"] and len(outs["host"]) > 100
    assert outs["device"] == outs["host"]

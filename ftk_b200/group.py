"""Several GPUs behind one tracker: Python mirror of ftkb_group (include/ftkb200.h, ftk_b200/csrc/group.cpp).

The reference hands a device list to every filter (filter.hh:47-51 set_device_ids); here one process drives the devices
through time chunks (chunk c = `chunk` consecutive timesteps, swept by a context of its own on device_ids[c mod N], one host
thread per device), or, with chunk=0 (3D), through z-slabs that every device sweeps at every step.  Results equal the
one-device tracker bit for bit; ftkb_group_finalize merges everything into one context, which this class then exposes through
the ordinary tracker getters.  streaming=True grows trajectories there as a single streaming tracker does; coords=(mode, data)
takes make_tracker's forms, for the whole array.

Snapshots are numpy arrays (host memory) or device arrays -- torch CUDA tensors, or anything with __cuda_array_interface__ --
on any visible device, one of the group's or not: every device then copies what it needs from the source device (peer copies
over NVLink), ordered after torch's current stream on the tensor's device.  Either kind is consumed before the push returns.
A producer decomposed over several GPUs pushes its pieces as they are (push_field_data_snapshot_pieces): every device then
copies only the planes it needs, from whichever pieces hold them; slab(s) tells where z-slab s needs planes.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .tracker import coords_arg, make_tracker, _dev_ptr, _RegularTracker, SOURCE_DERIVED, SOURCE_GIVEN, SOURCE_NONE


class _GroupRoot(_RegularTracker):
    """tracker view of the group's merged context (owned by the group: closing the view only forgets the handle)"""

    def close(self):
        self._h = None
        self._keep = []

    def __del__(self):
        pass


class GroupTracker:
    def __init__(self, dims, device_ids, field="scalar", chunk=8, lb=None, ub=None, jacobian_symmetric=None, robust=True,
                 compute_degrees=False, type_filter=None, start_timestep=0, streaming=False, coords=None,
                 scalar_source=None, vector_source=None, jacobian_source=None):
        nd = len(dims)
        if field == "scalar":
            ss, vs, js, sym, margin = SOURCE_GIVEN, SOURCE_DERIVED, SOURCE_DERIVED, True, 2
        else:
            ss, vs, js, sym, margin = SOURCE_NONE, SOURCE_GIVEN, SOURCE_DERIVED, False, 1
        lo = [margin] * nd if lb is None else list(lb)
        hi = [d - 2 for d in dims] if ub is None else list(ub)
        cfg = L.Config()
        cfg.abi_version = L.ABI_VERSION
        cfg.nd = nd
        for i in range(3):
            cfg.dims[i] = dims[i] if i < nd else 1
            cfg.lb[i] = lo[i] if i < nd else 0
            cfg.ub[i] = hi[i] if i < nd else 0
        cfg.scalar_source = ss if scalar_source is None else int(scalar_source)
        cfg.vector_source = vs if vector_source is None else int(vector_source)
        cfg.jacobian_source = js if jacobian_source is None else int(jacobian_source)
        cfg.jacobian_symmetric = int(sym if jacobian_symmetric is None else jacobian_symmetric)
        cfg.robust_detection = int(robust)
        cfg.compute_degrees = int(compute_degrees)
        cfg.use_type_filter = int(type_filter is not None)
        cfg.type_filter = int(type_filter or 0)
        cfg.start_timestep = int(start_timestep)
        ids = (C.c_int32 * len(device_ids))(*[int(d) for d in device_ids])
        g = C.c_void_p()
        rc = L.lib().ftkb_group_create(C.byref(cfg), ids, len(device_ids), int(chunk), C.byref(g))
        if rc:
            raise L.FTKBError(rc, "ftkb_group_create failed (device ids?)")
        self._g = g
        self._dims, self._field, self._nd = list(dims), field, nd
        self._root = None
        if streaming:
            self._check(L.lib().ftkb_group_set_streaming_trajectories(g, 1))
        if coords is not None:      # copied by the library before the call returns
            mode, data = coords_arg(coords)
            self._check(L.lib().ftkb_group_set_coords(g, mode, data.ctypes.data, data.size))

    def _check(self, rc):
        if rc:
            raise L.FTKBError(rc, L.lib().ftkb_group_last_error(self._g).decode())

    def push_scalar_field_snapshot(self, a):
        self.push_field_data_snapshot(scalar=a)

    def push_vector_field_snapshot(self, a):
        self.push_field_data_snapshot(vector=a)

    def push_field_data_snapshot(self, scalar=None, vector=None, jacobian=None):
        """ref: critical_point_tracker.hh:202-213.  Host arrays, or float64 device arrays on one device (any visible one):
        copied to every device of the group before the call returns."""
        n = self._nd
        shape = tuple(reversed(self._dims))
        ptrs, hold, on_device = [], [], None
        for a, trailing in ((scalar, ()), (vector, (n,)), (jacobian, (n, n))):
            if a is None:
                ptrs.append(None)
                continue
            dp = _dev_ptr(a)
            count = int(np.prod(shape + trailing))
            if dp is not None:
                if int(np.prod(tuple(a.shape))) != count or (hasattr(a, "is_contiguous") and not a.is_contiguous()):
                    raise ValueError("device array has the wrong size or is not contiguous")
                if str(getattr(a, "dtype", "")) != "torch.float64" and getattr(a, "__cuda_array_interface__", {}).get("typestr") != "<f8":
                    raise ValueError("device arrays must be float64")
                ptrs.append(dp)
            else:
                h = np.ascontiguousarray(a, dtype=np.float64)
                if h.size != count:
                    raise ValueError(f"array has {h.size} elements, expected {count}")
                ptrs.append(h.ctypes.data)
                a = h
            hold.append(a)
            if on_device is not None and on_device != (dp is not None):
                raise ValueError("scalar/vector/jacobian must all be host arrays or all be device arrays")
            on_device = dp is not None
        if on_device:
            self._order_after_producer(hold)
            self._check(L.lib().ftkb_group_push_snapshot_device(self._g, ptrs[0], ptrs[1], ptrs[2]))
        else:
            self._check(L.lib().ftkb_group_push_snapshot(self._g, ptrs[0], ptrs[1], ptrs[2]))

    def push_field_data_snapshot_pieces(self, scalar=None, vector=None, jacobian=None):
        """A snapshot in pieces along the slowest axis (z in 3D, y in 2D), the way a decomposed producer holds it: each argument
        is a list of float64 device arrays (torch CUDA tensors or __cuda_array_interface__ objects), one per piece, in plane
        order, each piece's arrays on one device (any visible one).  A piece's leading dimension is its plane count: shapes
        (count, H, W) for a 3D scalar, (count, W) for a 2D one, with trailing (n,) or (n, n) for vector and Jacobian.  Every copy
        from a torch tensor waits for torch's current stream on its device; other producers synchronise before pushing.  Copied
        to every device that needs the planes before the call returns (ftkb_group_push_pieces_device)."""
        n = self._nd
        lists = [list(a) if a is not None else None for a in (scalar, vector, jacobian)]
        given = [a for a in lists if a is not None]
        if not given or any(len(a) != len(given[0]) for a in given):
            raise ValueError("pass one array per piece for every array, the same number of pieces for each")
        plane = tuple(reversed(self._dims))[1:]
        pieces = (L.Piece * len(given[0]))()
        first = 0
        for i, p in enumerate(pieces):
            count = None
            for a, trailing, field in zip(lists, ((), (n,), (n, n)), ("scalar", "vector", "jacobian")):
                if a is None:
                    continue
                x = a[i]
                if x is None:       # (refused by the library: every piece passes the same arrays)
                    continue
                dp = _dev_ptr(x)
                if dp is None:
                    raise ValueError(f"piece {i}: the {field} array is not a device array")
                shape = tuple(x.shape)
                if len(shape) != 1 + len(plane) + len(trailing) or shape[1:] != plane + trailing or \
                        (hasattr(x, "is_contiguous") and not x.is_contiguous()):
                    raise ValueError(f"piece {i}: the {field} array has shape {shape}, expected (count,) + {plane + trailing}, contiguous")
                if str(getattr(x, "dtype", "")) != "torch.float64" and getattr(x, "__cuda_array_interface__", {}).get("typestr") != "<f8":
                    raise ValueError(f"piece {i}: device arrays must be float64")
                if count is not None and shape[0] != count:
                    raise ValueError(f"piece {i}: its arrays hold different numbers of planes")
                count = shape[0]
                setattr(p, field, dp)
                if getattr(x, "is_cuda", False) and hasattr(x, "data_ptr"):
                    import torch
                    p.stream = int(torch.cuda.current_stream(x.device).cuda_stream)
                    p.has_stream = 1
            p.first, p.count = first, count or 0
            first += count or 0
        self._check(L.lib().ftkb_group_push_pieces_device(self._g, pieces, len(pieces)))

    def slab(self, s):
        """z-slab mode: (c0, c1, a0, a1), the corner planes slab s owns and the array planes it holds (ftkb_group_get_slab)"""
        planes = (C.c_int32 * 4)()
        self._check(L.lib().ftkb_group_get_slab(self._g, int(s), planes))
        return tuple(planes)

    def _order_after_producer(self, arrays):
        """device inputs: every copy waits for torch's current stream on the tensor's device (ftkb_group_set_producer_stream);
        other producers synchronise before pushing"""
        for a in arrays:
            if getattr(a, "is_cuda", False) and hasattr(a, "data_ptr"):
                import torch
                stream = int(torch.cuda.current_stream(a.device).cuda_stream)
                self._check(L.lib().ftkb_group_set_producer_stream(self._g, C.c_void_p(stream), 1))
                return

    def push_synthetic_snapshot(self, kind, params, t):
        p = (C.c_double * max(len(params), 1))(*[float(v) for v in params])
        self._check(L.lib().ftkb_group_push_synthetic(self._g, int(kind), p, len(params), float(t)))

    def advance_timestep(self):
        self._check(L.lib().ftkb_group_advance_timestep(self._g))

    def update_timestep(self):
        self._check(L.lib().ftkb_group_update_timestep(self._g))

    def finalize(self):
        """merge every chunk's punctured simplices into one context on the first device and trace there; returns a tracker
        view of that context (owned by the group: valid until close())"""
        h = C.c_void_p()
        self._check(L.lib().ftkb_group_finalize(self._g, C.byref(h)))
        view = _GroupRoot()
        view.ND = self._nd
        view._h = h
        view._dims = list(self._dims)
        self._root = view
        return view

    def live_curveset(self):
        """streaming groups, at any time: (grown_through, CurveSet) after the grow steps of every interval swept so far --
        call for call what Tracker.live_curveset of one tracker fed the same series returns"""
        from .curves import CurveSet
        return CurveSet.live(L.lib().ftkb_group_get_live_curveset, self._g, self._check)

    def stats(self):
        s, n = L.Stats(), C.c_int32()
        self._check(L.lib().ftkb_group_get_stats(self._g, C.byref(s), C.byref(n)))
        d = s.as_dict()
        d["chunks_done"] = n.value
        return d

    def close(self):
        if self._g:
            if self._root is not None:
                self._root._h = None
            L.lib().ftkb_group_destroy(self._g)
            self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def track_on_devices(snapshots, dims, device_ids, field="scalar", chunk=8, **kw):
    """the reference's front-end loop (python/pyftk.cpp:110-117) on several devices; returns (group, root tracker view)"""
    g = GroupTracker(dims, device_ids, field=field, chunk=chunk, **kw)
    snaps = list(snapshots)
    for k, s in enumerate(snaps):
        if field == "scalar":
            g.push_scalar_field_snapshot(s)
        else:
            g.push_vector_field_snapshot(s)
        if k != 0:
            g.advance_timestep()
        if k == len(snaps) - 1:
            g.update_timestep()
    return g, g.finalize()

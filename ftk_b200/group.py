"""Several GPUs behind one tracker: Python mirror of ftkb_group (include/ftkb200.h, ftk_b200/csrc/group.cpp).

The reference hands a device list to every filter (filter.hh:47-51 set_device_ids); here one process drives the devices
through time chunks (chunk c = `chunk` consecutive timesteps, swept by a context of its own on device_ids[c mod N], one host
thread per device), or, with chunk=0 (3D), through z-slabs that every device sweeps at every step.  Results equal the
one-device tracker bit for bit; ftkb_group_finalize merges everything into one context, which this class then exposes through
the ordinary tracker getters.  streaming=True grows trajectories there as a single streaming tracker does; coords=(mode, data)
takes make_tracker's forms, for the whole array.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .tracker import coords_arg, make_tracker, _RegularTracker, SOURCE_DERIVED, SOURCE_GIVEN, SOURCE_NONE


class _GroupRoot(_RegularTracker):
    """tracker view of the group's merged context (owned by the group: closing the view only forgets the handle)"""

    def close(self):
        self._h = None
        self._keep = []

    def __del__(self):
        pass


class GroupTracker:
    def __init__(self, dims, device_ids, field="scalar", chunk=8, lb=None, ub=None, jacobian_symmetric=None, robust=True,
                 compute_degrees=False, type_filter=None, start_timestep=0, streaming=False, coords=None):
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
        cfg.scalar_source, cfg.vector_source, cfg.jacobian_source = ss, vs, js
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
        h = np.ascontiguousarray(a, dtype=np.float64)
        self._check(L.lib().ftkb_group_push_snapshot(self._g, h.ctypes.data, None, None))

    def push_vector_field_snapshot(self, a):
        h = np.ascontiguousarray(a, dtype=np.float64)
        self._check(L.lib().ftkb_group_push_snapshot(self._g, None, h.ctypes.data, None))

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

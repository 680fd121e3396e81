"""Traced trajectories as a mutable curve set + the reference's trajectory post-processing (SURVEY.md 8f3).

Mirror of ftk::feature_curve_set_t (include/ftk/features/feature_curve_set.hh) with
feature_curve_set_post_processor_t::filter (include/ftk/filters/feature_curve_set_post_processor.hh:23-70) and the legacy
json_interface::post_process() sequence (include/ftk/filters/json_interface.hh:758-800).  The work is host code inside
libftkb200.so (ftk_b200/csrc/curves.cpp); this module only moves arrays across the C ABI.
"""
import ctypes as C

import numpy as np

from . import _lib as L


class CurveSet:
    def __init__(self, handle):
        self._h = handle

    @classmethod
    def from_trajectories(cls, points, trajectories):
        """points: POINT_DTYPE array; trajectories: list of (index array, loop flag) in trace order (ids 0 .. n-1)"""
        pts = np.ascontiguousarray(points, dtype=L.POINT_DTYPE)
        off = np.zeros(len(trajectories) + 1, np.uint64)
        for i, (idx, _) in enumerate(trajectories):
            off[i + 1] = off[i] + len(idx)
        idx = (np.concatenate([np.asarray(t[0], np.uint64) for t in trajectories]) if trajectories else np.zeros(0, np.uint64))
        idx = np.ascontiguousarray(idx, np.uint64)
        loop = np.ascontiguousarray([1 if t[1] else 0 for t in trajectories], np.uint8)
        h = C.c_void_p()
        rc = L.lib().ftkb_curveset_create(pts.ctypes.data, len(pts), off.ctypes.data, idx.ctypes.data if len(idx) else None,
                                          loop.ctypes.data if len(loop) else None, len(trajectories), C.byref(h))
        if rc:
            raise L.FTKBError(rc, "curveset_create: bad trajectories")
        return cls(h)

    @classmethod
    def from_tracker(cls, tracker):
        """get_traced_critical_points() of a finalized tracker"""
        h = C.c_void_p()
        tracker._check(L.lib().ftkb_get_curveset(tracker._h, C.byref(h)))
        return cls(h)

    @classmethod
    def live(cls, get, handle, check):
        """(grown_through, CurveSet) of a streaming tracker or group at any time: `get` is ftkb_get_live_curveset or
        ftkb_group_get_live_curveset, `check` turns its return code into an exception"""
        h, t = C.c_void_p(), C.c_int32()
        check(get(handle, C.byref(t), C.byref(h)))
        return t.value, cls(h)

    def post_process(self, ops):
        rc = L.lib().ftkb_curveset_post_process(self._h, ops.encode())
        if rc:
            raise L.FTKBError(rc, L.lib().ftkb_curveset_last_error(self._h).decode())
        return self

    def arrays(self):
        """(infos: CURVE_INFO_DTYPE array in multimap order, points: CURVE_POINT_DTYPE array, curve i = points[first:first+count])"""
        nc, npt = C.c_uint64(), C.c_uint64()
        L.lib().ftkb_curveset_size(self._h, C.byref(nc), C.byref(npt))
        infos = np.zeros(nc.value, L.CURVE_INFO_DTYPE)
        pts = np.zeros(npt.value, L.CURVE_POINT_DTYPE)
        L.lib().ftkb_curveset_get(self._h, infos.ctypes.data if nc.value else None, pts.ctypes.data if npt.value else None)
        return infos, pts

    def slice(self, timestep):
        """sliced critical points of one timestep: the ordinal points of the curves (CURVE_POINT_DTYPE array)"""
        n = C.c_uint64()
        L.lib().ftkb_curveset_slice(self._h, int(timestep), None, 0, C.byref(n))
        out = np.zeros(n.value, L.CURVE_POINT_DTYPE)
        if n.value:
            L.lib().ftkb_curveset_slice(self._h, int(timestep), out.ctypes.data, n.value, C.byref(n))
        return out

    def curves(self):
        infos, pts = self.arrays()
        return [(infos[i], pts[int(infos[i]["first"]):int(infos[i]["first"] + infos[i]["count"])]) for i in range(len(infos))]

    def __len__(self):
        nc = C.c_uint64()
        L.lib().ftkb_curveset_size(self._h, C.byref(nc), None)
        return int(nc.value)

    def close(self):
        if self._h:
            L.lib().ftkb_curveset_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

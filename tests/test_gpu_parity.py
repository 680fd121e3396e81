"""GPU: the CUDA path, called through the C ABI (libftkb200.so), against the parity oracle and the
fixtures produced by the unmodified reference.

Bar (north_star / SURVEY.md App. A10): punctured set, simplex types, ordinal flags, timesteps and
critical-point types bit-exact; trajectories equal as a set of ordered sequences; interpolated
x/y/z/t and scalar within 1e-9 absolute in grid units.
"""
import numpy as np
import pytest

import _parity as P

pytestmark = pytest.mark.gpu

TOL = 1e-9   # north_star tolerance on interpolated coordinates / scalar


@pytest.fixture(scope="module")
def ftk():
    import ftk_b200
    from ftk_b200 import _lib
    if _lib.lib().ftkb_device_count() < 1:
        pytest.fail("no sm_100 device visible: the CUDA path cannot run (there is no fallback)")
    return ftk_b200


def cuda_result(tr):
    return {"points": tr.get_discrete_critical_points(), "trajectories": tr.get_trajectory_index()}


@pytest.mark.parametrize("name", P.golden_names())
def test_cuda_matches_reference_golden(name, ftk, oracle):
    meta, gold, inp = P.load_golden(name)
    snaps = P.golden_snapshots(meta, inp, oracle)
    field = "scalar" if meta["nv"] == 1 else "vector"
    tr = ftk.track(snaps, meta["dims"], field=field, jacobian_symmetric=meta["symmetric"])
    got = cuda_result(tr)
    P.assert_same_result(got, gold, tol=TOL, what=name)
    st = tr.stats()
    assert st["kernel_launches"] > 0 and st["simplices_tested"] > 0
    tr.close()


def _both(ftk, oracle, snaps, dims, field, **kw):
    o = oracle.track(snaps, dims, field=field, **kw)
    c = ftk.track(snaps, dims, field=field, **kw)
    return c, o


def _rand_series(rng, dims, T, nv, kind):
    shape = tuple(reversed(dims)) + ((nv,) if nv > 1 else ())
    if kind == "int":
        return [rng.integers(-3, 4, size=shape).astype(np.float64) for _ in range(T)]
    if kind == "smooth":
        grids = np.meshgrid(*[np.arange(d, dtype=np.float64) for d in reversed(dims)], indexing="ij")
        out = []
        for k in range(T):
            comps = []
            for c in range(max(nv, 1)):
                f = 0.0
                for q, g in enumerate(grids):
                    f = f + np.cos((0.7 + 0.17 * c * (q + 1)) * g + 0.3 * q + 0.11 * k + 1.3 * c) * (1.0 + 0.2 * q)
                comps.append(f + 0.05 * rng.standard_normal(size=f.shape))
            out.append(np.stack(comps, axis=-1) if nv > 1 else comps[0])
        return out
    return [rng.standard_normal(size=shape) for _ in range(T)]


CASES = [
    # dims, T, field, kind, extra tracker kwargs
    ([17, 13], 4, "scalar", "normal", {}),
    ([17, 13], 4, "scalar", "int", {}),
    ([40, 35], 5, "scalar", "smooth", {}),
    ([16, 12], 4, "vector", "normal", {}),
    ([16, 12], 4, "vector", "int", {}),
    ([16, 12], 4, "vector", "normal", {"jacobian_symmetric": True}),
    ([33, 9], 3, "vector", "smooth", {}),
    ([14, 12], 3, "scalar", "normal", {"compute_degrees": True}),
    ([14, 12], 3, "scalar", "normal", {"type_filter": 0x2 | 0x8}),
    ([14, 12], 3, "vector", "normal", {"lb": [0, 0], "ub": [13, 11]}),           # domain = whole array
    ([14, 12], 3, "scalar", "normal", {"lb": [3, 1], "ub": [9, 10]}),
    ([14, 12], 3, "scalar", "normal", {"start_timestep": 5}),
    ([70, 5], 3, "vector", "normal", {}),                                        # several x strips, ragged
    ([9, 8, 7], 3, "scalar", "normal", {}),
    ([9, 8, 7], 3, "scalar", "int", {}),
    ([12, 11, 10], 3, "scalar", "smooth", {}),
    ([8, 7, 7], 3, "vector", "normal", {}),
    ([8, 7, 7], 3, "vector", "int", {}),
    ([8, 7, 7], 3, "vector", "normal", {"jacobian_symmetric": True}),
    ([8, 7, 7], 3, "vector", "normal", {"robust": False}),
    ([8, 7, 6], 3, "vector", "normal", {"lb": [0, 0, 0], "ub": [7, 6, 5]}),
    ([36, 20, 5], 2, "vector", "smooth", {}),                                    # several x/y tiles
    ([7, 6, 40], 2, "scalar", "smooth", {}),                                     # several z chunks
    # fused 3D scan (even W: gradient derived inside the TMA-staged scan kernel)
    ([132, 70, 9], 2, "scalar", "smooth", {}),                                   # interior + edge tiles, 3 x strips, 3 y tiles
    ([14, 12, 10], 3, "scalar", "int", {}),                                      # ties and exact zeros
    ([20, 40, 30], 2, "scalar", "normal", {}),                                   # noise: every lane takes the per-cube path
    ([64, 36, 20], 2, "scalar", "smooth", {"lb": [0, 0, 0], "ub": [63, 35, 19]}),  # domain = whole array (zero-gradient border)
    ([66, 34, 12], 2, "scalar", "smooth", {"lb": [5, 3, 2], "ub": [60, 33, 7]}),
    ([16, 12, 60], 2, "scalar", "smooth", {}),                                   # z chunks
    ([64, 10, 8], 3, "scalar", "smooth", {"start_timestep": 3}),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_cuda_matches_oracle_random(case, ftk, oracle):
    dims, T, field, kind, kw = CASES[case]
    rng = np.random.default_rng(1000 + case)
    nv = 1 if field == "scalar" else len(dims)
    snaps = _rand_series(rng, dims, T, nv, kind)
    c, o = _both(ftk, oracle, snaps, dims, field, **kw)
    got, want = cuda_result(c), P.oracle_result(o)
    assert len(want["points"]) > 0, "degenerate test case: the oracle found nothing"
    P.assert_same_result(got, want, tol=TOL, what=f"case {case}")
    # component partition (special nodes included) and node degrees, bit-exact
    assert np.array_equal(c.get_component_labels(), o.component_labels())
    assert np.array_equal(c.get_degrees(), o.degrees())
    assert c.stats()["scaling_factor"] == o.scaling_factor
    c.close()


def test_fused_3d_scan_non_finite_scalars_fall_back(ftk, oracle):
    """NaN / Inf / huge scalars cannot be bracketed by the fused 3D scan's keys: it raises its poison flag and
    the step is redone on the unfused path -- results still match the oracle"""
    rng = np.random.default_rng(314)
    dims, T = [16, 14, 12], 3
    snaps = _rand_series(rng, dims, T, 1, "smooth")
    snaps[1][5, 6, 7] = np.nan
    snaps[1][3, 3, 3] = np.inf
    snaps[2][8, 9, 10] = 1e305
    c, o = _both(ftk, oracle, snaps, dims, "scalar")
    P.assert_same_result(cuda_result(c), P.oracle_result(o), tol=TOL, what="non-finite 3D scalars")
    assert c.stats()["sweeps_repeated"] >= 1
    c.close()


def test_fused_3d_scan_equals_unfused(ftk, monkeypatch):
    """FTKB_SCAN3D=plain materialises the gradient and runs the vector-layer scan: same points, same
    trajectories, same quantisation factor as the fused scan, and the fused worklist is a superset filter"""
    rng = np.random.default_rng(2718)
    dims, T = [130, 68, 10], 3
    snaps = _rand_series(rng, dims, T, 1, "smooth")
    a = ftk.track(snaps, dims, field="scalar")
    monkeypatch.setenv("FTKB_SCAN3D", "plain")
    b = ftk.track(snaps, dims, field="scalar")
    monkeypatch.delenv("FTKB_SCAN3D")
    pa, pb = a.get_discrete_critical_points(), b.get_discrete_critical_points()
    assert len(pa) > 0 and np.array_equal(pa, pb)
    assert P.canonical_trajectories(a.get_trajectory_index()) == P.canonical_trajectories(b.get_trajectory_index())
    sa, sb = a.stats(), b.stats()
    assert sa["scaling_factor"] == sb["scaling_factor"] and sa["resolution"] == sb["resolution"]
    assert sa["ms_derive"] == 0.0 and sb["ms_derive"] > 0.0          # the fused path never launches the gradient kernel
    # every punctured simplex's cube is in the fused scan's worklist (last sweep: ordinal simplices at T-1)
    wl = set(int(v) for v in a.get_last_worklist())
    last = pa[(pa["timestep"] == T - 1)]
    nc = [d - 3 for d in dims]
    for q in last:
        cx, cy, cz = int(q["corner"][0]) - 2, int(q["corner"][1]) - 2, int(q["corner"][2]) - 2
        assert cx + nc[0] * (cy + nc[1] * cz) in wl
    a.close()
    b.close()


@pytest.mark.parametrize("dims,T,env,value,field", [([200, 150], 4, "FTKB_SCAN2D", "f32", "scalar"), ([130, 70, 44], 3, "FTKB_SCAN3D", "plain", "scalar"),
                                                    ([200, 150], 4, "FTKB_VSCAN", "twolayer", "vector"), ([66, 70, 24], 3, "FTKB_VSCAN", "twolayer", "vector"),
                                                    ([131, 37], 3, "FTKB_VSCAN", "twolayer", "vector")])
def test_range_cell_scan_equals_fallback_scan(dims, T, env, value, field, ftk, oracle, monkeypatch):
    """default scan (each layer streamed once, 16-byte range cells kept per layer) against the fallback the same input takes
    when the default cannot run (FTKB_SCAN2D=f32: fp32-range build kernel; FTKB_SCAN3D=plain: materialised gradient;
    FTKB_VSCAN=twolayer: vector scan that re-reads both layers) and against the oracle: same points, same trajectories, same
    factor; every punctured simplex's cube is in the cell scan's worklist; a repeated sweep (cells only) changes nothing"""
    rng = np.random.default_rng(4242 + len(dims))
    snaps = _rand_series(rng, dims, T, 1 if field == "scalar" else len(dims), "smooth")
    a = ftk.track(snaps, dims, field=field)
    monkeypatch.setenv(env, value)
    b = ftk.track(snaps, dims, field=field)
    monkeypatch.delenv(env)
    pa, pb = a.get_discrete_critical_points(), b.get_discrete_critical_points()
    assert len(pa) > 0 and np.array_equal(pa, pb)
    assert P.canonical_trajectories(a.get_trajectory_index()) == P.canonical_trajectories(b.get_trajectory_index())
    assert a.stats()["scaling_factor"] == b.stats()["scaling_factor"] and a.stats()["resolution"] == b.stats()["resolution"]
    o = oracle.track(snaps, dims, field=field)
    P.assert_same_result(cuda_result(a), P.oracle_result(o), tol=TOL, what="range-cell scan")
    wl = set(int(v) for v in a.get_last_worklist())
    lo = 2 if field == "scalar" else 1
    nc = [d - 1 - lo for d in dims]
    for q in pa[pa["timestep"] == T - 1]:
        c = [int(v) - lo for v in q["corner"][:len(dims)]]
        lin = c[0] + nc[0] * (c[1] + (nc[1] * c[2] if len(dims) == 3 else 0))
        assert lin in wl
    a.close()
    b.close()
    # streaming form: an update_timestep repeated on resident layers sweeps from the cells alone
    tr = ftk.make_tracker(dims, field=field)
    for k in range(2):
        if field == "scalar":
            tr.push_scalar_field_snapshot(snaps[k])
        else:
            tr.push_vector_field_snapshot(snaps[k])
    tr.update_timestep()
    first = tr.get_discrete_critical_points().copy()
    tr.update_timestep()
    assert len(first) > 0 and np.array_equal(first, tr.get_discrete_critical_points())
    tr.close()


def test_2d_cell_scan_on_ragged_fields(ftk, oracle):
    """the 2D range-cell scan (16-byte aligned rows) on ragged fields over several CTA tiles, strips and row chunks: same
    results, scaling factor and resolution as the oracle"""
    rng = np.random.default_rng(9090)
    for dims, T in (([200, 150], 4), ([64, 35], 3), ([130, 17], 3)):
        snaps = _rand_series(rng, dims, T, 1, "smooth")
        c, o = _both(ftk, oracle, snaps, dims, "scalar")
        P.assert_same_result(cuda_result(c), P.oracle_result(o), tol=TOL, what=f"2D cell scan {dims}")
        assert c.stats()["scaling_factor"] == o.scaling_factor and c.stats()["resolution"] == o.resolution
        c.close()


def test_given_jacobian_and_scalar(ftk, oracle):
    """push_field_data_snapshot(scalar, vector, jacobian) with every field GIVEN"""
    rng = np.random.default_rng(5)
    dims, T = [13, 11], 3
    ot = oracle.Tracker(dims, field="vector", scalar_source=1, vector_source=1, jacobian_source=1, jacobian_symmetric=False)
    ct = ftk.make_tracker(dims, field="vector", scalar_source=1, vector_source=1, jacobian_source=1, jacobian_symmetric=False)
    for k in range(T):
        s, v, j = rng.standard_normal((11, 13)), rng.standard_normal((11, 13, 2)), rng.standard_normal((11, 13, 2, 2))
        for t in (ot, ct):
            t.push_field_data_snapshot(scalar=s, vector=v, jacobian=j)
            if k:
                t.advance_timestep()
            if k == T - 1:
                t.update_timestep()
    ot.finalize()
    ct.finalize()
    P.assert_same_result(cuda_result(ct), P.oracle_result(ot), tol=TOL, what="given jacobian")
    assert len(set(ct.get_discrete_critical_points()["cp_type"])) > 2   # foci / centres appear with a full Jacobian
    ct.close()


def test_empty_and_single_snapshot(ftk, oracle):
    """no punctured simplex at all; and a single snapshot (ordinal sweep only, extractors path)"""
    dims = [12, 10]
    s = np.ones((10, 12)) + np.arange(12)[None, :] * 1.0     # constant gradient: no critical point
    c, o = _both(ftk, oracle, [s, s + 1.0], dims, "scalar")
    assert len(c.get_discrete_critical_points()) == 0 == len(o.points())
    assert c.get_trajectory_index() == []
    c.close()
    rng = np.random.default_rng(11)
    c, o = _both(ftk, oracle, [rng.standard_normal((10, 12))], dims, "scalar")
    got = cuda_result(c)
    assert got["points"]["ordinal"].all() and len(got["points"]) > 0
    P.assert_same_result(got, P.oracle_result(o), tol=TOL, what="single snapshot")
    c.close()


def test_repeated_update_is_idempotent(ftk):
    """a second update_timestep on the same snapshots re-inserts the same map keys (std::map semantics)"""
    rng = np.random.default_rng(3)
    snaps = [rng.standard_normal((10, 12)) for _ in range(2)]
    tr = ftk.make_tracker([12, 10], field="scalar")
    tr.push_scalar_field_snapshot(snaps[0])
    tr.push_scalar_field_snapshot(snaps[1])
    tr.update_timestep()
    a = tr.get_discrete_critical_points().copy()
    tr.update_timestep()
    b = tr.get_discrete_critical_points()
    assert len(a) > 0 and np.array_equal(a, b)
    tr.close()


def test_buffers_grow_on_demand(ftk, oracle):
    """a noisy field larger than the initial worklist / point buffers: results still match the oracle"""
    rng = np.random.default_rng(21)
    dims, T = [300, 260], 2
    snaps = [rng.standard_normal((260, 300)) for _ in range(T)]
    c, o = _both(ftk, oracle, snaps, dims, "scalar", trace=False)
    got, want = c.get_discrete_critical_points(), o.points()
    assert len(want) > 2000
    P.assert_same_result({"points": got}, {"points": want}, check_trajectories=False, tol=TOL, what="noisy 300x260")
    st = c.stats()
    assert st["cells_refined"] > 65536    # the default worklist had to grow
    c.close()


def test_device_generator_matches_host_input(ftk, oracle):
    """ftkb_push_synthetic(moving_extremum) is bit-identical to pushing the host-generated field"""
    dims, T = [64, 48], 6
    x0, d = [30.3, 21.7], [0.4, 0.3]
    host = [oracle.gen_moving_extremum(dims, x0, d, float(k)) for k in range(T)]
    a = ftk.track(host, dims, field="scalar")
    b = ftk.make_tracker(dims, field="scalar")
    for k in range(T):
        b.push_synthetic_snapshot(0, x0 + d, float(k))
        if k:
            b.advance_timestep()
        if k == T - 1:
            b.update_timestep()
    b.finalize()
    pa, pb = a.get_discrete_critical_points(), b.get_discrete_critical_points()
    assert len(pa) > 0 and np.array_equal(pa, pb)
    assert P.canonical_trajectories(a.get_trajectory_index()) == P.canonical_trajectories(b.get_trajectory_index())
    a.close()
    b.close()


# ---- full-size properties (sizes the oracle cannot finish in seconds) ----------------------------
def _track_moving_extremum(ftk, dims, x0, d, T):
    tr = ftk.make_tracker(dims, field="scalar")
    for k in range(T):
        tr.push_synthetic_snapshot(0, list(x0) + list(d), float(k))
        if k:
            tr.advance_timestep()
        if k == T - 1:
            tr.update_timestep()
    tr.finalize()
    return tr


def test_moving_extremum_2d_full_width_line_equation(ftk):
    """BASELINE configs[1] at full spatial size (8192^2), 4 timesteps: exactly one trajectory, every
    point on x = x0 + dir t (the reference's own moving-extremum check,
    tests/test_critical_point_tracking_moving_extremum_2d.cpp:23-95), all minima, and the
    scan kernel refined only a handful of the 6.7e7 cubes per step."""
    dims, x0, d, T = [8192, 8192], (4096.3, 4095.7), (0.1, 0.1), 4
    tr = _track_moving_extremum(ftk, dims, x0, d, T)
    pts = tr.get_discrete_critical_points()
    trajs = tr.get_trajectory_index()
    assert len(trajs) == 1 and len(trajs[0][0]) == len(pts) and len(pts) >= 2 * T - 1
    for q in range(2):
        assert np.abs(pts["x"][:, q] - (x0[q] + d[q] * pts["t"])).max() < 1e-9
    assert (pts["cp_type"] == 2).all()
    st = tr.stats()
    assert st["simplices_tested"] == 8189 * 8189 * (12 * (T - 1) + 2)
    assert st["cells_refined"] < 64 * T
    tr.close()


def test_moving_extremum_3d_line_equation(ftk):
    """BASELINE configs[2] generator at 256^3 x 3 (pentachora mesh)"""
    dims, x0, d, T = [256, 256, 256], (128.3, 127.7, 128.1), (0.1, 0.11, 0.1), 3
    tr = _track_moving_extremum(ftk, dims, x0, d, T)
    pts = tr.get_discrete_critical_points()
    trajs = tr.get_trajectory_index()
    assert len(trajs) == 1 and len(trajs[0][0]) == len(pts) and len(pts) >= 2 * T - 1
    for q in range(3):
        assert np.abs(pts["x"][:, q] - (x0[q] + d[q] * pts["t"])).max() < 1e-9
    assert (pts["cp_type"] == 2).all()
    assert tr.stats()["simplices_tested"] == 253 ** 3 * (60 * (T - 1) + 6)
    tr.close()


def test_time_slab_split_equals_single_run(ftk, oracle):
    """two contexts, each owning a contiguous time slab (+ one halo layer and the inherited running
    resolution), merged by a final union-find over the imported points == one sequential run"""
    rng = np.random.default_rng(77)
    dims, T, cut = [24, 20], 8, 4
    snaps = _rand_series(rng, dims, T, 1, "smooth")
    whole = ftk.track(snaps, dims, field="scalar")
    want = cuda_result(whole)
    o = oracle.track(snaps, dims, field="scalar")
    P.assert_same_result(want, P.oracle_result(o), tol=TOL, what="whole run")
    # slab 0: timesteps [0, cut) needs layers 0..cut ; slab 1: [cut, T) needs layers cut..T-1
    a = ftk.make_tracker(dims, field="scalar")
    for k in range(0, cut + 1):
        a.push_scalar_field_snapshot(snaps[k])
        if k:
            a.advance_timestep()
    res = a.stats()["resolution"]
    b = ftk.make_tracker(dims, field="scalar", start_timestep=cut, resolution_init=res)
    for k in range(cut, T):
        b.push_scalar_field_snapshot(snaps[k])
        if k > cut:
            b.advance_timestep()
        if k == T - 1:
            b.update_timestep()
    a.import_points(b.get_discrete_critical_points())
    a.finalize()
    P.assert_same_result(cuda_result(a), want, tol=0.0, what="time-slab merge")
    for t in (whole, a, b):
        t.close()


# ---- time-slab halo through peer memory (two processes, IPC handles) --------------------------------------------
def _upper_slab_worker(dims, field, snaps_upper, cut, res_init, q_out, q_in):
    """process of the slab above: builds the range cells of its first layer, exports layer + cells, waits for the slab
    below to finish its last sweep, then completes its own slab"""
    import torch
    import ftk_b200
    from ftk_b200 import _lib
    ndev = torch.cuda.device_count()
    dev = torch.device("cuda", 1 if ndev >= 2 else 0)      # the upper slab on its own GPU when there is one: the halo then crosses NVLink
    torch.cuda.set_device(dev)
    first = torch.from_numpy(np.ascontiguousarray(snaps_upper[0])).to(dev)       # stays alive while the neighbour reads it
    tr = ftk_b200.make_tracker(dims, field=field, start_timestep=cut, resolution_init=res_init, device=dev.index)
    kw = "scalar" if field == "scalar" else "vector"
    tr.push_device_pointers(**{kw: int(first.data_ptr())})
    if field == "scalar":
        tr.push_scalar_field_snapshot(snaps_upper[1])
    else:
        tr.push_vector_field_snapshot(snaps_upper[1])
    tr.update_timestep()
    cptr, _, cres = tr.export_layer_cells(0)
    q_out.put((_lib.ipc_export(int(first.data_ptr())), _lib.ipc_export(cptr), cres))
    assert q_in.get(timeout=120) == "done"
    tr.advance_timestep()
    for k in range(2, len(snaps_upper)):
        if field == "scalar":
            tr.push_scalar_field_snapshot(snaps_upper[k])
        else:
            tr.push_vector_field_snapshot(snaps_upper[k])
        tr.advance_timestep()
    tr.update_timestep()
    q_out.put(tr.get_discrete_critical_points().tobytes())
    tr.close()


def _lower_slab_worker(dims, field, snaps_lower, q_from_upper, q_to_upper, q_out):
    """process of the slab below: its last sweep reads the neighbour's first layer in place (cells + sparse vertices)"""
    import ftk_b200
    from ftk_b200 import _lib
    lh, ch, cres = q_from_upper.get(timeout=120)
    layer, cells = _lib.ipc_import(lh, 0), _lib.ipc_import(ch, 0)
    tr = ftk_b200.make_tracker(dims, field=field)
    for k, s in enumerate(snaps_lower):
        if field == "scalar":
            tr.push_scalar_field_snapshot(s)
        else:
            tr.push_vector_field_snapshot(s)
        if k:
            tr.advance_timestep()
    kw = "scalar" if field == "scalar" else "vector"
    tr.push_remote_snapshot(**{kw: layer, "cells": cells, "resolution": cres})
    tr.advance_timestep()
    q_out.put((tr.get_discrete_critical_points().tobytes(), tr.stats()["kernel_launches"]))
    q_to_upper.put("done")
    tr.close()


@pytest.mark.parametrize("dims,field", [([70, 40], "scalar"), ([66, 36, 12], "scalar"), ([66, 36, 12], "vector"), ([70, 40], "vector")])
def test_time_slab_halo_through_peer_memory(dims, field, ftk, oracle):
    """two processes own the two time slabs; the lower one never receives the upper slab's first layer: it maps the
    neighbour's layer and range cells (CUDA IPC; NVLink peer memory between GPUs) and sweeps them in place.
    Merged result == one sequential run == the oracle."""
    import multiprocessing as mp
    from ftk_b200 import _lib
    rng = np.random.default_rng(555 + len(dims))
    T, cut = 6, 3
    snaps = _rand_series(rng, dims, T, 1 if field == "scalar" else len(dims), "smooth")
    whole = ftk.track(snaps, dims, field=field)
    want = cuda_result(whole)
    P.assert_same_result(want, P.oracle_result(oracle.track(snaps, dims, field=field)), tol=TOL, what="whole run")
    # the running resolution the upper slab inherits (layers 0 .. cut)
    probe = ftk.make_tracker(dims, field=field)
    for k in range(cut + 1):
        (probe.push_scalar_field_snapshot if field == "scalar" else probe.push_vector_field_snapshot)(snaps[k])
        if k:
            probe.advance_timestep()
    res = probe.stats()["resolution"]
    probe.close()
    ctx = mp.get_context("spawn")
    q_handles, q_done, q_up, q_lo = ctx.Queue(), ctx.Queue(), ctx.Queue(), ctx.Queue()
    up = ctx.Process(target=_upper_slab_worker, args=(dims, field, snaps[cut:], cut, res, q_up, q_done))
    up.start()
    handles = q_up.get(timeout=180)
    q_handles.put(handles)
    lo = ctx.Process(target=_lower_slab_worker, args=(dims, field, snaps[:cut], q_handles, q_done, q_lo))
    lo.start()
    lo_pts, lo_launches = q_lo.get(timeout=180)
    up_pts = q_up.get(timeout=180)
    lo.join(60)
    up.join(60)
    assert lo.exitcode == 0 and up.exitcode == 0 and lo_launches > 0
    merged = ftk.make_tracker(dims, field=field)
    merged.import_points(np.frombuffer(lo_pts, dtype=_lib.POINT_DTYPE))
    merged.import_points(np.frombuffer(up_pts, dtype=_lib.POINT_DTYPE))
    merged.finalize()
    P.assert_same_result(cuda_result(merged), want, tol=0.0, what="peer-memory halo")
    for t in (whole, merged):
        t.close()


# ---- sync-free (deferred) steps: results never depend on the mode -------------------------------------------------
def _woven_series(oracle, dims, T):
    return list(oracle.synthetic_series("woven", dims, T, None))


@pytest.mark.parametrize("mode", ["deferred", "sync"])
def test_deferred_steps_equal_synchronous_steps(mode, ftk, oracle, monkeypatch):
    """FTKB_DEFER=0 confirms every step before returning; the default enqueues step k+1 before reading step k"""
    monkeypatch.setenv("FTKB_DEFER", "0" if mode == "sync" else "1")
    dims, T = [96, 80], 7
    snaps = _woven_series(oracle, dims, T)
    want = P.oracle_result(oracle.track(snaps, dims, field="scalar"))
    tr = ftk.track(snaps, dims, field="scalar")
    P.assert_same_result(cuda_result(tr), want, tol=TOL, what=f"woven {mode}")
    st = tr.stats()
    assert st["scan_launches"] >= T and st["simplices_tested"] == (93 * 77) * (12 * (T - 1) + 2)
    tr.close()


@pytest.mark.parametrize("what", ["points", "worklist"])
def test_deferred_step_overflow_is_replayed(what, ftk, oracle, monkeypatch):
    """a step whose output buffers overflow while the next one is already enqueued: both are discarded and redone"""
    if what == "worklist":
        monkeypatch.setenv("FTKB_WL_CAP", "5")
    dims, T = [96, 80], 6
    snaps = _woven_series(oracle, dims, T)
    want = P.oracle_result(oracle.track(snaps, dims, field="scalar"))
    tr = ftk.track(snaps, dims, field="scalar", point_capacity=7 if what == "points" else 0)
    P.assert_same_result(cuda_result(tr), want, tol=TOL, what=f"overflow {what}")
    assert tr.stats()["sweeps_repeated"] > 0
    tr.close()


@pytest.mark.parametrize("dims,T,min_points", [([448, 384], 4, 1 << 20), ([60, 52, 48], 3, 800000)])
def test_feature_dense_field_deferred(dims, T, min_points, ftk, oracle):
    """white noise: nearly every cube survives the scan (1.7e5 per step) and a third of a million simplices per step are punctured --
    the paths only a dense field takes: survivors staged per warp and flushed 64 at a time, the test kernel moving from the second
    stream to the sweep's once the worklist is a GPU's worth of work, the point buffer (2^20 records) growing ahead of the steps in
    flight, several passes of the cold path per block"""
    rng = np.random.default_rng(5)
    snaps = [rng.standard_normal(tuple(reversed(dims))) for _ in range(T)]
    want = P.oracle_result(oracle.track(snaps, dims, field="scalar"))
    tr = ftk.track(snaps, dims, field="scalar")
    got = cuda_result(tr)
    assert len(got["points"]) > min_points                      # (2D: the buffer of 2^20 records did have to grow)
    P.assert_same_result(got, want, tol=TOL, what=f"white noise {dims} x {T}")
    st = tr.stats()
    assert st["cells_refined"] > 100000 * (T - 1)
    tr.close()


def test_deferred_steps_3d_and_vector(ftk, oracle):
    rng = np.random.default_rng(77)
    for dims, T, field in (([34, 20, 12], 5, "scalar"), ([40, 36], 6, "vector"), ([18, 16, 10], 4, "vector")):
        nv = 1 if field == "scalar" else len(dims)
        snaps = _rand_series(rng, dims, T, nv, "smooth")
        c, o = _both(ftk, oracle, snaps, dims, field)
        P.assert_same_result(cuda_result(c), P.oracle_result(o), tol=TOL, what=f"deferred {dims} {field}")
        assert c.stats()["scaling_factor"] == o.scaling_factor
        c.close()


# ---- SURVEY.md 8(c) sizes: the reduced extents of the benchmark generators, compared with the oracle -------------
def _ref_series(oracle, gen, dims, T, params=None):
    return list(oracle.synthetic_series(gen, dims, T, params))


@pytest.mark.parametrize("gen,dims,T,field,params", [
    ("woven", [512, 512], 16, "scalar", None),
    ("double_gyre", [512, 256], 16, "vector", None),
    ("moving_extremum", [96, 96, 96], 6, "scalar", [48.3, 47.7, 48.1, 0.1, 0.11, 0.1]),
    ("abc", [96, 96, 96], 6, "vector", None),                      # unsteady ABC: A(k) as in the C4 benchmark
])
def test_survey_8c_sizes_match_oracle(gen, dims, T, field, params, ftk, oracle):
    snaps = _ref_series(oracle, gen, dims, T, params)
    c, o = _both(ftk, oracle, snaps, dims, field)
    got, want = cuda_result(c), P.oracle_result(o)
    assert len(want["points"]) > 0
    P.assert_same_result(got, want, tol=TOL, what=f"{gen} {dims}x{T}")
    assert np.array_equal(c.get_component_labels(), o.component_labels())
    assert c.stats()["scaling_factor"] == o.scaling_factor
    c.close()


def test_scalar_2d_nonfinite_and_huge_values(ftk, oracle):
    """NaN / Inf / 2^1010 scalars cannot be ordered by the high-word keys of the default 2D build kernel: the layer is
    poisoned and the step redone with the fp32-range kernel; results equal the oracle's either way"""
    rng = np.random.default_rng(5)
    dims, T = [140, 90], 4
    snaps = [rng.standard_normal((90, 140)) for _ in range(T)]
    snaps[1][40, 70] = np.nan
    snaps[2][10:12, 100] = np.inf
    snaps[2][60, 20] = -2.0 ** 1010
    c, o = _both(ftk, oracle, snaps, dims, "scalar")
    P.assert_same_result(cuda_result(c), P.oracle_result(o), tol=TOL, what="non-finite 2D scalar")
    assert c.stats()["sweeps_repeated"] > 0
    c.close()


# ---- device-side generators (SURVEY.md 8f1): values against the reference's closed forms, and the tracker on exactly the
# field the device produced against the oracle on that same field --------------------------------------------------------
GENERATORS = [
    # kind, name, dims, field, params handed to ftkb_push_synthetic, time of snapshot k, host twin
    (0, "moving_extremum_2d", [64, 48], "scalar", [30.3, 21.7, 0.4, 0.3], lambda k, T: float(k)),
    (0, "moving_extremum_3d", [24, 20, 18], "scalar", [11.3, 9.7, 8.1, 0.3, 0.21, 0.1], lambda k, T: float(k)),
    (1, "woven", [96, 72], "scalar", [], lambda k, T: float(k) / (T - 1) + 1e-4),
    (2, "double_gyre", [96, 48], "vector", [0.1, 2 * np.pi, 0.25], lambda k, T: 0.1 * k),
    (3, "abc", [24, 22, 20], "vector", None, lambda k, T: 0.0),
    (4, "merger", [48, 40], "scalar", [], lambda k, T: 0.1 * k),
    (5, "tornado", [20, 18, 16], "vector", [], lambda k, T: float(k)),
]


def _host_twin(oracle, name, dims, params, t, k):
    if name.startswith("moving_extremum"):
        nd = len(dims)
        return oracle.gen_moving_extremum(dims, params[:nd], params[nd:], t)
    if name == "woven":
        return oracle.gen_woven(dims[0], dims[1], t)
    if name == "double_gyre":
        return oracle.gen_double_gyre(dims[0], dims[1], t, *params)
    if name == "abc":
        return oracle.gen_abc(dims[0], dims[1], dims[2], oracle.abc_amplitude(k))
    if name == "merger":
        return oracle.gen_merger(dims[0], dims[1], t)
    return oracle.gen_tornado(dims[0], dims[1], dims[2], int(t))


@pytest.mark.parametrize("case", range(len(GENERATORS)), ids=[g[1] for g in GENERATORS])
def test_device_generators(case, ftk, oracle):
    kind, name, dims, field, params, time_of = GENERATORS[case]
    T = 5
    tr = ftk.make_tracker(dims, field=field)
    device_fields = []
    for k in range(T):
        t = time_of(k, T)
        prm = [oracle.abc_amplitude(k), np.sqrt(2.0), 1.0] if name == "abc" else params
        tr.push_synthetic_snapshot(kind, prm, t)
        s, v = tr.get_layer(1 if k else 0)
        dev = s if field == "scalar" else v
        host = _host_twin(oracle, name, dims, prm, t, k)
        # the closed forms of include/ftk/ndarray/synthetic.hh: exact where they are pure arithmetic, within a few ulp of the
        # value scale where sin / cos / exp / sqrt of the device's libm round differently from the host's
        scale = max(1.0, float(np.abs(host).max()))
        if name.startswith("moving_extremum"):
            assert np.array_equal(dev, host), f"{name}: device generator differs from synthetic.hh"
        else:
            assert np.abs(dev - host).max() <= 64 * np.finfo(np.float64).eps * scale, f"{name}: max |d| = {np.abs(dev - host).max()}"
        device_fields.append(dev.copy())
        if k:
            tr.advance_timestep()
        if k == T - 1:
            tr.update_timestep()
    tr.finalize()
    o = oracle.track(device_fields, dims, field=field)           # the oracle on exactly what the device generated
    P.assert_same_result(cuda_result(tr), P.oracle_result(o), tol=TOL, what=f"generator {name}")
    tr.close()


@pytest.mark.parametrize("dims,field", [([19, 13], "scalar"), ([17, 11], "vector"), ([11, 9, 7], "scalar")])
def test_float32_snapshots_are_widened_on_the_device(dims, field, ftk, oracle):
    """float32 host arrays travel as float32 (ftkb_push_snapshot_f32) and are widened on the device: same result as widening
    on the host first, sizes that are not a multiple of four elements included"""
    rng = np.random.default_rng(77)
    nv = 1 if field == "scalar" else len(dims)
    snaps32 = [s.astype(np.float32) for s in _rand_series(rng, dims, 4, nv, "smooth")]
    o = oracle.track([s.astype(np.float64) for s in snaps32], dims, field=field)
    c = ftk.track(snaps32, dims, field=field)
    assert c.stats()["h2d_bytes"] == sum(s.nbytes for s in snaps32)
    P.assert_same_result(cuda_result(c), P.oracle_result(o), tol=TOL, what=f"float32 {field} {dims}")
    c.close()

"""The scan's cube exclusion at its edges: quantisation threshold, determinant guards, int64 conversion overflow, the
2^1000 poison bound and the placement of the minimum non-zero |v| that sets the quantisation factor.

Every scan kernel excludes whole space-time cubes before the exact per-simplex test.  That is only correct while the
exclusion is conservative: it may drop a cube only if the reference's predicate, evaluated on trunc(v * 2^nbits) in
(wrapping) int64 arithmetic, punctures none of its simplices.  The fields here are built so that many cubes hang on
one value within 2^-20 of the threshold, on a magnitude next to a guard bound, or on where the minimum sits, and every
scan path that can take a field runs it:

  * against the parity oracle (points, types, trajectories, component labels, factor, resolution), and
  * against a numpy restatement of the strict-sign rule: every cube that rule cannot exclude is in the worklist.

The CPU tests at the end check that each generator still reaches the regime it is meant for.
"""
import math

import numpy as np
import pytest

import _parity as P

TOL = 1e-9
U = 2.0 ** -21                  # one quantum at nbits = 21
I64_MIN = np.iinfo(np.int64).min


# ---- numpy restatement of the reference's quantisation (cp_oracle.c: gradient2D / gradient3D, resolution, factor) --------
def gradient(S):
    """gradient2D (clamped differences scaled by W-1, H-1) / gradient3D (halved differences, zero border) of a scalar
    snapshot in memory order -> (..., nd)"""
    if S.ndim == 2:
        H, W = S.shape
        ip, im = np.minimum(np.arange(W) + 1, W - 1), np.maximum(np.arange(W) - 1, 0)
        jp, jm = np.minimum(np.arange(H) + 1, H - 1), np.maximum(np.arange(H) - 1, 0)
        gx = (S[:, ip] - S[:, im]) * float(W - 1)
        gy = (S[jp, :] - S[jm, :]) * float(H - 1)
        return np.stack([gx, gy], -1)
    g = np.zeros(S.shape + (3,))
    c = (slice(1, -1),) * 3
    g[c + (0,)] = 0.5 * (S[1:-1, 1:-1, 2:] - S[1:-1, 1:-1, :-2])
    g[c + (1,)] = 0.5 * (S[1:-1, 2:, 1:-1] - S[1:-1, :-2, 1:-1])
    g[c + (2,)] = 0.5 * (S[2:, 1:-1, 1:-1] - S[:-2, 1:-1, 1:-1])
    return g


def vectors(snap, field):
    return gradient(snap) if field == "scalar" else snap


def resolution(vs):
    r = np.inf
    for v in vs:
        a = np.abs(v[v != 0])
        if a.size:
            r = min(r, float(a.min()))
    return r


def nbits_of(res):
    inv = 1.0 / res if res >= 2.0 ** -1023 else math.inf
    return min(max(int(math.ceil(math.log2(inv))), 8), 21) if inv < math.inf else 8   # (int)ceil(inf) is INT_MIN on x86-64


def quantise(v, nbits):
    """(int64)(v * 2^nbits) as x86-64 converts it: out of range and NaN give INT64_MIN"""
    p = v * float(1 << nbits)
    out = np.full(p.shape, I64_MIN, np.int64)
    ok = np.abs(p) < 2.0 ** 63
    out[ok] = np.trunc(p[ok]).astype(np.int64)
    return out


def excludable(layers_q, dims, field):
    """strict-sign rule per cube of the domain (corner c spans vertices c .. min(c+1, ub) in each dimension, over every
    layer given): some component >= 1 at all of them or <= -1 at all of them.  -> bool array (z,)y,x over corners"""
    lo = 2 if field == "scalar" else 1
    box = tuple(slice(lo, d - 1) for d in reversed(dims))
    pos = np.logical_and.reduce([q[box] >= 1 for q in layers_q])
    neg = np.logical_and.reduce([q[box] <= -1 for q in layers_q])
    for ax in range(len(dims)):
        def up(a):
            return np.concatenate([np.take(a, np.arange(1, a.shape[ax]), axis=ax), np.take(a, [-1], axis=ax)], axis=ax)
        pos, neg = pos & up(pos), neg & up(neg)
    return (pos | neg).any(-1)


# ---- field families ---------------------------------------------------------------------------------------------------
def _grids(dims):
    return np.meshgrid(*[np.arange(d, dtype=np.float64) for d in reversed(dims)], indexing="ij")


def _smooth(dims, k, c, f=0.21):
    out = 0.0
    for q, g in enumerate(_grids(dims)):
        out = out + np.cos((f + 0.05 * c + 0.03 * q) * g + 0.9 * q + 0.37 * k + 1.3 * c) * (1.0 + 0.2 * q)
    return out


OFFS_UP = np.array([0.0, 2.0 ** -52, 2.0 ** -24, 2.0 ** -21, 2.0 ** -5])
OFFS_ALL = np.concatenate([OFFS_UP, -OFFS_UP[1:]])


def lattice_vector(dims, T, seed):
    """v directly on the quantum lattice at nbits = 21: coherent sign regions of +-1, +-2 quanta, each offset by 0, +-1 ulp,
    +-2^-24, +-2^-21 or +-2^-5 relative; in 'edgy' regions also a band in (0.5, 1) quanta, exact zeros and -0.0.
    One value of 2^-40 pins the factor at 2^21."""
    rng = np.random.default_rng(seed)
    shape, nv = tuple(reversed(dims)), len(dims)
    out = []
    for k in range(T):
        edgy = _smooth(dims, k, 7, 0.13) > 0.6
        comps = []
        for c in range(nv):
            f = _smooth(dims, k, c)
            mag = np.where(np.abs(f) > 1.4, 2.0, 1.0)
            r = np.where(edgy, rng.choice(OFFS_ALL, size=shape), rng.choice(OFFS_UP, size=shape))
            v = np.where(f < 0, -1.0, 1.0) * mag * U * (1.0 + r)
            u = rng.random(shape)
            band = edgy & (u < 0.15)
            v[band] = np.sign(f[band]) * U * rng.uniform(0.5, 1.0, int(band.sum()))
            zero = edgy & (u >= 0.15) & (u < 0.25)
            v[zero] = np.where(rng.random(int(zero.sum())) < 0.5, 0.0, -0.0)
            comps.append(v)
        out.append(np.stack(comps, -1))
    out[0][tuple(s // 2 for s in shape) + (0,)] = 2.0 ** -40
    return out


def _ramp(n, rng, k):
    """cumulative sum of piecewise-constant slopes: +-1, +-0.5 (differences over two steps of 1 or 2 quanta), +-2, and
    +-0.375 / +-0.25 (a difference of 0.75 / 0.5 quanta: quantised to 0)"""
    mags = np.array([1.0, 1.0, 0.5, 0.5, 1.0, 2.0, 0.375, 0.25])
    s, sign, i = np.empty(n), 1.0, 0
    while i < n:
        ln = int(rng.integers(5, 13))
        if rng.random() < 0.45:
            sign = -sign
        s[i:i + ln] = sign * mags[rng.integers(len(mags))]
        i += ln
    return np.roll(np.cumsum(s), 3 * k)


def lattice_scalar(dims, T, seed):
    """scalars whose derived gradient lands on the nbits = 21 lattice.  3D: S = 2^-20 Z, Z in halves (v = d / 2); 2D: y differences
    scaled by H - 1 = 2^7 exactly, x differences RN(2^-21 / (W - 1)) per slope unit, so d * (W - 1) rounds to either
    side of the threshold.  A few ulp-sized nudges of S, and one interior difference of 2^-38 (pins nbits at 21)."""
    rng = np.random.default_rng(seed)
    shape = tuple(reversed(dims))
    out = []
    for k in range(T):
        if len(dims) == 3:
            D, H, W = shape
            Z = (_ramp(W, rng, k)[None, None, :] + _ramp(H, rng, k)[None, :, None] + _ramp(D, rng, k)[:, None, None] +
                 0.5 * np.round(2.0 * _smooth(dims, k, 3, 0.11)))     # (separable ramps alone leave no critical point)
            S = 2.0 ** -20 * Z
        else:
            H, W = shape
            assert H - 1 == 128
            S = 2.0 ** -28 * _ramp(H, rng, k)[:, None] + float(np.float64(U) / (W - 1)) * _ramp(W, rng, k)[None, :]
        nudge = (rng.random(shape) < 0.3) & (np.abs(S) >= 2.0 ** -30)     # (a nudge of 0 would be a denormal difference)
        S[nudge] = S[nudge] + rng.integers(-2, 3, int(nudge.sum())) * np.spacing(S[nudge])
        c = tuple(s // 2 for s in shape)
        lo = c[:-1] + (c[-1] - 1,)
        hi = c[:-1] + (c[-1] + 1,)
        S[hi] = S[lo] + 2.0 ** -38
        out.append(S)
    return out


def ladder(dims, field, T, e, kind, seed):
    """integer-valued smooth-plus-noise ('int') or smooth fields, times 2^e; scalar kinds 'offset40' (2^40 + small field:
    differences that round) and 'offset999' (2^999 + 2^960 * integer field)"""
    rng = np.random.default_rng(seed)
    nv = 1 if field == "scalar" else len(dims)
    out = []
    for k in range(T):
        comps = []
        for c in range(nv):
            f = _smooth(dims, k, c)
            if kind == "smooth":
                comps.append(np.ldexp(f, e))
            elif kind == "offset40":
                comps.append(2.0 ** 40 + f)
            elif kind == "offset999":
                comps.append(2.0 ** 999 + 2.0 ** 960 * np.round(2.5 * f + 0.8 * rng.standard_normal(f.shape)))
            else:
                comps.append(np.ldexp(np.round(2.5 * f + 0.8 * rng.standard_normal(f.shape)), e))
        out.append(np.stack(comps, -1) if nv > 1 else comps[0])
    return out


def poison(dims, T, scale, seed):
    """scalars whose magnitude peaks at `scale` (just under / just over 2^1000)"""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(T):
        n = np.round(2.5 * _smooth(dims, k, 0) + 0.8 * rng.standard_normal(tuple(reversed(dims))))
        out.append(n / np.abs(n).max() * scale)
    return out


B_RES = 2.0 ** -10.5            # background minimum: nbits = 11
PLACED = 2.0 ** -13.3           # placed minimum: nbits = 14 (or more: see place_scalar)
TIE = (1.5 + 2.0 ** -40) * 2.0 ** -11    # a minimum whose low word is not zero: its predecessor has the same high word


def place_vector(dims, T, where, layer, seed, tie=False):
    """background min non-zero |v| = B_RES (or TIE), one component of one vertex set to PLACED (or the double just below
    TIE) in snapshot `layer`"""
    rng = np.random.default_rng(seed)
    floor = TIE if tie else B_RES
    out = []
    for k in range(T):
        comps = []
        for c in range(len(dims)):
            f = _smooth(dims, k, c) + 0.05 * rng.standard_normal(tuple(reversed(dims)))
            v = np.where(f < 0, -1.0, 1.0) * np.maximum(np.abs(f), floor)
            v[rng.random(v.shape) < 0.02] = 0.0
            comps.append(v)
        out.append(np.stack(comps, -1))
    out[layer][tuple(reversed(where)) + (1,)] = -np.nextafter(TIE, 0.0) if tie else -PLACED
    return out


def place_scalar(dims, T, where, layer, seed, tie=False):
    """S = K q on an integer field q, so that min non-zero |v| = K * (smallest gradient scale) = B_RES (or TIE).  At vertex
    `where` the difference along the axis with the smallest scale (y in 2D) is made tiny in snapshot `layer`: its two
    stencil vertices get equal q, then one is moved by delta (tie: 0 and the double just below K).  The new minimum
    sits at `where` and possibly at vertices within two of it."""
    rng = np.random.default_rng(seed)
    nd = len(dims)
    scale = 0.5 if nd == 3 else float(min(dims) - 1)
    ax = 1 if nd == 2 else 0                       # x-major index of the axis
    K = (TIE if tie else B_RES) / scale
    out = []
    for k in range(T):
        # (a wide range of integers: few exactly singular Hessians, whose 3D types libm decides -- see assert_same)
        q = np.round(24.0 * _smooth(dims, k, 0) + 3.0 * rng.standard_normal(tuple(reversed(dims))))
        if k == layer:
            g = list(where)
            lo, hi = list(g), list(g)
            lo[ax], hi[ax] = max(g[ax] - 1, 0), min(g[ax] + 1, dims[ax] - 1)
            L, Hh = tuple(reversed(lo)), tuple(reversed(hi))
            if tie:
                q[L] = 0.0
                q[Hh] = 1.0
                for b in range(nd):                 # the other stencils through `hi` must not produce a smaller difference
                    for s in (-2, 2):
                        o = list(hi)
                        o[b] += s
                        if 0 <= o[b] < dims[b] and o != lo:
                            q[tuple(reversed(o))] = 0.0
            else:
                q[Hh] = q[L]
        S = K * q
        if k == layer:
            if tie:
                S[Hh] = np.nextafter(K, 0.0)
            else:
                S[Hh] += PLACED / scale
        out.append(S)
    return out


def filter_tie_scalar(dims, T, where, seed):
    """smooth scalars plus noise, so that no gradient component is exactly zero: the scalar build kernels' key filter
    (res_threshold_key, two key units above the running minimum) then decides alone which stages need the exact minimum.
    Snapshot 0 holds the minimum m at vertex `where` (0.7 of the field's own minimum: low word not zero), the last
    snapshot holds the double just below m at the vertex mirrored through the array's centre.  Both are made exactly along
    the axis whose scale is a power of two (y in 2D: H - 1; 3D: 1/2): S = 0 on one stencil vertex, value / scale on the other."""
    rng = np.random.default_rng(seed)
    nd = len(dims)
    shape = tuple(reversed(dims))
    scale = 0.5 if nd == 3 else float(dims[1] - 1)
    ax = 1 if nd == 2 else 0
    out = [_smooth(dims, k, 0) + 1e-3 * rng.standard_normal(shape) for k in range(T)]
    m = 0.7 * resolution([gradient(S) for S in out])

    def put(S, w, val):
        lo, hi = list(w), list(w)
        lo[ax], hi[ax] = w[ax] - 1, w[ax] + 1
        S[tuple(reversed(lo))] = 0.0
        S[tuple(reversed(hi))] = val / scale
    put(out[0], where, m)
    put(out[-1], [d - 1 - x for d, x in zip(dims, where)], np.nextafter(m, 0.0))
    return out


# ---- the field catalogue: name -> (dims, field, T, generator) ---------------------------------------------------------
S2, S2_ODD, V2 = [500, 129], [129, 65], [130, 70]
S3, S3_ODD, V3 = [66, 36, 32], [65, 35, 20], [66, 36, 20]

FIELDS = {}
FAMILY = {}


def _add(name, family, dims, field, T, gen):
    FIELDS[name] = (dims, field, T, gen)
    FAMILY[name] = family


for _dims, _f in ((S2, "scalar"), (S2_ODD, "scalar"), (V2, "vector"), (S3, "scalar"), (S3_ODD, "scalar"), (V3, "vector")):
    _tag = f"{len(_dims)}d{_f[0]}{'_odd' if _dims[0] % 2 else ''}"
    if _f == "vector":
        _add(f"lattice_{_tag}", "lattice", _dims, _f, 3, lambda d=_dims: lattice_vector(d, 3, 11))
    elif _dims[1] == 129 or len(_dims) == 3:
        _add(f"lattice_{_tag}", "lattice", _dims, _f, 3, lambda d=_dims: lattice_scalar(d, 3, 12))

# magnitude ladder: quantised |v| = |n| 2^(e + nbits) (vector), |dn| 2^(e + nbits) * (W-1 | H-1 | 1/2) (scalar)
LADDER = {
    "2dv": (V2, "vector", [-30, -22, 0, 12, 21, 22, 30, 54, 55, 56]),
    "3dv": (V3, "vector", [-30, -22, 0, 12, 20, 22, 30, 55, 56]),
    "2ds": (S2, "scalar", [-40, -28, 0, 13, 15, 24, 47, 48, 60]),
    "3ds": (S3, "scalar", [-40, -21, 0, 13, 22, 30, 56, 57]),
}
for _tag, (_dims, _f, _es) in LADDER.items():
    for _e in _es:
        _add(f"ladder_{_tag}_int_e{_e}", "ladder", _dims, _f, 3, lambda d=_dims, f=_f, e=_e: ladder(d, f, 3, e, "int", 100 + e))
    for _e in (-25, 0, 22, 55):
        _add(f"ladder_{_tag}_smooth_e{_e}", "ladder", _dims, _f, 3, lambda d=_dims, f=_f, e=_e: ladder(d, f, 3, e, "smooth", 0))
for _dims, _tag in ((S2, "2ds"), (S3, "3ds"), (S2_ODD, "2ds_odd")):
    _add(f"offset40_{_tag}", "ladder", _dims, "scalar", 3, lambda d=_dims: ladder(d, "scalar", 3, 0, "offset40", 5))
    _add(f"offset999_{_tag}", "ladder", _dims, "scalar", 3, lambda d=_dims: ladder(d, "scalar", 3, 0, "offset999", 6))
    _add(f"poison_below_{_tag}", "poison", _dims, "scalar", 3, lambda d=_dims: poison(d, 3, 2.0 ** 1000 * (1 - 2.0 ** -40), 7))
    _add(f"poison_above_{_tag}", "poison", _dims, "scalar", 3, lambda d=_dims: poison(d, 3, 2.0 ** 1000 * (1 + 2.0 ** -40), 7))
for _dims, _tag in ((V2, "2dv"), (V3, "3dv")):
    _add(f"poison_above_{_tag}", "poison", _dims, "vector", 3,
         lambda d=_dims: [v * 2.0 ** 1000 for v in ladder(d, "vector", 3, 0, "int", 8)])

# resolution placement: (dims, field, vertex (x-major), layer, tie)
T_PLACE = 5
PLACEMENTS = {
    "2ds": (S2, "scalar", {
        "first_row": ([250, 0], 0), "last_row": ([250, 128], 0), "first_col": ([0, 60], 0), "last_col": ([499, 60], 0),
        "chunk_edge": ([100, 19], 0), "block_edge": ([100, 27], 0), "cta_edge": ([434, 60], 0), "cta_edge_m1": ([433, 61], 0),
        "outside_domain": ([1, 1], 0), "layer1": ([300, 40], 1), "middle_layer": ([300, 40], 2), "layer0": ([300, 40], 0), "last_layer": ([300, 40], 4)}),
    "2ds_odd": (S2_ODD, "scalar", {"first_row": ([64, 0], 0), "last_col": ([128, 30], 0), "strip_edge": ([61, 30], 0),
                                   "middle_layer": ([40, 33], 2), "layer0": ([40, 33], 0)}),
    "2dv": (V2, "vector", {
        "first_row": ([60, 0], 0), "last_row": ([60, 69], 0), "first_col": ([0, 30], 0), "last_col": ([129, 30], 0),
        "strip_edge": ([62, 30], 0), "chunk_edge": ([40, 17], 0), "outside_domain": ([0, 0], 0), "layer1": ([70, 40], 1),
        "middle_layer": ([70, 40], 2), "layer0": ([70, 40], 0), "last_layer": ([70, 40], 4)}),
    "3ds": (S3, "scalar", {
        "near_border_x": ([1, 18, 16], 0), "near_border_xmax": ([64, 18, 16], 0), "near_border_z": ([30, 18, 1], 0),
        "tile_edge_x": ([62, 18, 16], 0), "tile_edge_y": ([30, 32, 16], 0), "zchunk_edge": ([30, 18, 16], 0),
        "zchunk_edge_p1": ([30, 18, 17], 0), "outside_domain": ([1, 1, 1], 0), "layer1": ([20, 10, 10], 1),
        "middle_layer": ([20, 10, 10], 2), "layer0": ([20, 10, 10], 0), "last_layer": ([20, 10, 10], 4)}),
    "3ds_odd": (S3_ODD, "scalar", {"near_border": ([63, 17, 10], 0), "middle_layer": ([20, 10, 10], 2), "layer0": ([20, 10, 10], 0)}),
    "3dv": (V3, "vector", {
        "border_x": ([0, 18, 10], 0), "border_zmax": ([30, 18, 19], 0), "tile_edge_x": ([62, 18, 10], 0),
        "tile_edge_y": ([30, 31, 10], 0), "outside_domain": ([0, 0, 0], 0), "layer1": ([20, 10, 10], 1),
        "middle_layer": ([20, 10, 10], 2), "layer0": ([20, 10, 10], 0), "last_layer": ([20, 10, 10], 4)}),
}
for _tag, (_dims, _f, _where) in PLACEMENTS.items():
    _gen = place_scalar if _f == "scalar" else place_vector
    for _name, (_w, _layer) in _where.items():
        _add(f"place_{_tag}_{_name}", "place", _dims, _f, T_PLACE, lambda d=_dims, w=_w, l=_layer, g=_gen: g(d, T_PLACE, w, l, 3))
    _w = [d // 3 for d in _dims]
    # (last layer: by then the running minimum is confirmed, so the scalar build kernels' key filter is armed with it)
    _add(f"place_{_tag}_tie", "tie", _dims, _f, T_PLACE, lambda d=_dims, w=_w, g=_gen: g(d, T_PLACE, w, T_PLACE - 1, 4, tie=True))

PLACED_AT = {f"place_{t}_{n}": (w, l) for t, (_, _, ws) in PLACEMENTS.items() for n, (w, l) in ws.items()}
PLACED_AT.update({f"place_{t}_tie": ([d // 3 for d in dims], T_PLACE - 1) for t, (dims, _, _) in PLACEMENTS.items()})
for _tag, (_dims, _f, _) in PLACEMENTS.items():
    if _f == "scalar":
        _w = [d // 3 for d in _dims]
        _add(f"place_{_tag}_filter_tie", "filter_tie", _dims, _f, T_PLACE, lambda d=_dims, w=_w: filter_tie_scalar(d, T_PLACE, w, 9))
        PLACED_AT[f"place_{_tag}_filter_tie"] = ([d - 1 - x for d, x in zip(_dims, _w)], T_PLACE - 1)

_SNAPS = {}


def snapshots(name):
    if name not in _SNAPS:
        _SNAPS[name] = FIELDS[name][3]()
    return _SNAPS[name]


# ---- scan paths ---------------------------------------------------------------------------------------------------------
# path -> (environment switch or None, borrowed at +8 bytes, robust, stats check)
PATHS = {
    "keys": (None, False, True, None),                          # 2D scalar, even W: scan2d_keys_build_kernel
    "f32": (("FTKB_SCAN2D", "f32"), False, True, None),         # 2D scalar: fp32-range build kernel
    "reg_borrow8": (None, True, True, None),                    # 2D scalar, rows off a 16-byte boundary: scan2d_fused_kernel
    "reg_odd": (None, False, True, None),                       # 2D scalar, odd W: scan2d_fused_kernel
    "vcells": (None, False, True, None),                        # vector input: vscan{2,3}d_build_kernel
    "twolayer": (("FTKB_VSCAN", "twolayer"), False, True, None),
    "nonrobust": (None, False, False, None),                    # 3D vector, robust detection off: every cube refined
    "fused": (None, False, True, "fused"),                      # 3D scalar, even W: scan3d_build_kernel
    "plain": (("FTKB_SCAN3D", "plain"), False, True, "derive"),  # 3D scalar: materialised gradient, scan3d_kernel
    "plain_borrow8": (None, True, True, "derive"),              # 3D scalar, no TMA descriptor for the layer
    "plain_odd": (None, False, True, "derive"),                 # 3D scalar, odd W
}


def paths_for(dims, field):
    nd, odd = len(dims), dims[0] % 2 == 1
    if field == "vector":
        return ["vcells", "twolayer"] + (["nonrobust"] if nd == 3 else [])
    if nd == 2:
        return ["reg_odd"] if odd else ["keys", "f32", "reg_borrow8"]
    return ["plain_odd"] if odd else ["fused", "plain", "plain_borrow8"]


MATRIX = [(n, p) for n in FIELDS for p in paths_for(FIELDS[n][0], FIELDS[n][1])]


# ---- GPU part -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ftk():
    import ftk_b200
    from ftk_b200 import _lib
    if _lib.lib().ftkb_device_count() < 1:
        pytest.fail("no sm_100 device visible: the CUDA path cannot run (there is no fallback)")
    return ftk_b200


_ORACLE = {}


def oracle_run(oracle, name, robust=True):
    key = (name, robust)
    if key not in _ORACLE:
        dims, field, T, _ = FIELDS[name]
        o = oracle.track(snapshots(name), dims, field=field, robust=robust)
        _ORACLE[key] = (P.oracle_result(o), o.component_labels(), o.scaling_factor, o.resolution)
    return _ORACLE[key]


class _Borrowed:
    """device copies of the snapshots, each starting 8 bytes past a 16-byte boundary, kept alive as long as the tracker"""
    def __init__(self):
        self.keep = []

    def ptr(self, a):
        import torch
        flat = torch.from_numpy(np.ascontiguousarray(a, np.float64).ravel())
        buf = torch.zeros(flat.numel() + 2, dtype=torch.float64, device="cuda")
        buf[1:1 + flat.numel()].copy_(flat)
        torch.cuda.synchronize()
        self.keep.append(buf)
        p = buf.data_ptr() + 8
        assert p % 16 == 8
        return p


def make(ftk, path, dims, field, monkeypatch, **kw):
    env, borrow, robust, _ = PATHS[path]
    if env:
        monkeypatch.setenv(*env)
    try:
        tr = ftk.make_tracker(dims, field=field, robust=robust, **kw)
    finally:
        if env:
            monkeypatch.delenv(env[0])
    tr._borrowed = _Borrowed() if borrow else None
    return tr


def push(tr, field, s):
    if tr._borrowed is not None:
        tr.push_device_pointers(**{field: tr._borrowed.ptr(s)})
    elif field == "scalar":
        tr.push_scalar_field_snapshot(s)
    else:
        tr.push_vector_field_snapshot(s)


def run(ftk, path, name, monkeypatch):
    dims, field, T, _ = FIELDS[name]
    tr = make(ftk, path, dims, field, monkeypatch)
    snaps = snapshots(name)
    for k, s in enumerate(snaps):
        push(tr, field, s)
        if k:
            tr.advance_timestep()
        if k == T - 1:
            tr.update_timestep()
    tr.finalize()
    return tr


def integer_valued(name):
    """scalar fields on a coarse grid of values (integer multiples of one step): their Hessians can be exactly singular"""
    return FAMILY[name] in ("lattice", "place", "tie", "poison") or "_int_" in name or "offset" in name


def small_integers(name):
    """3D lattices (half-integer ramps) and the integer ladder (|n| <= ~6): exactly singular Hessians are ten times as
    common there as on the wider-ranged placement fields (measured up to 2.0e-3 of the points, lattice_3ds)"""
    return FAMILY[name] == "lattice" or "_int_" in name


def assert_same(got, want, name, what):
    """_parity.assert_same_result.  On integer-valued 3D scalar fields, as in test_group.py, fewer than 1e-4 (3e-3 on small_integers) of the
    critical-point TYPES may differ (DESIGN.md §5: a Jacobian eigenvalue is exactly zero and the last bit of libm decides its
    sign); the punctured set, positions and ordered trajectories stay exact, and every other field is exact throughout"""
    dims, field = FIELDS[name][:2]
    g, w = got["points"], want["points"]
    if len(dims) == 3 and field == "scalar" and integer_valued(name) and len(g) == len(w) and len(w):
        d = g["cp_type"] != w["cp_type"]
        assert d.mean() < (3e-3 if small_integers(name) else 1e-4), f"{what}: {d.sum()} of {len(w)} critical-point types differ"
        g = g.copy()
        g["cp_type"] = w["cp_type"]
        got = dict(got, points=g)
    P.assert_same_result(got, want, tol=TOL, what=what)


def check_path_stats(path, st):
    what = PATHS[path][3]
    if what == "fused":
        assert st["ms_derive"] == 0.0, "the fused 3D scan never launches the gradient kernel"
    elif what == "derive":
        assert st["ms_derive"] > 0.0, "this input must take the materialised-gradient path"


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", MATRIX, ids=[f"{n}-{p}" for n, p in MATRIX])
def test_scan_path_matches_oracle(name, path, ftk, oracle, monkeypatch):
    """every field through every scan that can take it: points, types, ordered trajectories, component labels, factor and
    resolution equal the oracle's"""
    want, labels, factor, res = oracle_run(oracle, name, robust=PATHS[path][2])
    tr = run(ftk, path, name, monkeypatch)
    got = {"points": tr.get_discrete_critical_points(), "trajectories": tr.get_trajectory_index()}
    assert_same(got, want, name, f"{name} on {path}")
    assert np.array_equal(tr.get_component_labels(), labels)
    st = tr.stats()
    assert st["scaling_factor"] == factor and st["resolution"] == res, \
        f"{name} on {path}: factor {st['scaling_factor']} resolution {st['resolution']!r}, oracle {factor} {res!r}"
    fam = FAMILY[name]
    if fam != "poison":                # (a poisoned step is redone on the materialised gradient)
        check_path_stats(path, st)
    if fam == "poison" and name.startswith("poison_above") and path in ("keys", "fused", "vcells"):
        assert st["sweeps_repeated"] > 0, "values >= 2^1000 must poison the step and redo it"
    # (the two-layer, non-robust and materialised-gradient paths resolve a layer before they scan it: nothing to replay)
    # sweeps_repeated also counts poison fallbacks, buffer growth and the first step's own resolution: the same field with the
    # minimum placed in layer 0 instead must repeat fewer sweeps
    if fam == "place" and name.endswith("middle_layer") and path not in ("twolayer", "nonrobust", "plain", "plain_borrow8", "plain_odd"):
        t0 = run(ftk, path, name.replace("middle_layer", "layer0"), monkeypatch)
        n0 = t0.stats()["sweeps_repeated"]
        t0.close()
        assert st["sweeps_repeated"] > n0, "a minimum found in a later layer must replay the step with the new factor"
    tr.close()


def test_every_family_punctures_somewhere(oracle):
    """the oracle finds punctured simplices in (nearly) every field: a comparison of two empty sets checks nothing"""
    empty = [n for n in FIELDS if FAMILY[n] in ("lattice", "place", "tie", "filter_tie") and len(oracle_run(oracle, n)[0]["points"]) == 0]
    assert not empty, f"fields with no punctured simplex: {empty}"


# z-slabs over several contexts: the resolution of every slab (ghost planes included) merges into one factor
SLAB_CASES = [("place_3ds_zchunk_edge", [0, 0]), ("place_3ds_middle_layer", [0, 0, 0]), ("place_3ds_tie", [0, 0])]


@pytest.mark.gpu
@pytest.mark.parametrize("name,ids,z", [(n, i, z) for n, i in SLAB_CASES for z in (None, "cut", "ghost")])
def test_z_slabs_find_the_placed_minimum(name, ids, z, ftk, oracle):
    """the placed minimum through 2 / 3 z-slabs (repeated device ids), as placed, moved onto a cut plane (first plane of
    the second slab) and onto the plane just below it (a ghost plane of the second slab): points, trajectories, factor and
    resolution equal the one-device run's"""
    from ftk_b200.group import track_on_devices
    dims, field, T, _ = FIELDS[name]
    w, layer = PLACED_AT[name]
    if z is None:
        snaps = snapshots(name)
    else:
        cut = 2 + (dims[2] - 3) // len(ids)          # first plane of the second slab (group.cpp: glb + nplanes * s / n)
        w = [w[0], w[1], cut if z == "cut" else cut - 1]
        snaps = place_scalar(dims, T, w, layer, 3, tie=name.endswith("tie"))
    one = ftk.track(snaps, dims, field=field)
    o = oracle.track(snaps, dims, field=field)
    assert_same({"points": one.get_discrete_critical_points(), "trajectories": one.get_trajectory_index()},
                P.oracle_result(o), name, f"{name} one device")
    g, root = track_on_devices(snaps, dims, ids, field=field, chunk=0)
    P.assert_same_result({"points": root.get_discrete_critical_points(), "trajectories": root.get_trajectory_index()},
                         {"points": one.get_discrete_critical_points(), "trajectories": one.get_trajectory_index()},
                         tol=0.0, what=f"{name} z-slabs {ids} {z}")
    gs, st = g.stats(), one.stats()
    assert gs["scaling_factor"] == st["scaling_factor"] == o.scaling_factor and gs["resolution"] == st["resolution"] == o.resolution
    g.close()
    one.close()


# ---- the scan's decision against the strict-sign rule on exact quantised values ------------------------------------------
WL_CASES = [(n, p) for n, p in MATRIX if FAMILY[n] == "lattice" and p != "nonrobust"] + \
           [(n, p) for n, p in MATRIX if n in ("ladder_2dv_int_e55", "ladder_3dv_int_e55", "ladder_2ds_int_e60",
                                                 "ladder_3ds_int_e57", "ladder_3dv_int_e12", "ladder_2dv_int_e22")]


def _assert_worklist_covers(tr, layers, dims, field, nbits, what, min_excluded=0.0):
    qs = [quantise(vectors(s, field), nbits) for s in layers]
    ex = excludable(qs, dims, field)
    need = np.flatnonzero(~ex.ravel())
    wl = np.unique(tr.get_last_worklist().astype(np.int64))
    missing = np.setdiff1d(need, wl)
    if missing.size:
        nc = ex.shape[::-1]
        c = [(int(m % nc[0]), int(m // nc[0] % nc[1])) + ((int(m // (nc[0] * nc[1])),) if len(dims) == 3 else ()) for m in missing[:5]]
        raise AssertionError(f"{what}: {missing.size} cubes the strict-sign rule keeps are missing from the worklist, "
                             f"e.g. corners (domain-relative) {c}")
    assert wl.size <= ex.size and (wl < ex.size).all()
    assert 1.0 - wl.size / ex.size >= min_excluded, f"{what}: the scan excluded only {1 - wl.size / ex.size:.2%} of the cubes"
    return ex


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", WL_CASES, ids=[f"{n}-{p}" for n, p in WL_CASES])
def test_worklist_contains_every_cube_the_sign_rule_keeps(name, path, ftk, monkeypatch):
    """the interval sweep that builds the range cells, a repeated sweep from the cells alone and the final ordinal sweep:
    every cube whose exact quantised values are not all >= 1 / all <= -1 in some component is in the worklist.  On the
    lattice fields the scan must also exclude a good share of the cubes (the filter ran)"""
    dims, field, T, _ = FIELDS[name]
    s = snapshots(name)
    nbits = nbits_of(resolution([vectors(x, field) for x in s[:2]]))
    share = 0.15 if FAMILY[name] == "lattice" else 0.0
    tr = make(ftk, path, dims, field, monkeypatch)
    push(tr, field, s[0])
    push(tr, field, s[1])
    tr.update_timestep()
    assert tr.stats()["scaling_factor"] == float(1 << nbits)
    _assert_worklist_covers(tr, s[:2], dims, field, nbits, f"{name} {path} interval sweep", share)
    tr.update_timestep()
    _assert_worklist_covers(tr, s[:2], dims, field, nbits, f"{name} {path} repeated sweep", share)
    tr.advance_timestep()
    tr.update_timestep()
    _assert_worklist_covers(tr, s[1:2], dims, field, nbits, f"{name} {path} ordinal sweep", share)
    tr.close()


# ---- CPU: every family reaches the regime it is aimed at -------------------------------------------------------------------
def _near_threshold(name):
    """values within 2^-20 relative below / at-or-above one quantum, over all snapshots"""
    dims, field, T, _ = FIELDS[name]
    below = above = 0
    for s in snapshots(name):
        a = np.abs(vectors(s, field)) * 2.0 ** 21
        below += int(((a >= 1 - 2.0 ** -20) & (a < 1)).sum())
        above += int(((a >= 1) & (a <= 1 + 2.0 ** -20)).sum())
    return below, above


def _hanging_cubes(name):
    """cubes (first interval) the strict-sign rule excludes only thanks to a value in [1, 1 + 2^-20] quanta: read as just
    below the threshold, each of those values would make the cube a survivor"""
    dims, field, T, _ = FIELDS[name]
    vs = [vectors(s, field) for s in snapshots(name)[:2]]
    ex = excludable([quantise(v, 21) for v in vs], dims, field)
    lowered = [np.where((np.abs(v) * 2.0 ** 21 >= 1) & (np.abs(v) * 2.0 ** 21 <= 1 + 2.0 ** -20), 0.0, v) for v in vs]
    ex2 = excludable([quantise(v, 21) for v in lowered], dims, field)
    return int(ex.sum()), int((ex & ~ex2).sum())


LATTICE = [n for n in FIELDS if FAMILY[n] == "lattice"]


@pytest.mark.parametrize("name", LATTICE)
def test_lattice_sits_on_the_threshold(name):
    dims, field, T, _ = FIELDS[name]
    assert nbits_of(resolution([vectors(s, field) for s in snapshots(name)])) == 21
    below, above = _near_threshold(name)
    assert below >= 50 and above >= 200, (below, above)
    n_ex, hanging = _hanging_cubes(name)
    ncubes = int(np.prod([d - (3 if field == "scalar" else 2) for d in dims]))
    assert n_ex >= 0.15 * ncubes and hanging >= 50, (n_ex, hanging, ncubes)


def _guard_products(name):
    """per sign-excludable cube of the first interval: the 2D determinant bound Mx Ry + My Rx on exact quantised values
    (M = max |q| + 1, R = spread + 2); 3D: the largest pairwise bound"""
    dims, field, T, _ = FIELDS[name]
    vs = [vectors(s, field) for s in snapshots(name)[:2]]
    nb = nbits_of(resolution(vs))
    qs = [quantise(v, nb).astype(np.float64) for v in vs]
    lo = 2 if field == "scalar" else 1
    box = tuple(slice(lo, d - 1) for d in reversed(dims))
    mx = np.maximum.reduce([q[box] for q in qs])
    mn = np.minimum.reduce([q[box] for q in qs])
    for ax in range(len(dims)):
        def up(a, f):
            return f(a, np.concatenate([np.take(a, np.arange(1, a.shape[ax]), axis=ax), np.take(a, [-1], axis=ax)], axis=ax))
        mx, mn = up(mx, np.maximum), up(mn, np.minimum)
    M = np.maximum(np.abs(mx), np.abs(mn)) + 1
    R = mx - mn + 2
    nd = len(dims)
    prods = [M[..., a] * R[..., b] + M[..., b] * R[..., a] for a in range(nd) for b in range(a + 1, nd)]
    bound = np.maximum.reduce(prods)
    return bound[excludable([quantise(v, nb) for v in vs], dims, field)]


@pytest.mark.parametrize("name", ["ladder_2dv_int_e21", "ladder_2ds_int_e13", "ladder_3dv_int_e20", "ladder_3ds_int_e22"])
def test_ladder_straddles_the_guard(name):
    b = _guard_products(name)
    assert (b < 4.5e18).sum() >= 20 and (b >= 4.5e18).sum() >= 20, ((b < 4.5e18).sum(), (b >= 4.5e18).sum())


@pytest.mark.parametrize("name", ["ladder_2dv_int_e55", "ladder_3dv_int_e55", "ladder_2ds_int_e48", "ladder_3ds_int_e57",
                                  "offset999_2ds", "offset999_3ds"])
def test_ladder_overflows_int64(name):
    dims, field, T, _ = FIELDS[name]
    vs = [vectors(s, field) for s in snapshots(name)]
    p = np.abs(np.concatenate([v.ravel() for v in vs])) * float(1 << nbits_of(resolution(vs)))
    assert (p >= 2.0 ** 63).sum() >= 100 and (p < 2.0 ** 63).sum() >= 100
    if "ladder" in name and "3ds" not in name:
        assert ((p >= 2.0 ** 63) & (p < 2.0 ** 64)).sum() >= 100


def test_poison_fields_bracket_2_to_the_1000():
    for tag in ("2ds", "3ds", "2ds_odd"):
        assert np.abs(np.stack(snapshots(f"poison_below_{tag}"))).max() < 2.0 ** 1000
        assert np.abs(np.stack(snapshots(f"poison_above_{tag}"))).max() >= 2.0 ** 1000


@pytest.mark.parametrize("name", [n for n in FIELDS if FAMILY[n] in ("place", "tie", "filter_tie")])
def test_placed_minimum_is_the_global_one(name):
    """the placed value is the array's min non-zero |v| (within two vertices of where it was placed, in the snapshot it was
    placed in) and moves nbits from 11 to at least 14; the tie leaves nbits alone and lowers the resolution by one ulp"""
    dims, field, T, _ = FIELDS[name]
    w, layer = PLACED_AT[name]
    vs = [vectors(s, field) for s in snapshots(name)]
    others = resolution(vs[:layer] + vs[layer + 1:])
    r = resolution(vs)
    a = np.abs(vs[layer])
    at = np.argwhere((a == r).any(-1))
    assert len(at) and (np.abs(at[:, ::-1] - np.array(w)).max(1) <= 2).all(), (at[:4], w)
    if FAMILY[name] in ("tie", "filter_tie"):
        assert r == np.nextafter(others, 0.0) and nbits_of(r) == nbits_of(others)
        assert FAMILY[name] == "filter_tie" or nbits_of(r) == 11
        hi = lambda x: np.array([x]).view(np.uint64)[0] >> np.uint64(32)
        assert hi(r) == hi(others)
    else:
        assert nbits_of(others) == 11 and nbits_of(r) >= 14

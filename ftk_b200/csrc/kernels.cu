// Device code of the critical-point sweep, sm_100a.  Compile with -fmad=false: the reference's CPU
// path (x86-64, no FMA contraction) is the parity target, so every floating-point expression below
// keeps the reference's literal operation order and is never contracted; fma() appears only where
// the reference calls it.
//
// Kernels
//   scan2d / scan3d   streaming pass over the space-time cubes of one step: exact sign early-out
//                     (all vertices of the cube strictly on one side of zero in some component =>
//                     no simplex of the cube is punctured), survivors appended to a worklist.
//                     HBM-bound: each vertex of layers t and t+1 is read once.
//   test<ND>          the fused per-simplex test on the surviving cubes: ordinal->vertex decode,
//                     gather, fixed-point quantisation, simulation-of-simplicity predicates,
//                     inverse interpolation, lerp of position/time/scalar/Jacobian, type
//                     classification, warp-aggregated append.
//   gradient2d/3d, resolution, synthetic generators, element keys, neighbour search, union-find.
#include "kernels.h"

#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <string>
#include <climits>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

namespace ftkb {

typedef long long i64;
typedef unsigned long long u64;

__constant__ DeviceMeshTables c_mesh[2];   // [0]: 2D+t (12 triangle types), [1]: 3D+t (60 tetrahedron types)

void upload_mesh_tables(const DeviceMeshTables &t2, const DeviceMeshTables &t3) {
  DeviceMeshTables h[2] = {t2, t3};
  cudaMemcpyToSymbol(c_mesh, h, sizeof(h));
}

// =============================================================================================
// 1. scan: exact sign early-out on whole cubes
// =============================================================================================
//
// Only the high word of each fp64 component is inspected.  With factor = 2^nbits the scaled value
// p = v * factor has high word hi(v) + (nbits << 20) (exact for normal v), and the reference's
// quantised integer trunc(p) is >= 1 iff p >= 1.0 and <= -1 iff p <= -1.0.  An order-preserving
// 32-bit key k of p brackets it: p in [key_lo(k), key_hi(k)].  Per cube we keep min/max keys per
// component; "all vertices strictly positive" is  kmin >= key(1.0).
//
// The early-out claims "the reference's predicate returns false".  The reference evaluates its
// determinants in wrapping int64 arithmetic, which equals exact arithmetic only while the true
// determinant values fit; the magnitude guard below proves that from the cube's value range, and
// cubes that fail it are refined like any other survivor (they then go through the same wrapping
// arithmetic as the reference).
constexpr int KEY_ONE = 0x3FF00000;        // high word of 1.0
constexpr int KEY_POISON_EXP = 0x43E00000; // |p| >= 2^63 (also Inf / NaN after scaling)

__device__ __forceinline__ int clampi(int i, int n) { return i < 0 ? 0 : (i > n - 1 ? n - 1 : i); }

struct KeyRange { int mn, mx; };

__device__ __forceinline__ KeyRange neutral_range() { return KeyRange{INT_MAX, INT_MIN}; }

__device__ __forceinline__ KeyRange vertex_range(int hi, int nbits20) {
  const int m = hi & 0x7fffffff;
  const int ms = (m >> 20) ? m + nbits20 : 0;      // zero / denormal: |p| < 2^-1000
  const int k = hi < 0 ? -1 - ms : ms;
  const bool bad = ms >= KEY_POISON_EXP;
  return KeyRange{bad ? INT_MIN : k, bad ? INT_MAX : k};
}

__device__ __forceinline__ KeyRange merge(KeyRange a, KeyRange b) { return KeyRange{min(a.mn, b.mn), max(a.mx, b.mx)}; }

__device__ __forceinline__ KeyRange shfl_down1(KeyRange a) {
  return KeyRange{__shfl_down_sync(0xffffffffu, a.mn, 1), __shfl_down_sync(0xffffffffu, a.mx, 1)};
}

__device__ __forceinline__ double key_lo(int k) { return k >= 0 ? __hiloint2double(k, 0) : -__hiloint2double(-k, 0); }
__device__ __forceinline__ double key_hi(int k) { return k >= 0 ? __hiloint2double(k + 1, 0) : -__hiloint2double(-1 - k, 0); }

__device__ __forceinline__ bool one_sided(KeyRange r) { return r.mn >= KEY_ONE || r.mx <= -1 - KEY_ONE; }

// bound on |quantised value| and on the spread of quantised values over the cube (+ truncation slack)
__device__ __forceinline__ void magnitude_range(KeyRange r, double &M, double &R) {
  const double lo = key_lo(r.mn), hi = key_hi(r.mx);
  M = fmax(fabs(lo), fabs(hi)) + 1.0;
  R = (hi - lo) + 2.0;
}

// true: no simplex with vertices in this cube can be punctured, and the reference agrees
__device__ __forceinline__ bool cube_excluded2(KeyRange x, KeyRange y) {
  if (!(one_sided(x) || one_sided(y))) return false;
  if (x.mn == INT_MIN || y.mn == INT_MIN) return false;
  double Mx, Rx, My, Ry;
  magnitude_range(x, Mx, Rx);
  magnitude_range(y, My, Ry);
  // every determinant of the 2D cascade is bounded by 2 (Mx Ry + My Rx); require < 2^63 with slack
  return Mx * Ry + My * Rx < 4.5e18;
}

__device__ __forceinline__ bool cube_excluded3(KeyRange x, KeyRange y, KeyRange z) {
  if (!(one_sided(x) || one_sided(y) || one_sided(z))) return false;
  if (x.mn == INT_MIN || y.mn == INT_MIN || z.mn == INT_MIN) return false;
  double Mx, Rx, My, Ry, Mz, Rz;
  magnitude_range(x, Mx, Rx);
  magnitude_range(y, My, Ry);
  magnitude_range(z, Mz, Rz);
  // 4x4 level: <= 4 (Mx Ry Rz + My Rx Rz + Mz Rx Ry); 3x3 sub-levels: <= 2 (Ma Rb + Mb Ra)
  const bool d4 = 4.0 * (Mx * Ry * Rz + My * Rx * Rz + Mz * Rx * Ry) < 9.0e18;
  const bool d3 = (Mx * Ry + My * Rx < 4.5e18) && (Mx * Rz + Mz * Rx < 4.5e18) && (My * Rz + Mz * Ry < 4.5e18);
  return d4 && d3;
}

__device__ __forceinline__ void append_survivors(const SweepParams &p, bool surv, u64 lin) {
  const unsigned b = __ballot_sync(0xffffffffu, surv);
  if (b == 0) return;
  const int lane = threadIdx.x & 31;
  u64 base = 0;
  if (lane == __ffs(b) - 1) base = atomicAdd(p.wl_count, (u64)__popc(b));
  base = __shfl_sync(0xffffffffu, base, __ffs(b) - 1);
  if (surv) {
    const u64 i = base + __popc(b & ((1u << lane) - 1));
    if (i < p.wl_cap) p.wl[i] = lin;
  }
}

// Survivors staged per warp in shared memory and appended WL_STAGE_CAP at a time: on feature-dense fields (1e6 surviving cubes per
// step) one atomicAdd per pass of the cold path -- all on the same counter -- is what the scan waits for.
// stage (shared-memory address, 8-byte aligned): u32 count, pad, then WL_STAGE_CAP u64 entries; one per warp.
constexpr int WL_STAGE_CAP = 64;
constexpr uint32_t WL_STAGE_BYTES = 16u + 8u * WL_STAGE_CAP;     // (a multiple of 16: what follows the stagings is 16-byte aligned)
__device__ __forceinline__ void flush_survivors(const SweepParams &p, const uint32_t stage) {
  const int lane = threadIdx.x & 31;
  int cnt;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(cnt) : "r"(stage) : "memory");
  if (cnt == 0) return;                                         // (warp-uniform)
  u64 base = 0;
  if (lane == 0) base = atomicAdd(p.wl_count, (u64)cnt);
  base = __shfl_sync(0xffffffffu, base, 0);
  for (int i = lane; i < cnt; i += 32) {
    u64 lin;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(lin) : "r"(stage + 8u + 8u * (uint32_t)i) : "memory");
    if (base + (u64)i < p.wl_cap) p.wl[base + (u64)i] = lin;
  }
  __syncwarp();
  if (lane == 0) asm volatile("st.shared.s32 [%0], %1;" ::"r"(stage), "r"(0) : "memory");
  __syncwarp();
}
__device__ __forceinline__ void stage_survivors(const SweepParams &p, const uint32_t stage, const bool surv, const u64 lin) {
  const unsigned b = __ballot_sync(0xffffffffu, surv);
  if (b == 0) return;
  const int lane = threadIdx.x & 31, n = __popc(b);
  int cnt;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(cnt) : "r"(stage) : "memory");
  if (cnt + n > WL_STAGE_CAP) { flush_survivors(p, stage); cnt = 0; }
  if (surv) asm volatile("st.shared.u64 [%0], %1;" ::"r"(stage + 8u + 8u * (uint32_t)(cnt + __popc(b & ((1u << lane) - 1)))), "l"(lin) : "memory");
  __syncwarp();
  if (lane == 0) asm volatile("st.shared.s32 [%0], %1;" ::"r"(stage), "r"(cnt + n) : "memory");
  __syncwarp();
}

// ---- 2D: one warp owns a strip of 32 vertex columns (31 corners) and marches along y -------------
template <bool HAS_NEXT>
__global__ void __launch_bounds__(256) scan2d_kernel(const SweepParams p) {
  const int lane = threadIdx.x & 31;
  const i64 warp = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int sx = (int)(warp % p.nsx), cy = (int)(warp / p.nsx);
  if (cy >= p.nsy) return;
  const int x = p.lb[0] + sx * 31 + lane;
  const bool col_ok = x <= p.vmax[0];
  const bool corner_col = lane < 31 && x <= p.ub[0];
  const int ys = p.lb[1] + cy * p.rows;
  const int ye = min(ys + p.rows - 1, p.ub[1]);
  const int nbits20 = p.nbits << 20;
  const int4 *__restrict__ V0 = reinterpret_cast<const int4 *>(p.L[0].V);
  const int4 *__restrict__ V1 = reinterpret_cast<const int4 *>(p.L[1].V);
  // a borrowed layer may be 8-byte aligned only: such a launch reads the two high words with 4-byte loads
  const bool al16 = (((uintptr_t)p.L[0].V | (uintptr_t)p.L[1].V) & 15) == 0;
  auto load_hi = [&](const int4 *V, const size_t i) -> int2 {
    if (al16) { const int4 a = __ldg(V + i); return make_int2(a.y, a.w); }
    const int *q = reinterpret_cast<const int *>(V) + 4 * i;
    return make_int2(__ldg(q + 1), __ldg(q + 3));
  };

  KeyRange px = neutral_range(), py = neutral_range();   // previous row, already merged over t and x..x+1
#pragma unroll 2
  for (int y = ys; y <= ye + 1; y++) {
    KeyRange rx = neutral_range(), ry = neutral_range();
    if (col_ok && y <= p.vmax[1]) {
      const size_t i = (size_t)x + (size_t)p.W * (size_t)y;
      const int2 a = load_hi(V0, i);
      rx = vertex_range(a.x, nbits20);
      ry = vertex_range(a.y, nbits20);
      if (HAS_NEXT) {
        const int2 b = load_hi(V1, i);
        rx = merge(rx, vertex_range(b.x, nbits20));
        ry = merge(ry, vertex_range(b.y, nbits20));
      }
    }
    rx = merge(rx, shfl_down1(rx));
    ry = merge(ry, shfl_down1(ry));
    if (y > ys) {
      const bool active = corner_col;
      const bool surv = active && (p.no_filter || !cube_excluded2(merge(px, rx), merge(py, ry)));
      append_survivors(p, surv, (u64)(x - p.lb[0]) + (u64)p.nc[0] * (u64)(y - 1 - p.lb[1]));
    }
    px = rx;
    py = ry;
  }
}

// ---- 3D: a block owns a 32 x BY column tile (31 x (BY-1) corners) and marches along z -------------
constexpr int SCAN3_BY = 16;

template <bool HAS_NEXT>
__global__ void __launch_bounds__(32 * SCAN3_BY) scan3d_kernel(const SweepParams p) {
  __shared__ int sh[2][6][SCAN3_BY][32];
  const int lane = threadIdx.x, ty = threadIdx.y;
  int b = blockIdx.x;
  const int bx = b % p.nsx; b /= p.nsx;
  const int by = b % p.nsy;
  const int bz = b / p.nsy;
  const int x = p.lb[0] + bx * 31 + lane;
  const int y = p.lb[1] + by * (SCAN3_BY - 1) + ty;
  const bool col_ok = x <= p.vmax[0] && y <= p.vmax[1];
  const bool corner_col = lane < 31 && ty < SCAN3_BY - 1 && x <= p.ub[0] && y <= p.ub[1];
  const int zs = p.lb[2] + bz * p.rows;
  const int ze = min(zs + p.rows - 1, p.ub[2]);
  const int nbits20 = p.nbits << 20;
  const int *__restrict__ V0 = reinterpret_cast<const int *>(p.L[0].V);
  const int *__restrict__ V1 = reinterpret_cast<const int *>(p.L[1].V);
  const size_t plane = (size_t)p.W * (size_t)p.H;
  const size_t col = (size_t)x + (size_t)p.W * (size_t)y;

  KeyRange pr[3] = {neutral_range(), neutral_range(), neutral_range()};   // previous plane, merged over t, x, y
  for (int z = zs; z <= ze + 1; z++) {
    KeyRange r[3] = {neutral_range(), neutral_range(), neutral_range()};
    if (col_ok && z <= p.vmax[2]) {
      const size_t w = (col + plane * (size_t)z) * 6 + 1;   // high word of component 0
#pragma unroll
      for (int c = 0; c < 3; c++) {
        r[c] = vertex_range(__ldg(V0 + w + 2 * c), nbits20);
        if (HAS_NEXT) r[c] = merge(r[c], vertex_range(__ldg(V1 + w + 2 * c), nbits20));
      }
    }
    const int buf = z & 1;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      r[c] = merge(r[c], shfl_down1(r[c]));
      sh[buf][2 * c][ty][lane] = r[c].mn;
      sh[buf][2 * c + 1][ty][lane] = r[c].mx;
    }
    __syncthreads();
    if (ty < SCAN3_BY - 1) {
#pragma unroll
      for (int c = 0; c < 3; c++)
        r[c] = merge(r[c], KeyRange{sh[buf][2 * c][ty + 1][lane], sh[buf][2 * c + 1][ty + 1][lane]});
    }
    if (z > zs) {
      const bool surv = corner_col &&
          (p.no_filter || !cube_excluded3(merge(pr[0], r[0]), merge(pr[1], r[1]), merge(pr[2], r[2])));
      append_survivors(p, surv, (u64)(x - p.lb[0]) + (u64)p.nc[0] * ((u64)(y - p.lb[1]) + (u64)p.nc[1] * (u64)(z - 1 - p.lb[2])));
    }
#pragma unroll
    for (int c = 0; c < 3; c++) pr[c] = r[c];
  }
}

// ---- 2D, scalar input: central-difference gradient (grad.hh:10-31) fused into the scan -------------
// The vector field is never materialised.  A warp owns a strip of 64 vertex columns (two per lane,
// two 8-byte loads per lane, row and layer) and marches along y with a four-row register window
// per layer (three rows of stencil + one row of prefetch; the row loop is unrolled by four so the
// window rotates without register moves); x neighbours come from warp shuffles.  It runs where the
// rows are not 16-byte aligned (odd W, or a borrowed pointer off a 16-byte boundary); aligned rows
// take the range-cell kernels below.
//
// Per row the kernel derives the fp64 gradient of both layers exactly as gradient2D does, rounds
// each component to fp32 and keeps fp32 min/max ranges per component (merged over the two layers,
// then x..x+1, then y..y+1).  The exclusion test on those ranges is conservative in every rounding:
//   * sidedness uses thr+ = 2^-nbits (1 + 2^-20): approx(v) >= thr+  =>  v >= 2^-nbits  <=>
//     trunc(v 2^nbits) >= 1 (scaling by a power of two is exact); values closer to the threshold
//     than fp32 resolves simply leave the cube to the exact test;
//   * the magnitude bound pads M and R by more than the fp32 rounding of their inputs;
//   * vertices outside the tracker's domain or the array are NOT masked out of the ranges: a range
//     that covers more vertices than the valid simplices use can only refine more cubes;
//   * NaN components never enter a range (FMNMX drops them): a simplex with a NaN vertex is rejected
//     by the reference before the predicate; +-Inf makes the bound infinite, so the cube is refined.
// Survivors go to the same exact per-simplex test as in the vector-layer path, so results do not
// depend on any of these approximations.
//
// By-product: min non-zero |v| (ndarray.hh:769-779) of the layers whose resolution is still unknown,
// over the WHOLE array -- which is why strips cover the array and not only the tracker's domain.
struct FRange { float mn, mx; };

// raw high word of an fp64 value read as fp32: an order-preserving key (sign | 11 exponent bits | 20 mantissa bits) for
// magnitudes below 2^1017; FMNMX orders such keys like the values, NaN patterns (>= 2^1017, Inf, NaN) drop out
constexpr int KEYF_BIG = 0x7E700000;     // high word of 2^1000
constexpr int KEYF_NAN = 0x7FC00000;
__device__ __forceinline__ float hikey(double d) { return __int_as_float(__double2hiint(d)); }

__device__ __forceinline__ FRange fmerge(FRange a, FRange b) { return FRange{fminf(a.mn, b.mn), fmaxf(a.mx, b.mx)}; }
__device__ __forceinline__ FRange fshfl_down1(FRange a) {
  return FRange{__shfl_down_sync(0xffffffffu, a.mn, 1), __shfl_down_sync(0xffffffffu, a.mx, 1)};
}

// thrp = 2^-nbits (1 + 2^-20), thr2 = 2^(1-nbits), limf = 0.999 * 4.5e18 / factor^2; all values in field units
__device__ __forceinline__ bool cube_excluded2_f(FRange x, FRange y, float thrp, float thr2, float limf) {
  const bool sided = x.mn >= thrp || x.mx <= -thrp || y.mn >= thrp || y.mx <= -thrp;
  // |quantised| <= |v| factor; quantised spread <= spread factor + 1; fp32 rounding of the inputs is
  // covered by the relative pads (2^-20 >> 2^-24)
  const float Mx = __fmaf_rn(fmaxf(-x.mn, x.mx), 1.000001f, thr2), My = __fmaf_rn(fmaxf(-y.mn, y.mx), 1.000001f, thr2);
  const float Rx = __fmaf_rn(Mx, 9.5367431640625e-7f, x.mx - x.mn) + thr2;
  const float Ry = __fmaf_rn(My, 9.5367431640625e-7f, y.mx - y.mn) + thr2;
  return sided && (__fmaf_rn(Mx, Ry, My * Rx) < limf);      // NaN / Inf compare false: the cube is refined
}

__device__ __forceinline__ void warp_res_commit(double m, unsigned long long *slot) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m < DBL_MAX) atomicMin(slot, (unsigned long long)__double_as_longlong(m));
}

__device__ __forceinline__ double nz_abs_d(double v) { const double a = fabs(v); return (v != 0.0 && a < DBL_MAX) ? a : DBL_MAX; }

template <bool HAS_NEXT, bool BORDER>
__device__ __forceinline__ void fused2d_strip(const SweepParams &p, const int b, const int cy, const int lane) {
  constexpr int NL = HAS_NEXT ? 2 : 1;
  const int W = p.W, H = p.H;
  const int e = b + 2 * lane, o = e + 1;     // this lane's two columns
  const bool e_in = !BORDER || e < W, o_in = !BORDER || o < W, o1_in = !BORDER || o + 1 < W;
  // the gradient needs both x neighbours inside the strip (or the array border, where the index clamps)
  const bool e_valid = e_in && (lane > 0 || b == 0);
  const bool o_valid = o_in && (lane < 31 || o == W - 1);
  // corner columns b+1 .. b+60 belong to this strip (strip 0 also owns column 0)
  const bool e_own = ((lane >= 1 && lane <= 30) || (lane == 0 && b == 0)) && e >= p.lb[0] && e <= p.ub[0];
  const bool o_own = lane <= 29 && o >= p.lb[0] && o <= p.ub[0];
  const int r0 = cy * p.rows;
  const int r1 = min(r0 + p.rows - 1, H - 1);        // last corner row of the chunk
  const int jl = r1 + 1;                             // last gradient row visited
  const double cw = (double)(W - 1), ch = (double)(H - 1);
  const float cwf = (float)(W - 1), chf = (float)(H - 1);
  const float thrp = p.thrp_f, thr2 = p.thr2_f, limf = p.lim_f;
  const bool want_res[2] = {p.res_slot[0] != nullptr, HAS_NEXT && p.res_slot[1] != nullptr};
  double rmin[2] = {DBL_MAX, DBL_MAX};
  float rminf[2] = {3.4028234e38f, 3.4028234e38f};   // fp32 candidate filter: slightly above rmin

  // row pointers advance by one row per step; rows past the array's last row re-read it (index clamp)
  const double *q[NL];
  {
    const size_t off = (size_t)W * (size_t)clampi(r0 - 1, H) + e;
#pragma unroll
    for (int L = 0; L < NL; L++) q[L] = (L == 0 ? p.L[0].S : p.L[1].S) + off;
  }
  int qrow = clampi(r0 - 1, H);
  auto loadrow = [&](const int r, double (&dst)[NL][2]) {   // r is requested in increasing order, one row at a time
    const int rc = clampi(r, H);
    if (rc != qrow) {
      qrow = rc;
#pragma unroll
      for (int L = 0; L < NL; L++) q[L] += W;
    }
#pragma unroll
    for (int L = 0; L < NL; L++) {
      dst[L][0] = e_in ? __ldg(q[L]) : 0.0;
      dst[L][1] = o_in ? __ldg(q[L] + 1) : 0.0;
    }
  };

  // one gradient row j: stencil rows (m1, c0, p1); pf receives row j+2; prev/cur are the x-merged
  // ranges of rows j-1 / j for the corner columns e and o: [corner column][component]
  auto step = [&](const int j, double (&m1)[NL][2], double (&c0)[NL][2], double (&p1)[NL][2], double (&pf)[NL][2],
                  FRange (&prev)[2][2], FRange (&cur)[2][2]) {
    if (j + 1 <= jl) loadrow(j + 2, pf);
    FRange ve[2], vo[2];   // per component, layers merged
#pragma unroll
    for (int L = 0; L < NL; L++) {
      double left = __shfl_up_sync(0xffffffffu, c0[L][1], 1), right = __shfl_down_sync(0xffffffffu, c0[L][0], 1);
      double mid_e = c0[L][1];
      if (BORDER) {
        if (e == 0) left = c0[L][0];
        if (!o_in) mid_e = c0[L][0];
        if (!o1_in) right = c0[L][1];
      }
      // exact fp64 differences; the scaling by (W-1), (H-1) is done in fp32 here (only the conservative
      // ranges use it) and in fp64, as the reference does, wherever a value is needed exactly
      const double dxe = mid_e - left, dxo = right - c0[L][0], dye = p1[L][0] - m1[L][0], dyo = p1[L][1] - m1[L][1];
      const float fxe = __double2float_rn(dxe) * cwf, fxo = __double2float_rn(dxo) * cwf;
      const float fye = __double2float_rn(dye) * chf, fyo = __double2float_rn(dyo) * chf;
      if (want_res[L] && j < H) {
        // candidates for a new minimum of the non-zero |v|: decided in fp32 against a filter that sits
        // above the fp64 minimum; exact zeros (and fp32 underflow) also take the exact path
        const float ae = e_valid ? fminf(fabsf(fxe), fabsf(fye)) : 3.4028234e38f;
        const float ao = o_valid ? fminf(fabsf(fxo), fabsf(fyo)) : 3.4028234e38f;
        if (fminf(ae, ao) < rminf[L]) {
          double m = rmin[L];
          if (e_valid) m = fmin(m, fmin(nz_abs_d(dxe * cw), nz_abs_d(dye * ch)));
          if (o_valid) m = fmin(m, fmin(nz_abs_d(dxo * cw), nz_abs_d(dyo * ch)));
          rmin[L] = m;
          rminf[L] = m < 1e38 ? __double2float_ru(m) * 1.000001f : 3.4028234e38f;
        }
      }
      if (L == 0) {
        ve[0] = FRange{fxe, fxe}; ve[1] = FRange{fye, fye}; vo[0] = FRange{fxo, fxo}; vo[1] = FRange{fyo, fyo};
      } else {
        ve[0] = fmerge(ve[0], FRange{fxe, fxe}); ve[1] = fmerge(ve[1], FRange{fye, fye});
        vo[0] = fmerge(vo[0], FRange{fxo, fxo}); vo[1] = fmerge(vo[1], FRange{fyo, fyo});
      }
    }
    // x merge: corner column c covers vertex columns c and c+1
#pragma unroll
    for (int c = 0; c < 2; c++) {
      cur[0][c] = fmerge(ve[c], vo[c]);
      cur[1][c] = fmerge(vo[c], fshfl_down1(ve[c]));
    }
    if (j > r0) {
      const int y = j - 1;
      const bool yrow = y >= p.lb[1] && y <= p.ub[1];
      const bool se = yrow && e_own && !cube_excluded2_f(fmerge(prev[0][0], cur[0][0]), fmerge(prev[0][1], cur[0][1]), thrp, thr2, limf);
      const bool so = yrow && o_own && !cube_excluded2_f(fmerge(prev[1][0], cur[1][0]), fmerge(prev[1][1], cur[1][1]), thrp, thr2, limf);
      if (__any_sync(0xffffffffu, se || so)) {
        append_survivors(p, se, (u64)(e - p.lb[0]) + (u64)p.nc[0] * (u64)(y - p.lb[1]));
        append_survivors(p, so, (u64)(o - p.lb[0]) + (u64)p.nc[0] * (u64)(y - p.lb[1]));
      }
    }
  };

  double s[4][NL][2];
  FRange R[2][2][2];
  loadrow(r0 - 1, s[0]);
  loadrow(r0, s[1]);
  loadrow(r0 + 1, s[2]);
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int c = 0; c < 2; c++) R[1][a][c] = FRange{0.f, 0.f};   // never read: the first row has no previous row
  for (int j = r0; j <= jl; j += 4) {
    step(j, s[0], s[1], s[2], s[3], R[1], R[0]);
    if (j + 1 <= jl) step(j + 1, s[1], s[2], s[3], s[0], R[0], R[1]);
    if (j + 2 <= jl) step(j + 2, s[2], s[3], s[0], s[1], R[1], R[0]);
    if (j + 3 <= jl) step(j + 3, s[3], s[0], s[1], s[2], R[0], R[1]);
  }
#pragma unroll
  for (int L = 0; L < NL; L++)
    if (want_res[L]) warp_res_commit(rmin[L], p.res_slot[L]);
}

template <bool HAS_NEXT>
__global__ void __launch_bounds__(256, 2) scan2d_fused_kernel(const SweepParams p) {
  const int lane = threadIdx.x & 31;
  const i64 warp = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int sx = (int)(warp % p.nsx), cy = (int)(warp / p.nsx);
  if (cy >= p.nsy) return;
  const int b = sx * 60;                     // first loaded column of the strip (even)
  if (b == 0 || b + 65 > p.W) fused2d_strip<HAS_NEXT, true>(p, b, cy, lane);    // touches the array's left / right edge
  else fused2d_strip<HAS_NEXT, false>(p, b, cy, lane);
}

// ---- staging helpers of the range-cell scans ----------------------------------------------------------------------
// The scalar build kernels below stage rows (2D) or planes (3D) in a shared-memory ring with the async copy engine
// (cp.async.bulk / cp.async.bulk.tensor, completion on a stage's `full` mbarrier).  Consumer warps wait on `full` and
// never synchronise with each other; a stage is refilled once every consumer warp has released it (2D: a producer
// warp waits on the stage's `empty` mbarrier; 3D: the last warp to release it issues the copy).  A 2D strip owns
// FB_STRIDE corner columns and reads FB_SEG columns of a row.
constexpr int FB_SEG = 68;         // doubles per row segment of a strip: columns c0-2 .. c0+65
constexpr int FB_STRIDE = 62;      // corner columns owned per strip (c0 .. c0+61)

__device__ __forceinline__ uint32_t smem_u32(const void *q) { return (uint32_t)__cvta_generic_to_shared(q); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}

template <int K> struct IC { static constexpr int value = K; };

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// exact update of the running min non-zero |v| with the four gradient values of one step (v = d * c in
// fp64, as gradient2D computes them); m keeps the signed value with the smallest non-zero magnitude
__device__ __forceinline__ void res_update4(double &m, float &mf, bool e_in, bool o_in, double dxe, double dye, double dxo, double dyo, double cw, double ch) {
  const double vxe = dxe * cw, vye = dye * ch, vxo = dxo * cw, vyo = dyo * ch;
  if (e_in) {
    if (vxe != 0.0 && fabs(vxe) < fabs(m)) m = vxe;     // NaN / Inf never compare below
    if (vye != 0.0 && fabs(vye) < fabs(m)) m = vye;
  }
  if (o_in) {
    if (vxo != 0.0 && fabs(vxo) < fabs(m)) m = vxo;
    if (vyo != 0.0 && fabs(vyo) < fabs(m)) m = vyo;
  }
  mf = fabs(m) < 1e38 ? __double2float_ru(fabs(m)) * 1.000001f : 3.4028234e38f;
}

// ---- 2D, scalar input, per-layer range cells ("build once, test from cells") ---------------------------------
// Same idea as the 3D cells below: the fp32 ranges of the register scan above depend on one layer only, so
// a layer is streamed once -- by the step that first sees it -- and leaves a 16-byte cell {min vx, max vx, min vy,
// max vy} per (lane, block of C2_R corner rows); the step reads the CURRENT layer's cells instead of the layer.
// A cell spans the lane's two columns, the next lane's two, and gradient rows 9k .. 9k+9: a superset of the
// vertices of the lane's 2 x 9 cubes.  If the union of the two layers' cells passes cube_excluded2_f, all 18 cubes
// are excluded; otherwise they are tested one by one from global memory (cold) and survivors are appended.
// Traffic per step: 8 B/vertex of scalars + ~1 B/vertex of cells written + ~1 B/vertex read (16 B/vertex for a scan that re-reads both layers).
constexpr int C2_R = 9;                                // corner rows per cell block (a multiple of 3: the row window rotates by index)
constexpr int C2_NST = 9;                              // ring stages (rows) = unroll of the row loop = C2_R
constexpr int C2_CW = 7;                               // consumer warps per CTA (plus one producer warp)
constexpr int C2_SEG = C2_CW * FB_STRIDE + 8;          // staged doubles per row: columns C0-2 .. C0+439
static_assert(C2_R % 3 == 0 && C2_R == C2_NST && C2_R == SCAN2D_CELL_ROWS, "row window / ring / cell block must stay aligned");

__device__ __forceinline__ size_t cells2d_index(const SweepParams &p, const int strip, const int kb, const int lane) {
  const size_t nblk = (size_t)(p.H / C2_R + 2);
  return ((size_t)strip * nblk + (size_t)kb) * 32u + (size_t)lane;
}

// cold path: for every lane whose cell union failed (bit set in failmask), the WARP tests that lane's 2 x C2_R cubes,
// one lane per cube: ranges over the vertices valid simplices can use (<= ub) from global memory, gradient exactly
// as gradient2D indexes it (clamped at the array border); survivors are appended.
template <int NL>
__device__ __forceinline__ void cells2d_slow_cubes_t(const SweepParams &p, unsigned failmask, const int c0, const int y0, const uint32_t stage) {
  static_assert(2 * C2_R <= 32, "one lane per cube");
  const int W = p.W, H = p.H;
  const int lane = threadIdx.x & 31;
  const float cwf = (float)(W - 1), chf = (float)(H - 1);
  const float nanf_ = __int_as_float(0x7FC00000);
  // the 2 x C2_R cubes of every failing lane, packed 32 to a pass (a failing lane alone would keep 18 of 32 lanes busy)
  const int per = 2 * C2_R, total = per * __popc(failmask);
  for (int q0 = 0; q0 < total; q0 += 32) {
    const int qi = q0 + lane;
    const bool live = qi < total;
    const int which = live ? qi / per : 0, within = live ? qi % per : 0;
    const int src = (int)__fns(failmask, 0, which + 1);       // the which-th failing lane
    const int r = within >> 1, q = within & 1;
    const int x = c0 + 2 * src + q, y = y0 + r;
    const bool in = live && x >= p.lb[0] && x <= p.ub[0] && y >= p.lb[1] && y <= p.ub[1];
    // the cube's 3 x 3 (+ corners unused) stencil footprint: columns x-1 .. x+2, rows y-1 .. y+2, clamped like gradient2D clamps
    // them; every load of a layer is issued before the first one is used (a pass is one round trip to L2 per layer, not sixteen)
    const int xs[4] = {clampi(x - 1, W), clampi(x, W), clampi(x + 1, W), clampi(x + 2, W)};
    size_t rows_[4];
#pragma unroll
    for (int k = 0; k < 4; k++) rows_[k] = (size_t)W * (size_t)clampi(y - 1 + k, H);
    FRange rx{nanf_, nanf_}, ry{nanf_, nanf_};
#pragma unroll
    for (int L = 0; L < NL; L++) {
      const double *S = p.L[L].S;
      // h[j][k] = S(clamp(x - 1 + k), clamp(y + j)), lo / hi[i] = S(clamp(x + i), clamp(y - 1)) / S(clamp(x + i), clamp(y + 2)):
      // d/dx at vertex (x + i, y + j) = h[j][i + 2] - h[j][i], d/dy = (row y + j + 1) - (row y + j - 1) at column x + i
      double h[2][4], lo[2], hi[2];
#pragma unroll
      for (int j = 0; j < 2; j++)
#pragma unroll
        for (int k = 0; k < 4; k++) h[j][k] = __ldg(S + rows_[1 + j] + xs[k]);
#pragma unroll
      for (int i = 0; i < 2; i++) { lo[i] = __ldg(S + rows_[0] + xs[1 + i]); hi[i] = __ldg(S + rows_[3] + xs[1 + i]); }
#pragma unroll
      for (int v = 0; v < 4; v++) {
        const int i = v & 1, j = v >> 1;
        if (!in || x + i > p.ub[0] || y + j > p.ub[1]) continue;
        const double dx = h[j][i + 2] - h[j][i];
        const double dy = (j == 0 ? h[1][i + 1] : hi[i]) - (j == 0 ? lo[i] : h[0][i + 1]);
        const float fx = __double2float_rn(dx) * cwf, fy = __double2float_rn(dy) * chf;
        rx = fmerge(rx, FRange{fx, fx}); ry = fmerge(ry, FRange{fy, fy});
      }
    }
    const bool surv = in && !cube_excluded2_f(rx, ry, p.thrp_f, p.thr2_f, p.lim_f);
    const u64 lin = (u64)(x - p.lb[0]) + (u64)p.nc[0] * (u64)(y - p.lb[1]);
    if (stage) stage_survivors(p, stage, surv, lin);          // (warp-uniform)
    else append_survivors(p, surv, lin);
  }
}
// cold path: for every lane whose cell union failed (bit set in failmask), the WARP tests that lane's 2 x C2_R cubes,
// one lane per cube: ranges over the vertices valid simplices can use (<= ub) from global memory, gradient exactly
// as gradient2D indexes it (clamped at the array border); survivors are appended.
// stage: shared-memory staging of this warp's survivors (flushed by the caller at the end), or 0: append directly
__device__ __noinline__ void cells2d_slow_cubes(const SweepParams &p, unsigned failmask, const int c0, const int y0, const int nl, const uint32_t stage = 0) {
  if (nl == 1) cells2d_slow_cubes_t<1>(p, failmask, c0, y0, stage);
  else cells2d_slow_cubes_t<2>(p, failmask, c0, y0, stage);
}

// union of the cells of all layers for one block -> excluded, or the cold path
__device__ __forceinline__ void cells2d_decide(const SweepParams &p, const FRange ux, const FRange uy, const bool own, const int e, const int y0, const int nl) {
  const bool fail = own && !cube_excluded2_f(ux, uy, p.thrp_f, p.thr2_f, p.lim_f);
  const unsigned fm = __ballot_sync(0xffffffffu, fail);
  if (fm) cells2d_slow_cubes(p, fm, e - 2 * (int)(threadIdx.x & 31), y0, nl);
}

template <bool BORDER, int NPREV, bool TEST>
__device__ __forceinline__ void cells2d_strip(const SweepParams &p, const int c0, const int r0, const int r1, const int lane,
                                              const double *tile /* this warp's column 0 = c0-2 */, const uint32_t full0, const uint32_t empty0,
                                              const int strip) {
  const int W = p.W, H = p.H, B = p.build_layer;
  const int e = c0 + 2 * lane, o = e + 1;
  const bool e_in = !BORDER || e < W, o_in = !BORDER || o < W, o1_in = !BORDER || o + 1 < W;
  const bool own_cols = lane <= 30 && ((e >= p.lb[0] && e <= p.ub[0]) || (o >= p.lb[0] && o <= p.ub[0]));
  const int jl = r1 + 1;                             // last gradient row visited
  const float cwf = (float)(W - 1), chf = (float)(H - 1);
  const bool want_res = p.res_slot[B] != nullptr;
  double rmin = DBL_MAX;
  float rminf = 3.4028234e38f;
  const uint4 *sum_prev = NPREV ? p.sum_in[0] + cells2d_index(p, strip, 0, lane) : nullptr;
  uint4 *sum_out = p.sum_out + cells2d_index(p, strip, 0, lane);

  const double *lane_base = tile + 2 * lane;    // [1]: column e-1, [2..3]: e, o, [4]: o+1
  auto centre = [&](const int st, double (&dst)[2]) {
    const double2 t = *reinterpret_cast<const double2 *>(lane_base + st * C2_SEG + 2);
    dst[0] = t.x; dst[1] = t.y;
  };
  auto release = [&](const int st) {     // this warp is done with the stage
    __syncwarp();
    if (elect_one()) mbar_arrive(empty0 + 8u * st);
  };
  // a block of C2_R corner rows is complete: x-neighbour merge, store the cell, test against the other layer's cell
  auto finish_block = [&](const int kb, FRange bx, FRange by, const uint4 prevc) {
    bx = fmerge(bx, fshfl_down1(bx));
    by = fmerge(by, fshfl_down1(by));
    sum_out[(size_t)kb * 32u] = make_uint4(__float_as_uint(bx.mn), __float_as_uint(bx.mx), __float_as_uint(by.mn), __float_as_uint(by.mx));
    if (TEST) {
      if (NPREV) {
        bx = fmerge(bx, FRange{__uint_as_float(prevc.x), __uint_as_float(prevc.y)});
        by = fmerge(by, FRange{__uint_as_float(prevc.z), __uint_as_float(prevc.w)});
      }
      const int y0 = kb * C2_R;
      const bool own = own_cols && y0 <= p.ub[1] && y0 + C2_R - 1 >= p.lb[1];
      cells2d_decide(p, bx, by, own, e, y0, NPREV + 1);
    }
  };

  double win[3][2];
  mbar_wait(full0, 0);
  centre(0, win[0]);
  mbar_wait(full0 + 8, 0);
  centre(1, win[1]);
  release(0);                                      // row r0-1: only its centre columns are ever needed
  FRange bx{0.f, 0.f}, by{0.f, 0.f};
  uint4 prevc = make_uint4(0x7FC00000u, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u);

  // gradient row j = r0 + C2_NST i + K (r0 is a multiple of C2_R = C2_NST); ring index of row j is 1 + C2_NST i + K
  auto step = [&](auto KC, const int j, const int i) {
    constexpr int K = decltype(KC)::value;
    constexpr int ST_J = (1 + K) % C2_NST, ST_P = (2 + K) % C2_NST;
    double (&m1)[2] = win[K % 3];
    double (&c0v)[2] = win[(K + 1) % 3];
    double (&p1)[2] = win[(K + 2) % 3];
    mbar_wait(full0 + 8u * ST_P, (uint32_t)((i + (2 + K >= C2_NST ? 1 : 0)) & 1));
    centre(ST_P, p1);
    const double *rowj = lane_base + ST_J * C2_SEG;
    double left = rowj[1], right = rowj[4];
    double mid_e = c0v[1];
    if (BORDER) {
      if (e == 0) left = c0v[0];
      if (!o_in) mid_e = c0v[0];
      if (!o1_in) right = c0v[1];
    }
    const double dxe = mid_e - left, dxo = right - c0v[0], dye = p1[0] - m1[0], dyo = p1[1] - m1[1];
    const float fxe = __double2float_rn(dxe) * cwf, fxo = __double2float_rn(dxo) * cwf;
    const float fye = __double2float_rn(dye) * chf, fyo = __double2float_rn(dyo) * chf;
    if (want_res && j < H) {
      float a = fminf(fminf(fabsf(fxe), fabsf(fye)), fminf(fabsf(fxo), fabsf(fyo)));
      if (BORDER) a = fminf(e_in ? fminf(fabsf(fxe), fabsf(fye)) : 3.4028234e38f, o_in ? fminf(fabsf(fxo), fabsf(fyo)) : 3.4028234e38f);
      if (a < rminf) res_update4(rmin, rminf, e_in, o_in, dxe, dye, dxo, dyo, (double)(W - 1), (double)(H - 1));
    }
    const FRange rx{fminf(fxe, fxo), fmaxf(fxe, fxo)}, ry{fminf(fye, fyo), fmaxf(fye, fyo)};
    if (K == 0) {
      // gradient row C2_R k closes block k-1 and opens block k
      if (j > r0) finish_block(j / C2_R - 1, fmerge(bx, rx), fmerge(by, ry), prevc);
      bx = rx; by = ry;
      if (NPREV && j < jl) prevc = __ldg(sum_prev + (size_t)(j / C2_R) * 32u);
    } else {
      bx = fmerge(bx, rx); by = fmerge(by, ry);
    }
    release(ST_J);     // row j: its centre went into the window one step ago, its x neighbours were read above
  };

  for (int j = r0, i = 0; j <= jl; j += C2_NST, i++) {
    step(IC<0>{}, j, i);
    if (j + 1 <= jl) step(IC<1>{}, j + 1, i);
    if (j + 2 <= jl) step(IC<2>{}, j + 2, i);
    if (j + 3 <= jl) step(IC<3>{}, j + 3, i);
    if (j + 4 <= jl) step(IC<4>{}, j + 4, i);
    if (j + 5 <= jl) step(IC<5>{}, j + 5, i);
    if (j + 6 <= jl) step(IC<6>{}, j + 6, i);
    if (j + 7 <= jl) step(IC<7>{}, j + 7, i);
    if (j + 8 <= jl) step(IC<8>{}, j + 8, i);
  }
  if (jl % C2_R != 0) finish_block(jl / C2_R, bx, by, prevc);     // the array's last, partial block
  if (want_res) warp_res_commit(fabs(rmin), p.res_slot[B]);
}

template <int NPREV, bool TEST>
__global__ void __launch_bounds__((C2_CW + 1) * 32, 3) scan2d_build_kernel(const __grid_constant__ SweepParams p) {
  constexpr uint32_t STAGE_BYTES = C2_SEG * 8;
  extern __shared__ __align__(128) unsigned char fb_smem[];
  const int lane = threadIdx.x & 31;
  const int wib = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);     // warp-uniform by construction
  double *ring = reinterpret_cast<double *>(fb_smem);
  const uint32_t full0 = smem_u32(fb_smem + (size_t)C2_NST * STAGE_BYTES), empty0 = full0 + 8u * C2_NST;
  const int W = p.W, H = p.H;
  const int bx = blockIdx.x % p.nsx, cy = blockIdx.x / p.nsx;
  const int C0 = bx * (C2_CW * FB_STRIDE);
  const int nactive = min(C2_CW, (W - C0 + FB_STRIDE - 1) / FB_STRIDE);     // consumer warps whose strip starts inside the array
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < C2_NST; q++) { mbar_init(full0 + 8u * q, 1); mbar_init(empty0 + 8u * q, (uint32_t)nactive); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  const int r0 = cy * p.rows;                        // p.rows is a multiple of C2_R
  const int r1 = min(r0 + p.rows - 1, H - 1);
  const int nrows = (r1 + 1) - r0 + 3;               // staged rows r0-1 .. r1+2 (ring index 0 .. nrows-1)
  if (wib == C2_CW) {
    // producer: one elected lane walks the rows with the array's index clamp and keeps the ring full
    if (elect_one()) {
      const double *S = p.L[p.build_layer].S;
      const int col_lo = max(C0 - 2, 0), col_hi = min(C0 - 2 + C2_SEG, W);
      const uint32_t seg_bytes = (uint32_t)(col_hi - col_lo) * 8u;
      const uint32_t dst0 = smem_u32(ring) + (uint32_t)(col_lo - (C0 - 2)) * 8u;
      for (int rr = 0; rr < nrows; rr++) {
        const int st = rr % C2_NST;
        if (rr >= C2_NST) mbar_wait(empty0 + 8u * st, (uint32_t)((rr / C2_NST - 1) & 1));
        const size_t off = (size_t)W * (size_t)clampi(r0 - 1 + rr, H) + (size_t)col_lo;
        mbar_expect_tx(full0 + 8u * st, seg_bytes);
        bulk_g2s(dst0 + (uint32_t)st * STAGE_BYTES, S + off, seg_bytes, full0 + 8u * st);
      }
    }
    return;
  }
  if (wib >= nactive) return;
  const int c0 = C0 + wib * FB_STRIDE;
  const double *tile = ring + wib * FB_STRIDE;
  const bool border = c0 == 0 || c0 + FB_SEG - 2 > W;      // strips that touch the array's left / right edge clamp their columns
  if (border) cells2d_strip<true, NPREV, TEST>(p, c0, r0, r1, lane, tile, full0, empty0, bx * C2_CW + wib);
  else cells2d_strip<false, NPREV, TEST>(p, c0, r0, r1, lane, tile, full0, empty0, bx * C2_CW + wib);
}

// cells only: the final ordinal sweep (one layer) and re-sweeps (both layers' cells exist); thread per cell
template <int NL>
__global__ void __launch_bounds__(256) scan2d_cells_kernel(const __grid_constant__ SweepParams p, const int nstrips, const int nblk_used) {
  const int lane = threadIdx.x & 31;
  const long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);   // 8 warps per CTA
  if (w >= (long long)nstrips * nblk_used) return;
  const int strip = (int)(w / nblk_used), kb = (int)(w % nblk_used);
  const int e = strip * FB_STRIDE + 2 * lane, y0 = kb * C2_R;
  const bool own = lane <= 30 && ((e >= p.lb[0] && e <= p.ub[0]) || (e + 1 >= p.lb[0] && e + 1 <= p.ub[0])) && y0 <= p.ub[1] && y0 + C2_R - 1 >= p.lb[1];
  if (!__any_sync(0xffffffffu, own)) return;
  const float nanf_ = __int_as_float(0x7FC00000);
  FRange ux{nanf_, nanf_}, uy{nanf_, nanf_};
#pragma unroll
  for (int L = 0; L < NL; L++) {
    const uint4 c = __ldg(p.sum_in[L] + cells2d_index(p, strip, kb, lane));
    ux = fmerge(ux, FRange{__uint_as_float(c.x), __uint_as_float(c.y)});
    uy = fmerge(uy, FRange{__uint_as_float(c.z), __uint_as_float(c.w)});
  }
  cells2d_decide(p, ux, uy, own, e, y0, NL);
}

// ---- 2D, scalar input, range cells from high-word keys (default build kernel) -----------------------------------------
// Same cells, same geometry and the same consumers as scan2d_build_kernel (cells kernel, cold path, peer export), but the
// hot loop never converts fp64 to fp32: the raw high word of each fp64 difference d = S(x+1) - S(x-1) (not yet scaled by
// W-1) is used as an order-preserving fp32 key (sign | 11 exponent bits | 20 mantissa bits read as a float: monotone in d
// for |d| < 2^1017), so a row costs four DADD and four three-input FMNMX per lane.  Keys become conservative fp32 ranges of
// v = d (W-1) once per cell block of 9 rows: a key truncates |d| towards zero, so bounds that must move away from zero take
// the next key; key x (W-1) is exact in fp64 (21 x 31 significant bits), the final rounding is directed outwards.
// Staging: ring of K2_NST stages of K2_R = 3 rows each (cp.async.bulk + full/empty mbarriers, one producer warp); a consumer
// warp moves a whole stage into registers (3 x LDS.128 + 6 x LDS.64 through explicit shared-space loads) and releases it at
// once, so a stage is busy for a few dozen cycles and the ring is almost always in flight.
// Scalars >= 2^1000 / Inf / NaN cannot be ordered by the keys: they raise p.poison and the context redoes the step with
// scan2d_build_kernel (fp32 ranges, handles them).
constexpr int K2_R = 3;                                // rows per stage
constexpr int K2_NST = 4;                              // ring stages (42 KB per CTA)
constexpr int K2_CTAS = 3;                             // CTAs per SM
constexpr uint32_t K2_ROW_BYTES = C2_SEG * 8;
constexpr uint32_t K2_STAGE_BYTES = K2_R * K2_ROW_BYTES;
static_assert(C2_R % K2_R == 0, "cell block = whole stages");

__device__ __forceinline__ double2 lds128_f64(uint32_t a) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ double lds64_f64(uint32_t a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
// 16 bytes global -> shared without a register (LDGSTS); completion: cp_async_wait_all of the issuing thread
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds128_u32(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts64_f64(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
// max that keeps a NaN once it has seen one (FMNMX.NAN): the "magnitude too large for float keys" accumulator
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// running minimum of the non-zero magnitudes, branch-free (two DSETP + select per value): the moving-extremum fields are
// adversarial for a filtered slow path -- |dS/dy| shrinks row by row towards the extremum, so every row is a new minimum
__device__ __forceinline__ double nzmin(double m, double d) {     // m, d signed: |.| folds into the compare's operand modifiers
  double r;                                                      // (|d| < |m| && d != 0) ? d : m -- NaN compares false, Inf never below
  asm("{\n\t.reg .pred p, q;\n\t.reg .f64 ad, am;\n\tabs.f64 ad, %2;\n\tabs.f64 am, %1;\n\t"
      "setp.neu.f64 q, %2, 0d0000000000000000;\n\tsetp.lt.and.f64 p, ad, am, q;\n\tselp.f64 %0, %2, %1, p;\n\t}"
      : "=d"(r) : "d"(m), "d"(d));
  return r;
}

// conservative fp32 range of v = d * c over the values whose keys lie in [kmn, kmx]
__device__ __forceinline__ FRange k2_vrange(float kmn, float kmx, double c) {
  const int a = __float_as_int(kmn), b = __float_as_int(kmx);
  const double lo = __hiloint2double(a < 0 ? a + 1 : a, 0);     // negative: the truncated key is too close to zero
  const double hi = __hiloint2double(b < 0 ? b : b + 1, 0);     // positive: likewise
  return FRange{__double2float_rd(lo * c), __double2float_ru(hi * c)};
}

__device__ __forceinline__ void prefetch_l2(const void *q) { asm volatile("prefetch.global.L2 [%0];" ::"l"(q)); }

struct K2Acc { double mdx, mdy; float big; };     // per-lane accumulators carried across the segments of a persistent CTA

// one segment of one strip; a function of its own (not inlined) so that the hot loop gets the whole register file and the
// persistent loop's bookkeeping is saved once per segment, not kept live across it
template <bool BORDER, int NPREV, bool TEST>
__device__ __forceinline__ K2Acc keys2d_strip(const SweepParams &p, const int c0, const int r0, const int r1, const int lane,
                                           const uint32_t tile_u32 /* smem address of this warp's column c0-2, stage 0, row 0 */,
                                           const uint32_t full0, const uint32_t empty0, const int strip,
                                           const uint32_t sbase /* ring stages this CTA has consumed before this segment */,
                                           const uint32_t res_u32 /* smem: this thread's {min dx, min dy}; only the rare exact path touches them */,
                                           const uint32_t wl_stage /* smem: this warp's survivor staging (empty on entry and on exit) */,
                                           const uint32_t cell_stage /* smem: this lane's two 16-byte slots (512 bytes apart) for the other layer's cells */,
                                           const K2Acc acc) {
  float big = acc.big;
  const int W = p.W, H = p.H, B = p.build_layer;
  const int e = c0 + 2 * lane, o = e + 1;
  const bool e_in = !BORDER || e < W, o_in = !BORDER || o < W, o1_in = !BORDER || o + 1 < W;
  const bool own_cols = lane <= 30 && ((e >= p.lb[0] && e <= p.ub[0]) || (o >= p.lb[0] && o <= p.ub[0]));
  const int jl = r1 + 1;                              // last gradient row visited
  const int nrows = jl - r0 + 1;                      // gradient rows r0 .. jl; ring rows 0 .. nrows+1 hold array rows r0-1 .. jl+1
  const int ngroups = (nrows + K2_R - 1) / K2_R, nstages = (nrows + 2 + K2_R - 1) / K2_R;
  const double cw = (double)(W - 1), ch = (double)(H - 1);
  const bool want_res = p.res_slot[B] != nullptr;
  const float thrx = p.res_thr[0], thry = p.res_thr[1];
  const uint4 *sum_prev = NPREV ? p.sum_in[0] + cells2d_index(p, strip, 0, lane) : nullptr;
  uint4 *sum_out = p.sum_out + cells2d_index(p, strip, 0, lane);
  const uint32_t lane_u32 = tile_u32 + (uint32_t)lane * 16u;    // +8: column e-1, +16: e, o, +32: o+1
  const int kb0 = r0 / C2_R;                          // first block of the segment (a segment has at most 64 blocks)
  unsigned long long failbits = 0;
  const int kb_end = ((r1 + 1) + C2_R - 1) / C2_R;     // blocks up to kb_end-1 are closed by this segment

  // a block of C2_R corner rows is complete: x-neighbour merge on the keys, keys -> fp32 ranges of v, store the cell, test
  auto finish_block = [&](const int kb, float xmn, float xmx, float ymn, float ymx) {
    xmn = fminf(xmn, __shfl_down_sync(0xffffffffu, xmn, 1)); xmx = fmaxf(xmx, __shfl_down_sync(0xffffffffu, xmx, 1));
    ymn = fminf(ymn, __shfl_down_sync(0xffffffffu, ymn, 1)); ymx = fmaxf(ymx, __shfl_down_sync(0xffffffffu, ymx, 1));
    FRange bx = k2_vrange(xmn, xmx, cw), by = k2_vrange(ymn, ymx, ch);
    sum_out[(size_t)kb * 32u] = make_uint4(__float_as_uint(bx.mn), __float_as_uint(bx.mx), __float_as_uint(by.mn), __float_as_uint(by.mx));
    if (TEST) {
      if (NPREV && kb < kb_end) {
        // the other layer's cell of this block: requested into L2 two blocks ago (a DRAM miss: ~1 us), copied into shared memory
        // by cp.async when the block opened -- no register is live across the block's nine rows (four of them cost the loop six
        // spilled scalars), and the L2 latency is not waited for here (a plain load at this point was 8 % of the warp samples)
        cp_async_wait_all();
        const uint4 prevc = lds128_u32(cell_stage + ((uint32_t)kb & 1u) * 512u);
        bx = fmerge(bx, FRange{__uint_as_float(prevc.x), __uint_as_float(prevc.y)});
        by = fmerge(by, FRange{__uint_as_float(prevc.z), __uint_as_float(prevc.w)});
      }
      const int y0 = kb * C2_R;
      const bool own = own_cols && y0 <= p.ub[1] && y0 + C2_R - 1 >= p.lb[1];
      // a union that does not prove its 18 cubes excluded is only noted here (one bit per block of the segment): the per-cube
      // refinement runs after the row loop, so the hot loop contains no call and keeps its registers
      if (own && !cube_excluded2_f(bx, by, p.thrp_f, p.thr2_f, p.lim_f)) failbits |= 1ull << (kb - kb0);
    }
  };

  // two register sets of one stage each: the centre columns (e, o) of its three rows, and the keys of their x differences --
  // d/dx only involves the row itself, so it is formed (and its exact minimum taken) while the stage is unloaded and only
  // the two 32-bit keys stay live
  double C[2][K2_R][2];
  float KX[2][K2_R][2];
  auto load_stage = [&](auto PC, const int s) {
    constexpr int P = decltype(PC)::value;
    const uint32_t gs = sbase + (uint32_t)s, slot = gs % K2_NST;
    mbar_wait(full0 + 8u * slot, (gs / K2_NST) & 1u);
    const uint32_t base = lane_u32 + slot * K2_STAGE_BYTES;
    double nl[K2_R], nr[K2_R];
#pragma unroll
    for (int i = 0; i < K2_R; i++) {
      const double2 c = lds128_f64(base + (uint32_t)i * K2_ROW_BYTES + 16u);
      C[P][i][0] = c.x; C[P][i][1] = c.y;
      nl[i] = lds64_f64(base + (uint32_t)i * K2_ROW_BYTES + 8u);
      nr[i] = lds64_f64(base + (uint32_t)i * K2_ROW_BYTES + 32u);
    }
    float ax = __int_as_float(0x7F800000);
#pragma unroll
    for (int i = 0; i < K2_R; i++) {
      const float ke = fabsf(hikey(C[P][i][0])), ko = fabsf(hikey(C[P][i][1]));
      big = fmax_nan(big, BORDER ? (e_in ? ke : 0.f) : ke);
      big = fmax_nan(big, BORDER ? (o_in ? ko : 0.f) : ko);
      double left = nl[i], right = nr[i], mid_e = C[P][i][1];
      if (BORDER) {
        if (e == 0) left = C[P][i][0];
        if (!o_in) mid_e = C[P][i][0];
        if (!o1_in) right = C[P][i][1];
      }
      const double dxe = mid_e - left, dxo = right - C[P][i][0];
      KX[P][i][0] = hikey(dxe); KX[P][i][1] = hikey(dxo);
      ax = fminf(ax, fminf(fabsf(KX[P][i][0]), fabsf(KX[P][i][1])));
    }
    // exact minimum of the non-zero |d|: only values whose key does not exceed the running minimum's (known when the step was
    // enqueued; +inf until a layer has been resolved) can lower it -- one vote per stage instead of two DSETP + select per value.
    // The rare path reads the x neighbours again (the stage is released after it) so that the differences need not stay live.
    if (want_res && __any_sync(0xffffffffu, ax <= thrx)) {
      double mdx = lds64_f64(res_u32);
#pragma unroll
      for (int i = 0; i < K2_R; i++) {
        const int j = r0 + K2_R * s + i - 1;              // the gradient row this ring row is the centre of
        if (j >= r0 && j <= jl && j < H) {
          double left = lds64_f64(base + (uint32_t)i * K2_ROW_BYTES + 8u), right = lds64_f64(base + (uint32_t)i * K2_ROW_BYTES + 32u), mid_e = C[P][i][1];
          if (BORDER) {
            if (e == 0) left = C[P][i][0];
            if (!o_in) mid_e = C[P][i][0];
            if (!o1_in) right = C[P][i][1];
          }
          if (e_in) mdx = nzmin(mdx, mid_e - left);
          if (o_in) mdx = nzmin(mdx, right - C[P][i][0]);
        }
      }
      sts64_f64(res_u32, mdx);
    }
    __syncwarp();
    if (elect_one()) mbar_arrive(empty0 + 8u * slot);   // the stage lives in registers now
  };

  float bxmn = 0.f, bxmx = 0.f, bymn = 0.f, bymx = 0.f;
  const uint4 nanc = make_uint4(0x7FC00000u, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u);
  int kb = r0 / C2_R;                                  // the block the next row with K == 0 opens
  // the other layer's cells are requested into L2 two blocks ahead of their use
  if (NPREV && kb < kb_end) prefetch_l2(sum_prev + (size_t)kb * 32u);
  if (NPREV && kb + 1 < kb_end) prefetch_l2(sum_prev + (size_t)(kb + 1) * 32u);

  // group g = gradient rows r0 + 3 g + {0, 1, 2}; ring row q holds array row r0 - 1 + q, gradient row r0 + q reads ring rows
  // q (below), q + 1 (centre, x neighbours), q + 2 (above).  PC: register set of stage g; phase: rows since the last block opened.
  // r0 is a multiple of C2_R = 9 = three groups: only the first row of every third group opens a block (gphase counts groups)
  int gphase = 0;
  static_assert(C2_R == 3 * K2_R, "a cell block is three groups");
  auto group = [&](auto PC, const int g) {
    constexpr int P = decltype(PC)::value;
    if (g + 1 < nstages) load_stage(IC<1 - P>{}, g + 1);
    const bool opens_group = gphase == 0;               // warp-uniform
    gphase = gphase == 2 ? 0 : gphase + 1;
    const int j0 = r0 + K2_R * g;
    const bool full = j0 + K2_R - 1 <= min(jl, H - 1);  // (warp-uniform) all three rows exist and count for min |v|
    float ay = __int_as_float(0x7F800000);
#pragma unroll
    for (int i = 0; i < K2_R; i++) {
      const int j = j0 + i;
      if (!full && j > jl) break;
      const double *m1 = C[P][i];
      const float *kx = i + 1 < K2_R ? KX[P][i + 1] : KX[1 - P][i + 1 - K2_R];
      const double *p1 = i + 2 < K2_R ? C[P][i + 2] : C[1 - P][i + 2 - K2_R];
      const double dye = p1[0] - m1[0], dyo = p1[1] - m1[1];
      const float kxe = kx[0], kxo = kx[1], kye = hikey(dye), kyo = hikey(dyo);
      ay = fminf(ay, fminf(fabsf(kye), fabsf(kyo)));
      if (i == 0 && opens_group) {
        // gradient row C2_R k closes block k-1 and opens block k
        const float rxmn = fminf(kxe, kxo), rxmx = fmaxf(kxe, kxo), rymn = fminf(kye, kyo), rymx = fmaxf(kye, kyo);
        if (j > r0) finish_block(kb - 1, fminf(bxmn, rxmn), fmaxf(bxmx, rxmx), fminf(bymn, rymn), fmaxf(bymx, rymx));
        bxmn = rxmn; bxmx = rxmx; bymn = rymn; bymx = rymx;
        if (NPREV && kb < kb_end) cp_async16(cell_stage + ((uint32_t)kb & 1u) * 512u, sum_prev + (size_t)kb * 32u);     // the block this row opens
        kb++;
        if (NPREV && kb + 1 < kb_end) prefetch_l2(sum_prev + (size_t)(kb + 1) * 32u);
      } else {
        bxmn = fminf(fminf(bxmn, kxe), kxo); bxmx = fmaxf(fmaxf(bxmx, kxe), kxo);
        bymn = fminf(fminf(bymn, kye), kyo); bymx = fmaxf(fmaxf(bymx, kye), kyo);
      }
    }
    if (want_res && __any_sync(0xffffffffu, ay <= thry)) {     // see load_stage: the rows of this group are still in registers
      double mdy = lds64_f64(res_u32 + 8u);
#pragma unroll
      for (int i = 0; i < K2_R; i++) {
        const int j = j0 + i;
        if (!full && (j > jl || j >= H)) break;
        const double *m1 = C[P][i];
        const double *p1 = i + 2 < K2_R ? C[P][i + 2] : C[1 - P][i + 2 - K2_R];
        if (e_in) mdy = nzmin(mdy, p1[0] - m1[0]);
        if (o_in) mdy = nzmin(mdy, p1[1] - m1[1]);
      }
      sts64_f64(res_u32 + 8u, mdy);
    }
  };

  load_stage(IC<0>{}, 0);
#pragma unroll 1
  for (int g = 0; g < ngroups; g += 2) {
    group(IC<0>{}, g);
    if (g + 1 < ngroups) group(IC<1>{}, g + 1);
  }
  if (jl % C2_R != 0) finish_block(jl / C2_R, bxmn, bxmx, bymn, bymx);     // the array's last, partial block
  if (TEST) {
    // cold path: per-cube refinement of the blocks whose cell union failed (rows re-read through L2)
    for (int b = 0; b < 64; b++) {
      if (!__any_sync(0xffffffffu, (failbits >> b) != 0)) break;
      const unsigned fm = __ballot_sync(0xffffffffu, (failbits >> b) & 1ull);
      if (fm) cells2d_slow_cubes(p, fm, c0, (kb0 + b) * C2_R, NPREV + 1, wl_stage);
    }
    flush_survivors(p, wl_stage);
  }
  return K2Acc{lds64_f64(res_u32), lds64_f64(res_u32 + 8u), big};
}

// One CTA per (tile of C2_CW strips, chunk of p.rows corner rows); K2_CTAS CTAs per SM.
template <int NPREV, bool TEST>
__global__ void __launch_bounds__((C2_CW + 1) * 32, K2_CTAS) scan2d_keys_build_kernel(const __grid_constant__ SweepParams p) {
  extern __shared__ __align__(128) unsigned char fb_smem[];
  const int lane = threadIdx.x & 31;
  const int wib = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);     // warp-uniform by construction
  const uint32_t ring0 = smem_u32(fb_smem);
  const uint32_t full0 = ring0 + (uint32_t)K2_NST * K2_STAGE_BYTES, empty0 = full0 + 8u * K2_NST;
  const uint32_t res_u32 = empty0 + 8u * K2_NST + 16u * threadIdx.x;
  const uint32_t wl_stage = empty0 + 8u * K2_NST + 16u * (C2_CW + 1) * 32u + 32u + WL_STAGE_BYTES * (uint32_t)wib;
  const uint32_t cell_stage = empty0 + 8u * K2_NST + 16u * (C2_CW + 1) * 32u + 32u + WL_STAGE_BYTES * (uint32_t)C2_CW + 1024u * (uint32_t)wib + 16u * (uint32_t)lane;
  const int W = p.W, H = p.H;
  const int bx = blockIdx.x % p.nsx, cy = blockIdx.x / p.nsx;
  const int C0 = bx * (C2_CW * FB_STRIDE);
  const int nactive = min(C2_CW, (W - C0 + FB_STRIDE - 1) / FB_STRIDE);     // consumer warps whose strip starts inside the array
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < K2_NST; q++) { mbar_init(full0 + 8u * q, 1); mbar_init(empty0 + 8u * q, (uint32_t)nactive); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  const int r0 = cy * p.rows;                        // p.rows is a multiple of C2_R, at most 64 blocks (one fail bit each)
  const int r1 = min(r0 + p.rows - 1, H - 1);
  const int nstages = ((r1 + 1) - r0 + 1 + 2 + K2_R - 1) / K2_R;
  if (wib == C2_CW) {
    // producer: one elected lane walks the rows with the array's index clamp and keeps the ring full; a stage always gets
    // K2_R rows (rows past the chunk's last one repeat the clamp: valid data, never used)
    if (elect_one()) {
      const double *S = p.L[p.build_layer].S;
      const int col_lo = max(C0 - 2, 0), col_hi = min(C0 - 2 + C2_SEG, W);
      const uint32_t seg_bytes = (uint32_t)(col_hi - col_lo) * 8u;
      const uint32_t dst0 = ring0 + (uint32_t)(col_lo - (C0 - 2)) * 8u;
      for (int s = 0; s < nstages; s++) {
        const uint32_t slot = (uint32_t)s % K2_NST;
        if (s >= K2_NST) mbar_wait(empty0 + 8u * slot, (uint32_t)((s / K2_NST - 1) & 1));
        mbar_expect_tx(full0 + 8u * slot, seg_bytes * K2_R);
#pragma unroll
        for (int i = 0; i < K2_R; i++) {
          const size_t off = (size_t)W * (size_t)clampi(r0 - 1 + K2_R * s + i, H) + (size_t)col_lo;
          bulk_g2s(dst0 + slot * K2_STAGE_BYTES + (uint32_t)i * K2_ROW_BYTES, S + off, seg_bytes, full0 + 8u * slot);
        }
      }
    }
    return;
  }
  if (wib >= nactive) return;
  const int c0 = C0 + wib * FB_STRIDE;
  const uint32_t tile_u32 = ring0 + (uint32_t)(wib * FB_STRIDE) * 8u;
  const bool border = c0 == 0 || c0 + FB_SEG - 2 > W;      // strips that touch the array's left / right edge clamp their columns
  K2Acc acc{DBL_MAX, DBL_MAX, 0.f};                   // exact min non-zero |d| per component; scaled by (W-1), (H-1) at the end:
                                                      // v = fl(d c) is monotone in |d|, so min |v| = fl(min |d| c) (grad.hh:24-27)
  sts64_f64(res_u32, DBL_MAX); sts64_f64(res_u32 + 8u, DBL_MAX);
  if (lane == 0) asm volatile("st.shared.s32 [%0], %1;" ::"r"(wl_stage), "r"(0) : "memory");
  __syncwarp();
  if (border) acc = keys2d_strip<true, NPREV, TEST>(p, c0, r0, r1, lane, tile_u32, full0, empty0, bx * C2_CW + wib, 0u, res_u32, wl_stage, cell_stage, acc);
  else acc = keys2d_strip<false, NPREV, TEST>(p, c0, r0, r1, lane, tile_u32, full0, empty0, bx * C2_CW + wib, 0u, res_u32, wl_stage, cell_stage, acc);
  if (p.res_slot[p.build_layer] != nullptr) {
    const double cw = (double)(W - 1), ch = (double)(H - 1);
    const double ax = fabs(acc.mdx), ay = fabs(acc.mdy);
    const double vx = ax < DBL_MAX ? ax * cw : DBL_MAX, vy = ay < DBL_MAX ? ay * ch : DBL_MAX;      // W - 1, H - 1 >= 1: no underflow to zero
    warp_res_commit(fmin(vx > 0.0 ? vx : DBL_MAX, vy > 0.0 ? vy : DBL_MAX), p.res_slot[p.build_layer]);
  }
  if (!(acc.big < __int_as_float(KEYF_BIG))) atomicExch(p.poison, 1ull);
}

static size_t k2_smem_bytes() { return (size_t)K2_NST * K2_STAGE_BYTES + (size_t)2 * K2_NST * 8 + (size_t)16 * (C2_CW + 1) * 32 + 32 + (size_t)WL_STAGE_BYTES * C2_CW + (size_t)1024 * C2_CW; }
static size_t c2_smem_bytes() { return (size_t)C2_NST * C2_SEG * 8 + (size_t)2 * C2_NST * 8; }

size_t scan2d_cells_per_layer(const SweepParams &p) {
  return (size_t)p.nsx * C2_CW * (size_t)(p.H / C2_R + 2) * 32u;
}

void launch_scan2d_cells(const SweepParams &p, cudaStream_t s) {
  const unsigned grid = (unsigned)((i64)p.nsx * p.nsy);
  const int nstrips = (p.W + FB_STRIDE - 1) / FB_STRIDE, nblk = (p.H + C2_R - 1) / C2_R;
  const unsigned tgrid = (unsigned)(((i64)nstrips * nblk + 7) / 8);
  if (p.keys2d && p.sum_mode <= SUM_BUILD_TEST2) {
    switch (p.sum_mode) {
      case SUM_BUILD: scan2d_keys_build_kernel<0, false><<<grid, (C2_CW + 1) * 32, k2_smem_bytes(), s>>>(p); break;
      case SUM_BUILD_TEST1: scan2d_keys_build_kernel<0, true><<<grid, (C2_CW + 1) * 32, k2_smem_bytes(), s>>>(p); break;
      default: scan2d_keys_build_kernel<1, true><<<grid, (C2_CW + 1) * 32, k2_smem_bytes(), s>>>(p); break;
    }
    return;
  }
  switch (p.sum_mode) {
    case SUM_BUILD: scan2d_build_kernel<0, false><<<grid, (C2_CW + 1) * 32, c2_smem_bytes(), s>>>(p); break;
    case SUM_BUILD_TEST1: scan2d_build_kernel<0, true><<<grid, (C2_CW + 1) * 32, c2_smem_bytes(), s>>>(p); break;
    case SUM_BUILD_TEST2: scan2d_build_kernel<1, true><<<grid, (C2_CW + 1) * 32, c2_smem_bytes(), s>>>(p); break;
    case SUM_TEST1: scan2d_cells_kernel<1><<<tgrid, 256, 0, s>>>(p, nstrips, nblk); break;
    default: scan2d_cells_kernel<2><<<tgrid, 256, 0, s>>>(p, nstrips, nblk); break;
  }
}

// ---- 3D, scalar input: gradient (grad.hh:130-149) folded into per-layer range cells, planes staged by TMA --------
// The vector field is never materialised.  gradient3D is 1/2 (S[+1] - S[-1]) on the array interior and zero on its
// border, so the quantised value trunc(v 2^nbits) is trunc(d 2^(nbits-1)) with d the plain difference: scaling by a
// power of two is exact, and the HIGH WORD of the fp64 difference, reinterpreted as an fp32 bit pattern, is a monotone
// key of d (sign-magnitude order; truncated towards zero).  The kernels therefore keep min/max of those keys with
// FMNMX -- no conversion instruction at all -- and "every vertex >= 1 after quantisation" is the exact comparison
// key >= key(2^(1-nbits)) because the threshold is a power of two.  NaN keys are the neutral element (FMNMX drops
// NaN); real NaN / Inf / >= 2^1000 scalars raise p.poison instead and the host repeats the sweep with the gradient
// materialised (scan3d_kernel).
//
// Determinant guard, exponent form: with e_c the biased exponent of max |d_c| (at least that of 2^-nbits),
// |quantised v_c| < 2^(e_c - 1023 + nbits) and M_c := |quantised| + 1 <= 2^(e_c - 1022 + nbits).  Every determinant of
// the cascade is at most 48 Mx My Mz (cube_excluded3 with R <= 2 M) < 2^(6 + sum(e_c) - 3066 + 3 nbits), which stays
// below 2^59 for sum(e_c) <= 3119 - 3 nbits: three binades under 2^62, four under the int64 range.
constexpr int F3_LAYER_BYTES = ((F3_ROWS * F3_COLS * 8 + 127) / 128) * 128;   // one staged plane of one layer
constexpr uint32_t F3_BOX_BYTES = F3_ROWS * F3_COLS * 8;

// cold path: for every lane whose union failed (bit set in failmask), the WARP tests that lane's 2 x F3_RW cubes of
// plane z: four lanes per cube, two vertices each (ranges over the vertices valid simplices can use, <= ub, read from
// global memory with the same key logic as the vector-layer scan), combined by shuffles; survivors are appended.
// Warp-wide so that a failing lane costs a couple of memory round trips instead of several hundred serialised loads.
__device__ __noinline__ void fused3d_slow_cubes(const SweepParams &p, unsigned failmask, const int C0, const int y0, const int z, const int nl) {
  static_assert(2 * F3_RW * 4 == 32, "four lanes per cube");
  const int lane = threadIdx.x & 31;
  const bool vec = !p.fused;                          // vector input: the keys are the vertices' own components
  const int nbits20 = (p.nbits - (vec ? 0 : 1)) << 20;
  const size_t sy = (size_t)p.W, sz = (size_t)p.W * (size_t)p.H;
  const int cube = lane >> 2, sub = lane & 3;
  const int r = cube >> 1, q = cube & 1;
  while (failmask) {
    const int src = __ffs(failmask) - 1;
    failmask &= failmask - 1;
    const int x = C0 + 2 * src + q, y = y0 + r;
    const bool in = x >= p.lb[0] && x <= p.ub[0] && y >= p.lb[1] && y <= p.ub[1];
    KeyRange rg[3] = {neutral_range(), neutral_range(), neutral_range()};
#pragma unroll
    for (int vv = 0; vv < 2; vv++) {
      const int v = 2 * sub + vv;
      const int vx = x + (v & 1), vy = y + ((v >> 1) & 1), vz = z + (v >> 2);
      if (!in || vx > p.ub[0] || vy > p.ub[1] || vz > p.ub[2]) continue;
      const bool border = vx < 1 || vx > p.W - 2 || vy < 1 || vy > p.H - 2 || vz < 1 || vz > p.D - 2;
      const size_t idx = (size_t)vx + sy * (size_t)vy + sz * (size_t)vz;
      for (int L = 0; L < nl; L++) {
        const double *S = p.L[L].S;
        int h0 = 0, h1 = 0, h2 = 0;
        if (vec) {
          const int *Vh = reinterpret_cast<const int *>(p.L[L].V) + idx * 6 + 1;
          h0 = __ldg(Vh); h1 = __ldg(Vh + 2); h2 = __ldg(Vh + 4);
        } else if (!border) {
          h0 = __double2hiint(__ldg(S + idx + 1) - __ldg(S + idx - 1));
          h1 = __double2hiint(__ldg(S + idx + sy) - __ldg(S + idx - sy));
          h2 = __double2hiint(__ldg(S + idx + sz) - __ldg(S + idx - sz));
        }
        rg[0] = merge(rg[0], vertex_range(h0, nbits20));
        rg[1] = merge(rg[1], vertex_range(h1, nbits20));
        rg[2] = merge(rg[2], vertex_range(h2, nbits20));
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int off = 1; off <= 2; off <<= 1) {
        rg[c].mn = min(rg[c].mn, __shfl_xor_sync(0xffffffffu, rg[c].mn, off));
        rg[c].mx = max(rg[c].mx, __shfl_xor_sync(0xffffffffu, rg[c].mx, off));
      }
    const bool surv = in && sub == 0 && !cube_excluded3(rg[0], rg[1], rg[2]);
    append_survivors(p, surv, (u64)(x - p.lb[0]) + (u64)p.nc[0] * ((u64)(y - p.lb[1]) + (u64)p.nc[1] * (u64)(z - p.lb[2])));
  }
}

// exact path of the running min non-zero |v| (v = d / 2): m keeps the signed value of smallest magnitude
__device__ __forceinline__ void res_update3(double &m, const bool in, const double dx, const double dy, const double dz) {
  if (!in) return;
  const double vx = 0.5 * dx, vy = 0.5 * dy, vz = 0.5 * dz;
  if (vx != 0.0 && fabs(vx) < fabs(m)) m = vx;      // NaN / Inf never compare below
  if (vy != 0.0 && fabs(vy) < fabs(m)) m = vy;
  if (vz != 0.0 && fabs(vz) < fabs(m)) m = vz;
}

// ---- 3D, scalar input, per-layer range summaries ("build once, test from summaries") -----------------------
// A CTA of eight warps owns a tile of F3_STRIDE x F3_TROWS corner columns and marches along z over a chunk of
// planes; a thread covers 2 columns x S3_RW corner rows.  The per-thread unions of gradient keys depend on ONE
// layer only (raw keys of the gradient, domain masks), not on the quantisation factor.  A layer is therefore
// streamed from HBM once in its life: the step that first sees it (as the "next" layer) derives its gradient
// keys, folds min non-zero |v|, and stores each thread's union (after the x-neighbour merge) as a 16-byte cell
// -- six keys truncated to their upper 16 bits (sign, 11 exponent bits, 4 mantissa bits).  The exclusion test
// only compares keys against powers of two and sums exponents, so truncation towards zero changes none of its
// decisions.  The same step reads the CURRENT layer's cells (written one step earlier) instead of the layer
// itself: 8 B/vertex of scalars + 2 B/vertex of cells written + 2 B/vertex read, against 16 B/vertex for a scan
// that re-reads both layers, and half the arithmetic.  Re-sweeps (a stale speculated factor, worklist growth)
// and the final ordinal-only sweep read cells only.
//
// Staging: a ring of S3_NST planes of the layer being built, one TMA box (tile + halo, out-of-bounds elements
// zero-filled) per plane and stage; no producer warp (see S3Build::release).  Each consumer thread keeps a
// three-plane register window of its 2 columns x (S3_RW + 3) rows, so a plane is read from shared memory once
// (plus the two x-neighbour columns while it is the centre plane).
constexpr int S3_RW = F3_RW;                       // corner rows per consumer warp
constexpr int S3_WR = S3_RW + 1;                   // window rows per plane: the gradient rows y0 .. y0+RW (the two halo rows of the
                                                   // centre plane are re-read from shared memory while it is the centre)
constexpr int S3_NST = 5;                          // ring stages (planes)
constexpr int S3_STAGE_BYTES = F3_LAYER_BYTES;

__device__ __forceinline__ uint32_t pack_keys(float mn, float mx) {
  return __byte_perm((uint32_t)__float_as_int(mn), (uint32_t)__float_as_int(mx), 0x7632);
}
__device__ __forceinline__ void merge_cell(float (&mn)[3], float (&mx)[3], const uint4 w) {
  mn[0] = fminf(mn[0], __int_as_float((int)(w.x << 16))); mx[0] = fmaxf(mx[0], __int_as_float((int)(w.x & 0xffff0000u)));
  mn[1] = fminf(mn[1], __int_as_float((int)(w.y << 16))); mx[1] = fmaxf(mx[1], __int_as_float((int)(w.y & 0xffff0000u)));
  mn[2] = fminf(mn[2], __int_as_float((int)(w.z << 16))); mx[2] = fmaxf(mx[2], __int_as_float((int)(w.z & 0xffff0000u)));
}

struct S3Thresholds { float kthr, kfloor; int esum_max, nbits20; double half_factor; };
// vec = false: keys of d = 2 v (gradient differences of a scalar layer); vec = true: keys of v itself (vector input), i.e.
// every threshold one binade lower and every magnitude bound one bit larger
__device__ __forceinline__ S3Thresholds s3_thresholds(const int nbits, const bool vec) {
  const int s = vec ? 1 : 0;
  S3Thresholds t;
  t.kthr = __int_as_float((1023 + 1 - s - nbits) << 20);   // key of 2^(1-nbits) (d) / 2^-nbits (v): at or above it |quantised v| >= 1
  t.kfloor = __int_as_float((1023 - s - nbits) << 20);     // half of that: smaller magnitudes quantise to 0
  t.esum_max = 3119 - 3 * s - 3 * nbits;                    // determinant guard, see the 3D section header
  t.nbits20 = (nbits - 1 + s) << 20;
  t.half_factor = __hiloint2double((1023 + nbits - 1 + s) << 20, 0);   // v 2^nbits = d 2^(nbits-1)
  return t;
}

// third level of the determinant guard (rare): the range form of cube_excluded3.  Keys may have lost their low 16
// bits (cells are stored truncated towards zero), so bounds that truncation moved inwards are pushed back out.
__device__ __noinline__ bool s3_union_excluded_precise(const float mn0, const float mx0, const float mn1, const float mx1,
                                                       const float mn2, const float mx2, const int nbits20) {
  const auto lo = [](float f) { const int k = __float_as_int(f); return k < 0 ? (k | 0xFFFF) : k; };
  const auto hi = [](float f) { const int k = __float_as_int(f); return k < 0 ? k : (k | 0xFFFF); };
  // merged, not {lo.mn, hi.mx}: a poisoned upper end (|p| >= 2^63) must poison the range's mn, which the guards test
  const KeyRange x = merge(vertex_range(lo(mn0), nbits20), vertex_range(hi(mx0), nbits20));
  const KeyRange y = merge(vertex_range(lo(mn1), nbits20), vertex_range(hi(mx1), nbits20));
  const KeyRange z = merge(vertex_range(lo(mn2), nbits20), vertex_range(hi(mx2), nbits20));
  return cube_excluded3(x, y, z);
}

// exponent-level part of s3_test: true = every cube of the block is excluded (see s3_test for the bound)
__device__ __forceinline__ bool s3_excluded_level1(const S3Thresholds &T, const float (&cmn)[3], const float (&cmx)[3]) {
  bool sided = false;
  int esum = 0;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    sided = sided || cmn[c] >= T.kthr || cmx[c] <= -T.kthr;
    esum += (__float_as_int(fmaxf(fmaxf(fabsf(cmn[c]), fabsf(cmx[c])), T.kfloor)) >> 20);
  }
  return sided && esum <= T.esum_max && !(cmn[0] != cmn[0]);
}

// levels 2 and 3 of the determinant guard for a union that is one-sided in some component but failed the exponent-level bound
// (large magnitudes: on a 512^3 moving extremum at factor 2^21 that is every sixth block).  A function of its own, entered behind a
// warp vote, so that the plane loop pays a call only where it is needed and the blocks it clears never reach the retest after the loop.
__device__ __noinline__ bool s3_excluded_levels23(const float mn0, const float mx0, const float mn1, const float mx1, const float mn2, const float mx2,
                                                  const double half_factor, const int nbits20) {
  const float mag[3] = {fmaxf(fabsf(mn0), fabsf(mx0)), fmaxf(fabsf(mn1), fabsf(mx1)), fmaxf(fabsf(mn2), fabsf(mx2))};
  double P = 48.0;
#pragma unroll
  for (int c = 0; c < 3; c++) P *= fma(__hiloint2double((__float_as_int(mag[c]) | 0xFFFF) + 1, 0), half_factor, 1.0);
  if (P < 9.0e18) return true;           // Inf / NaN magnitudes compare false
  return s3_union_excluded_precise(mn0, mx0, mn1, mx1, mn2, mx2, nbits20);
}

// decide corner plane zc of this lane's 2 x S3_RW cubes from the union of the cells of planes zc, zc+1 (all layers)
__device__ __forceinline__ void s3_test(const SweepParams &p, const S3Thresholds &T, const float (&cmn)[3], const float (&cmx)[3],
                                        const bool own_any, const int e, const int y0, const int zc, const int nl) {
  bool sided = false;
  int esum = 0;
  float mag[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    sided = sided || cmn[c] >= T.kthr || cmx[c] <= -T.kthr;
    mag[c] = fmaxf(fabsf(cmn[c]), fabsf(cmx[c]));
    esum += (__float_as_int(fmaxf(mag[c], T.kfloor)) >> 20);
  }
  // determinant guard, level 1 (exponents only, see the 3D section header).  A NaN union (no vertex) fails every level and
  // takes the cold path, which is exact.
  bool excl = sided && esum <= T.esum_max && !(cmn[0] != cmn[0]);
  if (sided && !excl && own_any && !(cmn[0] != cmn[0])) {
    // level 2: M_c = |quantised v_c| + 1 <= D_c 2^(nbits-1) + 1 with D_c the next key above max |d_c| (also above every
    // value a truncated key stands for); every determinant of the cascade is at most 48 Mx My Mz (cube_excluded3, R <= 2 M)
    double P = 48.0;
#pragma unroll
    for (int c = 0; c < 3; c++) P *= fma(__hiloint2double((__float_as_int(mag[c]) | 0xFFFF) + 1, 0), T.half_factor, 1.0);
    excl = P < 9.0e18;           // Inf / NaN magnitudes compare false
    if (!excl) excl = s3_union_excluded_precise(cmn[0], cmx[0], cmn[1], cmx[1], cmn[2], cmx[2], T.nbits20);
  }
  const bool fail = own_any && !excl;
  const unsigned fm = __ballot_sync(0xffffffffu, fail);
  if (fm) fused3d_slow_cubes(p, fm, e - 2 * (int)(threadIdx.x & 31), y0, zc, nl);
}

__device__ __forceinline__ size_t s3_cell_index(const SweepParams &p, const int tile, const int wib, const int z, const int lane) {
  return (((size_t)tile * F3_CW + (size_t)wib) * (size_t)(p.D + 1) + (size_t)z) * 32u + (size_t)lane;
}

// cold path of the build kernels: corner plane zc of one warp's blocks, decided from the cells in memory (those of the layer
// being built were written by these very threads: plain loads; the other layer's cells are read-only here)
__device__ __noinline__ void s3_retest_plane(const SweepParams &p, const uint4 *built, const uint4 *other, const bool fail, const bool vec,
                                             const int e, const int y0, const int zc, const int zc0) {
  if (!__any_sync(0xffffffffu, fail)) return;
  const S3Thresholds T = s3_thresholds(p.nbits, vec);
  const float nanf_ = __int_as_float(KEYF_NAN);
  float cmn[3] = {nanf_, nanf_, nanf_}, cmx[3] = {nanf_, nanf_, nanf_};
#pragma unroll
  for (int dz = 0; dz < 2; dz++) {
    merge_cell(cmn, cmx, built[(size_t)(zc - zc0 + dz) * 32u]);
    if (other) merge_cell(cmn, cmx, __ldg(other + (size_t)(zc - zc0 + dz) * 32u));
  }
  s3_test(p, T, cmn, cmx, fail, e, y0, zc, other ? 2 : 1);
}

// exact (cold) part of the running min non-zero |v|: entered only when a key of this row undercuts the best so far
__device__ __noinline__ double s3_res_row(double rmin, const bool in_e, const bool in_o, const double dxe, const double dye,
                                          const double dze, const double dxo, const double dyo, const double dzo) {
  res_update3(rmin, in_e, dxe, dye, dze);
  res_update3(rmin, in_o, dxo, dyo, dzo);
  return rmin;
}

__device__ __forceinline__ double lds_f64(const uint32_t a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ double2 lds_f64x2(const uint32_t a) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
  return v;
}

// one plane step of the build: zm / zc / zp are the register windows of planes zg-1, zg, zg+1 (zp is loaded here)
//
// EDGE tiles (they touch the array border or leave the tracker's domain): vertices outside the domain stay out of
// the ranges (NaN key, the neutral element of FMNMX); a thread whose block holds in-domain vertices ON the array
// border, where gradient3D is zero (grad.hh:130-149), adds 0 to its ranges (whatever the stencil computed there from
// the zero-filled halo only widens them further: still a superset); border vertices stay out of min |v|.
template <bool EDGE, int NPREV, bool TEST>
struct S3Build {
  const SweepParams &p;
  uint32_t ring;             // shared-memory address of the ring
  uint32_t full0;
  uint32_t cnt;              // shared-memory address of the per-stage release counters
  const CUtensorMap *tm;
  int C0, Y0, nplanes;
  int lane, e, y0, zc0;
  uint32_t lane_off;         // byte offset of this thread's first window element within a stage
  int sidx;                  // index of the centre plane within this CTA's chunk (plane zc0-1 is 0)
  S3Thresholds T;
  bool want_res, bad, own_any, touches;
  // EDGE: bit r (+0 / +8): gradient row r of column e / e+1 lies in the array interior; bit r (+16 / +24): in the domain
  unsigned masks;
  double rmin, r2;           // signed value of smallest magnitude so far; 2 |rmin| (the differences are 2 v)
  float rkey;                // high word of r2
  double r2cap;              // what r2 / rkey start from: just above twice the running minimum of the earlier layers, or +inf
  float kcap;
  uint32_t pcell[3];         // previous plane's merged cell (packed like a stored cell)
  int st_c, st_p;
  uint32_t par_p;
  unsigned long long failbits;   // bit (zc - zc0): corner plane zc of this lane's block failed the exponent-level test (decided after the loop)
  uint32_t cellring;         // shared memory: this lane's four 16-byte slots (512 bytes apart) for the other layer's cells
  int zlast;                 // last plane of the chunk's loop (zc1 + 1)
  const uint4 *sum_prev;     // cells of the current layer at the plane being processed (this warp, this lane)
  uint4 *sum_out;            // cells of the layer being built, likewise

  __device__ __forceinline__ void load_plane(double2 (&P)[S3_WR], const int st) const {
    const uint32_t base = ring + (uint32_t)st * S3_STAGE_BYTES + lane_off + (uint32_t)(F3_COLS * 8) + 16u;
#pragma unroll
    for (int r = 0; r < S3_WR; r++) P[r] = lds_f64x2(base + (uint32_t)(r * F3_COLS * 8));
  }
  // Release the stage of plane `sx`.  There is no producer warp: the LAST consumer warp to release a stage
  // (a monotone shared-memory counter per stage) issues the TMA load of plane sx + S3_NST into it, so nobody
  // ever waits for a stage to drain.
  __device__ __forceinline__ void release(const int st, const int sx) const {
    __syncwarp();
    if (lane == 0) {
      unsigned old;
      asm volatile("atom.acq_rel.cta.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(cnt + 4u * (uint32_t)st) : "memory");
      if ((old + 1u) % F3_CW == 0u && sx + S3_NST < nplanes) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(full0 + 8u * st, F3_BOX_BYTES);
        tma_load_3d(ring + (uint32_t)st * S3_STAGE_BYTES, tm, C0 - 2, Y0 - 1, zc0 - 1 + sx + S3_NST, full0 + 8u * st);
      }
    }
  }
  __device__ __forceinline__ void advance_stage() {
    st_c = st_p;
    st_p = st_p + 1 == S3_NST ? 0 : st_p + 1;
    if (st_p == 0) par_p ^= 1u;
  }

  __device__ __forceinline__ void step(const double2 (&zm)[S3_WR], const double2 (&zc)[S3_WR], double2 (&zp)[S3_WR], const int zg) {
    const float nanf_ = __int_as_float(KEYF_NAN);
    const float inff_ = __int_as_float(0x7F800000);
    // the other layer's cells travel through a small shared-memory ring filled by cp.async three planes ahead (no register holds
    // a cell in flight: as a 128-bit load one plane ahead it was still waited for -- 16 % of the warp samples -- because an L2 hit
    // takes longer than a plane step while the TMA ring saturates the memory system); one commit group per plane
    if (NPREV) {
      if (zg + 3 <= zlast) cp_async16(cellring + (((uint32_t)zg + 3u) & 3u) * 512u, sum_prev + 3 * 32);
      cp_async_commit();
      if (zg + 5 <= p.D) prefetch_l2(sum_prev + 5 * 32);      // a DRAM miss each, requested into L2 five planes ahead
    }
    mbar_wait(full0 + 8u * st_p, par_p);
    load_plane(zp, st_p);
    const uint32_t cen = ring + (uint32_t)st_c * S3_STAGE_BYTES + lane_off + (uint32_t)(F3_COLS * 8);
    const bool zarr = zg >= 1 && zg <= p.D - 2;
    const bool zdom = zg >= p.lb[2] && zg <= p.ub[2];
    const bool res_now = want_res && zarr;
    const double2 top = lds_f64x2(cen - (uint32_t)(F3_COLS * 8) + 16u), bot = lds_f64x2(cen + (uint32_t)((S3_RW + 1) * F3_COLS * 8) + 16u);
    float umin[3] = {nanf_, nanf_, nanf_}, umax[3] = {nanf_, nanf_, nanf_};
    int big = 0;
    unsigned mk = masks;
    if (EDGE) asm volatile("" : "+r"(mk));       // keep the per-row tests as single bit tests of one register
#pragma unroll
    for (int r = 0; r <= S3_RW; r++) {
      const double left = lds_f64(cen + (uint32_t)(r * F3_COLS * 8 + 8)), right = lds_f64(cen + (uint32_t)(r * F3_COLS * 8 + 32));
      const double2 rc = zc[r];
      const double2 up = r == S3_RW ? bot : zc[r == S3_RW ? r : r + 1], dn = r == 0 ? top : zc[r == 0 ? r : r - 1];
      const double dxe = rc.y - left, dxo = right - rc.x;
      const double dye = up.x - dn.x, dyo = up.y - dn.y;
      const double dze = zp[r].x - zm[r].x, dzo = zp[r].y - zm[r].y;
      float kxe = hikey(dxe), kxo = hikey(dxo), kye = hikey(dye), kyo = hikey(dyo), kze = hikey(dze), kzo = hikey(dzo);
      big = max(big, max(__double2hiint(rc.x) & 0x7fffffff, __double2hiint(rc.y) & 0x7fffffff));   // NaN / Inf patterns compare high
      if (res_now) {
        float a = fminf(fminf(fabsf(kxe), fabsf(kye)), fabsf(kze)), b = fminf(fminf(fabsf(kxo), fabsf(kyo)), fabsf(kzo));
        bool in_e = true, in_o = true;
        if (EDGE) {
          in_e = (mk >> r) & 1u; in_o = (mk >> (r + 8)) & 1u;
          a = in_e ? a : inff_; b = in_o ? b : inff_;
        }
        const float m = fminf(a, b);
        if (m <= rkey) {
          // a high word below the best so far, or a tie on the high word that a low word may break
          bool go = m < rkey;
          // (no key of this row is below rkey here, so none of the six values is zero)
          if (!go) go = fabs(dxe) < r2 || fabs(dye) < r2 || fabs(dze) < r2 || fabs(dxo) < r2 || fabs(dyo) < r2 || fabs(dzo) < r2;
          if (go) {
            res_update3(rmin, in_e, dxe, dye, dze);       // inline: a call here would cost the plane loop its registers
            res_update3(rmin, in_o, dxo, dyo, dzo);
            // nothing found yet: back to the cap -- the running minimum known when the step was enqueued (SweepParams::res_thr;
            // +inf accepts every key)
            const double n2 = 2.0 * fabs(rmin);
            const bool capped = !(n2 < r2cap);
            r2 = capped ? r2cap : n2;
            rkey = capped ? kcap : hikey(n2);
          }
        }
      }
      if (EDGE) {
        const bool de = (mk >> (r + 16)) & 1u, dq = (mk >> (r + 24)) & 1u;
        kxe = de ? kxe : nanf_; kye = de ? kye : nanf_; kze = de ? kze : nanf_;
        kxo = dq ? kxo : nanf_; kyo = dq ? kyo : nanf_; kzo = dq ? kzo : nanf_;
      }
      umin[0] = fminf(umin[0], fminf(kxe, kxo)); umax[0] = fmaxf(umax[0], fmaxf(kxe, kxo));
      umin[1] = fminf(umin[1], fminf(kye, kyo)); umax[1] = fmaxf(umax[1], fmaxf(kye, kyo));
      umin[2] = fminf(umin[2], fminf(kze, kzo)); umax[2] = fmaxf(umax[2], fmaxf(kze, kzo));
    }
    bad = bad || big >= KEYF_BIG;
    release(st_c, sidx);                    // the centre plane's x neighbours were the last shared-memory reads of plane zg
    sidx++;
    if (EDGE && touches) {
#pragma unroll
      for (int c = 0; c < 3; c++) { umin[c] = fminf(umin[c], 0.f); umax[c] = fmaxf(umax[c], 0.f); }
    }
    // plane-level masks (warp-uniform): planes outside the domain stay out of the ranges; the array's first and
    // last plane have a zero gradient
    if (!zdom || !zarr) {
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const bool has = zdom && !(umin[c] != umin[c]);     // lanes with no in-domain vertex keep the neutral element
        umin[c] = has ? 0.f : nanf_; umax[c] = has ? 0.f : nanf_;
      }
    }
    // x neighbour: corner column e+1 also uses the next lane's first column
#pragma unroll
    for (int c = 0; c < 3; c++) {
      umin[c] = fminf(umin[c], __shfl_down_sync(0xffffffffu, umin[c], 1));
      umax[c] = fmaxf(umax[c], __shfl_down_sync(0xffffffffu, umax[c], 1));
    }
    *sum_out = make_uint4(pack_keys(umin[0], umax[0]), pack_keys(umin[1], umax[1]), pack_keys(umin[2], umax[2]), 0u);
    sum_out += 32;
    if (NPREV) sum_prev += 32;
    if (TEST) {
      if (NPREV) {
        cp_async_wait_group<3>();               // everything but the three newest groups: this plane's cell has landed
        merge_cell(umin, umax, lds128_u32(cellring + ((uint32_t)zg & 3u) * 512u));
      }
      if (zg > zc0) {
        const int zc_ = zg - 1;                   // corner plane decided now (warp-uniform)
        if (zc_ >= p.lb[2] && zc_ <= p.ub[2]) {
          float cmn[3] = {umin[0], umin[1], umin[2]}, cmx[3] = {umax[0], umax[1], umax[2]};
          merge_cell(cmn, cmx, make_uint4(pcell[0], pcell[1], pcell[2], 0u));
          // the exponent-level test runs here; a union it cannot exclude although some component is one-sided goes through
          // the magnitude / range bounds behind a vote (s3_excluded_levels23); what is still open is noted (one bit per corner
          // plane of the chunk) and decided after the plane loop from the stored cells
          bool open_ = own_any && !s3_excluded_level1(T, cmn, cmx);
          bool sided = false;
#pragma unroll
          for (int c = 0; c < 3; c++) sided = sided || cmn[c] >= T.kthr || cmx[c] <= -T.kthr;
          const bool try23 = open_ && sided && !(cmn[0] != cmn[0]);
          if (__any_sync(0xffffffffu, try23)) {
            if (try23 && s3_excluded_levels23(cmn[0], cmx[0], cmn[1], cmx[1], cmn[2], cmx[2], T.half_factor, T.nbits20)) open_ = false;
          }
          if (open_) failbits |= 1ull << (zc_ - zc0);
        }
      }
#pragma unroll
      for (int c = 0; c < 3; c++) pcell[c] = pack_keys(umin[c], umax[c]);
    }
    advance_stage();
  }
};

template <bool EDGE, int NPREV, bool TEST>
__device__ __forceinline__ void s3_consume(const SweepParams &p, const uint32_t ring, const uint32_t full0, const uint32_t cnt, const uint32_t cellring,
                                           const int tile, const int C0, const int Y0, const int zc0, const int zc1, const int wib, const int lane) {
  const int B = p.build_layer;
  S3Build<EDGE, NPREV, TEST> s{p, ring, full0, cnt};
  s.tm = &p.tmap[B];
  s.C0 = C0; s.Y0 = Y0; s.nplanes = zc1 - zc0 + 4;
  s.lane = lane;
  s.e = C0 + 2 * lane;
  s.y0 = Y0 + wib * S3_RW;
  s.lane_off = (uint32_t)((wib * S3_RW * F3_COLS + 2 * lane) * 8);
  s.zc0 = zc0;
  s.T = s3_thresholds(p.nbits, false);
  s.want_res = p.res_slot[B] != nullptr;
  s.bad = false;
  s.own_any = lane <= 30;
  s.touches = false;
  s.masks = 0xffffffffu;
  if (EDGE) {
    const bool arr_c0 = s.e >= 1 && s.e <= p.W - 2, arr_c1 = s.e + 1 >= 1 && s.e + 1 <= p.W - 2;
    const bool dom_c0 = s.e >= p.lb[0] && s.e <= p.ub[0], dom_c1 = s.e + 1 >= p.lb[0] && s.e + 1 <= p.ub[0];
    s.own_any = s.own_any && (dom_c0 || dom_c1) && s.y0 <= p.ub[1] && s.y0 + S3_RW - 1 >= p.lb[1];
    unsigned rows = 0, rows_dom = 0;
#pragma unroll
    for (int r = 0; r <= S3_RW; r++) {
      rows |= (s.y0 + r >= 1 && s.y0 + r <= p.H - 2) ? (1u << r) : 0u;
      rows_dom |= (s.y0 + r >= p.lb[1] && s.y0 + r <= p.ub[1]) ? (1u << r) : 0u;
    }
    const unsigned in_e = arr_c0 ? rows : 0u, in_o = arr_c1 ? rows : 0u, dom_e = dom_c0 ? rows_dom : 0u, dom_o = dom_c1 ? rows_dom : 0u;
    s.masks = in_e | (in_o << 8) | (dom_e << 16) | (dom_o << 24);
    // in-domain vertices of this thread's block that lie on the array border
    s.touches = ((dom_e & ~in_e) | (dom_o & ~in_o)) != 0u;
  }
  s.rmin = DBL_MAX;
  s.kcap = p.res_thr[0];
  s.r2cap = s.kcap < __int_as_float(0x7F800000) ? __hiloint2double(__float_as_int(s.kcap), 0) : __hiloint2double(0x7FF00000, 0);
  s.r2 = s.r2cap;
  s.rkey = s.kcap;
#pragma unroll
  for (int c = 0; c < 3; c++) s.pcell[c] = 0x7FC07FC0u;
  s.failbits = 0;
  const size_t cell0 = s3_cell_index(p, tile, wib, zc0, lane);
  s.sum_prev = NPREV ? p.sum_in[0] + cell0 : nullptr;
  s.sum_out = p.sum_out + cell0;
  if (NPREV) { prefetch_l2(s.sum_prev); prefetch_l2(s.sum_prev + 32); prefetch_l2(s.sum_prev + 64); }
  s.zlast = zc1 + 1;
  s.cellring = cellring + (uint32_t)wib * 2048u + (uint32_t)lane * 16u;
  if (NPREV) {
    // planes zc0 .. zc0 + 2 of the other layer's cells: three commit groups (a plane past the chunk's end commits an empty one)
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (zc0 + k <= s.zlast) cp_async16(s.cellring + (((uint32_t)zc0 + (uint32_t)k) & 3u) * 512u, s.sum_prev + k * 32);
      cp_async_commit();
    }
  }

  double2 A[S3_WR], Bw[S3_WR], Cw[S3_WR];
  mbar_wait(full0, 0);
  s.load_plane(A, 0);          // plane zc0-1: only ever the z-1 neighbour
  s.release(0, 0);
  mbar_wait(full0 + 8, 0);
  s.load_plane(Bw, 1);         // plane zc0: first centre plane
  s.st_c = 1; s.st_p = 2; s.par_p = 0; s.sidx = 1;
  const int zend = zc1 + 1;
  int zg = zc0;
  // ONE copy of the plane step; the three-plane register window rotates by moves (20 per plane).  Three unrolled steps with the
  // windows renamed (no moves) measured 2 % slower: the kernel is three times the code and 13 % of its warp samples were
  // instruction fetch.
  while (true) {
    s.step(A, Bw, Cw, zg); if (++zg > zend) break;
#pragma unroll
    for (int r = 0; r < S3_WR; r++) { A[r] = Bw[r]; Bw[r] = Cw[r]; }
  }
  if (s.want_res) warp_res_commit(fabs(s.rmin), p.res_slot[B]);
  if (s.bad) atomicExch(p.poison, 1ull);
  if (TEST) {
    // cold path: the corner planes whose cell union the exponent-level test could not exclude (a chunk has at most 64 planes)
    const unsigned long long fb = s.failbits;
    const int e = s.e, y0 = s.y0;
    for (int b = 0; b <= zc1 - zc0; b++) {
      if (!__any_sync(0xffffffffu, (fb >> b) != 0)) break;
      s3_retest_plane(p, p.sum_out + cell0, NPREV ? p.sum_in[0] + cell0 : nullptr, (fb >> b) & 1ull, false, e, y0, zc0 + b, zc0);
    }
  }
}

template <int NPREV, bool TEST>
__global__ void __launch_bounds__(F3_CW * 32, 2) scan3d_build_kernel(const __grid_constant__ SweepParams p) {
  extern __shared__ __align__(128) unsigned char fb_smem[];
  const int lane = threadIdx.x & 31;
  const int wib = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);     // warp-uniform by construction
  const uint32_t ring_u32 = smem_u32(fb_smem);
  const uint32_t full0 = ring_u32 + (uint32_t)S3_NST * S3_STAGE_BYTES;
  unsigned *cnt = reinterpret_cast<unsigned *>(fb_smem + (size_t)S3_NST * S3_STAGE_BYTES + 8u * S3_NST);
  const uint32_t cellring_u32 = (ring_u32 + (uint32_t)S3_NST * S3_STAGE_BYTES + 12u * S3_NST + 15u) & ~15u;     // 8 warps x 4 planes x 512 bytes
  int b = blockIdx.x;
  const int bx = b % p.nsx; b /= p.nsx;
  const int by = b % p.nsy;
  const int bz = b / p.nsy;
  const int C0 = bx * F3_STRIDE, Y0 = by * F3_TROWS;
  const int zc0 = bz * p.rows, zc1 = min(zc0 + p.rows - 1, p.D - 1);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < S3_NST; q++) { mbar_init(full0 + 8u * q, 1); cnt[q] = 0u; }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    // scalar planes zc0-1 .. zc1+2 of the layer being built, one TMA box (tile + halo) each: the first S3_NST here,
    // the rest by whichever warp drains a stage last
    const int nplanes = zc1 - zc0 + 4;
    for (int s = 0; s < min(S3_NST, nplanes); s++) {
      mbar_expect_tx(full0 + 8u * s, F3_BOX_BYTES);
      tma_load_3d(ring_u32 + (uint32_t)s * S3_STAGE_BYTES, &p.tmap[p.build_layer], C0 - 2, Y0 - 1, zc0 - 1 + s, full0 + 8u * s);
    }
  }
  __syncthreads();
  const int tile = by * p.nsx + bx;
  const bool interior = C0 >= max(1, p.lb[0]) && C0 + 63 <= min(p.W - 2, p.ub[0]) && Y0 >= max(1, p.lb[1]) && Y0 + F3_TROWS <= min(p.H - 2, p.ub[1]);
  if (interior) s3_consume<false, NPREV, TEST>(p, ring_u32, full0, smem_u32(cnt), cellring_u32, tile, C0, Y0, zc0, zc1, wib, lane);
  else s3_consume<true, NPREV, TEST>(p, ring_u32, full0, smem_u32(cnt), cellring_u32, tile, C0, Y0, zc0, zc1, wib, lane);
}

// cells only: the final ordinal sweep (one layer) and re-sweeps (both layers' cells exist)
template <int NL>
__global__ void __launch_bounds__(F3_CW * 32) scan3d_cells_kernel(const __grid_constant__ SweepParams p) {
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  int b = blockIdx.x;
  const int bx = b % p.nsx; b /= p.nsx;
  const int by = b % p.nsy;
  const int bz = b / p.nsy;
  const int C0 = bx * F3_STRIDE, Y0 = by * F3_TROWS;
  const int zc0 = bz * p.rows, zc1 = min(zc0 + p.rows - 1, p.D - 1);
  const int e = C0 + 2 * lane, y0 = Y0 + wib * S3_RW;
  const bool any_col = (e >= p.lb[0] && e <= p.ub[0]) || (e + 1 >= p.lb[0] && e + 1 <= p.ub[0]);
  const bool own_any = lane <= 30 && any_col && y0 <= p.ub[1] && y0 + S3_RW - 1 >= p.lb[1];
  if (!__any_sync(0xffffffffu, own_any)) return;
  const S3Thresholds T = s3_thresholds(p.nbits, !p.fused);
  const size_t cell0 = s3_cell_index(p, by * p.nsx + bx, wib, 0, lane);
  const float nanf_ = __int_as_float(KEYF_NAN);
  float pmn[3] = {nanf_, nanf_, nanf_}, pmx[3] = {nanf_, nanf_, nanf_};
  for (int zg = zc0; zg <= zc1 + 1; zg++) {
    float umn[3] = {nanf_, nanf_, nanf_}, umx[3] = {nanf_, nanf_, nanf_};
#pragma unroll
    for (int L = 0; L < NL; L++) merge_cell(umn, umx, __ldg(p.sum_in[L] + cell0 + (size_t)zg * 32u));
    if (zg > zc0) {
      const int zc_ = zg - 1;
      if (zc_ >= p.lb[2] && zc_ <= p.ub[2]) {
        float cmn[3], cmx[3];
#pragma unroll
        for (int c = 0; c < 3; c++) { cmn[c] = fminf(pmn[c], umn[c]); cmx[c] = fmaxf(pmx[c], umx[c]); }
        s3_test(p, T, cmn, cmx, own_any, e, y0, zc_, NL);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) { pmn[c] = umn[c]; pmx[c] = umx[c]; }
  }
}

static size_t s3_smem_bytes() { return (size_t)S3_NST * S3_STAGE_BYTES + (size_t)S3_NST * 8 + (size_t)S3_NST * 4 + 16 + (size_t)F3_CW * 2048; }

size_t scan3d_cells_per_layer(const SweepParams &p) { return (size_t)p.nsx * p.nsy * F3_CW * (size_t)(p.D + 1) * 32u; }

// =============================================================================================
// 1c. vector input (field GIVEN): range cells as well -- each vector layer is streamed once
// =============================================================================================
// No stencil here: a vertex's keys are the high words of its own components, so the build kernels read global memory
// directly (16-byte loads, two vertices per lane).  They also fold min non-zero |v| of the layer (the separate
// resolution pass over the whole layer disappears) and raise p.poison for magnitudes the float keys cannot order
// (>= 2^1000; the context then falls back to the two-layer scans).  Cell layouts and tests are those of the scalar
// paths: 3D = six 16-bit keys per (lane, 4-row block, plane), s3_test with thresholds for v instead of d = 2 v;
// 2D = four full high-word keys per (lane, 8-row block), cube_excluded2 on the key ranges.
constexpr int V2_R = 8;                                // 2D: corner rows per cell block

__device__ __forceinline__ size_t vcells2d_index(const SweepParams &p, const int strip, const int kb, const int lane) {
  return ((size_t)strip * (size_t)(p.H / V2_R + 2) + (size_t)kb) * 32u + (size_t)lane;
}

// exact (cold) update of the running min non-zero |v| with one vertex's components
template <int N>
__device__ __noinline__ double vres_vertex(double rmin, const double v0, const double v1, const double v2) {
  if (v0 != 0.0 && fabs(v0) < fabs(rmin)) rmin = v0;
  if (v1 != 0.0 && fabs(v1) < fabs(rmin)) rmin = v1;
  if (N == 3 && v2 != 0.0 && fabs(v2) < fabs(rmin)) rmin = v2;
  return rmin;
}

// cold path, 2D vector input: one lane per cube of the failing lane's 2 x V2_R cubes
__device__ __noinline__ void vcells2d_slow_cubes(const SweepParams &p, unsigned failmask, const int c0, const int y0, const int nl) {
  static_assert(2 * V2_R <= 32, "one lane per cube");
  const int lane = threadIdx.x & 31;
  const int nbits20 = p.nbits << 20;
  const int r = lane >> 1, q = lane & 1;
  while (failmask) {
    const int src = __ffs(failmask) - 1;
    failmask &= failmask - 1;
    const int x = c0 + 2 * src + q, y = y0 + r;
    const bool in = lane < 2 * V2_R && x >= p.lb[0] && x <= p.ub[0] && y >= p.lb[1] && y <= p.ub[1];
    KeyRange rx = neutral_range(), ry = neutral_range();
#pragma unroll
    for (int v = 0; v < 4; v++) {
      const int vx = x + (v & 1), vy = y + (v >> 1);
      if (!in || vx > p.ub[0] || vy > p.ub[1]) continue;
      const size_t i = (size_t)vx + (size_t)p.W * (size_t)vy;
      for (int L = 0; L < nl; L++) {
        const int4 a = __ldg(reinterpret_cast<const int4 *>(p.L[L].V) + i);
        rx = merge(rx, vertex_range(a.y, nbits20));
        ry = merge(ry, vertex_range(a.w, nbits20));
      }
    }
    const bool surv = in && !cube_excluded2(rx, ry);
    append_survivors(p, surv, (u64)(x - p.lb[0]) + (u64)p.nc[0] * (u64)(y - p.lb[1]));
  }
}

// float-key ranges (raw high words) -> excluded, or the cold path
__device__ __forceinline__ void vcells2d_decide(const SweepParams &p, const float xmn, const float xmx, const float ymn, const float ymx,
                                                const bool own, const int c0, const int y0, const int nl) {
  const int nbits20 = p.nbits << 20;
  bool excl = false;
  if (!(xmn != xmn) && !(ymn != ymn)) {       // a NaN union (no vertex) goes to the cold path, which is exact
    // merged, not {min.mn, max.mx}: a positive value with |p| >= 2^63 (INT64_MIN in the reference) at the upper end must poison
    // the range's mn, which cube_excluded2 tests
    const KeyRange x = merge(vertex_range(__float_as_int(xmn), nbits20), vertex_range(__float_as_int(xmx), nbits20));
    const KeyRange y = merge(vertex_range(__float_as_int(ymn), nbits20), vertex_range(__float_as_int(ymx), nbits20));
    excl = cube_excluded2(x, y);
  }
  const unsigned fm = __ballot_sync(0xffffffffu, own && !excl);
  if (fm) vcells2d_slow_cubes(p, fm, c0, y0, nl);
}

// warp = strip of 62 corner columns (64 vertex columns, two per lane) x a chunk of rows (a multiple of V2_R)
template <int NPREV, bool TEST>
__global__ void __launch_bounds__(256) vscan2d_build_kernel(const __grid_constant__ SweepParams p) {
  const int lane = threadIdx.x & 31;
  const i64 w = (i64)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int strip = (int)(w % p.nsx), cy = (int)(w / p.nsx);
  if (cy >= p.nsy) return;
  const int W = p.W, H = p.H, B = p.build_layer;
  const int c0 = strip * FB_STRIDE, e = c0 + 2 * lane;
  const bool e_ok = e < W, o_ok = e + 1 < W;
  const bool e_dom = e >= p.lb[0] && e <= p.ub[0], o_dom = e + 1 >= p.lb[0] && e + 1 <= p.ub[0];
  const bool own_cols = lane <= 30 && (e_dom || o_dom);
  const int r0 = cy * p.rows, r1 = min(r0 + p.rows - 1, H - 1), jl = min(r1 + 1, H - 1);
  const int4 *__restrict__ V = reinterpret_cast<const int4 *>(p.L[B].V);
  const bool want_res = p.res_slot[B] != nullptr;
  const float nanf_ = __int_as_float(KEYF_NAN), inff_ = __int_as_float(0x7F800000);
  double rmin = DBL_MAX;
  float rkey = inff_;
  int big = 0;
  const uint4 *sum_prev = NPREV ? p.sum_in[0] + vcells2d_index(p, strip, 0, lane) : nullptr;
  uint4 *sum_out = p.sum_out + vcells2d_index(p, strip, 0, lane);
  float bxmn = nanf_, bxmx = nanf_, bymn = nanf_, bymx = nanf_;
  uint4 prevc = make_uint4(0x7FC00000u, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u);

  auto finish_block = [&](const int kb, float xmn, float xmx, float ymn, float ymx) {
    xmn = fminf(xmn, __shfl_down_sync(0xffffffffu, xmn, 1)); xmx = fmaxf(xmx, __shfl_down_sync(0xffffffffu, xmx, 1));
    ymn = fminf(ymn, __shfl_down_sync(0xffffffffu, ymn, 1)); ymx = fmaxf(ymx, __shfl_down_sync(0xffffffffu, ymx, 1));
    sum_out[(size_t)kb * 32u] = make_uint4(__float_as_uint(xmn), __float_as_uint(xmx), __float_as_uint(ymn), __float_as_uint(ymx));
    if (TEST) {
      if (NPREV) {
        xmn = fminf(xmn, __uint_as_float(prevc.x)); xmx = fmaxf(xmx, __uint_as_float(prevc.y));
        ymn = fminf(ymn, __uint_as_float(prevc.z)); ymx = fmaxf(ymx, __uint_as_float(prevc.w));
      }
      const int y0 = kb * V2_R;
      vcells2d_decide(p, xmn, xmx, ymn, ymx, own_cols && y0 <= p.ub[1] && y0 + V2_R - 1 >= p.lb[1], c0, y0, NPREV + 1);
    }
  };

  for (int j0 = r0; j0 <= jl; j0 += V2_R) {
    // the rows of this block are independent loads: issue them all, then consume
    int4 a[V2_R][2];
#pragma unroll
    for (int k = 0; k < V2_R; k++) {
      const int j = j0 + k;
      const size_t i = (size_t)W * (size_t)min(j, H - 1) + (size_t)e;
      a[k][0] = (e_ok && j <= jl) ? __ldg(V + i) : make_int4(0, 0, 0, 0);
      a[k][1] = (o_ok && j <= jl) ? __ldg(V + i + 1) : make_int4(0, 0, 0, 0);
    }
    uint4 prevn = prevc;
    if (NPREV) prevn = __ldg(sum_prev + (size_t)(j0 / V2_R) * 32u);     // the block this row opens
#pragma unroll
    for (int k = 0; k < V2_R; k++) {
      const int j = j0 + k;
      if (j > jl) break;
      const bool dom_y = j >= p.lb[1] && j <= p.ub[1];
      float kxe = __int_as_float(a[k][0].y), kye = __int_as_float(a[k][0].w), kxo = __int_as_float(a[k][1].y), kyo = __int_as_float(a[k][1].w);
      big = max(big, max(max(a[k][0].y & 0x7fffffff, a[k][0].w & 0x7fffffff), max(a[k][1].y & 0x7fffffff, a[k][1].w & 0x7fffffff)));
      if (want_res) {
        const float m = fminf(e_ok ? fminf(fabsf(kxe), fabsf(kye)) : inff_, o_ok ? fminf(fabsf(kxo), fabsf(kyo)) : inff_);
        if (m <= rkey) {
          const double vxe = __hiloint2double(a[k][0].y, a[k][0].x), vye = __hiloint2double(a[k][0].w, a[k][0].z);
          const double vxo = __hiloint2double(a[k][1].y, a[k][1].x), vyo = __hiloint2double(a[k][1].w, a[k][1].z);
          bool go = m < rkey;
          if (!go) go = (e_ok && (fabs(vxe) < fabs(rmin) || fabs(vye) < fabs(rmin))) || (o_ok && (fabs(vxo) < fabs(rmin) || fabs(vyo) < fabs(rmin)));
          if (go) {
            if (e_ok) rmin = vres_vertex<2>(rmin, vxe, vye, 0.0);
            if (o_ok) rmin = vres_vertex<2>(rmin, vxo, vyo, 0.0);
            rkey = rmin == DBL_MAX ? inff_ : hikey(fabs(rmin));
          }
        }
      }
      if (!(e_dom && dom_y)) { kxe = nanf_; kye = nanf_; }
      if (!(o_dom && dom_y)) { kxo = nanf_; kyo = nanf_; }
      const float rxmn = fminf(kxe, kxo), rxmx = fmaxf(kxe, kxo), rymn = fminf(kye, kyo), rymx = fmaxf(kye, kyo);
      if (k == 0) {
        // vertex row V2_R k closes block k-1 and opens block k
        if (j > r0) finish_block(j / V2_R - 1, fminf(bxmn, rxmn), fmaxf(bxmx, rxmx), fminf(bymn, rymn), fmaxf(bymx, rymx));
        bxmn = rxmn; bxmx = rxmx; bymn = rymn; bymx = rymx;
        prevc = prevn;
      } else {
        bxmn = fminf(bxmn, rxmn); bxmx = fmaxf(bxmx, rxmx); bymn = fminf(bymn, rymn); bymx = fmaxf(bymx, rymx);
      }
    }
  }
  // a chunk's last block is closed by the next chunk's first row (read above as row jl); the array's last block ends at row H-1
  if (jl == H - 1) finish_block(jl / V2_R, bxmn, bxmx, bymn, bymx);
  if (want_res) warp_res_commit(fabs(rmin), p.res_slot[B]);
  if (big >= KEYF_BIG) atomicExch(p.poison, 1ull);
}

template <int NL>
__global__ void __launch_bounds__(256) vscan2d_cells_kernel(const __grid_constant__ SweepParams p, const int nstrips, const int nblk_used) {
  const int lane = threadIdx.x & 31;
  const long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (w >= (long long)nstrips * nblk_used) return;
  const int strip = (int)(w / nblk_used), kb = (int)(w % nblk_used);
  const int c0 = strip * FB_STRIDE, e = c0 + 2 * lane, y0 = kb * V2_R;
  const bool own = lane <= 30 && ((e >= p.lb[0] && e <= p.ub[0]) || (e + 1 >= p.lb[0] && e + 1 <= p.ub[0])) && y0 <= p.ub[1] && y0 + V2_R - 1 >= p.lb[1];
  if (!__any_sync(0xffffffffu, own)) return;
  const float nanf_ = __int_as_float(KEYF_NAN);
  float xmn = nanf_, xmx = nanf_, ymn = nanf_, ymx = nanf_;
#pragma unroll
  for (int L = 0; L < NL; L++) {
    const uint4 c = __ldg(p.sum_in[L] + vcells2d_index(p, strip, kb, lane));
    xmn = fminf(xmn, __uint_as_float(c.x)); xmx = fmaxf(xmx, __uint_as_float(c.y));
    ymn = fminf(ymn, __uint_as_float(c.z)); ymx = fmaxf(ymx, __uint_as_float(c.w));
  }
  vcells2d_decide(p, xmn, xmx, ymn, ymx, own, c0, y0, NL);
}


// 3D: CTA = 8 warps over a tile of 62 x 32 corner columns, marching along a chunk of planes; per plane a thread reads
// its 2 columns x (S3_RW + 1) rows (three 16-byte loads per row)
template <bool EDGE, int NPREV, bool TEST>
__device__ __forceinline__ void vs3_consume(const SweepParams &p, const int tile, const int C0, const int Y0, const int zc0, const int zc1,
                                            const int wib, const int lane) {
  const int B = p.build_layer, W = p.W, H = p.H, D = p.D;
  const int e = C0 + 2 * lane, y0 = Y0 + wib * S3_RW;
  const S3Thresholds T = s3_thresholds(p.nbits, true);
  const bool want_res = p.res_slot[B] != nullptr;
  const float nanf_ = __int_as_float(KEYF_NAN), inff_ = __int_as_float(0x7F800000);
  const int4 *__restrict__ V = reinterpret_cast<const int4 *>(p.L[B].V);
  bool own_any = lane <= 30;
  unsigned mk = 0xffffffffu;     // bit r (+0 / +8): vertex (e / e+1, y0 + r) exists; bit r (+16 / +24): and lies in the domain
  if (EDGE) {
    unsigned ok = 0, dom = 0;
#pragma unroll
    for (int r = 0; r <= S3_RW; r++) {
      ok |= (y0 + r < H) ? (1u << r) : 0u;
      dom |= (y0 + r >= p.lb[1] && y0 + r <= p.ub[1]) ? (1u << r) : 0u;
    }
    const bool e_ok = e < W, o_ok = e + 1 < W;
    const bool e_dom = e >= p.lb[0] && e <= p.ub[0], o_dom = e + 1 >= p.lb[0] && e + 1 <= p.ub[0];
    mk = (e_ok ? ok : 0u) | ((o_ok ? ok : 0u) << 8) | ((e_dom ? dom : 0u) << 16) | ((o_dom ? dom : 0u) << 24);
    own_any = own_any && (e_dom || o_dom) && y0 <= p.ub[1] && y0 + S3_RW - 1 >= p.lb[1];
  }
  double rmin = DBL_MAX;
  float rkey = inff_;
  int big = 0;
  uint32_t pcell[3] = {0x7FC07FC0u, 0x7FC07FC0u, 0x7FC07FC0u};
  const size_t cell0 = s3_cell_index(p, tile, wib, zc0, lane);
  const uint4 *sum_prev = NPREV ? p.sum_in[0] + cell0 : nullptr;
  uint4 *sum_out = p.sum_out + cell0;
  const size_t row3 = (size_t)W * 3 / 2;            // int4 per row (W even)
  for (int zg = zc0; zg <= zc1 + 1; zg++) {
    uint4 prev = make_uint4(0x7FC07FC0u, 0x7FC07FC0u, 0x7FC07FC0u, 0u);
    if (NPREV) prev = __ldg(sum_prev);
    const bool zok = zg < D;
    const bool zdom = zg >= p.lb[2] && zg <= p.ub[2];
    float umin[3] = {nanf_, nanf_, nanf_}, umax[3] = {nanf_, nanf_, nanf_};
    if (zok) {
      unsigned m2 = mk;
      if (EDGE) asm volatile("" : "+r"(m2));
      int4 a[S3_RW + 1][3];
      const int4 *base = V + ((size_t)zg * (size_t)H + (size_t)y0) * row3 + (size_t)e * 3 / 2;
#pragma unroll
      for (int r = 0; r <= S3_RW; r++) {
        const bool ld = !EDGE || (((m2 >> r) | (m2 >> (r + 8))) & 1u);     // e + 1 < W whenever e < W (W even)
#pragma unroll
        for (int q = 0; q < 3; q++) a[r][q] = ld ? __ldg(base + (size_t)r * row3 + q) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int r = 0; r <= S3_RW; r++) {
        // vertex e: (x,y) = a0.xyzw, z = a1.xy; vertex e+1: x = a1.zw, (y,z) = a2.xyzw
        float kxe = __int_as_float(a[r][0].y), kye = __int_as_float(a[r][0].w), kze = __int_as_float(a[r][1].y);
        float kxo = __int_as_float(a[r][1].w), kyo = __int_as_float(a[r][2].y), kzo = __int_as_float(a[r][2].w);
        big = max(big, max(max(a[r][0].y & 0x7fffffff, a[r][0].w & 0x7fffffff), a[r][1].y & 0x7fffffff));
        big = max(big, max(max(a[r][1].w & 0x7fffffff, a[r][2].y & 0x7fffffff), a[r][2].w & 0x7fffffff));
        if (want_res) {
          float ma = fminf(fminf(fabsf(kxe), fabsf(kye)), fabsf(kze)), mb = fminf(fminf(fabsf(kxo), fabsf(kyo)), fabsf(kzo));
          bool in_e = true, in_o = true;
          if (EDGE) { in_e = (m2 >> r) & 1u; in_o = (m2 >> (r + 8)) & 1u; ma = in_e ? ma : inff_; mb = in_o ? mb : inff_; }
          const float m = fminf(ma, mb);
          if (m <= rkey) {
            const double vxe = __hiloint2double(a[r][0].y, a[r][0].x), vye = __hiloint2double(a[r][0].w, a[r][0].z), vze = __hiloint2double(a[r][1].y, a[r][1].x);
            const double vxo = __hiloint2double(a[r][1].w, a[r][1].z), vyo = __hiloint2double(a[r][2].y, a[r][2].x), vzo = __hiloint2double(a[r][2].w, a[r][2].z);
            bool go = m < rkey;
            const double ar = fabs(rmin);
            if (!go) go = (in_e && (fabs(vxe) < ar || fabs(vye) < ar || fabs(vze) < ar)) || (in_o && (fabs(vxo) < ar || fabs(vyo) < ar || fabs(vzo) < ar));
            if (go) {
              if (in_e) rmin = vres_vertex<3>(rmin, vxe, vye, vze);
              if (in_o) rmin = vres_vertex<3>(rmin, vxo, vyo, vzo);
              rkey = rmin == DBL_MAX ? inff_ : hikey(fabs(rmin));
            }
          }
        }
        if (EDGE) {
          const bool de = (m2 >> (r + 16)) & 1u, dq = (m2 >> (r + 24)) & 1u;
          kxe = de ? kxe : nanf_; kye = de ? kye : nanf_; kze = de ? kze : nanf_;
          kxo = dq ? kxo : nanf_; kyo = dq ? kyo : nanf_; kzo = dq ? kzo : nanf_;
        }
        umin[0] = fminf(umin[0], fminf(kxe, kxo)); umax[0] = fmaxf(umax[0], fmaxf(kxe, kxo));
        umin[1] = fminf(umin[1], fminf(kye, kyo)); umax[1] = fmaxf(umax[1], fmaxf(kye, kyo));
        umin[2] = fminf(umin[2], fminf(kze, kzo)); umax[2] = fmaxf(umax[2], fmaxf(kze, kzo));
      }
    }
    if (!zdom) {
#pragma unroll
      for (int c = 0; c < 3; c++) { umin[c] = nanf_; umax[c] = nanf_; }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) {
      umin[c] = fminf(umin[c], __shfl_down_sync(0xffffffffu, umin[c], 1));
      umax[c] = fmaxf(umax[c], __shfl_down_sync(0xffffffffu, umax[c], 1));
    }
    *sum_out = make_uint4(pack_keys(umin[0], umax[0]), pack_keys(umin[1], umax[1]), pack_keys(umin[2], umax[2]), 0u);
    sum_out += 32;
    if (NPREV) sum_prev += 32;
    if (TEST) {
      if (NPREV) merge_cell(umin, umax, prev);
      if (zg > zc0) {
        const int zc_ = zg - 1;
        if (zc_ >= p.lb[2] && zc_ <= p.ub[2]) {
          float cmn[3] = {umin[0], umin[1], umin[2]}, cmx[3] = {umax[0], umax[1], umax[2]};
          merge_cell(cmn, cmx, make_uint4(pcell[0], pcell[1], pcell[2], 0u));
          s3_test(p, T, cmn, cmx, own_any, e, y0, zc_, NPREV + 1);
        }
      }
#pragma unroll
      for (int c = 0; c < 3; c++) pcell[c] = pack_keys(umin[c], umax[c]);
    }
  }
  if (want_res) warp_res_commit(fabs(rmin), p.res_slot[B]);
  if (big >= KEYF_BIG) atomicExch(p.poison, 1ull);
}

template <int NPREV, bool TEST>
__global__ void __launch_bounds__(F3_CW * 32, 2) vscan3d_build_kernel(const __grid_constant__ SweepParams p) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int b = blockIdx.x;
  const int bx = b % p.nsx; b /= p.nsx;
  const int by = b % p.nsy;
  const int bz = b / p.nsy;
  const int C0 = bx * F3_STRIDE, Y0 = by * F3_TROWS;
  const int zc0 = bz * p.rows, zc1 = min(zc0 + p.rows - 1, p.D - 1);
  const int tile = by * p.nsx + bx;
  const bool interior = C0 >= p.lb[0] && C0 + 63 <= min(p.W - 1, p.ub[0]) && Y0 >= p.lb[1] && Y0 + F3_TROWS <= min(p.H - 1, p.ub[1]);
  if (interior) vs3_consume<false, NPREV, TEST>(p, tile, C0, Y0, zc0, zc1, wib, lane);
  else vs3_consume<true, NPREV, TEST>(p, tile, C0, Y0, zc0, zc1, wib, lane);
}

size_t vscan2d_cells_per_layer(const SweepParams &p) { return (size_t)p.nsx * (size_t)(p.H / V2_R + 2) * 32u; }

void launch_vscan_cells(const SweepParams &p, cudaStream_t s) {
  if (p.nd == 3) {
    const unsigned grid = (unsigned)((i64)p.nsx * p.nsy * p.nsz);
    switch (p.sum_mode) {
      case SUM_BUILD: vscan3d_build_kernel<0, false><<<grid, F3_CW * 32, 0, s>>>(p); break;
      case SUM_BUILD_TEST1: vscan3d_build_kernel<0, true><<<grid, F3_CW * 32, 0, s>>>(p); break;
      case SUM_BUILD_TEST2: vscan3d_build_kernel<1, true><<<grid, F3_CW * 32, 0, s>>>(p); break;
      case SUM_TEST1: scan3d_cells_kernel<1><<<grid, F3_CW * 32, 0, s>>>(p); break;
      default: scan3d_cells_kernel<2><<<grid, F3_CW * 32, 0, s>>>(p); break;
    }
    return;
  }
  const unsigned grid = (unsigned)(((i64)p.nsx * p.nsy + 7) / 8);
  const int nblk = (p.H + V2_R - 1) / V2_R;
  const unsigned tgrid = (unsigned)(((i64)p.nsx * nblk + 7) / 8);
  switch (p.sum_mode) {
    case SUM_BUILD: vscan2d_build_kernel<0, false><<<grid, 256, 0, s>>>(p); break;
    case SUM_BUILD_TEST1: vscan2d_build_kernel<0, true><<<grid, 256, 0, s>>>(p); break;
    case SUM_BUILD_TEST2: vscan2d_build_kernel<1, true><<<grid, 256, 0, s>>>(p); break;
    case SUM_TEST1: vscan2d_cells_kernel<1><<<tgrid, 256, 0, s>>>(p, p.nsx, nblk); break;
    default: vscan2d_cells_kernel<2><<<tgrid, 256, 0, s>>>(p, p.nsx, nblk); break;
  }
}


typedef CUresult (*TmapEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                 const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

bool encode_scalar_tmap3d(const double *S, int W, int H, int D, CUtensorMap *out) {
  static TmapEncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<TmapEncodeFn>(ptr);
    else cudaGetLastError();
  }
  if (!fn || (W & 1) || ((uintptr_t)S & 15)) return false;     // strides must be multiples of 16 B
  const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D};
  const cuuint64_t gstride[2] = {(cuuint64_t)W * 8, (cuuint64_t)W * (cuuint64_t)H * 8};
  const cuuint32_t box[3] = {F3_COLS, F3_ROWS, 1}, estr[3] = {1, 1, 1};
  return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double *>(S), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

void init_kernel_attributes() {
  cudaFuncSetAttribute(scan2d_build_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c2_smem_bytes());
  cudaFuncSetAttribute(scan2d_build_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c2_smem_bytes());
  cudaFuncSetAttribute(scan2d_build_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c2_smem_bytes());
  cudaFuncSetAttribute(scan2d_keys_build_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem_bytes());
  cudaFuncSetAttribute(scan2d_keys_build_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem_bytes());
  cudaFuncSetAttribute(scan2d_keys_build_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem_bytes());
  cudaFuncSetAttribute(scan3d_build_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s3_smem_bytes());
  cudaFuncSetAttribute(scan3d_build_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s3_smem_bytes());
  cudaFuncSetAttribute(scan3d_build_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s3_smem_bytes());
}

// summary path of the fused 3D scan: p.sum_mode selects what one launch does (see SweepParams)
void launch_scan3d_cells(const SweepParams &p, cudaStream_t s) {
  const unsigned grid = (unsigned)((i64)p.nsx * p.nsy * p.nsz);
  switch (p.sum_mode) {
    case SUM_BUILD: scan3d_build_kernel<0, false><<<grid, F3_CW * 32, s3_smem_bytes(), s>>>(p); break;
    case SUM_BUILD_TEST1: scan3d_build_kernel<0, true><<<grid, F3_CW * 32, s3_smem_bytes(), s>>>(p); break;
    case SUM_BUILD_TEST2: scan3d_build_kernel<1, true><<<grid, F3_CW * 32, s3_smem_bytes(), s>>>(p); break;
    case SUM_TEST1: scan3d_cells_kernel<1><<<grid, F3_CW * 32, 0, s>>>(p); break;
    default: scan3d_cells_kernel<2><<<grid, F3_CW * 32, 0, s>>>(p); break;
  }
}

void launch_scan(const SweepParams &p, cudaStream_t s) {
  const unsigned grid = p.nd == 2 ? (unsigned)(((i64)p.nsx * p.nsy + 7) / 8) : (unsigned)((i64)p.nsx * p.nsy * p.nsz);
  if (p.nd == 2 && p.fused) {     // rows that are not 16-byte aligned (aligned ones take the range-cell kernels)
    if (p.has_next) scan2d_fused_kernel<true><<<grid, 256, 0, s>>>(p);
    else scan2d_fused_kernel<false><<<grid, 256, 0, s>>>(p);
  } else if (p.nd == 2) {
    if (p.has_next) scan2d_kernel<true><<<grid, 256, 0, s>>>(p);
    else scan2d_kernel<false><<<grid, 256, 0, s>>>(p);
  } else {
    const dim3 block(32, SCAN3_BY);
    if (p.has_next) scan3d_kernel<true><<<grid, block, 0, s>>>(p);
    else scan3d_kernel<false><<<grid, block, 0, s>>>(p);
  }
}

// =============================================================================================
// 2. exact predicates (ref: include/ftk/numeric/sign_det.hh, det.hh, critical_point_test.hh)
// =============================================================================================
// All integer arithmetic wraps mod 2^64 exactly like the reference's int64 (-fwrapv) evaluation;
// the determinant expansions below are polynomial identities of the reference's, hence equal
// mod 2^64 term order notwithstanding.
// [host-testable: begin]  (tests/test_predicate_fast_path.py compiles the lines up to the matching end marker with g++)
__device__ __forceinline__ int sgn(i64 v) { return (v > 0) - (v < 0); }
__device__ __forceinline__ u64 U(i64 v) { return (u64)v; }

// | a0 a1 1 |
// | b0 b1 1 |
// | c0 c1 1 |
__device__ __forceinline__ i64 det3_h(i64 a0, i64 a1, i64 b0, i64 b1, i64 c0, i64 c1) {
  return (i64)(U(a0) * (U(b1) - U(c1)) - U(a1) * (U(b0) - U(c0)) + (U(b0) * U(c1) - U(b1) * U(c0)));
}

// 4x4 determinant of rows (x, y, z, 1): subtracting row 0 and expanding along the last column
// gives -det3 of the difference rows
__device__ __forceinline__ i64 det4_h(const i64 X[4][3]) {
  u64 d[3][3];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) d[i][j] = U(X[i + 1][j]) - U(X[0][j]);
  const u64 det = d[0][0] * (d[1][1] * d[2][2] - d[1][2] * d[2][1])
                - d[0][1] * (d[1][0] * d[2][2] - d[1][2] * d[2][0])
                + d[0][2] * (d[1][0] * d[2][1] - d[1][1] * d[2][0]);
  return (i64)(0 - det);
}

// sign of the 3x3 orientation determinant with the symbolic perturbation cascade (sign_det.hh:44-90)
__device__ int sos_sign3(const i64 X[3][2]) {
  int s = sgn(det3_h(X[0][0], X[0][1], X[1][0], X[1][1], X[2][0], X[2][1]));
  if (s) return s;
  s = -sgn((i64)(U(X[1][0]) - U(X[2][0])));
  if (s) return s;
  s = sgn((i64)(U(X[1][1]) - U(X[2][1])));
  if (s) return s;
  s = sgn((i64)(U(X[0][0]) - U(X[2][0])));
  if (s) return s;
  return 1;
}

// 4x4 cascade (sign_det.hh:92-200): 15 levels
__device__ int sos_sign4(const i64 X[4][3]) {
  int s = sgn(det4_h(X));
  if (s) return s;
#define D3(r0, r1, r2, c0, c1) det3_h(X[r0][c0], X[r0][c1], X[r1][c0], X[r1][c1], X[r2][c0], X[r2][c1])
#define D2(r0, r1, c) ((i64)(U(X[r0][c]) - U(X[r1][c])))
  s = sgn(D3(1, 2, 3, 0, 1)); if (s) return s;
  s = -sgn(D3(1, 2, 3, 0, 2)); if (s) return s;
  s = sgn(D3(1, 2, 3, 1, 2)); if (s) return s;
  s = -sgn(D3(0, 2, 3, 0, 1)); if (s) return s;
  s = sgn(D2(2, 3, 0)); if (s) return s;
  s = -sgn(D2(2, 3, 1)); if (s) return s;
  s = sgn(D3(0, 2, 3, 0, 2)); if (s) return s;
  s = sgn(D2(2, 3, 2)); if (s) return s;
  s = -sgn(D3(0, 2, 3, 1, 2)); if (s) return s;
  s = sgn(D3(0, 1, 3, 0, 1)); if (s) return s;
  s = -sgn(D2(1, 3, 0)); if (s) return s;
  s = sgn(D2(1, 3, 1)); if (s) return s;
  s = sgn(D2(0, 3, 0)); if (s) return s;
#undef D3
#undef D2
  return 1;
}

// rows sorted by vertex rank with the reference's bubble sort (strict >, adjacent swaps); the
// sign flips with the parity of the number of swaps (sign_det.hh:203-289)
template <int NV, int NC>
__device__ int oriented_sign(const i64 Xin[NV][NC], const int idx_in[NV]) {
  int idx[NV], ord[NV];
#pragma unroll
  for (int i = 0; i < NV; i++) { idx[i] = idx_in[i]; ord[i] = i; }
  int swaps = 0;
#pragma unroll
  for (int i = 0; i < NV - 1; i++)
#pragma unroll
    for (int j = 0; j < NV - 1 - i; j++)
      if (idx[j] > idx[j + 1]) {
        int t = idx[j]; idx[j] = idx[j + 1]; idx[j + 1] = t;
        t = ord[j]; ord[j] = ord[j + 1]; ord[j + 1] = t;
        swaps++;
      }
  i64 X[NV][NC];
#pragma unroll
  for (int i = 0; i < NV; i++)
#pragma unroll
    for (int j = 0; j < NC; j++) {
      // ord[] is a register-resident permutation: select without dynamic indexing
      i64 v = 0;
#pragma unroll
      for (int q = 0; q < NV; q++) v = (ord[i] == q) ? Xin[q][j] : v;
      X[i][j] = v;
    }
  int s;
  if constexpr (NV == 3) s = sos_sign3(X);
  else s = sos_sign4(X);
  return (swaps & 1) ? -s : s;
}

// origin (rank -1) inside the simplex: the orientation must not change when any one row is
// replaced by the origin (sign_det.hh:360-414, critical_point_test.hh:22-34)
template <int NV, int NC>
__device__ __noinline__ bool origin_in_simplex(const i64 X[NV][NC], const int idx[NV]) {
  const int s = oriented_sign<NV, NC>(X, idx);
#pragma unroll 1
  for (int i = 0; i < NV; i++) {
    i64 Y[NV][NC];
    int my[NV];
#pragma unroll
    for (int j = 0; j < NV; j++) {
      const bool rep = (j == i);
      my[j] = rep ? -1 : idx[j];
#pragma unroll
      for (int c = 0; c < NC; c++) Y[j][c] = rep ? 0 : X[j][c];
    }
    if (oriented_sign<NV, NC>(Y, my) != s) return false;
  }
  return true;
}

// Fast paths of origin_in_simplex.  The reference sorts the rows by vertex rank and multiplies the sign by the parity of the
// swaps; the determinant is an alternating polynomial of the rows, and the arithmetic is mod 2^64 (a ring), so
// det(sorted) = (-1)^swaps det(unsorted) exactly -- whenever a determinant is neither 0 (the symbolic cascade decides) nor
// -2^63 (the one value whose negation has the same sign) the sorted, parity-corrected sign IS the sign of the unsorted
// determinant.  A row replaced by the origin leaves a minor: expanding along the column of ones, det = sum of the replaced
// determinants D_i.  All D_i and their sum usable -> compare signs; anything else -> the full cascade above.
__device__ __forceinline__ bool usable_det(i64 v) { return v != 0 && v != LLONG_MIN; }

__device__ __forceinline__ bool origin_in_simplex_fast(const i64 X[3][2], const int idx[3]) {
  const u64 a0 = U(X[0][0]), a1 = U(X[0][1]), b0 = U(X[1][0]), b1 = U(X[1][1]), c0 = U(X[2][0]), c1 = U(X[2][1]);
  const i64 Da = (i64)(b0 * c1 - b1 * c0);      // det3_h with row 0 = origin
  const i64 Db = (i64)(a1 * c0 - a0 * c1);      // row 1 = origin
  const i64 Dc = (i64)(a0 * b1 - a1 * b0);      // row 2 = origin
  const i64 D = (i64)(U(Da) + U(Db) + U(Dc));   // det3_h of the simplex itself
  if (usable_det(D) && usable_det(Da) && usable_det(Db) && usable_det(Dc)) {
    const bool pos = D > 0;
    return (Da > 0) == pos && (Db > 0) == pos && (Dc > 0) == pos;
  }
  return origin_in_simplex<3, 2>(X, idx);
}

__device__ __forceinline__ u64 det3_rows(const u64 r0[3], const u64 r1[3], const u64 r2[3]) {
  return r0[0] * (r1[1] * r2[2] - r1[2] * r2[1]) - r0[1] * (r1[0] * r2[2] - r1[2] * r2[0]) + r0[2] * (r1[0] * r2[1] - r1[1] * r2[0]);
}

__device__ __forceinline__ bool origin_in_simplex_fast(const i64 X[4][3], const int idx[4]) {
  u64 r[4][3];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) r[i][j] = U(X[i][j]);
  // det of rows (x, y, z, 1) with row i replaced by (0, 0, 0, 1): (-1)^(i+3) times the minor of the other rows
  const i64 D0 = (i64)(0 - det3_rows(r[1], r[2], r[3]));
  const i64 D1 = (i64)det3_rows(r[0], r[2], r[3]);
  const i64 D2 = (i64)(0 - det3_rows(r[0], r[1], r[3]));
  const i64 D3 = (i64)det3_rows(r[0], r[1], r[2]);
  const i64 D = (i64)(U(D0) + U(D1) + U(D2) + U(D3));
  if (usable_det(D) && usable_det(D0) && usable_det(D1) && usable_det(D2) && usable_det(D3)) {
    const bool pos = D > 0;
    return (D0 > 0) == pos && (D1 > 0) == pos && (D2 > 0) == pos && (D3 > 0) == pos;
  }
  return origin_in_simplex<4, 3>(X, idx);
}
// [host-testable: end]

// =============================================================================================
// 3. floating-point leaves (literal operation order of the reference)
// =============================================================================================
__device__ __forceinline__ double std_max(double a, double b) { return (a < b) ? b : a; }
__device__ __forceinline__ double std_min(double a, double b) { return (b < a) ? b : a; }

// ref: include/ftk/numeric/clamp.hh:15-37
template <int N>
__device__ __forceinline__ void clamp_barycentric(double *x) {
  double sum = 0.0;
#pragma unroll
  for (int i = 0; i < N; i++) { x[i] = std_min(std_max(0.0, x[i]), 1.0); sum += x[i]; }
#pragma unroll
  for (int i = 0; i < N; i++) x[i] /= sum;
  if (isnan(x[0]) || isinf(x[0])) {
#pragma unroll
    for (int i = 0; i < N; i++) x[i] = 1.0 / N;
  }
}

// ref: inverse_linear_interpolation_solver.hh:32-54, linear_solver.hh:22-34 (Cramer)
__device__ bool inverse_lerp2(const double V[3][2], double mu[3]) {
  const double eps = DBL_EPSILON;
  const double A00 = V[0][0] - V[2][0], A01 = V[1][0] - V[2][0], A10 = V[0][1] - V[2][1], A11 = V[1][1] - V[2][1];
  const double b0 = -V[2][0], b1 = -V[2][1];
  const double D = A00 * A11 - A10 * A01, Dx = b0 * A11 - A01 * b1, Dy = A00 * b1 - b0 * A10;
  mu[0] = Dx / D;
  mu[1] = Dy / D;
  mu[2] = 1.0 - mu[0] - mu[1];
  return mu[0] >= -eps && mu[0] <= 1.0 + eps && mu[1] >= -eps && mu[1] <= 1.0 + eps && mu[2] >= -eps && mu[2] <= 1.0 + eps;
}

// ref: inverse_linear_interpolation_solver.hh:143-167, linear_solver.hh:12-20, matrix_inverse.hh:23-45
__device__ bool inverse_lerp3(const double V[4][3], double l[4]) {
  const double eps = DBL_EPSILON;
  double m[3][3], inv[3][3];
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) m[r][c] = V[c][r] - V[3][r];
  const double b[3] = {-V[3][0], -V[3][1], -V[3][2]};
  inv[0][0] = m[1][1] * m[2][2] - m[1][2] * m[2][1];
  inv[0][1] = -m[0][1] * m[2][2] + m[0][2] * m[2][1];
  inv[0][2] = m[0][1] * m[1][2] - m[0][2] * m[1][1];
  inv[1][0] = -m[1][0] * m[2][2] + m[1][2] * m[2][0];
  inv[1][1] = m[0][0] * m[2][2] - m[0][2] * m[2][0];
  inv[1][2] = -m[0][0] * m[1][2] + m[0][2] * m[1][0];
  inv[2][0] = m[1][0] * m[2][1] - m[1][1] * m[2][0];
  inv[2][1] = -m[0][0] * m[2][1] + m[0][1] * m[2][0];
  inv[2][2] = m[0][0] * m[1][1] - m[0][1] * m[1][0];
  const double det = m[0][0] * inv[0][0] + m[0][1] * inv[1][0] + m[0][2] * inv[2][0];
  const double invdet = 1.0 / det;
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) inv[r][c] = inv[r][c] * invdet;
#pragma unroll
  for (int r = 0; r < 3; r++) l[r] = inv[r][0] * b[0] + inv[r][1] * b[1] + inv[r][2] * b[2];
  l[3] = 1.0 - l[0] - l[1] - l[2];
  return l[0] >= -eps && l[0] < 1.0 + eps && l[1] >= -eps && l[1] < 1.0 + eps &&
         l[2] >= -eps && l[2] < 1.0 + eps && l[3] >= -eps && l[3] < 1.0 + eps;
}

// ref: critical_point_type.hh:40-72, eigen_solver2.hh:18-41,63-68, quadratic_solver.hh:12-25
__device__ unsigned cp_type_2d(const double J[2][2], bool symmetric) {
  if (symmetric) {
    const double m00 = J[0][0], m10 = J[1][0], m11 = J[1][1];
    const double b = -(m00 + m11), c = m00 * m11 - m10 * m10;
    const double delta = fma(b, b, -4 * c);
    const double sq = delta < 0 ? 0 : sqrt(delta);
    double e0 = 0.5 * (-b + sq), e1 = 0.5 * (-b - sq);
    if (fabs(e0) < fabs(e1)) { const double t = e0; e0 = e1; e1 = t; }
    if (e0 > 0 && e1 > 0) return 2;
    if (e0 < 0 && e1 < 0) return 8;
    if (e0 * e1 < 0) return 4;
    return 1;
  }
  const double P1 = -(J[0][0] + J[1][1]), P0 = J[0][0] * J[1][1] - J[1][0] * J[0][1];
  const double delta = P1 * P1 - 4 * 1.0 * P0;
  if (delta >= 0) {
    const double r0 = (-P1 + sqrt(delta)) / 2.0, r1 = (-P1 - sqrt(delta)) / 2.0;
    if (r0 * r1 < 0) return 4;
    if (r0 > 0 && r1 > 0) return 2;
    if (r0 < 0 && r1 < 0) return 8;
    return 1;
  }
  // conjugate pair (or NaN): real part of (-P1 + pow(complex(delta), 0.5)) / 2, evaluated the way
  // libstdc++ does (polar form), so a vanishing trace still yields the tiny positive real part
  const double rho = exp(0.5 * log(fabs(delta))), theta = 0.5 * atan2(0.0, delta);
  const double re = (-P1 + rho * cos(theta)) / 2.0;
  if (re < 0) return 16;
  if (re > 0) return 32;
  return 64;
}

// ref: critical_point_type.hh:74-93, eigen_solver3.hh:16-47, characteristic_polynomial.hh:36-47
__device__ unsigned cp_type_3d(const double A[3][3], bool symmetric) {
  if (!symmetric) return 0;
  const double b = -(A[0][0] + A[1][1] + A[2][2]);
  const double c = A[1][1] * A[2][2] + A[0][0] * A[2][2] + A[0][0] * A[1][1] - A[0][1] * A[1][0] - A[1][2] * A[2][1] - A[0][2] * A[2][0];
  const double d = -(A[0][0] * (A[1][1] * A[2][2] - A[1][2] * A[2][1]) - A[0][1] * (A[1][0] * A[2][2] - A[1][2] * A[2][0]) +
                     A[0][2] * (A[1][0] * A[2][1] - A[1][1] * A[2][0]));
  double x0, x1, x2;
  double q = (3.0 * c - (b * b)) / 9.0;
  const double r = (-(27.0 * d) + b * (9.0 * c - 2.0 * (b * b))) / 54.0;
  const double disc = q * q * q + r * r;
  const double term1 = (b / 3.0);
  if (disc >= 0) {
    const double r13 = (r < 0) ? -pow(-r, (1.0 / 3.0)) : pow(r, (1.0 / 3.0));
    x0 = -term1 + 2.0 * r13;
    x1 = -(r13 + term1);
    x2 = -(r13 + term1);
  } else {
    const double kPi = 3.14159265358979323846;
    q = -q;
    double dum1 = q * q * q;
    dum1 = acos(r / sqrt(dum1));
    const double r13 = 2.0 * sqrt(q);
    x0 = -term1 + r13 * cos(dum1 / 3.0);
    x1 = -term1 + r13 * cos((dum1 + 2.0 * kPi) / 3.0);
    x2 = -term1 + r13 * cos((dum1 + 4.0 * kPi) / 3.0);
  }
  if (x0 * x1 * x2 == 0.0) return 1;
  if (x0 < 0 && x1 < 0 && x2 < 0) return 8;
  if (x0 > 0 && x1 > 0 && x2 > 0) return 2;
  return 4;
}

// =============================================================================================
// 4. the fused per-simplex test
// =============================================================================================

// x86-64 cvttsd2si semantics: out-of-range and NaN give INT64_MIN (the reference's cast, compiled for x86-64)
__device__ __forceinline__ i64 quantise(double v, double factor) {
  const double pq = v * factor;
  if (!(pq < 9223372036854775808.0) || pq < -9223372036854775808.0) return LLONG_MIN;
  return (i64)pq;
}

// Jacobian at one vertex, derived on demand from the resident vector layer with the reference's
// formulas (ref: include/ftk/ndarray/grad.hh:54-86, incl. the unscaled first term and the
// non-symmetric variant's off-diagonals landing on array element 0 only).
// component c of the vector field at vertex (i, j) (indices clamped to the array like the reference's
// accessor lambdas): read from the resident vector layer, or -- when the layer only holds the scalar
// field -- derived with gradient2D's formula (grad.hh:10-31)
__device__ __forceinline__ double vec2_at(const SweepParams &p, const LayerPtrs &L, int c, int i, int j) {
  const int W = p.W, H = p.H;
  i = clampi(i, W); j = clampi(j, H);
  if (L.V) return __ldg(L.V + c + 2 * ((size_t)i + (size_t)W * j));
#define SF(ii, jj) __ldg(L.S + (size_t)clampi(ii, W) + (size_t)W * clampi(jj, H))
  return c == 0 ? (SF(i + 1, j) - SF(i - 1, j)) * (W - 1) : (SF(i, j + 1) - SF(i, j - 1)) * (H - 1);
#undef SF
}

// gradient3D (grad.hh:130-149): 1/2 central differences on the interior, zero on the array border
__device__ __forceinline__ double vec3_at(const SweepParams &p, const LayerPtrs &L, int c, int i, int j, int k) {
  const int W = p.W, H = p.H, D = p.D;
  const size_t idx = (size_t)i + (size_t)W * ((size_t)j + (size_t)H * (size_t)k);
  if (L.V) return __ldg(L.V + c + 3 * idx);
  if (!(i >= 1 && i < W - 1 && j >= 1 && j < H - 1 && k >= 1 && k < D - 1)) return 0.0;
  const size_t st = c == 0 ? 1 : (c == 1 ? (size_t)W : (size_t)W * H);
  return 0.5 * (__ldg(L.S + idx + st) - __ldg(L.S + idx - st));
}

__device__ void jacobian2d_at(const SweepParams &p, const LayerPtrs &L, int i, int j, double G[2][2] /* G[a][b] = jacobian(a,b,i,j) */) {
  const int W = p.W, H = p.H;
#define F2(c, ii, jj) vec2_at(p, L, c, ii, jj)
  const double H00 = F2(0, i + 1, j) - F2(0, i - 1, j) * (W - 1), H11 = F2(1, i, j + 1) - F2(1, i, j - 1) * (H - 1);
  G[0][0] = H00;
  G[1][1] = H11;
  if (p.derived_symmetric) {
    const double H01 = F2(0, i, j + 1) - F2(0, i, j - 1) * (H - 1), H10 = F2(1, i + 1, j) - F2(1, i - 1, j) * (W - 1);
    G[0][1] = G[1][0] = (H01 + H10) * 0.5;
  } else if (i == 0 && j == 0) {
    const int li = W - 1, lj = H - 1;   // the last vertex written by the reference's loop
    G[0][1] = F2(0, li, lj + 1) - F2(0, li, lj - 1) * (H - 1);
    G[1][0] = F2(1, li + 1, lj) - F2(1, li - 1, lj) * (W - 1);
  } else {
    G[0][1] = G[1][0] = 0.0;
  }
#undef F2
}

// ref: grad.hh:175-212 (interior [2, D-3] only, zero elsewhere)
__device__ void jacobian3d_at(const SweepParams &p, const LayerPtrs &L, int i, int j, int k, double G[3][3] /* G[c][d] = dV_c/dx_d * 0.5 form */) {
  const int W = p.W, H = p.H, D = p.D;
  const bool in = i >= 2 && i < W - 2 && j >= 2 && j < H - 2 && k >= 2 && k < D - 2;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    if (!in) { G[c][0] = G[c][1] = G[c][2] = 0.0; continue; }
#define F3(c, ii, jj, kk) vec3_at(p, L, c, ii, jj, kk)
    G[c][0] = 0.5 * (F3(c, i + 1, j, k) - F3(c, i - 1, j, k));
    G[c][1] = 0.5 * (F3(c, i, j + 1, k) - F3(c, i, j - 1, k));
    G[c][2] = 0.5 * (F3(c, i, j, k + 1) - F3(c, i, j, k - 1));
#undef F3
  }
}

// physical coordinates of one vertex v = (x, y[, z], t) -> X = (x, y, z, t)
// (ref: critical_point_tracker_2d_regular.hh:494-526, critical_point_tracker_3d_regular.hh:343-379; the array domain starts at 0).
// The 3D explicit mode is the reference's as it stands: looked up by (x, y) only, and the time slot receives z.
// A z-slab looks its vertices up in the whole array's frame: z + voff[2], of coords_D planes.
template <int ND>
__device__ __forceinline__ void simplex_coordinates(const SweepParams &p, const int *v, double X[4]) {
  const int dims[3] = {p.W, p.H, p.coords_D};
  const int g[3] = {v[0], v[1], ND == 3 ? v[2] + p.voff[2] : v[2]};      // (2D: g[2] is the time)
  if (p.coords_mode == 1) {
#pragma unroll
    for (int j = 0; j < ND; j++)
      X[j] = ((double)g[j] / (double)(dims[j] - 1)) * (p.coords_bounds[2 * j + 1] - p.coords_bounds[2 * j]) + p.coords_bounds[2 * j];
    if (ND == 2) X[2] = 0.0;
    X[3] = (double)v[ND];
  } else if (p.coords_mode == 2) {
    int off = 0;
#pragma unroll
    for (int j = 0; j < ND; j++) { X[j] = __ldg(p.coords + off + g[j]); off += dims[j]; }
    if (ND == 2) X[2] = 0.0;
    X[3] = (double)v[ND];
  } else {
    const size_t nc = (size_t)p.coords_ncomp, k = (size_t)v[0] + (size_t)p.W * (size_t)v[1];
    X[0] = __ldg(p.coords + nc * k);
    X[1] = __ldg(p.coords + 1 + nc * k);
    if (ND == 2) X[2] = nc > 2 ? __ldg(p.coords + 2 + nc * k) : 0.0;
    else X[2] = __ldg(p.coords + 2 + nc * k);
    X[3] = (double)g[2];
  }
}

// SoS vertex rank: position in the mesh lattice (domain x time), uint64 truncated to int
// (ref: regular_tracker.hh:188-194, lattice.hh:196-207)
template <int ND>
__device__ __forceinline__ int sos_rank(const SweepParams &p, const int *v /* ND spatial + time */) {
  u64 prod = 1, i = 0;
#pragma unroll
  for (int j = 0; j <= ND; j++) {
    // (the whole lattice's frame: a spatial slab ranks its vertices as the undivided domain would)
    const u64 d = j < ND ? (u64)(i64)(v[j] + p.voff[j] - p.rank_lb[j]) : (u64)(i64)v[j];
    i += d * prod;
    if (j < ND) prod *= (u64)p.rank_nc[j];
  }
  return (int)(unsigned)i;
}

// vcache: the cube's 2^(ND+1) vertex vectors, [vertex mask][component], gathered once per cube by the block (test_kernel)
template <int ND>
__device__ bool check_simplex(const SweepParams &p, const DeviceMeshTables &mt, const int corner[3], int type, ftkb_point &cp, const double *vcache) {
  constexpr int NV = ND + 1;
  int vt[NV][ND + 1];
  const LayerPtrs *L[NV];
  size_t vi[NV];
  // vertices + validity (ref: simplicial_regular_mesh.hh:356-386)
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const int m = mt.vmask[type][k];
#pragma unroll
    for (int j = 0; j < ND; j++) {
      vt[k][j] = corner[j] + ((m >> j) & 1);
      if (vt[k][j] < p.lb[j] || vt[k][j] > p.ub[j]) return false;
    }
    const int dt = (m >> ND) & 1;
    vt[k][ND] = p.t + dt;
    if (vt[k][ND] < 0) return false;
    L[k] = &p.L[dt];
    vi[k] = ND == 2 ? (size_t)vt[k][0] + (size_t)p.W * (size_t)vt[k][1]
                    : (size_t)vt[k][0] + (size_t)p.W * ((size_t)vt[k][1] + (size_t)p.H * (size_t)vt[k][2]);
  }
  double v[NV][ND];
#pragma unroll
  for (int k = 0; k < NV; k++)
#pragma unroll
    for (int c = 0; c < ND; c++) v[k][c] = vcache[mt.vmask[type][k] * ND + c];

  double mu[NV];
  bool inside = false;
  if constexpr (ND == 3) inside = inverse_lerp3(v, mu);

  i64 vf[NV][ND];
  int rank[NV];
  if (ND == 2 || p.robust) {
#pragma unroll
    for (int k = 0; k < NV; k++)
#pragma unroll
      for (int c = 0; c < ND; c++) {
        if (isnan(v[k][c]) || isinf(v[k][c])) return false;
        vf[k][c] = quantise(v[k][c], p.factor);
      }
#pragma unroll
    for (int k = 0; k < NV; k++) rank[k] = sos_rank<ND>(p, vt[k]);
    // cheap exact exclusion on the quantised integers before the full cascade: one strictly
    // signed component, with magnitudes small enough that no determinant can leave int64
    {
      const i64 lim = ND == 2 ? (1ll << 29) : (1ll << 19);
      bool small = true, sided = false;
#pragma unroll
      for (int c = 0; c < ND; c++) {
        bool pos = true, neg = true;
#pragma unroll
        for (int k = 0; k < NV; k++) {
          pos = pos && vf[k][c] > 0;
          neg = neg && vf[k][c] < 0;
          small = small && vf[k][c] < lim && vf[k][c] > -lim;
        }
        sided = sided || pos || neg;
      }
      if (small && sided) return false;
    }
    if (!origin_in_simplex_fast(vf, rank)) return false;
  } else {
    if (!inside) return false;
  }

  if constexpr (ND == 2) {
    inside = inverse_lerp2(v, mu);
    if (!inside) clamp_barycentric<3>(mu);
  } else {
    clamp_barycentric<4>(mu);
  }

  // position / time: lerp of the vertex coordinates, ref linear_interpolation.hh:81-99
  double xo[4];
  if (p.coords_mode == 0) {     // REGULAR_COORDS_SIMPLE: the integer vertex coordinates
#pragma unroll
    for (int q = 0; q < 4; q++) {
      double acc;
      if constexpr (ND == 2) {
        const double c0 = q < 2 ? (double)(vt[0][q] + p.voff[q]) : (q == 2 ? 0.0 : (double)vt[0][2]);
        const double c1 = q < 2 ? (double)(vt[1][q] + p.voff[q]) : (q == 2 ? 0.0 : (double)vt[1][2]);
        const double c2 = q < 2 ? (double)(vt[2][q] + p.voff[q]) : (q == 2 ? 0.0 : (double)vt[2][2]);
        acc = c0 * mu[0] + c1 * mu[1] + c2 * mu[2];
      } else {
        const int og = q < ND ? p.voff[q < ND ? q : 0] : 0;      // a slab reports positions in the whole array's frame
        acc = (double)(vt[0][q] + og) * mu[0] + (double)(vt[1][q] + og) * mu[1] + (double)(vt[2][q] + og) * mu[2] + (double)(vt[ND][q] + og) * mu[ND];
      }
      xo[q] = acc;
    }
  } else {                      // bounds / rectilinear / explicit physical coordinates
    double X[ND + 1][4];
#pragma unroll
    for (int k = 0; k <= ND; k++) simplex_coordinates<ND>(p, vt[k], X[k]);
#pragma unroll
    for (int q = 0; q < 4; q++) {
      double acc = X[0][q] * mu[0] + X[1][q] * mu[1] + X[2][q] * mu[2];
      if constexpr (ND == 3) acc = acc + X[ND][q] * mu[ND];
      xo[q] = acc;
    }
  }
  cp.x[0] = xo[0]; cp.x[1] = xo[1]; cp.x[2] = xo[2]; cp.t = xo[3];

  cp.scalar = 0.0;
  if (p.scalar_source != FTKB_SOURCE_NONE) {
    double acc = __ldg(L[0]->S + vi[0]) * mu[0] + __ldg(L[1]->S + vi[1]) * mu[1] + __ldg(L[2]->S + vi[2]) * mu[2];
    if constexpr (ND == 3) acc = acc + __ldg(L[ND]->S + vi[ND]) * mu[ND];
    cp.scalar = acc;
  }
  cp.corner[0] = corner[0] + p.voff[0]; cp.corner[1] = corner[1] + p.voff[1];
  cp.corner[2] = ND == 3 ? corner[2] + p.voff[2] : 0;
  cp.corner[3] = p.t;
  cp.simplex_type = type;
  cp.ordinal = mt.ordinal[type];
  cp.timestep = p.t;

  if constexpr (ND == 2) {
    if (p.compute_degrees) {
      if (cp.ordinal) {
        int deg = oriented_sign<3, 2>(vf, rank);
        deg *= (type == 4) ? 1 : -1;
        cp.cp_type = deg == 1 ? 1 : 2;
      } else cp.cp_type = 0;
    } else {
      double J[2][2] = {{0, 0}, {0, 0}};
      if (p.jacobian_source != FTKB_SOURCE_NONE) {
        double Js[3][2][2];
#pragma unroll
        for (int k = 0; k < 3; k++) {
          if (L[k]->J) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
              for (int b = 0; b < 2; b++) Js[k][a][b] = __ldg(L[k]->J + b + 2 * (a + 2 * vi[k]));
          } else {
            double G[2][2];
            jacobian2d_at(p, *L[k], vt[k][0], vt[k][1], G);
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
              for (int b = 0; b < 2; b++) Js[k][a][b] = G[b][a];
          }
        }
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
          for (int b = 0; b < 2; b++) J[a][b] = Js[0][a][b] * mu[0] + Js[1][a][b] * mu[1] + Js[2][a][b] * mu[2];
        const double sym = 0.5 * (J[0][1] + J[1][0]);
        J[0][1] = J[1][0] = sym;
      }
      cp.cp_type = cp_type_2d(J, p.jacobian_symmetric != 0);
    }
    if (p.use_type_filter && !(p.type_filter & cp.cp_type)) return false;
  } else {
    double Js[4][3][3];
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
      if (L[k]->J) {
        for (int a = 0; a < 3; a++)
          for (int b = 0; b < 3; b++) Js[k][a][b] = __ldg(L[k]->J + b + 3 * (a + 3 * vi[k]));
      } else if (p.jacobian_source == FTKB_SOURCE_DERIVED) {
        double G[3][3];
        jacobian3d_at(p, *L[k], vt[k][0], vt[k][1], vt[k][2], G);
        for (int a = 0; a < 3; a++)
          for (int b = 0; b < 3; b++) Js[k][a][b] = G[b][a];
      } else {
        for (int a = 0; a < 3; a++)
          for (int b = 0; b < 3; b++) Js[k][a][b] = 0.0;
      }
    }
    double J[3][3];
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
      for (int b = 0; b < 3; b++) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 4; k++) acc += Js[k][a][b] * mu[k];
        J[a][b] = acc;
      }
    cp.cp_type = cp_type_3d(J, p.jacobian_symmetric != 0);
  }
  return true;
}

// A block works on CPB surviving cubes per round: the 2^(ND+1) vertices of every cube are gathered (the vector field
// read or derived ONCE per vertex -- a vertex is shared by up to 9 / 36 simplices of its cube), then one thread per
// (cube, simplex type) runs the exact test on the cached vectors.  The gather is software-pipelined: while round r is
// tested, the loads of round r + 1 are in flight (their results sit in registers until the test is over and then go into
// the other half of the cache), and the worklist entry of round r + 2 is on its way -- one barrier per round, and neither
// the worklist read nor the dependent field reads are waited for.
template <int ND>
struct VertexLoads {
  double a[ND], b[ND];        // component c = finish(a[c], b[c]): the value itself (vector input) or the two ends of a difference
  int corner[3];
  bool item, ok;              // this thread holds a (cube, vertex) item of the round / the vertex is one valid simplices use
};

template <int ND>
__device__ __forceinline__ void vertex_loads_issue(const SweepParams &p, const LayerPtrs &L, const int *vx, VertexLoads<ND> &g) {
  const int W = p.W, H = p.H;
  if constexpr (ND == 2) {
    const int i = clampi(vx[0], W), j = clampi(vx[1], H);
    if (L.V) {
      const double *v = L.V + 2 * ((size_t)i + (size_t)W * j);      // (8-byte loads: a borrowed layer need not be 16-byte aligned)
      g.a[0] = __ldg(v); g.a[1] = __ldg(v + 1); g.b[0] = g.b[1] = 0.0;
      return;
    }
#define SF(ii, jj) __ldg(L.S + (size_t)clampi(ii, W) + (size_t)W * clampi(jj, H))
    g.a[0] = SF(i + 1, j); g.b[0] = SF(i - 1, j);
    g.a[1] = SF(i, j + 1); g.b[1] = SF(i, j - 1);
#undef SF
  } else {
    const int D = p.D, i = vx[0], j = vx[1], k = vx[2];
    const size_t idx = (size_t)i + (size_t)W * ((size_t)j + (size_t)H * (size_t)k);
    if (L.V) {
#pragma unroll
      for (int c = 0; c < 3; c++) { g.a[c] = __ldg(L.V + c + 3 * idx); g.b[c] = 0.0; }
      return;
    }
    const bool interior = i >= 1 && i < W - 1 && j >= 1 && j < H - 1 && k >= 1 && k < D - 1;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const size_t st = c == 0 ? 1 : (c == 1 ? (size_t)W : (size_t)W * H);
      g.a[c] = interior ? __ldg(L.S + idx + st) : 0.0;
      g.b[c] = interior ? __ldg(L.S + idx - st) : 0.0;
    }
  }
}

// the arithmetic of vec2_at / vec3_at on the loaded values (same operations, same order)
template <int ND>
__device__ __forceinline__ double vertex_loads_finish(const SweepParams &p, const LayerPtrs &L, const VertexLoads<ND> &g, const int c) {
  if (L.V) return g.a[c];
  if constexpr (ND == 2) return (g.a[c] - g.b[c]) * (c == 0 ? p.W - 1 : p.H - 1);
  else return 0.5 * (g.a[c] - g.b[c]);
}

template <int ND>
__global__ void __launch_bounds__(128, ND == 2 ? 5 : 3) test_kernel(const __grid_constant__ SweepParams p) {
  const DeviceMeshTables &mt = c_mesh[ND - 2];
  constexpr int ntypes = ND == 2 ? 12 : 60;
  constexpr int NVC = 1 << (ND + 1);                  // vertices of a space-time cube
  constexpr int CPB = 128 / ntypes;                   // cubes per block and round (10 in 2D, 2 in 3D)
  static_assert(CPB * NVC <= 128, "one (cube, vertex) item per thread");
  __shared__ double vcache[2][CPB][NVC * ND];
  __shared__ int ccorner[2][CPB][3];
  u64 ncubes = *p.wl_count;
  if (ncubes > p.wl_cap) ncubes = p.wl_cap;
  const u64 stride = (u64)gridDim.x * CPB;
  const u64 rounds = (ncubes + stride - 1) / stride;
  const int lane = threadIdx.x & 31;
  const int gci = threadIdx.x / NVC, gm = threadIdx.x % NVC;       // this thread's gather item: cube gci of the round, vertex mask gm
  const bool gthread = (int)threadIdx.x < CPB * NVC;
  const int gdt = (gm >> ND) & 1;
  // worklist entry of this thread's cube in round r (all ones: none)
  auto wl_entry = [&](const u64 r) -> u64 {
    const u64 cube = r * stride + (u64)blockIdx.x * CPB + (u64)gci;
    return (gthread && r < rounds && cube < ncubes) ? p.wl[cube] : ~0ull;
  };
  auto issue = [&](u64 q, VertexLoads<ND> &g) {
    g.item = q != ~0ull;
    g.ok = false;
#pragma unroll
    for (int c = 0; c < ND; c++) { g.a[c] = 0.0; g.b[c] = 0.0; }
    if (!g.item) return;
    g.corner[0] = (int)(q % (u64)p.nc[0]) + p.lb[0]; q /= (u64)p.nc[0];
    g.corner[1] = (int)(q % (u64)p.nc[1]) + p.lb[1]; q /= (u64)p.nc[1];
    g.corner[2] = ND == 3 ? (int)q + p.lb[2] : 0;
    int vx[3] = {0, 0, 0};
    bool ok = true;
#pragma unroll
    for (int j = 0; j < ND; j++) { vx[j] = g.corner[j] + ((gm >> j) & 1); ok = ok && vx[j] >= p.lb[j] && vx[j] <= p.ub[j]; }
    ok = ok && (p.has_next || gdt == 0);              // (no second layer: the interval vertices belong to no simplex that is tested)
    g.ok = ok;
    if (ok) vertex_loads_issue<ND>(p, p.L[gdt], vx, g);   // a vertex outside the domain belongs to no valid simplex: never read
  };
  auto commit = [&](const int buf, const VertexLoads<ND> &g) {
    if (!g.item) return;
    if (gm == 0) { ccorner[buf][gci][0] = g.corner[0]; ccorner[buf][gci][1] = g.corner[1]; ccorner[buf][gci][2] = g.corner[2]; }
#pragma unroll
    for (int c = 0; c < ND; c++) vcache[buf][gci][gm * ND + c] = g.ok ? vertex_loads_finish<ND>(p, p.L[gdt], g, c) : 0.0;
  };

  int cur = 0;
  u64 qnext = ~0ull;
  {
    VertexLoads<ND> g0;
    issue(wl_entry(0), g0);
    qnext = wl_entry(1);
    commit(0, g0);
  }
  __syncthreads();
  for (u64 r = 0; r < rounds; r++) {
    const u64 cube0 = r * stride + (u64)blockIdx.x * CPB;
    // ---- round r + 1: field loads issued now, worklist entry of round r + 2 requested
    VertexLoads<ND> gn;
    issue(qnext, gn);
    qnext = wl_entry(r + 2);
    // ---- test: thread t -> (cube t / ntypes, type t % ntypes)
    bool hit = false;
    ftkb_point cp;
    {
      const int ci = threadIdx.x / ntypes, type = threadIdx.x % ntypes;
      if (ci < CPB && cube0 + (u64)ci < ncubes && (p.has_next || mt.ordinal[type])) {
        const int corner[3] = {ccorner[cur][ci][0], ccorner[cur][ci][1], ccorner[cur][ci][2]};
        hit = check_simplex<ND>(p, mt, corner, type, cp, vcache[cur][ci]);
      }
    }
    const unsigned b = __ballot_sync(0xffffffffu, hit);
    if (b) {
      u64 base = 0;
      const int leader = __ffs(b) - 1;
      if (lane == leader) base = atomicAdd(p.pt_count, (u64)__popc(b));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (hit) {
        const u64 o = base + __popc(b & ((1u << lane) - 1));
        if (o < p.pt_cap) p.pts[o] = cp;
      }
    }
    commit(cur ^ 1, gn);
    __syncthreads();                                  // round r + 1 is in the other half; this half is free again
    cur ^= 1;
  }
  if (p.step_out == nullptr) return;
  // deferred step: the last block to finish publishes the counters to the host (mapped memory) and re-arms the
  // device-side counters for the next step -- no copy, memset or host round trip sits between two sweeps
  __syncthreads();
  if (threadIdx.x != 0) return;
  __threadfence();
  if (atomicAdd(p.ticket, 1ull) != (u64)gridDim.x - 1) return;
  __threadfence();
  volatile unsigned long long *out = p.step_out;
  out[0] = *(volatile unsigned long long *)p.wl_count;
  out[1] = *(volatile unsigned long long *)p.pt_count;
  out[2] = *(volatile unsigned long long *)p.poison;
  out[3] = p.res_slot[0] ? *(volatile unsigned long long *)p.res_slot[0] : ~0ull;
  out[4] = p.res_slot[1] ? *(volatile unsigned long long *)p.res_slot[1] : ~0ull;
  out[5] = p.step_seq;
  // re-arm this step's set (the other set belongs to the next step, whose scan may be running already)
  *p.ticket = 0;
  *p.poison = 0;
  *p.wl_count = 0;
  if (p.res_reset) *p.res_reset = ~0ull;
  __threadfence_system();
}

void launch_test(const SweepParams &p, cudaStream_t s) {
  // the number of surviving cubes is only known on the device: grid sized by the caller from the previous step's count,
  // grid-stride loop over whatever the scan really left
  const unsigned grid = (unsigned)(p.test_blocks > 0 ? p.test_blocks : 148 * 8);
  if (p.nd == 2) test_kernel<2><<<grid, 128, 0, s>>>(p);
  else test_kernel<3><<<grid, 128, 0, s>>>(p);
}


// =============================================================================================
// 5. field derivation + resolution
// =============================================================================================
__device__ __forceinline__ void block_min_nonzero(double m, unsigned long long *res_bits) {
  // positive doubles order like their bit patterns
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ double sm[32];
  const int tid = threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z);
  const int nw = (blockDim.x * blockDim.y * blockDim.z + 31) >> 5;
  if ((tid & 31) == 0) sm[tid >> 5] = m;
  __syncthreads();
  if (tid < 32) {
    m = tid < nw ? sm[tid] : DBL_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (tid == 0 && m < DBL_MAX) atomicMin(res_bits, (unsigned long long)__double_as_longlong(m));
  }
}

__device__ __forceinline__ double nz_abs(double v) { const double a = fabs(v); return (v != 0.0 && !isnan(v)) ? a : DBL_MAX; }

// ref: grad.hh:10-31 (clamped one-sided borders, scaled by (DW-1)/(DH-1), no 1/2)
__global__ void __launch_bounds__(256) gradient2d_kernel(const double *__restrict__ S, double2 *__restrict__ V, int W, int H, unsigned long long *res_bits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
  double m = DBL_MAX;
  if (i < W && j < H) {
    const size_t row = (size_t)W * j;
    const double gx = (__ldg(S + row + clampi(i + 1, W)) - __ldg(S + row + clampi(i - 1, W))) * (W - 1);
    const double gy = (__ldg(S + (size_t)W * clampi(j + 1, H) + i) - __ldg(S + (size_t)W * clampi(j - 1, H) + i)) * (H - 1);
    V[row + i] = make_double2(gx, gy);
    m = fmin(nz_abs(gx), nz_abs(gy));
  }
  block_min_nonzero(m, res_bits);
}

// ref: grad.hh:130-149 (interior only, 1/2 central difference, border stays zero)
__global__ void __launch_bounds__(256) gradient3d_kernel(const double *__restrict__ S, double *__restrict__ V, int W, int H, int D, unsigned long long *res_bits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y, k = blockIdx.z;
  double m = DBL_MAX;
  if (i < W && j < H) {
    const size_t idx = (size_t)i + (size_t)W * ((size_t)j + (size_t)H * k);
    double g0 = 0.0, g1 = 0.0, g2 = 0.0;
    if (i >= 1 && i < W - 1 && j >= 1 && j < H - 1 && k >= 1 && k < D - 1) {
      const size_t sy = W, sz = (size_t)W * H;
      g0 = 0.5 * (__ldg(S + idx + 1) - __ldg(S + idx - 1));
      g1 = 0.5 * (__ldg(S + idx + sy) - __ldg(S + idx - sy));
      g2 = 0.5 * (__ldg(S + idx + sz) - __ldg(S + idx - sz));
    }
    V[3 * idx] = g0; V[3 * idx + 1] = g1; V[3 * idx + 2] = g2;
    m = fmin(nz_abs(g0), fmin(nz_abs(g1), nz_abs(g2)));
  }
  block_min_nonzero(m, res_bits);
}

void launch_gradient(int nd, const double *S, double *V, int W, int H, int D, unsigned long long *res_bits, cudaStream_t s) {
  const dim3 block(64, 4);
  if (nd == 2) {
    const dim3 grid((W + 63) / 64, (H + 3) / 4);
    gradient2d_kernel<<<grid, block, 0, s>>>(S, reinterpret_cast<double2 *>(V), W, H, res_bits);
  } else {
    const dim3 grid((W + 63) / 64, (H + 3) / 4, D);
    gradient3d_kernel<<<grid, block, 0, s>>>(S, V, W, H, D, res_bits);
  }
}

// ref: ndarray.hh:769-779 resolution(): min |p| over the non-zero entries
__global__ void __launch_bounds__(256) resolution_kernel(const double *__restrict__ p, u64 n, unsigned long long *res_bits) {
  double m = DBL_MAX;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) m = fmin(m, nz_abs(__ldg(p + i)));
  block_min_nonzero(m, res_bits);
}

void launch_resolution(const double *p, uint64_t n, unsigned long long *res_bits, cudaStream_t s) {
  const u64 blocks = (n + 255) / 256;
  const unsigned grid = (unsigned)(blocks < 148ull * 16 ? (blocks ? blocks : 1) : 148ull * 16);
  resolution_kernel<<<grid, 256, 0, s>>>(p, n, res_bits);
}

// float32 -> float64 widening of a snapshot that travelled as float32 (raw float32 file series: half the PCIe bytes)
__global__ void __launch_bounds__(256) widen_f32_kernel(const float4 *__restrict__ in, double *__restrict__ out, u64 n4, const float *__restrict__ tail_in, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (u64)gridDim.x * blockDim.x) {
    const float4 v = __ldg(in + i);
    reinterpret_cast<double2 *>(out)[2 * i] = make_double2((double)v.x, (double)v.y);
    reinterpret_cast<double2 *>(out)[2 * i + 1] = make_double2((double)v.z, (double)v.w);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) out[4 * n4 + threadIdx.x] = (double)tail_in[4 * n4 + threadIdx.x];
}
void launch_widen_f32(const float *in, double *out, uint64_t n, cudaStream_t s) {
  const u64 n4 = n / 4;
  const unsigned grid = (unsigned)std::max<u64>(1, std::min<u64>((n4 + 255) / 256, 148ull * 16));
  widen_f32_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const float4 *>(in), out, n4, in, n);
}

__global__ void fill_u64_kernel(unsigned long long *p, unsigned long long v) { *p = v; }
void launch_fill_u64(unsigned long long *p, unsigned long long v, cudaStream_t s) { fill_u64_kernel<<<1, 1, 0, s>>>(p, v); }

// =============================================================================================
// 6. synthetic generators (benchmark inputs; ref: include/ftk/ndarray/synthetic.hh)
// =============================================================================================
struct SynParams { double p[8]; };

__global__ void __launch_bounds__(256) synthetic_kernel(int kind, int nd, int W, int H, int Dg, SynParams sp, double t, double *__restrict__ out, int zoff) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y, kl = blockIdx.z;
  if (i >= W || j >= H) return;
  const size_t idx = (size_t)i + (size_t)W * ((size_t)j + (size_t)H * kl);
  const int k = kl + zoff, D = Dg;          // a slab generates its planes of the whole array
  const double kPi = 3.14159265358979323846;
  switch (kind) {
    case FTKB_SYN_MOVING_EXTREMUM: {   // synthetic.hh:332-354; pow(d, 2) is the correctly rounded square
      const int xi[3] = {i, j, k};
      double d = 0;
      for (int q = 0; q < nd; q++) {
        const double xc = sp.p[q] + sp.p[nd + q] * t;
        const double e = xi[q] - xc;
        d += e * e;
      }
      out[idx] = d;
    } break;
    case FTKB_SYN_WOVEN: {             // synthetic.hh:32-48, scaling_factor = 15
      const double x = (((double)i / (W - 1)) - 0.5) * 15, y = (((double)j / (H - 1)) - 0.5) * 15;
      out[idx] = cos(x * cos(t) - y * sin(t)) * sin(x * sin(t) + y * cos(t));
    } break;
    case FTKB_SYN_MERGER: {            // synthetic.hh:262-297
      double x = (((double)i / (W - 1)) - 0.5) * 4, y = (((double)j / (H - 1)) - 0.5) * 4;
      const double xp = x * cos(t) - y * sin(t), yp = x * sin(t) + y * cos(t);
      x = xp; y = yp;
      const double cx0 = sin(t - kPi / 2), cx1 = sin(t + kPi / 2), cy = 1e-4;
      const double f0 = exp(-((x - cx0) * (x - cx0) + (y - cy) * (y - cy))), f1 = exp(-((x - cx1) * (x - cx1) + (y - cy) * (y - cy)));
      out[idx] = std_max(f0, f1);
    } break;
    case FTKB_SYN_DOUBLE_GYRE: {       // synthetic.hh:130-150,193-217 on [0,2]x[0,1]
      const double A = sp.p[0], omega = sp.p[1], eps = sp.p[2];
      const double x = ((double)i / (W - 1)) * 2, y = ((double)j / (H - 1));
      const double a = eps * sin(omega * t), b = 1 - 2 * eps * sin(omega * t);
      const double f = a * x * x + b * x, dfdx = 2 * a * x + b;
      out[2 * idx] = -kPi * A * sin(kPi * f) * cos(kPi * y);
      out[2 * idx + 1] = kPi * A * cos(kPi * f) * sin(kPi * y) * dfdx;
    } break;
    case FTKB_SYN_TORNADO: {           // synthetic.hh:441-494; t = integer time step
      const double SMALL = 0.00000000001;
      const double x = i * (1.0 / (W - 1.0)), y = j * (1.0 / (H - 1.0)), z = k * (1.0 / (D - 1.0));
      const double xc = 0.5 + 0.1 * sin(0.04 * t + 10.0 * z), yc = 0.5 + 0.1 * cos(0.03 * t + 3.0 * z);
      const double r = 0.1 + 0.4 * z * z + 0.1 * z * sin(8.0 * z), r2 = 0.2 + 0.1 * z;
      double temp = sqrt((y - yc) * (y - yc) + (x - xc) * (x - xc));
      double scale = fabs(r - temp);
      scale = scale > r2 ? 0.8 - scale : 1.0;
      double z0 = 0.1 * (0.1 - temp * z);
      if (z0 < 0.0) z0 = 0.0;
      temp = sqrt(temp * temp + z0 * z0);
      scale = (r + r2 - temp) * scale / (temp + SMALL);
      scale = scale / (1 + z);
      out[3 * idx] = scale * (y - yc) + 0.1 * (x - xc);
      out[3 * idx + 1] = scale * -(x - xc) + 0.1 * (y - yc);
      out[3 * idx + 2] = scale * z0;
    } break;
    case FTKB_SYN_ABC: {               // synthetic.hh:239-260 on [0, 2 pi]^3
      const double A = sp.p[0], B = sp.p[1], C = sp.p[2];
      const double x = (((double)i / (W - 1))) * 2 * kPi, y = (((double)j / (H - 1))) * 2 * kPi, z = (((double)k / (D - 1))) * 2 * kPi;
      out[3 * idx] = A * sin(z) + C * cos(y);
      out[3 * idx + 1] = B * sin(x) + A * cos(z);
      out[3 * idx + 2] = C * sin(y) + B * cos(x);
    } break;
  }
}

void launch_synthetic(int kind, int nd, int W, int H, int D, const double *params, double t, double *out, cudaStream_t s, int zoff, int Dg) {
  SynParams sp;
  for (int i = 0; i < 8; i++) sp.p[i] = params[i];
  const dim3 block(64, 4), grid((W + 63) / 64, (H + 3) / 4, D);
  synthetic_kernel<<<grid, block, 0, s>>>(kind, nd, W, H, Dg > 0 ? Dg : D, sp, t, out, zoff);
}

// =============================================================================================
// 7. trajectory construction: element keys, neighbour search, union-find
// =============================================================================================
// element key = reference element order (corner compared x first, then y[, z], t, then type;
// simplicial_regular_mesh.hh:327-337) packed into 64 bits
__device__ __forceinline__ bool element_key(const TraceParams &tp, int x, int y, int z, int t, int type, u64 &key) {
  if (x < tp.lb[0] || x > tp.ub[0] || y < tp.lb[1] || y > tp.ub[1] || t < 0 || t >= (1 << KEY_TIME_BITS)) return false;
  if (tp.nd == 3 && (z < tp.lb[2] || z > tp.ub[2])) return false;
  u64 k = (u64)(x - tp.lb[0]);
  k = k * (u64)tp.ny + (u64)(y - tp.lb[1]);
  k = k * (u64)tp.nz + (u64)(tp.nd == 3 ? z - tp.lb[2] : 0);
  k = (k << KEY_TIME_BITS) | (u64)t;
  key = (k << KEY_TYPE_BITS) | (u64)type;
  return true;
}

__global__ void point_keys_kernel(const ftkb_point *__restrict__ pts, u64 n, TraceParams tp, u64 *keys, uint32_t *idx) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 k = ~0ull;
  element_key(tp, pts[i].corner[0], pts[i].corner[1], pts[i].corner[2], pts[i].corner[3], pts[i].simplex_type, k);
  keys[i] = k;
  idx[i] = (uint32_t)i;
}

void launch_point_keys(const ftkb_point *pts, uint64_t n, const TraceParams &tp, unsigned long long *keys, uint32_t *idx, cudaStream_t s) {
  if (n) point_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pts, n, tp, keys, idx);
}

__global__ void gather_points_kernel(const ftkb_point *__restrict__ src, const uint32_t *__restrict__ idx, u64 n, ftkb_point *dst) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}

void launch_gather_points(const ftkb_point *src, const uint32_t *idx, uint64_t n, ftkb_point *dst, cudaStream_t s) {
  if (n) gather_points_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, idx, n, dst);
}

// neighbours of a punctured simplex = the other facets of its two cofaces that are punctured too
// (ref: critical_point_tracker_2d_regular.hh:189-197); found by binary search in the sorted keys
__global__ void neighbors_kernel(TraceParams tp) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tp.n) return;
  const DeviceMeshTables &mt = c_mesh[tp.nd - 2];
  const ftkb_point pt = tp.pts[i];
  const int type = pt.simplex_type;
  uint32_t found[8];
  int cnt = 0;
  for (int q = 0; q < mt.n_nb[type]; q++) {
    const int x = pt.corner[0] + mt.nb_off[type][q][0], y = pt.corner[1] + mt.nb_off[type][q][1];
    const int z = tp.nd == 3 ? pt.corner[2] + mt.nb_off[type][q][2] : 0;
    const int t = pt.corner[3] + mt.nb_off[type][q][tp.nd];
    u64 key;
    if (!element_key(tp, x, y, z, t, mt.nb_type[type][q], key)) continue;
    u64 lo = 0, hi = tp.n;
    while (lo < hi) {
      const u64 mid = (lo + hi) >> 1;
      if (tp.keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < tp.n && tp.keys[lo] == key) found[cnt++] = (uint32_t)lo;
  }
  // ascending order (= element order); candidates are distinct elements
  for (int a = 1; a < cnt; a++)
    for (int b = a; b > 0 && found[b - 1] > found[b]; b--) { const uint32_t t = found[b]; found[b] = found[b - 1]; found[b - 1] = t; }
  for (int q = 0; q < 8; q++) tp.nb[i * 8 + q] = q < cnt ? found[q] : 0xffffffffu;
  tp.deg[i] = cnt;
  tp.parent_all[i] = (uint32_t)i;
  tp.parent_ord[i] = (uint32_t)i;
}

void launch_neighbors(const TraceParams &tp, cudaStream_t s) {
  if (tp.n) neighbors_kernel<<<(unsigned)((tp.n + 127) / 128), 128, 0, s>>>(tp);
}

// streaming grow step (online.cpp: OnlineTracer::grow_sorted): the step's batch, sorted and unique; thread i moves point
// idx[i] into place (dst != nullptr) and lists the batch indices of its punctured neighbours in ascending element order, ITSELF INCLUDED
// (the reference unites an element with itself, which is visible in its union-find sizes).  *n_ptr = unique elements.
__global__ void batch_neighbors_kernel(TraceParams tp, const u64 *__restrict__ n_ptr, const ftkb_point *__restrict__ src,
                                       const uint32_t *__restrict__ idx, ftkb_point *dst, uint32_t *nb9, uint8_t *cnt_out) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const u64 n = *n_ptr;
  if (i >= n) return;
  const DeviceMeshTables &mt = c_mesh[tp.nd - 2];
  const ftkb_point &pt = src[idx[i]];
  if (dst) dst[i] = pt;
  const int type = pt.simplex_type;
  uint32_t found[9];
  int cnt = 0;
  found[cnt++] = (uint32_t)i;
  for (int q = 0; q < mt.n_nb[type]; q++) {
    const int x = pt.corner[0] + mt.nb_off[type][q][0], y = pt.corner[1] + mt.nb_off[type][q][1];
    const int z = tp.nd == 3 ? pt.corner[2] + mt.nb_off[type][q][2] : 0;
    const int t = pt.corner[3] + mt.nb_off[type][q][tp.nd];
    u64 key;
    if (!element_key(tp, x, y, z, t, mt.nb_type[type][q], key)) continue;
    u64 lo = 0, hi = n;
    while (lo < hi) {
      const u64 mid = (lo + hi) >> 1;
      if (tp.keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < n && tp.keys[lo] == key) found[cnt++] = (uint32_t)lo;
  }
  for (int a = 1; a < cnt; a++)
    for (int b = a; b > 0 && found[b - 1] > found[b]; b--) { const uint32_t t = found[b]; found[b] = found[b - 1]; found[b - 1] = t; }
  for (int q = 0; q < 9; q++) nb9[i * 9 + q] = q < cnt ? found[q] : 0xffffffffu;
  cnt_out[i] = (uint8_t)cnt;
}

void launch_batch_neighbors(const TraceParams &tp, const unsigned long long *n_ptr, uint64_t n_max, const ftkb_point *src, const uint32_t *idx,
                            ftkb_point *dst, uint32_t *nb9, uint8_t *cnt, cudaStream_t s) {
  if (n_max) batch_neighbors_kernel<<<(unsigned)((n_max + 127) / 128), 128, 0, s>>>(tp, n_ptr, src, idx, dst, nb9, cnt);
}

// union-find with atomicMin hooking: the larger root is hooked under the smaller one, so the root of
// every tree is its smallest member (the reference's duf hooks the same way, basic/duf.hh:41-72)
__device__ __forceinline__ uint32_t uf_find(uint32_t *parent, uint32_t i) {
  uint32_t p = parent[i];
  while (p != i) {
    const uint32_t g = parent[p];
    if (g != p) atomicMin(parent + i, g);   // path halving; parents only ever decrease towards the root
    i = p;
    p = g;
  }
  return i;
}

__device__ void uf_unite(uint32_t *parent, uint32_t a, uint32_t b) {
  while (true) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const uint32_t t = a; a = b; b = t; }
    const uint32_t old = atomicMin(parent + a, b);
    if (old == a) return;
    a = old;
  }
}

__global__ void uf_hook_kernel(TraceParams tp) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tp.n) return;
  const bool special = tp.deg[i] > 2;
  for (int q = 0; q < 8; q++) {
    const uint32_t j = tp.nb[i * 8 + q];
    if (j == 0xffffffffu) break;
    if (j < i) continue;                       // each edge once
    uf_unite(tp.parent_all, (uint32_t)i, j);
    if (!special && tp.deg[j] <= 2) uf_unite(tp.parent_ord, (uint32_t)i, j);
  }
}

// pointer jumping to the root
__global__ void uf_flatten_kernel(TraceParams tp) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tp.n) return;
  uint32_t r = tp.parent_all[i];
  while (tp.parent_all[r] != r) r = tp.parent_all[r];
  uint32_t o = tp.parent_ord[i];
  while (tp.parent_ord[o] != o) o = tp.parent_ord[o];
  tp.parent_all[i] = r;
  tp.parent_ord[i] = o;
}

void launch_union_find(const TraceParams &tp, cudaStream_t s) {
  if (!tp.n) return;
  const unsigned grid = (unsigned)((tp.n + 127) / 128);
  uf_hook_kernel<<<grid, 128, 0, s>>>(tp);
  uf_flatten_kernel<<<grid, 128, 0, s>>>(tp);
}

// ---- cub wrappers ---------------------------------------------------------------------------------
size_t sort_pairs_u64(void *temp, size_t temp_bytes, const unsigned long long *kin, unsigned long long *kout,
                      const uint32_t *vin, uint32_t *vout, uint64_t n, cudaStream_t s) {
  size_t bytes = temp_bytes;
  cub::DeviceRadixSort::SortPairs(temp, bytes, kin, kout, vin, vout, (int64_t)n, 0, 64, s);
  return bytes;
}

size_t unique_by_key_u64(void *temp, size_t temp_bytes, const unsigned long long *kin, const uint32_t *vin,
                         unsigned long long *kout, uint32_t *vout, unsigned long long *n_out, uint64_t n, cudaStream_t s) {
  size_t bytes = temp_bytes;
  cub::DeviceSelect::UniqueByKey(temp, bytes, kin, vin, kout, vout, n_out, (int64_t)n, s);
  return bytes;
}

}  // namespace ftkb

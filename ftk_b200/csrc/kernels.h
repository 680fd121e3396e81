// Kernel parameter blocks and launchers (host-callable).  Device code lives in kernels.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/ftkb200.h"
#include "mesh_tables.h"

namespace ftkb {

// One resident time layer (device pointers; any may be null)
struct LayerPtrs {
  const double *S;  // (W,H[,D])
  const double *V;  // (n,W,H[,D])
  const double *J;  // (n,n,W,H[,D]) only when the Jacobian is GIVEN
};

struct SweepParams {
  int32_t nd;                 // 2 or 3
  int32_t W, H, D;            // array dims (D = 1 in 2D)
  int32_t lb[3], ub[3];       // domain (inclusive)
  int32_t nc[3];              // corners per dimension = ub - lb + 1 (1 for the unused dim)
  int32_t vmax[3];            // last vertex that enters a cube's value range per dim (= ub)
  // global frame of a spatial slab (all zero / equal to lb, nc when the context is not a slab): offset of the local array in
  // the whole one, and the whole domain's lower bound / extent -- SoS vertex rank, interpolated position, reported corner
  int32_t voff[3], rank_lb[3], rank_nc[3];
  int32_t t;                  // current timestep (time of layer 0)
  int32_t has_next;           // layer 1 present -> interval simplices are swept too
  int32_t nbits;              // factor = 2^nbits
  double factor;
  int32_t no_filter;          // 3D with robust detection off: every cube is refined
  // sources / options (see ftkb_config)
  int32_t scalar_source, jacobian_source, jacobian_symmetric, derived_symmetric;
  int32_t robust, compute_degrees, use_type_filter;
  uint32_t type_filter;
  LayerPtrs L[2];
  // physical coordinates of the vertices (regular_tracker.hh:12-17,38-40): 0 grid units, 1 bounds, 2 rectilinear, 3 explicit
  int32_t coords_mode, coords_ncomp;
  double coords_bounds[6];
  const double *coords;       // device: rectilinear x[W] y[H] [z[D]], or explicit (ncomp, W, H)
  // fused mode: the vector field is derived from the scalar layers on the fly (L[].V == nullptr)
  int32_t fused;
  int32_t keys2d;             // 2D scalar build: high-word keys of the differences instead of fp32 ranges (scan2d_keys_build_kernel)
  float thrp_f;               // 2^-nbits (1 + 2^-20): approx(v) >= thrp_f  =>  |quantised v| >= 1
  float thr2_f;               // 2^(1-nbits)
  float lim_f;                // 0.999 * 4.5e18 / factor^2 (determinant magnitude bound, field units)
  unsigned long long *res_slot[2];   // non-null: accumulate min non-zero |v| of that layer during the scan
  // key filter of that accumulation (scalar build kernels): a difference d (v = d * scale of the component) whose high-word key
  // exceeds res_thr[component] cannot lower the running minimum known when the step was enqueued; +inf: nothing is known yet.
  // What the slot then receives is the minimum over the values under the threshold -- equal to the layer's own minimum whenever
  // that one would lower the running minimum, which is all the tracker uses it for.
  float res_thr[3];
  unsigned long long *poison;        // fused 3D scan: set non-zero when a scalar is NaN / Inf / >= 2^1000 (the sweep is redone unfused)
  // fused 3D scan: TMA descriptors of the two scalar layers (box = one tile plane incl. halo)
  alignas(64) CUtensorMap tmap[2];
  // fused 3D scan, summary path: 16-byte range cells per (tile, warp, plane, lane), one buffer per layer
  int32_t sum_mode;                  // SUM_*: what this launch does
  int32_t build_layer;               // which of L[0] / L[1] (tmap, res_slot) the build streams
  const uint4 *sum_in[2];            // cells read (layer order as L[])
  uint4 *sum_out;                    // cells written by a build
  // scan decomposition
  int32_t nsx;                // x strips (31 corners each)
  int32_t nsy;                // 2D: row chunks; 3D: y tiles (BY-1 corners each)
  int32_t nsz;                // 3D: z chunks
  int32_t rows;               // corner rows (2D) / corner planes (3D) per chunk
  // worklist of surviving cubes (linear corner index, x fastest over the domain)
  unsigned long long *wl_count;
  unsigned long long wl_cap;
  unsigned long long *wl;
  // output
  unsigned long long *pt_count;
  unsigned long long pt_cap;
  ftkb_point *pts;
  // deferred step (context.cpp, "sync-free step"): the test kernel's last block publishes the step's counters into
  // mapped host memory and re-arms the device counters for the next step, so that the host never has to touch the
  // stream between two sweeps.  step_out == nullptr: the host resets / reads the counters itself (synchronous step).
  unsigned long long *step_out;      // mapped pinned host memory: {worklist count, point count, poison, res[0], res[1], sequence}
  unsigned long long step_seq;
  unsigned long long *ticket;        // blocks of the test kernel that are done
  unsigned long long *res_reset;     // resolution slot to re-arm (all ones) for the step after next, or nullptr
  int32_t test_blocks;               // grid of the test kernel (grid-stride: any worklist size is covered)
  int32_t sm_count;                  // SMs of the device (persistent kernels size their grid by it)
};

// threshold key for SweepParams::res_thr: R = running minimum of the non-zero |v| (DBL_MAX: unknown), v = d * scale
inline float res_threshold_key(double R, double scale) {
  if (!(R < 0x1p1000) || !(scale > 0.0)) return __builtin_inff();
  const double T = R / scale;
  unsigned long long bits;
  __builtin_memcpy(&bits, &T, 8);
  const int hi = (int)(bits >> 32) + 2;     // two key units (2^-19 relative) above T: far beyond the rounding of T and of d * scale
  float f;
  __builtin_memcpy(&f, &hi, 4);
  return f;
}

void upload_mesh_tables(const DeviceMeshTables &t2, const DeviceMeshTables &t3);
void init_kernel_attributes();   // opt-in shared memory sizes; once per device

// fused 3D scan geometry (host needs it for the grid decomposition and the TMA box)
constexpr int F3_CW = 8;                       // consumer warps per CTA
constexpr int F3_RW = 4;                       // corner rows per consumer warp
constexpr int F3_STRIDE = 62;                  // corner columns per tile
constexpr int F3_COLS = 68;                    // staged columns: C0-2 .. C0+65
constexpr int F3_TROWS = F3_CW * F3_RW;        // corner rows per tile
constexpr int F3_ROWS = F3_TROWS + 3;          // staged rows: Y0-1 .. Y0+TROWS+1
// encode the TMA descriptor of one scalar layer (W,H,D) fp64 for the fused 3D scan; false if the driver
// entry point is unavailable or the layer does not meet TMA's alignment rules
bool encode_scalar_tmap3d(const double *S, int W, int H, int D, CUtensorMap *out);

void launch_scan(const SweepParams &p, cudaStream_t s);
// summary path of the fused 3D scan
enum { SUM_BUILD = 0,          // stream layer build_layer, write its cells (+ min |v|); no cube is tested
       SUM_BUILD_TEST1 = 1,    // ... and test the ordinal cubes of that single layer (single-snapshot sweep)
       SUM_BUILD_TEST2 = 2,    // stream L[1], write its cells, read L[0]'s cells, test the cubes over both layers
       SUM_TEST1 = 3,          // cells of L[0] only (final ordinal sweep, repeats)
       SUM_TEST2 = 4 };        // cells of L[0] and L[1] (repeats)
void launch_scan3d_cells(const SweepParams &p, cudaStream_t s);
size_t scan3d_cells_per_layer(const SweepParams &p);
constexpr int SCAN2D_CELL_ROWS = 9;
void launch_scan2d_cells(const SweepParams &p, cudaStream_t s);     // needs 16-byte aligned rows, the CTA tiling of 7 strips and p.rows a multiple of SCAN2D_CELL_ROWS
size_t scan2d_cells_per_layer(const SweepParams &p);
// vector input (field GIVEN): p.fused == 0, p.L[].V set; 2D needs p.nsx = strips of 62 columns and p.rows a multiple of 8,
// 3D the tile / chunk geometry of the fused 3D scan and W even
constexpr int VSCAN2D_CELL_ROWS = 8;
void launch_vscan_cells(const SweepParams &p, cudaStream_t s);
size_t vscan2d_cells_per_layer(const SweepParams &p);
// thread-per-(surviving cube, type) exact test; grid sized for `expected` cubes, grid-stride otherwise
void launch_test(const SweepParams &p, cudaStream_t s);

// field derivation (ref: include/ftk/ndarray/grad.hh) + min non-zero |v| (ndarray.hh:769-779).
// res_bits: the running minimum as the bit pattern of a positive double (atomicMin on u64).
void launch_gradient(int nd, const double *S, double *V, int W, int H, int D, unsigned long long *res_bits, cudaStream_t s);
void launch_resolution(const double *p, uint64_t n, unsigned long long *res_bits, cudaStream_t s);
void launch_fill_u64(unsigned long long *p, unsigned long long v, cudaStream_t s);
void launch_widen_f32(const float *in, double *out, uint64_t n, cudaStream_t s);   // in, out 16-byte aligned

// synthetic generators (ref: include/ftk/ndarray/synthetic.hh); out is S (scalar kinds) or V (vector kinds)
// zoff / Dg: the slab's first plane and the whole array's depth (3D; zoff = 0, Dg = D when the context is not a slab)
void launch_synthetic(int kind, int nd, int W, int H, int D, const double *params, double t, double *out, cudaStream_t s, int zoff = 0, int Dg = 0);

// finalize
struct TraceParams {
  int32_t nd;
  int32_t lb[3], ub[3];
  int64_t ny, nz;             // domain extents used by the element key
  uint64_t n;                 // number of (sorted, unique) points
  const unsigned long long *keys;   // sorted
  const ftkb_point *pts;            // sorted
  uint32_t *nb;               // n * 8 neighbour indices (ascending), 0xffffffff padded
  int32_t *deg;
  uint32_t *parent_all;       // union-find over every punctured simplex
  uint32_t *parent_ord;       // union-find over ordinary nodes (degree <= 2)
};
constexpr int KEY_TYPE_BITS = 6;
constexpr int KEY_TIME_BITS = 22;

void launch_point_keys(const ftkb_point *pts, uint64_t n, const TraceParams &tp, unsigned long long *keys, uint32_t *idx, cudaStream_t s);
void launch_gather_points(const ftkb_point *src, const uint32_t *idx, uint64_t n, ftkb_point *dst, cudaStream_t s);
void launch_neighbors(const TraceParams &tp, cudaStream_t s);
void launch_union_find(const TraceParams &tp, cudaStream_t s);
// streaming grow step: tp.keys = the batch's sorted unique keys, *n_ptr of them (n_max bounds the grid); writes the sorted points (dst may be nullptr),
// nine neighbour indices per element (ascending, itself included, 0xffffffff padded) and how many
void launch_batch_neighbors(const TraceParams &tp, const unsigned long long *n_ptr, uint64_t n_max, const ftkb_point *src, const uint32_t *idx,
                            ftkb_point *dst, uint32_t *nb9, uint8_t *cnt, cudaStream_t s);

// cub wrappers (sort by key, then drop duplicate keys); return bytes of temp storage needed when temp == nullptr
size_t sort_pairs_u64(void *temp, size_t temp_bytes, const unsigned long long *kin, unsigned long long *kout,
                      const uint32_t *vin, uint32_t *vout, uint64_t n, cudaStream_t s);
size_t unique_by_key_u64(void *temp, size_t temp_bytes, const unsigned long long *kin, const uint32_t *vin,
                         unsigned long long *kout, uint32_t *vout, unsigned long long *n_out, uint64_t n, cudaStream_t s);

}  // namespace ftkb

// K1 — Karto correlative scan matcher on B200 (sm_100a).  Product code: CUDA only, no CPU fallback.
//
// Reference behaviour (paths relative to /root/reference/lesson6/lib/open_karto):
//   ScanMatcher::Create / MatchScan / CorrelateScan / GetResponse / AddScans / FindValidPoints  src/Mapper.cpp:126-856
//   CorrelationGrid (smear kernel, ROI)                                   include/open_karto/Mapper.h:900-1118
//   GridIndexLookup::ComputeOffsets, Grid<T>, CoordinateConverter          include/open_karto/Karto.h:6409-6501, 4209-4767
//   LocalizedRangeScan::Update (point readings)                            include/open_karto/Karto.h:5362-5428
//
// Data layout in HBM (per handle, B = batch capacity, N = beams):
//   grids   [B][grid_pitch] u8      one correlation grid per match, same flat row-major layout as the reference
//                                   (index = x + y*width_step); grid_pitch = data_size rounded up to 128 B (+pad, zero)
//   lut     [B][nA][N]      i32     per-angle flat offsets (GridIndexLookup), INT32_MAX = INVALID_SCAN
//   sums    [B][nA][nY][nX] i32     integer numerators of GetResponse for the whole (x,y,theta) volume
//   probs   [B][side*side]  f64     per-cell maximum over theta (m_pSearchSpaceProbs)
//
// Kernels:
//   k_scan_points      point readings + scan-local points                              (fp64, O(B*N))
//   k_add_scan         FindValidPoints state machine + rasterise + max-smear           (byte atomics, O(B*S*N))
//   k_offsets          per-angle lookup tables                                         (fp64 -> i32)
//   k_sweep_window     THE HOT KERNEL: whole grid staged into shared memory by TMA bulk copy; one warp per
//                      angle, one lane per candidate row; each 32-bit shared-memory word feeds 4 adjacent-x
//                      candidates (byte-permute into packed u16 accumulators)           (int, smem-gather bound)
//   k_sweep_generic    any lattice / any grid size: one warp per (x,y) candidate, lanes over beams,
//                      gathers from global memory through L1/L2
//   k_reduce           penalties, best response, tie-averaged pose, positional covariance (fp64, one CTA per match)
//   k_angular_cov      fine-stage angular covariance (re-evaluates GetResponse at the best cell)
#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include <math_constants.h>

#include "common.cuh"
#include "nccl_dl.cuh"
#include "scan_kernels.cuh"

namespace b2s {

static thread_local std::string g_last_error;
void set_last_error(const std::string &s) { g_last_error = s; }
std::string &last_error_ref() { return g_last_error; }

// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t addr = smem_u32(bar);
  while (!done) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// PRMT, default mode: selector nibble bit 3 replicates the sign bit of the selected byte.  Grid bytes are
// <= 100 < 128, so a "sign-replicated" byte is 0x00: one PRMT extracts two bytes into packed u16 lanes.
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

// per-byte atomic max on a u8 array (no native byte atomics): CAS on the containing aligned word
// returns the byte's previous value
__device__ __forceinline__ uint32_t atomic_max_u8(uint8_t *base, int idx, uint32_t val) {
  uint32_t *w = reinterpret_cast<uint32_t *>(base + (idx & ~3));
  uint32_t shift = (idx & 3) * 8;
  uint32_t v = val << shift;
  uint32_t old = *w, assumed;
  do {
    if (((old >> shift) & 0xffu) >= val) return (old >> shift) & 0xffu;
    assumed = old;
    old = atomicCAS(w, assumed, __vmaxu4(assumed, v));
  } while (assumed != old);
  return (old >> shift) & 0xffu;
}

// ----------------------------------------------------------------------------------------------
// handle
// ----------------------------------------------------------------------------------------------

struct SweepDims {
  int nx = 0, ny = 0, na = 0;
};

// launch configuration of the last k_sweep_window call (re-run densely when the full volume is asked for)
struct WinLaunch {
  int stride = 1;
  bool gen = false;
  size_t smem = 0;
  int ctas = 0, copy_bytes = 0, band_rows = 0, nbands = 1, band_bytes = 0, neg_bands = 0;
};

}  // namespace b2s

using namespace b2s;

struct b2s_matcher {
  b2s_matcher_params p;
  b2s_laser l;
  b2s_grid_info g;
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int max_batch = 0, max_base = 0;
  int batch = 0, n = 0, n_base = 0;
  bool scans_set = false, grids_set = false;
  bool smear_degenerate = false;  // an off-centre kernel value reaches 100: AddScan becomes order-dependent
  size_t grid_pitch = 0;
  int force_kernel = 0;
  int num_sms = 148;
  int smem_optin = 0;

  uint8_t *d_kernel = nullptr;
  double *d_ranges = nullptr, *d_poses = nullptr, *d_sensor = nullptr, *d_pts = nullptr, *d_local = nullptr;
  uint8_t *d_grids = nullptr;
  double *d_grid_off = nullptr;
  double *d_base_ranges = nullptr, *d_base_poses = nullptr, *d_base_pts = nullptr;
  size_t base_cap = 0;
  double *d_pool = nullptr;        // scan pool: readings of scans that serve as base scans again and again
  size_t pool_cap = 0, pool_count = 0;
  int32_t *d_base_src = nullptr;   // [batch * n_base] pool rows of the current base sets
  size_t base_src_cap = 0;
  int32_t *d_lut = nullptr;
  size_t lut_cap = 0;
  int32_t *d_lists = nullptr, *d_counts = nullptr, *d_starts = nullptr;  // window kernel: per-(match, angle) grouped window origins
  size_t lists_cap = 0, counts_cap = 0, starts_cap = 0;
  double *d_part_best = nullptr, *d_glob_best = nullptr, *d_tie = nullptr;  // split-sweep phases: [B], [B], [B][5]
  int32_t *d_status = nullptr;                                              // [B] statuses of a split sweep
  cudaEvent_t ev_split[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double last_split_ms[4] = {0, 0, 0, 0};
  int last_k_first = 0;
  uint16_t *d_sat = nullptr;  // [B][(sby+1)(sbx+1)] block summed-area tables of the grids
  int sbx = 0, sby = 0;
  bool sat_valid = false;
  unsigned long long *d_stats = nullptr;  // [0] beam-angle pairs dropped as empty windows in the last sweep,
                                          // [1] (match, angle) pairs k_prune_select kept
  unsigned long long *h_stats = nullptr;  // pinned copy, read back with the results
  uint8_t *d_mp4 = nullptr;               // [B][mp_pitch] phase-split 4x4 max-pool images (k_grid_mp4)
  size_t mp_pitch = 0;
  int mp_guard = 0, mp_lq = 0;
  bool mp_valid = false;
  int32_t *d_keep = nullptr, *d_nkeep = nullptr;  // [B][na], [B]: angles a pruned sweep visits
  size_t keep_cap = 0, nkeep_cap = 0;
  bool last_pruned = false;  // the last sweep visited only the kept angles: d_sums holds only those
  bool sums_dense = false;   // d_sums holds every angle of the last sweep
  WinLaunch win;
  double last_prune[2] = {1.0, 0.0};
  bool pending = false;                   // a correlate_scan_begin awaits its _end
  int pending_batch = 0;                  // batch size that _begin enqueued
  double last_empty_frac = 0.0;
  bool grid_high_bytes = false;  // set_grids saw a byte > 127: the packed-byte window kernel is not applicable
  int32_t *d_sums = nullptr;
  size_t sums_cap = 0;
  int32_t *d_bases = nullptr;  // [B][ny*nx] candidate base indices
  size_t bases_cap = 0;
  int32_t *d_flags = nullptr;  // [B] per-match: bit0 lattice regular stride-1, bits 8.. status
  double *d_probs = nullptr;
  double *d_centers = nullptr;
  b2s_match_result *d_results = nullptr;
  b2s_match_result *h_results = nullptr;  // pinned
  int *d_work = nullptr;                   // persistent-CTA work counter
  SweepDims last;
  b2s_search last_search;
  bool have_sweep = false;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  double last_ms[4] = {0, 0, 0, 0};
  int last_path = 0;
};

namespace b2s {

// MatchScan steps 2-4 (Mapper.cpp:212-220): grid offset so that the ROI centre is the scan's sensor position
__global__ void k_grid_offsets(const double *__restrict__ sensor, double *__restrict__ grid_off, int batch, int roi_w,
                               int roi_h, double resolution) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  grid_off[2 * b] = sensor[3 * b] - (0.5 * (double)(roi_w - 1) * resolution);
  grid_off[2 * b + 1] = sensor[3 * b + 1] - (0.5 * (double)(roi_h - 1) * resolution);
}

// ----------------------------------------------------------------------------------------------
// k_add_scan: ScanMatcher::AddScan (Mapper.cpp:716-748) for one (match, base scan) per block:
// the FindValidPoints state machine (Mapper.cpp:756-811) runs over points staged in shared memory (see below),
// then all threads rasterise the valid points and max-stamp the smear kernel (Mapper.h:971-1005).
// The result is a per-byte maximum, hence independent of the order in which points / scans are applied,
// EXCEPT when an off-centre kernel value equals 100 (sigma ~ 10*res); that case takes k_add_scans_seq.
// ----------------------------------------------------------------------------------------------
// The state machine in parallel.  Its only carried state is the "first point of the current segment" f and the
// trailing index, and after every segment boundary (a point farther than 0.1 m from f) trailing == that boundary's
// index whichever branch ran.  Hence: (1) next[i] = first j > i with |p_i - p_j|^2 > 0.01 (same expression, so NaN /
// inf readings behave as in the loop) is computed for all i at once; (2) one thread follows f -> next[f] from the first
// non-NaN point — a chain of ~n/5 dependent shared-memory loads instead of n iterations of fp64 arithmetic; (3) for
// boundary k (f = b[k-1], c = b[k]) the side test is evaluated in parallel and the points [b[k-1]', b[k]) — from index 0
// for the first boundary — are valid iff ss >= 0 (i.e. !(ss < 0), NaN included).  Points after the last boundary are
// never pushed (the reference drops the tail, SURVEY.md §8 a3).  Bit-identical flags to the sequential loop (kept verbatim in k_add_scans_seq).
__global__ void k_add_scan(const double *__restrict__ base_pts, const double *__restrict__ sensor,
                           const double *__restrict__ grid_off, uint8_t *__restrict__ grids, size_t grid_pitch,
                           const uint8_t *__restrict__ kernel, b2s_grid_info g, double scale, int n, int n_base) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *px = reinterpret_cast<double *>(smem_raw);
  double *py = px + n;
  int *nxt = reinterpret_cast<int *>(py + n);  // next[i]; reused as the boundary list b[k]
  int *bnd = nxt + n;
  uint8_t *valid = reinterpret_cast<uint8_t *>(bnd + n + 1);
  __shared__ int n_bnd, first_pt;
  const int bs = blockIdx.x;  // b * n_base + s
  const int b = bs / n_base;
  if (threadIdx.x == 0) first_pt = n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    px[i] = base_pts[((size_t)bs * n + i) * 2];
    py[i] = base_pts[((size_t)bs * n + i) * 2 + 1];
    valid[i] = 0;
  }
  __syncthreads();
  const double min_sq = 0.1 * 0.1;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double fx = px[i], fy = py[i];
    if (!isnan(fx) && !isnan(fy)) atomicMin(&first_pt, i);
    int j = i + 1;
    for (; j < n; j++) {
      const double dx = fx - px[j], dy = fy - py[j];
      if (dx * dx + dy * dy > min_sq) break;
    }
    nxt[i] = j;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int k = 0;
    for (int f = first_pt; f < n; f = nxt[f]) bnd[k++] = f;
    n_bnd = k;
  }
  __syncthreads();
  const double vx = sensor[3 * b], vy = sensor[3 * b + 1];
  for (int k = 1 + threadIdx.x; k < n_bnd; k += blockDim.x) {
    const int f = bnd[k - 1], c = bnd[k];
    const double fx = px[f], fy = py[f], cx = px[c], cy = py[c];
    const double a = vy - fy;
    const double bb = fx - vx;
    const double cc = fy * vx - fx * vy;
    const double ss = cx * a + cy * bb + cc;
    if (!(ss < 0.0))
      for (int t = (k == 1 ? 0 : f); t < c; t++) valid[t] = 1;
  }
  __syncthreads();
  // Rasterise + smear.  The result is max over occupied cells of the kernel stamped around them, and a cell holds 100
  // only as the centre of some point (no off-centre kernel value reaches 100 on this path), so each occupied cell is
  // stamped ONCE, by whichever thread raises its centre byte to 100 (running-window base scans hit the same walls many
  // times over).  Winners are queued in shared memory and stamped a warp at a time, lanes over the kernel cells.
  const double ox = grid_off[2 * b], oy = grid_off[2 * b + 1];
  uint8_t *grid = grids + (size_t)b * grid_pitch;
  const int half = g.kernel_size / 2;
  int *win = nxt;  // the chain arrays are free again
  if (threadIdx.x == 0) n_bnd = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    if (!valid[i]) continue;
    double gxd = kround((px[i] - ox) * scale);
    double gyd = kround((py[i] - oy) * scale);
    // IsUpTo on static_cast<int>: non-finite / out-of-int-range values are rejected (see SURVEY.md §8 a3)
    if (!(gxd >= 0.0 && gxd < (double)g.roi_w) || !(gyd >= 0.0 && gyd < (double)g.roi_h)) continue;
    const int idx = ((int)gxd + g.roi_x) + ((int)gyd + g.roi_y) * g.width_step;
    if (atomic_max_u8(grid, idx, GRID_OCCUPIED) != GRID_OCCUPIED) win[atomicAdd(&n_bnd, 1)] = idx;
  }
  __syncthreads();
  // one lane per aligned 32-bit WORD of the stamp (a kernel row covers <= kernel_size/4 + 2 words): the four byte
  // maxima of a word go out as one packed CAS, so lanes of a warp never contend with each other
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5, n_win = n_bnd;
  const int ks = g.kernel_size, wpr = (ks + 3) / 4 + 1;  // words per kernel row, whatever the alignment
  for (int w = warp; w < n_win; w += nwarps) {
    const int idx = win[w];
    for (int t = lane; t < ks * wpr; t += 32) {
      const int j = t / wpr - half, q = t % wpr;
      const int row0 = idx - half + j * g.width_step;   // byte index of the stamp row's first cell
      const int wbase = (row0 & ~3) + 4 * q;            // this lane's aligned word
      uint32_t v = 0;
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int k = wbase + e - row0;                 // kernel column of byte e
        if (k >= 0 && k < ks) v |= (uint32_t)kernel[k + ks * (j + half)] << (8 * e);
      }
      if (v == 0) continue;
      uint32_t *wp = reinterpret_cast<uint32_t *>(grid + wbase);
      uint32_t old = *wp, assumed;
      do {
        const uint32_t mx = __vmaxu4(old, v);
        if (mx == old) break;
        assumed = old;
        old = atomicCAS(wp, assumed, mx);
      } while (assumed != old);
    }
  }
}

// exact sequential AddScans for the degenerate smear kernel (see above): one thread per match
__global__ void k_add_scans_seq(const double *__restrict__ base_pts, const double *__restrict__ sensor,
                                const double *__restrict__ grid_off, uint8_t *__restrict__ grids, size_t grid_pitch,
                                const uint8_t *__restrict__ kernel, b2s_grid_info g, double scale, int n, int n_base,
                                int batch, uint8_t *__restrict__ valid_scratch) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  uint8_t *grid = grids + (size_t)b * grid_pitch;
  uint8_t *valid = valid_scratch + (size_t)b * n;
  const int half = g.kernel_size / 2;
  for (int s = 0; s < n_base; s++) {
    const double *p = base_pts + ((size_t)(b * n_base + s) * n) * 2;
    // FindValidPoints on strided xy pairs
    const double min_sq = 0.1 * 0.1;
    const double vx = sensor[3 * b], vy = sensor[3 * b + 1];
    for (int i = 0; i < n; i++) valid[i] = 0;
    int trailing = 0;
    double fx = 0.0, fy = 0.0;
    bool first_time = true;
    for (int it = 0; it < n; it++) {
      double cx = p[2 * it], cy = p[2 * it + 1];
      if (first_time && !isnan(cx) && !isnan(cy)) { fx = cx; fy = cy; first_time = false; }
      double dx = fx - cx, dy = fy - cy;
      if (dx * dx + dy * dy > min_sq) {
        double a = vy - fy, bb = fx - vx, c = fy * vx - fx * vy;
        double ss = cx * a + cy * bb + c;
        fx = cx; fy = cy;
        if (ss < 0.0) trailing = it;
        else for (; trailing != it; ++trailing) valid[trailing] = 1;
      }
    }
    for (int i = 0; i < n; i++) {
      if (!valid[i]) continue;
      double gxd = kround((p[2 * i] - grid_off[2 * b]) * scale);
      double gyd = kround((p[2 * i + 1] - grid_off[2 * b + 1]) * scale);
      if (!(gxd >= 0.0 && gxd < (double)g.roi_w) || !(gyd >= 0.0 && gyd < (double)g.roi_h)) continue;
      int gx = (int)gxd + g.roi_x, gy = (int)gyd + g.roi_y;
      int idx = gx + gy * g.width_step;
      if (grid[idx] == GRID_OCCUPIED) continue;  // Mapper.cpp:734-738
      grid[idx] = GRID_OCCUPIED;
      for (int j = -half; j <= half; j++)
        for (int k = -half; k <= half; k++) {
          uint8_t kv = kernel[(k + half) + g.kernel_size * (j + half)];
          uint8_t *c = grid + (gx + k) + (gy + j) * g.width_step;
          if (kv > *c) *c = kv;
        }
    }
  }
}

// GridIndexLookup::ComputeOffsets for one reading (Karto.h:6474-6499)
__device__ __forceinline__ int32_t lut_value(double r, double lx, double ly, double cosine, double sine, double gox,
                                             double goy, double scale, int width_step) {
  if (isnan(r) || isinf(r)) return INVALID_SCAN;
  double ox = __dsub_rn(__dmul_rn(cosine, lx), __dmul_rn(sine, ly));
  double oy = __dadd_rn(__dmul_rn(sine, lx), __dmul_rn(cosine, ly));
  // WorldToGrid(offset + rGridOffset): ((o + off) - off) * scale (Karto.h:6491, 4239-4251)
  int32_t gx = cast_i32(kround(__dmul_rn(__dsub_rn(__dadd_rn(ox, gox), gox), scale)));
  int32_t gy = cast_i32(kround(__dmul_rn(__dsub_rn(__dadd_rn(oy, goy), goy), scale)));
  return (int32_t)((uint32_t)gx + (uint32_t)gy * (uint32_t)width_step);  // Grid<T>::GridIndex, no ROI
}

// ----------------------------------------------------------------------------------------------
// k_offsets: GridIndexLookup::ComputeOffsets (Karto.h:6455-6501).  One block per (match, angle).
// ----------------------------------------------------------------------------------------------
__global__ void k_offsets(const double *__restrict__ ranges, const double *__restrict__ local,
                          const double *__restrict__ grid_off, const double *__restrict__ centers, int center_stride,
                          double angle_center_override, int use_override, double angle_offset, double angle_res,
                          int n_angles, int n, int width_step, double scale, int32_t *__restrict__ lut, int k_first) {
  const int b = blockIdx.x / n_angles, k = blockIdx.x % n_angles;
  const double center = use_override ? angle_center_override : centers[(size_t)b * center_stride + 2];
  const double start = center - angle_offset;
  const double angle = start + (double)(uint32_t)(k_first + k) * angle_res;  // k_first: angle subset of a split sweep
  const double cosine = cos(angle), sine = sin(angle);
  const double gox = grid_off[2 * b], goy = grid_off[2 * b + 1];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int32_t v = lut_value(ranges[(size_t)b * n + i], local[((size_t)b * n + i) * 2], local[((size_t)b * n + i) * 2 + 1],
                                cosine, sine, gox, goy, scale, width_step);
    lut[((size_t)b * n_angles + k) * n + i] = v;
  }
}

// ----------------------------------------------------------------------------------------------
// k_bases: candidate lattice of CorrelateScan (Mapper.cpp:338-358, 373-386) -> flat base index per (iy, ix).
// flags[b]: bit0 = lattice is the regular raster base00 + stride*(ix + iy*width_step), stride = 1 or 2 cells;
//           bit1 = some candidate fell outside the grid (reference throws karto::Exception, Karto.h:4490-4499)
// ----------------------------------------------------------------------------------------------
__global__ void k_bases(const double *__restrict__ centers, const double *__restrict__ grid_off, b2s_search s,
                        b2s_grid_info g, double scale, int nx, int ny, int32_t *__restrict__ bases,
                        int32_t *__restrict__ flags, int stride) {
  const int b = blockIdx.x;
  __shared__ int irregular, oob;
  if (threadIdx.x == 0) { irregular = 0; oob = 0; }
  __syncthreads();
  const double cx = centers[3 * b], cy = centers[3 * b + 1];
  const double gox = grid_off[2 * b], goy = grid_off[2 * b + 1];
  const double start_x = -s.offset_x, start_y = -s.offset_y;
  const int32_t gx0 = world_to_grid_1(cx + start_x, gox, scale) + g.roi_x;
  const int32_t gy0 = world_to_grid_1(cy + start_y, goy, scale) + g.roi_y;
  for (int c = threadIdx.x; c < nx * ny; c += blockDim.x) {
    int iy = c / nx, ix = c % nx;
    double y = start_y + (double)(uint32_t)iy * s.res_y;
    double x = start_x + (double)(uint32_t)ix * s.res_x;
    int32_t gx = world_to_grid_1(cx + x, gox, scale) + g.roi_x;  // CorrelationGrid::GridIndex (Mapper.h:941-947)
    int32_t gy = world_to_grid_1(cy + y, goy, scale) + g.roi_y;
    if (!(gx >= 0 && gx < g.width && gy >= 0 && gy < g.height)) oob = 1;
    if (gx != gx0 + stride * ix || gy != gy0 + stride * iy) irregular = 1;
    bases[(size_t)b * nx * ny + c] = gx + gy * g.width_step;
  }
  __syncthreads();
  if (threadIdx.x == 0) flags[b] = (irregular ? 0 : 1) | (oob ? 2 : 0);
}

// ----------------------------------------------------------------------------------------------
// k_sweep_generic: integer numerators of GetResponse (Mapper.cpp:819-856) for every candidate.
// One warp per (x,y) candidate, looping over all angles; lanes stride over beams; grid + LUT read from
// global memory (L1/L2).  Handles any lattice and any grid size.  mode 0: all matches; mode 1: only matches
// whose lattice is NOT regular (the window kernel did the others).
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sweep_generic(const uint8_t *__restrict__ grids, size_t grid_pitch,
                                                       int data_size, const int32_t *__restrict__ lut,
                                                       const int32_t *__restrict__ bases,
                                                       const int32_t *__restrict__ flags, int mode, int n, int na,
                                                       int ncell, int32_t *__restrict__ sums,
                                                       const double *__restrict__ ranges,
                                                       const double *__restrict__ local,
                                                       const double *__restrict__ grid_off,
                                                       const double *__restrict__ centers, double angle_offset,
                                                       double angle_res, int width_step, double scale, int k_first) {
  const int b = blockIdx.y;
  const int f = flags[b];
  if (f & 2) return;
  if (mode == 1 && (f & 1)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint8_t *grid = grids + (size_t)b * grid_pitch;
  for (int c = blockIdx.x * (blockDim.x >> 5) + warp; c < ncell; c += gridDim.x * (blockDim.x >> 5)) {
  const int32_t base = bases[(size_t)b * ncell + c];
  for (int k = 0; k < na; k++) {
    const int32_t *offs = lut ? lut + ((size_t)b * na + k) * n : nullptr;
    double cosine = 0, sine = 0, gox = 0, goy = 0;
    if (!lut) {  // no materialised table (window mode fall-through): GridIndexLookup values on the fly
      const double angle = (centers[(size_t)b * 3 + 2] - angle_offset) + (double)(uint32_t)(k_first + k) * angle_res;
      cosine = cos(angle); sine = sin(angle);
      gox = grid_off[2 * b]; goy = grid_off[2 * b + 1];
    }
    int32_t sum = 0;
    if (lut) {
      // 8 independent (offset, cell) load chains in flight per lane: the gather is latency bound
      constexpr int U = 8;
      for (int i0 = lane; i0 < n; i0 += 32 * U) {
        int32_t o[U];
#pragma unroll
        for (int u = 0; u < U; u++) o[u] = (i0 + 32 * u < n) ? __ldg(offs + i0 + 32 * u) : INVALID_SCAN;
        uint32_t v[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const int32_t idx = (int32_t)((uint32_t)base + (uint32_t)o[u]);
          v[u] = (o[u] != INVALID_SCAN && idx >= 0 && idx < data_size) ? (uint32_t)__ldg(grid + idx) : 0u;
        }
#pragma unroll
        for (int u = 0; u < U; u++) sum += (int32_t)v[u];
      }
    } else {
      for (int i = lane; i < n; i += 32) {
        const int32_t o = lut_value(ranges[(size_t)b * n + i], local[((size_t)b * n + i) * 2],
                                    local[((size_t)b * n + i) * 2 + 1], cosine, sine, gox, goy, scale, width_step);
        if (o == INVALID_SCAN) continue;
        const int32_t idx = (int32_t)((uint32_t)base + (uint32_t)o);
        if (idx >= 0 && idx < data_size) sum += __ldg(grid + idx);
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    if (lane == 0) sums[((size_t)b * na + k) * ncell + c] = sum;
  }
  }
}

// ----------------------------------------------------------------------------------------------
// k_sweep_window — the hot kernel (stride-1 lattices, grid fits in shared memory).
//
// For a fixed angle k and beam i, the cells read by all (ix, iy) candidates form the nY x nX window of the
// grid whose origin is  a = base00 + lut[k][i]  (flat index; rows are width_step apart).  So
//     sums[k][iy][ix] = SUM_i grid[a_i + iy*width_step + ix].
// A persistent CTA stages one match's whole grid into shared memory with TMA bulk copies and its warps take
// (angle, 32x32 window tile) work items.  Within a warp lane r owns candidate row r.
//
// k_offsets_sorted prepares, per (match, angle), the window origins a_i grouped by byte alignment (a & 3) and
// split into INTERIOR beams (every byte any lane will touch lies inside the staged image, no checks needed) and
// EDGE beams (some row leaves [0, data_size): per-row redirect to a zero guard), with beams whose whole window is
// outside dropped.  Integer sums commute, so the regrouping is free.
//
// Inner loop, per PAIR of same-alignment beams and per lane: 2 x 9 aligned 32-bit shared-memory loads (the 36
// bytes covering the lane's 32 candidate cells), 9 packed-byte adds of the two beams' words (cell values <= 100,
// so two fit a byte), then each summed word is split into two packed-u16 halves (bytes 0,2 / bytes 1,3) and added
// to 18 packed-u16 accumulators kept in WORD-ALIGNED coordinates — the alignment (a compile-time constant of the
// class) is only applied when the u16 lanes are flushed into the 32 per-candidate 32-bit sums.  One shared-memory
// word therefore feeds 4 adjacent-x candidates and costs ~2.3 integer instructions per beam.
//
// Flat-index semantics of the reference are kept bit-exactly: rows wrap exactly as `base + offset` does, and
// positions outside [0, data_size) read zeros (guard bands, zero padding of the HBM image, redirect of rows that
// are entirely outside).  Lanes 16..31 fetch their 9 words rotated by one so that the two half-warps hit odd /
// even banks (width_step/4 is even, so rows r and r+16 would otherwise always collide).
// ----------------------------------------------------------------------------------------------
constexpr int WIN_THREADS = 512;
constexpr int WIN_GUARD = 128;          // zero bytes before and after the grid image in shared memory
constexpr int WIN_FLUSH_BEAMS = 512;    // beams accumulated in u16 lanes between flushes (512 * 127 < 65536)
constexpr int32_t WIN_SKIP = -(1 << 29);
constexpr int WIN_MAX_BANDS = 32;      // row bands a grid larger than shared memory is swept in
constexpr int LIST_PAD = 16;            // per-(match, angle) list capacity = n + LIST_PAD * nbands

// ----------------------------------------------------------------------------------------------
// k_grid_sat: per match, a summed-area table over 4x4-cell blocks of "block holds a non-zero cell".  A beam whose
// whole nY x nX window covers only empty blocks adds 0 to every candidate, so k_offsets_sorted may drop it — the
// response volume stays bit-identical.  sat[(by+1) x (bx+1)] u16, one block per match.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_grid_sat(const uint8_t *__restrict__ grids, size_t grid_pitch, int width_step, int height, int bx, int by,
               uint16_t *__restrict__ sat_all) {
  extern __shared__ uint32_t s_sat[];  // (by+1) x (bx+1)
  const int b = blockIdx.x;
  const uint8_t *grid = grids + (size_t)b * grid_pitch;
  const int W = bx + 1;
  for (int i = threadIdx.x; i < (by + 1) * W; i += blockDim.x) s_sat[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < bx * by; i += blockDim.x) {
    const int cy = i / bx, cx = i % bx;
    uint32_t any = 0;
    for (int r = 0; r < 4; r++) {
      const int y = cy * 4 + r;
      if (y < height) any |= *reinterpret_cast<const uint32_t *>(grid + (size_t)y * width_step + cx * 4);  // width_step % 4 == 0
    }
    s_sat[(cy + 1) * W + (cx + 1)] = any ? 1u : 0u;
  }
  __syncthreads();
  for (int y = threadIdx.x + 1; y <= by; y += blockDim.x) {  // row prefix sums
    uint32_t acc = 0;
    for (int x = 1; x <= bx; x++) { acc += s_sat[y * W + x]; s_sat[y * W + x] = acc; }
  }
  __syncthreads();
  for (int x = threadIdx.x + 1; x <= bx; x += blockDim.x) {  // column prefix sums
    uint32_t acc = 0;
    for (int y = 1; y <= by; y++) { acc += s_sat[y * W + x]; s_sat[y * W + x] = acc; }
  }
  __syncthreads();
  uint16_t *out = sat_all + (size_t)b * (size_t)(((by + 1) * W + 7) & ~7);  // padded stride: k_offsets_sorted copies 16 bytes at a time
  for (int i = threadIdx.x; i < (by + 1) * W; i += blockDim.x) out[i] = (uint16_t)s_sat[i];  // < 65536 blocks (checked by the host)
}

// ----------------------------------------------------------------------------------------------
// k_grid_mp4: per match, the 4x4 max-pool MP4[j] = max over dy, dx in [0, 4) of grid[j + dy*width_step + dx] in flat
// index space (zero outside [0, data_size)), for j in [-guard, data_size + guard).  guard >= 3*width_step + 3 + 64, so
// every j whose pool reaches the grid is covered, including origins just below flat index 0, and the first 12 bytes of
// phase 0 are zero (k_prune_select redirects rows outside the image there).  k_prune_select reads the
// pool values of the 8 block columns of one beam row, j + 4*bx, as 8 consecutive bytes: the image is stored split into
// four column phases, phase p = (j + guard) & 3 at byte p*lq + ((j + guard) >> 2).  One thread per 16 flat bytes
// (one 32-bit word of each phase); guard % 16 == 0 and width_step % 8 == 0 keep every grid read word-aligned.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_grid_mp4(const uint8_t *__restrict__ grids, size_t grid_pitch, int data_size, int width_step, int guard, int lq,
               uint8_t *__restrict__ mp_all, size_t mp_pitch) {
  const int b = blockIdx.y;
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= lq / 4) return;
  const uint8_t *grid = grids + (size_t)b * grid_pitch;
  const int j = 16 * w - guard;
  uint32_t o[4] = {0u, 0u, 0u, 0u};  // pool bytes of flat j + 4k + q (word k, byte q)
#pragma unroll
  for (int dy = 0; dy < 4; dy++) {
    const int r = j + dy * width_step;
    uint32_t W[5], m1[5];
#pragma unroll
    for (int q = 0; q < 5; q++) {
      const int x = r + 4 * q;
      W[q] = (x >= 0 && x < data_size) ? __ldg(reinterpret_cast<const uint32_t *>(grid + x)) : 0u;
    }
#pragma unroll
    for (int q = 0; q < 5; q++) m1[q] = __vmaxu4(W[q], __funnelshift_r(W[q], q < 4 ? W[q + 1] : 0u, 8));  // max of bytes i, i+1
#pragma unroll
    for (int k = 0; k < 4; k++) o[k] = __vmaxu4(o[k], __vmaxu4(m1[k], __funnelshift_r(m1[k], m1[k + 1], 16)));  // i .. i+3
  }
  // 4x4 byte transpose: phase p's word w holds byte p of o[0..3]
  const uint32_t t01l = __byte_perm(o[0], o[1], 0x5140), t01h = __byte_perm(o[0], o[1], 0x7362);
  const uint32_t t23l = __byte_perm(o[2], o[3], 0x5140), t23h = __byte_perm(o[2], o[3], 0x7362);
  uint8_t *mp = mp_all + (size_t)b * mp_pitch + 4 * (size_t)w;
  *reinterpret_cast<uint32_t *>(mp) = __byte_perm(t01l, t23l, 0x5410);
  *reinterpret_cast<uint32_t *>(mp + lq) = __byte_perm(t01l, t23l, 0x7632);
  *reinterpret_cast<uint32_t *>(mp + 2 * (size_t)lq) = __byte_perm(t01h, t23h, 0x5410);
  *reinterpret_cast<uint32_t *>(mp + 3 * (size_t)lq) = __byte_perm(t01h, t23h, 0x7632);
}

// One block per (match, chunk of OFF_CHUNK angles): window origins grouped as [I0 I1 I2 I3 E0 E1 E2 E3] (I = interior,
// E = edge, index = a & 3), every group a multiple of 4 long (an interior group donates its 0..3 surplus beams to its edge
// group; edge groups are padded with far-negative sentinels of the same alignment).  counts[8] holds the group lengths.
// The scan's readings and local points are staged in shared memory once per block and reused for every angle of
// the chunk (16x less L2 traffic than one block per angle).  A non-finite reading (INVALID_SCAN, Karto.h:6478) always
// yields a non-finite local point (inf/NaN propagate through the inverse transform), so only the points are staged.
constexpr int OFF_CHUNK = 16;
constexpr int OFF_Q = 2;                              // angles classified per pass
constexpr int OFF_GS = 8 * WIN_MAX_BANDS;             // group slots per angle
constexpr int OFF_SMEM_PER_BEAM = 16 + 5 * OFF_Q;     // two doubles + OFF_Q x (origin int32 + class byte)
__global__ void __launch_bounds__(256)
    k_offsets_sorted(const double *__restrict__ ranges, const double *__restrict__ local,
                     const double *__restrict__ grid_off, const double *__restrict__ centers,
                     const int32_t *__restrict__ bases, const int32_t *__restrict__ flags, double angle_offset,
                     double angle_res, int n_angles, int n, int ncell, int width_step, int data_size, double scale,
                     int rows_total, int cols_total, int32_t *__restrict__ lists, int32_t *__restrict__ counts,
                     const uint16_t *__restrict__ sat_all, int sbx, int sby, int height, int nx, int ny,
                     unsigned long long *__restrict__ stats, int band_rows, int nbands,
                     int32_t *__restrict__ starts, int stride, int k_first, int neg_bands) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  double *s_lx = reinterpret_cast<double *>(s_raw), *s_ly = s_lx + n;  // [n] scan-local points
  int32_t *s_vals = reinterpret_cast<int32_t *>(s_ly + n);             // [OFF_Q][n] window origins
  uint8_t *s_cls = reinterpret_cast<uint8_t *>(s_vals + OFF_Q * n);    // [OFF_Q][n] group ids
  uint16_t *s_sat = reinterpret_cast<uint16_t *>(s_raw + (((size_t)n * OFF_SMEM_PER_BEAM + 15) & ~(size_t)15));  // [(sby+1)(sbx+1)] or unused
  __shared__ int cnt[OFF_Q * OFF_GS], fill[OFF_Q * OFF_GS], seg[OFF_Q * OFF_GS];  // [angle][band][group]
  __shared__ int n_empty;
  const int ngroups = 8 * nbands;
  const int list_cap = n + LIST_PAD * nbands;
  const int chunks = (n_angles + OFF_CHUNK - 1) / OFF_CHUNK;
  const int b = blockIdx.x / chunks, k0 = (blockIdx.x % chunks) * OFF_CHUNK;
  const int f = flags[b];
  if ((f & 2) || !(f & 1)) return;  // error / irregular lattice: the generic kernel handles this match
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    s_lx[i] = local[((size_t)b * n + i) * 2];
    s_ly[i] = local[((size_t)b * n + i) * 2 + 1];
  }
  const int SW = sbx + 1;
  if (sat_all) {  // per-match tables are padded to a multiple of 8 entries: 16-byte copies
    const int sat_stride = ((sby + 1) * SW + 7) & ~7;
    const uint4 *src = reinterpret_cast<const uint4 *>(sat_all + (size_t)b * sat_stride);
    uint4 *dst = reinterpret_cast<uint4 *>(s_sat);
    for (int i = threadIdx.x; i < sat_stride / 8; i += blockDim.x) dst[i] = src[i];
  }
  if (threadIdx.x == 0) n_empty = 0;
  const double center = centers[(size_t)b * 3 + 2];
  __shared__ double s_cos[OFF_CHUNK], s_sin[OFF_CHUNK];
  if (threadIdx.x < OFF_CHUNK && k0 + threadIdx.x < n_angles) {  // one sincos per angle, not per thread
    const double ang = (center - angle_offset) + (double)(uint32_t)(k_first + k0 + threadIdx.x) * angle_res;
    s_cos[threadIdx.x] = cos(ang);
    s_sin[threadIdx.x] = sin(ang);
  }
  const double gox = grid_off[2 * b], goy = grid_off[2 * b + 1];
  const int32_t base00 = bases[(size_t)b * ncell];
  const long long span = (long long)stride * (rows_total - 1) * width_step + cols_total + 8;  // last byte any lane may touch
  const int32_t span32 = (int32_t)min(span, (long long)(1 << 29));
  const int fx = stride * (nx - 1) + 1, fy = stride * (ny - 1) + 1;  // footprint of the candidate lattice in cells
  const float inv_step = 1.0f / (float)width_step, inv_band = 1.0f / (float)band_rows;
  const int kend = min(k0 + OFF_CHUNK, n_angles);
  for (int kq = k0; kq < kend; kq += OFF_Q) {  // OFF_Q angles per pass: half the barriers, one read of the points
    const int nq = min(OFF_Q, kend - kq);
    __syncthreads();  // staging done / previous angles' smem fully consumed
    for (int t = threadIdx.x; t < OFF_Q * OFF_GS; t += blockDim.x) { cnt[t] = 0; fill[t] = 0; }
    __syncthreads();
    int empty_here = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double plx = s_lx[i], ply = s_ly[i];
#pragma unroll
      for (int q = 0; q < OFF_Q; q++) {
        if (q >= nq) break;
        const double cosine = s_cos[kq - k0 + q], sine = s_sin[kq - k0 + q];
        // lut_value() inlined: a non-finite local point (INVALID_SCAN reading) makes ox/oy non-finite
        const double ox = __dsub_rn(__dmul_rn(cosine, plx), __dmul_rn(sine, ply));
        const double oy = __dadd_rn(__dmul_rn(sine, plx), __dmul_rn(cosine, ply));
        int cls = 255;  // dropped
        int32_t a = 0;
        if (isfinite(ox) && isfinite(oy)) {
          const int32_t gx = cast_i32(kround(__dmul_rn(__dsub_rn(__dadd_rn(ox, gox), gox), scale)));
          const int32_t gy = cast_i32(kround(__dmul_rn(__dsub_rn(__dadd_rn(oy, goy), goy), scale)));
          const int32_t o = (int32_t)((uint32_t)gx + (uint32_t)gy * (uint32_t)width_step);
          a = (int32_t)((uint32_t)base00 + (uint32_t)o);
          // window [a - 8, a + span] against [0, data_size): 32-bit arithmetic after clamping far-away origins
          const int32_t ac = max(min(a, (int32_t)(1 << 29)), -(int32_t)(1 << 29));
          const int32_t lo = ac - 8, hi = ac + span32;
          if (hi < 0 || lo >= data_size) cls = 255;  // whole window outside: contributes 0
          else if (lo >= -(WIN_GUARD - 16) && hi <= data_size + (WIN_GUARD - 16)) cls = a & 3;  // interior
          else cls = 4 + (a & 3);                                                                // edge
          int y = 0, x = 0;
          if ((sat_all || nbands > 1) && cls < 255 && (a >= 0 || neg_bands > 0)) {
            // floor(a / width_step) by float reciprocal + fix-up (|a| < 2^24 is exact in float; larger values are
            // corrected too); a < 0 only matters when origins below the grid get row bands of their own (neg_bands)
            if (data_size <= (1 << 24) && ac == a) {
              y = (int)((float)a * inv_step);
              if (y * width_step > a) y--;
              else if ((y + 1) * width_step <= a) y++;
            } else {
              y = a / width_step;
              if (y * width_step > a) y--;
            }
            x = a - y * width_step;
          }
          if (nbands > 1 && cls < 8) {
            int band = (int)((float)y * inv_band);
            if (band * band_rows > y) band--;
            else if ((band + 1) * band_rows <= y) band++;
            cls += 8 * max(min(band + neg_bands, nbands - 1), 0);  // the row band that holds the window origin
          }
          if (sat_all && cls < 255 && a >= 0) {
            // empty-window test on the 4x4-block summed-area table (only for windows that do not wrap a row end)
            if (x + fx <= width_step && y + fy <= height) {
              const int bx0 = x >> 2, bx1 = (x + fx - 1) >> 2, by0 = y >> 2, by1 = (y + fy - 1) >> 2;
              const uint32_t c = (uint32_t)s_sat[(by1 + 1) * SW + bx1 + 1] - (uint32_t)s_sat[by0 * SW + bx1 + 1] -
                                 (uint32_t)s_sat[(by1 + 1) * SW + bx0] + (uint32_t)s_sat[by0 * SW + bx0];
              if (c == 0) { cls = 255; empty_here++; }
            }
          }
        }
        s_vals[q * n + i] = a;
        s_cls[q * n + i] = (uint8_t)cls;
        if (cls < 255) atomicAdd(&cnt[q * OFF_GS + cls], 1);
      }
    }
    if (empty_here) atomicAdd(&n_empty, empty_here);
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && (threadIdx.x >> 5) < nq) {  // one thread (of its own warp) per angle
      int *c_ = cnt + (threadIdx.x >> 5) * OFF_GS, *seg_ = seg + (threadIdx.x >> 5) * OFF_GS;
      int pos = 0;
      for (int g8 = 0; g8 < ngroups; g8 += 8) {
        for (int c = 0; c < 4; c++) {
          const int d = c_[g8 + c] & 3;  // interior groups are multiples of 4: the last-placed 0..3 beams go to the edge group
          c_[g8 + c] -= d;
          c_[g8 + 4 + c] += d;
        }
        for (int c = 0; c < 8; c++) {
          seg_[g8 + c] = pos;
          pos += (c_[g8 + c] + 3) & ~3;
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
#pragma unroll
      for (int q = 0; q < OFF_Q; q++) {
        if (q >= nq) break;
        int cls = s_cls[q * n + i];
        if (cls == 255) continue;
        int slot = atomicAdd(&fill[q * OFF_GS + cls], 1);
        if ((cls & 7) < 4 && slot >= cnt[q * OFF_GS + cls]) {  // a donated one
          cls += 4;
          slot = atomicAdd(&fill[q * OFF_GS + cls], 1);
        }
        lists[((size_t)b * n_angles + kq + q) * list_cap + seg[q * OFF_GS + cls] + slot] = s_vals[q * n + i];
      }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nq * ngroups; t += blockDim.x) {
      const int q = t / ngroups, g = t % ngroups;
      const int cg = cnt[q * OFF_GS + g], sg_ = seg[q * OFF_GS + g];
      int32_t *out = lists + ((size_t)b * n_angles + kq + q) * list_cap;
      if ((g & 7) >= 4)
        for (int r = cg; r < ((cg + 3) & ~3); r++)
          out[sg_ + r] = WIN_SKIP + (g & 3);  // pad: all-outside beams of the same alignment
      counts[((size_t)b * n_angles + kq + q) * ngroups + g] = (cg + 3) & ~3;
      starts[((size_t)b * n_angles + kq + q) * ngroups + g] = sg_;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && stats && n_empty) atomicAdd(stats, (unsigned long long)n_empty);
}

// flush the packed-u16 accumulators (word-aligned coordinates, alignment class SH) into the per-candidate sums.
// slots 0..7 hold aligned word j (lanes 0..15) or aligned word (j+1)%8 (lanes 16..31); slot 8 holds aligned word 8;
// byte q of word w is candidate x = 4*w + q - SH.
// With STRIDE = 2 (candidates every other cell) only the bytes at even distance from the origin are candidates:
// byte position p = 4*w + q - SH is candidate x = p / 2 when p is even; a tile then holds 16 candidates in 32 bytes.
template <int SH, int STRIDE, int ROT>
__device__ __forceinline__ void win_flush_rot(const uint32_t (&lo)[9], const uint32_t (&hi)[9], uint32_t (&acc)[32]) {
#define B2S_FLUSH_ONE(P, VAL)                                                        \
  if ((P) >= 0 && ((P) % STRIDE) == 0 && (P) / STRIDE < 32 / STRIDE) acc[((P) / STRIDE) & 31] += (VAL);
#define B2S_FLUSH_SLOT(J, W)                                                         \
  {                                                                                  \
    const int x0 = 4 * (W) - SH;                                                     \
    B2S_FLUSH_ONE(x0 + 0, lo[J] & 0xffffu)                                           \
    B2S_FLUSH_ONE(x0 + 1, hi[J] & 0xffffu)                                           \
    B2S_FLUSH_ONE(x0 + 2, lo[J] >> 16)                                               \
    B2S_FLUSH_ONE(x0 + 3, hi[J] >> 16)                                               \
  }
#pragma unroll
  for (int j = 0; j < 8; j++) B2S_FLUSH_SLOT(j, (j + ROT) % 8)
  B2S_FLUSH_SLOT(8, 8)
#undef B2S_FLUSH_SLOT
#undef B2S_FLUSH_ONE
}

// `rot` = this lane's word rotation: slot j holds aligned word (j + rot) % 8 (see win_load).  GEN = false: rot is 0 for
// lanes 0..15 and 1 for lanes 16..31; GEN = true: any of 0..7.
template <int SH, int STRIDE, bool GEN>
__device__ __forceinline__ void win_flush(uint32_t (&lo)[9], uint32_t (&hi)[9], uint32_t (&acc)[32], int rot) {
  if (!GEN) {
    if (!rot) win_flush_rot<SH, STRIDE, 0>(lo, hi, acc);
    else win_flush_rot<SH, STRIDE, 1>(lo, hi, acc);
  } else {
    switch (rot) {
      case 0: win_flush_rot<SH, STRIDE, 0>(lo, hi, acc); break;
      case 1: win_flush_rot<SH, STRIDE, 1>(lo, hi, acc); break;
      case 2: win_flush_rot<SH, STRIDE, 2>(lo, hi, acc); break;
      case 3: win_flush_rot<SH, STRIDE, 3>(lo, hi, acc); break;
      case 4: win_flush_rot<SH, STRIDE, 4>(lo, hi, acc); break;
      case 5: win_flush_rot<SH, STRIDE, 5>(lo, hi, acc); break;
      case 6: win_flush_rot<SH, STRIDE, 6>(lo, hi, acc); break;
      default: win_flush_rot<SH, STRIDE, 7>(lo, hi, acc); break;
    }
  }
#pragma unroll
  for (int j = 0; j < 9; j++) { lo[j] = 0; hi[j] = 0; }
}

// load the 8 (+1) words of one beam's row; `base` = byte address in sgrid of aligned word 0 of this lane's row.
// Bank conflicts: lane L's row starts (L * STRIDE * width_step / 4) mod 32 banks after lane 0's; with width_step a
// multiple of 8 that step is even, so m = gcd(step, 32) >= 2 lanes share every row-start bank.  Rotating the order in
// which a lane fetches its 8 words by rot = L / (32 / m) gives each of those m lanes a different bank at every load
// instruction, and the m-lane groups tile the 32 banks when m <= 8: conflict-free.  The common case m = 2 (cfg 1/2's
// 408-byte step: 102 words) is the GEN = false path, lanes 16..31 fetch words 1..7,0 with immediate offsets; GEN =
// true takes any rotation through per-lane byte offsets `loff`.  Word 8 (only needed when the window's last
// candidates spill past 32 bytes) cannot be de-conflicted and is loaded only when W9.
template <bool W9, bool GEN>
__device__ __forceinline__ void win_load(const uint8_t *__restrict__ sgrid, int base, int rot, const int (&loff)[8],
                                         uint32_t (&v)[9]) {
  if (!GEN) {
    const uint32_t *w0 = reinterpret_cast<const uint32_t *>(sgrid + base);
    const uint32_t *wp = w0 + rot;
#pragma unroll
    for (int j = 0; j < 7; j++) v[j] = wp[j];
    v[7] = wp[7 - 8 * rot];
    v[8] = W9 ? w0[8] : 0u;
  } else {
    const uint8_t *p = sgrid + base;
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = *reinterpret_cast<const uint32_t *>(p + loff[j]);
    v[8] = W9 ? *reinterpret_cast<const uint32_t *>(p + 32) : 0u;
  }
}

template <bool W9>
__device__ __forceinline__ void win_accumulate2(const uint32_t (&v1)[9], const uint32_t (&v2)[9], uint32_t (&lo)[9],
                                                uint32_t (&hi)[9]) {
#pragma unroll
  for (int q = 0; q < (W9 ? 9 : 8); q++) {
    const uint32_t w = v1[q] + v2[q];      // packed bytes, each <= 254
    lo[q] += w & 0x00ff00ffu;              // bytes 0, 2 -> u16 lanes
    hi[q] += __byte_perm(w, 0u, 0x4341);   // bytes 1, 3 -> u16 lanes
  }
}

// all beams of one alignment class; count is a multiple of 4.  CHECK = per-row range test (edge beams).
template <int SH, int STRIDE, bool CHECK, bool W9, bool GEN>
__device__ __forceinline__ void win_class(const uint8_t *__restrict__ sgrid, const int32_t *__restrict__ list,
                                          int count, int lane, int hi_half, const int (&loff)[8], int bias, int row_delta,
                                          int data_size, int32_t *__restrict__ s_off, uint32_t (&lo)[9],
                                          uint32_t (&hi)[9], uint32_t (&acc)[32], int &pending) {
  for (int ib = 0; ib < count; ib += 32) {
    const int cnt = min(32, count - ib);
    __syncwarp();
    s_off[lane] = (lane < cnt) ? __ldg(list + ib + lane) : 0;  // this warp's staging row
    __syncwarp();
    if (pending + cnt > WIN_FLUSH_BEAMS) {
      win_flush<SH, STRIDE, GEN>(lo, hi, acc, hi_half);
      pending = 0;
    }
    pending += cnt;
    for (int j = 0; j < cnt; j += 4) {
      const int4 a = *reinterpret_cast<const int4 *>(s_off + j);  // one broadcast load: four window origins
      int b0, b1, b2, b3;
      if (CHECK) {
        const int32_t i0 = a.x + row_delta, i1 = a.y + row_delta, i2 = a.z + row_delta, i3 = a.w + row_delta;
        b0 = (((uint32_t)i0 + 35u) < ((uint32_t)data_size + 35u)) ? (i0 + (bias - SH)) : 0;
        b1 = (((uint32_t)i1 + 35u) < ((uint32_t)data_size + 35u)) ? (i1 + (bias - SH)) : 0;
        b2 = (((uint32_t)i2 + 35u) < ((uint32_t)data_size + 35u)) ? (i2 + (bias - SH)) : 0;
        b3 = (((uint32_t)i3 + 35u) < ((uint32_t)data_size + 35u)) ? (i3 + (bias - SH)) : 0;
      } else {
        const int lane_const = row_delta + bias - SH;
        b0 = a.x + lane_const; b1 = a.y + lane_const; b2 = a.z + lane_const; b3 = a.w + lane_const;
      }
      uint32_t v1[9], v2[9];
      win_load<W9, GEN>(sgrid, b0, hi_half, loff, v1);
      win_load<W9, GEN>(sgrid, b1, hi_half, loff, v2);
      win_accumulate2<W9>(v1, v2, lo, hi);
      win_load<W9, GEN>(sgrid, b2, hi_half, loff, v1);
      win_load<W9, GEN>(sgrid, b3, hi_half, loff, v2);
      win_accumulate2<W9>(v1, v2, lo, hi);
    }
  }
}

template <int SH, int STRIDE, bool GEN>
__device__ __forceinline__ void win_class_pair(const uint8_t *__restrict__ sgrid, const int32_t *__restrict__ li,
                                               int ci, const int32_t *__restrict__ le, int ce, int cols, int lane,
                                               int hi_half, const int (&loff)[8], int row_delta, int bias, int data_size, int32_t *__restrict__ s_off,
                                               uint32_t (&lo)[9], uint32_t (&hi)[9], uint32_t (&acc)[32]) {
  int pending = 0;
  if (SH + STRIDE * (cols - 1) + 1 > 32) {  // the last candidates need aligned word 8
    win_class<SH, STRIDE, false, true, GEN>(sgrid, li, ci, lane, hi_half, loff, bias, row_delta, data_size, s_off, lo, hi, acc, pending);
    win_class<SH, STRIDE, true, true, GEN>(sgrid, le, ce, lane, hi_half, loff, bias, row_delta, data_size, s_off, lo, hi, acc, pending);
  } else {
    win_class<SH, STRIDE, false, false, GEN>(sgrid, li, ci, lane, hi_half, loff, bias, row_delta, data_size, s_off, lo, hi, acc, pending);
    win_class<SH, STRIDE, true, false, GEN>(sgrid, le, ce, lane, hi_half, loff, bias, row_delta, data_size, s_off, lo, hi, acc, pending);
  }
  win_flush<SH, STRIDE, GEN>(lo, hi, acc, hi_half);
}

struct ReduceArgs {
  const int32_t *sums;
  const double *centers;
  int32_t *flags;
  b2s_matcher_params p;
  b2s_search s;
  b2s_grid_info g;
  double scale;
  int n, nx, ny, na;
  double *probs_all;
  b2s_match_result *results;
  int k_first, mode;
  double *part_best;
  const double *glob_best;
  double *tie_out;
  const double *tie_in;
  const int32_t *keep;   // [B][na] angles left by k_prune_select (nullptr: every angle)
  const int32_t *nkeep;  // [B]
};


template <int STRIDE, bool GEN>
__global__ void __launch_bounds__(WIN_THREADS, 1)
    k_sweep_window(const uint8_t *__restrict__ grids, size_t grid_pitch, int data_size, int copy_bytes,
                   const int32_t *__restrict__ lists, const int32_t *__restrict__ counts,
                   const int32_t *__restrict__ starts, const int32_t *__restrict__ flags, int batch, int n, int na,
                   int nx, int ny, int width_step, int32_t *__restrict__ sums, int *__restrict__ work_counter,
                   int band_rows, int nbands, int band_bytes, int neg_bands, const int32_t *__restrict__ keep,
                   const int32_t *__restrict__ nkeep) {
  // Grids larger than shared memory are swept in `nbands` row bands: a work unit is (match, band, 32-row candidate
  // tile); the image holds the rows that tile of a window whose ORIGIN lies in the band can touch (band_rows +
  // STRIDE * 31 + 2), k_offsets_sorted grouped the beams by the band of their origin (bands [0, neg_bands) hold origins
  // BELOW the grid, whose upper tiles still reach it), and the partial sums of the bands are combined with RED.ADD.
  // keep != nullptr: only the angles keep[b][0 .. nkeep[b]) of match b are swept (k_prune_select; nbands == 1).
  extern __shared__ __align__(128) unsigned char smem[];
  uint8_t *sgrid = smem;  // [WIN_GUARD zeros][band image][WIN_GUARD zeros]
  __shared__ uint64_t bar;
  __shared__ int s_unit, s_item;
  __shared__ __align__(16) int32_t s_offsets[WIN_THREADS / 32][32];  // per-warp staging of 32 window origins

  const int lane = threadIdx.x & 31;
  int32_t *s_off = s_offsets[threadIdx.x >> 5];
  constexpr int CPT = 32 / STRIDE;  // candidates per tile row (a tile row is always 32 bytes)
  const int tiles_x = (nx + CPT - 1) / CPT, tiles_y = (ny + 31) >> 5;
  const int unit_tiles_y = nbands > 1 ? tiles_y : 1;        // banded: one row tile per unit
  const int tiles_per_angle = tiles_x * (nbands > 1 ? 1 : tiles_y);
  // word rotation of this lane (see win_load): lanes whose rows start in the same bank get different rotations
  int hi_half = lane >> 4;
  int loff[8];
  if (GEN) {
    const int step = ((width_step >> 2) * STRIDE) & 31;
    const int m = step ? (step & -step) : 32;  // gcd(step, 32): lanes L and L + 32/m share a row-start bank
    hi_half = ((lane * m) >> 5) & 7;
  }
#pragma unroll
  for (int j = 0; j < 8; j++) loff[j] = 4 * ((j + hi_half) & 7);
  const int list_cap = n + LIST_PAD * nbands;
  const int ngroups = 8 * nbands;

  for (int i = threadIdx.x; i < WIN_GUARD / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(sgrid)[i] = 0;  // leading guard
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  uint32_t parity = 0;

  while (true) {
    if (threadIdx.x == 0) {
      s_unit = atomicAdd(work_counter, 1);
      s_item = 0;
    }
    __syncthreads();
    const int unit = s_unit;
    if (unit >= batch * nbands * unit_tiles_y) break;
    const int b = unit / (nbands * unit_tiles_y), band = (unit / unit_tiles_y) % nbands, unit_ty = unit % unit_tiles_y;
    const int f = flags[b];
    if ((f & 2) || !(f & 1)) {  // out-of-range lattice (error) or irregular lattice (generic kernel takes it)
      __syncthreads();
      continue;
    }
    // first / one-past-last grid row of this unit's image (the whole grid when nbands == 1)
    const int row0 = (band - neg_bands) * band_rows + STRIDE * unit_ty * 32;
    const int lo_row = max(row0, 0);
    const int band_lo = lo_row * width_step;  // flat index of the first staged byte (multiple of 16)
    int bytes = nbands > 1 ? min((((row0 - lo_row) * width_step + band_bytes) + 15) & ~15, copy_bytes - band_lo) : copy_bytes;
    if (nbands > 1) {
      // nothing to do when the image misses the grid or no beam of any angle has its origin in this band
      int any = 0;
      if (bytes > 0)
        for (int i = threadIdx.x; i < na * 8; i += blockDim.x) any |= counts[((size_t)b * na + (i >> 3)) * ngroups + band * 8 + (i & 7)];
      if (!__syncthreads_or(any)) continue;
    }
    // ---- stage this unit's band image: TMA bulk copies, 32 KB each, one mbarrier phase ----
    if (threadIdx.x == 0) {
      fence_proxy_async();  // earlier generic-proxy reads of sgrid are ordered before the async-proxy writes
      mbar_expect_tx(&bar, (uint32_t)bytes);
      const uint8_t *src = grids + (size_t)b * grid_pitch + band_lo;
      for (int off = 0; off < bytes; off += 32768) {
        int len = min(32768, bytes - off);
        bulk_g2s(sgrid + WIN_GUARD + off, src + off, (uint32_t)len, &bar);
      }
    }
    if (threadIdx.x < WIN_GUARD / 4) reinterpret_cast<uint32_t *>(sgrid + WIN_GUARD + bytes)[threadIdx.x] = 0;  // trailing guard
    mbar_wait(&bar, parity);
    parity ^= 1;
    __syncthreads();
    const int bias = WIN_GUARD - band_lo;

    int32_t *bsums = sums + (size_t)b * na * nx * ny;
    const int items = (keep ? nkeep[b] : na) * tiles_per_angle;
    while (true) {
      int item = 0;
      if (lane == 0) item = atomicAdd(&s_item, 1);
      item = __shfl_sync(0xffffffffu, item, 0);
      if (item >= items) break;
      int k, ty, tx;
      if (nbands > 1) {
        k = item / tiles_x; tx = item % tiles_x; ty = unit_ty;
      } else {
        k = item / (tiles_x * tiles_y);
        const int t = item % (tiles_x * tiles_y);
        ty = t / tiles_x; tx = t % tiles_x;
      }
      if (keep) k = keep[(size_t)b * na + k];
      const int row_delta = STRIDE * (ty * 32 + lane) * width_step + tx * 32;  // this lane's row start relative to a beam's origin
      const int32_t *list = lists + ((size_t)b * na + k) * list_cap;
      const int32_t *cn = counts + ((size_t)b * na + k) * ngroups + band * 8;
      const int32_t *sg = starts + ((size_t)b * na + k) * ngroups + band * 8;

      uint32_t acc[32];
#pragma unroll
      for (int j = 0; j < 32; j++) acc[j] = 0;
      uint32_t lo[9], hi[9];
#pragma unroll
      for (int j = 0; j < 9; j++) { lo[j] = 0; hi[j] = 0; }
      // groups of this band: I0 I1 I2 I3 E0 E1 E2 E3 (interior / edge beams of each alignment class)
      const int cols = min(CPT, nx - tx * CPT);
      win_class_pair<0, STRIDE, GEN>(sgrid, list + sg[0], cn[0], list + sg[4], cn[4], cols, lane, hi_half, loff, row_delta, bias, data_size, s_off, lo, hi, acc);
      win_class_pair<1, STRIDE, GEN>(sgrid, list + sg[1], cn[1], list + sg[5], cn[5], cols, lane, hi_half, loff, row_delta, bias, data_size, s_off, lo, hi, acc);
      win_class_pair<2, STRIDE, GEN>(sgrid, list + sg[2], cn[2], list + sg[6], cn[6], cols, lane, hi_half, loff, row_delta, bias, data_size, s_off, lo, hi, acc);
      win_class_pair<3, STRIDE, GEN>(sgrid, list + sg[3], cn[3], list + sg[7], cn[7], cols, lane, hi_half, loff, row_delta, bias, data_size, s_off, lo, hi, acc);

      // ---- write / accumulate this lane's row ----
      const int iy = ty * 32 + lane;
      if (iy < ny) {
        int32_t *dst = bsums + ((size_t)k * ny + iy) * nx + tx * CPT;
        if (nbands == 1) {
#pragma unroll
          for (int x = 0; x < CPT; x++)
            if (tx * CPT + x < nx) dst[x] = (int32_t)acc[x];
        } else {
#pragma unroll
          for (int x = 0; x < CPT; x++)
            if (tx * CPT + x < nx && acc[x]) atomicAdd(dst + x, (int32_t)acc[x]);
        }
      }
    }
    __syncthreads();  // everyone is done with sgrid before the next unit's copy is issued
  }
}

// ----------------------------------------------------------------------------------------------
// k_reduce: the fp64 tail of CorrelateScan (Mapper.cpp:397-523): penalties, best response, per-cell maxima,
// tie-averaged pose, positional covariance.  One CTA per match.  Candidate order of the reference is
// (iy, ix, k) with linear index (iy*nx + ix)*na + k; ties are summed sequentially in that order when there are
// at most RED_MAX_TIES of them (bit-identical to the reference), otherwise by a fixed-order tree.
// ----------------------------------------------------------------------------------------------
constexpr int RED_THREADS = 512;
// (stand-alone k_reduce: 60 registers, two CTAs per SM, so one match's serial tail overlaps another's streaming pass)
constexpr int RED_MAX_TIES = 512;
constexpr int RED_UNROLL = 8;

__device__ __forceinline__ double candidate_response(int32_t isum, int n, bool do_penalize, double sq_xy,
                                                     double angle, double center_h, const b2s_matcher_params &p) {
  double response = (double)isum;
  response /= (double)((uint32_t)n * (uint32_t)GRID_OCCUPIED);  // Mapper.cpp:852
  if (do_penalize && !double_equal(response, 0.0)) {
    double dpen = 1.0 - (DISTANCE_PENALTY_GAIN * sq_xy / p.distance_variance_penalty);
    dpen = dmax(dpen, p.minimum_distance_penalty);
    double sq_a = (angle - center_h) * (angle - center_h);
    double apen = 1.0 - (ANGLE_PENALTY_GAIN * sq_a / p.angle_variance_penalty);
    apen = dmax(apen, p.minimum_angle_penalty);
    response *= (dpen * apen);
  }
  return response;
}

// float score of a candidate (see k_reduce): relative error < 3e-7 vs candidate_response
__device__ __forceinline__ float red_fscore(int32_t isum, float apf_k, float dpf, float inv_d, bool do_penalize,
                                            bool &ambiguous) {
  const float u = (float)isum * inv_d;  // unpenalised response
  ambiguous = (u > 0.5e-6f) && (u < 2.0e-6f);
  if (!do_penalize || u <= 1.0e-6f) return u;
  return (float)isum * apf_k * dpf;
}

__device__ __forceinline__ void reduce_match_body(const int b, const ReduceArgs &A) {
  const int32_t *sums = A.sums;  // no __restrict__ / no read-only path: the fused sweep wrote them in this very launch
  const double *__restrict__ centers = A.centers;
  const int32_t *__restrict__ flags = A.flags;
  const b2s_matcher_params &p = A.p;
  const b2s_search &s = A.s;
  const b2s_grid_info &g = A.g;
  const double scale = A.scale;
  const int n = A.n, nx = A.nx, ny = A.ny, na = A.na;
  double *__restrict__ probs_all = A.probs_all;
  b2s_match_result *__restrict__ results = A.results;
  const int k_first = A.k_first, mode = A.mode;
  double *__restrict__ part_best = A.part_best;
  const double *__restrict__ glob_best = A.glob_best;
  double *__restrict__ tie_out = A.tie_out;
  const double *__restrict__ tie_in = A.tie_in;
  const int tid = threadIdx.x;
  const int ncell = nx * ny;
  b2s_match_result *res = results + b;
  if (flags[b] & 2) {
    if (tid == 0) res->status = B2S_ERR_OUT_OF_RANGE;
    return;
  }
  const int32_t *bs = sums + (size_t)b * na * ncell;
  const double cx = centers[3 * b], cy = centers[3 * b + 1], ch = centers[3 * b + 2];
  const double start_x = -s.offset_x, start_y = -s.offset_y, start_a = ch - s.angle_offset;
  const int pstep = (g.search_side + 7) & ~7;
  double *probs = probs_all + (size_t)b * pstep * g.search_side;
  const double pox = cx - s.offset_x, poy = cy - s.offset_y;  // Mapper.cpp:332-333
  const bool pen = s.do_penalize != 0;

  __shared__ double red[8];
  __shared__ double cov_terms[4][RED_THREADS];  // also the scratch of the block-wide max reduction
  __shared__ float s_apf[1024];  // per-angle factor (anglePenalty / (N*100)) as float
  __shared__ int s_err, s_count;
  __shared__ int tie_idx[RED_MAX_TIES];
  __shared__ int sorted[RED_MAX_TIES];
  __shared__ double s_best;
  __shared__ double s_mean[3];
  __shared__ int s_keep[1024];  // angle indices the table-driven passes visit, ascending
  if (tid == 0) { s_err = 0; s_count = 0; }
  if (!s.fine && mode <= 1)
    for (int i = tid; i < pstep * g.search_side; i += RED_THREADS) probs[i] = 0.0;  // Clear (Mapper.cpp:329)

  // Float pre-filter.  The exact fp64 response (reference operation order, candidate_response) is only needed for
  // candidates that can be a maximum or a tie; a float score f = isum * w(c,k) with relative error < 3e-7 bounds it:
  // a candidate whose f is more than 2e-6 (relative) below the largest f of its cell / below (best - 1e-6) cannot
  // be the cell maximum / a tie.  Candidates whose unpenalised response is near the 1e-6 DoubleEqual threshold of
  // the penalty test (Mapper.cpp:399) are always evaluated exactly.
  const bool tab = na <= 1024;
  const double D = (double)((uint32_t)n * (uint32_t)GRID_OCCUPIED);
  const float inv_d = (float)(1.0 / D);
  for (int k = tid; k < na && tab; k += RED_THREADS) {
    double apen = 1.0;
    if (pen) {
      const double angle = start_a + (double)(uint32_t)(k_first + k) * s.angle_res;
      apen = dmax(1.0 - (ANGLE_PENALTY_GAIN * ((angle - ch) * (angle - ch)) / p.angle_variance_penalty), p.minimum_angle_penalty);
    }
    s_apf[k] = (float)(apen / D);
  }
  // a pruned sweep computed only the angles k_prune_select kept; every candidate that can be the best, a tie or a
  // per-cell maximum the covariance reads lies in one of them (see k_prune_select)
  const int nk = (tab && A.keep) ? A.nkeep[b] : na;
  for (int j = tid; j < nk && tab; j += RED_THREADS) s_keep[j] = A.keep ? A.keep[(size_t)b * na + j] : j;
  __syncthreads();

  // ---- pass 1: best response + per-cell maxima (Mapper.cpp:430-451); one thread per (x,y) cell ----
  // One read of the cell's nA sums: the running float maximum remembers its angle and whether any OTHER candidate
  // came within the filter margin of it; if none did, the exact maximum is at that angle and needs one fp64
  // evaluation, otherwise (near-ties, e.g. equal sums under the clamped penalty) the row is re-read and every
  // candidate inside the margin is evaluated exactly.
  double best = -1.0;
  float fmax0 = 0.0f, fmax1 = 0.0f;  // float maxima of this thread's first two cells, kept for pass 2
  bool known0 = false, known1 = false;
  for (int c = tid; c < ncell && mode <= 1; c += RED_THREADS) {
    const int iy = c / nx, ix = c % nx;
    const double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
    const double sq = x * x + y * y;
    double cell_best = -1.0;
    if (tab) {
      const float dpf = (float)dmax(1.0 - (DISTANCE_PENALTY_GAIN * sq / p.distance_variance_penalty), p.minimum_distance_penalty);
      float fmax = -1.0f;
      int kmax = 0;
      int32_t vmax = 0;
      bool near = false, any_amb = false;
      for (int j0 = 0; j0 < nk; j0 += RED_UNROLL) {
        int32_t v[RED_UNROLL];
#pragma unroll
        for (int u = 0; u < RED_UNROLL; u++) v[u] = (j0 + u < nk) ? __ldcg(bs + (size_t)s_keep[j0 + u] * ncell + c) : 0;
#pragma unroll
        for (int u = 0; u < RED_UNROLL; u++) {
          if (j0 + u >= nk) continue;
          const int k = s_keep[j0 + u];
          bool amb;
          const float f = red_fscore(v[u], s_apf[k], dpf, inv_d, pen, amb);
          any_amb |= amb;
          if (f > fmax) {
            near = fmax >= f * (1.0f - 2.0e-6f) - 1.0e-30f;  // the old maximum (and only it or its own near ones) may still be near
            fmax = f; kmax = k; vmax = v[u];
          } else if (f >= fmax * (1.0f - 2.0e-6f) - 1.0e-30f) {
            near = true;
          }
        }
      }
      if (c == tid) { fmax0 = fmax; known0 = !any_amb; }
      else if (c == tid + RED_THREADS) { fmax1 = fmax; known1 = !any_amb; }
      if (!near && !any_amb) {
        const double angle = start_a + (double)(uint32_t)(k_first + kmax) * s.angle_res;
        cell_best = candidate_response(vmax, n, pen, sq, angle, ch, p);
      } else if (fmax == 0.0f && !any_amb) {
        cell_best = 0.0;  // every sum is 0: response 0 / D, never penalised (Mapper.cpp:399)
      } else {
        const float thr = fmax * (1.0f - 2.0e-6f) - 1.0e-30f;
        for (int j0 = 0; j0 < nk; j0 += RED_UNROLL) {
          int32_t v[RED_UNROLL];
#pragma unroll
          for (int u = 0; u < RED_UNROLL; u++) v[u] = (j0 + u < nk) ? __ldcg(bs + (size_t)s_keep[j0 + u] * ncell + c) : 0;
#pragma unroll
          for (int u = 0; u < RED_UNROLL; u++) {
            if (j0 + u >= nk) continue;
            const int k = s_keep[j0 + u];
            bool amb;
            const float f = red_fscore(v[u], s_apf[k], dpf, inv_d, pen, amb);
            if (f >= thr || amb) {
              const double angle = start_a + (double)(uint32_t)(k_first + k) * s.angle_res;
              cell_best = dmax(cell_best, candidate_response(v[u], n, pen, sq, angle, ch, p));
            }
          }
        }
      }
    } else {
      for (int k = 0; k < na; k++) {
        const double angle = start_a + (double)(uint32_t)(k_first + k) * s.angle_res;
        cell_best = dmax(cell_best, candidate_response(__ldcg(bs + (size_t)k * ncell + c), n, pen, sq, angle, ch, p));
      }
    }
    best = dmax(best, cell_best);
    if (!s.fine) {
      const int32_t px = world_to_grid_1(cx + x, pox, scale), py = world_to_grid_1(cy + y, poy, scale);
      if (!(px >= 0 && px < g.search_side && py >= 0 && py < g.search_side)) {
        s_err = 1;  // GetDataPointer -> GridIndex throws (Karto.h:4553-4557)
      } else {
        // distinct candidates can share a probs cell only on degenerate lattices; max is order-free
        unsigned long long *pp = reinterpret_cast<unsigned long long *>(probs + px + (size_t)py * pstep);
        atomicMax(pp, (unsigned long long)__double_as_longlong(dmax(cell_best, 0.0)));
      }
    }
  }
  cov_terms[0][tid] = best;
  __syncthreads();
  for (int d = RED_THREADS / 2; d > 0; d >>= 1) {
    if (tid < d) cov_terms[0][tid] = dmax(cov_terms[0][tid], cov_terms[0][tid + d]);
    __syncthreads();
  }
  if (tid == 0) s_best = mode <= 1 ? cov_terms[0][0] : glob_best[b];
  __syncthreads();
  best = s_best;
  if (s_err) {
    if (tid == 0) res->status = B2S_ERR_OUT_OF_RANGE;
    return;
  }
  if (mode == 1) {  // split sweep, phase 1: this angle subset's best (the per-cell maxima are in `probs`)
    if (tid == 0) { part_best[b] = best; res->status = B2S_OK; }
    return;
  }

  // ---- pass 2: poses tied with the best (Mapper.cpp:455-487) ----
  double ax = 0, ay = 0, tx = 0, ty = 0;
  const float tie_thr = (float)((best - KT_TOLERANCE) * (1.0 - 1.0e-6)) - 1.0e-9f;
  for (int c = tid; c < ncell && mode != 3; c += RED_THREADS) {
    if (c == tid && known0 && fmax0 < tie_thr) continue;  // no candidate of this cell can tie (pass 1's maximum)
    if (c == tid + RED_THREADS && known1 && fmax1 < tie_thr) continue;
    const int iy = c / nx, ix = c % nx;
    const double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
    const double sq = x * x + y * y;
    const float dpf = (float)dmax(1.0 - (DISTANCE_PENALTY_GAIN * sq / p.distance_variance_penalty), p.minimum_distance_penalty);
    for (int j0 = 0; j0 < nk; j0 += RED_UNROLL) {
      int32_t v[RED_UNROLL];
#pragma unroll
      for (int u = 0; u < RED_UNROLL; u++)
        v[u] = (j0 + u < nk) ? __ldcg(bs + (size_t)(tab ? s_keep[j0 + u] : j0 + u) * ncell + c) : 0;
#pragma unroll
      for (int u = 0; u < RED_UNROLL; u++) {
        if (j0 + u >= nk) continue;
        const int k = tab ? s_keep[j0 + u] : j0 + u;
        if (tab) {
          bool amb;
          const float f = red_fscore(v[u], s_apf[k], dpf, inv_d, pen, amb);
          if (f < tie_thr && !amb) continue;
        }
        const double angle = start_a + (double)(uint32_t)(k_first + k) * s.angle_res;
        const double r = candidate_response(v[u], n, pen, sq, angle, ch, p);
        if (double_equal(r, best)) {
          const double h = normalize_angle(angle);
          ax += cx + x; ay += cy + y; tx += cos(h); ty += sin(h);
          int slot = atomicAdd(&s_count, 1);
          if (slot < RED_MAX_TIES) tie_idx[slot] = c * na + k;
        }
      }
    }
  }
  __syncthreads();
  if (mode == 3 && tid == 0) s_count = (int)tie_in[5 * b + 4];
  __syncthreads();
  const int total = s_count;
  if (total == 0 && mode != 2) {
    if (tid == 0) res->status = B2S_ERR_NO_BEST_POSE;  // Mapper.cpp:484-487
    return;
  }
  if (mode == 3) {
    if (tid == 0) { red[0] = tie_in[5 * b]; red[1] = tie_in[5 * b + 1]; red[2] = tie_in[5 * b + 2]; red[3] = tie_in[5 * b + 3]; }
    __syncthreads();
  } else if (total <= RED_MAX_TIES && mode == 0) {
    // rank-sort the tie list by reference linear index, then one thread sums in that exact order
    for (int i = tid; i < total; i += RED_THREADS) {
      int v = tie_idx[i], rank = 0;
      for (int j = 0; j < total; j++) rank += (tie_idx[j] < v);
      sorted[rank] = v;
    }
    __syncthreads();
    if (tid == 0) {
      double sx = 0, sy = 0, cxs = 0, sys = 0;
      for (int i = 0; i < total; i++) {
        int v = sorted[i];
        int c = v / na, k = v % na;
        int iy = c / nx, ix = c % nx;
        double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
        double h = normalize_angle(start_a + (double)(uint32_t)(k_first + k) * s.angle_res);
        sx += cx + x; sy += cy + y; cxs += cos(h); sys += sin(h);
      }
      red[0] = sx; red[1] = sy; red[2] = cxs; red[3] = sys;
    }
    __syncthreads();
  } else {
    // fixed-order tree reduction (deterministic; differs from the sequential sum only in the last bits)
    cov_terms[0][tid] = ax; cov_terms[1][tid] = ay; cov_terms[2][tid] = tx; cov_terms[3][tid] = ty;
    __syncthreads();
    for (int d = RED_THREADS / 2; d > 0; d >>= 1) {
      if (tid < d)
        for (int q = 0; q < 4; q++) cov_terms[q][tid] += cov_terms[q][tid + d];
      __syncthreads();
    }
    if (tid == 0) { red[0] = cov_terms[0][0]; red[1] = cov_terms[1][0]; red[2] = cov_terms[2][0]; red[3] = cov_terms[3][0]; }
    __syncthreads();
  }
  if (mode == 2) {  // split sweep, phase 2: this subset's tie sums {x, y, cos, sin, count}
    if (tid == 0) {
      tie_out[5 * b] = red[0]; tie_out[5 * b + 1] = red[1]; tie_out[5 * b + 2] = red[2]; tie_out[5 * b + 3] = red[3];
      tie_out[5 * b + 4] = (double)total;
    }
    return;
  }
  if (tid == 0) {
    double sx = red[0], sy = red[1], cxs = red[2], sys = red[3];
    sx /= total; sy /= total; cxs /= total; sys /= total;
    s_mean[0] = sx; s_mean[1] = sy; s_mean[2] = atan2(sys, cxs);
  }
  __syncthreads();
  const double mean0 = s_mean[0], mean1 = s_mean[1], mean2 = s_mean[2];

  // ---- covariance ----
  if (!s.fine) {
    // ComputePositionalCovariance (Mapper.cpp:535-630).  The four running sums are accumulated in the reference's
    // (y, x) order: the per-cell terms are produced in parallel (0.0 for cells the reference skips, which leaves a
    // sum unchanged), then four threads add one series each sequentially.
    double cov[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    const bool tiny = best < KT_TOLERANCE;
    double axx = 0, axy = 0, ayy = 0, norm = 0;  // live in threads 0..3 (one series each)
    const double dx = mean0 - cx, dy = mean1 - cy;
    if (!tiny) {
      for (int base = 0; base < ncell; base += RED_THREADS) {
        const int c = base + tid;
        double t0 = 0, t1 = 0, t2 = 0, t3 = 0;
        if (c < ncell) {
          const int iy = c / nx, ix = c % nx;
          const double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
          const int32_t px = world_to_grid_1(cx + x, pox, scale), py = world_to_grid_1(cy + y, poy, scale);
          if (!(px >= 0 && px < g.search_side && py >= 0 && py < g.search_side)) {
            s_err = 1;
          } else {
            const double response = probs[px + (size_t)py * pstep];
            if (response >= (best - 0.1)) {
              t0 = response;
              t1 = ((x - dx) * (x - dx) * response);
              t2 = ((x - dx) * (y - dy) * response);
              t3 = ((y - dy) * (y - dy) * response);
            }
          }
        }
        cov_terms[0][tid] = t0; cov_terms[1][tid] = t1; cov_terms[2][tid] = t2; cov_terms[3][tid] = t3;
        __syncthreads();
        const int cnt = min(RED_THREADS, ncell - base);
        if (tid < 4) {
          double acc = tid == 0 ? norm : (tid == 1 ? axx : (tid == 2 ? axy : ayy));
          for (int i = 0; i < cnt; i++) acc += cov_terms[tid][i];
          if (tid == 0) norm = acc; else if (tid == 1) axx = acc; else if (tid == 2) axy = acc; else ayy = acc;
        }
        __syncthreads();
      }
      if (tid == 1) red[1] = axx;
      if (tid == 2) red[2] = axy;
      if (tid == 3) red[3] = ayy;
      __syncthreads();
    }
    if (s_err) {
      if (tid == 0) res->status = B2S_ERR_OUT_OF_RANGE;
      return;
    }
    if (tid != 0) return;
    if (tiny) {
      cov[0] = MAX_VARIANCE; cov[4] = MAX_VARIANCE;
      cov[8] = 4 * (s.angle_res * s.angle_res);
    } else {
      axx = red[1]; axy = red[2]; ayy = red[3];
      if (norm > KT_TOLERANCE) {
        double vxx = axx / norm, vxy = axy / norm, vyy = ayy / norm;
        const double vthth = 4 * (s.angle_res * s.angle_res);
        vxx = dmax(vxx, 0.1 * (s.res_x * s.res_x));
        vyy = dmax(vyy, 0.1 * (s.res_y * s.res_y));
        const double mult = 1.0 / best;
        cov[0] = vxx * mult; cov[1] = vxy * mult; cov[3] = vxy * mult; cov[4] = vyy * mult; cov[8] = vthth;
      }
      if (double_equal(cov[0], 0.0)) cov[0] = MAX_VARIANCE;
      if (double_equal(cov[4], 0.0)) cov[4] = MAX_VARIANCE;
    }
    for (int i = 0; i < 9; i++) res->cov[i] = cov[i];
  }
  if (tid != 0) return;
  res->pose[0] = mean0; res->pose[1] = mean1; res->pose[2] = mean2;
  // un-clamped best goes through `response` for k_angular_cov; it clamps afterwards.  Coarse: clamp here.
  res->response = s.fine ? best : (best > 1.0 ? 1.0 : best);  // Mapper.cpp:514-517
  res->status = B2S_OK;
  res->tie_count = total;
}

__global__ void __launch_bounds__(RED_THREADS, 2) k_reduce(ReduceArgs A) {
  reduce_match_body(blockIdx.x, A);
}

// ----------------------------------------------------------------------------------------------
// k_prune_select: which angles of a stride-1, one-tile (nx, ny <= 32) window sweep can change a result.  One CTA per
// match, the phase-split 4x4 max-pool image (k_grid_mp4) staged into shared memory by TMA bulk copy.
//
// 1. Bound.  For angle k and 4x4 candidate block (by, bx), every candidate's integer sum is at most
//    S(k, by, bx) = sum over the listed beams i of MP4[a_i + 4*by*width_step + 4*bx]  (a_i = window origin).  Beams
//    k_offsets_sorted dropped as empty windows add 0 to every exact sum and are left out here too.  The penalised bound
//    applies the reference's fp64 operations to S, the block's largest distance penalty and the angle's penalty;
//    correctly rounded operations are monotone, so it is >= every candidate's response.  A candidate whose unpenalised
//    response is within KT_TOLERANCE of 0 is not penalised (Mapper.cpp:399): it is <= min(S / (N*100), 1.1e-6).
//    Warps pull angles; lane = (beam group g, block row by); a beam row's 8 block columns are 8 consecutive bytes of
//    one phase, summed as packed u16 lanes.  bound[k] = max over the angle's blocks; the top (bound, angle, block)
//    is kept with a packed 64-bit atomicMax.
// 2. Seed.  The 16 candidates of the top block are evaluated exactly (same fp64 operations as k_reduce); their
//    maximum L is a response of the volume, so L <= best.
// 3. Select.  Angle k is kept iff bound[k] >= L - 0.1 - 1e-9 (the 1e-9 only ever keeps more).
// Why the results are unchanged: the outputs of CorrelateScan depend on the best response, on the candidates within
// KT_TOLERANCE of it (the ties, summed in (y, x, theta) order) and, for the covariance, on the per-cell maxima over
// angles of the cells whose maximum is >= best - 0.1 (ComputePositionalCovariance, Mapper.cpp:586).  Each of these is a
// candidate with response >= best - 0.1 >= L - 0.1, so its block bound, and hence its angle's bound, clears the cut:
// its angle is kept.  So the best, the tie set and its order, and every per-cell maximum the covariance reads come out
// identical when k_sweep_window and k_reduce visit only the kept angles.  A cell whose true maximum is below the cut
// may get a smaller partial maximum, but it is excluded either way.  (When best < 0.1 every bound clears the cut.)
// Irregular lattices (k_sweep_generic sweeps every angle) keep every angle; out-of-range lattices keep none.
// ----------------------------------------------------------------------------------------------
constexpr int PRUNE_THREADS = 512;
constexpr double PRUNE_CUT = 0.1;     // ComputePositionalCovariance's window below the best response
constexpr double PRUNE_EPS = 1e-9;    // guard against rounding in the bound product
__global__ void __launch_bounds__(PRUNE_THREADS, 1)
    k_prune_select(const uint8_t *__restrict__ mp_all, size_t mp_pitch, int lq, int mp_guard,
                   const uint8_t *__restrict__ grids, size_t grid_pitch, int data_size, int width_step,
                   const int32_t *__restrict__ lists, const int32_t *__restrict__ counts,
                   const int32_t *__restrict__ starts, const int32_t *__restrict__ flags,
                   const double *__restrict__ centers, b2s_matcher_params p, b2s_search s, int n, int na, int nx,
                   int ny, int32_t *__restrict__ keep, int32_t *__restrict__ nkeep,
                   unsigned long long *__restrict__ stats) {
  extern __shared__ __align__(128) unsigned char smp[];  // [4][lq] phase-split MP4 image
  __shared__ uint64_t bar;
  __shared__ double s_ab[1024];     // per-angle bound
  __shared__ double s_dp[64];       // per-block largest distance penalty
  __shared__ double s_cand[16];     // exact responses of the top block's candidates
  __shared__ unsigned long long s_top;
  __shared__ int s_wc[PRUNE_THREADS / 32], s_kept;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int f = flags[b];
  if ((f & 2) || !(f & 1)) {
    const int nk = (f & 2) ? 0 : na;  // irregular: k_sweep_generic sweeps every angle, k_reduce reads every angle
    for (int k = tid; k < nk; k += PRUNE_THREADS) keep[(size_t)b * na + k] = k;
    if (tid == 0) {
      nkeep[b] = nk;
      if (nk) atomicAdd(stats + 1, (unsigned long long)nk);
    }
    return;
  }
  const int mp_bytes = 4 * lq;
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
    s_top = 0ull;
    s_kept = 0;
  }
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(&bar, (uint32_t)mp_bytes);
    const uint8_t *src = mp_all + (size_t)b * mp_pitch;
    for (int off = 0; off < mp_bytes; off += 32768) bulk_g2s(smp + off, src + off, (uint32_t)min(32768, mp_bytes - off), &bar);
  }
  const bool pen = s.do_penalize != 0;
  const double ch = centers[3 * b + 2];
  const double start_x = -s.offset_x, start_y = -s.offset_y, start_a = ch - s.angle_offset;
  const int nbx = (nx + 3) >> 2, nby = (ny + 3) >> 2;
  if (tid < 64) {
    const int by = tid >> 3, bx = tid & 7;
    double dp = 0.0;
    for (int dy = 0; dy < 4; dy++)
      for (int dx = 0; dx < 4; dx++) {
        const int iy = 4 * by + dy, ix = 4 * bx + dx;
        if (iy >= ny || ix >= nx) continue;
        const double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
        const double sq = x * x + y * y;
        dp = dmax(dp, dmax(1.0 - (DISTANCE_PENALTY_GAIN * sq / p.distance_variance_penalty), p.minimum_distance_penalty));
      }
    s_dp[tid] = dp;
  }
  mbar_wait(&bar, 0);
  __syncthreads();

  // ---- 1. bounds ----
  const int list_cap = n + LIST_PAD;
  const double D = (double)((uint32_t)n * (uint32_t)GRID_OCCUPIED);
  const int g = lane >> 3, by = lane & 7;
  const uint32_t row_off = (uint32_t)(4 * by * width_step + mp_guard);
  const uint32_t lim = (uint32_t)(data_size + 2 * mp_guard - 32);  // a row starting above lim reads only zero pool values
  for (int k = warp; k < na; k += PRUNE_THREADS / 32) {
    const size_t bk = (size_t)b * na + k;
    const int32_t *list = lists + bk * list_cap;
    const int total = starts[bk * 8 + 7] + counts[bk * 8 + 7];  // the 8 groups are contiguous
    uint32_t e0 = 0, o0 = 0, e1 = 0, o1 = 0;  // packed u16: block columns (0, 2), (1, 3), (4, 6), (5, 7)
    uint32_t sum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    auto flush = [&]() {
      sum[0] += e0 & 0xffffu; sum[2] += e0 >> 16; sum[1] += o0 & 0xffffu; sum[3] += o0 >> 16;
      sum[4] += e1 & 0xffffu; sum[6] += e1 >> 16; sum[5] += o1 & 0xffffu; sum[7] += o1 >> 16;
      e0 = o0 = e1 = o1 = 0;
    };
    int chunks = 0;
    for (int ib = 0; ib < total; ib += 32) {
      const int32_t mine = (ib + lane < total) ? __ldg(list + ib + lane) : WIN_SKIP;
#pragma unroll
      for (int jj = 0; jj < 8; jj++) {
        uint32_t u = (uint32_t)__shfl_sync(0xffffffffu, mine, jj * 4 + g) + row_off;
        // below -mp_guard or past data_size + mp_guard - 32 every pool value of the row is 0: read the zero-valued
        // start of phase 0 instead (branch-free, so the unrolled beams' loads overlap)
        u = u <= lim ? u : 0u;
        const uint32_t t = u >> 2, sh = (t & 3) * 8;
        const uint32_t *w = reinterpret_cast<const uint32_t *>(smp + (u & 3) * lq + (t & ~3u));
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
        const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
        e0 += lo & 0x00ff00ffu; o0 += (lo >> 8) & 0x00ff00ffu;
        e1 += hi & 0x00ff00ffu; o1 += (hi >> 8) & 0x00ff00ffu;
      }
      if (++chunks == 64) { flush(); chunks = 0; }  // 64 x 8 beams x 127 < 65536
    }
    flush();
#pragma unroll
    for (int q = 0; q < 8; q++) {
      sum[q] += __shfl_xor_sync(0xffffffffu, sum[q], 8);
      sum[q] += __shfl_xor_sync(0xffffffffu, sum[q], 16);
    }
    const double angle = start_a + (double)(uint32_t)k * s.angle_res;
    const double apen = dmax(1.0 - (ANGLE_PENALTY_GAIN * ((angle - ch) * (angle - ch)) / p.angle_variance_penalty),
                             p.minimum_angle_penalty);
    double bk_best = -1.0;
    unsigned long long key = 0ull;
    if (g == 0 && by < nby) {
#pragma unroll
      for (int bx = 0; bx < 8; bx++) {
        if (bx >= nbx) continue;
        const double r = (double)sum[bx] / D;
        const double bd = pen ? dmax(r * (s_dp[by * 8 + bx] * apen), r < 1.1e-6 ? r : 1.1e-6) : r;
        if (bd > bk_best) {
          bk_best = bd;
          key = ((unsigned long long)__double_as_longlong(bd) & ~0xffffull) | (unsigned long long)((k << 6) | (by << 3) | bx);
        }
      }
    }
#pragma unroll
    for (int d = 4; d > 0; d >>= 1) {
      bk_best = dmax(bk_best, __shfl_xor_sync(0xffffffffu, bk_best, d));
      const unsigned long long o = __shfl_xor_sync(0xffffffffu, key, d);
      key = o > key ? o : key;
    }
    if (lane == 0) {
      s_ab[k] = bk_best;
      atomicMax(&s_top, key);
    }
  }
  __syncthreads();

  // ---- 2. seed: the top block's candidates, exactly ----
  {
    const unsigned long long key = s_top;
    const int k = (int)((key >> 6) & 1023), tby = (int)((key >> 3) & 7), tbx = (int)(key & 7);
    const int iy = 4 * tby + (warp >> 2), ix = 4 * tbx + (warp & 3);  // 16 warps, one candidate each
    const bool valid = iy < ny && ix < nx;
    int32_t isum = 0;
    if (valid) {
      const size_t bk = (size_t)b * na + k;
      const int32_t *list = lists + bk * list_cap;
      const int total = starts[bk * 8 + 7] + counts[bk * 8 + 7];
      const uint8_t *grid = grids + (size_t)b * grid_pitch;
      const int32_t rel = iy * width_step + ix;
      for (int i = lane; i < total; i += 32) {
        const int32_t idx = (int32_t)((uint32_t)__ldg(list + i) + (uint32_t)rel);
        if ((uint32_t)idx < (uint32_t)data_size) isum += grid[idx];
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) isum += __shfl_xor_sync(0xffffffffu, isum, d);
    if (lane == 0) {
      double r = -1.0;
      if (valid) {
        const double y = start_y + (double)(uint32_t)iy * s.res_y, x = start_x + (double)(uint32_t)ix * s.res_x;
        r = candidate_response(isum, n, pen, x * x + y * y, start_a + (double)(uint32_t)k * s.angle_res, ch, p);
      }
      s_cand[warp] = r;
    }
  }
  __syncthreads();
  double L = s_cand[0];
  for (int i = 1; i < 16; i++) L = dmax(L, s_cand[i]);
  const double cut = L - PRUNE_CUT - PRUNE_EPS;

  // ---- 3. select: compact the kept angles in ascending order ----
  for (int k0 = 0; k0 < na; k0 += PRUNE_THREADS) {
    const int k = k0 + tid;
    const bool kp = k < na && s_ab[k] >= cut;
    const unsigned bal = __ballot_sync(0xffffffffu, kp);
    if (lane == 0) s_wc[warp] = __popc(bal);
    __syncthreads();
    int off = s_kept;
    for (int w = 0; w < warp; w++) off += s_wc[w];
    off += __popc(bal & ((1u << lane) - 1u));
    if (kp) keep[(size_t)b * na + off] = k;
    __syncthreads();
    if (tid == 0)
      for (int w = 0; w < PRUNE_THREADS / 32; w++) s_kept += s_wc[w];
    __syncthreads();
  }
  if (tid == 0) {
    nkeep[b] = s_kept;
    atomicAdd(stats + 1, (unsigned long long)s_kept);
  }
}

// ----------------------------------------------------------------------------------------------
// k_angular_cov: ComputeAngularCovariance (Mapper.cpp:641-692).  One CTA per match; warps over angles,
// lanes over beams (GetResponse at the best cell), then thread 0 accumulates in angle order.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_angular_cov(const uint8_t *__restrict__ grids, size_t grid_pitch, b2s_grid_info g,
                  const double *__restrict__ grid_off, const int32_t *__restrict__ lut,
                  const double *__restrict__ centers, b2s_search s, double scale, int n, int na,
                  b2s_match_result *__restrict__ results) {
  const int b = blockIdx.x;
  b2s_match_result *res = results + b;
  if (res->status != B2S_OK) return;
  extern __shared__ double s_resp[];  // [na]
  __shared__ int32_t s_base;
  __shared__ int s_bad;
  const double best = res->response;
  if (threadIdx.x == 0) {
    int32_t gx = world_to_grid_1(res->pose[0], grid_off[2 * b], scale) + g.roi_x;
    int32_t gy = world_to_grid_1(res->pose[1], grid_off[2 * b + 1], scale) + g.roi_y;
    s_bad = !(gx >= 0 && gx < g.width && gy >= 0 && gy < g.height);
    s_base = gx + gy * g.width_step;
  }
  __syncthreads();
  if (s_bad) {
    if (threadIdx.x == 0) res->status = B2S_ERR_OUT_OF_RANGE;
    return;
  }
  const uint8_t *grid = grids + (size_t)b * grid_pitch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int k = warp; k < na; k += nw) {
    const int32_t *offs = lut + ((size_t)b * na + k) * n;
    int32_t sum = 0;
    for (int i = lane; i < n; i += 32) {
      int32_t o = offs[i];
      if (o == INVALID_SCAN) continue;
      int32_t idx = (int32_t)((uint32_t)s_base + (uint32_t)o);
      if (idx >= 0 && idx < g.data_size) sum += grid[idx];
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    if (lane == 0) {
      double r = (double)sum;
      r /= (double)((uint32_t)n * (uint32_t)GRID_OCCUPIED);
      s_resp[k] = r;
    }
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  const double ch = centers[3 * b + 2];
  const double best_angle = normalize_angle_difference(res->pose[2], ch);
  const double start = ch - s.angle_offset;
  double norm = 0.0, acc = 0.0;
  for (int k = 0; k < na; k++) {
    const double angle = start + (double)(uint32_t)k * s.angle_res;
    const double response = s_resp[k];
    if (response >= (best - 0.1)) {
      norm += response;
      acc += ((angle - best_angle) * (angle - best_angle) * response);
    }
  }
  if (norm > KT_TOLERANCE) {
    if (acc < KT_TOLERANCE) acc = s.angle_res * s.angle_res;
    acc /= norm;
  } else {
    acc = 1000 * (s.angle_res * s.angle_res);
  }
  res->cov[8] = acc;
  if (best > 1.0) res->response = 1.0;
}

// fine-stage search centre = coarse mean (Mapper.cpp:278): copy result poses into the centre array
__global__ void k_results_to_centers(const b2s_match_result *__restrict__ results, double *__restrict__ centers,
                                     int batch) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  centers[3 * b] = results[b].pose[0];
  centers[3 * b + 1] = results[b].pose[1];
  centers[3 * b + 2] = results[b].pose[2];
}

// split sweep: per-match status out of / back into the result records (all-reduced with MAX between the phases)
__global__ void k_status_pack(const b2s_match_result *__restrict__ results, int32_t *__restrict__ st, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < batch) st[b] = results[b].status;
}
__global__ void k_status_apply(b2s_match_result *__restrict__ results, const int32_t *__restrict__ st, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < batch && st[b] != 0) results[b].status = st[b];  // a rank saw an out-of-range candidate: the reference throws
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------

static b2s_status layout_from_params(const b2s_matcher_params *p, b2s_grid_info *g) {
  // ScanMatcher::Create (Mapper.cpp:126-172) + CorrelationGrid ctor (Mapper.h:920-1027) + Grid::Resize (Karto.h:4438)
  if (p->resolution <= 0 || p->search_size <= 0 || p->smear_deviation < 0 || p->range_threshold <= 0)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "ScanMatcher::Create: invalid parameters");
  uint32_t side = cast_u32(kround(p->search_size / p->resolution) + 1);
  uint32_t margin = cast_u32(ceil(p->range_threshold / p->resolution));
  int32_t grid_size = (int32_t)(side + 2 * margin);
  int32_t half_kernel = cast_i32(kround(2.0 * p->smear_deviation / p->resolution));
  uint32_t border = (uint32_t)(half_kernel + 1);
  g->width = grid_size + 2 * (int32_t)border;
  g->height = grid_size + 2 * (int32_t)border;
  g->width_step = (int32_t)(((size_t)g->width + 7) & ~(size_t)7);
  g->data_size = g->width_step * g->height;
  g->roi_x = g->roi_y = (int32_t)border;
  g->roi_w = g->roi_h = grid_size;
  g->kernel_size = 2 * half_kernel + 1;
  g->search_side = (int32_t)side;
  double resolution = 1.0 / (1.0 / p->resolution);
  double min_dev = 0.5 * resolution, max_dev = 10 * resolution;  // Mapper.h:1041-1053 throws
  if (!(p->smear_deviation >= min_dev && p->smear_deviation <= max_dev))
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "Mapper Error: smear deviation must be within [0.5, 10] x resolution");
  return B2S_OK;
}

template <class T>
static b2s_status dev_alloc(T **p, size_t count) {
  B2S_CUDA_CHECK(cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(count, 1) * sizeof(T)));
  return B2S_OK;
}

template <class T>
static b2s_status ensure_cap(T **p, size_t *cap, size_t count) {
  if (count <= *cap && *p) return B2S_OK;
  if (*p) B2S_CUDA_CHECK(cudaFree(*p));
  *p = nullptr;
  B2S_CUDA_CHECK(cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(count, 1) * sizeof(T)));
  *cap = count;
  return B2S_OK;
}

static b2s_status run_correlate(b2s_matcher *m, const b2s_search *s, bool centers_on_device, int k_first = 0,
                                int na_override = -1, int mode = 0);

// k_sweep_window over the lists of the last lookup stage with m->win's configuration; pruned: only the kept angles
static b2s_status launch_window(b2s_matcher *m, int B, int n, int na, int nx, int ny, bool pruned) {
  const WinLaunch &w = m->win;
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_work, 0, sizeof(int), m->stream));
  if (w.nbands > 1)  // bands accumulate with RED.ADD
    B2S_CUDA_CHECK(cudaMemsetAsync(m->d_sums, 0, sizeof(int32_t) * (size_t)B * na * nx * ny, m->stream));
  auto launch = [&](auto kern) -> b2s_status {
    B2S_CUDA_CHECK(raise_dyn_smem(kern, w.smem));
    kern<<<w.ctas, WIN_THREADS, w.smem, m->stream>>>(m->d_grids, m->grid_pitch, m->g.data_size, w.copy_bytes, m->d_lists,
                                                     m->d_counts, m->d_starts, m->d_flags, B, n, na, nx, ny,
                                                     m->g.width_step, m->d_sums, m->d_work, w.band_rows, w.nbands,
                                                     w.band_bytes, w.neg_bands, pruned ? m->d_keep : nullptr,
                                                     pruned ? m->d_nkeep : nullptr);
    return B2S_OK;
  };
  if (w.stride == 2) return w.gen ? launch(k_sweep_window<2, true>) : launch(k_sweep_window<2, false>);
  return w.gen ? launch(k_sweep_window<1, true>) : launch(k_sweep_window<1, false>);
}

// (re)build the per-match max-pool images k_prune_select stages into shared memory, when one fits there
static b2s_status build_mp4(b2s_matcher *m) {
  m->mp_valid = false;
  const b2s_grid_info &g = m->g;
  if (g.width_step % 8 != 0 || m->grid_high_bytes) return B2S_OK;  // no pruned sweep
  // >= 3*width_step + 3 + 32 (see k_grid_mp4) and > 3*width_step + 47: phase 0's first 12 bytes pool no grid cell
  m->mp_guard = (3 * g.width_step + 3 + 64 + 15) & ~15;
  m->mp_lq = ((g.data_size + 2 * m->mp_guard) / 4 + 16 + 15) & ~15;
  static size_t prune_static = 0;
  if (!prune_static) {
    cudaFuncAttributes fa;
    B2S_CUDA_CHECK(cudaFuncGetAttributes(&fa, k_prune_select));
    prune_static = fa.sharedSizeBytes;
  }
  const size_t bytes = 4 * (size_t)m->mp_lq;
  if (bytes + prune_static + 512 > (size_t)m->smem_optin) return B2S_OK;
  if (!m->d_mp4) {
    m->mp_pitch = (bytes + 127) & ~(size_t)127;
    b2s_status st = dev_alloc(&m->d_mp4, (size_t)m->max_batch * m->mp_pitch);
    if (st) return st;
  }
  const dim3 grid((unsigned)ceil_div(m->mp_lq / 4, 256), (unsigned)m->batch);
  k_grid_mp4<<<grid, 256, 0, m->stream>>>(m->d_grids, m->grid_pitch, g.data_size, g.width_step, m->mp_guard, m->mp_lq,
                                          m->d_mp4, m->mp_pitch);
  B2S_CUDA_CHECK(cudaGetLastError());
  m->mp_valid = true;
  return B2S_OK;
}

// (re)build the per-match block summed-area tables and max-pool images after the grids changed
static b2s_status build_sat(b2s_matcher *m) {
  b2s_status st = build_mp4(m);
  if (st) return st;
  const size_t sm = sizeof(uint32_t) * (size_t)(m->sbx + 1) * (m->sby + 1);
  m->sat_valid = false;
  if (sm > 200 * 1024 || (m->g.width_step % 4) != 0 || (long long)m->sbx * m->sby >= 65535) return B2S_OK;  // no skipping
  if (sm > 16 * 1024) B2S_CUDA_CHECK(raise_dyn_smem(k_grid_sat, sm));
  k_grid_sat<<<m->batch, 256, sm, m->stream>>>(m->d_grids, m->grid_pitch, m->g.width_step, m->g.height, m->sbx, m->sby, m->d_sat);
  B2S_CUDA_CHECK(cudaGetLastError());
  m->sat_valid = true;
  return B2S_OK;
}

}  // namespace b2s

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int b2s_abi_version(void) { return B2S_ABI_VERSION; }
const char *b2s_last_error(void) { return b2s::last_error_ref().c_str(); }
int b2s_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

void b2s_matcher_destroy(b2s_matcher *m);
static b2s_status matcher_create_impl(const b2s_matcher_params *params, const b2s_laser *laser, int device, int max_batch,
                                      int max_base_scans, void *cuda_stream, b2s_matcher *m, const b2s_grid_info &g) {
  b2s_status st;
  m->p = *params; m->l = *laser; m->g = g; m->device = device;
  m->max_batch = max_batch; m->max_base = max_base_scans; m->n = laser->n_readings;
  cudaDeviceProp prop;
  B2S_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  m->num_sms = prop.multiProcessorCount;
  m->smem_optin = (int)prop.sharedMemPerBlockOptin;
  if (cuda_stream) {
    m->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  } else {
    B2S_CUDA_CHECK(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    m->own_stream = true;
  }
  for (auto &e : m->ev) B2S_CUDA_CHECK(cudaEventCreate(&e));
  // smear kernel on the host with glibc, exactly CorrelationGrid::CalculateKernel (Mapper.h:1032-1087)
  {
    int ks = g.kernel_size, half = ks / 2;
    std::vector<uint8_t> K((size_t)ks * ks);
    double resolution = 1.0 / (1.0 / params->resolution);
    for (int i = -half; i <= half; i++)
      for (int j = -half; j <= half; j++) {
        double d = hypot(i * resolution, j * resolution);
        double z = exp(-0.5 * pow(d / params->smear_deviation, 2));
        uint32_t kv = cast_u32(kround(z * GRID_OCCUPIED));
        K[(i + half) + ks * (j + half)] = (uint8_t)kv;
        if ((i != 0 || j != 0) && kv >= (uint32_t)GRID_OCCUPIED) m->smear_degenerate = true;
      }
    if ((st = dev_alloc(&m->d_kernel, K.size()))) return st;
    B2S_CUDA_CHECK(cudaMemcpy(m->d_kernel, K.data(), K.size(), cudaMemcpyHostToDevice));
  }
  const size_t B = (size_t)max_batch, N = (size_t)std::max(m->n, 1);
  m->grid_pitch = (((size_t)g.data_size + 16) + 127) & ~(size_t)127;
  const int pstep = (g.search_side + 7) & ~7;
  if ((st = dev_alloc(&m->d_ranges, B * N))) return st;
  if ((st = dev_alloc(&m->d_poses, B * 3))) return st;
  if ((st = dev_alloc(&m->d_sensor, B * 3))) return st;
  if ((st = dev_alloc(&m->d_pts, B * N * 2))) return st;
  if ((st = dev_alloc(&m->d_local, B * N * 2))) return st;
  if ((st = dev_alloc(&m->d_grids, B * m->grid_pitch))) return st;
  if ((st = dev_alloc(&m->d_grid_off, B * 2))) return st;
  if ((st = dev_alloc(&m->d_flags, B))) return st;
  if ((st = dev_alloc(&m->d_probs, B * (size_t)pstep * g.search_side))) return st;
  if ((st = dev_alloc(&m->d_centers, B * 3))) return st;
  if ((st = dev_alloc(&m->d_results, B))) return st;
  if ((st = dev_alloc(&m->d_work, 1))) return st;
  m->sbx = (g.width_step + 3) / 4;
  m->sby = (g.height + 3) / 4;
  if ((st = dev_alloc(&m->d_sat, B * (size_t)((((m->sbx + 1) * (m->sby + 1)) + 7) & ~7)))) return st;  // per-match stride padded to 16 bytes
  if ((st = dev_alloc(&m->d_stats, 2))) return st;
  if ((st = dev_alloc(&m->d_part_best, B))) return st;
  if ((st = dev_alloc(&m->d_glob_best, B))) return st;
  if ((st = dev_alloc(&m->d_tie, B * 5))) return st;
  if ((st = dev_alloc(&m->d_status, B))) return st;
  B2S_CUDA_CHECK(cudaMallocHost(reinterpret_cast<void **>(&m->h_results), B * sizeof(b2s_match_result)));
  B2S_CUDA_CHECK(cudaMallocHost(reinterpret_cast<void **>(&m->h_stats), 2 * sizeof(unsigned long long)));
  m->h_stats[0] = m->h_stats[1] = 0;
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_grids, 0, B * m->grid_pitch, m->stream));
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_results, 0, B * sizeof(b2s_match_result), m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  return B2S_OK;
}

b2s_status b2s_matcher_create(const b2s_matcher_params *params, const b2s_laser *laser, int device, int max_batch,
                              int max_base_scans, void *cuda_stream, b2s_matcher **out) {
  if (!params || !laser || !out || max_batch <= 0 || laser->n_readings < 0 || max_base_scans < 0)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_matcher_create: null/negative argument");
  *out = nullptr;
  b2s_grid_info g;
  b2s_status st = layout_from_params(params, &g);
  if (st) return st;
  if (b2s_device_count() <= device) B2S_FAIL(B2S_ERR_NO_DEVICE, "no usable CUDA device (the product path has no CPU fallback)");
  B2S_CUDA_CHECK(cudaSetDevice(device));
  keep_pool_memory(device);
  b2s_matcher *m = new (std::nothrow) b2s_matcher();
  if (!m) B2S_FAIL(B2S_ERR_CUDA, "out of host memory");
  st = matcher_create_impl(params, laser, device, max_batch, max_base_scans, cuda_stream, m, g);
  if (st) {  // release whatever was allocated before the failure
    const std::string why = b2s::last_error_ref();
    b2s_matcher_destroy(m);
    b2s::set_last_error(why);
    return st;
  }
  *out = m;
  return B2S_OK;
}

void b2s_matcher_destroy(b2s_matcher *m) {
  if (!m) return;
  cudaSetDevice(m->device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  void *ptrs[] = {m->d_kernel, m->d_ranges, m->d_poses, m->d_sensor, m->d_pts, m->d_local, m->d_grids,
                  m->d_grid_off, m->d_base_ranges, m->d_base_poses, m->d_base_pts, m->d_pool, m->d_base_src, m->d_lut, m->d_lists, m->d_counts, m->d_starts, m->d_sat, m->d_stats, m->d_mp4, m->d_keep, m->d_nkeep, m->d_part_best, m->d_glob_best, m->d_tie, m->d_status, m->d_sums, m->d_bases,
                  m->d_flags, m->d_probs, m->d_centers, m->d_results, m->d_work};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  if (m->h_results) cudaFreeHost(m->h_results);
  if (m->h_stats) cudaFreeHost(m->h_stats);
  for (auto &e : m->ev)
    if (e) cudaEventDestroy(e);
  for (auto &e : m->ev_split)
    if (e) cudaEventDestroy(e);
  if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
  delete m;
}

b2s_status b2s_matcher_grid_info(const b2s_matcher *m, b2s_grid_info *out) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  *out = m->g;
  return B2S_OK;
}

b2s_status b2s_matcher_set_kernel(b2s_matcher *m, int which) {
  if (!m || which < 0 || which > 3) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad kernel selector");
  m->force_kernel = which;
  return B2S_OK;
}

b2s_status b2s_matcher_sync(b2s_matcher *m) {
  if (!m) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  return B2S_OK;
}

b2s_status b2s_matcher_set_scans(b2s_matcher *m, int batch, const double *ranges, const double *poses) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !ranges || !poses) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (batch <= 0 || batch > m->max_batch) B2S_FAIL(B2S_ERR_TOO_LARGE, "batch exceeds the handle's max_batch");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  m->batch = batch;
  const size_t n = (size_t)m->n;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_ranges, ranges, sizeof(double) * batch * n, cudaMemcpyHostToDevice, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_poses, poses, sizeof(double) * batch * 3, cudaMemcpyHostToDevice, m->stream));
  k_scan_points<<<batch, 256, 0, m->stream>>>(m->d_ranges, m->d_poses, m->l, m->d_sensor, m->d_pts, m->d_local, nullptr);
  B2S_CUDA_CHECK(cudaGetLastError());
  m->scans_set = true;
  m->grids_set = false;
  m->have_sweep = false;
  return B2S_OK;
}

// base_ranges != NULL: the base scans' readings come from the host; otherwise pool_rows ([batch * n_base], host) names
// rows of the handle's device-resident scan pool
static b2s_status add_scans_impl(b2s_matcher *m, int n_base, const double *base_ranges, const int32_t *pool_rows,
                                 const double *base_poses) {
  B2S_NVTX("K1 add_scans (rasterise + smear)");
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || n_base < 0 || (n_base > 0 && ((!base_ranges && !pool_rows) || !base_poses))) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->scans_set) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_set_scans must precede b2s_matcher_add_scans");
  if (n_base > m->max_base) B2S_FAIL(B2S_ERR_TOO_LARGE, "n_base exceeds the handle's max_base_scans");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  const size_t n = (size_t)m->n;
  const double resolution = 1.0 / (1.0 / m->p.resolution);
  const double scale = 1.0 / m->p.resolution;  // CorrelationGrid ctor SetScale (Mapper.h:1020)
  k_grid_offsets<<<ceil_div(B, 128), 128, 0, m->stream>>>(m->d_sensor, m->d_grid_off, B, m->g.roi_w, m->g.roi_h,
                                                          resolution);
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_grids, 0, (size_t)B * m->grid_pitch, m->stream));  // Grid::Clear
  m->n_base = n_base;
  if (n_base > 0 && n > 0) {
    const size_t need = (size_t)B * n_base;
    if (need > m->base_cap) {
      for (double **p : {&m->d_base_ranges, &m->d_base_poses, &m->d_base_pts})
        if (*p) { B2S_CUDA_CHECK(cudaFree(*p)); *p = nullptr; }
      b2s_status st;
      if ((st = dev_alloc(&m->d_base_ranges, need * n))) return st;
      if ((st = dev_alloc(&m->d_base_poses, need * 3))) return st;
      if ((st = dev_alloc(&m->d_base_pts, need * n * 2))) return st;
      m->base_cap = need;
    }
    B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_base_poses, base_poses, sizeof(double) * need * 3, cudaMemcpyHostToDevice, m->stream));
    if (base_ranges) {
      B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_base_ranges, base_ranges, sizeof(double) * need * n, cudaMemcpyHostToDevice, m->stream));
      k_scan_points<<<(unsigned)need, 256, 0, m->stream>>>(m->d_base_ranges, m->d_base_poses, m->l, nullptr, m->d_base_pts, nullptr, nullptr);
    } else {
      for (size_t i = 0; i < need; i++)
        if (pool_rows[i] < 0 || (size_t)pool_rows[i] >= m->pool_count) B2S_FAIL(B2S_ERR_OUT_OF_RANGE, "scan pool row out of range");
      if (need > m->base_src_cap) {
        if (m->d_base_src) { B2S_CUDA_CHECK(cudaFree(m->d_base_src)); m->d_base_src = nullptr; }
        B2S_CUDA_CHECK(cudaMalloc(reinterpret_cast<void **>(&m->d_base_src), sizeof(int32_t) * need));
        m->base_src_cap = need;
      }
      B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_base_src, pool_rows, sizeof(int32_t) * need, cudaMemcpyHostToDevice, m->stream));
      k_scan_points<<<(unsigned)need, 256, 0, m->stream>>>(m->d_pool, m->d_base_poses, m->l, nullptr, m->d_base_pts, nullptr, m->d_base_src);
    }
    if (!m->smear_degenerate) {
      size_t smem = n * (2 * sizeof(double) + 2 * sizeof(int) + 1) + sizeof(int) + 16;
      if (smem > 16 * 1024)
        B2S_CUDA_CHECK(raise_dyn_smem(k_add_scan, smem));
      k_add_scan<<<(unsigned)need, 256, smem, m->stream>>>(m->d_base_pts, m->d_sensor, m->d_grid_off, m->d_grids,
                                                           m->grid_pitch, m->d_kernel, m->g, scale, (int)n, n_base);
    } else {
      uint8_t *scratch = nullptr;
      B2S_CUDA_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&scratch), (size_t)B * n, m->stream));
      k_add_scans_seq<<<ceil_div(B, 32), 32, 0, m->stream>>>(m->d_base_pts, m->d_sensor, m->d_grid_off, m->d_grids,
                                                             m->grid_pitch, m->d_kernel, m->g, scale, (int)n, n_base,
                                                             B, scratch);
      B2S_CUDA_CHECK(cudaFreeAsync(scratch, m->stream));
    }
    B2S_CUDA_CHECK(cudaGetLastError());
  }
  m->grids_set = true;
  m->grid_high_bytes = false;
  m->have_sweep = false;
  return build_sat(m);
}

b2s_status b2s_matcher_add_scans(b2s_matcher *m, int n_base, const double *base_ranges, const double *base_poses) {
  if (n_base > 0 && !base_ranges) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  return add_scans_impl(m, n_base, base_ranges, nullptr, base_poses);
}

// ---- scan pool: readings that serve as base scans of many matches (a mapper's running window, near chains, loop
// candidates) are uploaded once and referenced by row afterwards
b2s_status b2s_matcher_pool_append(b2s_matcher *m, const double *ranges, int32_t *out_row) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !ranges) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const size_t n = (size_t)std::max(m->l.n_readings, 1);
  if (m->pool_count == m->pool_cap) {
    const size_t cap = std::max<size_t>(256, m->pool_cap * 2);
    double *fresh = nullptr;
    b2s_status st = dev_alloc(&fresh, cap * n);
    if (st) return st;
    if (m->pool_count)
      B2S_CUDA_CHECK(cudaMemcpyAsync(fresh, m->d_pool, sizeof(double) * m->pool_count * n, cudaMemcpyDeviceToDevice, m->stream));
    B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
    if (m->d_pool) B2S_CUDA_CHECK(cudaFree(m->d_pool));
    m->d_pool = fresh;
    m->pool_cap = cap;
  }
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_pool + m->pool_count * n, ranges, sizeof(double) * n, cudaMemcpyHostToDevice, m->stream));
  if (out_row) *out_row = (int32_t)m->pool_count;
  m->pool_count++;
  return B2S_OK;
}

int32_t b2s_matcher_pool_count(const b2s_matcher *m) { return m ? (int32_t)m->pool_count : 0; }

b2s_status b2s_matcher_add_scans_pool(b2s_matcher *m, int n_base, const int32_t *pool_rows, const double *base_poses) {
  if (n_base > 0 && !pool_rows) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  return add_scans_impl(m, n_base, nullptr, pool_rows, base_poses);
}

b2s_status b2s_matcher_set_grids(b2s_matcher *m, const uint8_t *grids, const double *offsets) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !grids || !offsets) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->scans_set) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_set_scans must precede b2s_matcher_set_grids");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  m->grid_high_bytes = false;  // the reference's grids hold 0..100; anything above 127 needs the generic kernel
  for (size_t i = 0, e = (size_t)B * m->g.data_size; i < e; i++)
    if (grids[i] > 127) { m->grid_high_bytes = true; break; }
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_grids, 0, (size_t)B * m->grid_pitch, m->stream));
  B2S_CUDA_CHECK(cudaMemcpy2DAsync(m->d_grids, m->grid_pitch, grids, (size_t)m->g.data_size, (size_t)m->g.data_size, B,
                                   cudaMemcpyHostToDevice, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_grid_off, offsets, sizeof(double) * 2 * B, cudaMemcpyHostToDevice, m->stream));
  m->grids_set = true;
  m->have_sweep = false;
  return build_sat(m);
}

b2s_status b2s_matcher_get_grid(b2s_matcher *m, int b, uint8_t *out_bytes, double out_offset[2]) {
  if (!m || b < 0 || b >= m->batch || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "no grid for this match");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  if (out_bytes)
    B2S_CUDA_CHECK(cudaMemcpyAsync(out_bytes, m->d_grids + (size_t)b * m->grid_pitch, (size_t)m->g.data_size,
                                   cudaMemcpyDeviceToHost, m->stream));
  if (out_offset)
    B2S_CUDA_CHECK(cudaMemcpyAsync(out_offset, m->d_grid_off + 2 * b, 2 * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  return B2S_OK;
}

b2s_status b2s_matcher_get_point_readings(b2s_matcher *m, int b, double *out_xy) {
  if (!m || !out_xy || b < 0 || b >= m->batch || !m->scans_set) B2S_FAIL(B2S_ERR_BAD_STATE, "no scan for this match");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  B2S_CUDA_CHECK(cudaMemcpyAsync(out_xy, m->d_pts + (size_t)b * m->n * 2, sizeof(double) * 2 * m->n,
                                 cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  return B2S_OK;
}

b2s_status b2s_matcher_compute_offsets(b2s_matcher *m, int b, double angle_center, double angle_offset,
                                       double angle_res, int32_t *out, int32_t *out_n_angles) {
  if (!m || !out || b < 0 || b >= m->batch) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad argument");
  if (!m->scans_set || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "scans and grids must be set first");
  if (angle_res == 0.0) B2S_FAIL(B2S_ERR_BAD_PARAMS, "angle resolution must be non-zero");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int na = n_steps(angle_offset, angle_res);
  const size_t n = (size_t)m->n;
  int32_t *tmp = nullptr;
  B2S_CUDA_CHECK(cudaMalloc(reinterpret_cast<void **>(&tmp), sizeof(int32_t) * std::max<size_t>(na * n, 1)));
  // one-match launch on the slices of match b
  k_offsets<<<na, 256, 0, m->stream>>>(m->d_ranges + (size_t)b * n, m->d_local + (size_t)b * n * 2,
                                       m->d_grid_off + 2 * b, nullptr, 0, angle_center, 1, angle_offset, angle_res, na,
                                       (int)n, m->g.width_step, 1.0 / m->p.resolution, tmp, 0);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, tmp, sizeof(int32_t) * na * n, cudaMemcpyDeviceToHost, m->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
  cudaFree(tmp);
  B2S_CUDA_CHECK(e);
  if (out_n_angles) *out_n_angles = na;
  return B2S_OK;
}

// Enqueue a CorrelateScan (centers H2D, lookup lists, sweep, reduce, results D2H into the handle's pinned buffer) on the
// handle's stream and return without waiting: a caller with two handles overlaps one batch's uploads and small kernels
// with the other batch's sweep.  b2s_matcher_correlate_scan_end waits and hands the results out.
b2s_status b2s_matcher_correlate_scan_begin(b2s_matcher *m, const double *centers, const b2s_search *search,
                                            const b2s_match_result *cov_in) {
  if (!m || !centers || !search) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->scans_set || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "scans and grids must be set first");
  if (search->fine && !cov_in) B2S_FAIL(B2S_ERR_BAD_PARAMS, "the fine stage needs the incoming covariances (rCovariance is IN/OUT)");
  if (m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_correlate_scan_begin while an earlier one awaits its _end");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_centers, centers, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, m->stream));
  if (search->fine) {  // rCovariance is IN/OUT for the fine stage (Mapper.cpp:648)
    for (int b = 0; b < B; b++) m->h_results[b] = cov_in[b];
    B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_results, m->h_results, sizeof(b2s_match_result) * B, cudaMemcpyHostToDevice, m->stream));
  }
  b2s_status st = run_correlate(m, search, true);
  if (st) return st;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_stats, m->d_stats, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, m->stream));
  m->pending = true;
  m->pending_batch = B;
  return B2S_OK;
}

b2s_status b2s_matcher_correlate_scan_end(b2s_matcher *m, b2s_match_result *results) {
  if (!m || !results) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_correlate_scan_end without a pending b2s_matcher_correlate_scan_begin");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->pending_batch;  // the batch the _begin enqueued
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  m->pending = false;
  std::memcpy(results, m->h_results, sizeof(b2s_match_result) * B);
  if (m->last_path == 2 && m->last.na > 0 && m->n > 0) m->last_empty_frac = (double)*m->h_stats / ((double)B * m->last.na * m->n);
  else m->last_empty_frac = 0.0;
  const double pairs = (double)B * m->last.na;
  if (m->last_pruned) { m->last_prune[0] = pairs > 0 ? (double)m->h_stats[1] / pairs : 1.0; m->last_prune[1] = (double)m->h_stats[1]; }
  else { m->last_prune[0] = 1.0; m->last_prune[1] = pairs; }
  for (int i = 1; i < 3; i++) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, m->ev[i - 1], m->ev[i]) == cudaSuccess) m->last_ms[i - 1] = ms;
  }
  {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, m->ev[2], m->ev[3]) == cudaSuccess) m->last_ms[2] = ms;
  }
  return B2S_OK;
}

b2s_status b2s_matcher_correlate_scan(b2s_matcher *m, const double *centers, const b2s_search *search,
                                      b2s_match_result *results) {
  if (!results) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  b2s_status st = b2s_matcher_correlate_scan_begin(m, centers, search, results);
  if (st) return st;
  return b2s_matcher_correlate_scan_end(m, results);
}

b2s_status b2s_matcher_match_scan(b2s_matcher *m, int do_penalize, int do_refine, b2s_match_result *results) {
  B2S_NVTX("K1 MatchScan (coarse + fine)");
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !results) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->scans_set || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "scans and grids must be set first");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  if (m->n == 0) {  // Mapper.cpp:199-209: no readings -> pose passthrough, maximum covariance
    std::vector<double> sp((size_t)3 * B);
    B2S_CUDA_CHECK(cudaMemcpyAsync(sp.data(), m->d_sensor, sizeof(double) * 3 * B, cudaMemcpyDeviceToHost, m->stream));
    B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
    for (int b = 0; b < B; b++) {
      std::memset(&results[b], 0, sizeof(b2s_match_result));
      for (int i = 0; i < 3; i++) results[b].pose[i] = sp[3 * b + i];
      results[b].cov[0] = MAX_VARIANCE; results[b].cov[4] = MAX_VARIANCE;
      results[b].cov[8] = 4 * (m->p.coarse_angle_resolution * m->p.coarse_angle_resolution);
    }
    return B2S_OK;
  }
  const double resolution = 1.0 / (1.0 / m->p.resolution);
  b2s_search coarse;
  coarse.offset_x = 0.5 * ((double)m->g.search_side - 1) * resolution;  // Mapper.cpp:228-230
  coarse.offset_y = coarse.offset_x;
  coarse.res_x = 2 * resolution;  // Mapper.cpp:233-234
  coarse.res_y = 2 * resolution;
  coarse.angle_offset = m->p.coarse_search_angle_offset;
  coarse.angle_res = m->p.coarse_angle_resolution;
  coarse.do_penalize = do_penalize;
  coarse.fine = 0;
  // search centre = scan (sensor) pose (Mapper.cpp:237)
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_centers, m->d_sensor, sizeof(double) * 3 * B, cudaMemcpyDeviceToDevice, m->stream));
  b2s_status st = run_correlate(m, &coarse, true);
  if (st) return st;
  if (m->p.use_response_expansion) {  // Mapper.cpp:242-272 — applied to the matches whose response is ~0
    B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
    B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
    std::vector<b2s_match_result> keep(m->h_results, m->h_results + B);
    std::vector<char> pending(B, 0);
    bool any = false;
    for (int b = 0; b < B; b++)
      if (keep[b].status == B2S_OK && double_equal(keep[b].response, 0.0)) { pending[b] = 1; any = true; }
    double new_off = m->p.coarse_search_angle_offset;
    for (int it = 0; it < 3 && any; it++) {
      new_off += 20 * 0.01745329251994329577;  // math::DegreesToRadians(20)
      b2s_search ex = coarse;
      ex.angle_offset = new_off;
      B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_centers, m->d_sensor, sizeof(double) * 3 * B, cudaMemcpyDeviceToDevice, m->stream));
      st = run_correlate(m, &ex, true);
      if (st) return st;
      B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
      B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
      any = false;
      for (int b = 0; b < B; b++) {
        if (!pending[b]) continue;
        keep[b] = m->h_results[b];
        if (keep[b].status != B2S_OK || !double_equal(keep[b].response, 0.0)) pending[b] = 0;
        else any = true;
      }
    }
    for (int b = 0; b < B; b++) m->h_results[b] = keep[b];
    B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_results, m->h_results, sizeof(b2s_match_result) * B, cudaMemcpyHostToDevice, m->stream));
  }
  if (do_refine) {  // Mapper.cpp:274-282
    b2s_search fine;
    fine.offset_x = coarse.res_x * 0.5;
    fine.offset_y = coarse.res_y * 0.5;
    fine.res_x = resolution;
    fine.res_y = resolution;
    fine.angle_offset = 0.5 * m->p.coarse_angle_resolution;
    fine.angle_res = m->p.fine_search_angle_offset;
    fine.do_penalize = do_penalize;
    fine.fine = 1;
    k_results_to_centers<<<ceil_div(B, 128), 128, 0, m->stream>>>(m->d_results, m->d_centers, B);
    st = run_correlate(m, &fine, true);
    if (st) return st;
  }
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  std::memcpy(results, m->h_results, sizeof(b2s_match_result) * B);
  return B2S_OK;
}

b2s_status b2s_matcher_match_scan_host(b2s_matcher *m, int batch, const double *ranges, const double *poses,
                                       int n_base, const double *base_ranges, const double *base_poses,
                                       int do_penalize, int do_refine, b2s_match_result *results) {
  b2s_status st = b2s_matcher_set_scans(m, batch, ranges, poses);
  if (st) return st;
  st = b2s_matcher_add_scans(m, n_base, base_ranges, base_poses);
  if (st) return st;
  return b2s_matcher_match_scan(m, do_penalize, do_refine, results);
}

/* ---- a CorrelateScan whose ANGLES are split over several GPUs (SURVEY.md §8(e)(ii)) ----
 * Every rank holds the same scans + grids and sweeps angle indices [k_first, k_first + k_count) of the search.
 * Between the three phases the caller all-reduces small host arrays (torch.distributed / NCCL):
 *   begin : out best[B] (MAX), per-cell maxima plane probs[B][probs_len] (MAX), status[B] (MAX)
 *   ties  : in global best; out tie sums {x, y, cos, sin, count}[B][5] (SUM)
 *   finish: in global best / tie sums / plane; out the same results as b2s_matcher_correlate_scan (coarse stage). */
b2s_status b2s_matcher_correlate_split_begin(b2s_matcher *m, const double *centers, const b2s_search *search, int k_first,
                                             int k_count, double *best, double *probs, int32_t *status) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !centers || !search || !best || !probs || !status || k_count < 0) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (search->fine) B2S_FAIL(B2S_ERR_BAD_PARAMS, "only the coarse stage (doingFineMatch = false) can be split");
  if (!m->scans_set || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "scans and grids must be set first");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  const size_t plen = (size_t)((m->g.search_side + 7) & ~7) * m->g.search_side;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_centers, centers, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, m->stream));
  b2s_status st = run_correlate(m, search, true, k_first, k_count, 1);
  if (st) return st;
  B2S_CUDA_CHECK(cudaMemcpyAsync(best, m->d_part_best, sizeof(double) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(probs, m->d_probs, sizeof(double) * plen * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  for (int b = 0; b < B; b++) status[b] = m->h_results[b].status;
  return B2S_OK;
}

static ReduceArgs reduce_args(b2s_matcher *m, const b2s_search &s, int nx, int ny, int na, int k_first, int mode) {
  ReduceArgs A;
  A.sums = m->d_sums; A.centers = m->d_centers; A.flags = m->d_flags;
  A.p = m->p; A.s = s; A.g = m->g; A.scale = 1.0 / m->p.resolution;
  A.n = m->n; A.nx = nx; A.ny = ny; A.na = na;
  A.probs_all = m->d_probs; A.results = m->d_results;
  A.k_first = k_first; A.mode = mode;
  A.part_best = m->d_part_best; A.glob_best = m->d_glob_best; A.tie_out = m->d_tie; A.tie_in = m->d_tie;
  A.keep = nullptr; A.nkeep = nullptr;
  return A;
}

static b2s_status split_phase(b2s_matcher *m, int mode) {
  k_reduce<<<m->batch, RED_THREADS, 0, m->stream>>>(reduce_args(m, m->last_search, m->last.nx, m->last.ny, m->last.na, m->last_k_first, mode));
  B2S_CUDA_CHECK(cudaGetLastError());
  return B2S_OK;
}

b2s_status b2s_matcher_correlate_split_ties(b2s_matcher *m, const double *global_best, double *tie_sums) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !global_best || !tie_sums) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->have_sweep) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_correlate_split_begin must come first");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_glob_best, global_best, sizeof(double) * B, cudaMemcpyHostToDevice, m->stream));
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_tie, 0, sizeof(double) * 5 * B, m->stream));
  b2s_status st = split_phase(m, 2);
  if (st) return st;
  B2S_CUDA_CHECK(cudaMemcpyAsync(tie_sums, m->d_tie, sizeof(double) * 5 * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  return B2S_OK;
}

b2s_status b2s_matcher_correlate_split_finish(b2s_matcher *m, const double *global_best, const double *tie_sums,
                                              const double *probs, b2s_match_result *results) {
  if (m && m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end: the handle cannot change state in between");
  if (!m || !global_best || !tie_sums || !probs || !results) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (!m->have_sweep) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_matcher_correlate_split_begin must come first");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int B = m->batch;
  const size_t plen = (size_t)((m->g.search_side + 7) & ~7) * m->g.search_side;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_glob_best, global_best, sizeof(double) * B, cudaMemcpyHostToDevice, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_tie, tie_sums, sizeof(double) * 5 * B, cudaMemcpyHostToDevice, m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_probs, probs, sizeof(double) * plen * B, cudaMemcpyHostToDevice, m->stream));
  b2s_status st = split_phase(m, 3);
  if (st) return st;
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  std::memcpy(results, m->h_results, sizeof(b2s_match_result) * B);
  return B2S_OK;
}

/* The same angle-split CorrelateScan with the collectives INSIDE the library (SURVEY.md §8(e)(ii); north_star: "a single
 * NCCL all-reduce on the per-scan best-score"): every rank holds the same scans + grids and calls this with its rank; the
 * angle steps are partitioned by rank, and between the three phases the library all-reduces device buffers on the
 * handle's stream through the caller's NCCL communicator — best response (MAX, B doubles), per-cell maxima plane (MAX,
 * B x probs_len doubles), status (MAX), tie sums (SUM, 5B doubles).  No host staging; results equal the single-GPU
 * b2s_matcher_correlate_scan on every rank. */
b2s_status b2s_matcher_correlate_scan_split(b2s_matcher *m, void *nccl_comm, int rank, int world, const double *centers,
                                            const b2s_search *search, b2s_match_result *results) {
  if (!m || !nccl_comm || !centers || !search || !results || world < 1 || rank < 0 || rank >= world)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "null / bad argument");
  if (m->pending) B2S_FAIL(B2S_ERR_BAD_STATE, "a b2s_matcher_correlate_scan_begin awaits its _end");
  if (search->fine) B2S_FAIL(B2S_ERR_BAD_PARAMS, "only the coarse stage (doingFineMatch = false) can be split");
  if (!m->scans_set || !m->grids_set) B2S_FAIL(B2S_ERR_BAD_STATE, "scans and grids must be set first");
  const NcclApi &nc = nccl_api();
  if (!nc.ok) B2S_FAIL(B2S_ERR_BAD_STATE, "libnccl.so.2 could not be loaded (dlopen)");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  for (auto &e : m->ev_split)
    if (!e) B2S_CUDA_CHECK(cudaEventCreate(&e));
  const int B = m->batch;
  const size_t plen = (size_t)((m->g.search_side + 7) & ~7) * m->g.search_side;
  const int na_full = n_steps(search->angle_offset, search->angle_res);
  const int base = na_full / world, extra = na_full % world;  // contiguous, balanced (parallel.shard_bounds)
  const int k_first = rank * base + std::min(rank, extra), k_count = base + (rank < extra ? 1 : 0);
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->d_centers, centers, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, m->stream));
  b2s_status st = run_correlate(m, search, true, k_first, k_count, 1);
  if (st) return st;
  k_status_pack<<<ceil_div(B, 128), 128, 0, m->stream>>>(m->d_results, m->d_status, B);
  auto check_nccl = [&](int rc, const char *what) -> b2s_status {
    if (rc == 0) return B2S_OK;
    set_last_error(std::string(what) + " failed: " + (nc.error_string ? nc.error_string(rc) : "NCCL error"));
    return B2S_ERR_CUDA;
  };
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[0], m->stream));
  if ((st = check_nccl(nc.all_reduce(m->d_part_best, m->d_glob_best, (size_t)B, NCCL_FLOAT64, NCCL_MAX, nccl_comm, m->stream), "ncclAllReduce(best)"))) return st;
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[1], m->stream));
  if ((st = check_nccl(nc.all_reduce(m->d_probs, m->d_probs, plen * B, NCCL_FLOAT64, NCCL_MAX, nccl_comm, m->stream), "ncclAllReduce(plane)"))) return st;
  if ((st = check_nccl(nc.all_reduce(m->d_status, m->d_status, (size_t)B, NCCL_INT32, NCCL_MAX, nccl_comm, m->stream), "ncclAllReduce(status)"))) return st;
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[2], m->stream));
  B2S_CUDA_CHECK(cudaMemsetAsync(m->d_tie, 0, sizeof(double) * 5 * B, m->stream));
  if ((st = split_phase(m, 2))) return st;
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[3], m->stream));
  if ((st = check_nccl(nc.all_reduce(m->d_tie, m->d_tie, (size_t)5 * B, NCCL_FLOAT64, NCCL_SUM, nccl_comm, m->stream), "ncclAllReduce(ties)"))) return st;
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[4], m->stream));
  if ((st = split_phase(m, 3))) return st;
  k_status_apply<<<ceil_div(B, 128), 128, 0, m->stream>>>(m->d_results, m->d_status, B);
  B2S_CUDA_CHECK(cudaGetLastError());
  B2S_CUDA_CHECK(cudaEventRecord(m->ev_split[5], m->stream));
  B2S_CUDA_CHECK(cudaMemcpyAsync(m->h_results, m->d_results, sizeof(b2s_match_result) * B, cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  std::memcpy(results, m->h_results, sizeof(b2s_match_result) * B);
  float ms = 0;
  if (cudaEventElapsedTime(&ms, m->ev_split[0], m->ev_split[1]) == cudaSuccess) m->last_split_ms[0] = ms;  // best
  if (cudaEventElapsedTime(&ms, m->ev_split[1], m->ev_split[2]) == cudaSuccess) m->last_split_ms[1] = ms;  // plane + status
  if (cudaEventElapsedTime(&ms, m->ev_split[3], m->ev_split[4]) == cudaSuccess) m->last_split_ms[2] = ms;  // tie sums
  if (cudaEventElapsedTime(&ms, m->ev_split[0], m->ev_split[5]) == cudaSuccess) m->last_split_ms[3] = ms;  // all phases after the sweep
  return B2S_OK;
}

/* ms of the last b2s_matcher_correlate_scan_split: all-reduce(best), all-reduce(plane + status), all-reduce(tie sums),
 * everything between the end of the local sweep and the final results */
b2s_status b2s_matcher_last_split_timing(b2s_matcher *m, double out[4]) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  for (int i = 0; i < 4; i++) out[i] = m->last_split_ms[i];
  return B2S_OK;
}

b2s_status b2s_matcher_get_response_sums(b2s_matcher *m, int b, int32_t *out, int32_t dims[3]) {
  if (!m || !out || b < 0 || b >= m->batch) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad argument");
  if (!m->have_sweep) B2S_FAIL(B2S_ERR_BAD_STATE, "no sweep has been run");
  B2S_CUDA_CHECK(cudaSetDevice(m->device));
  const int nx = m->last.nx, ny = m->last.ny, na = m->last.na;
  if (!m->sums_dense) {  // a pruned sweep left the other angles unswept: sweep every angle once from the held lists
    b2s_status st = launch_window(m, m->batch, m->n, na, nx, ny, false);
    if (st) return st;
    B2S_CUDA_CHECK(cudaGetLastError());
    m->sums_dense = true;
  }
  std::vector<int32_t> tmp((size_t)nx * ny * na);
  B2S_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), m->d_sums + (size_t)b * nx * ny * na, sizeof(int32_t) * tmp.size(),
                                 cudaMemcpyDeviceToHost, m->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(m->stream));
  // device layout [k][iy][ix] -> reference loop order [iy][ix][k]
  for (int k = 0; k < na; k++)
    for (int c = 0; c < nx * ny; c++) out[(size_t)c * na + k] = tmp[(size_t)k * nx * ny + c];
  if (dims) { dims[0] = ny; dims[1] = nx; dims[2] = na; }
  return B2S_OK;
}

b2s_status b2s_matcher_last_stats(b2s_matcher *m, double out[4]) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  out[0] = m->last_empty_frac;
  out[1] = (double)m->last_path;
  out[2] = (double)m->last.na * m->last.nx * m->last.ny;
  out[3] = (double)m->n;
  return B2S_OK;
}

b2s_status b2s_matcher_last_prune_stats(b2s_matcher *m, double out[2]) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  out[0] = m->last_prune[0];
  out[1] = m->last_prune[1];
  return B2S_OK;
}

b2s_status b2s_matcher_last_timing(b2s_matcher *m, double out[4]) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (m->have_sweep && !m->pending && cudaSetDevice(m->device) == cudaSuccess && cudaStreamSynchronize(m->stream) == cudaSuccess) {
    // the events of the LAST sweep (whichever entry point ran it: correlate_scan, match_scan's last stage, a split phase)
    for (int i = 0; i < 3; i++) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, m->ev[i], m->ev[i + 1]) == cudaSuccess) m->last_ms[i] = ms;
    }
    cudaGetLastError();
  }
  out[0] = m->last_ms[0]; out[1] = m->last_ms[1]; out[2] = m->last_ms[2]; out[3] = (double)m->last_path;
  return B2S_OK;
}

}  // extern "C"

namespace b2s {

// One CorrelateScan over the batch with centres already in d_centers.  Results stay in d_results.
static b2s_status run_correlate(b2s_matcher *m, const b2s_search *s, bool /*centers_on_device*/, int k_first, int na_override,
                                int mode) {
  B2S_NVTX("K1 correlate (lists + sweep + tail)");
  if (s->angle_res == 0.0 || s->res_x == 0.0 || s->res_y == 0.0)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "search resolutions must be non-zero");  // assert at Mapper.cpp:319
  const int B = m->batch, n = m->n;
  const int nx = n_steps(s->offset_x, s->res_x), ny = n_steps(s->offset_y, s->res_y);
  const int na_full = n_steps(s->angle_offset, s->angle_res);
  const int na = na_override >= 0 ? na_override : na_full;  // angles swept by THIS call (a subset when the sweep is split)
  if (k_first < 0 || k_first + na > na_full) B2S_FAIL(B2S_ERR_BAD_PARAMS, "angle subset outside the search");
  if (nx <= 0 || ny <= 0 || na_full <= 0 || (long long)nx * ny * std::max(na, 1) > (1ll << 28))
    B2S_FAIL(B2S_ERR_TOO_LARGE, "search volume too large");
  const double scale = 1.0 / m->p.resolution;
  const int ncell = nx * ny;
  b2s_status st;
  if ((st = ensure_cap(&m->d_sums, &m->sums_cap, (size_t)B * na * ncell))) return st;
  if ((st = ensure_cap(&m->d_bases, &m->bases_cap, (size_t)B * ncell))) return st;

  // ---- which sweep kernel ----
  // The window kernel needs a stride-1 lattice and a band of the grid in shared memory: the whole grid when it fits
  // (nbands = 1), otherwise nbands row bands of band_rows origin rows + (window rows + 1) halo rows each.
  const int copy_bytes = (m->g.data_size + 15) & ~15;
  // candidate stride in grid cells: 1 (search resolution == grid resolution) or 2 (the coarse stage of MatchScan,
  // Mapper.cpp:233-234); anything else goes to the generic kernel
  const double gres = 1.0 / (1.0 / m->p.resolution);
  auto stride_of = [&](double r) { return (r == gres || r == m->p.resolution) ? 1 : ((r == 2 * gres || r == 2 * m->p.resolution) ? 2 : 0); };
  const int stride = (stride_of(s->res_x) == stride_of(s->res_y)) ? stride_of(s->res_x) : 0;
  const int cpt = stride == 2 ? 16 : 32;  // candidates per 32-byte tile row
  const int tiles_x_w = (nx + cpt - 1) / cpt, tiles_y_w = (ny + 31) / 32;
  const int rows_total = tiles_y_w * 32;
  const int halo_rows = std::max(stride, 1) * 31 + 2;  // rows below the first row of a 32-row candidate tile that a lane may touch
  // static shared memory of the sweep kernel (its own + the fused tail's scratch) comes out of the opt-in budget
  static size_t win_static = 0;
  if (!win_static) {
    cudaFuncAttributes fa;
    B2S_CUDA_CHECK(cudaFuncGetAttributes(&fa, k_sweep_window<1, false>));
    win_static = fa.sharedSizeBytes;
  }
  const long long smem_limit = (long long)m->smem_optin - (long long)win_static - 512;
  int band_rows = std::max(m->g.height, 1), nbands = 1, band_bytes = copy_bytes, neg_bands = 0;
  bool bands_ok = true;
  if ((long long)copy_bytes + 2 * WIN_GUARD > smem_limit) {
    const long long rows_fit = (smem_limit - 2 * WIN_GUARD) / m->g.width_step;
    band_rows = (int)((rows_fit - halo_rows) & ~1LL);  // even: band starts stay 16-byte aligned (width_step % 8 == 0)
    if (band_rows < 8) {
      bands_ok = false;
    } else {
      // origins up to (window rows) below the grid still reach it from their upper row tiles: bands of their own
      neg_bands = tiles_y_w > 1 ? (std::max(stride, 1) * (rows_total - 1) + 1 + band_rows - 1) / band_rows : 0;
      nbands = (m->g.height + band_rows - 1) / band_rows + neg_bands;
      band_bytes = (int)((long long)(band_rows + halo_rows) * m->g.width_step);
      if (nbands > WIN_MAX_BANDS) bands_ok = false;
    }
  }
  const size_t win_smem = (size_t)((band_bytes + 15) & ~15) + 2 * WIN_GUARD;
  const bool win_fits = bands_ok && stride != 0 && (m->g.width_step % 8) == 0 && n > 0 &&
                        (size_t)n * OFF_SMEM_PER_BEAM + 64 <= 200 * 1024 && !m->grid_high_bytes;
  bool use_window = win_fits;
  if (m->force_kernel == 1) use_window = false;
  if (m->force_kernel >= 2 && !win_fits)
    B2S_FAIL(B2S_ERR_TOO_LARGE, "window kernel forced but not applicable to this lattice / grid / beam count");
  if (m->force_kernel >= 2) use_window = true;
  const bool need_plain_lut = !use_window || s->fine;  // generic sweep and the angular covariance read the plain table
  if (need_plain_lut && (st = ensure_cap(&m->d_lut, &m->lut_cap, (size_t)B * na * std::max(n, 1)))) return st;

  B2S_CUDA_CHECK(cudaEventRecord(m->ev[0], m->stream));
  k_bases<<<B, 256, 0, m->stream>>>(m->d_centers, m->d_grid_off, *s, m->g, scale, nx, ny, m->d_bases, m->d_flags,
                                    std::max(stride, 1));
  if (need_plain_lut && na > 0)
    k_offsets<<<B * na, 256, 0, m->stream>>>(m->d_ranges, m->d_local, m->d_grid_off, m->d_centers, 3, 0.0, 0,
                                             s->angle_offset, s->angle_res, na, n, m->g.width_step, scale, m->d_lut, k_first);
  const dim3 ggrid((unsigned)ceil_div(ncell, 8), (unsigned)B);
  if (use_window && na > 0) {
    if ((st = ensure_cap(&m->d_lists, &m->lists_cap, (size_t)B * na * (n + LIST_PAD * nbands)))) return st;
    if ((st = ensure_cap(&m->d_counts, &m->counts_cap, (size_t)B * na * 8 * nbands))) return st;
    if ((st = ensure_cap(&m->d_starts, &m->starts_cap, (size_t)B * na * 8 * nbands))) return st;
    bool skip_empty = m->sat_valid && m->force_kernel != 3;
    if ((((size_t)n * OFF_SMEM_PER_BEAM + 15) & ~(size_t)15) + sizeof(uint16_t) * (size_t)((((m->sbx + 1) * (m->sby + 1)) + 7) & ~7) + 64 > 200 * 1024) skip_empty = false;
    const size_t sat_bytes = skip_empty ? sizeof(uint16_t) * (size_t)((((m->sbx + 1) * (m->sby + 1)) + 7) & ~7) : 0;
    const size_t osm = (((size_t)n * OFF_SMEM_PER_BEAM + 15) & ~(size_t)15) + sat_bytes + 64;
    B2S_CUDA_CHECK(cudaMemsetAsync(m->d_stats, 0, 2 * sizeof(unsigned long long), m->stream));
    if (osm > 16 * 1024)  // static + dynamic shared memory together must stay under the 48 KB default: opt in early
      B2S_CUDA_CHECK(raise_dyn_smem(k_offsets_sorted, osm));
    k_offsets_sorted<<<B * ((na + OFF_CHUNK - 1) / OFF_CHUNK), 256, osm, m->stream>>>(
        m->d_ranges, m->d_local, m->d_grid_off, m->d_centers, m->d_bases, m->d_flags, s->angle_offset, s->angle_res, na, n,
        ncell, m->g.width_step, m->g.data_size, scale, rows_total, tiles_x_w * 32, m->d_lists, m->d_counts,
        skip_empty ? m->d_sat : nullptr, m->sbx, m->sby, m->g.height, nx, ny, m->d_stats, band_rows, nbands, m->d_starts,
        stride, k_first, neg_bands);
  }
  B2S_CUDA_CHECK(cudaGetLastError());
  B2S_CUDA_CHECK(cudaEventRecord(m->ev[1], m->stream));

  // ---- response sweep ----
  // Pruned sweep (k_prune_select): only the angles that can change a result are swept.  It covers the one-tile,
  // stride-1, whole-grid window sweep of a complete coarse-stage CorrelateScan; kernel selector 3 keeps the dense sweep.
  const bool prune = use_window && na > 0 && m->force_kernel != 3 && m->mp_valid && stride == 1 && nbands == 1 &&
                     !s->fine && k_first == 0 && na == na_full && mode == 0 && nx <= 32 && ny <= 32 && na <= 1024;
  m->last_pruned = prune;
  m->sums_dense = !prune;
  if (na == 0) {
    m->last_path = use_window ? 2 : 1;  // empty angle subset of a split sweep: nothing to sweep
  } else if (use_window) {
    // (A variant that ran each match's fp64 tail inside the sweep CTA right after its last tile — volume read back from
    // L2, no k_reduce pass — was built, parity-tested and measured SLOWER on cfg 2, 8.80 -> 9.06 ms per 1024 matches: the
    // sweep kernel owns its SM, so the tail's serial stretches are no longer hidden by a second resident CTA as they are
    // in the stand-alone k_reduce.  Removed again; DESIGN.md §4.)
    // the GEN = false instantiation assumes exactly two lanes per row-start bank (see win_load)
    const int bank_step = ((m->g.width_step >> 2) * std::max(stride, 1)) & 31;
    m->win.stride = stride;
    m->win.gen = (bank_step & 3) != 2;
    m->win.smem = win_smem;
    m->win.ctas = (int)std::min<long long>((long long)B * nbands * (nbands > 1 ? tiles_y_w : 1), m->num_sms);
    m->win.copy_bytes = copy_bytes; m->win.band_rows = band_rows; m->win.nbands = nbands;
    m->win.band_bytes = band_bytes; m->win.neg_bands = neg_bands;
    if (prune) {
      if ((st = ensure_cap(&m->d_keep, &m->keep_cap, (size_t)B * na))) return st;
      if ((st = ensure_cap(&m->d_nkeep, &m->nkeep_cap, (size_t)B))) return st;
      const size_t psm = 4 * (size_t)m->mp_lq;
      B2S_CUDA_CHECK(raise_dyn_smem(k_prune_select, psm));
      k_prune_select<<<B, PRUNE_THREADS, psm, m->stream>>>(
          m->d_mp4, m->mp_pitch, m->mp_lq, m->mp_guard, m->d_grids, m->grid_pitch, m->g.data_size, m->g.width_step,
          m->d_lists, m->d_counts, m->d_starts, m->d_flags, m->d_centers, m->p, *s, n, na, nx, ny, m->d_keep,
          m->d_nkeep, m->d_stats);
      B2S_CUDA_CHECK(cudaGetLastError());
    }
    if ((st = launch_window(m, B, n, na, nx, ny, prune))) return st;
    // matches whose lattice is not the regular raster (a centre exactly on a rounding tie) fall through;
    // they compute their lookup values on the fly (no table was materialised for them)
    // (a few CTAs per match that exit at once unless the lattice is irregular: the kernel loops over the cells)
    k_sweep_generic<<<dim3(4, (unsigned)B), 256, 0, m->stream>>>(m->d_grids, m->grid_pitch, m->g.data_size, nullptr, m->d_bases,
                                                  m->d_flags, 1, n, na, ncell, m->d_sums, m->d_ranges, m->d_local,
                                                  m->d_grid_off, m->d_centers, s->angle_offset, s->angle_res,
                                                  m->g.width_step, scale, k_first);
    m->last_path = 2;
  } else {
    k_sweep_generic<<<ggrid, 256, 0, m->stream>>>(m->d_grids, m->grid_pitch, m->g.data_size, m->d_lut, m->d_bases,
                                                  m->d_flags, 0, n, na, ncell, m->d_sums, m->d_ranges, m->d_local,
                                                  m->d_grid_off, m->d_centers, s->angle_offset, s->angle_res,
                                                  m->g.width_step, scale, k_first);
    m->last_path = 1;
  }
  B2S_CUDA_CHECK(cudaGetLastError());
  B2S_CUDA_CHECK(cudaEventRecord(m->ev[2], m->stream));

  // ---- fp64 tail ----
  ReduceArgs ra = reduce_args(m, *s, nx, ny, na, k_first, mode);
  if (prune) { ra.keep = m->d_keep; ra.nkeep = m->d_nkeep; }
  k_reduce<<<B, RED_THREADS, 0, m->stream>>>(ra);
  if (s->fine) {
    size_t sm = sizeof(double) * (size_t)na;
    if (sm > 48 * 1024) B2S_FAIL(B2S_ERR_TOO_LARGE, "too many angles for the angular-covariance kernel");
    k_angular_cov<<<B, 256, sm, m->stream>>>(m->d_grids, m->grid_pitch, m->g, m->d_grid_off, m->d_lut, m->d_centers, *s,
                                             scale, n, na, m->d_results);
  }
  B2S_CUDA_CHECK(cudaGetLastError());
  B2S_CUDA_CHECK(cudaEventRecord(m->ev[3], m->stream));
  m->last.nx = nx; m->last.ny = ny; m->last.na = na;
  m->last_search = *s;
  m->last_k_first = k_first;
  m->have_sweep = true;
  return B2S_OK;
}

}  // namespace b2s

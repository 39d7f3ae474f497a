// lesson4 front end — hectorslam::HectorSlamProcessor on B200 (sm_100a).  Product code: CUDA only.
//
// Reference behaviour (paths relative to /root/reference/lesson4/include/lesson4/hector_mapping):
//   HectorSlamProcessor::update / reset                                  slam_main/HectorSlamProcessor.h:81-116
//   MapRepMultiMap ctor / matchData / updateByScan                       slam_main/MapRepMultiMap.h:56-191
//   ScanMatcher::matchData / estimateTransformationLogLh                 matcher/ScanMatcher.h:60-141
//   OccGridMapUtil::getCompleteHessianDerivs / interpMapValueWithDerivatives / getTransformForState
//                                                                        map/OccGridMapUtil.h:77-228, 437-440
//   OccGridMapBase::updateByScan / Bresenham / bresenhamCellFree/Occ     map/OccGridMapBase.h:118-168, 220-330
//   GridMapLogOddsFunctions::getGridProbability                          map/GridMapLogOdds.h:136-140
//   util::poseDifferenceLargerThan / normalize_angle                     util/UtilFunctions.h:36-48, 72-90
//   node loop: update(container, getLastScanMatchPose())                 lesson4/src/hector_mapping/hector_slam.cc:195-204
//
// Everything of one LaserScan runs on the device: the coarse-to-fine Gauss-Newton match, the map-update gate, the
// pose -> cell transform of the update and the Bresenham mark / apply passes.  The processor's state (last poses,
// update indices, stamp epochs, the coarse levels' data containers) lives in device memory, so a stream of scans needs
// no host round trip between scans (b2s_hector_slam_process_stream: ONE cooperative kernel walks the whole stream;
// b2s_hector_slam_update: one launch per scan, the pose comes back through a host-mapped mailbox as soon as the match
// is done while the map update still runs).  A handle holds B independent processors (independent robots / maps,
// SURVEY.md §8(e): "shard over independent maps"); B = 1 is the reference's single processor.
//
// Arithmetic: float32 in the reference's operation order, no FMA (-fmad=false).  EXACT mode (default) reproduces the
// reference bit for bit: the nine sums of getCompleteHessianDerivs are accumulated sequentially in point order (one lane
// per sum), Rotation2Df's std::cos / std::sin(float) are glibc's sincosf restated (glibc_math.cuh), the unqualified
// sin / cos / exp of the reference (C library DOUBLE functions rounded to float) are the device's double functions
// rounded to float (both are within 2 ulp of the exact double, so the float agrees unless the exact value lies within
// ~1e-16 relative of a float rounding boundary: ~5e-9 per evaluation).  FAST mode differs in ONE thing: the nine sums are
// tree-reduced (warp shuffles) instead of accumulated in point order, so its Hessians / poses differ in the last float bits
// (~1e-6 m per scan, inside the 1e-4 contract) and a cell can move when a pose lands an ulp away.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include <cooperative_groups.h>

#include "common.cuh"
#include "glibc_math.cuh"

using namespace b2s;

namespace b2s {

constexpr int HS_L = B2S_HECTOR_MAX_LEVELS;
constexpr int HS_THREADS = 576;          // 18 warps: two points per thread cover a 1081-beam scan in one pass
constexpr int HS_MAX_PTS = 4096;         // beams per scan (12-bit beam field of the stamps; shared-memory staging)
constexpr int HS_EPOCH_BITS = 20;
constexpr unsigned HS_EPOCH_MAX = (1u << HS_EPOCH_BITS) - 1;
constexpr int HS_STREAM_CTAS = 48;       // cooperative grid of the stream kernel (one CTA per SM, all co-resident)

struct HsLevel {  // one MapRepMultiMap level, all B processors ([b][cells] planes)
  float4 *quad;   // per cell (x, y): getGridProbability of the four cells (x, y), (x+1, y), (x, y+1), (x+1, y+1) — what one
                  // bilinear look-up of the matcher reads — refreshed whenever a cell's log-odds changes (the device-side
                  // form of the reference's per-scan GridMapCacheArray).  ONE 16-byte load per scan point instead of four
                  // scattered 4-byte ones: the match's per-point phase was bound by L1 tag throughput (gathers)
  float *lo;
  int32_t *ui;
  uint32_t *free_st, *occ_st;  // per-scan stamps: (epoch << 12) | (4095 - beam)
  float *pts;                  // [b][cap][2] data container of this level (level 0: the current scan)
  int sx, sy;
  float tw_lin, tw_tx, tw_ty, wt_lin, wt_tx, wt_ty;
  int iterations;  // 1 + maxIterations of MapRepMultiMap::matchData (:144-166): 1+5 on level 0, 1+3 above
};

struct HsState {  // device-resident state of ONE processor
  float last_update_pose[3], last_match_pose[3], last_cov[9];
  int curr_update_index[HS_L];
  unsigned int epoch[HS_L];
  int n_pts[HS_L];
  float origo[HS_L][2];
  // the update the gate decided for the current scan
  int do_update;
  float uc[HS_L], us[HS_L], umx[HS_L], umy[HS_L];
  int bx[HS_L], by[HS_L];
  unsigned int epoch_hi[HS_L];
  int mark_free[HS_L], mark_occ[HS_L];
  int bb_x0[HS_L], bb_y0[HS_L], bb_x1[HS_L], bb_y1[HS_L];  // cells the update's rays can touch (inclusive; empty: x1 < x0)
  unsigned long long visits, n_matched, n_updated;
  unsigned long long t_match_ns, t_update_ns;
};

struct HsBatch {  // kernel parameter
  HsLevel l[HS_L];
  int levels, batch, cap;
  float lo_free, lo_occ, min_dist, min_angle;
  int exact, use_fma;
  HsState *state;  // [batch]
};

struct HsCall {  // one scan per processor
  const float *pts0;    // [b][pts_stride][2] level-0 points (device, or host-mapped for the per-scan call)
  const int *n0;        // [b] (device / host-mapped) or NULL -> n0_uniform
  int n0_uniform, pts_stride;
  const float *hints;   // [b][3] or NULL -> the processor's last scan-match pose (the node's loop)
  float origo_x, origo_y;
  int map_without_matching;
  float *out;           // [b][16] device: pose[3], cov[9], updated, matched, exchange-lost, -
  volatile float *mailbox;  // host-mapped copy of out for processor 0 + sequence word, or NULL
  unsigned int seq;
  unsigned int tag;     // != 0: published (release, gpu scope) in out[b][15] once the scan's state is complete
  float *carry;         // shared-memory [3] or NULL: receives the scan-match pose (the next scan's hint in a stream)
};

__device__ __forceinline__ unsigned long long hs_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- thread-block cluster exchange of the fast single-stream match (k_hs_stream<false, true>) ----
// The per-point phase of a Gauss-Newton iteration is issue-bound on ONE SM (2600 of the iteration's 3700 cycles), so the
// CTAs of cluster 0 split the scan's points: rank 0 (the master) solves, the helpers receive the pose + sine / cosine and
// return their nine partial sums through distributed shared memory.  Data and signal travel together (st.async with
// mbarrier complete_tx): no cluster-scope fence, hence no L1 invalidation (CCTL.IVALL) inside the iteration loop.
// (Measured alternative: 8-byte {value, sequence} messages written with plain st.shared::cluster and polled with volatile
// shared loads — no mbarrier at all — took ~1000 cycles MORE per hop than st.async + try_wait: 21.5 k vs 29.9 k scans/s.)
constexpr int HS_CLUSTER = 4;
constexpr int HS_POSE_WORDS = 7;  // e0, e1, cos, sin, sinRot, cosRot, spare
struct __align__(16) HsXchg {
  unsigned long long bar_pose, bar_part;  // mbarriers: pose arrived (helpers) / all partial sums arrived (master)
  float pose[8];
  float part[8][12];                      // [rank][sum]
};
__device__ __forceinline__ uint32_t hs_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t hs_cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t hs_cluster_size() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t hs_mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void hs_st_async(uint32_t remote_addr, float v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr),
               "r"(__float_as_uint(v)), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void hs_mbar_init(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(hs_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void hs_mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(hs_smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded: a lost exchange must not hang the device (the host reports B2S_ERR_CUDA when the flag is set)
__device__ __forceinline__ bool hs_mbar_wait(unsigned long long *bar, uint32_t parity) {
  const uint32_t addr = hs_smem_u32(bar);
  const long long t0 = clock64();
  while (true) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return true;
    if (clock64() - t0 > (1ll << 25)) return false;  // ~17 ms; a legitimate wait is microseconds
  }
}
__device__ __forceinline__ void hs_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the points [p0, p1) of rank r when n points are split over `size` CTAs
__device__ __forceinline__ void hs_share(int n, int rank, int size, int &p0, int &p1) {
  const int chunk = (n + size - 1) / size;
  p0 = min(n, rank * chunk);
  p1 = min(n, p0 + chunk);
}

// interpMapValueWithDerivatives (OccGridMapUtil.h:139-228) in two halves so that the four cell loads of SEVERAL points are
// in flight together.  Plain loads (L1): within one launch the planes are only rewritten by the update passes, and every
// CTA passes the grid barrier's gpu-scope acquire (which drops the SM's L1 lines) between an update and the next match.
struct HsFetch {
  float i0, i1, i2, i3, fx, fy;
  bool inside;
};
__device__ __forceinline__ HsFetch hs_fetch(const float4 *__restrict__ quad, int sx, int sy, float x, float y) {
  HsFetch f;
  const float lim_x = (float)sx - 2.0f, lim_y = (float)sy - 2.0f;  // setMapCellDims: dims - 2
  f.inside = !(x < 0.0f || x > lim_x || y < 0.0f || y > lim_y);
  f.i0 = f.i1 = f.i2 = f.i3 = 0.0f; f.fx = f.fy = 0.0f;
  if (f.inside) {
    const int ix = (int)x, iy = (int)y;
    f.fx = x - (float)ix; f.fy = y - (float)iy;
    const float4 *c = quad + (iy * sx + ix);
    const float4 q = *c;
    f.i0 = q.x; f.i1 = q.y; f.i2 = q.z; f.i3 = q.w;
  }
  return f;
}
__device__ __forceinline__ void hs_finish(const HsFetch &f, float out[3]) {
  if (!f.inside) { out[0] = out[1] = out[2] = 0.0f; return; }
  const float dx1 = f.i0 - f.i1, dx2 = f.i2 - f.i3, dy1 = f.i0 - f.i2, dy2 = f.i1 - f.i3;
  const float xfi = 1.0f - f.fx, yfi = 1.0f - f.fy;
  out[0] = ((f.i0 * xfi + f.i1 * f.fx) * yfi) + ((f.i2 * xfi + f.i3 * f.fx) * f.fy);
  out[1] = -((dx1 * yfi) + (dx2 * f.fy));
  out[2] = -((dy1 * xfi) + (dy2 * f.fx));
}

__device__ __forceinline__ void hs_inv3_mul(const float m[9], const float v[3], float out[3]) {  // Matrix3f::inverse() * v
  const float c00 = m[4] * m[8] - m[5] * m[7], c10 = m[5] * m[6] - m[3] * m[8], c20 = m[3] * m[7] - m[4] * m[6];
  const float det = c00 * m[0] + (c10 * m[1] + c20 * m[2]);  /* Eigen's unrolled 3-term redux: a0 + (a1 + a2) */
  const float invdet = 1.0f / det;
  float inv[9];
  inv[0] = c00 * invdet; inv[3] = c10 * invdet; inv[6] = c20 * invdet;
  inv[1] = (m[2] * m[7] - m[1] * m[8]) * invdet;
  inv[4] = (m[0] * m[8] - m[2] * m[6]) * invdet;
  inv[7] = (m[1] * m[6] - m[0] * m[7]) * invdet;
  inv[2] = (m[1] * m[5] - m[2] * m[4]) * invdet;
  inv[5] = (m[2] * m[3] - m[0] * m[5]) * invdet;
  inv[8] = (m[0] * m[4] - m[1] * m[3]) * invdet;
  for (int r = 0; r < 3; r++) out[r] = inv[3 * r] * v[0] + (inv[3 * r + 1] * v[1] + inv[3 * r + 2] * v[2]);
}

// util::poseDifferenceLargerThan (UtilFunctions.h:72-90).  Only <cmath> is included there, so the unqualified
// abs(angleDiff) is int abs(int): the difference is truncated to an integer before the compare.
__device__ inline bool hs_pose_difference_larger_than(const float a[3], const float b[3], float dist_thresh,
                                                      float angle_thresh) {
  const float dx = a[0] - b[0], dy = a[1] - b[1];
  if (sqrtf(dx * dx + dy * dy) > dist_thresh) return true;
  float d = a[2] - b[2];
  const double pi = 3.14159265358979323846;
  if ((double)d > pi) d = (float)((double)d - pi * 2.0f);
  else if ((double)d < -pi) d = (float)((double)d + pi * 2.0f);
  const int t = (int)d;
  return (float)(t < 0 ? -t : t) > angle_thresh;
}

// terms of one point for getCompleteHessianDerivs (OccGridMapUtil.h:99-126)
__device__ __forceinline__ HsFetch hs_point_fetch(const float4 *__restrict__ prob, int sx, int sy, float2 p, float c, float s,
                                                  float e0, float e1) {
  const float tx = (c * p.x + (-s) * p.y) + e0, ty = (s * p.x + c * p.y) + e1;
  return hs_fetch(prob, sx, sy, tx, ty);
}
__device__ __forceinline__ void hs_point_terms(const HsFetch &f, float2 p, float sin_rot, float cos_rot, float a[9]) {
  float t[3];
  hs_finish(f, t);
  const float rot = ((-sin_rot * p.x - cos_rot * p.y) * t[1] + (cos_rot * p.x - sin_rot * p.y) * t[2]);
  const float fun = 1.0f - t[0];
  a[0] = t[1] * fun; a[1] = t[2] * fun; a[2] = rot * fun;    // dTr
  a[3] = t[1] * t[1]; a[4] = t[2] * t[2]; a[5] = rot * rot;  // H00 H11 H22
  a[6] = t[1] * t[2]; a[7] = t[1] * rot; a[8] = t[2] * rot;  // H01 H02 H12
}

// util::normalize_angle (UtilFunctions.h:36-48): double fmod, float result
__device__ __noinline__ float hs_normalize_angle(float e2) {
  const double two_pi = 2.0f * 3.14159265358979323846;
  const double d = (double)e2;
  double r;
  if (fabs(d) < two_pi) {
    // fmod(d, 2pi) = d here, and for x = d + 2pi in (0, 4pi): fmod(x, 2pi) = x - 2pi when x >= 2pi (exact: Sterbenz), else x.
    // Bit for bit the reference's two fmod calls, without the two software remainder loops (~1000 cycles per scan).
    const double x = d + two_pi;
    r = x >= two_pi ? x - two_pi : x;
  } else {
    r = fmod(fmod(d, two_pi) + two_pi, two_pi);
  }
  float a = (float)r;
  if ((double)a > 3.14159265358979323846) a = (float)((double)a - two_pi);  // `a -= 2.0f*M_PI` promotes to double
  return a;
}

struct HsTrig {
  float c, s;              // Rotation2Df(angle): std::cos / std::sin(float) = glibc cosf / sinf
  float sin_rot, cos_rot;  // OccGridMapUtil.h:87-88: the C library's double sin / cos, rounded to float
};
// (out of line on purpose: the Gauss-Newton loop is executed by few warps, so its code must stay inside the instruction
// cache — 60-90 KB kernels with the double-precision sincos / fmod expansions inlined at every use ran 2x slower)
__device__ __noinline__ HsTrig hs_trig(float angle, bool exact, bool use_fma) {
  HsTrig t;
  if (exact) {
    glibc_sincosf(angle, use_fma, &t.s, &t.c);
    double ds, dc;
    sincos((double)angle, &ds, &dc);
    t.sin_rot = (float)ds;
    t.cos_rot = (float)dc;
  } else {
    // fast mode: the glibc-exact float sine / cosine also stand in for sinRot / cosRot (they differ from the rounded
    // double ones on ~1 % of angles, by one ulp).  The device's own sincosf was tried here and broke the 1e-4 contract on
    // one scan of the test stream: a few Gauss-Newton iterations amplify an ulp of the rotation noticeably.
    glibc_sincosf(angle, use_fma, &t.s, &t.c);
    t.sin_rot = t.s;
    t.cos_rot = t.c;
  }
  return t;
}

struct HsLine {
  bool ok;
  int x0, y0, x1, y1;
  unsigned int da, db;
  int err0, off_a, off_b;
};

// endpoints (OccGridMapBase.h:127-154) + updateLineBresenhami set-up (:220-258)
__device__ __forceinline__ HsLine hs_line(float c, float s, float mx, float my, int bx, int by, float px, float py, int sx,
                                          int sy) {
  HsLine L;
  float ex = __fadd_rn(__fadd_rn(__fmul_rn(c, px), __fmul_rn(-s, py)), mx);
  float ey = __fadd_rn(__fadd_rn(__fmul_rn(s, px), __fmul_rn(c, py)), my);
  ex = __fadd_rn(ex, 0.5f);
  ey = __fadd_rn(ey, 0.5f);
  L.x0 = bx; L.y0 = by;
  L.x1 = (int)ex; L.y1 = (int)ey;  // Vector2f::cast<int>(): truncation
  L.ok = !(L.x0 == L.x1 && L.y0 == L.y1);
  if ((L.x0 < 0) || (L.x0 >= sx) || (L.y0 < 0) || (L.y0 >= sy)) L.ok = false;
  if ((L.x1 < 0) || (L.x1 >= sx) || (L.y1 < 0) || (L.y1 >= sy)) L.ok = false;
  const int dx = L.x1 - L.x0, dy = L.y1 - L.y0;
  const unsigned int adx = (unsigned int)abs(dx), ady = (unsigned int)abs(dy);
  const int odx = dx > 0 ? 1 : -1, ody = (dy > 0 ? 1 : -1) * sx;  // util::sign: sign(0) = -1
  if (adx >= ady) { L.da = adx; L.db = ady; L.err0 = (int)(adx / 2); L.off_a = odx; L.off_b = ody; }
  else { L.da = ady; L.db = adx; L.err0 = (int)(ady / 2); L.off_a = ody; L.off_b = odx; }
  return L;
}

// Fast mode, cluster variant: the per-point phase of this CTA's share (points [0, cnt) of `pts`) and the CTA's nine sums.
// The phase is ISSUE-bound (one SM retires ~500 warp instructions per warp and iteration in the two-points-per-thread
// form), so: only the warps that own points run it, every thread stores its nine terms as columns (9 STS instead of a
// 45-shuffle tree per warp), and warps 0..8 then sum one column each.  Returns sum `warp` in every lane of warps 0..8.
// Contains one __syncthreads.
__device__ __forceinline__ float hs_share_sums(const float4 *__restrict__ prob, int sx, int sy, const float2 *pts, int cnt,
                                               float factor, float e0, float e1, float c, float s, float sin_rot,
                                               float cos_rot, float *terms, int pitch, int tid, int lane, int warp) {
  if (warp * 32 < cnt) {
#pragma unroll 1
    for (int i = tid; i < cnt; i += HS_THREADS) {
      const float2 p = make_float2(__fmul_rn(pts[i].x, factor), __fmul_rn(pts[i].y, factor));
      const HsFetch f = hs_point_fetch(prob, sx, sy, p, c, s, e0, e1);
      float t[9];
      hs_point_terms(f, p, sin_rot, cos_rot, t);
#pragma unroll
      for (int q = 0; q < 9; q++) terms[q * pitch + i] = t[q];
    }
  }
  __syncthreads();
  float v = 0.0f;
  if (warp < 9) {
    const float *col = terms + warp * pitch;
    // (not unrolled on purpose: this runs once per iteration on cold instruction lines — the L0 instruction cache holds
    // ~6 KB and the iteration loop is larger — so executed code BYTES cost more than instructions)
    float v1 = 0.0f, v2 = 0.0f, v3 = 0.0f;  // four loads in flight: the loop is a latency chain, not a throughput one
    int i = lane;
#pragma unroll 1
    for (; i + 96 < cnt; i += 128) { v += col[i]; v1 += col[i + 32]; v2 += col[i + 64]; v3 += col[i + 96]; }
#pragma unroll 1
    for (; i < cnt; i += 32) v += col[i];
    v = (v + v1) + (v2 + v3);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  }
  return v;
}

// shared memory of the match: [cap] float2 staged scan, then (EXACT) 9 term columns of `pitch` floats / (FAST) per-warp partials
__host__ __device__ inline int hs_pitch(int cap) { return ((cap + 3) & ~3) + 4; }
__host__ __device__ inline size_t hs_terms_offset(int cap) { return (sizeof(float2) * (size_t)cap + 15) & ~(size_t)15; }  // float4 reads of the columns
__host__ __device__ inline size_t hs_smem_bytes(int cap) { return hs_terms_offset(cap) + sizeof(float) * 9 * (size_t)hs_pitch(cap) + 64; }

// MapRepMultiMap::matchData (:144-166) on every level, coarsest first, + the gate and the update parameters of
// HectorSlamProcessor::update (:81-108), by ONE CTA for processor b.
// Returns the gate's verdict (map update or not).
template <bool EXACT, bool CLUSTER>
__device__ bool hs_match_cta(const HsBatch &P, const HsCall &C, int b, unsigned char *smem, HsXchg *xc = nullptr,
                             uint32_t *xc_parity = nullptr) {
  static_assert(!(EXACT && CLUSTER), "the bit-exact sums are one sequential chain: nothing to split");
  HsState *st = P.state + b;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = HS_THREADS / 32;
  const int n = C.n0 ? C.n0[b] : C.n0_uniform;
  constexpr bool exact = EXACT;  // compile-time: each mode's kernel carries only its own code
  const bool use_fma = P.use_fma != 0;
  float2 *spts = reinterpret_cast<float2 *>(smem);
  float *terms = reinterpret_cast<float *>(smem + hs_terms_offset(P.cap));
  const int pitch = hs_pitch(P.cap);
  __shared__ float bc[8];    // estimate + trig published by the solving thread
  __shared__ float tot[9];
  __shared__ float s_world[3];
  __shared__ int s_do;
  __shared__ int s_bb[HS_L][4];
  __shared__ int s_lost;
  const uint32_t csize = CLUSTER ? hs_cluster_size() : 1u;
  uint32_t part_parity = CLUSTER ? *xc_parity : 0u;
  int my0 = 0, my1 = n;  // this CTA's share of the points in the per-point phase
  if (CLUSTER) hs_share(n, 0, (int)csize, my0, my1);
  if (CLUSTER && tid == 0) s_lost = 0;
  // master -> helpers: the pose of the next iteration (bc[0..6]) into every helper's HsXchg::pose; one st.async per lane
  // of warp 0 (the solving thread publishes nothing itself: 21 serial remote stores cost it ~300 cycles)
  auto publish = [&]() {
    if constexpr (CLUSTER) {
      const uint32_t a_pose = hs_smem_u32(xc->pose), a_bar = hs_smem_u32(&xc->bar_pose);
#pragma unroll 1
      for (uint32_t l = (uint32_t)lane; l + HS_POSE_WORDS < HS_POSE_WORDS * csize; l += 32) {
        const uint32_t r = 1 + l / HS_POSE_WORDS, q = l % HS_POSE_WORDS;
        hs_st_async(hs_mapa(a_pose + 4 * q, r), bc[q], hs_mapa(a_bar, r));
      }
    }
  };
  // state the serial tail needs, requested now so that the loads' latency hides behind the match (written last by this
  // same thread, or by an earlier kernel)
  float lup[3] = {0.0f, 0.0f, 0.0f}, lcov[9];
  unsigned long long n_matched0 = 0;
  if (tid == 0) {
    lup[0] = st->last_update_pose[0]; lup[1] = st->last_update_pose[1]; lup[2] = st->last_update_pose[2];
    n_matched0 = st->n_matched;
#pragma unroll
    for (int q = 0; q < 9; q++) lcov[q] = st->last_cov[q];
  }
  const unsigned long long t0 = hs_now_ns();
  const float2 *gp = reinterpret_cast<const float2 *>(C.pts0) + (size_t)b * C.pts_stride;
  for (int i = tid; i < n; i += HS_THREADS) {
    const float2 p = gp[i];
    spts[i] = p;
    reinterpret_cast<float2 *>(P.l[0].pts)[(size_t)b * P.cap + i] = p;  // level-0 container for the update passes
  }
  if (tid == 0) {
    const float *h = C.hints ? C.hints + 3 * b : st->last_match_pose;
    s_world[0] = h[0]; s_world[1] = h[1]; s_world[2] = h[2];
  }
  __syncthreads();
  float world0 = s_world[0], world1 = s_world[1], world2 = s_world[2];
  bool any = false;
  if (!C.map_without_matching && n > 0) {
    float factor = 1.0f;
    for (int l = 1; l < P.levels; l++) factor *= 0.5f;  // static_cast<float>(1.0 / pow(2.0, l)) is exactly 2^-l
    for (int lv = P.levels - 1; lv >= 0; lv--, factor *= 2.0f) {
      const HsLevel &m = P.l[lv];
      const float4 *prob = m.quad + (size_t)b * m.sx * m.sy;
      if (lv > 0)  // dataContainers[lv-1].setFrom(dataContainer, 2^-lv) (DataPointContainer.h:46-59): exact scaling
        for (int i = tid; i < n; i += HS_THREADS)
          reinterpret_cast<float2 *>(m.pts)[(size_t)b * P.cap + i] = make_float2(__fmul_rn(spts[i].x, factor), __fmul_rn(spts[i].y, factor));
      // getMapCoordsPose (GridMapBase.h:238-242)
      if (tid == 0) {
        const float e0 = (m.tw_lin * world0 + 0.0f * world1) + m.tw_tx;
        const float e1 = (0.0f * world0 + m.tw_lin * world1) + m.tw_ty;
        const HsTrig tr = hs_trig(world2, exact, use_fma);
        bc[0] = e0; bc[1] = e1; bc[2] = world2; bc[3] = tr.c; bc[4] = tr.s; bc[5] = tr.sin_rot; bc[6] = tr.cos_rot;
      }
      if (CLUSTER && warp == 0) {
        __syncwarp();
        publish();
      }
      __syncthreads();
      for (int it = 0; it < m.iterations; it++) {
        const float e0 = bc[0], e1 = bc[1], c = bc[3], s = bc[4], sin_rot = bc[5], cos_rot = bc[6];
        if constexpr (CLUSTER) {
          float v = 0.0f;
          if (my1 > 0) v = hs_share_sums(prob, m.sx, m.sy, spts, my1, factor, e0, e1, c, s, sin_rot, cos_rot, terms, pitch, tid, lane, warp);
          if (warp < 9) {
            if (csize > 1) {  // + the helpers' partial sums, in rank order
              if (tid == 0) hs_mbar_expect_tx(&xc->bar_part, 36u * (csize - 1));
              if (!hs_mbar_wait(&xc->bar_part, part_parity)) s_lost = 1;  // every reading thread observes the phase itself
#pragma unroll 1
              for (uint32_t r = 1; r < csize; r++) v += xc->part[r][warp];
            }
            if (lane == 0) tot[warp] = v;
          }
          if (csize > 1) part_parity ^= 1u;
          __syncthreads();
        } else {
        float acc[9];
#pragma unroll
        for (int q = 0; q < 9; q++) acc[q] = 0.0f;
        for (int base = my0; base < my1; base += 2 * HS_THREADS) {  // two points per thread, their eight cell loads in flight together
          const int ia = base + tid, ib = base + tid + HS_THREADS;
          const int n = my1;  // (shadows the scan length inside the per-point phase: this CTA's share ends at my1)
          float2 pa = make_float2(0.0f, 0.0f), pb = pa;
          HsFetch fa, fb;
          fa.inside = fb.inside = false;
          if (ia < n) { pa = make_float2(__fmul_rn(spts[ia].x, factor), __fmul_rn(spts[ia].y, factor)); fa = hs_point_fetch(prob, m.sx, m.sy, pa, c, s, e0, e1); }
          if (ib < n) { pb = make_float2(__fmul_rn(spts[ib].x, factor), __fmul_rn(spts[ib].y, factor)); fb = hs_point_fetch(prob, m.sx, m.sy, pb, c, s, e0, e1); }
          float ta[9], tb[9];
          if (ia < n) {
            hs_point_terms(fa, pa, sin_rot, cos_rot, ta);
            if (exact) {
#pragma unroll
              for (int q = 0; q < 9; q++) terms[q * pitch + ia] = ta[q];
            } else {
#pragma unroll
              for (int q = 0; q < 9; q++) acc[q] += ta[q];
            }
          }
          if (ib < n) {
            hs_point_terms(fb, pb, sin_rot, cos_rot, tb);
            if (exact) {
#pragma unroll
              for (int q = 0; q < 9; q++) terms[q * pitch + ib] = tb[q];
            } else {
#pragma unroll
              for (int q = 0; q < 9; q++) acc[q] += tb[q];
            }
          }
        }
        if (!exact) {
#pragma unroll
          for (int q = 0; q < 9; q++) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], d);
          }
          if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 9; q++) terms[q * NW + warp] = acc[q];
          }
        }
        __syncthreads();
        if (exact) {
          // The reference's float32 sums, in point order (OccGridMapUtil.h:99-126): ONE warp instruction advances all nine
          // chains (lane q owns sum q), so the floor is one dependent FADD per point.  (Nine warps with one chain each
          // share four schedulers and measured 2.5x slower.)
          if (warp == 0 && lane < 9) {
            float acc = 0.0f;
            const float *col = terms + lane * pitch;
            int i = 0;
            for (; i + 32 <= n; i += 32) {  // eight 16-byte loads in flight ahead of the 32 dependent adds they feed
              float4 t[8];
#pragma unroll
              for (int j = 0; j < 8; j++) t[j] = *reinterpret_cast<const float4 *>(col + i + 4 * j);
#pragma unroll
              for (int j = 0; j < 8; j++) {
                acc = __fadd_rn(acc, t[j].x); acc = __fadd_rn(acc, t[j].y); acc = __fadd_rn(acc, t[j].z); acc = __fadd_rn(acc, t[j].w);
              }
            }
            for (; i + 8 <= n; i += 8) {
              const float4 u = *reinterpret_cast<const float4 *>(col + i), w = *reinterpret_cast<const float4 *>(col + i + 4);
              acc = __fadd_rn(acc, u.x); acc = __fadd_rn(acc, u.y); acc = __fadd_rn(acc, u.z); acc = __fadd_rn(acc, u.w);
              acc = __fadd_rn(acc, w.x); acc = __fadd_rn(acc, w.y); acc = __fadd_rn(acc, w.z); acc = __fadd_rn(acc, w.w);
            }
            for (; i < n; i++) acc = __fadd_rn(acc, col[i]);
            tot[lane] = acc;
          }
          __syncthreads();
        } else if (warp == 0) {
          float v = 0.0f;
          if (lane < 9)
            for (int w = 0; w < NW; w++) v += terms[lane * NW + w];
          if (lane < 9) tot[lane] = v;
          __syncwarp();
        }
        }  // !CLUSTER
        if (tid == 0) {  // estimateTransformationLogLh (ScanMatcher.h:107-141)
          const float dTr[3] = {tot[0], tot[1], tot[2]};
          float Hm[9];
          Hm[0] = tot[3]; Hm[4] = tot[4]; Hm[8] = tot[5];
          Hm[1] = Hm[3] = tot[6]; Hm[2] = Hm[6] = tot[7]; Hm[5] = Hm[7] = tot[8];
          float n0 = bc[0], n1 = bc[1], n2 = bc[2];
          if (Hm[0] != 0.0f && Hm[4] != 0.0f) {
            float dir[3];
            hs_inv3_mul(Hm, dTr, dir);
            if (dir[2] > 0.2f) dir[2] = 0.2f;
            else if (dir[2] < -0.2f) dir[2] = -0.2f;
            n0 += dir[0]; n1 += dir[1]; n2 += dir[2];
          }
          bc[0] = n0; bc[1] = n1; bc[2] = n2;
          if (it + 1 < m.iterations) {
            const HsTrig tr = hs_trig(n2, exact, use_fma);
            bc[3] = tr.c; bc[4] = tr.s; bc[5] = tr.sin_rot; bc[6] = tr.cos_rot;
          }
        }
        if (CLUSTER && warp == 0 && it + 1 < m.iterations) {
          __syncwarp();
          publish();
        }
        __syncthreads();
      }
      {
        const float e0 = bc[0], e1 = bc[1], e2 = bc[2];
        const float a = hs_normalize_angle(e2);
        world0 = (m.wt_lin * e0 + (-0.0f) * e1) + m.wt_tx;  // getWorldCoordsPose (GridMapBase.h:229-233)
        world1 = ((-0.0f) * e0 + m.wt_lin * e1) + m.wt_ty;
        world2 = a;
        any = true;
      }
      __syncthreads();  // bc / tot are rewritten by the next level
    }
  }
  if (tid == 0) {
    // ---- HectorSlamProcessor::update after the match (:88-107) ----
    float est[3] = {world0, world1, world2};
    if (any) {  // covMatrix = H of the last level matched (level 0)
      lcov[0] = tot[3]; lcov[4] = tot[4]; lcov[8] = tot[5];
      lcov[1] = lcov[3] = tot[6]; lcov[2] = lcov[6] = tot[7];
      lcov[5] = lcov[7] = tot[8];
#pragma unroll
      for (int q = 0; q < 9; q++) st->last_cov[q] = lcov[q];
    }
    if (!C.map_without_matching) {
      st->n_matched = n_matched0 + 1;
      if (n > 0) {
        float factor = 1.0f;
        for (int l = 1; l < P.levels; l++) {
          factor *= 0.5f;
          st->n_pts[l] = n;
          st->origo[l][0] = C.origo_x * factor; st->origo[l][1] = C.origo_y * factor;
        }
      } else {
        for (int l = 1; l < P.levels; l++) st->n_pts[l] = 0;  // setFrom of an empty container
      }
    }
    st->n_pts[0] = n;
    st->origo[0][0] = C.origo_x; st->origo[0][1] = C.origo_y;
    st->last_match_pose[0] = est[0]; st->last_match_pose[1] = est[1]; st->last_match_pose[2] = est[2];
    if (C.carry) { C.carry[0] = est[0]; C.carry[1] = est[1]; C.carry[2] = est[2]; }
    const bool do_update = hs_pose_difference_larger_than(est, lup, P.min_dist, P.min_angle) ||
                           C.map_without_matching;
    st->do_update = do_update ? 1 : 0;
    if (do_update) {
      float uc, us;  // Rotation2Df of the update transform: glibc cosf / sinf -> the same cells as the CPU
      glibc_sincosf(est[2], use_fma, &us, &uc);
      for (int l = 0; l < P.levels; l++) {
        const HsLevel &m = P.l[l];
        const float mx = (m.tw_lin * est[0] + 0.0f * est[1]) + m.tw_tx;  // getMapCoordsPose (GridMapBase.h:238-242)
        const float my = (0.0f * est[0] + m.tw_lin * est[1]) + m.tw_ty;
        st->uc[l] = uc; st->us[l] = us; st->umx[l] = mx; st->umy[l] = my;
        const float bxf = (uc * st->origo[l][0] + (-us) * st->origo[l][1]) + mx;
        const float byf = (us * st->origo[l][0] + uc * st->origo[l][1]) + my;
        st->bx[l] = (int)(bxf + 0.5f); st->by[l] = (int)(byf + 0.5f);  // Vector2i(float, float): truncation
        st->epoch[l] += 1;
        st->epoch_hi[l] = st->epoch[l] << 12;
        st->mark_free[l] = st->curr_update_index[l] + 1;  // OccGridMapBase.h:120-121
        st->mark_occ[l] = st->curr_update_index[l] + 2;
        st->curr_update_index[l] += 3;                    // :167
      }
      st->last_update_pose[0] = est[0]; st->last_update_pose[1] = est[1]; st->last_update_pose[2] = est[2];
      st->n_updated += 1;
    }
    float *o = C.out + 16 * (size_t)b;
    o[0] = est[0]; o[1] = est[1]; o[2] = est[2];
    for (int q = 0; q < 9; q++) o[3 + q] = lcov[q];
    o[12] = do_update ? 1.0f : 0.0f;
    o[13] = any ? 1.0f : 0.0f;
    o[14] = (CLUSTER && s_lost) ? 1.0f : 0.0f;  // a cluster exchange timed out: the host fails the call
    if (C.mailbox && b == 0) {
      for (int q = 0; q < 15; q++) C.mailbox[q] = o[q];
      __threadfence_system();
      reinterpret_cast<volatile unsigned int *>(C.mailbox)[15] = C.seq;
      __threadfence_system();
    }
    s_do = do_update ? 1 : 0;
  }
  __syncthreads();
  if (s_do) {
    // cells the rays of this update can touch, per level: the apply pass sweeps this box instead of re-walking the rays
    if (tid < HS_L * 4) s_bb[tid >> 2][tid & 3] = (tid & 2) ? -2147483647 : 2147483647;  // {min x, min y, max x, max y}
    __syncthreads();
    for (int lv = 0; lv < P.levels; lv++) {
      const HsLevel &m = P.l[lv];
      const int nl = st->n_pts[lv];
      const float c = st->uc[lv], s = st->us[lv], mx = st->umx[lv], my = st->umy[lv];
      const int bx = st->bx[lv], by = st->by[lv];
      const float2 *pp = reinterpret_cast<const float2 *>(m.pts) + (size_t)b * P.cap;
      int lo_x = 2147483647, lo_y = 2147483647, hi_x = -2147483647, hi_y = -2147483647;
      for (int i = tid; i < nl; i += HS_THREADS) {
        const float2 pt = pp[i];
        const HsLine ln = hs_line(c, s, mx, my, bx, by, pt.x, pt.y, m.sx, m.sy);
        if (!ln.ok) continue;
        lo_x = min(lo_x, min(ln.x0, ln.x1)); hi_x = max(hi_x, max(ln.x0, ln.x1));
        lo_y = min(lo_y, min(ln.y0, ln.y1)); hi_y = max(hi_y, max(ln.y0, ln.y1));
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        lo_x = min(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, d)); lo_y = min(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, d));
        hi_x = max(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, d)); hi_y = max(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, d));
      }
      if (lane == 0) {
        atomicMin(&s_bb[lv][0], lo_x); atomicMin(&s_bb[lv][1], lo_y);
        atomicMax(&s_bb[lv][2], hi_x); atomicMax(&s_bb[lv][3], hi_y);
      }
    }
    __syncthreads();
    if (tid < P.levels) {
      st->bb_x0[tid] = s_bb[tid][0]; st->bb_y0[tid] = s_bb[tid][1];
      st->bb_x1[tid] = s_bb[tid][2]; st->bb_y1[tid] = s_bb[tid][3];  // no ray: max < min -> an empty box
    }
  }
  if (tid == 0) st->t_match_ns = hs_now_ns() - t0;
  if (CLUSTER) *xc_parity = part_parity;
  const bool verdict = s_do != 0;
  if (C.tag) {
    __syncthreads();  // the bounding boxes (other threads' stores) are ordered before the release below
    if (tid == 0)
      asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(C.out + 16 * (size_t)b + 15), "r"(C.tag) : "memory");
  }
  return verdict;
}

// every CTA but the matching one: wait until scan i's row carries this launch's tag, then read the gate's verdict
__device__ __forceinline__ bool hs_wait_decision(const float *row, unsigned int tag, int *s_flag) {
  if (threadIdx.x == 0) {
    while (true) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(row + 15) : "memory");
      if (v == tag) break;
      __nanosleep(40);
    }
    *s_flag = __ldcg(row + 12) != 0.0f ? 1 : 0;
  }
  __syncthreads();
  const bool r = *s_flag != 0;
  __syncthreads();  // s_flag may be rewritten for the next scan
  return r;
}

// A helper CTA of cluster 0 (rank >= 1): the same level / iteration loops as hs_match_cta, but only the per-point phase of
// its share of the scan; the pose comes from the master, the nine partial sums go back to it.
__device__ void hs_match_helper(const HsBatch &P, const HsCall &C, unsigned char *smem, HsXchg *xc, uint32_t rank,
                                uint32_t csize, uint32_t &pose_parity) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = C.n0_uniform;
  if (C.map_without_matching || n <= 0) return;
  float2 *spts = reinterpret_cast<float2 *>(smem);
  float *terms = reinterpret_cast<float *>(smem + hs_terms_offset(P.cap));
  int p0, p1;
  hs_share(n, (int)rank, (int)csize, p0, p1);
  const int cnt = p1 - p0;
  const float2 *gp = reinterpret_cast<const float2 *>(C.pts0);
  for (int i = tid; i < cnt; i += HS_THREADS) spts[i] = gp[p0 + i];
  __syncthreads();
  const int pitch = hs_pitch(P.cap);
  const uint32_t r_part = hs_mapa(hs_smem_u32(&xc->part[rank][0]), 0), r_bar = hs_mapa(hs_smem_u32(&xc->bar_part), 0);
  float factor = 1.0f;
  for (int l = 1; l < P.levels; l++) factor *= 0.5f;
  for (int lv = P.levels - 1; lv >= 0; lv--, factor *= 2.0f) {
    const HsLevel &m = P.l[lv];
    const float4 *prob = m.quad;
    for (int it = 0; it < m.iterations; it++) {
      if (tid == 0) hs_mbar_expect_tx(&xc->bar_pose, 4u * HS_POSE_WORDS);
      hs_mbar_wait(&xc->bar_pose, pose_parity);  // every thread observes the phase itself (a time-out is reported by the master)
      pose_parity ^= 1u;
      // Not needed for ordering — the master sends this pose only after it holds all nine sums of the previous iteration,
      // which are sent after the column reads — but that chain runs through another CTA, which compute-sanitizer's
      // racecheck cannot follow: the barrier (~50 cycles) keeps the tool's report clean.
      __syncthreads();
      const float e0 = xc->pose[0], e1 = xc->pose[1], c = xc->pose[3], s = xc->pose[4], sin_rot = xc->pose[5], cos_rot = xc->pose[6];
      const float v = hs_share_sums(prob, m.sx, m.sy, spts, cnt, factor, e0, e1, c, s, sin_rot, cos_rot, terms, pitch, tid, lane, warp);
      if (warp < 9 && lane == 0) hs_st_async(r_part + 4 * warp, v, r_bar);
    }
  }
}

// the update parameters of one level as the gate wrote them.  Plain (L1) loads: within the persistent launch every CTA
// passes the grid barrier between the gate's writes and these reads, and the barrier's gpu-scope acquire drops the SM's
// L1 (CCTL.IVALL); in the batch path a kernel boundary lies in between.  (With L2 loads the ~dozen dependent state reads
// at the head of every warp were 47 % of k_hs_apply's stall samples.)
struct HsUpd {
  int n;
  float c, s, mx, my;
  int bx, by;
  uint32_t ehi;
  int mark_free, mark_occ;
};
__device__ __forceinline__ HsUpd hs_load_upd(const HsState *st, int lv) {
  HsUpd u;
  u.n = st->n_pts[lv];
  u.c = st->uc[lv]; u.s = st->us[lv]; u.mx = st->umx[lv]; u.my = st->umy[lv];
  u.bx = st->bx[lv]; u.by = st->by[lv];
  u.ehi = st->epoch_hi[lv];
  u.mark_free = st->mark_free[lv]; u.mark_occ = st->mark_occ[lv];
  return u;
}

__device__ __forceinline__ float hs_prob_of(float lo) {  // getGridProbability (GridMapLogOdds.h:136-140)
  const float odds = (float)exp((double)lo);  // unqualified exp(): the C library's double exp, rounded to float
  return odds / (odds + 1.0f);
}

// MapRepMultiMap::updateByScan (:174-191) for processor b, PASS 1 (mark): work item = (level, beam), flattened over
// the levels, one warp each; lanes over Bresenham steps in closed form.  Every traversed cell records the LOWEST beam
// index that frees it / ends on it (32-bit atomicMax of epoch | ~beam).  Returns this warp's cell visits.
__device__ unsigned long long hs_mark_pass(const HsBatch &P, int b, int w, int nw, int lane) {
  const HsState *st = P.state + b;
  unsigned long long my_visits = 0;
  int first[HS_L + 1];
  first[0] = 0;
  for (int lv = 0; lv < P.levels; lv++) first[lv + 1] = first[lv] + st->n_pts[lv];
  int lv = 0;
  HsUpd u = hs_load_upd(st, 0);
  for (int j = w; j < first[P.levels]; j += nw) {
    if (j >= first[lv + 1]) {
      while (j >= first[lv + 1]) lv++;
      u = hs_load_upd(st, lv);
    }
    const int i = j - first[lv];
    const HsLevel &m = P.l[lv];
    const size_t cells = (size_t)m.sx * m.sy;
    uint32_t *fs = m.free_st + (size_t)b * cells, *os = m.occ_st + (size_t)b * cells;
    const float2 pt = __ldcg(reinterpret_cast<const float2 *>(m.pts) + (size_t)b * P.cap + i);
    const HsLine ln = hs_line(u.c, u.s, u.mx, u.my, u.bx, u.by, pt.x, pt.y, m.sx, m.sy);
    if (!ln.ok) continue;
    const uint32_t stamp = u.ehi | (uint32_t)(4095 - i);
    const int start = ln.y0 * m.sx + ln.x0;
    for (unsigned int k = lane; k < ln.da; k += 32) {  // bresenham2D: da cells from the start, end excluded
      const unsigned int inc = (unsigned int)(((unsigned long long)ln.err0 + (unsigned long long)k * ln.db) / ln.da);
      atomicMax(fs + (start + (int)k * ln.off_a + (int)inc * ln.off_b), stamp);
    }
    if (lane == 0) {
      atomicMax(os + (ln.y1 * m.sx + ln.x1), stamp);
      my_visits += (unsigned long long)ln.da + 1;
    }
  }
  return my_visits;
}

// the probability of cell (x, y) enters the quads of (x, y), (x-1, y), (x, y-1), (x-1, y-1)
__device__ __forceinline__ void hs_publish_prob(float4 *__restrict__ quad, int sx, int x, int y, float p) {
  float *q = reinterpret_cast<float *>(quad + (y * sx + x));
  q[0] = p;
  if (x > 0) q[-4 + 1] = p;
  if (y > 0) {
    q[-4 * sx + 2] = p;
    if (x > 0) q[-4 * sx - 4 + 3] = p;
  }
}

// PASS 2 (apply): a dense, coalesced sweep over each level's bounding box of the rays (work item = 128 consecutive
// cells of a row: four 128-byte loads per stamp plane per warp).  A cell stamped in this epoch gets the reference's
// update exactly once: end cells (occ stamp of this epoch; the stamp's winner is the lowest beam ending there) take
// bresenhamCellOcc — with the "(v + f) - f" un-free rounding iff a LOWER beam index had freed the cell first (its
// free stamp, same epoch, is larger) — then += logOddsOccupied if v < 50; cells only freed take bresenhamCellFree.
// The floats are those of the sequential loop (OccGridMapBase.h:302-330), whatever the execution order.
__device__ void hs_apply_pass(const HsBatch &P, int b, int w, int nw, int lane) {
  const HsState *st = P.state + b;
  int first[HS_L + 1], x0[HS_L], y0[HS_L], x1[HS_L], chunks[HS_L];
  first[0] = 0;
  for (int lv = 0; lv < P.levels; lv++) {
    x0[lv] = st->bb_x0[lv]; y0[lv] = st->bb_y0[lv];
    x1[lv] = st->bb_x1[lv];
    const int y1 = st->bb_y1[lv];
    const bool any = x1[lv] >= x0[lv] && y1 >= y0[lv];
    chunks[lv] = any ? (x1[lv] - x0[lv] + 128) / 128 : 0;
    first[lv + 1] = first[lv] + (any ? (y1 - y0[lv] + 1) * chunks[lv] : 0);
  }
  int lv = 0;
  for (int j = w; j < first[P.levels]; j += nw) {
    while (j >= first[lv + 1]) lv++;
    const HsLevel &m = P.l[lv];
    const size_t cells = (size_t)m.sx * m.sy;
    const uint32_t *fs = m.free_st + (size_t)b * cells, *os = m.occ_st + (size_t)b * cells;
    float *lo = m.lo + (size_t)b * cells;
    float4 *quad = m.quad + (size_t)b * cells;
    int32_t *ui = m.ui + (size_t)b * cells;
    const uint32_t ep = st->epoch_hi[lv] >> 12;
    const int mark_free = st->mark_free[lv], mark_occ = st->mark_occ[lv];
    const int r = j - first[lv];
    const int y = y0[lv] + r / chunks[lv];
    const int xb = x0[lv] + (r % chunks[lv]) * 128 + lane;
    uint32_t f[4], o[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int x = xb + 32 * q;
      f[q] = o[q] = 0;
      if (x <= x1[lv]) {
        f[q] = __ldcg(fs + (y * m.sx + x));
        o[q] = __ldcg(os + (y * m.sx + x));
      }
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int off = y * m.sx + xb + 32 * q;
      if (o[q] != 0 && (o[q] >> 12) == ep) {  // bresenhamCellOcc (:315-330)
        float v = __ldcg(lo + off);
        if ((f[q] >> 12) == ep && f[q] > o[q]) {  // a lower beam index freed it first: set free, then unset
          v = __fadd_rn(v, P.lo_free);
          v = __fsub_rn(v, P.lo_free);
        }
        if (v < 50.0f) v = __fadd_rn(v, P.lo_occ);
        lo[off] = v;
        hs_publish_prob(quad, m.sx, xb + 32 * q, y, hs_prob_of(v));
        ui[off] = mark_occ;
      } else if (f[q] != 0 && (f[q] >> 12) == ep) {  // bresenhamCellFree (:302-312)
        const float v = __fadd_rn(__ldcg(lo + off), P.lo_free);
        lo[off] = v;
        hs_publish_prob(quad, m.sx, xb + 32 * q, y, hs_prob_of(v));
        ui[off] = mark_free;
      }
    }
  }
}

// ---- batch path: three launches per step over all B processors ----
// The matching kernels ask for one CTA per SM: the Gauss-Newton loop keeps its terms in registers (90-96 per thread).
// Without the minimum ptxas may cap them at 56 so that two CTAs fit, and spill inside the per-point phase.
template <bool EXACT>
__global__ void __launch_bounds__(HS_THREADS, 1) k_hs_match(HsBatch P, HsCall C) {
  extern __shared__ __align__(16) unsigned char hs_smem[];
  hs_match_cta<EXACT, false>(P, C, blockIdx.x, hs_smem);
}
__global__ void __launch_bounds__(256) k_hs_mark(HsBatch P) {
  const int b = blockIdx.y;
  if (!P.state[b].do_update) return;
  const int lane = threadIdx.x & 31;
  const unsigned long long v = hs_mark_pass(P, b, (blockIdx.x * blockDim.x + threadIdx.x) >> 5, (gridDim.x * blockDim.x) >> 5, lane);
  if (lane == 0 && v) atomicAdd(&P.state[b].visits, v);  // lane 0 carries the warp's count
}
__global__ void __launch_bounds__(256) k_hs_apply(HsBatch P) {
  const int b = blockIdx.y;
  if (!P.state[b].do_update) return;
  hs_apply_pass(P, b, (blockIdx.x * blockDim.x + threadIdx.x) >> 5, (gridDim.x * blockDim.x) >> 5, threadIdx.x & 31);
}

// ---- single-processor path: ONE cooperative launch walks n_scans scans (n_scans = 1 for b2s_hector_slam_update) ----
// CTA 0 matches while the other CTAs wait at the grid barrier; then every CTA takes beams of the update passes.
__device__ __forceinline__ void hs_grid_barrier(unsigned int *counter, unsigned int &generation) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int target = (generation + 1) * gridDim.x;
    atomicAdd(counter, 1u);
    while (true) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= target) break;
      __nanosleep(40);
    }
    __threadfence();
  }
  generation++;
  __syncthreads();
}

struct HsStream {
  const float *pts;      // concatenated scans (device, or host-mapped for a single scan)
  const int *offsets;    // [n_scans] first point of each scan, or NULL (single scan at 0)
  const int *counts;     // [n_scans] or NULL -> count0
  int count0, n_scans;
  const float *hints;    // [n_scans][3] or NULL (chain through the processor's last scan-match pose)
  const float *first_hint;  // device [3] or NULL
  float origo_x, origo_y;
  int map_without_matching;
  float *out;            // [n_scans][16]
  volatile float *mailbox;
  unsigned int seq;
  unsigned int *barrier;
  unsigned int tag;      // this launch's id (never 0): scan i is decided once out[i][15] holds it
};

template <bool EXACT, bool CLUSTER>
__global__ void __launch_bounds__(HS_THREADS, 1) k_hs_stream(HsBatch P, HsStream S) {
  extern __shared__ __align__(16) unsigned char hs_smem[];
  __shared__ HsXchg xc;  // same offset in every CTA of the kernel: mapa() of a local address names the peer's copy
  __shared__ int s_flag;
  uint32_t crank = 0, csize = 1, pose_parity = 0, part_parity = 0;
  if (CLUSTER) {
    crank = hs_cluster_rank();
    csize = hs_cluster_size();
    if (threadIdx.x == 0) {
      hs_mbar_init(&xc.bar_pose, 1);
      hs_mbar_init(&xc.bar_part, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    hs_cluster_sync();  // no peer signals a barrier that is not initialised yet (once per launch)
  }
  const bool helper = CLUSTER && blockIdx.x < csize && crank != 0;  // cluster 0 = CTAs [0, csize)
  unsigned int generation = 0;
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * HS_THREADS + threadIdx.x) >> 5, nw = (gridDim.x * HS_THREADS) >> 5;
  HsState *st = P.state;
  __shared__ float s_last[3];  // the matching CTA's last scan-match pose: the next scan's hint without a global round trip
  int next_off = (S.offsets && S.n_scans > 0) ? S.offsets[0] : 0, next_cnt = (S.counts && S.n_scans > 0) ? S.counts[0] : S.count0;
  for (int i = 0; i < S.n_scans; i++) {
    bool update;
    HsCall C;
    const int off = next_off, cnt_i = next_cnt;
    if (i + 1 < S.n_scans) {  // requested a whole scan ahead of their use
      if (S.offsets) next_off = S.offsets[i + 1];
      if (S.counts) next_cnt = S.counts[i + 1];
    }
    C.pts0 = S.pts + 2 * (size_t)off;
    C.n0 = nullptr;
    C.n0_uniform = cnt_i;
    C.pts_stride = 0;
    C.hints = S.hints ? S.hints + 3 * (size_t)i : ((i == 0 && S.first_hint) ? S.first_hint : (i > 0 ? s_last : nullptr));
    C.carry = s_last;
    C.origo_x = S.origo_x; C.origo_y = S.origo_y;
    C.map_without_matching = S.map_without_matching;
    C.out = S.out + 16 * (size_t)i;
    C.mailbox = S.mailbox;
    C.seq = S.seq;
    C.tag = S.tag;
    // The matching CTA never waits for the others unless the map is updated: it publishes the scan's verdict (release) and
    // goes on to the next scan; the other CTAs follow the verdicts and meet it at the update's barriers.  (A grid barrier
    // per scan cost the matching CTA ~1 us: two fences and an L2 round trip.)
    if (blockIdx.x == 0) {
      update = hs_match_cta<EXACT, CLUSTER>(P, C, 0, hs_smem, &xc, &part_parity);
    } else {
      if (helper) hs_match_helper(P, C, hs_smem, &xc, crank, csize, pose_parity);
      update = hs_wait_decision(C.out, S.tag, &s_flag);
    }
    if (update) {
      const unsigned long long t0 = hs_now_ns();
      const unsigned long long v = hs_mark_pass(P, 0, w, nw, lane);
      if (lane == 0 && v) atomicAdd(&st->visits, v);
      hs_grid_barrier(S.barrier, generation);
      hs_apply_pass(P, 0, w, nw, lane);
      hs_grid_barrier(S.barrier, generation);  // the next match reads the refreshed probability planes
      if (blockIdx.x == 0 && threadIdx.x == 0) st->t_update_ns = hs_now_ns() - t0;
    }
  }
}

__global__ void k_hs_fill(float *__restrict__ p, size_t n, float v) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__global__ void k_hs_state_init(HsState *st, int batch, int reset_maps) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  HsState &s = st[b];
  // HectorSlamProcessor::reset (:111-116)
  s.last_update_pose[0] = s.last_update_pose[1] = s.last_update_pose[2] = 3.402823466e+38F;
  s.last_match_pose[0] = s.last_match_pose[1] = s.last_match_pose[2] = 0.0f;
  s.do_update = 0;
  if (reset_maps == 2) {  // create
    for (int q = 0; q < 9; q++) s.last_cov[q] = 0.0f;
    for (int l = 0; l < HS_L; l++) { s.curr_update_index[l] = 0; s.epoch[l] = 0; s.n_pts[l] = 0; s.origo[l][0] = s.origo[l][1] = 0.0f; }
    s.visits = s.n_matched = s.n_updated = 0;
    s.t_match_ns = s.t_update_ns = 0;
    for (int l = 0; l < HS_L; l++) { s.bb_x0[l] = s.bb_y0[l] = 0; s.bb_x1[l] = s.bb_y1[l] = -1; }
  }
}

__global__ void k_hs_epoch_reset(HsState *st, int batch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  for (int l = 0; l < HS_L; l++) st[b].epoch[l] = 0;
}

__global__ void k_hs_ros(const float *__restrict__ lo, int n, int8_t *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = lo[i];
  out[i] = v < 0.0f ? 0 : (v > 0.0f ? 100 : -1);  // HectorMappingRos::publishMap (hector_slam.cc:254-317)
}

static float hs_prob_to_log_odds(float prob) {  // GridMapLogOdds.h:153-157
  float odds = prob / (1.0f - prob);
  return (float)log((double)odds);
}

}  // namespace b2s

struct b2s_hector_slam {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int levels = 0, batch = 1, cap = 0;
  int sx[HS_L] = {}, sy[HS_L] = {};
  float cell_length[HS_L] = {};
  HsBatch P;
  void *allocs[HS_L * 6 + 8] = {};
  int n_allocs = 0;
  HsState *d_state = nullptr;
  float *d_out = nullptr;        // [batch][16] (per-scan / batch calls)
  float *h_out = nullptr;        // pinned [batch][16]
  float *h_pts = nullptr;        // host-mapped pinned staging of one scan (single-processor call)
  float *h_pts_dev = nullptr;    // its device alias
  volatile float *h_mail = nullptr;  // host-mapped mailbox [16]
  float *h_mail_dev = nullptr;
  float *h_hint = nullptr, *h_hint_dev = nullptr;  // host-mapped [3] pose hint of the per-scan call
  unsigned int seq = 0;
  unsigned int *d_barrier = nullptr;
  unsigned long long host_updates = 0;  // upper bound of every level's device epoch
  int stream_ctas = HS_STREAM_CTAS;
  bool coop = true;
  unsigned int launch_tag = 0;  // id of the last stream launch (the kernel publishes per-scan verdicts under it)
  int cluster = 1;  // CTAs per thread-block cluster of the fast-mode stream kernel (1: no cluster launch)
  cudaEvent_t ev_done = nullptr;
  bool launch_pending = false;  // a per-scan launch may still be running its update passes
};

static void hs_free_all(b2s_hector_slam *p) {
  for (int i = 0; i < p->n_allocs; i++)
    if (p->allocs[i]) cudaFree(p->allocs[i]);
  p->n_allocs = 0;
  if (p->d_state) cudaFree(p->d_state);
  if (p->d_out) cudaFree(p->d_out);
  if (p->d_barrier) cudaFree(p->d_barrier);
  if (p->h_out) cudaFreeHost(p->h_out);
  if (p->h_pts) cudaFreeHost(p->h_pts);
  if (p->h_mail) cudaFreeHost(const_cast<float *>(p->h_mail));
  if (p->h_hint) cudaFreeHost(p->h_hint);
  if (p->ev_done) cudaEventDestroy(p->ev_done);
}

extern "C" void b2s_hector_slam_destroy(b2s_hector_slam *p);

static b2s_status hs_clear_maps(b2s_hector_slam *p) {  // GridMapBase::reset -> clear(): resetGridCell on every cell (:93-113)
  for (int l = 0; l < p->levels; l++) {
    const HsLevel &m = p->P.l[l];
    const size_t cells = (size_t)m.sx * m.sy * p->batch;
    B2S_CUDA_CHECK(cudaMemsetAsync(m.lo, 0, cells * 4, p->stream));       // logOdds 0
    B2S_CUDA_CHECK(cudaMemsetAsync(m.ui, 0xff, cells * 4, p->stream));    // updateIndex -1
    B2S_CUDA_CHECK(cudaMemsetAsync(m.free_st, 0, cells * 4, p->stream));
    B2S_CUDA_CHECK(cudaMemsetAsync(m.occ_st, 0, cells * 4, p->stream));
    k_hs_fill<<<ceil_div((long long)cells * 4, 256), 256, 0, p->stream>>>(reinterpret_cast<float *>(m.quad), cells * 4, 0.5f);  // e^0 / (e^0 + 1)
  }
  B2S_CUDA_CHECK(cudaGetLastError());
  return B2S_OK;
}

// stamps carry a 20-bit epoch: before any level's epoch could overflow, clear the stamps and restart the epochs.
// host_updates counts calls (>= every device epoch), so the test needs no device read-back.
static b2s_status hs_reserve_epochs(b2s_hector_slam *p, unsigned long long n_updates) {
  if (p->host_updates + n_updates < HS_EPOCH_MAX) {
    p->host_updates += n_updates;
    return B2S_OK;
  }
  if (n_updates >= HS_EPOCH_MAX) B2S_FAIL(B2S_ERR_TOO_LARGE, "too many scans in one call (stamp epochs are 20 bits)");
  for (int l = 0; l < p->levels; l++) {
    const HsLevel &m = p->P.l[l];
    const size_t cells = (size_t)m.sx * m.sy * p->batch;
    B2S_CUDA_CHECK(cudaMemsetAsync(m.free_st, 0, cells * 4, p->stream));
    B2S_CUDA_CHECK(cudaMemsetAsync(m.occ_st, 0, cells * 4, p->stream));
  }
  k_hs_epoch_reset<<<ceil_div(p->batch, 128), 128, 0, p->stream>>>(p->d_state, p->batch);
  B2S_CUDA_CHECK(cudaGetLastError());
  p->host_updates = n_updates;
  return B2S_OK;
}

static b2s_status hs_create(float map_resolution, int map_size_x, int map_size_y, float start_x, float start_y, int levels,
                            int batch, int max_points, int device, void *cuda_stream, b2s_hector_slam **out) {
  if (!out || levels < 1 || levels > B2S_HECTOR_MAX_LEVELS || !(map_resolution > 0.0f) || (map_size_x >> (levels - 1)) <= 2 ||
      (map_size_y >> (levels - 1)) <= 2 || batch < 1 || max_points < 1)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_hector_slam_create: bad levels / size / resolution / batch");
  *out = nullptr;
  if (max_points > HS_MAX_PTS) B2S_FAIL(B2S_ERR_TOO_LARGE, "at most 4096 points per scan");
  if (b2s_device_count() <= device) B2S_FAIL(B2S_ERR_NO_DEVICE, "no usable CUDA device (the product path has no CPU fallback)");
  B2S_CUDA_CHECK(cudaSetDevice(device));
  keep_pool_memory(device);
  b2s_hector_slam *p = new (std::nothrow) b2s_hector_slam();
  if (!p) B2S_FAIL(B2S_ERR_CUDA, "out of host memory");
  p->device = device;
  p->levels = levels;
  p->batch = batch;
  p->cap = max_points;
#define HS_CHECK(expr) B2S_CUDA_CHECK_CLEAN(b2s_hector_slam_destroy(p), expr)
  if (cuda_stream) {
    p->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  } else {
    HS_CHECK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    p->own_stream = true;
  }
  std::memset(&p->P, 0, sizeof(p->P));
  p->P.levels = levels; p->P.batch = batch; p->P.cap = max_points;
  p->P.lo_free = hs_prob_to_log_odds(0.4f);  // GridMapLogOdds.h:98-102
  p->P.lo_occ = hs_prob_to_log_odds(0.6f);
  p->P.min_dist = 0.4f; p->P.min_angle = 0.13f;  // HectorSlamProcessor.h:63-64
  p->P.exact = 1;
  const int variant = glibc_sincosf_variant_of_host();
  p->P.use_fma = variant == 0 ? 0 : 1;
  // MapRepMultiMap ctor (MapRepMultiMap.h:56-89): one offset for every level, dims halve, cell length doubles
  const float total_x = map_resolution * static_cast<float>(map_size_x), total_y = map_resolution * static_cast<float>(map_size_y);
  const float off_x = total_x * start_x, off_y = total_y * start_y;
  int sx = map_size_x, sy = map_size_y;
  float res = map_resolution;
  for (int l = 0; l < levels; l++) {
    HsLevel &m = p->P.l[l];
    m.sx = sx; m.sy = sy;
    p->sx[l] = sx; p->sy[l] = sy; p->cell_length[l] = res;
    // GridMapBase::setMapTransformation (GridMapBase.h:270-286): AlignedScaling2f(s,s) * Translation2f(off)
    const float scale_to_map = 1.0f / res;
    m.tw_lin = scale_to_map;
    m.tw_tx = scale_to_map * off_x; m.tw_ty = scale_to_map * off_y;
    const float det = m.tw_lin * m.tw_lin - 0.0f * 0.0f, invdet = 1.0f / det, i01 = -0.0f * invdet;  // Affine inverse, cofactor form
    m.wt_lin = m.tw_lin * invdet;
    m.wt_tx = -(m.wt_lin * m.tw_tx + i01 * m.tw_ty);
    m.wt_ty = -(i01 * m.tw_tx + m.wt_lin * m.tw_ty);
    m.iterations = 1 + (l == 0 ? 5 : 3);
    const size_t cells = (size_t)sx * sy * batch;
    void **slots[4] = {(void **)&m.lo, (void **)&m.ui, (void **)&m.free_st, (void **)&m.occ_st};
    for (void **s : slots) {
      HS_CHECK(cudaMalloc(s, cells * 4));
      p->allocs[p->n_allocs++] = *s;
    }
    HS_CHECK(cudaMalloc(reinterpret_cast<void **>(&m.quad), cells * 16));
    p->allocs[p->n_allocs++] = m.quad;
    HS_CHECK(cudaMalloc(reinterpret_cast<void **>(&m.pts), sizeof(float) * 2 * (size_t)max_points * batch));
    p->allocs[p->n_allocs++] = m.pts;
    sx /= 2; sy /= 2;
    res *= 2.0f;
  }
  HS_CHECK(cudaMalloc(reinterpret_cast<void **>(&p->d_state), sizeof(HsState) * (size_t)batch));
  p->P.state = p->d_state;
  HS_CHECK(cudaMalloc(reinterpret_cast<void **>(&p->d_out), sizeof(float) * 16 * (size_t)batch));
  HS_CHECK(cudaMalloc(reinterpret_cast<void **>(&p->d_barrier), sizeof(unsigned int)));
  HS_CHECK(cudaMallocHost(reinterpret_cast<void **>(&p->h_out), sizeof(float) * 16 * (size_t)batch));
  HS_CHECK(cudaHostAlloc(reinterpret_cast<void **>(&p->h_pts), sizeof(float) * 2 * (size_t)max_points, cudaHostAllocMapped));
  HS_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void **>(&p->h_pts_dev), p->h_pts, 0));
  {
    float *mail = nullptr;
    HS_CHECK(cudaHostAlloc(reinterpret_cast<void **>(&mail), sizeof(float) * 16, cudaHostAllocMapped));
    std::memset(mail, 0, sizeof(float) * 16);
    p->h_mail = mail;
    HS_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void **>(&p->h_mail_dev), mail, 0));
  }
  HS_CHECK(cudaHostAlloc(reinterpret_cast<void **>(&p->h_hint), sizeof(float) * 4, cudaHostAllocMapped));
  HS_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void **>(&p->h_hint_dev), p->h_hint, 0));
  HS_CHECK(cudaEventCreateWithFlags(&p->ev_done, cudaEventDisableTiming));
  const size_t smem = hs_smem_bytes(max_points);
  HS_CHECK(raise_dyn_smem(k_hs_match<true>, smem));
  HS_CHECK(raise_dyn_smem(k_hs_match<false>, smem));
  HS_CHECK(raise_dyn_smem(k_hs_stream<true, false>, smem));
  HS_CHECK(raise_dyn_smem(k_hs_stream<false, false>, smem));
  HS_CHECK(raise_dyn_smem(k_hs_stream<false, true>, smem));
  {
    int coop = 0, sms = 0, per_sm = 0;
    HS_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
    HS_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    HS_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_hs_stream<true, false>, HS_THREADS, smem));
    p->coop = coop != 0;
    p->stream_ctas = std::max(1, std::min(HS_STREAM_CTAS, sms * std::max(per_sm, 0)));
    if (!p->coop) p->stream_ctas = 1;  // without a co-residency guarantee a spinning grid barrier could deadlock
    // fast mode: the matching CTA's cluster.  Needs the whole cooperative grid co-resident AS clusters.
    if (p->coop && p->stream_ctas >= HS_CLUSTER) {
      cudaLaunchConfig_t cfg;
      std::memset(&cfg, 0, sizeof(cfg));
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = (unsigned)HS_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.gridDim = dim3((p->stream_ctas / HS_CLUSTER) * HS_CLUSTER);
      cfg.blockDim = dim3(HS_THREADS);
      cfg.dynamicSmemBytes = smem;
      cfg.attrs = at; cfg.numAttrs = 1;
      int n_clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&n_clusters, k_hs_stream<false, true>, &cfg) == cudaSuccess &&
          n_clusters * HS_CLUSTER >= (int)cfg.gridDim.x)
        p->cluster = HS_CLUSTER;
      else
        cudaGetLastError();
    }
  }
  k_hs_state_init<<<ceil_div(batch, 128), 128, 0, p->stream>>>(p->d_state, batch, 2);
  {
    b2s_status st = hs_clear_maps(p);
    if (st) { b2s_hector_slam_destroy(p); return st; }
  }
  HS_CHECK(cudaGetLastError());
  HS_CHECK(cudaStreamSynchronize(p->stream));
#undef HS_CHECK
  *out = p;
  return B2S_OK;
}

// wait until the previous per-scan launch (its update passes) has left the host-mapped staging buffers alone
static b2s_status hs_wait_launch(b2s_hector_slam *p) {
  if (p->launch_pending) {
    B2S_CUDA_CHECK(cudaEventSynchronize(p->ev_done));
    p->launch_pending = false;
  }
  return B2S_OK;
}

static b2s_status hs_launch_stream(b2s_hector_slam *p, const HsStream &S) {
  B2S_CUDA_CHECK(cudaMemsetAsync(p->d_barrier, 0, sizeof(unsigned int), p->stream));
  HsBatch P = p->P;
  HsStream Sv = S;
  Sv.barrier = p->d_barrier;
  p->launch_tag += 1;
  if (p->launch_tag == 0) p->launch_tag = 1;
  Sv.tag = p->launch_tag;
  const size_t smem = hs_smem_bytes(p->cap);
  if (p->coop && !P.exact && p->cluster > 1) {
    // cooperative (all CTAs co-resident for the grid barrier) AND clustered (CTAs [0, cluster) share the match)
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    at[1].id = cudaLaunchAttributeClusterDimension;
    at[1].val.clusterDim.x = (unsigned)p->cluster; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
    cfg.gridDim = dim3((p->stream_ctas / p->cluster) * p->cluster);
    cfg.blockDim = dim3(HS_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = p->stream;
    cfg.attrs = at; cfg.numAttrs = 2;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, k_hs_stream<false, true>, P, Sv);
    if (e == cudaSuccess) return B2S_OK;
    cudaGetLastError();
    p->cluster = 1;  // this driver refuses the combination: the one-CTA match from now on
  }
  if (p->coop) {
    void *args[2] = {&P, &Sv};
    const void *kern = P.exact ? reinterpret_cast<const void *>(k_hs_stream<true, false>) : reinterpret_cast<const void *>(k_hs_stream<false, false>);
    B2S_CUDA_CHECK(cudaLaunchCooperativeKernel(kern, dim3(p->stream_ctas), dim3(HS_THREADS), args, smem, p->stream));
  } else {
    if (P.exact) k_hs_stream<true, false><<<1, HS_THREADS, smem, p->stream>>>(P, Sv);
    else k_hs_stream<false, false><<<1, HS_THREADS, smem, p->stream>>>(P, Sv);
    B2S_CUDA_CHECK(cudaGetLastError());
  }
  return B2S_OK;
}

extern "C" {

b2s_status b2s_hector_slam_create(float map_resolution, int map_size_x, int map_size_y, float start_x, float start_y,
                                  int levels, int device, void *cuda_stream, b2s_hector_slam **out) {
  return hs_create(map_resolution, map_size_x, map_size_y, start_x, start_y, levels, 1, 2048, device, cuda_stream, out);
}

b2s_status b2s_hector_slam_create_batch(int batch, int max_points, float map_resolution, int map_size_x, int map_size_y,
                                        float start_x, float start_y, int levels, int device, void *cuda_stream,
                                        b2s_hector_slam **out) {
  return hs_create(map_resolution, map_size_x, map_size_y, start_x, start_y, levels, batch, max_points, device, cuda_stream, out);
}

void b2s_hector_slam_destroy(b2s_hector_slam *p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->stream) cudaStreamSynchronize(p->stream);
  hs_free_all(p);
  if (p->own_stream && p->stream) cudaStreamDestroy(p->stream);
  delete p;
}

b2s_status b2s_hector_slam_set_update_factors(b2s_hector_slam *p, float update_free, float update_occupied) {
  if (!p) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  p->P.lo_free = hs_prob_to_log_odds(update_free);
  p->P.lo_occ = hs_prob_to_log_odds(update_occupied);
  return B2S_OK;
}

b2s_status b2s_hector_slam_set_map_update_min_diff(b2s_hector_slam *p, float min_dist, float min_angle) {
  if (!p) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  p->P.min_dist = min_dist;
  p->P.min_angle = min_angle;
  return B2S_OK;
}

b2s_status b2s_hector_slam_set_exact(b2s_hector_slam *p, int exact) {
  if (!p) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  p->P.exact = exact ? 1 : 0;
  return B2S_OK;
}

int32_t b2s_hector_slam_match_cluster_size(const b2s_hector_slam *p) { return p ? (int32_t)p->cluster : 0; }

b2s_status b2s_hector_slam_reset(b2s_hector_slam *p) {
  if (!p) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  b2s_status st = hs_wait_launch(p);
  if (st) return st;
  k_hs_state_init<<<ceil_div(p->batch, 128), 128, 0, p->stream>>>(p->d_state, p->batch, 1);
  return hs_clear_maps(p);
}

b2s_status b2s_hector_slam_update(b2s_hector_slam *p, const float *points, int n_points, const float origo[2],
                                  const float pose_hint_world[3], int map_without_matching, float out_pose[3],
                                  float out_cov[9], int *out_map_updated) {
  B2S_NVTX("Hector update (match + gate + map update)");
  if (!p || !origo || !pose_hint_world || !out_pose || n_points < 0 || (n_points > 0 && !points))
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (p->batch != 1) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_hector_slam_update serves single-processor handles; use b2s_hector_slam_update_batch");
  if (n_points > p->cap) B2S_FAIL(B2S_ERR_TOO_LARGE, "more points than the handle's capacity (2048 for b2s_hector_slam_create)");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  b2s_status st = hs_wait_launch(p);  // the previous call's update passes still read nothing of ours, but its kernel reads h_hint / h_pts
  if (st) return st;
  if ((st = hs_reserve_epochs(p, 1))) return st;
  if (n_points > 0) std::memcpy(p->h_pts, points, sizeof(float) * 2 * (size_t)n_points);
  p->h_hint[0] = pose_hint_world[0]; p->h_hint[1] = pose_hint_world[1]; p->h_hint[2] = pose_hint_world[2];
  p->seq += 1;
  if (p->seq == 0) p->seq = 1;
  HsStream S;
  std::memset(&S, 0, sizeof(S));
  S.pts = p->h_pts_dev;        // read over the host link by the matching CTA (8.6 KB for 1081 beams)
  S.count0 = n_points;
  S.n_scans = 1;
  S.first_hint = p->h_hint_dev;
  S.origo_x = origo[0]; S.origo_y = origo[1];
  S.map_without_matching = map_without_matching;
  S.out = p->d_out;
  S.mailbox = p->h_mail_dev;
  S.seq = p->seq;
  if ((st = hs_launch_stream(p, S))) return st;
  B2S_CUDA_CHECK(cudaEventRecord(p->ev_done, p->stream));
  p->launch_pending = true;
  // the pose arrives through the mailbox as soon as the match is done; the update passes keep running
  const volatile unsigned int *flag = reinterpret_cast<const volatile unsigned int *>(p->h_mail) + 15;
  for (unsigned long long spin = 0;; spin++) {
    if (*flag == p->seq) break;
    if ((spin & 0x3fff) == 0x3fff) {
      const cudaError_t q = cudaEventQuery(p->ev_done);
      if (q == cudaSuccess) {
        if (*flag == p->seq) break;
        B2S_FAIL(B2S_ERR_CUDA, "b2s_hector_slam_update: the kernel finished without posting its result");
      }
      if (q != cudaErrorNotReady) B2S_CUDA_CHECK(q);
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  float r[15];
  for (int q = 0; q < 15; q++) r[q] = p->h_mail[q];
  if (r[14] != 0.0f) B2S_FAIL(B2S_ERR_CUDA, "b2s_hector_slam_update: a cluster exchange of the match timed out");
  out_pose[0] = r[0]; out_pose[1] = r[1]; out_pose[2] = r[2];
  if (out_cov && !map_without_matching) std::memcpy(out_cov, r + 3, 9 * sizeof(float));
  if (out_map_updated) *out_map_updated = r[12] != 0.0f ? 1 : 0;
  return B2S_OK;
}

b2s_status b2s_hector_slam_process_stream(b2s_hector_slam *p, int n_scans, const float *points, const int32_t *n_points,
                                          const float origo[2], const float *first_pose_hint, const float *pose_hints,
                                          int map_without_matching, float *out_poses, int32_t *out_map_updated,
                                          float *out_last_cov) {
  B2S_NVTX("Hector stream");
  if (!p || n_scans < 0 || !origo || !out_poses || (n_scans > 0 && (!points || !n_points)))
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (map_without_matching && !pose_hints) B2S_FAIL(B2S_ERR_BAD_PARAMS, "map_without_matching needs a pose per scan (pose_hints)");
  if (p->batch != 1) B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_hector_slam_process_stream serves single-processor handles");
  if (n_scans == 0) return B2S_OK;
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  b2s_status st = hs_wait_launch(p);
  if (st) return st;
  std::vector<int> offs((size_t)n_scans);
  long long total = 0;
  for (int i = 0; i < n_scans; i++) {
    if (n_points[i] < 0 || n_points[i] > p->cap) B2S_FAIL(B2S_ERR_TOO_LARGE, "a scan has more points than the handle's capacity");
    offs[i] = (int)total;
    total += n_points[i];
    if (total > 0x7fffffffLL / 2) B2S_FAIL(B2S_ERR_TOO_LARGE, "stream too long for one call");
  }
  if ((st = hs_reserve_epochs(p, (unsigned long long)n_scans))) return st;
  float *d_pts = nullptr, *d_hints = nullptr, *d_first = nullptr, *d_out = nullptr;
  int *d_offs = nullptr, *d_cnt = nullptr;
  auto release = [&]() {
    for (void *q : {(void *)d_pts, (void *)d_hints, (void *)d_first, (void *)d_out, (void *)d_offs, (void *)d_cnt})
      if (q) cudaFreeAsync(q, p->stream);
    cudaStreamSynchronize(p->stream);
  };
#define HS_CHECK(expr) B2S_CUDA_CHECK_CLEAN(release(), expr)
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_pts), sizeof(float) * 2 * (size_t)std::max<long long>(total, 1), p->stream));
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_out), sizeof(float) * 16 * (size_t)n_scans, p->stream));
  HS_CHECK(cudaMemsetAsync(d_out, 0, sizeof(float) * 16 * (size_t)n_scans, p->stream));  // no stale verdict tags
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_offs), sizeof(int) * (size_t)n_scans, p->stream));
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_cnt), sizeof(int) * (size_t)n_scans, p->stream));
  if (total > 0) HS_CHECK(cudaMemcpyAsync(d_pts, points, sizeof(float) * 2 * (size_t)total, cudaMemcpyHostToDevice, p->stream));
  HS_CHECK(cudaMemcpyAsync(d_offs, offs.data(), sizeof(int) * (size_t)n_scans, cudaMemcpyHostToDevice, p->stream));
  HS_CHECK(cudaMemcpyAsync(d_cnt, n_points, sizeof(int) * (size_t)n_scans, cudaMemcpyHostToDevice, p->stream));
  if (pose_hints) {
    HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_hints), sizeof(float) * 3 * (size_t)n_scans, p->stream));
    HS_CHECK(cudaMemcpyAsync(d_hints, pose_hints, sizeof(float) * 3 * (size_t)n_scans, cudaMemcpyHostToDevice, p->stream));
  } else if (first_pose_hint) {
    HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_first), sizeof(float) * 3, p->stream));
    HS_CHECK(cudaMemcpyAsync(d_first, first_pose_hint, sizeof(float) * 3, cudaMemcpyHostToDevice, p->stream));
  }
  HsStream S;
  std::memset(&S, 0, sizeof(S));
  S.pts = d_pts; S.offsets = d_offs; S.counts = d_cnt; S.n_scans = n_scans;
  S.hints = d_hints; S.first_hint = d_first;
  S.origo_x = origo[0]; S.origo_y = origo[1];
  S.map_without_matching = map_without_matching;
  S.out = d_out;
  if ((st = hs_launch_stream(p, S))) { release(); return st; }
  std::vector<float> host((size_t)n_scans * 16);
  HS_CHECK(cudaMemcpyAsync(host.data(), d_out, sizeof(float) * 16 * (size_t)n_scans, cudaMemcpyDeviceToHost, p->stream));
  HS_CHECK(cudaStreamSynchronize(p->stream));
#undef HS_CHECK
  release();
  for (int i = 0; i < n_scans; i++) {
    if (host[16 * (size_t)i + 14] != 0.0f) B2S_FAIL(B2S_ERR_CUDA, "b2s_hector_slam_process_stream: a cluster exchange of the match timed out");
    std::memcpy(out_poses + 3 * (size_t)i, host.data() + 16 * (size_t)i, 3 * sizeof(float));
    if (out_map_updated) out_map_updated[i] = host[16 * (size_t)i + 12] != 0.0f ? 1 : 0;
  }
  if (out_last_cov && !map_without_matching) std::memcpy(out_last_cov, host.data() + 16 * (size_t)(n_scans - 1) + 3, 9 * sizeof(float));
  return B2S_OK;
}

b2s_status b2s_hector_slam_update_batch(b2s_hector_slam *p, const float *points, const int32_t *n_points, const float origo[2],
                                        const float *pose_hints, int map_without_matching, float *out_poses, float *out_covs,
                                        int32_t *out_map_updated) {
  if (!p || !points || !n_points || !origo || !out_poses) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (map_without_matching && !pose_hints) B2S_FAIL(B2S_ERR_BAD_PARAMS, "map_without_matching needs the poses (pose_hints)");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  b2s_status st = hs_wait_launch(p);
  if (st) return st;
  const int B = p->batch;
  for (int b = 0; b < B; b++)
    if (n_points[b] < 0 || n_points[b] > p->cap) B2S_FAIL(B2S_ERR_TOO_LARGE, "a scan has more points than the handle's capacity");
  if ((st = hs_reserve_epochs(p, 1))) return st;
  float *d_pts = nullptr, *d_hints = nullptr;
  int *d_cnt = nullptr;
  auto release = [&]() {
    for (void *q : {(void *)d_pts, (void *)d_hints, (void *)d_cnt})
      if (q) cudaFreeAsync(q, p->stream);
  };
#define HS_CHECK(expr) B2S_CUDA_CHECK_CLEAN((release(), cudaStreamSynchronize(p->stream)), expr)
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_pts), sizeof(float) * 2 * (size_t)p->cap * B, p->stream));
  HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_cnt), sizeof(int) * (size_t)B, p->stream));
  HS_CHECK(cudaMemcpyAsync(d_pts, points, sizeof(float) * 2 * (size_t)p->cap * B, cudaMemcpyHostToDevice, p->stream));
  HS_CHECK(cudaMemcpyAsync(d_cnt, n_points, sizeof(int) * (size_t)B, cudaMemcpyHostToDevice, p->stream));
  if (pose_hints) {
    HS_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d_hints), sizeof(float) * 3 * (size_t)B, p->stream));
    HS_CHECK(cudaMemcpyAsync(d_hints, pose_hints, sizeof(float) * 3 * (size_t)B, cudaMemcpyHostToDevice, p->stream));
  }
  HsCall C;
  std::memset(&C, 0, sizeof(C));
  C.pts0 = d_pts; C.n0 = d_cnt; C.pts_stride = p->cap;
  C.hints = d_hints;
  C.origo_x = origo[0]; C.origo_y = origo[1];
  C.map_without_matching = map_without_matching;
  C.out = p->d_out;
  int max_n = 0;
  for (int b = 0; b < B; b++) max_n = std::max(max_n, n_points[b]);
  if (p->P.exact) k_hs_match<true><<<B, HS_THREADS, hs_smem_bytes(p->cap), p->stream>>>(p->P, C);
  else k_hs_match<false><<<B, HS_THREADS, hs_smem_bytes(p->cap), p->stream>>>(p->P, C);
  // data containers of the coarse levels may hold more points than this step's scans (map_without_matching): size the
  // update grid by the capacity bound
  const dim3 grid(std::max(1, std::min(ceil_div(std::max(max_n, 1) * p->levels, 8), 148 * 8 / std::max(1, std::min(B, 8)))), B);
  k_hs_mark<<<grid, 256, 0, p->stream>>>(p->P);
  k_hs_apply<<<grid, 256, 0, p->stream>>>(p->P);
  HS_CHECK(cudaGetLastError());
  HS_CHECK(cudaMemcpyAsync(p->h_out, p->d_out, sizeof(float) * 16 * (size_t)B, cudaMemcpyDeviceToHost, p->stream));
  release();
  HS_CHECK(cudaStreamSynchronize(p->stream));
#undef HS_CHECK
  for (int b = 0; b < B; b++) {
    std::memcpy(out_poses + 3 * (size_t)b, p->h_out + 16 * (size_t)b, 3 * sizeof(float));
    if (out_covs && !map_without_matching) std::memcpy(out_covs + 9 * (size_t)b, p->h_out + 16 * (size_t)b + 3, 9 * sizeof(float));
    if (out_map_updated) out_map_updated[b] = p->h_out[16 * (size_t)b + 12] != 0.0f ? 1 : 0;
  }
  return B2S_OK;
}

/* the same step with the scans ALREADY on the device (device pointers; nothing is copied, nothing is returned to the
 * host): the resident-in-HBM form the throughput of the batched update is measured on */
b2s_status b2s_hector_slam_update_batch_device(b2s_hector_slam *p, const float *d_points, const int32_t *d_n_points, int max_n,
                                               const float origo[2], const float *d_pose_hints, int map_without_matching) {
  B2S_NVTX("Hector batch step");
  if (!p || !d_points || !d_n_points || !origo) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  if (map_without_matching && !d_pose_hints) B2S_FAIL(B2S_ERR_BAD_PARAMS, "map_without_matching needs the poses");
  if (max_n < 0 || max_n > p->cap) B2S_FAIL(B2S_ERR_TOO_LARGE, "more points than the handle's capacity");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  b2s_status st = hs_wait_launch(p);
  if (st) return st;
  if ((st = hs_reserve_epochs(p, 1))) return st;
  const int B = p->batch;
  HsCall C;
  std::memset(&C, 0, sizeof(C));
  C.pts0 = d_points; C.n0 = d_n_points; C.pts_stride = p->cap;
  C.hints = d_pose_hints;
  C.origo_x = origo[0]; C.origo_y = origo[1];
  C.map_without_matching = map_without_matching;
  C.out = p->d_out;
  if (p->P.exact) k_hs_match<true><<<B, HS_THREADS, hs_smem_bytes(p->cap), p->stream>>>(p->P, C);
  else k_hs_match<false><<<B, HS_THREADS, hs_smem_bytes(p->cap), p->stream>>>(p->P, C);
  const dim3 grid(std::max(1, std::min(ceil_div(std::max(max_n, 1) * p->levels, 8), 148 * 8 / std::max(1, std::min(B, 8)))), B);
  k_hs_mark<<<grid, 256, 0, p->stream>>>(p->P);
  k_hs_apply<<<grid, 256, 0, p->stream>>>(p->P);
  B2S_CUDA_CHECK(cudaGetLastError());
  return B2S_OK;
}

b2s_status b2s_hector_slam_sync(b2s_hector_slam *p) {
  if (!p) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  B2S_CUDA_CHECK(cudaStreamSynchronize(p->stream));
  p->launch_pending = false;
  return B2S_OK;
}

b2s_status b2s_hector_slam_level_dims(b2s_hector_slam *p, int level, int dims[2], float *cell_length) {
  if (!p || !dims || level < 0 || level >= p->levels) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad level");
  dims[0] = p->sx[level];
  dims[1] = p->sy[level];
  if (cell_length) *cell_length = p->cell_length[level];
  return B2S_OK;
}

b2s_status b2s_hector_slam_copy_level_of(b2s_hector_slam *p, int b, int level, float *log_odds, int32_t *update_index) {
  if (!p || level < 0 || level >= p->levels || b < 0 || b >= p->batch) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad level / processor");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  const HsLevel &m = p->P.l[level];
  const size_t cells = (size_t)m.sx * m.sy;
  if (log_odds) B2S_CUDA_CHECK(cudaMemcpyAsync(log_odds, m.lo + (size_t)b * cells, cells * 4, cudaMemcpyDeviceToHost, p->stream));
  if (update_index) B2S_CUDA_CHECK(cudaMemcpyAsync(update_index, m.ui + (size_t)b * cells, cells * 4, cudaMemcpyDeviceToHost, p->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(p->stream));
  p->launch_pending = false;
  return B2S_OK;
}

b2s_status b2s_hector_slam_copy_level(b2s_hector_slam *p, int level, float *log_odds, int32_t *update_index) {
  return b2s_hector_slam_copy_level_of(p, 0, level, log_odds, update_index);
}

b2s_status b2s_hector_slam_copy_level_ros(b2s_hector_slam *p, int level, int8_t *out) {
  if (!p || !out || level < 0 || level >= p->levels) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad level");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  const HsLevel &m = p->P.l[level];
  const int n = m.sx * m.sy;
  int8_t *d = nullptr;
  B2S_CUDA_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&d), (size_t)n, p->stream));
  k_hs_ros<<<ceil_div(n, 256), 256, 0, p->stream>>>(m.lo, n, d);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, d, (size_t)n, cudaMemcpyDeviceToHost, p->stream);
  cudaFreeAsync(d, p->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
  B2S_CUDA_CHECK(e);
  p->launch_pending = false;
  return B2S_OK;
}

b2s_status b2s_hector_slam_stats(b2s_hector_slam *p, double out[5]) {
  if (!p || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  std::vector<HsState> s((size_t)p->batch);
  B2S_CUDA_CHECK(cudaMemcpyAsync(s.data(), p->d_state, sizeof(HsState) * (size_t)p->batch, cudaMemcpyDeviceToHost, p->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(p->stream));
  p->launch_pending = false;
  out[0] = out[1] = out[2] = 0.0;
  for (const HsState &x : s) { out[0] += (double)x.n_matched; out[1] += (double)x.n_updated; out[2] += (double)x.visits; }
  out[3] = (double)s[0].t_match_ns * 1e-6;   // ms of processor 0's last match / update (device %globaltimer)
  out[4] = (double)s[0].t_update_ns * 1e-6;
  return B2S_OK;
}

/* the processor's own last poses (getLastScanMatchPose / getLastMapUpdatePose, HectorSlamProcessor.h:118-119) */
b2s_status b2s_hector_slam_last_poses(b2s_hector_slam *p, int b, float last_scan_match_pose[3], float last_map_update_pose[3]) {
  if (!p || b < 0 || b >= p->batch) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad processor");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  HsState s;
  B2S_CUDA_CHECK(cudaMemcpyAsync(&s, p->d_state + b, sizeof(HsState), cudaMemcpyDeviceToHost, p->stream));
  B2S_CUDA_CHECK(cudaStreamSynchronize(p->stream));
  p->launch_pending = false;
  if (last_scan_match_pose) std::memcpy(last_scan_match_pose, s.last_match_pose, 3 * sizeof(float));
  if (last_map_update_pose) std::memcpy(last_map_update_pose, s.last_update_pose, 3 * sizeof(float));
  return B2S_OK;
}

/* test hook: pretend `updates` map updates have already consumed stamp epochs (exercises the 20-bit epoch wrap) */
b2s_status b2s_hector_slam_debug_set_epoch(b2s_hector_slam *p, unsigned int updates) {
  if (!p || updates >= HS_EPOCH_MAX) B2S_FAIL(B2S_ERR_BAD_PARAMS, "bad epoch");
  B2S_CUDA_CHECK(cudaSetDevice(p->device));
  B2S_CUDA_CHECK(cudaStreamSynchronize(p->stream));
  std::vector<HsState> s((size_t)p->batch);
  B2S_CUDA_CHECK(cudaMemcpy(s.data(), p->d_state, sizeof(HsState) * (size_t)p->batch, cudaMemcpyDeviceToHost));
  unsigned int have = 0;
  for (const HsState &x : s)
    for (int l = 0; l < p->levels; l++) have = std::max(have, x.epoch[l]);
  if (updates < have) B2S_FAIL(B2S_ERR_BAD_PARAMS, "epochs only move forward");
  for (HsState &x : s)
    for (int l = 0; l < p->levels; l++) x.epoch[l] = updates;
  B2S_CUDA_CHECK(cudaMemcpy(p->d_state, s.data(), sizeof(HsState) * (size_t)p->batch, cudaMemcpyHostToDevice));
  p->host_updates = updates;
  return B2S_OK;
}

}  // extern "C"

// lesson6 front end on top of K1 — the host driver of karto::Mapper / MapperGraph / MapperSensorManager (host C++).
// Product code.  It decides WHAT to match (key frames, running window, near chains, loop-closure candidates) and keeps
// the pose graph; every ScanMatcher::MatchScan runs on the device through the matcher ABI of this library, and the
// independent matches of one Process call are sent as one batch.
//
// Reference behaviour (paths relative to /root/reference/lesson6/lib/open_karto):
//   Mapper::Process / HasMovedEnough / Initialize                          src/Mapper.cpp:1959-2125
//   MapperGraph::{AddVertex, AddEdges, TryCloseLoop, GetClosestScanToPose, AddEdge, LinkScans, LinkNearChains,
//                 LinkChainToScan, FindNearChains, FindNearLinkedScans, ComputeWeightedMean,
//                 FindPossibleLoopClosure, CorrectPoses}                   src/Mapper.cpp:862-1414
//   ScanManager / MapperSensorManager (running-scan window)                include/open_karto/Mapper.h:1288-1404
//   LinkInfo, Vertex, Edge, BreadthFirstTraversal, NearScanVisitor         include/open_karto/Mapper.h:108-643
//   LocalizedRangeScan::{Update, SetSensorPose, GetReferencePose}          include/open_karto/Karto.h:5243-5428
//   Transform, Matrix3, Pose2                                              include/open_karto/Karto.h:2085-2160, 2392-2600, 2853-2944
// All pose arithmetic is double precision in the reference's operation order, so poses, link means and covariances agree
// with the reference to the matcher's own tolerance (1e-9 in the parity tests) and every threshold decision is the same.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <deque>
#include <list>
#include <new>
#include <queue>
#include <string>
#include <vector>

#include "common.cuh"

using namespace b2s;

namespace {

struct P3 {
  double x = 0, y = 0, h = 0;
};
inline P3 p3(const double v[3]) { return P3{v[0], v[1], v[2]}; }
inline double sqdist(const P3 &a, const P3 &b) {  // Vector2::SquaredDistance -> (a - b).SquaredLength()
  const double dx = a.x - b.x, dy = a.y - b.y;
  return dx * dx + dy * dy;
}
inline double sq(double v) { return v * v; }  // math::Square

struct M3 {
  double m[3][3];
  M3() { std::memset(m, 0, sizeof(m)); }  // Matrix3(): Clear()
  static M3 identity() {
    M3 r;
    r.m[0][0] = r.m[1][1] = r.m[2][2] = 1.0;
    return r;
  }
  static M3 axis_z(double radians) {  // FromAxisAngle(0, 0, 1, radians) (Karto.h:2392-2421)
    const double c = cos(radians), s = sin(radians), omc = 1.0 - c;
    const double x = 0, y = 0, z = 1;
    const double xyM = x * y * omc, xzM = x * z * omc, yzM = y * z * omc, xS = x * s, yS = y * s, zS = z * s;
    M3 r;
    r.m[0][0] = x * x * omc + c; r.m[0][1] = xyM - zS; r.m[0][2] = xzM + yS;
    r.m[1][0] = xyM + zS; r.m[1][1] = y * y * omc + c; r.m[1][2] = yzM - xS;
    r.m[2][0] = xzM - yS; r.m[2][1] = yzM + xS; r.m[2][2] = z * z * omc + c;
    return r;
  }
  M3 operator*(const M3 &o) const {  // Karto.h:2544-2556
    M3 r;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) r.m[i][j] = m[i][0] * o.m[0][j] + m[i][1] * o.m[1][j] + m[i][2] * o.m[2][j];
    return r;
  }
  P3 operator*(const P3 &p) const {  // Karto.h:2557-2564
    P3 r;
    r.x = m[0][0] * p.x + m[0][1] * p.y + m[0][2] * p.h;
    r.y = m[1][0] * p.x + m[1][1] * p.y + m[1][2] * p.h;
    r.h = m[2][0] * p.x + m[2][1] * p.y + m[2][2] * p.h;
    return r;
  }
  M3 transpose() const {
    M3 r;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) r.m[i][j] = m[j][i];
    return r;
  }
  void add(const M3 &o) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) m[i][j] += o.m[i][j];
  }
  bool inverse(M3 &k) const {  // Inverse() -> InverseFast(k, 1e-14) (Karto.h:2445-2493)
    k.m[0][0] = m[1][1] * m[2][2] - m[1][2] * m[2][1];
    k.m[0][1] = m[0][2] * m[2][1] - m[0][1] * m[2][2];
    k.m[0][2] = m[0][1] * m[1][2] - m[0][2] * m[1][1];
    k.m[1][0] = m[1][2] * m[2][0] - m[1][0] * m[2][2];
    k.m[1][1] = m[0][0] * m[2][2] - m[0][2] * m[2][0];
    k.m[1][2] = m[0][2] * m[1][0] - m[0][0] * m[1][2];
    k.m[2][0] = m[1][0] * m[2][1] - m[1][1] * m[2][0];
    k.m[2][1] = m[0][1] * m[2][0] - m[0][0] * m[2][1];
    k.m[2][2] = m[0][0] * m[1][1] - m[0][1] * m[1][0];
    const double det = m[0][0] * k.m[0][0] + m[0][1] * k.m[1][0] + m[0][2] * k.m[2][0];
    if (fabs(det) <= 1e-14) return false;
    const double inv = 1.0 / det;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) k.m[i][j] *= inv;
    return true;
  }
};

struct Xform {  // karto::Transform (Karto.h:2853-2944)
  P3 t;
  M3 rot;
  Xform(const P3 &a, const P3 &b) {
    if (a.x == b.x && a.y == b.y && a.h == b.h) {
      rot = M3::identity();
      t = P3();
      return;
    }
    rot = M3::axis_z(b.h - a.h);
    P3 np;
    if (a.x != 0.0 || a.y != 0.0) {
      const P3 ra = rot * a;  // rPose2 - m_Rotation * rPose1 (Pose2 operator-)
      np.x = b.x - ra.x;
      np.y = b.y - ra.y;
    } else {
      np = b;
    }
    t.x = np.x; t.y = np.y; t.h = b.h - a.h;
  }
  P3 apply(const P3 &s) const {  // TransformPose
    const P3 r = rot * s;
    P3 o;
    o.x = t.x + r.x;
    o.y = t.y + r.y;
    o.h = normalize_angle(s.h + t.h);
    return o;
  }
};

struct MScan {
  std::vector<double> ranges;
  P3 odom, corrected, sensor, bary;
  double time = 0;
  int id = -1;      // unique id (MapperSensorManager::m_NextScanId): index into b2s_mapper::scans
  int dev = 0;      // index into b2s_mapper::sensors
  int state = -1;   // state id: index into that sensor's scan list (ScanManager::AddScan, Mapper.h:1290-1303)
  std::vector<int> edges;  // Vertex::m_Edges: indices into Mapper::edges, in insertion order
};

struct MEdge {
  int src, dst;
  P3 pose1, pose2, diff;
  M3 cov;
};

struct SensorState {  // one ScanManager (Mapper.h:1265-1410): the scans, running window and last scan of one sensor
  std::string name;
  std::vector<int> ids;      // ScanManager::m_Scans as unique ids, indexed by state id
  std::vector<int> running;  // ScanManager::m_RunningScans
  int last_scan = -1;        // ScanManager::m_pLastScan
};

struct CudaBackend {  // the two ScanMatcher instances a Mapper owns, as b2s_matcher handles
  int device = 0;
  b2s_laser laser{};
  b2s_matcher_params params[2]{};
  b2s_matcher *h[2] = {nullptr, nullptr};
  int cap_batch[2] = {0, 0}, cap_base[2] = {0, 0};
  int min_base = 32;  // scan_buffer_size + 1: the sequential matcher's base set is the running window
  std::vector<double> base_r, base_p;
  std::vector<int32_t> base_rows;
  size_t pool_n[2] = {0, 0};  // scans of the mapper already appended to each handle's device-resident pool
  ~CudaBackend() {
    for (auto *p : h)
      if (p) b2s_matcher_destroy(p);
  }
};

}  // namespace

struct b2s_mapper {
  bool failed = false;  // a Process call failed after the scan entered the graph: the handle must be discarded
  b2s_mapper_params prm{};
  b2s_laser laser{};
  b2s_match_scan_fn match = nullptr;
  void *match_user = nullptr;
  CudaBackend *cuda = nullptr;
  b2s_scan_solver solver{};
  bool have_solver = false;
  std::deque<MScan> scans;  // MapperSensorManager::m_Scans (every sensor's scans by unique id); deque: stable addresses
  std::vector<MEdge> edges;
  std::vector<SensorState> sensors;  // in registration order
  std::vector<int> by_name;          // sensor indices in the order of std::map<Name, ScanManager*> (Name::operator<, Karto.h:484)
  int last_sensor = 0;
  double n_match_calls = 0, n_batches = 0, n_loop_candidates = 0, n_loops_closed = 0;
};

namespace {

// LocalizedRangeScan::Update (Karto.h:5362-5428): sensor pose and barycenter of the in-range readings
void scan_update(const b2s_mapper *m, MScan &s) {
  const double c[3] = {s.corrected.x, s.corrected.y, s.corrected.h};
  double sp[3];
  sensor_pose_of(c, m->laser.offset_pose, sp);
  s.sensor = p3(sp);
  double sx = 0, sy = 0, n = 0;
  for (int i = 0; i < m->laser.n_readings; i++) {
    const double r = s.ranges[i];
    if (!(r >= m->laser.min_range && r <= m->laser.range_threshold)) continue;  // math::InRange
    const double angle = s.sensor.h + m->laser.min_angle + i * m->laser.angular_resolution;
    sx += s.sensor.x + (r * cos(angle));
    sy += s.sensor.y + (r * sin(angle));
    n += 1.0;
  }
  if (n != 0.0) {
    s.bary.x = sx / n; s.bary.y = sy / n; s.bary.h = 0.0;
  } else {
    s.bary = s.sensor;
  }
}

// LocalizedRangeScan::SetSensorPose (Karto.h:5289-5303)
void set_sensor_pose(const b2s_mapper *m, MScan &s, const P3 &scan_pose) {
  const double ox = m->laser.offset_pose[0], oy = m->laser.offset_pose[1], oh = m->laser.offset_pose[2];
  const double len = sqrt(ox * ox + oy * oy);
  const double angleoffset = atan2(oy, ox);
  const double ch = normalize_angle(scan_pose.h);
  const double wx = len * cos(ch + angleoffset - oh), wy = len * sin(ch + angleoffset - oh);
  s.corrected.x = scan_pose.x - wx;  // Pose2 operator-: heading normalised
  s.corrected.y = scan_pose.y - wy;
  s.corrected.h = normalize_angle(scan_pose.h - oh);
  scan_update(m, s);
}

inline const P3 &ref_pose(const b2s_mapper *m, const MScan &s) { return m->prm.use_scan_barycenter ? s.bary : s.sensor; }

struct MatchJob {
  P3 robot_pose;                 // the scan's corrected pose at match time
  const std::vector<double> *ranges;
  std::vector<int> chain;        // base scans (indices into m->scans)
};

b2s_status cuda_ensure_handle(CudaBackend *c, int which, int batch, int max_base);

// The CUDA path proper: base scans are referenced by their row in the handle's device-resident scan pool (every scan
// of the mapper is uploaded once per handle), so a match uploads only the matched scans, the chain rows and the
// chain poses.  Ragged chains are padded to the longest chain of the batch by repeating the last row.
b2s_status cuda_match_ids(b2s_mapper *m, int which, const std::vector<MatchJob> &jobs, bool do_penalize, bool do_refine,
                          std::vector<b2s_match_result> &out) {
  CudaBackend *c = m->cuda;
  const int B = (int)jobs.size(), N = m->laser.n_readings;
  int max_base = 1;
  for (const MatchJob &j : jobs) {
    if (j.chain.empty()) B2S_FAIL(B2S_ERR_BAD_PARAMS, "mapper: MatchScan against an empty chain");
    max_base = std::max(max_base, (int)j.chain.size());
  }
  b2s_status st = cuda_ensure_handle(c, which, B, max_base);
  if (st) return st;
  for (; c->pool_n[which] < m->scans.size(); c->pool_n[which]++) {  // new scans (all of them after a handle re-creation)
    st = b2s_matcher_pool_append(c->h[which], m->scans[c->pool_n[which]].ranges.data(), nullptr);
    if (st) return st;
  }
  std::vector<double> ranges((size_t)B * N), poses((size_t)B * 3);
  c->base_rows.resize((size_t)B * max_base);
  c->base_p.resize((size_t)B * max_base * 3);
  for (int b = 0; b < B; b++) {
    std::memcpy(&ranges[(size_t)b * N], jobs[b].ranges->data(), sizeof(double) * N);
    poses[3 * b] = jobs[b].robot_pose.x; poses[3 * b + 1] = jobs[b].robot_pose.y; poses[3 * b + 2] = jobs[b].robot_pose.h;
    const int nb = (int)jobs[b].chain.size();
    for (int j = 0; j < max_base; j++) {
      const int id = jobs[b].chain[std::min(j, nb - 1)];
      const MScan &sc = m->scans[id];
      const size_t k = (size_t)b * max_base + j;
      c->base_rows[k] = id;
      c->base_p[3 * k] = sc.corrected.x; c->base_p[3 * k + 1] = sc.corrected.y; c->base_p[3 * k + 2] = sc.corrected.h;
    }
  }
  st = b2s_matcher_set_scans(c->h[which], B, ranges.data(), poses.data());
  if (!st) st = b2s_matcher_add_scans_pool(c->h[which], max_base, c->base_rows.data(), c->base_p.data());
  if (!st) st = b2s_matcher_match_scan(c->h[which], do_penalize ? 1 : 0, do_refine ? 1 : 0, out.data());
  return st;
}

b2s_status run_matches(b2s_mapper *m, int which, const std::vector<MatchJob> &jobs, bool do_penalize, bool do_refine,
                       std::vector<b2s_match_result> &out) {
  const int B = (int)jobs.size(), N = m->laser.n_readings;
  out.assign(B, b2s_match_result{});
  if (B == 0) return B2S_OK;
  if (m->cuda) {
    m->n_match_calls += B;
    m->n_batches += 1;
    return cuda_match_ids(m, which, jobs, do_penalize, do_refine, out);
  }
  std::vector<double> ranges((size_t)B * N), poses((size_t)B * 3);
  std::vector<int32_t> first(B), count(B);
  size_t total = 0;
  for (int b = 0; b < B; b++) {
    std::memcpy(&ranges[(size_t)b * N], jobs[b].ranges->data(), sizeof(double) * N);
    poses[3 * b] = jobs[b].robot_pose.x; poses[3 * b + 1] = jobs[b].robot_pose.y; poses[3 * b + 2] = jobs[b].robot_pose.h;
    first[b] = (int32_t)total;
    count[b] = (int32_t)jobs[b].chain.size();
    total += jobs[b].chain.size();
  }
  std::vector<double> br(total * N), bp(total * 3);
  size_t k = 0;
  for (int b = 0; b < B; b++)
    for (int id : jobs[b].chain) {
      const MScan &s = m->scans[id];
      std::memcpy(&br[k * N], s.ranges.data(), sizeof(double) * N);
      bp[3 * k] = s.corrected.x; bp[3 * k + 1] = s.corrected.y; bp[3 * k + 2] = s.corrected.h;
      k++;
    }
  m->n_match_calls += B;
  m->n_batches += 1;
  return m->match(m->match_user, which, B, ranges.data(), poses.data(), first.data(), count.data(), br.data(), bp.data(),
                  do_penalize ? 1 : 0, do_refine ? 1 : 0, out.data());
}

// (re)creating a handle costs tens of ms (device + pinned allocations): size it for the running window up front and
// double on growth so that a stream re-creates it a handful of times at most
b2s_status cuda_ensure_handle(CudaBackend *c, int which, int batch, int max_base) {
  if (c->h[which] && batch <= c->cap_batch[which] && max_base <= c->cap_base[which]) return B2S_OK;
  if (c->h[which]) b2s_matcher_destroy(c->h[which]);
  c->h[which] = nullptr;
  c->pool_n[which] = 0;
  const int cb = std::max(std::max(batch, c->cap_batch[which] * 2), 8);
  const int cs = std::max(std::max(max_base, c->cap_base[which] * 2), c->min_base);
  b2s_status st = b2s_matcher_create(&c->params[which], &c->laser, c->device, cb, cs, nullptr, &c->h[which]);
  if (st) return st;
  c->cap_batch[which] = cb;
  c->cap_base[which] = cs;
  return B2S_OK;
}

// ---- the CUDA matcher behind the generic plug-in signature (host arrays in; the mapper itself takes the pooled path
// above, this form serves callers that drive b2s_match_scan_fn directly): ragged chains are padded to the longest chain of the batch by repeating each
// match's last base scan (rasterising a scan twice leaves the correlation grid unchanged)
b2s_status cuda_match(void *user, int which, int batch, const double *ranges, const double *poses, const int32_t *base_first,
                      const int32_t *n_base, const double *base_ranges, const double *base_poses, int do_penalize,
                      int do_refine, b2s_match_result *results) {
  CudaBackend *c = static_cast<CudaBackend *>(user);
  const int N = c->laser.n_readings;
  int max_base = 1;
  for (int b = 0; b < batch; b++) max_base = std::max(max_base, (int)n_base[b]);
  {
    b2s_status st = cuda_ensure_handle(c, which, batch, max_base);
    if (st) return st;
  }
  for (int b = 0; b < batch; b++)
    if (n_base[b] <= 0) B2S_FAIL(B2S_ERR_BAD_PARAMS, "mapper: MatchScan against an empty chain");
  c->base_r.resize((size_t)batch * max_base * N);
  c->base_p.resize((size_t)batch * max_base * 3);
  for (int b = 0; b < batch; b++)
    for (int j = 0; j < max_base; j++) {
      const size_t src = (size_t)base_first[b] + std::min(j, (int)n_base[b] - 1), dst = (size_t)b * max_base + j;
      std::memcpy(&c->base_r[dst * N], base_ranges + src * N, sizeof(double) * N);
      std::memcpy(&c->base_p[dst * 3], base_poses + src * 3, sizeof(double) * 3);
    }
  return b2s_matcher_match_scan_host(c->h[which], batch, ranges, poses, max_base, c->base_r.data(), c->base_p.data(),
                                     do_penalize, do_refine, results);
}

// ---- MapperGraph

// BreadthFirstTraversal::Traverse with a NearScanVisitor (Mapper.h:568-643): scans linked to `start` by a path of
// edges whose every vertex lies within max_distance of it, in visiting order
std::vector<int> find_near_linked_scans(const b2s_mapper *m, int start, double max_distance) {
  const double max_sq = sq(max_distance);
  const P3 center = ref_pose(m, m->scans[start]);
  std::vector<int> valid;
  std::vector<char> seen(m->scans.size(), 0);
  std::queue<int> to_visit;
  to_visit.push(start);
  seen[start] = 1;
  do {
    const int next = to_visit.front();
    to_visit.pop();
    if (sqdist(ref_pose(m, m->scans[next]), center) <= max_sq - KT_TOLERANCE) {
      valid.push_back(next);
      for (int e : m->scans[next].edges) {  // Vertex::GetAdjacentVertices (Mapper.h:208-225)
        const MEdge &ed = m->edges[e];
        for (int adj : {ed.src, ed.dst}) {
          if (adj == next) continue;
          if (!seen[adj]) {
            to_visit.push(adj);
            seen[adj] = 1;
          }
        }
      }
    }
  } while (!to_visit.empty());
  return valid;
}

// MapperGraph::LinkScans + AddEdge (Mapper.cpp:1075-1120) with LinkInfo::Update (Mapper.h:125-151)
void link_scans(b2s_mapper *m, int from, int to, const P3 &mean, const M3 &cov) {
  for (int e : m->scans[from].edges)
    if (m->edges[e].dst == to) return;  // the edge exists: nothing is attached (isNewEdge == false)
  MEdge ed;
  ed.src = from; ed.dst = to;
  ed.pose1 = m->scans[from].sensor;
  ed.pose2 = mean;
  ed.diff = Xform(ed.pose1, P3()).apply(ed.pose2);
  const M3 rot = M3::axis_z(-ed.pose1.h);
  ed.cov = rot * cov * rot.transpose();
  const int idx = (int)m->edges.size();
  m->edges.push_back(ed);
  m->scans[from].edges.push_back(idx);
  m->scans[to].edges.push_back(idx);
  if (m->have_solver && m->solver.add_constraint) {
    const double d[3] = {ed.diff.x, ed.diff.y, ed.diff.h};
    m->solver.add_constraint(m->solver.user, from, to, d, &ed.cov.m[0][0]);
  }
}

// MapperGraph::LinkChainToScan + GetClosestScanToPose (Mapper.cpp:1054-1073, 1152-1167)
void link_chain_to_scan(b2s_mapper *m, const std::vector<int> &chain, int scan, const P3 &mean, const M3 &cov) {
  const P3 pose = ref_pose(m, m->scans[scan]);
  int closest = -1;
  double best = 1.7976931348623157e308;  // DBL_MAX
  for (int id : chain) {
    const double d = sqdist(pose, ref_pose(m, m->scans[id]));
    if (d < best) { best = d; closest = id; }
  }
  if (closest < 0) return;
  const double d = sqdist(pose, ref_pose(m, m->scans[closest]));
  if (d < sq(m->prm.link_scan_maximum_distance) + KT_TOLERANCE) link_scans(m, closest, scan, mean, cov);
}

// MapperGraph::FindNearChains (Mapper.cpp:1170-1275)
std::vector<std::vector<int>> find_near_chains(const b2s_mapper *m, int scan) {
  std::vector<std::vector<int>> chains;
  const P3 scan_pose = ref_pose(m, m->scans[scan]);
  std::vector<char> processed(m->scans.size(), 0);
  const std::vector<int> near = find_near_linked_scans(m, scan, m->prm.link_scan_maximum_distance);
  const double lim = sq(m->prm.link_scan_maximum_distance) + KT_TOLERANCE;
  for (int near_id : near) {
    if (near_id == scan) continue;
    if (processed[near_id]) continue;
    processed[near_id] = 1;
    bool valid = true;
    std::list<int> chain;
    // the chain grows along the state ids of the NEAR scan's own sensor (Mapper.cpp:1208-1262)
    const std::vector<int> &ids = m->sensors[m->scans[near_id].dev].ids;
    const int st = m->scans[near_id].state, n_scans = (int)ids.size();
    for (int cs = st - 1; cs >= 0; cs--) {
      const int c = ids[cs];
      if (c == scan) valid = false;
      if (sqdist(scan_pose, ref_pose(m, m->scans[c])) < lim) {
        chain.push_front(c);
        processed[c] = 1;
      } else {
        break;
      }
    }
    chain.push_back(near_id);
    for (int cs = st + 1; cs < n_scans; cs++) {
      const int c = ids[cs];
      if (c == scan) valid = false;
      if (sqdist(scan_pose, ref_pose(m, m->scans[c])) < lim) {
        chain.push_back(c);
        processed[c] = 1;
      } else {
        break;
      }
    }
    if (valid) chains.emplace_back(chain.begin(), chain.end());
  }
  return chains;
}

// MapperGraph::ComputeWeightedMean (Mapper.cpp:1288-1330)
b2s_status weighted_mean(const std::vector<P3> &means, const std::vector<M3> &covs, P3 &out) {
  std::vector<M3> inverses;
  inverses.reserve(covs.size());
  M3 sum;
  for (const M3 &c : covs) {
    M3 inv;
    if (!c.inverse(inv)) B2S_FAIL(B2S_ERR_BAD_STATE, "mapper: singular link covariance (the reference asserts here)");
    inverses.push_back(inv);
    sum.add(inv);
  }
  M3 inv_sum;
  if (!sum.inverse(inv_sum)) B2S_FAIL(B2S_ERR_BAD_STATE, "mapper: singular covariance sum (the reference asserts here)");
  P3 acc;
  double tx = 0.0, ty = 0.0;
  for (size_t i = 0; i < means.size(); i++) {
    const P3 &pose = means[i];
    tx += cos(pose.h);
    ty += sin(pose.h);
    const M3 weight = inv_sum * inverses[i];
    const P3 w = weight * pose;
    acc.x += w.x; acc.y += w.y;
    acc.h = normalize_angle(acc.h + w.h);  // Pose2::operator+=
  }
  tx /= (double)means.size();
  ty /= (double)means.size();
  acc.h = atan2(ty, tx);
  out = acc;
  return B2S_OK;
}

M3 cov_of(const b2s_match_result &r) {
  M3 c;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) c.m[i][j] = r.cov[3 * i + j];
  return c;
}

// MapperGraph::LinkNearChains (Mapper.cpp:1124-1149): all chains matched as one batch
b2s_status link_near_chains(b2s_mapper *m, int scan, std::vector<P3> &means, std::vector<M3> &covs) {
  const std::vector<std::vector<int>> near = find_near_chains(m, scan);
  std::vector<MatchJob> jobs;
  std::vector<int> which;
  for (size_t i = 0; i < near.size(); i++) {
    if ((int)near[i].size() < m->prm.loop_match_minimum_chain_size) continue;
    jobs.push_back(MatchJob{m->scans[scan].corrected, &m->scans[scan].ranges, near[i]});
    which.push_back((int)i);
  }
  std::vector<b2s_match_result> res;
  b2s_status st = run_matches(m, 0, jobs, false, true, res);
  if (st) return st;
  for (size_t j = 0; j < jobs.size(); j++) {
    if (res[j].status) B2S_FAIL((b2s_status)res[j].status, "mapper: near-chain MatchScan failed");
    if (res[j].response > m->prm.link_match_minimum_response_fine - KT_TOLERANCE) {
      const P3 mean = p3(res[j].pose);
      const M3 cov = cov_of(res[j]);
      means.push_back(mean);
      covs.push_back(cov);
      link_chain_to_scan(m, near[which[j]], scan, mean, cov);
    }
  }
  return B2S_OK;
}

// MapperGraph::AddEdges (Mapper.cpp:902-973)
b2s_status add_edges(b2s_mapper *m, int scan, const M3 &cov) {
  const int sensor = m->scans[scan].dev;
  const SensorState &S = m->sensors[sensor];
  const bool have_last = S.last_scan >= 0;
  if (have_last) link_scans(m, S.ids[m->scans[scan].state - 1], scan, m->scans[scan].sensor, cov);
  std::vector<P3> means;
  std::vector<M3> covs;
  if (have_last) {
    const P3 scan_pose = m->scans[scan].sensor;
    means.push_back(scan_pose);
    covs.push_back(cov);
    link_chain_to_scan(m, S.running, scan, scan_pose, cov);
  } else {
    // a sensor's first scan is matched against ALL scans of every other sensor (in name order) and linked to that
    // sensor's first scan whatever the response (Mapper.cpp:920-952); the matches do not depend on each other
    std::vector<MatchJob> jobs;
    std::vector<int> firsts;
    for (int other : m->by_name) {
      if (other == sensor || m->sensors[other].ids.empty()) continue;
      jobs.push_back(MatchJob{m->scans[scan].corrected, &m->scans[scan].ranges, m->sensors[other].ids});
      firsts.push_back(m->sensors[other].ids[0]);
    }
    if (!jobs.empty()) {
      std::vector<b2s_match_result> res;
      b2s_status st = run_matches(m, 0, jobs, true, true, res);
      if (st) return st;
      for (size_t j = 0; j < jobs.size(); j++) {
        if (res[j].status) B2S_FAIL((b2s_status)res[j].status, "mapper: first-scan MatchScan against another sensor failed");
        const P3 best = p3(res[j].pose);
        const M3 c = cov_of(res[j]);
        link_scans(m, firsts[j], scan, best, c);
        if (res[j].response > m->prm.link_match_minimum_response_fine) {
          means.push_back(best);
          covs.push_back(c);
        }
      }
    }
  }
  b2s_status st = link_near_chains(m, scan, means, covs);
  if (st) return st;
  if (!means.empty()) {
    P3 mean;
    st = weighted_mean(means, covs, mean);
    if (st) return st;
    set_sensor_pose(m, m->scans[scan], mean);
  }
  return B2S_OK;
}

// ScanManager::AddRunningScan (Mapper.h:1365-1386)
void add_running_scan(b2s_mapper *m, int scan) {
  std::vector<int> &running = m->sensors[m->scans[scan].dev].running;
  running.push_back(scan);
  auto d = [&]() { return sqdist(m->scans[running.front()].sensor, m->scans[running.back()].sensor); };
  double sd = d();
  while (running.size() > (size_t)m->prm.scan_buffer_size ||
         sd > sq(m->prm.scan_buffer_maximum_scan_distance) - KT_TOLERANCE) {
    running.erase(running.begin());
    sd = d();
  }
}

// MapperGraph::FindPossibleLoopClosure (Mapper.cpp:1333-1394)
std::vector<int> find_possible_loop_closure(const b2s_mapper *m, int scan, int sensor, const std::vector<char> &near_linked,
                                            unsigned &start) {
  std::vector<int> chain;
  const P3 pose = ref_pose(m, m->scans[scan]);
  const std::vector<int> &ids = m->sensors[sensor].ids;  // the candidate sensor's scans, by state id
  const unsigned n_scans = (unsigned)ids.size();
  const double lim = sq(m->prm.loop_search_maximum_distance) + KT_TOLERANCE;
  for (; start < n_scans; start++) {
    const int id = ids[start];
    if (sqdist(ref_pose(m, m->scans[id]), pose) < lim) {
      if (near_linked[id]) chain.clear();
      else chain.push_back(id);
    } else {
      if (chain.size() >= (size_t)m->prm.loop_match_minimum_chain_size) return chain;
      chain.clear();
    }
  }
  return chain;
}

// MapperGraph::CorrectPoses (Mapper.cpp:1397-1414)
void correct_poses(b2s_mapper *m) {
  if (!m->have_solver || !m->solver.compute) return;
  const int cap = (int)m->scans.size();
  std::vector<int32_t> ids(cap);
  std::vector<double> poses((size_t)cap * 3);
  const int n = m->solver.compute(m->solver.user, cap, ids.data(), poses.data());
  for (int i = 0; i < n && i < cap; i++)
    if (ids[i] >= 0 && ids[i] < cap) set_sensor_pose(m, m->scans[ids[i]], p3(&poses[3 * i]));
  if (m->solver.clear) m->solver.clear(m->solver.user);
}

// MapperGraph::TryCloseLoop (Mapper.cpp:976-1051).  The reference examines candidate chains one after another; the
// coarse matches of successive candidates are independent until a loop is actually closed (which moves the scan and,
// with a solver, every pose), so all candidates that the CURRENT state yields are matched as one batch and then
// walked in order; after an accepted closure the remaining candidates are re-enumerated from the new state.
b2s_status try_close_loop(b2s_mapper *m, int scan, int sensor) {
  unsigned scan_index = 0;
  for (;;) {
    std::vector<char> near_linked(m->scans.size(), 0);
    for (int id : find_near_linked_scans(m, scan, m->prm.loop_search_maximum_distance)) near_linked[id] = 1;
    std::vector<std::vector<int>> chains;
    std::vector<unsigned> index_after;
    for (unsigned idx = scan_index;;) {
      std::vector<int> chain = find_possible_loop_closure(m, scan, sensor, near_linked, idx);
      if (chain.empty()) break;
      chains.push_back(std::move(chain));
      index_after.push_back(idx);
    }
    if (chains.empty()) return B2S_OK;
    std::vector<MatchJob> jobs;
    for (const auto &c : chains) jobs.push_back(MatchJob{m->scans[scan].corrected, &m->scans[scan].ranges, c});
    std::vector<b2s_match_result> coarse;
    b2s_status st = run_matches(m, 1, jobs, false, false, coarse);
    if (st) return st;
    bool closed = false;
    for (size_t k = 0; k < chains.size() && !closed; k++) {
      m->n_loop_candidates += 1;
      if (coarse[k].status) B2S_FAIL((b2s_status)coarse[k].status, "mapper: loop-closure coarse MatchScan failed");
      const double lim = m->prm.loop_match_maximum_variance_coarse;
      if (coarse[k].response > m->prm.loop_match_minimum_response_coarse && coarse[k].cov[0] < lim && coarse[k].cov[4] < lim) {
        // tmpScan: same readings, corrected pose derived from the coarse best sensor pose (Mapper.cpp:1007-1012)
        MScan tmp;
        tmp.ranges = m->scans[scan].ranges;
        tmp.corrected = m->scans[scan].corrected;
        set_sensor_pose(m, tmp, p3(coarse[k].pose));
        std::vector<MatchJob> fine_job{MatchJob{tmp.corrected, &tmp.ranges, chains[k]}};
        std::vector<b2s_match_result> fine;
        st = run_matches(m, 0, fine_job, false, true, fine);
        if (st) return st;
        if (fine[0].status) B2S_FAIL((b2s_status)fine[0].status, "mapper: loop-closure fine MatchScan failed");
        if (!(fine[0].response < m->prm.loop_match_minimum_response_fine)) {
          const P3 best = p3(fine[0].pose);
          set_sensor_pose(m, m->scans[scan], best);
          link_chain_to_scan(m, chains[k], scan, best, cov_of(fine[0]));
          correct_poses(m);
          m->n_loops_closed += 1;
          closed = true;
          scan_index = index_after[k];
        }
      }
    }
    if (!closed) return B2S_OK;
  }
}

// Mapper::HasMovedEnough (Mapper.cpp:2087-2119)
bool has_moved_enough(const b2s_mapper *m, const MScan &scan, const MScan *last) {
  if (!last) return true;
  if (scan.time - last->time >= m->prm.minimum_time_interval) return true;
  double a[3], b[3];
  const double lo[3] = {last->odom.x, last->odom.y, last->odom.h}, so[3] = {scan.odom.x, scan.odom.y, scan.odom.h};
  sensor_pose_of(lo, m->laser.offset_pose, a);
  sensor_pose_of(so, m->laser.offset_pose, b);
  const double dh = normalize_angle(b[2] - a[2]);
  if (fabs(dh) >= m->prm.minimum_travel_heading) return true;
  const double d = sqdist(p3(a), p3(b));
  return d >= sq(m->prm.minimum_travel_distance) - KT_TOLERANCE;
}

b2s_status check_params(const b2s_mapper_params *p, const b2s_laser *l) {
  if (!p || !l) B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_mapper_create: null argument");
  if (l->n_readings <= 0 || p->scan_buffer_size < 1 || p->loop_match_minimum_chain_size < 0)
    B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_mapper_create: bad laser / buffer parameters");
  return B2S_OK;
}

}  // namespace

extern "C" {

void b2s_mapper_default_params(b2s_mapper_params *o, double range_threshold) {
  if (!o) return;
  std::memset(o, 0, sizeof(*o));
  const double deg = KT_PI / 180.0;
  o->use_scan_matching = 1;
  o->use_scan_barycenter = 1;
  o->minimum_time_interval = 3600;
  o->minimum_travel_distance = 0.2;
  o->minimum_travel_heading = 10 * deg;
  o->scan_buffer_size = 70;
  o->scan_buffer_maximum_scan_distance = 20.0;
  o->link_match_minimum_response_fine = 0.8;
  o->link_scan_maximum_distance = 10.0;
  o->loop_search_maximum_distance = 4.0;
  o->do_loop_closing = 1;
  o->loop_match_minimum_chain_size = 10;
  o->loop_match_maximum_variance_coarse = 0.4 * 0.4;
  o->loop_match_minimum_response_coarse = 0.8;
  o->loop_match_minimum_response_fine = 0.8;
  b2s_matcher_params t;
  std::memset(&t, 0, sizeof(t));
  t.range_threshold = range_threshold;
  t.distance_variance_penalty = 0.3 * 0.3;
  t.angle_variance_penalty = (20 * deg) * (20 * deg);
  t.fine_search_angle_offset = 0.2 * deg;
  t.coarse_search_angle_offset = 20 * deg;
  t.coarse_angle_resolution = 2 * deg;
  t.minimum_angle_penalty = 0.9;
  t.minimum_distance_penalty = 0.5;
  t.use_response_expansion = 0;
  o->sequential = t;
  o->sequential.search_size = 0.3; o->sequential.resolution = 0.01; o->sequential.smear_deviation = 0.03;
  o->loop = t;
  o->loop.search_size = 8.0; o->loop.resolution = 0.05; o->loop.smear_deviation = 0.03;
}

b2s_status b2s_mapper_create_with_matcher(const b2s_mapper_params *params, const b2s_laser *laser, b2s_match_scan_fn match,
                                          void *user, b2s_mapper **out) {
  if (!out || !match) B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_mapper_create_with_matcher: null argument");
  *out = nullptr;
  b2s_status st = check_params(params, laser);
  if (st) return st;
  b2s_mapper *m = new (std::nothrow) b2s_mapper();
  if (!m) B2S_FAIL(B2S_ERR_CUDA, "out of host memory");
  m->prm = *params;
  m->laser = *laser;
  m->match = match;
  m->match_user = user;
  *out = m;
  return B2S_OK;
}

b2s_status b2s_mapper_create(const b2s_mapper_params *params, const b2s_laser *laser, int device, b2s_mapper **out) {
  if (!out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_mapper_create: null argument");
  *out = nullptr;
  b2s_status st = check_params(params, laser);
  if (st) return st;
  if (b2s_device_count() <= device) B2S_FAIL(B2S_ERR_NO_DEVICE, "no usable CUDA device (the product path has no CPU fallback)");
  CudaBackend *c = new (std::nothrow) CudaBackend();
  if (!c) B2S_FAIL(B2S_ERR_CUDA, "out of host memory");
  c->device = device;
  c->laser = *laser;
  c->params[0] = params->sequential;
  c->params[1] = params->loop;
  c->min_base = std::max(32, params->scan_buffer_size + 1);
  st = b2s_mapper_create_with_matcher(params, laser, cuda_match, c, out);
  if (st) {
    delete c;
    return st;
  }
  (*out)->cuda = c;
  return B2S_OK;
}

void b2s_mapper_destroy(b2s_mapper *m) {
  if (!m) return;
  delete m->cuda;
  delete m;
}

b2s_status b2s_mapper_set_scan_solver(b2s_mapper *m, const b2s_scan_solver *solver) {
  if (!m) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  if (solver) {
    m->solver = *solver;
    m->have_solver = true;
  } else {
    m->have_solver = false;
  }
  return B2S_OK;
}

b2s_status b2s_mapper_process(b2s_mapper *m, const double *ranges, const double odometric_pose[3], double time,
                              int32_t *out_processed, double out_corrected_pose[3]) {
  return b2s_mapper_process_sensor(m, "laser", ranges, odometric_pose, time, out_processed, out_corrected_pose);
}

b2s_status b2s_mapper_process_sensor(b2s_mapper *m, const char *sensor_name, const double *ranges,
                                     const double odometric_pose[3], double time, int32_t *out_processed,
                                     double out_corrected_pose[3]) {
  B2S_NVTX("Mapper::Process");
  if (!m || !ranges || !odometric_pose || !sensor_name) B2S_FAIL(B2S_ERR_BAD_PARAMS, "b2s_mapper_process: null argument");
  if (out_processed) *out_processed = 0;
  if (m->failed)
    B2S_FAIL(B2S_ERR_BAD_STATE, "b2s_mapper_process: an earlier call failed half-way (the reference aborts there); destroy the handle");
  // MapperSensorManager::GetLastScan registers an unknown sensor (Mapper.h:1470-1475, Mapper.cpp:45-52)
  int sensor = -1;
  for (size_t i = 0; i < m->sensors.size(); i++)
    if (m->sensors[i].name == sensor_name) sensor = (int)i;
  if (sensor < 0) {
    sensor = (int)m->sensors.size();
    m->sensors.emplace_back();
    m->sensors.back().name = sensor_name;
    m->by_name.push_back(sensor);
    std::sort(m->by_name.begin(), m->by_name.end(), [&](int a, int b) { return m->sensors[a].name < m->sensors[b].name; });
  }
  m->last_sensor = sensor;
  MScan scan;
  scan.dev = sensor;
  scan.ranges.assign(ranges, ranges + m->laser.n_readings);
  scan.odom = p3(odometric_pose);
  scan.corrected = scan.odom;  // karto_slam.cc:437-440 sets both poses from odometry before Process
  scan.time = time;
  const MScan *last = m->sensors[sensor].last_scan >= 0 ? &m->scans[m->sensors[sensor].last_scan] : nullptr;
  if (last) scan.corrected = Xform(last->odom, last->corrected).apply(scan.odom);  // Mapper.cpp:2021-2026
  if (out_corrected_pose) { out_corrected_pose[0] = scan.corrected.x; out_corrected_pose[1] = scan.corrected.y; out_corrected_pose[2] = scan.corrected.h; }
  if (!has_moved_enough(m, scan, last)) return B2S_OK;
  scan_update(m, scan);
  M3 cov = M3::identity();
  if (m->prm.use_scan_matching && last) {
    std::vector<MatchJob> job{MatchJob{scan.corrected, &scan.ranges, m->sensors[sensor].running}};
    std::vector<b2s_match_result> res;
    b2s_status st = run_matches(m, 0, job, true, true, res);
    if (st) return st;
    if (res[0].status) B2S_FAIL((b2s_status)res[0].status, "mapper: sequential MatchScan failed");
    cov = cov_of(res[0]);
    set_sensor_pose(m, scan, p3(res[0].pose));
  }
  scan.id = (int)m->scans.size();                    // MapperSensorManager::AddScan (Mapper.cpp:75-80): unique id
  scan.state = (int)m->sensors[sensor].ids.size();   // ScanManager::AddScan: state id within the sensor
  m->scans.push_back(std::move(scan));
  const int id = (int)m->scans.size() - 1;
  m->sensors[sensor].ids.push_back(id);
  if (m->prm.use_scan_matching) {
    if (m->have_solver && m->solver.add_node) {  // MapperGraph::AddVertex -> ScanSolver::AddNode
      const MScan &s = m->scans[id];
      const double c[3] = {s.corrected.x, s.corrected.y, s.corrected.h};
      m->solver.add_node(m->solver.user, id, c);
    }
    // from here on the scan is part of the graph: a failure leaves a vertex without its edges / running-window entry,
    // so the handle is marked failed and every later Process returns B2S_ERR_BAD_STATE
    b2s_status st = add_edges(m, id, cov);
    if (st) { m->failed = true; return st; }
    add_running_scan(m, id);
    if (m->prm.do_loop_closing) {
      for (size_t k = 0; k < m->by_name.size(); k++) {  // against every sensor's scans, in name order (Mapper.cpp:2063-2070)
        st = try_close_loop(m, id, m->by_name[k]);
        if (st) { m->failed = true; return st; }
      }
    }
  }
  m->sensors[sensor].last_scan = id;
  if (out_processed) *out_processed = 1;
  if (out_corrected_pose) {
    const MScan &s = m->scans[id];
    out_corrected_pose[0] = s.corrected.x; out_corrected_pose[1] = s.corrected.y; out_corrected_pose[2] = s.corrected.h;
  }
  return B2S_OK;
}

int32_t b2s_mapper_scan_count(const b2s_mapper *m) { return m ? (int32_t)m->scans.size() : 0; }

b2s_status b2s_mapper_get_poses(const b2s_mapper *m, double *out) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  for (size_t i = 0; i < m->scans.size(); i++) {
    out[3 * i] = m->scans[i].corrected.x; out[3 * i + 1] = m->scans[i].corrected.y; out[3 * i + 2] = m->scans[i].corrected.h;
  }
  return B2S_OK;
}

int32_t b2s_mapper_sensor_count(const b2s_mapper *m) { return m ? (int32_t)m->sensors.size() : 0; }

b2s_status b2s_mapper_get_scan_sensors(const b2s_mapper *m, int32_t *out) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  std::vector<int> rank(m->sensors.size());
  for (size_t k = 0; k < m->by_name.size(); k++) rank[m->by_name[k]] = (int)k;
  for (size_t i = 0; i < m->scans.size(); i++) out[i] = rank[m->scans[i].dev];
  return B2S_OK;
}

int32_t b2s_mapper_edge_count(const b2s_mapper *m) { return m ? (int32_t)m->edges.size() : 0; }

b2s_status b2s_mapper_get_edges(const b2s_mapper *m, int32_t *ids, double *pose_difference, double *covariance) {
  if (!m) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null handle");
  for (size_t i = 0; i < m->edges.size(); i++) {
    const MEdge &e = m->edges[i];
    if (ids) { ids[2 * i] = e.src; ids[2 * i + 1] = e.dst; }
    if (pose_difference) { pose_difference[3 * i] = e.diff.x; pose_difference[3 * i + 1] = e.diff.y; pose_difference[3 * i + 2] = e.diff.h; }
    if (covariance) std::memcpy(covariance + 9 * i, &e.cov.m[0][0], 9 * sizeof(double));
  }
  return B2S_OK;
}

b2s_status b2s_mapper_stats(const b2s_mapper *m, double out[5]) {
  if (!m || !out) B2S_FAIL(B2S_ERR_BAD_PARAMS, "null argument");
  out[0] = m->n_match_calls; out[1] = m->n_batches; out[2] = m->n_loop_candidates; out[3] = m->n_loops_closed;
  out[4] = m->sensors.empty() ? 0.0 : (double)m->sensors[m->last_sensor].running.size();  // of the sensor processed last
  return B2S_OK;
}

}  // extern "C"

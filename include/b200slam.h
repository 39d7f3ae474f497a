/*
 * b200slam.h — the C ABI of the B200-native 2-D laser SLAM front-end hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8(b)).  The reference
 * (xiangli0608/Creating-2D-laser-slam-from-scratch) has no C ABI; its seams are C++ class
 * methods called in-process.  Every entry point below names the reference method it stands in
 * for (file:line relative to /root/reference).  A reference-side façade with the reference's own
 * signatures is in include/b200slam/karto_facade.hpp; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types; all arrays are caller-owned HOST memory
 *     unless the name says `_device`.
 *   - every function returns a b2s_status (0 = OK); exceptions of the reference map to codes.
 *   - a handle is single-threaded like the reference's ScanMatcher (Mapper.h:1273-1278 shares
 *     m_pCorrelationGrid / m_pGridLookup); DISTINCT handles may be used concurrently
 *     (one CUDA stream each).
 *   - "batch" = B independent scan-matches, each with its OWN correlation grid (SURVEY.md §8(e)(i)).
 *   - poses are (x, y, heading) doubles; covariances are row-major 3x3 doubles.
 *   - the product path is CUDA only: if no device is usable every compute entry point returns
 *     B2S_ERR_NO_DEVICE.  There is no CPU fallback.
 */
#ifndef B200SLAM_H
#define B200SLAM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2S_ABI_VERSION 1

typedef enum b2s_status {
  B2S_OK = 0,
  B2S_ERR_BAD_PARAMS = 1,   /* ScanMatcher::Create -> NULL (Mapper.cpp:130-145); smear out of range (Mapper.h:1045-1053) */
  B2S_ERR_OUT_OF_RANGE = 2, /* karto::Exception "Index out of range" (Karto.h:4492-4498) */
  B2S_ERR_NO_BEST_POSE = 3, /* std::runtime_error "Unable to find best position" (Mapper.cpp:486) */
  B2S_ERR_CUDA = 4,         /* a CUDA runtime call failed; see b2s_last_error() */
  B2S_ERR_NO_DEVICE = 5,    /* no CUDA device: the product path never falls back to the CPU */
  B2S_ERR_BAD_STATE = 6,    /* call order violated (e.g. correlate before scans are set) */
  B2S_ERR_TOO_LARGE = 7     /* batch / beam count / window exceeds what the handle was created for */
} b2s_status;

/* ScanMatcher::Create arguments (Mapper.cpp:126-127) + the 8 tuning values the matcher reads from its
 * Mapper through friend access (Mapper.cpp:206,238-239,250,256,279-280,405-411).  Values are the ones
 * STORED in the Mapper: setParamDistanceVariancePenalty/AngleVariancePenalty square their argument
 * (Mapper.cpp:1919-1927) — do that before filling this struct.  Defaults: Mapper.cpp:1569-1652. */
typedef struct b2s_matcher_params {
  double search_size;                /* CorrelationSearchSpaceDimension, m */
  double resolution;                 /* CorrelationSearchSpaceResolution, m/cell */
  double smear_deviation;            /* CorrelationSearchSpaceSmearDeviation, m */
  double range_threshold;            /* LaserRangeFinder range threshold, m */
  double distance_variance_penalty;  /* default 0.3^2 */
  double angle_variance_penalty;     /* default (20 deg)^2 */
  double fine_search_angle_offset;   /* default 0.2 deg */
  double coarse_search_angle_offset; /* default 20 deg */
  double coarse_angle_resolution;    /* default 2 deg */
  double minimum_angle_penalty;      /* default 0.9 */
  double minimum_distance_penalty;   /* default 0.5 */
  int32_t use_response_expansion;    /* default 0 */
  int32_t reserved;
} b2s_matcher_params;

/* The part of karto::LaserRangeFinder (Karto.h:3700-4184) the hot path reads. */
typedef struct b2s_laser {
  int32_t n_readings; /* LaserRangeFinder::GetNumberOfRangeReadings (1081 for Hokuyo_UTM_30LX; a Custom
                         sensor yields round((max-min)/res) WITHOUT +1, Karto.h:4158-4160) */
  int32_t reserved;
  double min_angle;          /* rad */
  double angular_resolution; /* rad */
  double min_range;          /* m */
  double max_range;          /* m */
  double range_threshold;    /* m */
  double offset_pose[3];     /* sensor pose in the robot frame (Sensor::GetOffsetPose) */
} b2s_laser;

/* CorrelationGrid geometry (Mapper.h:900-1118, Karto.h:4381-4767). */
typedef struct b2s_grid_info {
  int32_t width, height; /* allocation incl. smear border */
  int32_t width_step;    /* AlignValue(width, 8) (Karto.h:4442) */
  int32_t data_size;     /* width_step * height bytes */
  int32_t roi_x, roi_y, roi_w, roi_h;
  int32_t kernel_size;   /* smear kernel side, 2*round(2*sigma/res)+1 */
  int32_t search_side;   /* m_pSearchSpaceProbs side = round(search_size/res)+1 */
} b2s_grid_info;

/* CorrelateScan arguments (Mapper.cpp:309-317), shared by every match of a batch. */
typedef struct b2s_search {
  double offset_x, offset_y;   /* rSearchSpaceOffset */
  double res_x, res_y;         /* rSearchSpaceResolution */
  double angle_offset;         /* searchAngleOffset */
  double angle_res;            /* searchAngleResolution */
  int32_t do_penalize;
  int32_t fine;                /* doingFineMatch */
} b2s_search;

typedef struct b2s_match_result {
  double response;   /* return value of CorrelateScan / MatchScan, clamped to <= 1 */
  double pose[3];    /* rMean */
  double cov[9];     /* rCovariance, row-major */
  int32_t status;    /* per-match b2s_status (B2S_ERR_NO_BEST_POSE ...) */
  int32_t tie_count; /* averagePoseCount (Mapper.cpp:459-471) */
} b2s_match_result;

typedef struct b2s_matcher b2s_matcher; /* opaque: replaces karto::ScanMatcher* */

/* ---------------------------------------------------------------- library */
int b2s_abi_version(void);
const char *b2s_last_error(void);              /* thread-local text of the last failure */
int b2s_device_count(void);                    /* 0 when no usable CUDA device */

/* ---------------------------------------------------------------- K1: Karto correlative scan matcher
 * Host arrays are caller-owned.  Uploads are enqueued on the handle's stream: out of pageable memory the CUDA runtime
 * stages them before the call returns; out of PINNED memory they are asynchronous, so such buffers must stay unchanged
 * until the next call that waits for the stream (correlate_scan, match_scan, _end, sync). */

/* ScanMatcher::Create (Mapper.cpp:126-172).  `max_batch` matches share one handle, each with up to
 * `max_base_scans` base scans; buffers that depend on the search volume grow on demand.  `cuda_stream` may be NULL
 * (the handle then creates its own non-blocking stream) or a cudaStream_t owned by the caller. */
b2s_status b2s_matcher_create(const b2s_matcher_params *params, const b2s_laser *laser, int device,
                              int max_batch, int max_base_scans, void *cuda_stream, b2s_matcher **out);
void b2s_matcher_destroy(b2s_matcher *m);      /* ScanMatcher::~ScanMatcher (Mapper.cpp:119-124) */
b2s_status b2s_matcher_grid_info(const b2s_matcher *m, b2s_grid_info *out);

/* The scans being matched: B x (ranges[n_readings], robot pose).  Replaces building B
 * LocalizedRangeScan objects + SetOdometricPose/SetCorrectedPose (karto_slam.cc:437-440).
 * Point readings are derived on the device as LocalizedRangeScan::Update does (Karto.h:5362-5428). */
b2s_status b2s_matcher_set_scans(b2s_matcher *m, int batch, const double *ranges, const double *poses);

/* MatchScan steps 1-4 + AddScans (Mapper.cpp:195-225, 699-811; Mapper.h:971-1005): centre grid b on scan
 * b's sensor pose and rasterise + smear its `n_base` base scans.  base_ranges: [batch][n_base][n_readings],
 * base_poses: [batch][n_base][3]. */
b2s_status b2s_matcher_add_scans(b2s_matcher *m, int n_base, const double *base_ranges, const double *base_poses);

/* Scan pool: readings that serve as base scans of many matches (a mapper's running window, near chains, loop-closure
 * candidate chains) are uploaded once (_pool_append returns the row) and referenced by row afterwards;
 * _add_scans_pool is b2s_matcher_add_scans with pool rows ([batch][n_base], host) in place of base_ranges. */
b2s_status b2s_matcher_pool_append(b2s_matcher *m, const double *ranges, int32_t *out_row);
int32_t b2s_matcher_pool_count(const b2s_matcher *m);
b2s_status b2s_matcher_add_scans_pool(b2s_matcher *m, int n_base, const int32_t *pool_rows, const double *base_poses);

/* Alternative to add_scans for callers that keep grids themselves: upload ready-made correlation grids
 * ([batch][data_size] bytes) and their world offsets ([batch][2], CoordinateConverter::SetOffset). */
b2s_status b2s_matcher_set_grids(b2s_matcher *m, const uint8_t *grids, const double *offsets);

/* ScanMatcher::CorrelateScan (Mapper.cpp:309-523) for every match of the batch; centers: [batch][3].
 * For fine=1 results[b].cov is IN/OUT exactly like rCovariance (only cov[8] is overwritten, Mapper.cpp:648,691). */
b2s_status b2s_matcher_correlate_scan(b2s_matcher *m, const double *centers, const b2s_search *search,
                                      b2s_match_result *results);

/* The same call split in two so that a caller can pipeline batches on two handles (one batch's uploads, rasterisation and
 * lookup lists overlap the other batch's sweep): _begin enqueues everything incl. the result read-back on the handle's
 * stream and returns; _end waits and hands the results out.  cov_in is only read for fine = 1 (may be NULL otherwise).
 * Host buffers handed to set_scans / add_scans / _begin must stay unchanged until _end returns when they are pinned
 * (uploads out of pinned memory are asynchronous). */
b2s_status b2s_matcher_correlate_scan_begin(b2s_matcher *m, const double *centers, const b2s_search *search,
                                            const b2s_match_result *cov_in);
b2s_status b2s_matcher_correlate_scan_end(b2s_matcher *m, b2s_match_result *results);

/* ScanMatcher::MatchScan (Mapper.cpp:184-291): coarse sweep (+ optional response expansion) + fine sweep.
 * Requires set_scans + add_scans (or set_grids). */
b2s_status b2s_matcher_match_scan(b2s_matcher *m, int do_penalize, int do_refine, b2s_match_result *results);

/* One-call host-buffer form (what a reference node's MatchScan call costs end to end):
 * set_scans + add_scans + match_scan. */
b2s_status b2s_matcher_match_scan_host(b2s_matcher *m, int batch, const double *ranges, const double *poses,
                                       int n_base, const double *base_ranges, const double *base_poses,
                                       int do_penalize, int do_refine, b2s_match_result *results);

/* A coarse CorrelateScan whose ANGLES are split over several GPUs (SURVEY.md §8(e)(ii)): every rank holds the same
 * scans + grids and sweeps angle indices [k_first, k_first + k_count).  Between the three phases the caller
 * all-reduces the small host arrays (NCCL via torch.distributed in creating-..._b200/parallel.py):
 *   begin : best[batch] (MAX), probs[batch][probs_len] per-cell maxima plane (MAX), status[batch] (MAX);
 *           probs_len = AlignValue(search_side, 8) * search_side
 *   ties  : global best in; tie_sums[batch][5] = {sum x, sum y, sum cos, sum sin, count} out (SUM)
 *   finish: global best / tie sums / plane in; results as b2s_matcher_correlate_scan (positional covariance incl.) */
b2s_status b2s_matcher_correlate_split_begin(b2s_matcher *m, const double *centers, const b2s_search *search, int k_first,
                                             int k_count, double *best, double *probs, int32_t *status);
b2s_status b2s_matcher_correlate_split_ties(b2s_matcher *m, const double *global_best, double *tie_sums);
b2s_status b2s_matcher_correlate_split_finish(b2s_matcher *m, const double *global_best, const double *tie_sums,
                                              const double *probs, b2s_match_result *results);

/* Inspection (parity tests; also ScanMatcher::GetCorrelationGrid, Mapper.h:1192). */
b2s_status b2s_matcher_get_grid(b2s_matcher *m, int b, uint8_t *out_bytes, double out_offset[2]);
b2s_status b2s_matcher_get_point_readings(b2s_matcher *m, int b, double *out_xy /* [n_readings][2] */);
/* GridIndexLookup::ComputeOffsets (Karto.h:6409-6501): out[n_angles][n_readings]; INT32_MAX = INVALID_SCAN */
b2s_status b2s_matcher_compute_offsets(b2s_matcher *m, int b, double angle_center, double angle_offset,
                                       double angle_res, int32_t *out, int32_t *out_n_angles);
/* integer numerators of GetResponse (Mapper.cpp:819-856) of the LAST correlate_scan sweep for match b,
 * in the reference's loop order out[nY][nX][nAngles] (Mapper.cpp:373-424). */
/* The angle-split sweep with the collectives INSIDE the library: nccl_comm is the caller's ncclComm_t (the library
 * dlopens libnccl.so.2 and calls ncclAllReduce on the handle's stream; no host staging, no Python).  Every rank calls
 * it with the same scans / grids / centres and its own rank; results are those of b2s_matcher_correlate_scan on
 * every rank.  Collectives: best response MAX (B doubles), per-cell plane MAX (B x probs_len doubles), status MAX,
 * tie sums SUM (5B doubles). */
b2s_status b2s_matcher_correlate_scan_split(b2s_matcher *m, void *nccl_comm, int rank, int world, const double *centers,
                                            const b2s_search *search, b2s_match_result *results);
/* ms of its last call: all-reduce(best), all-reduce(plane + status), all-reduce(tie sums), sweep end -> results */
b2s_status b2s_matcher_last_split_timing(b2s_matcher *m, double out[4]);
/* The whole integer response volume of the last sweep.  After a pruned sweep (b2s_matcher_last_prune_stats) the first
 * call sweeps every angle once more from the lookup lists the handle still holds. */
b2s_status b2s_matcher_get_response_sums(b2s_matcher *m, int b, int32_t *out, int32_t dims[3]);

/* Device time (ms, CUDA events on the handle's stream) of the stages of the LAST correlate_scan call:
 * out[0] = offsets/LUT, out[1] = response sweep (with the angle-pruning bound and select kernel when it runs),
 * out[2] = reduce (max / tie-average / covariance),
 * out[3] = number of sweep kernel launches. */
b2s_status b2s_matcher_last_timing(b2s_matcher *m, double out[4]);
/* Statistics of the LAST correlate_scan call: out[0] = fraction of (beam, angle) windows the window kernel dropped
 * because every cell of the nY x nX window lies in empty 4x4 blocks of the grid (they add 0 to every candidate, so
 * results are unchanged); out[1] = sweep path (1 generic, 2 window); out[2] = candidates per match; out[3] = beams. */
b2s_status b2s_matcher_last_stats(b2s_matcher *m, double out[4]);
/* Angle pruning of the LAST correlate_scan call: out[0] = fraction of (match, angle) pairs the window kernel swept,
 * out[1] = number of (match, angle) pairs swept.  A coarse-stage, stride-1 search of at most 32 x 32 cells whose grid
 * fits shared memory first bounds every (angle, 4x4 candidate block) from a max-pooled grid and sweeps only the angles
 * that can hold the best response, a tie or a cell the covariance reads; results are unchanged.  Without pruning
 * out = {1, batch x angles}. */
b2s_status b2s_matcher_last_prune_stats(b2s_matcher *m, double out[2]);
b2s_status b2s_matcher_sync(b2s_matcher *m);
/* 0 = automatic, 1 = force the generic global-memory gather kernel, 2 = force the shared-memory window kernel,
 * 3 = window kernel without dropping empty windows and without angle pruning (every beam and every angle is swept) */
b2s_status b2s_matcher_set_kernel(b2s_matcher *m, int which);

/* ---------------------------------------------------------------- lesson6 front end: karto::Mapper / MapperGraph
 * The host driver that feeds K1 (SURVEY.md §8(f).1): key-frame gate, running-scan window, sequential MatchScan,
 * pose-graph vertices / edges, near-chain links and loop-closure candidates (Mapper.cpp:883-1414, 1999-2125;
 * Mapper.h:1288-1404).  Every MatchScan runs on the device; independent matches of one Process call (all near
 * chains of LinkNearChains, all candidate chains of TryCloseLoop up to the first accepted closure) go out as ONE
 * batch.  Several sensors (robots) may feed one mapper: b2s_mapper_process_sensor (MapperSensorManager semantics, the
 * first-scan linking of Mapper.cpp:920-952 included). */

/* Values as the Mapper STORES them (Mapper.cpp:1448-1653); the setParam* squaring of distance_variance_penalty,
 * angle_variance_penalty and loop_match_maximum_variance_coarse (Mapper.cpp:1871-1874,1919-1927) is the caller's job. */
typedef struct b2s_mapper_params {
  int32_t use_scan_matching;                 /* true */
  int32_t use_scan_barycenter;               /* true */
  double minimum_time_interval;              /* 3600 s */
  double minimum_travel_distance;            /* 0.2 m */
  double minimum_travel_heading;             /* 10 deg in rad */
  int32_t scan_buffer_size;                  /* 70 */
  int32_t do_loop_closing;                   /* true */
  double scan_buffer_maximum_scan_distance;  /* 20 m */
  double link_match_minimum_response_fine;   /* 0.8 */
  double link_scan_maximum_distance;         /* 10 m */
  double loop_search_maximum_distance;       /* 4 m */
  int32_t loop_match_minimum_chain_size;     /* 10 */
  int32_t reserved;
  double loop_match_maximum_variance_coarse; /* 0.4^2 */
  double loop_match_minimum_response_coarse; /* 0.8 */
  double loop_match_minimum_response_fine;   /* 0.8 */
  b2s_matcher_params sequential;             /* CorrelationSearchSpace* 0.3 / 0.01 / 0.03 + the shared tuning values */
  b2s_matcher_params loop;                   /* LoopSearchSpace* 8.0 / 0.05 / 0.03 + the same tuning values */
} b2s_mapper_params;

/* Mapper::InitializeParameters defaults (Mapper.cpp:1448-1653); range_threshold of both matchers = the laser's */
void b2s_mapper_default_params(b2s_mapper_params *out, double range_threshold);

/* The matcher plug-in: ScanMatcher::MatchScan (Mapper.cpp:184-291) for a batch of independent matches.
 * which = 0 the sequential matcher (Mapper::m_pSequentialScanMatcher), 1 the loop matcher
 * (MapperGraph::m_pLoopScanMatcher).  ranges [batch][N], poses [batch][3] (robot poses); the base scans of match b are
 * base_ranges/base_poses[base_first[b] .. base_first[b] + n_base[b]).  The in-tree implementation is the CUDA matcher
 * (b2s_mapper_create); the hook exists so that the graph logic can be exercised without a device. */
typedef b2s_status (*b2s_match_scan_fn)(void *user, int which, int batch, const double *ranges, const double *poses,
                                        const int32_t *base_first, const int32_t *n_base, const double *base_ranges,
                                        const double *base_poses, int do_penalize, int do_refine,
                                        b2s_match_result *results);

/* karto::ScanSolver (Mapper.h:825-891) as a C vtable — the reference's own back-end plug-in interface. */
typedef struct b2s_scan_solver {
  void *user;
  void (*add_node)(void *user, int32_t unique_id, const double corrected_pose[3]);          /* AddNode */
  void (*add_constraint)(void *user, int32_t source_id, int32_t target_id, const double pose_difference[3],
                         const double covariance[9]);                                       /* AddConstraint(LinkInfo) */
  int32_t (*compute)(void *user, int32_t capacity, int32_t *ids, double *poses /* [capacity][3] */);
                                                                                             /* Compute + GetCorrections */
  void (*clear)(void *user);                                                                /* Clear */
} b2s_scan_solver;

typedef struct b2s_mapper b2s_mapper; /* opaque: replaces karto::Mapper (+ MapperGraph, MapperSensorManager) */

b2s_status b2s_mapper_create(const b2s_mapper_params *params, const b2s_laser *laser, int device, b2s_mapper **out);
b2s_status b2s_mapper_create_with_matcher(const b2s_mapper_params *params, const b2s_laser *laser,
                                          b2s_match_scan_fn match, void *user, b2s_mapper **out);
void b2s_mapper_destroy(b2s_mapper *m);
/* Mapper::SetScanSolver (Mapper.cpp:2220); NULL = no back end (poses are never corrected, as with use_back_end false) */
b2s_status b2s_mapper_set_scan_solver(b2s_mapper *m, const b2s_scan_solver *solver);
/* Mapper::Process(LocalizedRangeScan*) (Mapper.cpp:1999-2079): ranges[n_readings], odometric robot pose, time stamp (s).
 * out_processed = the kt_bool it returns (false: rejected by HasMovedEnough); out_corrected_pose = GetCorrectedPose().
 * A non-OK status returned after the scan entered the graph (edge building / loop closing failed: CUDA error,
 * B2S_ERR_NO_BEST_POSE, or B2S_ERR_BAD_STATE where the reference's Matrix3::Inverse asserts) leaves the mapper where
 * the reference process would have aborted: the handle is marked failed, later calls return B2S_ERR_BAD_STATE, and it
 * must be destroyed. */
b2s_status b2s_mapper_process(b2s_mapper *m, const double *ranges, const double odometric_pose[3], double time,
                              int32_t *out_processed, double out_corrected_pose[3]);
/* The same for a scan of the NAMED sensor (LocalizedRangeScan::GetSensorName; karto_slam.cc passes the laser frame id).
 * MapperSensorManager semantics (Mapper.h:1412-1577, Mapper.cpp:45-100): a sensor is registered by its first scan; each
 * sensor has its own scan list (state ids), running window and last scan, unique ids count over all sensors; a sensor's
 * first scan is matched against ALL scans of every other sensor (name order = Name::operator<, Karto.h:484) and linked
 * to that sensor's first scan (Mapper.cpp:920-952); near chains follow the near scan's own sensor and loop closures are
 * searched against every sensor's scans in name order (Mapper.cpp:2063-2070).  All sensors share the handle's b2s_laser
 * (same LaserRangeFinder parameters on every robot).  b2s_mapper_process is this call with the name "laser". */
b2s_status b2s_mapper_process_sensor(b2s_mapper *m, const char *sensor_name, const double *ranges,
                                     const double odometric_pose[3], double time, int32_t *out_processed,
                                     double out_corrected_pose[3]);
int32_t b2s_mapper_sensor_count(const b2s_mapper *m);
/* per processed scan (unique-id order): the rank of its sensor in name order, [count] */
b2s_status b2s_mapper_get_scan_sensors(const b2s_mapper *m, int32_t *out);
int32_t b2s_mapper_scan_count(const b2s_mapper *m);   /* GetAllProcessedScans().size() */
/* corrected poses of every processed scan in unique-id order, [count][3] (they move when a loop closes and a solver is
 * set) */
b2s_status b2s_mapper_get_poses(const b2s_mapper *m, double *out);
int32_t b2s_mapper_edge_count(const b2s_mapper *m);
/* graph edges in creation order: ids [count][2] (source, target), LinkInfo pose difference [count][3] and covariance
 * [count][9] (Mapper.h:108-175) */
b2s_status b2s_mapper_get_edges(const b2s_mapper *m, int32_t *ids, double *pose_difference, double *covariance);
/* out[0] = MatchScan calls so far, out[1] = device batches they were sent in, out[2] = loop-closure candidate chains
 * examined, out[3] = loops closed, out[4] = running-scan window size of the sensor processed last */
b2s_status b2s_mapper_stats(const b2s_mapper *m, double out[5]);

/* ---------------------------------------------------------------- back end: a ScanSolver for the mapper (host only)
 * SURVEY.md §8(f).3: the reference's back ends (sparse bundle adjustment / g2o / Ceres / GTSAM, lesson6/src/<name>_solver)
 * need Eigen + SuiteSparse and stay on the CPU in every BASELINE config.  This is a small dependency-free 2-D pose-graph
 * optimiser with the same role: nodes = scan poses, constraints = LinkInfo pose differences weighted by the inverse
 * covariance (lesson6/src/spa_solver/spa_solver.cc:65-93), Levenberg-Marquardt outer loop, block-Jacobi preconditioned
 * conjugate gradients inside, first node fixed.  It is NOT a restatement of sba::SysSPA2d (parity unpinned: that
 * library is not under /root/reference); tests plug the SAME solver into the reference Mapper and into ours. */
typedef struct b2s_pose_graph b2s_pose_graph;
b2s_status b2s_pose_graph_create(b2s_pose_graph **out);
void b2s_pose_graph_destroy(b2s_pose_graph *g);
/* fills `out` with callbacks bound to `g` (valid while g lives): pass it to b2s_mapper_set_scan_solver */
b2s_status b2s_pose_graph_as_scan_solver(b2s_pose_graph *g, b2s_scan_solver *out);
/* SpaSolver::Compute runs doSPA(40) (spa_solver.cc:44-63): max LM iterations (default 40), PCG iterations per step */
b2s_status b2s_pose_graph_set_iterations(b2s_pose_graph *g, int lm_iterations, int cg_iterations);
/* out[0] = nodes, out[1] = constraints, out[2] = chi^2 before the last Compute, out[3] = after, out[4] = LM steps taken */
b2s_status b2s_pose_graph_stats(const b2s_pose_graph *g, double out[5]);

/* ---------------------------------------------------------------- K2c: karto::OccupancyGrid */

typedef struct b2s_occ_grid_info {
  int32_t width, height, width_step, data_size;
  double offset[2];  /* CoordinateConverter offset = bounding-box minimum (Karto.h:5821) */
  double resolution;
  uint64_t cell_visits; /* Bresenham cells touched incl. end cells (SURVEY.md §8(d) V) */
} b2s_occ_grid_info;

typedef struct b2s_occ_grid b2s_occ_grid; /* opaque: replaces karto::OccupancyGrid* */

/* OccupancyGrid::CreateFromScans (Karto.h:5659-5673, 5804-5990): n_scans x (ranges, robot pose).
 * Returns B2S_OK with *out == NULL when n_scans == 0 (the reference returns NULL). */
b2s_status b2s_occ_grid_create_from_scans(const b2s_laser *laser, int n_scans, const double *ranges,
                                          const double *poses, double resolution, int device,
                                          void *cuda_stream, b2s_occ_grid **out);
/* The same map built from a scan list SHARDED over several GPUs (SURVEY.md §8(e)(iii)): pass/hit counters are
 * commutative, so each rank ray-traces its shard into a grid sized by the GLOBAL bounding box and the counters are
 * summed (NCCL all-reduce, in place on the device pointers) before OccupancyGrid::Update thresholds them.
 *   1. b2s_occ_grid_scans_bbox  -> this shard's BoundingBox2 {min x, min y, max x, max y} (Karto.h:5810-5814);
 *                                  the caller reduces MIN on [0..1], MAX on [2..3] over the ranks
 *   2. b2s_occ_grid_create_shard -> grid dimensioned by the global box (ComputeDimensions, Karto.h:5816-5821),
 *                                  counters = this shard's rays; n_scans may be 0
 *   3. b2s_occ_grid_device_counters (all-reduce SUM on both) or b2s_occ_grid_set_counters (host arrays)
 *   4. b2s_occ_grid_update       -> cells from the summed counters (OccupancyGrid::Update, Karto.h:5953-5968) */
b2s_status b2s_occ_grid_scans_bbox(const b2s_laser *laser, int n_scans, const double *ranges, const double *poses,
                                   int device, void *cuda_stream, double bbox[4]);
b2s_status b2s_occ_grid_create_shard(const b2s_laser *laser, int n_scans, const double *ranges, const double *poses,
                                     double resolution, const double bbox[4], int device, void *cuda_stream,
                                     b2s_occ_grid **out);
b2s_status b2s_occ_grid_device_counters(b2s_occ_grid *g, uint32_t **d_pass, uint32_t **d_hit);
b2s_status b2s_occ_grid_set_counters(b2s_occ_grid *g, const uint32_t *pass, const uint32_t *hit);
/* step 3 with the collective inside the library: ncclAllReduce(SUM) of both counter planes in place through the caller's
 * ncclComm_t (dlopened libnccl.so.2), on the grid's stream */
b2s_status b2s_occ_grid_allreduce_counters(b2s_occ_grid *g, void *nccl_comm);
b2s_status b2s_occ_grid_update(b2s_occ_grid *g);
b2s_status b2s_occ_grid_info_get(const b2s_occ_grid *g, b2s_occ_grid_info *out);
/* cells: uint8 {0 unknown, 100 occupied, 255 free}; pass/hit: uint32 counters; any pointer may be NULL */
b2s_status b2s_occ_grid_copy(b2s_occ_grid *g, uint8_t *cells, uint32_t *pass, uint32_t *hit);
/* nav_msgs/OccupancyGrid payload as SlamKarto::updateMap fills it (karto_slam.cc:546-569):
 * int8 {-1,100,0}, row-major width x height (no width_step padding) */
b2s_status b2s_occ_grid_copy_ros(b2s_occ_grid *g, int8_t *out);
b2s_status b2s_occ_grid_last_timing(b2s_occ_grid *g, double out[2]); /* ms: ray-trace kernel, threshold kernel */
void b2s_occ_grid_destroy(b2s_occ_grid *g);

/* ---------------------------------------------------------------- K2a / K3: Hector log-odds grid map */

typedef struct b2s_hector_map b2s_hector_map; /* opaque: replaces hectorslam::GridMap (OccGridMapP) */

/* GridMap(mapResolution, size, offset) (GridMapBase.h:54-66, MapRepMultiMap.h:63-67): size x size cells,
 * start_x/start_y in [0,1] (fraction of the map at which the world origin sits). */
b2s_status b2s_hector_map_create(int size_x, int size_y, float resolution, float start_x, float start_y,
                                 int device, void *cuda_stream, b2s_hector_map **out);
void b2s_hector_map_destroy(b2s_hector_map *m);
/* GridMapLogOddsFunctions::setUpdateFreeFactor / setUpdateOccupiedFactor (GridMapLogOdds.h:116-134) */
b2s_status b2s_hector_map_set_factors(b2s_hector_map *m, float update_free, float update_occupied);
/* OccGridMapBase::updateByScan (OccGridMapBase.h:118-168): points are the DataContainer in map-cell units
 * ([n][2] float, already scaled by 1/resolution as hector_slam.cc:320-362 does), origo = sensor origin in the
 * same frame, pose = robot pose in WORLD coordinates (x, y, heading). */
b2s_status b2s_hector_map_update_by_scan(b2s_hector_map *m, const float *points, int n_points,
                                         const float origo[2], const float world_pose[3]);
/* OccGridMapBase::updateByScanJustOnce (OccGridMapBase.h:175-217), the make-map demo variant of lesson4
 * (hector_mapping/src/hector_mapping/...: map pose fixed at cell (800, 800), heading 0; points in METRES, the end cell is
 * begin + (int)round(p / 0.05)). */
b2s_status b2s_hector_map_update_by_scan_just_once(b2s_hector_map *m, const float *points, int n_points,
                                                   const float origo[2]);
/* ScanMatcher::matchData (ScanMatcher.h:60-98) on ONE grid level: Gauss-Newton scan-to-map alignment.
 * begin_world_pose in, new world pose + 3x3 Hessian ("covariance") out. */
b2s_status b2s_hector_map_match_data(b2s_hector_map *m, const float *points, int n_points,
                                     const float begin_world_pose[3], int max_iterations,
                                     float out_world_pose[3], float out_cov[9]);
/* raw cells: logOdds float + updateIndex int per cell (GridMapLogOdds.h:37-75) */
b2s_status b2s_hector_map_copy(b2s_hector_map *m, float *log_odds, int32_t *update_index);
/* nav_msgs/OccupancyGrid payload as HectorMappingRos::publishMap does (hector_slam.cc:254-317) */
b2s_status b2s_hector_map_copy_ros(b2s_hector_map *m, int8_t *out);
b2s_status b2s_hector_map_last_timing(b2s_hector_map *m, double out[2]);

/* ---------------------------------------------------------------- lesson4 front end: HectorSlamProcessor
 * One call per LaserScan = MapRepMultiMap::matchData (coarse-to-fine Gauss-Newton over all pyramid levels) + the
 * map-update gate + MapRepMultiMap::updateByScan (all levels) — all on the device: the processor's state (last poses,
 * update indices, the coarse levels' data containers) is device-resident, one cooperative launch does match + gate +
 * update, and the pose returns through a host-mapped mailbox as soon as the match is done.  A whole stream of scans can
 * be handed over at once (b2s_hector_slam_process_stream: no host round trip between scans), and a handle may hold B
 * independent processors (b2s_hector_slam_create_batch).
 * EXACT mode (default): bit-identical poses, Hessians and cells to the reference (sequential float32 sums in point
 * order, glibc's sinf / cosf restated on the device); b2s_hector_slam_set_exact(p, 0) sums with a tree instead and
 * spreads the per-point phase of the match over a 4-CTA cluster (faster; poses within 1e-4). */

typedef struct b2s_hector_slam b2s_hector_slam; /* opaque: replaces hectorslam::HectorSlamProcessor
                                                   (slam_main/HectorSlamProcessor.h:50-150) */

#define B2S_HECTOR_MAX_LEVELS 8

/* HectorSlamProcessor(mapResolution, mapSizeX, mapSizeY, startCoords, multi_res_size) (HectorSlamProcessor.h:56-65):
 * level l has cell length resolution * 2^l and size >> l cells; every level shares the level-0 offset
 * (MapRepMultiMap.h:56-89).  Defaults as the constructor sets them: update factors 0.4 / 0.6
 * (GridMapLogOdds.h:98-102), map-update gate 0.4 m / 0.13 rad. */
b2s_status b2s_hector_slam_create(float map_resolution, int map_size_x, int map_size_y, float start_x, float start_y,
                                  int levels, int device, void *cuda_stream, b2s_hector_slam **out);
void b2s_hector_slam_destroy(b2s_hector_slam *p);
/* setUpdateFactorFree / setUpdateFactorOccupied (HectorSlamProcessor.h:128-129) */
b2s_status b2s_hector_slam_set_update_factors(b2s_hector_slam *p, float update_free, float update_occupied);
/* setMapUpdateMinDistDiff / setMapUpdateMinAngleDiff (HectorSlamProcessor.h:130-131).  The gate is
 * util::poseDifferenceLargerThan (UtilFunctions.h:72-90), including its integer-truncating abs() on the angle. */
b2s_status b2s_hector_slam_set_map_update_min_diff(b2s_hector_slam *p, float min_dist, float min_angle);
/* reset() (HectorSlamProcessor.h:111-116): clears every level and the last poses */
b2s_status b2s_hector_slam_reset(b2s_hector_slam *p);
/* update(dataContainer, poseHintWorld, map_without_matching) (HectorSlamProcessor.h:81-108).  points = the
 * DataContainer in LEVEL-0 map-cell units ([n][2] float, as hector_slam.cc:320-362 fills it), origo likewise, pose
 * hint in world coordinates.  out_pose = getLastScanMatchPose(); out_cov (may be NULL) = getLastScanMatchCovariance()
 * (the level-0 Hessian; untouched when map_without_matching).  out_map_updated (may be NULL) tells whether the gate
 * let this scan into the maps. */
b2s_status b2s_hector_slam_update(b2s_hector_slam *p, const float *points, int n_points, const float origo[2],
                                  const float pose_hint_world[3], int map_without_matching, float out_pose[3],
                                  float out_cov[9], int *out_map_updated);
/* getMapLevels / getGridMap(level) (HectorSlamProcessor.h:124-125) */
b2s_status b2s_hector_slam_level_dims(b2s_hector_slam *p, int level, int dims[2], float *cell_length);
b2s_status b2s_hector_slam_copy_level(b2s_hector_slam *p, int level, float *log_odds, int32_t *update_index);
/* nav_msgs/OccupancyGrid payload of one level as HectorMappingRos::publishMap fills it (hector_slam.cc:254-317) */
b2s_status b2s_hector_slam_copy_level_ros(b2s_hector_slam *p, int level, int8_t *out);
/* out[0] = scans matched, out[1] = scans let into the maps, out[2] = Bresenham cell visits so far (all levels; summed
 * over the processors of a batched handle), out[3] / out[4] = ms of processor 0's last match / update (device timer) */
b2s_status b2s_hector_slam_stats(b2s_hector_slam *p, double out[5]);
/* 1 (default) = the reference's arithmetic bit for bit; 0 = the nine Gauss-Newton sums are tree-reduced instead of
 * accumulated in point order (everything else unchanged): faster, poses agree to ~1e-6 m */
b2s_status b2s_hector_slam_set_exact(b2s_hector_slam *p, int exact);
/* Non-exact mode, single-processor handles: the CTAs of one thread-block cluster share the per-point phase of every
 * Gauss-Newton iteration (pose out / nine partial sums back through distributed shared memory).  Returns the CTAs per
 * cluster in use (1: no cluster launch — the device cannot co-schedule the grid as clusters, or refused the launch). */
int32_t b2s_hector_slam_match_cluster_size(const b2s_hector_slam *p);
/* The node's loop over a recorded stream (hector_slam.cc:195-204: update(container, getLastScanMatchPose())) in ONE
 * call: n_scans scans, points concatenated ([sum n_points][2], level-0 map-cell units), hint of scan i = pose of scan
 * i-1 (first_pose_hint for scan 0; NULL = the processor's current last scan-match pose), or pose_hints[i] when given
 * (required with map_without_matching).  out_poses [n_scans][3]; out_map_updated [n_scans] and out_last_cov[9] may be
 * NULL.  Identical results to n_scans b2s_hector_slam_update calls. */
b2s_status b2s_hector_slam_process_stream(b2s_hector_slam *p, int n_scans, const float *points, const int32_t *n_points,
                                          const float origo[2], const float *first_pose_hint, const float *pose_hints,
                                          int map_without_matching, float *out_poses, int32_t *out_map_updated,
                                          float *out_last_cov);
/* B independent HectorSlamProcessors (robots / maps) behind one handle (SURVEY.md §8(e): Hector maps shard over
 * independent maps, not within one).  max_points = capacity of one scan (<= 4096). */
b2s_status b2s_hector_slam_create_batch(int batch, int max_points, float map_resolution, int map_size_x, int map_size_y,
                                        float start_x, float start_y, int levels, int device, void *cuda_stream,
                                        b2s_hector_slam **out);
/* update() of every processor with its own scan: points [B][max_points][2] (rows padded), n_points [B], pose_hints
 * [B][3] (NULL = each processor's last scan-match pose); out_poses [B][3], out_covs [B][9] / out_map_updated [B] may
 * be NULL. */
b2s_status b2s_hector_slam_update_batch(b2s_hector_slam *p, const float *points, const int32_t *n_points,
                                        const float origo[2], const float *pose_hints, int map_without_matching,
                                        float *out_poses, float *out_covs, int32_t *out_map_updated);
/* the same step on scans already in device memory (DEVICE pointers; asynchronous on the handle's stream, nothing
 * returned to the host; max_n = upper bound of n_points): the resident-in-HBM form */
b2s_status b2s_hector_slam_update_batch_device(b2s_hector_slam *p, const float *d_points, const int32_t *d_n_points,
                                               int max_n, const float origo[2], const float *d_pose_hints,
                                               int map_without_matching);
b2s_status b2s_hector_slam_sync(b2s_hector_slam *p);
b2s_status b2s_hector_slam_copy_level_of(b2s_hector_slam *p, int processor, int level, float *log_odds,
                                         int32_t *update_index);
/* getLastScanMatchPose / getLastMapUpdatePose (HectorSlamProcessor.h:118-119) of one processor; either may be NULL */
b2s_status b2s_hector_slam_last_poses(b2s_hector_slam *p, int processor, float last_scan_match_pose[3],
                                      float last_map_update_pose[3]);
/* test hook: pretend `updates` map updates already consumed per-scan stamp epochs (exercises the 20-bit epoch wrap) */
b2s_status b2s_hector_slam_debug_set_epoch(b2s_hector_slam *p, unsigned int updates);

/* ---------------------------------------------------------------- ROS-shaped input adapters (host only; SURVEY.md §8(f).4)
 * The wire formats either side of the path: sensor_msgs/LaserScan in (here), nav_msgs/OccupancyGrid payloads out
 * (b2s_occ_grid_copy_ros, b2s_hector_map_copy_ros / b2s_hector_slam_copy_level_ros, b2s_gmap_copy_ros).  ROS itself is
 * out of scope; these are the conversions the lesson nodes perform on the message fields. */
typedef struct b2s_laser_scan_msg { /* the sensor_msgs/LaserScan fields the nodes read */
  float angle_min, angle_max, angle_increment, range_min, range_max;
  int32_t n_ranges;
  const float *ranges;
} b2s_laser_scan_msg;
/* SlamKarto::getLaser (lesson6/src/karto_slam.cc:323-395): the Custom LaserRangeFinder made from the first scan —
 * angles / ranges from the message, offset = laser pose in base_link (x, y, yaw), range threshold clipped into
 * [range_min, range_max] (Karto.h:3778-3787), n_readings = Round((max - min) / resolution) WITHOUT + 1
 * (LaserRangeFinder::Update, Karto.h:4152-4161).  Returns B2S_ERR_BAD_PARAMS if the message carries a different
 * number of ranges than that (LaserRangeFinder::Validate would reject every scan). */
b2s_status b2s_ros_karto_laser(const b2s_laser_scan_msg *scan, const double laser_pose_in_base[3], double use_scan_range,
                               b2s_laser *out);
/* SlamKarto::addScan (karto_slam.cc:407-434): float32 ranges -> kt_double readings, in reverse order for a laser
 * mounted upside-down (lasers_inverted_) */
b2s_status b2s_ros_karto_readings(const b2s_laser_scan_msg *scan, int inverted, double *out_readings);
/* HectorMappingRos::rosPointCloudToDataContainer (lesson4/src/hector_mapping/hector_slam.cc:320-362): laser-frame points
 * ([n][3] float x, y, z as laser_geometry projected them) -> DataContainer entries in map-cell units.  laser_in_base =
 * (x, y, z, yaw) of the laser in base_link.  Filters: squared distance in (min_dist^2, max_dist^2), not behind the robot
 * within 0.5 m^2, not beyond use_max_scan_range, height window (z_min, z_max).  out_points [n][2] (capacity n),
 * out_origo[2] = laser position * scale_to_map.  Returns the number of points kept in *out_n. */
b2s_status b2s_ros_hector_points(const float *points_xyz, int n, const float laser_in_base[4], float scale_to_map,
                                 float min_dist, float max_dist, double use_max_scan_range, float z_min, float z_max,
                                 float *out_points, float out_origo[2], int32_t *out_n);

/* ---------------------------------------------------------------- K2b: GMapping hit/visit map */

typedef struct b2s_gmap b2s_gmap; /* opaque: replaces GMapping::ScanMatcherMap (gmapping.cc:135) */

/* ScanMatcherMap(center, xmin, ymin, xmax, ymax, delta) (map.h:117-140): note the (cells >> 5) patch rounding. */
b2s_status b2s_gmap_create(double center_x, double center_y, double xmin, double ymin, double xmax, double ymax,
                           double delta, int device, void *cuda_stream, b2s_gmap **out);
void b2s_gmap_destroy(b2s_gmap *g);
b2s_status b2s_gmap_size(const b2s_gmap *g, int32_t size_xy[2]);
/* GMapping::ComputeMap (gmapping.cc:171-242) for one scan: ranges[n], angles[n] (beam angles in the laser
 * frame), laser pose in world, max_range / max_urange. */
b2s_status b2s_gmap_compute_map(b2s_gmap *g, const double *ranges, const double *angles, int n,
                                const double laser_pose[3], double max_range, double max_urange);
/* PointAccumulator per cell (map.h:17-48): n, visits, acc.x, acc.y */
b2s_status b2s_gmap_copy(b2s_gmap *g, int32_t *n, int32_t *visits, float *acc_x, float *acc_y);
/* the published map (gmapping.cc:141-159): -1 unknown, 100 if n/visits > 0.25 else 0 */
b2s_status b2s_gmap_copy_ros(b2s_gmap *g, int8_t *out);

/* ---------------------------------------------------------------- K3 (lesson3): PL-ICP fine alignment */

/* The subset of CSM's sm_params the reference sets (lesson3/src/plicp_odometry.cc:72-185), defaults in comments. */
typedef struct b2s_icp_params {
  double max_angular_correction_deg; /* 45 */
  double max_linear_correction;      /* 1.0 m (the node's yaml default; CSM's is 0.5) */
  double epsilon_xy;                 /* 1e-6 */
  double epsilon_theta;              /* 1e-6 */
  double max_correspondence_dist;    /* 1.0 m */
  double outliers_maxPerc;           /* 0.90 */
  double outliers_adaptive_order;    /* 0.7 */
  double outliers_adaptive_mult;     /* 2.0 */
  int32_t max_iterations;            /* 10 */
  int32_t use_point_to_line_distance;/* 1 */
  int32_t outliers_remove_doubles;   /* 1 */
  int32_t reserved;
} b2s_icp_params;

typedef struct b2s_icp_result {
  double x[3];        /* sm_result.x: pose of the current scan in the reference scan's frame (plicp_odometry.cc:399-403) */
  double error;       /* sum of point-to-segment distances of the kept correspondences */
  int32_t valid;      /* sm_result.valid */
  int32_t iterations;
  int32_t nvalid;     /* correspondences kept in the last iteration */
  int32_t reserved;
} b2s_icp_result;

/* sm_icp (plicp_odometry.cc:391) for `batch` independent scan pairs: ref_ranges / sens_ranges [batch][n] on the beam
 * angles theta[n] (LaserScanToLDP, :285-322: a reading is valid iff range_min < r < range_max), first_guess [batch][3].
 * PARITY UNPINNED: CSM is an external, un-versioned dependency absent from the reference tree; this follows the
 * published algorithm (Censi, ICRA 2008) — see DESIGN.md §7. */
b2s_status b2s_plicp_match(const b2s_icp_params *params, int batch, int n, const double *ref_ranges,
                           const double *sens_ranges, const double *theta, double range_min, double range_max,
                           const double *first_guess, int device, void *cuda_stream, b2s_icp_result *results);

/* ---------------------------------------------------------------- lesson5: motion de-skew pre-stage (SURVEY.md §8(f).4)
 * LidarUndistortion (lesson5/src/lidar_undistortion.cc): every reading of a LaserScan is moved into the sensor frame
 * of the scan's first valid reading, using IMU angles integrated over the scan and the odometry increment across it.
 * The per-beam loop (CorrectLaserScan, :339-393) runs on the device for a batch of scans; the per-scan preparation is
 * host arithmetic.  PARITY UNPINNED: pcl::getTransformation and Eigen::Affine3f inverse / product are third-party
 * header code absent from the reference tree (PCL 1.8, Eigen 3.3); their published algorithms are restated. */
typedef struct b2s_deskew_scan {
  double time_start, time_increment;   /* header.stamp (start of the sweep), LaserScan::time_increment */
  float range_min, range_max;          /* readings outside [range_min, range_max] or non-finite are skipped (:349-352) */
  int32_t use_imu, use_odom;           /* the node's use_imu_ / use_odom_ */
  int32_t imu_last, reserved;          /* current_imu_index_ after PruneImuDeque: index of the last table entry */
  double odom_start_time, odom_end_time; /* stamps of start_odom_msg_ / end_odom_msg_ */
  float odom_incre[3];                 /* odom_incre_x_/y_/z_ */
  float reserved2;
} b2s_deskew_scan;

/* PruneImuDeque's integration (:196-238) over the IMU messages of the (already pruned) queue: stamp[n_imu],
 * angular_velocity[n_imu][3]; fills imu_time / rot_x / rot_y / rot_z [capacity] (zeroed first, as ResetParameters does)
 * and returns current_imu_index_ (the last entry), or -2 where the node would run outside its arrays. */
int32_t b2s_deskew_integrate_imu(int n_imu, const double *stamp, const double *angular_velocity, double scan_time_start,
                                 double scan_time_end, int capacity, double *imu_time, double *rot_x, double *rot_y,
                                 double *rot_z);
/* PruneOdomDeque's increment (:296-333): start / end pose as (x, y, z, roll, pitch, yaw) — the position of the
 * odometry message and tf::Matrix3x3(orientation).getRPY — gives odom_incre_x_/y_/z_. */
void b2s_deskew_odom_increment(const double start_pose[6], const double end_pose[6], float out_increment[3]);
/* CorrectLaserScan for `batch` scans: ranges [batch][n_beams] (host), beam angles angle_min + i * angle_increment
 * (CreateAngleCache, :160-172), per-scan parameters, IMU tables [batch][imu_stride]; out_xyz [batch][n_beams][3] (host):
 * the corrected point cloud, skipped readings as (0, 0, 0) (the cloud is cleared and resized per scan). */
b2s_status b2s_lidar_undistort(int batch, int n_beams, const float *ranges, double angle_min, double angle_increment,
                               const b2s_deskew_scan *scans, const double *imu_time, const double *imu_rot_x,
                               const double *imu_rot_y, const double *imu_rot_z, int imu_stride, float *out_xyz, int device,
                               void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SLAM_H */

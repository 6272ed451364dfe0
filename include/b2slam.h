/*
 * b2slam C ABI -- the drop-in boundary of the B200-native ICP / occupancy-grid hot path.
 *
 * The reference (zjwzcx/A-2D-LiDAR-based-SLAM-System-for-Wheeled-Mobile-Robots) has no FFI
 * layer: its boundary is the Python class API of course_agv_slam/scripts/{icp,mapping,
 * bresenham}.py (SURVEY.md section 8b).  Each entry point below names the reference
 * interface it replaces (paths relative to the reference root):
 *   [ICP]  W9_Fusion Localization (LiDAR Odometry)/course_agv_slam/scripts/icp.py
 *   [MAP]  W12_LiDAR SLAM/w12-mapping/course_agv_slam/scripts/mapping.py
 *   [MAPO] W12_LiDAR SLAM/w12-mapping-online/course_agv_slam/scripts/mapping.py
 *   [BRES] W12_LiDAR SLAM/w12-mapping/course_agv_slam/scripts/bresenham.py
 *   [SLAM] W12_LiDAR SLAM/w12-mapping/course_agv_slam/scripts/slam_ekf.py
 *
 * Two layers:
 *   layer 1  b2s_*            device pointers, asynchronous on the given CUDA stream
 *   layer 2  b2s_icp_* / b2s_mapping_*  host buffers in, host buffers out (the calls the
 *            Python classes ICP / Mapping make); copies and kernels run on the object's stream
 *
 * All functions return 0 (B2S_OK) or a negative status; b2s_last_error() gives the detail.
 * Plain pointers and sizes only; there is no CPU fallback -- without a CUDA device every
 * compute entry point returns B2S_ERR_CUDA.
 */
#ifndef B2SLAM_H
#define B2SLAM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2S_OK 0
#define B2S_ERR_INVALID_ARG (-1) /* bad shape / null pointer / negative size */
#define B2S_ERR_NONFINITE (-2)   /* NaN/inf coordinate the reference raises ValueError/OverflowError on */
#define B2S_ERR_CUDA (-3)        /* CUDA runtime error or no device */
#define B2S_ERR_TOO_LONG (-4)    /* a beam longer than B2S_MAX_PATH_CELLS cells */
#define B2S_ERR_NCCL (-5)        /* NCCL missing or failed */
#define B2S_ERR_NOMEM (-6)

#define B2S_MAX_PATH_CELLS (1 << 22)

/* index into the optional device counters of b2s_grid_raycast */
#define B2S_CNT_NONFINITE 0 /* beams dropped: a NaN coordinate (int(nan) -> ValueError in the reference) */
#define B2S_CNT_TOO_LONG 1  /* beams dropped: longer than B2S_MAX_PATH_CELLS */
#define B2S_CNT_SKIPPED_INF 2 /* beams skipped because ox is +-inf ([MAP]:30), not an error */
#define B2S_CNT_OVERFLOW 3  /* beams dropped: inf in oy or the sensor position (int(inf) -> OverflowError) */
#define B2S_CNT_WORDS 4

int b2s_version(void);
const char *b2s_status_string(int status);
const char *b2s_last_error(void); /* thread-local, valid until the next call on this thread */
int b2s_device_count(int *count);
/* Kernel-variant switch for benchmarking.  Keys: "grid_variant" 1 = one RED per visit, 2 = warp-aggregated
 * runs, 3 = lean loop, 4 = transposed scratch plane, 5 = 4 + test-free core phase, 6 = consecutive scans counted
 * in a shared-memory tile, 5 where the tile does not fit (default; 4..6 need a workspace, else 3; a roll-back runs 5);
 * "grid_tile_layout" (variant 6) 0 = 1024 threads, one 32-beam unit per warp, 1 = 512 threads, two units per warp,
 * longest paired with shortest (default); "icp_prune"
 * 0 = brute force, 1 = per-lane block pruning, 2 = warp-level + per-lane with whole-warp block visits,
 * 3 = warp-level only, 4 = both tests, surviving (point, block) pairs queued and spread over the lanes
 * (default); "icp_block" 0 (automatic) / 8 / 16 / 32 targets per pruning block; "icp_layout" 0 strided /
 * 1 balanced / 2 automatic point groups per warp; "icp_src_per_thread" 0 (automatic) / 2 / 3 / 4; "icp_graph" 0 / 1
 * (single-pair calls replay a captured CUDA graph); "h2d_chunks" 0 (automatic) .. 16 pipeline depth of the
 * host-buffer calls.  Not part of the reference surface; process-global, set it before the calls it should
 * affect (cached single-pair graphs are re-captured after a change). */
int b2s_tune(const char *key, int value);
/* Same-run FP64 FMA issue peak of the current device in TFLOP/s (8 independent DFMA chains per thread);
 * bench.py quotes the ICP kernel against it.  Not part of the reference surface. */
int b2s_measure_fp64_peak(double *tflops_out);

/* ===================================================================== layer 1: device */

/* ICP.process for a batch of independent scan pairs -- replaces [ICP]:38-88 (and through it
 * findNearest [ICP]:90-114 and getTransform [ICP]:149-179).
 *   tar_xy [pairs][2][n_tar], src_xy [pairs][2][n_src]: x row then y row, i.e. rows 0-1 of the
 *   3xN homogeneous arrays the reference passes.  T_out [pairs][9] row-major 3x3 float64 mapping
 *   the source scan into the target frame; iters_out [pairs] iterations run (may be NULL).
 *   max_iter / tol are rospy.get_param('/icp/max_iter', 30) / ('/icp/tolerance', 0.001).
 *   Limits: n_src <= 2304 (one CTA holds a pair's source points in registers), n_tar bounded by the 227 KB of
 *   shared memory (about 7000 points); beyond them the call returns B2S_ERR_INVALID_ARG. */
int b2s_icp_batch_f32(const float *tar_xy, const float *src_xy, int pairs, int n_src, int n_tar,
                      int max_iter, double tol, double *T_out, int32_t *iters_out, void *stream);
/* The same from raw scans (fused ingestion): tar_ranges / src_ranges [pairs][n] float ranges, beam_cs [n][2] =
 * cos, sin of the beam angles (device, 16-byte aligned).  The kernel forms the points as laserToNumpy does
 * ([ICP]:216-229; +inf -> clamp_inf_to when > 0, [SLAM]:119) in float64 before the solve. */
int b2s_icp_batch_ranges(const float *tar_ranges, const float *src_ranges, const double *beam_cs,
                         double clamp_inf_to, int pairs, int n, int max_iter, double tol, double *T_out,
                         int32_t *iters_out, void *stream);
int b2s_icp_batch_f64(const double *tar_xy, const double *src_xy, int pairs, int n_src, int n_tar,
                      int max_iter, double tol, double *T_out, int32_t *iters_out, void *stream);
/* b2s_icp_batch_f64 that also reports each pair's score: err_out [pairs] (may be NULL) receives the reference's
 * mean_error = sum(dist) / N of the last iteration that ran ([ICP]:75-76), i.e. the mean matched distance before that
 * iteration's move and the value the stop rule last compared; unmatched (inf / NaN) distances count as 0 ([ICP]:95).
 * T_out and iters_out are those of b2s_icp_batch_f64, bit for bit.  max_iter == 0 gives 0. */
int b2s_icp_batch_f64_err(const double *tar_xy, const double *src_xy, int pairs, int n_src, int n_tar,
                          int max_iter, double tol, double *T_out, int32_t *iters_out, double *err_out, void *stream);

/* ICP.findNearest -- replaces [ICP]:90-114.  src_xy [n][2], tar_xy [m][2] (row = point, as the
 * reference passes them); dist_out [n] float64, idx_out [n] int64.  Lowest index wins ties. */
int b2s_nearest_f64(const double *src_xy, int n, const double *tar_xy, int m, double *dist_out,
                    int64_t *idx_out, void *stream);

/* ICP.getTransform -- replaces [ICP]:149-179.  src_xy, tar_xy [n][2] row-matched; T_out [9]. */
int b2s_rigid_fit_f64(const double *src_xy, const double *tar_xy, int n, double *T_out,
                      void *stream);

/* Mapping.update in integer form -- replaces [MAP]:22-51 with bresenham [BRES]:2-58 inlined.
 *   hit, miss [xw][yw] int32, x-major like the reference's datamap[x][y]; updated atomically.
 *   ox, oy [scans][beams] world-frame endpoints; cx, cy [scans] sensor positions.
 *   cell = (int)(cells_per_m * (v + off)) in float64, truncating ([MAP]:33-36: 10, 10).
 *   counters: device int32[B2S_CNT_WORDS] accumulating dropped/skipped beams, or NULL. */
int b2s_grid_raycast(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                     double off_x, double off_y, const float *ox, const float *oy,
                     const float *cx, const float *cy, int scans, int beams, int32_t *counters,
                     void *stream);

/* The same update on float64 endpoints and sensor positions -- the dtype the reference's callers pass
 * ([SLAM]:89-90: obs = u2T(xEst).dot(np_msg) and xEst are float64, and [MAP]:33-36 applies int() to the
 * float64 value).  Nothing is narrowed before the cell transform, so a coordinate on or next to a cell
 * boundary lands in the reference's cell; float32 input upcast to float64 gives the float32 entry point's result. */
int b2s_grid_raycast_f64(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                         double off_x, double off_y, const double *ox, const double *oy,
                         const double *cx, const double *cy, int scans, int beams, int32_t *counters,
                         void *stream);

/* Same update with a caller-provided workspace, which enables the fastest kernel: y-major beams
 * accumulate into a transposed scratch plane inside the workspace (so that the 32 beams of a warp
 * touch consecutive words in either orientation) and a transpose-add folds it into `miss` before the
 * call's work completes on the stream.  Result and planes are identical to b2s_grid_raycast.
 * workspace: device memory of b2s_grid_workspace_bytes(xw, yw) bytes, 16-byte aligned, prepared once
 * by b2s_grid_workspace_init and reusable across calls on the same stream; NULL falls back to
 * b2s_grid_raycast. */
size_t b2s_grid_workspace_bytes(int xw, int yw);
int b2s_grid_workspace_init(void *workspace, int xw, int yw, void *stream);
int b2s_grid_raycast_ws(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                        double off_x, double off_y, const float *ox, const float *oy,
                        const float *cx, const float *cy, int scans, int beams, int32_t *counters,
                        void *workspace, void *stream);

int b2s_grid_raycast_ws_f64(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                            double off_x, double off_y, const double *ox, const double *oy,
                            const double *cx, const double *cy, int scans, int beams,
                            int32_t *counters, void *workspace, void *stream);

/* Fused scan ingestion -- replaces laserToNumpy ([SLAM]:115-123), u2T(xEst).dot(np_msg) ([SLAM]:130-137,89)
 * and Mapping.update ([MAP]:22-51) in one kernel: raw ranges [scans][beams] float32 and, per scan,
 * pose4 = (x, y, cos yaw, sin yaw) float64; beam_cs [beams][2] = cos / sin of the beam angles
 * (np.cos / np.sin of np.linspace(angle_min, angle_max, beams), computed by the caller exactly as the
 * reference does).  Endpoints are formed in float64 with the reference's operation order; +inf ranges are
 * replaced by clamp_inf_to when it is > 0 (MAX_LASER_RANGE = 30, [SLAM]:18,119).  Half the input bytes of
 * the endpoint form.  Requires a workspace (see b2s_grid_raycast_ws). */
int b2s_grid_raycast_ranges(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                            double off_x, double off_y, const float *ranges, const double *pose4,
                            const double *beam_cs, double clamp_inf_to, int scans, int beams,
                            int32_t *counters, void *workspace, void *stream);

/* Screening of a batch before it is applied: flags[0] |= 1 if a NaN is present, flags[1] |= 1 if
 * oy or a sensor position holds an inf -- the values int() raises on in [MAP]:33-36 (ValueError /
 * OverflowError); ox = +-inf alone is legal ([MAP]:30).  flags: device int32[2], caller-zeroed. */
int b2s_grid_validate(const float *ox, const float *oy, const float *cx, const float *cy, int scans,
                      int beams, int32_t *flags, void *stream);

int b2s_grid_validate_f64(const double *ox, const double *oy, const double *cx, const double *cy, int scans,
                          int beams, int32_t *flags, void *stream);

/* Evidence score and occupancy from the counts -- replaces the per-visit rule of [MAP]:42-50
 * (w_hit 20) / [MAPO]:43-51 (w_hit 4): datamap = w_miss*miss + w_hit*hit (float32 out),
 * pmap = 50 if untouched else (100 if datamap > thresh else 0).  Either output may be NULL. */
int b2s_grid_finalize(const int32_t *hit, const int32_t *miss, int xw, int yw, double w_hit,
                      double w_miss, double thresh, float *datamap, int8_t *pmap, void *stream);

/* OccupancyGrid payload -- replaces [SLAM]:270-271: data[y*xw + x] = (int8) pmap[x][y]. */
int b2s_grid_pack_ros(const int8_t *pmap, int xw, int yw, int8_t *data, void *stream);

/* bresenham(start, end).path for a batch of segments -- replaces [BRES]:2-58.
 *   segs [count][4] = x0,y0,x1,y1; offsets [count+1] exclusive prefix sums of the path lengths
 *   (max(|dx|,|dy|)+1, 0 for a same-cell segment); cells_xy [offsets[count]][2]. */
int b2s_bresenham_paths(const int32_t *segs, int count, const int64_t *offsets, int32_t *cells_xy,
                        void *stream);

/* Odometry chain over a stream of per-pair transforms -- replaces the sequential accumulation of
 * [ICP]:185-190 / W9 localization.py:79-83 (x += cos(th) T02 - sin(th) T12; y += sin(th) T02 + cos(th) T12;
 * th += atan2(T10, T00)) with a parallel prefix.  T [pairs][9] row-major, traj [pairs+1][3] = x, y, th
 * (traj[0] is the start state).  Equal to the sequential float64 loop up to summation order (~1e-13). */
int b2s_pose_chain(const double *T, int pairs, double x0, double y0, double th0, double *traj,
                   void *stream);
int b2s_pose_chain_host(const double *T, int pairs, double x0, double y0, double th0, double *traj);

/* Virtual scan from the static map -- replaces laserEstimation, W9 localization.py:128-150: for every
 * obstacle cell centre (obs_x, obs_y) the range hypot(x - ox, y - oy) is min-reduced into bearing bin
 * int((atan2(oy - y, ox - x) - angle_min - yaw) / angle_increment), wrapped into [0, beams); bins nobody
 * hits keep far_range (100.0 in the reference).  ranges [beams] float64. */
int b2s_virtual_scan(const double *obs_x, const double *obs_y, int count, double x, double y,
                     double yaw, double angle_min, double angle_increment, int beams,
                     double far_range, double *ranges, void *stream);
int b2s_virtual_scan_host(const double *obs_x, const double *obs_y, int count, double x, double y,
                          double yaw, double angle_min, double angle_increment, int beams,
                          double far_range, double *ranges);
/* laserEstimation (W9 localization.py:128-150) for `scans` poses at once: poses3 [scans][3] = x, y, yaw.
 * ranges [scans][beams] (may be NULL) gets exactly what b2s_virtual_scan gives per pose; tar_xy [scans][2][beams]
 * (may be NULL; needs beam_cs [beams][2], 16-byte aligned) gets laserToNumpy of those ranges, the target layout of
 * b2s_icp_batch_f64.  At least one of the two is set; beams <= B2S_VSCAN_MAX_BEAMS (the bins of a pose live in
 * shared memory).  Like b2s_virtual_scan, an obstacle whose bin is NaN or overflows int is skipped: the host-buffer
 * caller rejects NaN poses before the launch. */
#define B2S_VSCAN_MAX_BEAMS 6144
int b2s_virtual_scan_batch(const double *obs_x, const double *obs_y, int count, const double *poses3, int scans,
                           double angle_min, double angle_increment, int beams, double far_range,
                           const double *beam_cs, double *ranges, double *tar_xy, void *stream);
/* Selection of a relocalization (no reference counterpart: the reference has no global localization; this picks among
 * map observations, [LOC9]:128-157, at many candidate poses).  score [scans][hyps] (b2s_icp_batch_f64_err's err_out),
 * T [scans][hyps][9] (the transforms of those solves), candidates3 [hyps][3] = x, y, yaw.  Per scan, best_out[k] is
 * the h with the smallest score among the hypotheses whose score and all nine entries of T are finite, the lowest h
 * on ties; pose_out[k] = candidates3[best] composed with T[k][best] by the pose-chain step of [ICP]:185-190
 * (x + cos(yaw) T02 - sin(yaw) T12, y + sin(yaw) T02 + cos(yaw) T12, yaw + atan2(T10, T00)), in float64: the sensor pose
 * in the map frame.  A scan without a finite hypothesis gets -1 and a NaN pose. */
int b2s_relocalize_select(const double *score, const double *T, const double *candidates3, int scans, int hyps,
                          int32_t *best_out, double *pose_out, void *stream);

/* Sum of per-GPU count deltas (no reference counterpart: the reference is single-process).
 * In-place ncclAllReduce(int32, sum) of both planes on an existing communicator. */
int b2s_grid_allreduce(int32_t *hit, int32_t *miss, size_t cells, void *nccl_comm, void *stream);

/* Fused merge over NVLink peer memory (one process per GPU; no reference counterpart): ONE kernel
 * reduce-scatters the ranks' delta planes (this rank sums cells [cell_lo, cell_hi) of every rank's
 * delta_hit / delta_miss -- its own pointer for itself, CUDA-IPC-mapped pointers for the peers), adds
 * the sums into its shard of the global counts (global_*_shard, int32 [cell_hi - cell_lo]), applies the
 * evidence rule of [MAP]:42-50 and all-gathers the int8 occupancy by storing its shard into every
 * rank's full map pmap[r].  Shard bounds are multiples of 4096 cells.  The caller orders the launch
 * after every rank's ray-cast and fences the maps afterwards (dist.ShardedMappingP2P uses two tiny
 * stream-ordered all-reduces). */
int b2s_grid_merge_p2p(const int32_t *const *delta_hit, const int32_t *const *delta_miss,
                       int8_t *const *pmap, int nranks, size_t cell_lo, size_t cell_hi,
                       int32_t *global_hit_shard, int32_t *global_miss_shard, double w_hit,
                       double w_miss, double thresh, void *stream);

/* Tile-sparse form of the same merge.  b2s_grid_raycast_ws / _ranges mark every 64 x 64-cell tile they
 * touch in a dirty map inside the workspace (b2s_grid_workspace_dirty: one byte per tile, row-major over
 * b2s_grid_tile_count).  all_dirty [nranks][tiles] holds every rank's map (gather them first; the gather
 * doubles as the fence after the ray-casts).  This rank merges tiles [tile_lo, tile_hi): untouched tiles
 * cost nothing, touched ones read only the ranks that touched them.  The shard of global counts is
 * tile-major int32 [tile_hi - tile_lo][64][64].  b2s_grid_clear_dirty re-zeroes a pair of delta planes
 * (only their dirty tiles) and clears the map. */
int b2s_grid_merge_p2p_tiles(const int32_t *const *delta_hit, const int32_t *const *delta_miss,
                             int8_t *const *pmap, const uint8_t *all_dirty, int nranks, int xw, int yw,
                             int tile_lo, int tile_hi, int32_t *global_hit_shard,
                             int32_t *global_miss_shard, double w_hit, double w_miss, double thresh,
                             void *stream);
/* The same step without a collective around it (dist.ShardedMappingP2P, the default): the two rendezvous of the step
 * -- "every rank's ray-cast is done and its dirty map has arrived" before the merge, "every rank's merge is done"
 * after it -- are epoch words in CUDA-IPC-mapped flag blocks that the ranks push to each other (st.release.sys) and
 * wait on locally (ld.acquire.sys), inside the kernels.  Per rank: a flag block of b2s_p2p_flag_bytes(nranks) bytes,
 * zeroed once, and a table all_dirty [nranks][b2s_p2p_dirty_stride(xw, yw)] for the gathered dirty maps, both
 * cudaMalloc'ed (b2s_device_alloc) and mapped into every peer; flags[r] / all_dirty[r] are rank r's buffers as seen
 * from this process.  One step, all on one stream, epoch = 1, 2, 3, ... (the same on every rank):
 *   b2s_grid_clear_dirty -> b2s_grid_raycast_ws / _ranges (private delta planes)
 *   -> b2s_p2p_publish                 copies this rank's dirty map into every rank's table and raises ready[rank]
 *                                      there; counters (may be NULL) = the ray-cast's B2S_CNT_* words, whose error
 *                                      count travels along
 *   -> b2s_grid_merge_p2p_tiles_sync   waits for every ready flag inside the kernel, merges as above, and its last
 *                                      CTA raises done[rank] in every rank's block
 *   -> b2s_p2p_wait_done               returns (on the stream) once every rank's merge is done: this rank's map is
 *                                      complete and its delta planes may be cleared.
 * A wait gives up after 20 s and sets an error word instead of hanging the GPU; b2s_p2p_status copies the error
 * word and the ranks' dropped-beam counts of the last step to the host (it synchronizes the stream). */
size_t b2s_p2p_flag_bytes(int nranks);
size_t b2s_p2p_dirty_stride(int xw, int yw);
int b2s_p2p_publish(const void *workspace, const int32_t *counters, uint8_t *const *all_dirty, uint32_t *const *flags,
                    int nranks, int rank, int xw, int yw, uint32_t epoch, void *stream);
int b2s_grid_merge_p2p_tiles_sync(const int32_t *const *delta_hit, const int32_t *const *delta_miss,
                                  int8_t *const *pmap, const uint8_t *all_dirty, uint32_t *const *flags, int nranks,
                                  int rank, uint32_t epoch, int xw, int yw, int tile_lo, int tile_hi,
                                  int32_t *global_hit_shard, int32_t *global_miss_shard, double w_hit, double w_miss,
                                  double thresh, void *stream);
int b2s_p2p_wait_done(uint32_t *my_flags, int nranks, uint32_t epoch, void *stream);
int b2s_p2p_status(const uint32_t *my_flags, int nranks, int *timed_out, int64_t *dropped_beams, void *stream);
void *b2s_grid_workspace_dirty(void *workspace);
int b2s_grid_tile_count(int xw, int yw, int *tiles_x, int *tiles_y);
int b2s_grid_clear_dirty(int32_t *hit, int32_t *miss, int xw, int yw, void *workspace, void *stream);

/* cudaMalloc'ed (IPC-exportable) device memory and CUDA IPC handles (64 bytes) for the peer mapping. */
int b2s_device_alloc(void **out, size_t bytes);
int b2s_device_free(void *p);
int b2s_ipc_export(const void *dev_ptr, void *handle64);
int b2s_ipc_open(const void *handle64, void **dev_ptr_out);
int b2s_ipc_close(void *dev_ptr);

/* NCCL plumbing for callers that do not bring their own communicator. */
int b2s_nccl_unique_id(void *id128);
int b2s_nccl_comm_init(void **comm_out, int nranks, int rank, const void *id128);
int b2s_nccl_comm_destroy(void *comm);

/* ===================================================================== layer 2: host */

/* Page-locked host buffers (full-speed, truly asynchronous copies). */
int b2s_host_alloc(void **out, size_t bytes);
int b2s_host_free(void *p);

typedef struct b2s_icp b2s_icp;
typedef struct b2s_mapping b2s_mapping;

/* ICP() -- [ICP]:11-36.  device < 0 selects the current device. */
int b2s_icp_create(b2s_icp **out, int device);
int b2s_icp_destroy(b2s_icp *icp);
/* ICP.process on host arrays; is_f64 selects const double* (the reference's dtype) or const float*. */
int b2s_icp_process(b2s_icp *icp, const void *tar_xy, const void *src_xy, int is_f64, int pairs,
                    int n_src, int n_tar, int max_iter, double tol, double *T_out,
                    int32_t *iters_out);
/* ICP.process over the consecutive pairs of a scan stream: calc_odometry's loop, [LOC9]:159-168 / [SLAM]:109-113
 * (target = scan k, source = scan k + 1).  scans_xy [scans][2][n]; T_out [scans-1][9], iters_out [scans-1] (may be
 * NULL).  Same results as b2s_icp_process on the pairs, half the host-to-device bytes. */
int b2s_icp_process_sequence(b2s_icp *icp, const void *scans_xy, int is_f64, int scans, int n, int max_iter,
                             double tol, double *T_out, int32_t *iters_out);
/* The whole LiDAR-odometry loop of [LOC9]:66-83 for a recorded stream: b2s_icp_process_sequence followed by the
 * pose chain of [LOC9]:79-83 / [ICP]:185-190 (b2s_pose_chain) on the device.  traj_out [scans][3] = x, y, yaw,
 * row 0 = (x0, y0, th0); T_out [scans-1][9] and iters_out [scans-1] may be NULL. */
int b2s_icp_odometry(b2s_icp *icp, const void *scans_xy, int is_f64, int scans, int n, int max_iter, double tol,
                     double x0, double y0, double th0, double *traj_out, double *T_out, int32_t *iters_out);
/* The same loop fed with what the sensor delivers: ranges [scans][n] (LaserScan.ranges) + the beam table [n][2]
 * (cos, sin of linspace(angle_min, angle_max, n)); laserToNumpy runs inside the kernel (b2s_icp_batch_ranges).
 * state3 = (x0, y0, th0) and traj_out [scans][3] are both NULL (transforms only) or both set (with the pose chain). */
int b2s_icp_process_scans(b2s_icp *icp, const float *ranges, const double *beam_cs, double clamp_inf_to, int scans,
                          int n, int max_iter, double tol, const double *state3, double *traj_out, double *T_out,
                          int32_t *iters_out);
/* Streaming forms of b2s_icp_process_sequence / b2s_icp_process_scans (transforms only): submit enqueues the uploads, the
 * solves and the read-back of T_out [scans-1][9] / iters_out [scans-1] (may be NULL) and returns a ticket; two calls may be
 * in flight, so the scans of the next stream cross PCIe while this one is being solved.  The input array and the output
 * buffers (page-locked for truly asynchronous copies) must stay valid and untouched until b2s_icp_wait(ticket) returns. */
int b2s_icp_submit_sequence(b2s_icp *icp, const void *scans_xy, int is_f64, int scans, int n, int max_iter, double tol,
                            double *T_out, int32_t *iters_out, int *ticket_out);
int b2s_icp_submit_scans(b2s_icp *icp, const float *ranges, const double *beam_cs, double clamp_inf_to, int scans, int n,
                         int max_iter, double tol, double *T_out, int32_t *iters_out, int *ticket_out);
int b2s_icp_wait(b2s_icp *icp, int ticket);
/* The static map of the localization node (self.obstacle): obstacle cell centres, uploaded once and kept on the
 * device until replaced.  count == 0 clears it.  A NaN coordinate is rejected (B2S_ERR_NONFINITE, the map is then
 * cleared): the reference's int() raises on it.  +-inf coordinates are kept; they never win a bin. */
int b2s_icp_set_map(b2s_icp *icp, const double *obs_x, const double *obs_y, int count);
/* calc_map_observation ([LOC9]:152-157) for a recorded stream: for scan k, target = laserToNumpy(virtual scan of the
 * map at poses3[k]), source = laserToNumpy(ranges[k]) (clamp_inf_to > 0: the W12 inf clamp), T_out[k] =
 * ICP.process(target, source).  beam_cs [n][2] = cos, sin of linspace(angle_min, angle_max, n); the virtual scan bins
 * with angle_min / angle_increment.  virtual_out [scans][n] (may be NULL) receives the virtual ranges, iters_out
 * [scans] (may be NULL) the iteration counts.  A NaN pose fails with B2S_ERR_NONFINITE before anything runs; no map
 * set is B2S_ERR_INVALID_ARG.  Same transforms as b2s_icp_process on the float64 point pairs, bit for bit. */
int b2s_icp_map_observation(b2s_icp *icp, const float *ranges, const double *poses3, const double *beam_cs,
                            double clamp_inf_to, int scans, int n, double angle_min, double angle_increment,
                            double far_range, int max_iter, double tol, double *T_out, int32_t *iters_out,
                            double *virtual_out);
/* Relocalization in the static map: the map observation ([LOC9]:128-157) of each scan at every candidate pose,
 * scored and chosen on the device.  ranges [scans][n], candidates3 [hyps][3] = x, y, yaw, shared by all scans.
 * Hypothesis (k, h) is b2s_icp_map_observation of ranges[k] at candidates3[h], bit for bit: the virtual scans are built
 * once per call and reused for every scan.  score_out [scans][hyps] is its mean_error of the last iteration
 * ([ICP]:75-76), iters_out [scans][hyps] and T_out [scans][hyps][9] its iterations and transform; best_out [scans] and
 * pose_out [scans][3] come from b2s_relocalize_select ([ICP]:185-190).  score_out, iters_out and T_out may be NULL.
 * hyps >= 1, n <= 2304.  A NaN candidate fails with B2S_ERR_NONFINITE before anything runs; no map set is
 * B2S_ERR_INVALID_ARG. */
int b2s_icp_relocalize(b2s_icp *icp, const float *ranges, const double *candidates3, const double *beam_cs,
                       double clamp_inf_to, int scans, int hyps, int n, double angle_min, double angle_increment,
                       double far_range, int max_iter, double tol, int32_t *best_out, double *pose_out,
                       double *score_out, int32_t *iters_out, double *T_out);
int b2s_icp_find_nearest(b2s_icp *icp, const double *src_xy, int n, const double *tar_xy, int m,
                         double *dist_out, int64_t *idx_out);
int b2s_icp_get_transform(b2s_icp *icp, const double *src_xy, const double *tar_xy, int n,
                          double *T_out);

/* Mapping(xw, yw, xyreso) -- [MAP]:8-20.  Owns zeroed int32 hit/miss planes on the device. */
int b2s_mapping_create(b2s_mapping **out, int xw, int yw, double xyreso, double w_hit,
                       double w_miss, double thresh, int device);
int b2s_mapping_destroy(b2s_mapping *map);
int b2s_mapping_reset(b2s_mapping *map);
/* Mapping.update -- [MAP]:22-51 for `scans` scans at once, all-or-nothing: a batch holding a coordinate the
 * reference's int() raises on (B2S_ERR_NONFINITE) or an over-long beam (B2S_ERR_TOO_LONG) leaves the planes
 * as they were.  The chunks are applied while the later ones still cross PCIe (the kernels skip and count
 * the offending beams); a rejected batch is then taken back out with the sign -1 kernel, which is exact on
 * integer counts.  When pmap_out is not NULL it receives the refreshed occupancy [xw][yw].
 * b2s_mapping_update consumes float32 coordinates (the fast path: half the bytes over PCIe);
 * b2s_mapping_update_f64 consumes the float64 the reference's callers pass and is the form that is
 * bit-identical to [MAP]:33-36 on any input. */
int b2s_mapping_update(b2s_mapping *map, const float *ox, const float *oy, const float *cx,
                       const float *cy, int scans, int beams, int8_t *pmap_out);
int b2s_mapping_update_f64(b2s_mapping *map, const double *ox, const double *oy, const double *cx,
                           const double *cy, int scans, int beams, int8_t *pmap_out);
/* Mapping.update with an incremental read-back: pmap_inout must still hold the map written by the previous
 * call on this object (any of the update calls with a map pointer); only the 64 x 64-cell tiles this batch
 * touched are finalized, copied and patched into it, so a single scan on a large map costs microseconds
 * instead of a full-map transfer.  tiles_out / tiles_count (optional) report the patched tile indices
 * (row-major over b2s_grid_tile_count); *tiles_count = -1 means the whole map was rewritten (first call,
 * after reset / write, too many tiles, or more than tiles_cap). */
int b2s_mapping_update_incremental(b2s_mapping *map, const float *ox, const float *oy, const float *cx,
                                   const float *cy, int scans, int beams, int8_t *pmap_inout,
                                   int32_t *tiles_out, int tiles_cap, int *tiles_count);
int b2s_mapping_update_incremental_f64(b2s_mapping *map, const double *ox, const double *oy, const double *cx,
                                       const double *cy, int scans, int beams, int8_t *pmap_inout,
                                       int32_t *tiles_out, int tiles_cap, int *tiles_count);
/* The same for raw scans (fused ingestion, see b2s_grid_raycast_ranges): ranges [scans][beams], pose4
 * [scans][4], beam_cs [beams][2] on the host. */
int b2s_mapping_update_ranges(b2s_mapping *map, const float *ranges, const double *pose4,
                              const double *beam_cs, double clamp_inf_to, int scans, int beams,
                              int8_t *pmap_out);
/* The same with raw poses: poses3 [scans][3] = x, y, yaw.  cos / sin of the yaw (u2T, [SLAM]:130-137: math.cos,
 * math.sin) are evaluated with libm inside the call, one pipeline chunk ahead of the device. */
int b2s_mapping_update_scans(b2s_mapping *m, const float *ranges, const double *poses3, const double *beam_cs,
                             double clamp_inf_to, int scans, int beams, int8_t *pmap_out);
/* Streaming forms of b2s_mapping_update / b2s_mapping_update_scans: submit enqueues the whole step -- chunked upload,
 * ray-cast, finalize into the step's own device map, read-back into pmap_out on a third stream -- and returns a
 * ticket at once; up to two steps are in flight, so the upload and ray-cast of step k + 1 run while the map of step k
 * is still crossing PCIe the other way.  zero_first != 0 clears the counts before the step.  pmap_out [xw][yw]
 * (page-locked for a truly asynchronous copy; may be NULL) and the input arrays must stay valid and untouched until
 * b2s_mapping_wait(ticket) has returned; submitting a third step first waits for the first one implicitly.
 * b2s_mapping_wait returns the step's verdict: B2S_ERR_NONFINITE / B2S_ERR_TOO_LONG mean the batch held a coordinate the
 * reference's int() raises on ([MAP]:33-36) / an over-long beam and has been taken back out of the counts (exact, sign -1
 * kernels); maps of steps submitted after it and before the wait were finalized with it still applied. */
int b2s_mapping_submit(b2s_mapping *map, const float *ox, const float *oy, const float *cx, const float *cy, int scans,
                       int beams, int zero_first, int8_t *pmap_out, int *ticket_out);
int b2s_mapping_submit_scans(b2s_mapping *map, const float *ranges, const double *poses3, const double *beam_cs,
                             double clamp_inf_to, int scans, int beams, int zero_first, int8_t *pmap_out, int *ticket_out);
int b2s_mapping_wait(b2s_mapping *map, int ticket);
/* Snapshot to host; any pointer may be NULL. */
int b2s_mapping_read(b2s_mapping *map, int32_t *hit, int32_t *miss, float *datamap, int8_t *pmap);
/* Overwrite the count planes from host arrays [xw][yw] (checkpoint restore; the reference has none). */
int b2s_mapping_write(b2s_mapping *map, const int32_t *hit, const int32_t *miss);
/* The planes themselves, for layer-1 calls and collectives.  Handing them out invalidates the object's cached
 * occupancy: the next update call with a map pointer refreshes the whole map instead of patching dirty tiles. */
int b2s_mapping_planes(b2s_mapping *map, int32_t **hit, int32_t **miss, void **stream);
/* bresenham(start,end).path on host arrays (segs [count][4], cells_xy sized by the caller). */
int b2s_bresenham_host(const int32_t *segs, int count, const int64_t *offsets, int32_t *cells_xy);

#ifdef __cplusplus
}
#endif
#endif /* B2SLAM_H */

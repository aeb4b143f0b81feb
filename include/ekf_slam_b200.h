/* ekf_slam_b200.h — C ABI of the B200-native EKF-SLAM hot path.
 *
 * The reference (tonylitianyu/EKF-SLAM-ML) has no FFI: its boundary is the public C++ class API of
 * librigid2d (rigid2d/include/rigid2d/ekf_slam.hpp:19-91, circle_fitting.hpp:18-60), called in-process
 * by the nuslam ROS nodes (nuslam/src/slam.cpp:428-434, unknown_data_assoc.cpp:409-415,
 * landmarks.cpp:133-141).  The C++ facade in include/rigid2d/ keeps those class signatures and is a thin
 * shell over the functions below; every function names the reference member it stands in for.
 *
 * Conventions
 *   - plain pointers and sizes only; all host pointers stay owned by the caller;
 *   - every function returns 0 on success, < 0 for an invalid argument / unsupported request,
 *     > 0 for a CUDA runtime error code (cudaError_t); nothing throws across this boundary;
 *   - ekf_last_error() returns a thread-local human-readable message for the last failure;
 *   - a handle is single-caller (like the reference object, driven from one ros::spin thread);
 *     verbs enqueue on the handle's CUDA stream, getters synchronise;
 *   - state layout: [theta, x, y, m1x, m1y, ..., mnx, mny], N = 3 + 2n doubles (ekf_slam.cpp:72-74, 15-21);
 *     covariance: row-major N x N doubles with caller-chosen leading dimension `ld` >= N;
 *   - there is NO CPU fallback: without a usable CUDA device every create call fails.
 */
#ifndef EKF_SLAM_B200_H
#define EKF_SLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EKF_OK 0
#define EKF_ERR_INVALID (-1)
#define EKF_ERR_UNSUPPORTED (-2)
#define EKF_ERR_STATE (-3)

/* the reference's noise covariances (ekf_slam.cpp:41-43, :172-175): Q = EKF_DEFAULT_Q I_3 on (theta, x, y),
 * R = EKF_DEFAULT_R I_2 on (range, bearing); what every filter uses until ekf_set_noise / ekf_batch_set_noise */
#define EKF_DEFAULT_Q 0.0001
#define EKF_DEFAULT_R 0.01

/* engine selection for ekf_create_ex */
#define EKF_ENGINE_AUTO 0  /* fused on-chip engine when Sigma fits shared memory, streamed otherwise */
#define EKF_ENGINE_FUSED 1 /* one kernel per call, Sigma resident in shared memory (n <= 64) */
#define EKF_ENGINE_STREAM 2/* Sigma in HBM, gain + streamed rank-2 sweep per correction (any n) */

const char* ekf_version(void);
const char* ekf_last_error(void);
int ekf_device_count(int* count_out);

/* Pinned host memory for buffers handed to the batched verbs (makes their copies asynchronous). */
int ekf_host_alloc(void** out, uint64_t bytes);
int ekf_host_free(void* p);

/* ------------------------------------------------------------------ single filter: rigid2d::EKF_SLAM */
typedef struct ekf_filter ekf_filter;

/* EKF_SLAM::EKF_SLAM(int n_measurements)                       rigid2d/src/ekf_slam.cpp:27-53 */
int ekf_create(int n_landmarks, int device, ekf_filter** out);
int ekf_create_ex(int n_landmarks, int device, int engine, ekf_filter** out);
/* copy construction / assignment (the node copy-assigns a fresh filter in INIT, nuslam/src/slam.cpp:428) */
int ekf_clone(ekf_filter* src, ekf_filter** out);
int ekf_destroy(ekf_filter* h);
int ekf_num_landmarks(const ekf_filter* h);
int ekf_engine(const ekf_filter* h);

/* EKF_SLAM::prediction(const Twist2D&): dtheta = twist.angular(), dx = twist.linearX();
 * linearY is ignored by the reference (:70)                     rigid2d/src/ekf_slam.cpp:55-106
 * Fused engine: the call records the twist and returns; the prediction is applied by the next ekf_measurement() /
 * ekf_data_association() kernel, or by whichever other verb looks at or changes the filter first (results are the
 * same for every call order; a launch error of the deferred work is returned by that later verb). */
int ekf_predict(ekf_filter* h, double dtheta, double dx);

/* EKF_SLAM::measurement(mat sensor_reading, vector<bool> visible_list, vector<bool> known_list)
 * xy: 2n robot-frame readings (x0,y0,x1,y1,...); visible: n flags.  known_list is unused by the
 * reference and therefore not part of this call.                rigid2d/src/ekf_slam.cpp:108-197 */
int ekf_measurement(ekf_filter* h, const double* xy, const uint8_t* visible);

/* EKF_SLAM::data_association(vector<Vector2D> measures, vector<bool>& known_list)
 * xy: m robot-frame measurements; known: n flags, in/out.  Optional outputs (may be NULL), m entries each:
 *   assoc_out   landmark index corrected by measurement j, -1 if the measurement was dropped
 *   dmin_out    min_maha_dis before the new-landmark reset (10.0 when nothing was below the gate)
 *   second_out  runner-up distance (tie-margin diagnostics; +inf if none)
 *   created_out 1 if measurement j initialised a new landmark  rigid2d/src/ekf_slam.cpp:278-402 */
int ekf_data_association(ekf_filter* h, const double* xy, int m, uint8_t* known, int32_t* assoc_out,
                         double* dmin_out, double* second_out, uint8_t* created_out);

/* EKF_SLAM::calculate_maha_dis(Vector2D, int) — private in the reference, exposed as a test seam
 *                                                               rigid2d/src/ekf_slam.cpp:217-276 */
int ekf_maha(ekf_filter* h, double mx, double my, int landmark, double* d_out);

/* getStateTheta / getStateX / getStateY -> out3 = {theta, x, y}  rigid2d/src/ekf_slam.cpp:404-414 */
int ekf_get_pose(ekf_filter* h, double* out3);
/* getStateLandmark -> 2n doubles                                rigid2d/src/ekf_slam.cpp:416-418 */
int ekf_get_landmarks(ekf_filter* h, double* out);
/* full state / covariance access (parity dumps, checkpoint / resume; no reference counterpart) */
int ekf_get_state(ekf_filter* h, double* out);
int ekf_set_state(ekf_filter* h, const double* in);
/* Per-step association log (the reference only prints these decisions, ekf_slam.cpp:290-329): from now on every
 * ekf_data_association() call appends one CSV line per measurement - call,index,x,y,landmark (-1 = dropped),
 * min_distance,runner_up,created - to `path`; NULL closes the log. */
int ekf_association_log_open(ekf_filter* h, const char* path);
int ekf_get_sigma(ekf_filter* h, double* out, int64_t ld);
/* `count` selected rows (N doubles each, row stride ld in `out`) and the diagonal (N doubles): for parity checks of
 * maps whose whole covariance is too large to pull to the host */
int ekf_get_sigma_rows(ekf_filter* h, const int64_t* rows, int count, double* out, int64_t ld);
int ekf_get_sigma_diag(ekf_filter* h, double* out);
int ekf_set_sigma(ekf_filter* h, const double* in, int64_t ld);
int ekf_get_init_flag(ekf_filter* h, int* out);  /* landmark_init_flag, ekf_slam.cpp:50 */
int ekf_set_init_flag(ekf_filter* h, int v);
int ekf_update_count(ekf_filter* h, uint64_t* out); /* landmark corrections executed so far */
int ekf_sync(ekf_filter* h);
/* Streamed engine only: corrections accumulated before Sigma is swept (1..20, default 14: the deepest group for
 * which the sweep still runs at the HBM copy rate; 15..20 give more corrections per second with a sweep bound by the
 * FP64 pipe instead).  Within a measurement() call the delayed application is bit-identical to one sweep per
 * correction (1 reproduces the reference's schedule); across calls see ekf_set_carry_pending. */
int ekf_set_max_pending(ekf_filter* h, int max_pending);
/* 1 (default): correction factors may stay pending across prediction() and measurement() calls (prediction() maps
 * them through the motion Jacobian in O(1)), so every sweep of the streamed engine carries max_pending corrections;
 * 0: Sigma is swept at the end of every measurement().  Every verb that reads Sigma or the update counter settles the
 * pending factors first, so the difference is only visible in rounding (1e-15 relative) and in speed. */
int ekf_set_carry_pending(ekf_filter* h, int carry);
/* Noise covariances of the filter: noise5 = {q_theta, q_x, q_y, r_range, r_bearing}, Q = diag(q) added to the robot
 * block in prediction, R = diag(r) added to S in measurement(), data_association() and ekf_maha.  Every entry finite,
 * q >= 0, r > 0, or EKF_ERR_INVALID and nothing changes; NULL restores EKF_DEFAULT_Q / EKF_DEFAULT_R.  Takes effect
 * from the next verb (a prediction the fused engine still defers is applied first, with the old Q); noise5 may be
 * reused on return.  ekf_clone copies it; it is configuration, not state (ekf_set_state / ekf_set_sigma keep it). */
int ekf_set_noise(ekf_filter* h, const double* noise5);
int ekf_get_noise(ekf_filter* h, double* out5);
/* Normalised innovation squared of the single filter, with the scoring rule of ekf_batch_set_nis: every correction a
 * measurement() / data_association() call applies is scored from exactly the S^-1 and nu of its gain, except those of
 * the filter's first measurement() (landmark_init_flag == 0 on entry) and a data_association() correction of a landmark
 * created by the same reading.  A call's values are summed in correction order and the sum is then added to
 * {sum NIS, sum NIS^2, #scored, #non-finite}, so a streamed filter with ekf_set_carry_pending(h, 0) gets accumulators
 * bit-identical to the same filter in a wide batch.  No kernel launch is added: ekf_launch_count is the same either way.
 *
 * 1: the following measurement() / data_association() calls run the NIS variants of the filter's kernels and
 * accumulate (buffers allocated and zeroed on first use); 0: the plain kernels again, accumulators kept.  ekf_clone
 * copies the switch and the accumulators; ekf_set_state, ekf_set_sigma and ekf_set_noise leave them alone. */
int ekf_set_nis(ekf_filter* h, int on);
/* out4 = {sum NIS, sum NIS^2, #scored, #non-finite}; reset != 0 zeroes them after the read.  EKF_ERR_STATE before NIS
 * was ever enabled.  Synchronises. */
int ekf_nis(ekf_filter* h, double* out4, int reset);
/* The NIS of the last measurement() / data_association() call that ran with NIS on, aligned with that call's inputs:
 * n values (slot order) after measurement(), m values (measurement order) after data_association(); *count_out says
 * which (0 before the first such call).  -1.0 where no correction was scored; a scored value that is not finite is
 * written as it is.  out may be NULL to ask for the count only.  EKF_ERR_STATE before NIS was ever enabled.
 * Synchronises. */
int ekf_last_nis(ekf_filter* h, double* out, int* count_out);
/* passes over Sigma the streamed engine has made so far (for the roofline accounting of bench.py) */
int ekf_sweep_count(ekf_filter* h, uint64_t* out);
/* raw device pointers for callers that live on the GPU already (bench, fused pipelines) */
int ekf_device_pointers(ekf_filter* h, void** sigma, int64_t* ld, void** state);
void* ekf_stream(ekf_filter* h); /* cudaStream_t */

/* ------------------------------------------------------------------ batch of independent filters */
typedef struct ekf_batch ekf_batch;

/* n_landmarks <= 64: Sigma stays on chip during a step (EKF_ENGINE_FUSED engines).  64 < n_landmarks <= 1024: the
 * "wide" engine (EKF_ENGINE_STREAM): every filter's Sigma lives in HBM and each filter is bit-identical to an
 * ekf_create_ex(n, device, EKF_ENGINE_STREAM, ...) filter with ekf_set_carry_pending(h, 0) fed the same inputs; it
 * serves the known-association verbs (dense, marker list for n <= 256, device-resident), and ekf_batch_step_unknown
 * returns EKF_ERR_UNSUPPORTED.  n_landmarks > 1024 returns EKF_ERR_UNSUPPORTED: one streamed filter per map. */
int ekf_batch_create(int64_t n_filters, int n_landmarks, int device, ekf_batch** out);
int ekf_batch_destroy(ekf_batch* b);
int64_t ekf_batch_size(const ekf_batch* b);
/* EKF_ENGINE_FUSED (Sigma on chip, n <= 64) or EKF_ENGINE_STREAM (Sigma in HBM, the wide engine); mirrors ekf_engine */
int ekf_batch_engine(const ekf_batch* b);
/* passes over a filter's Sigma in HBM so far, summed over the filters (0 for the on-chip engines); mirrors
 * ekf_sweep_count.  A wide filter sweeps ceil(c / 14) times in a step with c corrections. */
int ekf_batch_sweep_count(ekf_batch* b, uint64_t* out);

/* One SLAM-node step for every filter: prediction(twist) then measurement(xy, visible)
 * (nuslam/src/slam.cpp:433-434).  HOST buffers: twists [B][2] = {dtheta, dx}, xy [B][2n], visible [B][n].
 * The copies and the kernel are enqueued and the call returns; with buffers from ekf_host_alloc() nothing
 * blocks, and the caller must leave them untouched until ekf_batch_sync() (cudaMemcpyAsync rules). */
int ekf_batch_step_known(ekf_batch* b, const double* twists, const double* xy, const uint8_t* visible);
/* prediction(twist) then data_association(measures) (nuslam/src/unknown_data_assoc.cpp:414-415).
 * meas [B][m_max][2], count [B] valid measurements per filter; assoc_out [B][m_max] host, optional.
 * A count below 0 is an empty list (prediction only, that filter's outputs all -1), a count above m_max is m_max;
 * assoc_out[b][j] = -1 for every j at or beyond filter b's count. */
int ekf_batch_step_unknown(ekf_batch* b, const double* twists, const double* meas, const int32_t* count,
                           int m_max, int32_t* assoc_out);
/* The same step fed with the fake_sensor message as it is on the wire: only the visible markers, each with its
 * landmark id (published at nurtlesim/src/tube_world.cpp:369-414, unpacked into the dense arrays at
 * nuslam/src/slam.cpp:232-262).  CSR: offsets [B + 1] (filter b owns entries offsets[b] .. offsets[b+1]-1, at most n,
 * ids unique within a filter), ids [total] < n, xy [total][2]; a filter whose offsets do not lie inside [0, total]
 * gets an empty list, an id >= n is ignored.  A slot that is not listed is not visible and reads
 * (0, 0), exactly what the node's dense arrays hold for it; results are bit-identical to ekf_batch_step_known() on
 * those dense arrays, with about a third of the host-to-device bytes. */
int ekf_batch_step_known_sparse(ekf_batch* b, const double* twists, const int32_t* offsets, const uint8_t* ids,
                                const double* xy, int64_t total);
/* Same verbs with inputs already resident in HBM (device pointers, same layouts).  ekf_batch_step_unknown_dev clamps
 * the counts as above; a null d_count means m_max measurements for every filter. */
int ekf_batch_step_known_sparse_dev(ekf_batch* b, const double* d_twists, const int32_t* d_offsets, const uint8_t* d_ids,
                                    const double* d_xy, int64_t total);
int ekf_batch_step_known_dev(ekf_batch* b, const double* d_twists, const double* d_xy, const uint8_t* d_visible);
int ekf_batch_step_unknown_dev(ekf_batch* b, const double* d_twists, const double* d_meas, const int32_t* d_count,
                               int m_max, int32_t* d_assoc_out);

int ekf_batch_get_poses(ekf_batch* b, double* out /* [B][3] theta,x,y */);
/* asynchronous read-back into pinned memory; complete after ekf_batch_sync() */
int ekf_batch_get_poses_async(ekf_batch* b, double* pinned_out);
int ekf_batch_get_states(ekf_batch* b, double* out /* [B][N] */);
/* one filter's covariance as a dense row-major N x N matrix (expanded from the on-chip engines' storage) */
int ekf_batch_get_sigma(ekf_batch* b, int64_t filter, double* out, int64_t ld);
int ekf_batch_get_known(ekf_batch* b, uint8_t* out /* [B][n] */);
int ekf_batch_set_known(ekf_batch* b, const uint8_t* in);
int ekf_batch_update_count(ekf_batch* b, uint64_t* out);
/* Checkpoint / resume (the reference keeps the filter only in the node's memory, slam.cpp:427-430): the batch's arrays
 * exactly as the engine holds them — Sigma in the layout of ekf_batch_device_pointers, sizes from
 * ekf_batch_checkpoint_size — plus
 * landmark_init_flag [B], known_list [B][n] and the update counter.  A batch of the same shape restored with
 * ekf_batch_import continues bit-identically. */
int ekf_batch_checkpoint_size(ekf_batch* b, int64_t* sigma_doubles, int64_t* state_doubles);
int ekf_batch_export(ekf_batch* b, double* sigma, double* state, int32_t* init_flag, uint8_t* known, uint64_t* updates);
int ekf_batch_import(ekf_batch* b, const double* sigma, const double* state, const int32_t* init_flag,
                     const uint8_t* known, uint64_t updates);
/* error statistics against ground-truth poses truth[B][3] = {x, y, theta}:
 * out4 = {sum dx^2, sum dy^2, sum wrap(dtheta)^2, B} — the per-GPU partial that ranks all-reduce. */
int ekf_batch_pose_error(ekf_batch* b, const double* truth, double* out4);
/* Consistency of the batch (no reference counterpart: the reference never scores its covariance).  One kernel reads
 * each filter's stored Sigma entries in place, in any of the three layouts below, plus the state, landmark_init_flag and
 * known_list; it writes nothing the filters own.  It is enqueued on ekf_batch_stream(), after any step already there.
 *
 * Marginals: pose_cov [B][6] = (00, 01, 02, 11, 12, 22) of Sigma[0:3, 0:3] (state order theta, x, y), lm_cov [B][n][3]
 * = (xx, xy, yy) of each landmark slot's 2 x 2 block; either may be NULL.  Bit-identical to the same entries
 * (row <= column) of ekf_batch_get_sigma(). */
int ekf_batch_get_marginals(ekf_batch* b, double* pose_cov, double* lm_cov);
/* Normalised estimation error squared against truth [B][3] = {x, y, theta} (the convention of ekf_batch_pose_error):
 *   NEES_pose = e^T P^-1 e, e = (wrap(theta_hat - theta), x_hat - x, y_hat - y), P = Sigma[0:3, 0:3];
 *   NEES_i    = the same with landmark slot i's 2 x 2 block and lm_truth.
 * lm_truth is [n][2] shared by every filter (lm_truth_stride = 0) or [B][n][2] (lm_truth_stride = 2n); NULL scores no
 * landmark.  Slot i of filter b is scored iff its truth is finite and (landmark_init_flag[b] != 0 or known_list[b][i]
 * != 0).  A block whose Cholesky pivot is not positive and finite is singular: its NEES is NaN and it is counted apart.
 * per_filter [B][3] = {NEES_pose, sum of NEES_i, number of NEES_i}, optional.
 * out8 = {sum NEES_pose, sum NEES_pose^2, #pose, sum NEES_i, sum NEES_i^2, #landmarks, #singular pose, #singular
 * landmark}: additive, so ranks all-reduce it like out4.  The reduction runs in a fixed order without floating-point
 * atomics: two calls on the same state and device return bit-identical results.  HOST buffers; synchronises. */
int ekf_batch_nees(ekf_batch* b, const double* truth, const double* lm_truth, int64_t lm_truth_stride,
                   double* per_filter, double* out8);
/* The same with DEVICE pointers (e.g. the truth of tubeworld_outputs()), enqueued on ekf_batch_stream() and not
 * synchronised: the results are valid after ekf_batch_sync(), so a per-step series costs no host round trip. */
int ekf_batch_nees_dev(ekf_batch* b, const double* d_truth, const double* d_lm_truth, int64_t lm_truth_stride,
                       double* d_per_filter, double* d_out8);
/* Normalised innovation squared, the consistency test that needs no truth.  Per correction NIS = nu^T S^-1 nu with
 * nu = (z_r - zhat_r, wrap(z_phi - zhat_phi)) and S = H_j Sigma H_j^T + R, from exactly the S^-1 and nu of the
 * correction's gain (known association: entry-time pose; unknown: live pose); chi^2(2) for a consistent filter.  Every
 * correction a step applies is scored, except those of a filter's first measurement (landmark_init_flag == 0 at step
 * entry) and, with unknown association, that of a landmark created by the same reading (nu ~ 0 in both).  Per filter
 * the kernel sums the step's values in correction order and adds them to {sum NIS, sum NIS^2, #scored, #non-finite};
 * a value that is not finite counts in #non-finite only.  No floating-point atomics: replicas of one trajectory get
 * bit-identical accumulators.
 *
 * 1: the following steps run the NIS variants of the step kernels and accumulate per filter (allocated and zeroed on
 * first use); 0: the plain kernels again, accumulators kept.  Not part of checkpoints: export / import ignore them. */
int ekf_batch_set_nis(ekf_batch* b, int on);
/* per_filter [B][4] = {sum NIS, sum NIS^2, #scored, #non-finite} (optional), out4 = the same summed over the batch in a
 * fixed order (additive across ranks).  reset != 0 zeroes the accumulators after the read.  EKF_ERR_STATE before NIS
 * was ever enabled.  HOST buffers; synchronises. */
int ekf_batch_nis(ekf_batch* b, double* per_filter, double* out4, int reset);
/* the same with DEVICE pointers, enqueued on ekf_batch_stream(), no synchronisation (a per-step series with reset = 1) */
int ekf_batch_nis_dev(ekf_batch* b, double* d_per_filter, double* d_out4, int reset);
/* Per-filter noise covariances, rows {q_theta, q_x, q_y, r_range, r_bearing} as in ekf_set_noise: stride 0 gives every
 * filter the row at `noise`, stride 5 reads [B][5].  The following steps run the NOISE variants of the step kernels
 * (still one launch per step); NULL returns to EKF_DEFAULT_Q / EKF_DEFAULT_R and the default kernels.  Rows are
 * checked on the host (any invalid row: EKF_ERR_INVALID, nothing changes) and copied in stream order behind the work
 * already enqueued; `noise` may be reused on return.  Not part of checkpoints: set it again after ekf_batch_import. */
int ekf_batch_set_noise(ekf_batch* b, const double* noise, int64_t stride);
/* out [B][5]: the rows in use (the defaults when none are set); synchronises */
int ekf_batch_get_noise(ekf_batch* b, double* out);
int ekf_batch_sync(ekf_batch* b);
/* Raw device arrays of the batch.  state: [B][state_stride] doubles (theta, x, y, m1x, m1y, ...).  sigma:
 * [B][sigma_stride] doubles in the engine's layout:
 *   n == 20      the tile engine's register-fragment layout, with the state inside each filter's block;
 *   n <= 64      the SYMMETRIC block-staircase layout: row r stores the columns [16*floor(r/16), N) only, rows back to
 *                back (element (r, c) with c < 16*floor(r/16) is the stored (c, r));
 *   64 < n       (wide engine) a dense row-major N x ld matrix, ld = N rounded up to a multiple of 16 doubles (the
 *                streamed engine's layout; columns N..ld-1 are padding), sigma_stride = N * ld.
 * ekf_batch_get_sigma() returns a dense copy of any of them. */
int ekf_batch_device_pointers(ekf_batch* b, void** sigma, int64_t* sigma_stride, void** state,
                              int64_t* state_stride);
void* ekf_batch_stream(ekf_batch* b);
/* CUDA-event stopwatches on the handles' own streams (for bench.py: torch.cuda.Event sees only torch's
 * streams).  The batch stop returns the latest completion over its compute, copy and output streams. */
int ekf_timer_start(ekf_filter* h);
int ekf_timer_stop(ekf_filter* h, float* ms_out);
int ekf_batch_timer_start(ekf_batch* b);
int ekf_batch_timer_stop(ekf_batch* b, float* ms_out);
/* kernels launched by this handle so far (bench.py's gpu_launches) */
int ekf_batch_launch_count(ekf_batch* b, uint64_t* out);
int ekf_launch_count(ekf_filter* h, uint64_t* out);

/* ------------------------------------------------------------------ helpers on the path */
/* rigid2d::normalize_angle                                      rigid2d/src/rigid2d.cpp:336-345
 * evaluated ON THE DEVICE for `count` values (parity seam for the device twin). */
int ekf_normalize_angles(const double* in, double* out, int64_t count, int device);
/* DiffDrive::getBodyTwistForUpdate(left, right) -> out2 = {angular, linear_x}
 *                                                               rigid2d/src/diff_drive.cpp:38-47 */
int ekf_body_twist(double wheel_base, double wheel_radius, double left, double right, double* out2);
/* DiffDrive::updatePose for `count` independent odometers (rigid2d/src/diff_drive.cpp:50-67 with integrateTwist,
 * rigid2d/src/rigid2d.cpp:304-333, and the acos / asin rotation of Transform2D::operator*=, :222-245):
 * poses [count][3] = {x, y, theta} are advanced in place by the wheel angle increments left / right [count].
 * HOST buffers; theta is not wrapped (as in the reference). */
int ekf_update_pose(double wheel_base, double wheel_radius, int64_t count, double* poses, const double* left,
                    const double* right);

#ifdef __cplusplus
}
#endif
#endif /* EKF_SLAM_B200_H */

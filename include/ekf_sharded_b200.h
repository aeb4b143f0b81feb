/* ekf_sharded_b200.h — one EKF-SLAM filter whose covariance is row-block-sharded over several GPUs
 * (BASELINE.json cfg5: n = 40,000 landmarks, Sigma = 80,003^2 fp64 = 51 GB).  Same verbs as ekf_slam_b200.h
 * (rigid2d::EKF_SLAM, rigid2d/src/ekf_slam.cpp:27-418); one process per GPU, every rank calls every verb with the
 * same arguments (SPMD).  Library: ekf-slam-ml_b200/libekfslam_sharded_b200.so (links NCCL).
 *
 * Partition: rank g owns the rows of landmarks [L_g, L_g+1) (two rows each, never split) and rank 0 additionally
 * the three robot rows; every rank holds all N columns of its rows, a replica of the state vector, and runs the
 * rank-2 sweep on its own rows only.  Per correction the ranks exchange
 *   W = Hj*Sigma (2 x N): the sum of the owners' partial products (W comes from ROWS, as in the reference) - an
 *   ncclAllReduce, or, with an attached exchange buffer (below), stores of the at most two non-zero partials into every
 *   rank's buffer from inside the correction kernel;
 *   every replica then forms K = W^T S^-1 (Sigma symmetric) and the state update locally, so K is not exchanged;
 * per associated measurement additionally the 3 x N robot rows (broadcast from rank 0) and one 24-byte
 * (distance, runner-up, index) triple per rank.
 */
#ifndef EKF_SHARDED_B200_H
#define EKF_SHARDED_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ekf_sharded ekf_sharded;

const char* ekf_sharded_last_error(void);
/* ncclGetUniqueId on one rank; ship the 128 bytes to the others (torch.distributed, MPI, a file ...) */
int ekf_sharded_unique_id(void* id128);
/* collective: one rank of a `world`-way sharded filter on `device` */
int ekf_sharded_create(int n_landmarks, int rank, int world, const void* id128, int device, ekf_sharded** out);
/* single-process emulation of `world` ranks on ONE device (exchanges become device copies): lets the sharding
 * arithmetic be parity-tested on a single GPU, as B200_PROFILING.md asks for when ranks outnumber GPUs */
int ekf_sharded_create_local(int n_landmarks, int world, int device, ekf_sharded** out);
int ekf_sharded_destroy(ekf_sharded* h);
/* Optional: exchange W without a collective.  Per correction only rank 0 (robot rows) and the landmark's owner hold
 * non-zero parts of W = Hj*Sigma; with an attached exchange buffer they store their parts straight into every rank's
 * buffer over NVLink (through the NVSwitch multicast address when one is given) and the correction kernel - one launch
 * for partial W, stores, flags, gain and state update - waits on per-block flags instead of on an ncclAllReduce.  The caller allocates one symmetric, zero-filled buffer of
 * ekf_sharded_exchange_bytes() bytes per rank (e.g. torch.distributed._symmetric_memory, or cudaIpc) and passes every
 * rank's mapping of it (peer_bases[0..world-1]) and the multicast address (0 = none).  Collective; the buffers must
 * outlive the handle.  Results are identical to the all-reduce path.  The correction kernel's CTAs wait for one another,
 * so its whole grid (ld / 256 CTAs) has to be resident on the device at once: for larger maps (on a B200, from about
 * n = 94,700 landmarks) the call returns an error, attaches nothing, and the handle keeps the all-reduce. */
int ekf_sharded_exchange_bytes(ekf_sharded* h, uint64_t* bytes);
int ekf_sharded_attach_exchange(ekf_sharded* h, int world, const uint64_t* peer_bases, uint64_t multicast_base);

int ekf_sharded_predict(ekf_sharded* h, double dtheta, double dx);                         /* ekf_slam.cpp:55-106  */
int ekf_sharded_measurement(ekf_sharded* h, const double* xy, const uint8_t* visible);     /* ekf_slam.cpp:108-197 */
int ekf_sharded_data_association(ekf_sharded* h, const double* xy, int m, uint8_t* known, int32_t* assoc_out,
                                 double* dmin_out, double* second_out, uint8_t* created_out); /* :278-402 */

int ekf_sharded_get_state(ekf_sharded* h, double* out /* N */);
/* rows [row_begin, row_end) owned by shard `shard` (NCCL mode: shard must be 0 = this rank) */
int ekf_sharded_rows(ekf_sharded* h, int shard, int64_t* row_begin, int64_t* row_end);
int ekf_sharded_get_sigma_rows(ekf_sharded* h, int shard, double* out, int64_t ld);
/* `count` selected GLOBAL rows, all owned by `shard` (N doubles each, row stride ld in `out`) */
int ekf_sharded_get_sigma_row_list(ekf_sharded* h, int shard, const int64_t* rows, int count, double* out, int64_t ld);
int ekf_sharded_update_count(ekf_sharded* h, uint64_t* out);
/* As ekf_set_carry_pending / ekf_sweep_count of ekf_slam_b200.h: correction factors stay pending across prediction()
 * and measurement() calls by default (every rank must use the same setting); verbs that read Sigma settle them. */
int ekf_sharded_set_carry_pending(ekf_sharded* h, int carry);
/* As ekf_set_max_pending (1..20, default 14); collective: every rank must use the same setting */
int ekf_sharded_set_max_pending(ekf_sharded* h, int max_pending);
int ekf_sharded_sweep_count(ekf_sharded* h, uint64_t* out);
int ekf_sharded_launch_count(ekf_sharded* h, uint64_t* out);
int ekf_sharded_sync(ekf_sharded* h);
int ekf_sharded_timer_start(ekf_sharded* h);
int ekf_sharded_timer_stop(ekf_sharded* h, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* EKF_SHARDED_B200_H */

/*
 * include/icet_b200.h -- C ABI of the B200-native ICET registration hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  It replaces the
 * work done inside the reference constructor
 *     ICET::ICET(MatrixXf& scan1, MatrixXf& scan2, int runlen, VectorXf X0, int num_bins_phi,
 *                int num_bins_theta, int n, float thresh, float buff)
 *                                              reference include/icet.h:38-40, src/icet.cpp:29-63
 * i.e. fitScan1 (src/icet.cpp:68-107), prepScan2 (:254-277) and runlen x fitScan2 (:372-436).
 * The reference has no FFI/plugin layer of its own (SURVEY.md 8b): its boundary is `class ICET`,
 * which include/icet.h of this repo re-declares and forwards to the entry points below.
 *
 * Everything runs on the GPU (hand-written sm_100a kernels).  There is NO CPU fallback: every
 * entry point fails with a non-zero status if no CUDA device is usable.
 *
 * Clouds are column-major N x 3 float32 (x-plane | y-plane | z-plane, leading dimension ld >= n),
 * which is the memory of Eigen::MatrixXf::data() -- zero-copy from the reference's caller types.
 */
#ifndef ICET_B200_H
#define ICET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICET_B200_VERSION 105

/* status codes (return values; also icet_b200_result.status for per-pair conditions) */
enum {
  ICET_B200_OK = 0,
  ICET_B200_COND_OVERFLOW = 1, /* checkCondition (src/icet.cpp:469-486) ran out of axes: the
                                  reference would abort on an Eigen bounds assert here          */
  ICET_B200_LOOP_TIMEOUT = 2,  /* internal: a wait inside the persistent loop kernel gave up (results invalid)   */
  ICET_B200_E_INVALID = -1,    /* bad argument                                                   */
  ICET_B200_E_CUDA = -2,       /* CUDA runtime error (see icet_b200_last_error)                  */
  ICET_B200_E_NODEVICE = -3,   /* no usable CUDA device / wrong architecture                     */
  ICET_B200_E_NOMEM = -4
};

/* ctor arguments of the reference (include/icet.h:38-40) */
typedef struct {
  int32_t runlen;     /* Gauss-Newton iterations (7 in icet_cpp_demo / odometry, 12 in simpleMapMaker) */
  int32_t bins_phi;   /* num_bins_phi   (elevation, pi / bins_phi each)   -- NB: phi comes first        */
  int32_t bins_theta; /* num_bins_theta (azimuth, 2 pi / bins_theta each)                               */
  int32_t n;          /* minimum cluster size (default 25)                                              */
  float thresh;       /* radial jump threshold (default 0.1)                                            */
  float buff;         /* radial buffer added to the cluster bounds (default 0.1)                        */
  int32_t flags;      /* ICET_B200_FLAG_*                                                               */
  int32_t reserved;
} icet_b200_params;

enum {
  ICET_B200_FLAG_FULL_EIG = 1, /* always run the 6x6 eigen-decomposition of checkCondition (reports the
                                 exact condition number); default: only when a cheap bound cannot
                                 prove cond <= 1e6 (identical results either way)                      */
  /* The Gauss-Newton loop has two forms with the same per-voxel arithmetic: ONE persistent kernel for all
   * iterations (warps draw dependency-ordered tasks; lowest latency for a single pair) and three launches per
   * iteration (highest throughput for large chunks).  Default: persistent for single-pair chunks. */
  ICET_B200_FLAG_UNFUSED_LOOP = 2,   /* always three launches per iteration */
  ICET_B200_FLAG_PERSISTENT_LOOP = 4, /* always the persistent kernel        */
  /* Odometry chaining (odometry.cpp:82 `X0 << X[0], X[1], ...`): the pairs of a batch / sequence call are
   * registered in order and pair k+1 starts from the solution of pair k.  `x0` then holds ONE seed (6 floats, pair 0)
   * or NULL.  Runs as the persistent kernel with pair-major task order; nothing returns to the host in between. */
  ICET_B200_FLAG_CHAIN_X0 = 8,
  /* Compatibility / validation mode, single pair only (icet_b200_register, icet_b200_register_clouds): findCluster
   * walks the points of each cell in the row order the reference ACTUALLY ends up with.  Its "radial sort"
   * (src/icet.cpp:72-83) index-sorts by range and then applies the permutation with a loop that is not a valid
   * permutation application, so the rows stay in a pseudo-random order; findCluster (:557-607) then finds far fewer
   * clusters than the sorted order the comments intend (89 instead of 336 Gaussians on the bundled pair).  The default
   * of this library is the intended, sorted order.  With this flag the host reproduces the shipped row order (the very
   * same std::sort call and swap loop, on the ranges the device computed) and the device clusters in that order --
   * slower (one host round trip), for checking results against an unmodified reference build. */
  ICET_B200_FLAG_SHIPPED_ORDER = 16,
  /* Scan 2 in the Gauss-Newton loop.  Default: INCREMENTAL -- exact integer moments of the untransformed members of
   * every voxel are kept across iterations, a point is re-evaluated (transform, spherical coordinates, voxel, cluster
   * box) only when the transform has moved it further than its margin to the nearest deciding threshold, and the
   * voxel mean / covariance follow from the moments analytically ((mean + t) R, R^T Cov R).  Voxel membership is the
   * per-point pipeline's in every iteration; mean / covariance differ from the reference's by the rounding noise of
   * its per-point fp32 round trip (DESIGN.md).
   * EXACT_PASS: every iteration runs the reference's per-point pipeline on every point (transform, c2s, filter,
   * sphericalToCartesian, src/icet.cpp:375-403 + :303-306) -- the validation form, about 3x slower in the loop.
   * FULL_REBUILD (diagnostic): incremental bookkeeping, but every iteration re-evaluates every point. */
  ICET_B200_FLAG_EXACT_PASS = 32,
  ICET_B200_FLAG_FULL_REBUILD = 64,
  /* Self-check of the incremental loop (tests): every point is re-evaluated in every iteration, and a point that the
   * margin test would have skipped but whose class changed is counted in icet_b200_result.reserved[0]; every point
   * whose filtered (approximate-angle) evaluation disagrees with the exact fp32 pipeline in reserved[1].  Both must
   * stay 0.  Results are bit-identical to the default form. */
  ICET_B200_FLAG_VERIFY_INCREMENTAL = 128,
  /* Form of the loop for the latency shape (single pairs, chained pairs): default = the loop of a pair inside ONE
   * thread-block cluster (hardware cluster barriers between the phases of an iteration, the 28 partial sums reduced
   * through distributed shared memory); ICET_B200_FLAG_PERSISTENT_LOOP selects the older GPU-wide persistent kernel
   * (global-memory flags).  CLUSTER_LOOP forces the cluster form for any chunk (one cluster per pair, round robin). */
  ICET_B200_FLAG_CLUSTER_LOOP = 256
};

/* per-pair result: the members callers of `class ICET` read (X: all four callers; pred_stds:
 * odometry.cpp:79, simpleMapMaker.cpp:122) plus the 6x6 error-bound covariance the reference
 * computes but drops (noise_mat, src/icet.cpp:410-411). */
typedef struct {
  float X[6];          /* x, y, z, phi, theta, psi   (p' = (p + t) * R(phi,theta,psi), src/icet.cpp:375-378) */
  float pred_stds[6];  /* sqrt|diag Q| (+ the checkCondition inflation of :479 when axes are dropped)         */
  float Q[36];         /* pinv(H^T W H) of the last iteration, row-major                                      */
  int32_t status;      /* ICET_B200_OK or ICET_B200_COND_OVERFLOW                                             */
  int32_t n_gauss1;    /* voxels that got a scan-1 Gaussian                                                   */
  int32_t n_used;      /* voxels that contributed to H^T W H in the last iteration                            */
  int32_t n_dropped;   /* solution axes dropped by checkCondition in the last iteration                       */
  float cond;          /* lambda_max/lambda_min of H^T W H if the eigen-decomposition ran, else the upper
                          bound trace(A)*trace(A^-1) negated (always <= 1e6 in magnitude then)                */
  int32_t reserved[3];
} icet_b200_result;    /* 56 x 4 bytes */

typedef struct icet_b200_ctx icet_b200_ctx; /* device workspace + stream; one per host thread */

/* -- lifecycle ------------------------------------------------------------------------------ */
int icet_b200_version(void);
/* Thread-local description of the last failure on the calling thread. */
const char* icet_b200_last_error(void);
/* device < 0: use the current CUDA device.  Fails (no fallback) when none is present. */
int icet_b200_create(int device, icet_b200_ctx** ctx);
int icet_b200_destroy(icet_b200_ctx* ctx);
/* All work of a context is issued on one stream (default: a private non-blocking stream).
 * `stream` is a cudaStream_t; pass the caller's stream to order against its own work. */
int icet_b200_set_stream(icet_b200_ctx* ctx, void* stream);
/* Upper bound on the number of pairs processed per internal chunk (workspace ~7.3 MB/pair at
 * 131 072-point scans, per compute lane in use). 0 restores the default (512). */
int icet_b200_set_chunk(icet_b200_ctx* ctx, int32_t max_pairs_per_chunk);
/* Chunk size of the HOST-buffer batch entry point (icet_b200_register_batch): the upload of one chunk overlaps the
 * registration of the previous one, so smaller chunks hide more of the PCIe transfer. 0 restores the default (64). */
int icet_b200_set_host_chunk(icet_b200_ctx* ctx, int32_t pairs_per_chunk);

/* -- registration ---------------------------------------------------------------------------- */
/* One pair, HOST buffers: replaces `ICET it(scan1, scan2, runlen, X0, nPhi, nTheta, n, thresh, buff)`
 * (src/icet.cpp:29-63).  Blocking; copies the inputs to the device and the result back. */
int icet_b200_register(icet_b200_ctx* ctx, const icet_b200_params* p, const float* scan1, int32_t n1,
                       int32_t ld1, const float* scan2, int32_t n2, int32_t ld2, const float x0[6],
                       icet_b200_result* out);

/* A batch of independent pairs, HOST buffers.  scan1[i]/scan2[i] point to clouds of n1[i]/n2[i]
 * points (leading dimension = point count).  x0: npairs*6 floats or NULL (zeros).  A scan that is
 * scan2 of pair i and scan1 of pair i+1 (same pointer, odometry.cpp:73-76 usage) is uploaded once.
 * Blocking. */
int icet_b200_register_batch(icet_b200_ctx* ctx, const icet_b200_params* p, int32_t npairs,
                             const float* const* scan1, const int32_t* n1, const float* const* scan2,
                             const int32_t* n2, const float* x0, icet_b200_result* out);

/* Same, DEVICE buffers: every scan pointer is device memory, x0 (or NULL) and `out` are device
 * memory too.  Asynchronous on the context's stream; nothing is copied to the host. */
int icet_b200_register_batch_device(icet_b200_ctx* ctx, const icet_b200_params* p, int32_t npairs,
                                    const float* const* scan1, const int32_t* n1,
                                    const float* const* scan2, const int32_t* n2, const float* x0,
                                    icet_b200_result* out);

/* Convenience for an odometry sequence stored back to back on the DEVICE: nscans clouds of n points
 * each (scan k at scans + k*3*n); registers the nscans-1 consecutive pairs (k, k+1) with X0 = 0.
 * `out` is device memory for nscans-1 results.  Asynchronous on the context's stream. */
int icet_b200_register_sequence_device(icet_b200_ctx* ctx, const icet_b200_params* p, int32_t nscans,
                                       const float* scans, int32_t n, icet_b200_result* out);

int icet_b200_synchronize(icet_b200_ctx* ctx);
/* Number of compute lanes (streams with their own workspace) consecutive chunks rotate over: 1 .. 8
 * (0 = default 8; a batch uses at most one lane per 512-pair chunk, batches below 4096 pairs at most four). */
int icet_b200_set_lanes(icet_b200_ctx* ctx, int32_t lanes);

/* -- keyframes ---------------------------------------------------------------------------------------------------------
 * Many registrations often share their scan 1: a scan against an accumulated map (scan-to-map localisation), one pair
 * from several initial guesses, scans k+1 .. k+m against keyframe k.  The scan-1 half of the reference's constructor
 * (fitScan1, src/icet.cpp:68-107) depends only on scan 1 and the bin parameters, so a keyframe runs it once and keeps
 * its result (cluster bounds, Gaussians, L / U of every voxel) on the device; registrations against it start from there.
 * Results are bit-identical to registering the same pairs with the cloud as scan 1.
 * A keyframe belongs to the context that created it and, like the context, is not thread-safe; destroy it before the
 * context.  Keyframe registrations record no per-voxel dump and, like batches, end the get_points2 / classify_scan2
 * record of the last icet_b200_register call. */
typedef struct icet_b200_keyframe icet_b200_keyframe; /* scan-1 state of one cloud, resident on the ctx's device */

/* fitScan1 once.  p: bins_phi, bins_theta, n, thresh, buff and ICET_B200_FLAG_SHIPPED_ORDER are fixed for the keyframe;
 * runlen and the other flags are ignored.  HOST planes (leading dimension ld1), blocking. */
int icet_b200_keyframe_create(icet_b200_ctx* ctx, const icet_b200_params* p, const float* scan1, int32_t n1,
                              int32_t ld1, icet_b200_keyframe** kf);
/* Same, scan1 in DEVICE memory (e.g. a map from icet_b200_map_get_device with a host-known count).  Blocking. */
int icet_b200_keyframe_create_device(icet_b200_ctx* ctx, const icet_b200_params* p, const float* scan1, int32_t n1,
                                     int32_t ld1, icet_b200_keyframe** kf);
int icet_b200_keyframe_destroy(icet_b200_keyframe* kf);   /* synchronises the ctx's stream first */
int icet_b200_keyframe_gaussians(icet_b200_keyframe* kf); /* = result.n_gauss1 of every registration against it */

/* The registrations below require p to agree with the keyframe in bins_phi, bins_theta, n, thresh, buff and
 * ICET_B200_FLAG_SHIPPED_ORDER, and reject ICET_B200_FLAG_CHAIN_X0 (ICET_B200_E_INVALID).  runlen and the loop / scan-2
 * flags apply per call, as in a batch. */
/* icet_b200_register with scan 1 = the keyframe.  HOST scan 2, blocking. */
int icet_b200_register_keyframe(icet_b200_keyframe* kf, const icet_b200_params* p, const float* scan2, int32_t n2,
                                int32_t ld2, const float x0[6], icet_b200_result* out);
/* icet_b200_register_batch_device with scan1[i] = the keyframe for every i: scan2[i] DEVICE pointers (host table),
 * x0 (npairs*6 or NULL) and out DEVICE memory, asynchronous on the ctx's stream. */
int icet_b200_register_keyframe_batch_device(icet_b200_keyframe* kf, const icet_b200_params* p, int32_t npairs,
                                             const float* const* scan2, const int32_t* n2, const float* x0,
                                             icet_b200_result* out);

/* -- per-voxel state of the most recent single-pair call (icet_b200_register) ------------------
 * Mirrors the public members the reference exposes for visualisation / debugging:
 *   clusterBounds (include/icet.h:83), sigma1/mu1/L/U (:89-94), pointIndices sizes (:95-96).
 * Any pointer may be NULL.  ncell = bins_phi*bins_theta, cell = bins_theta*phi + theta. HOST memory. */
typedef struct {
  int32_t* cnt1;     /* [ncell] points of scan 1 per angular bin                                  */
  float* bounds;     /* [ncell*6] azMin azMax elMin elMax inner outer (clusterBounds rows)        */
  int32_t* nin1;     /* [ncell] scan-1 points inside the cluster box                              */
  uint8_t* has1;     /* [ncell] Gaussian fitted                                                   */
  float* mu1;        /* [ncell*3]                                                                 */
  float* sigma1;     /* [ncell*9]                                                                 */
  float* evec1;      /* [ncell*9] row-major V (columns = eigenvectors, ascending eigenvalues)     */
  float* eval1;      /* [ncell*3]                                                                 */
  uint8_t* lmask;    /* [ncell*3] diagonal of L                                                   */
  /* scan 2 per iteration [runlen][ncell...] */
  int32_t* cnt2;
  int32_t* nin2;
  uint8_t* used2;
  float* mu2;        /* [runlen*ncell*3] */
  float* sigma2;     /* [runlen*ncell*9] */
  float* Xit;        /* [runlen*6]  X after each iteration     */
  float* HTWH;       /* [runlen*36] */
  float* HTWdz;      /* [runlen*6]  */
  float* TRit;       /* [runlen*12] trans (3) | rot_mat (9, row-major) every iteration used (src/icet.cpp:375-376) */
  float* testPoints; /* [ncell*6*3] the reference's public member testPoints (include/icet.h:84), row-major 6*ncell x 3:
                        rows 6*cell+2k, +2k+1 hold the two 2-sigma test points of axis k when that axis was found
                        extended (L(k,k) = 0, src/icet.cpp:214-232); all other rows are 0 (uninitialised in the
                        reference)                                                                               */
} icet_b200_voxel_dump;

/* Enable (1) / disable (0) recording of the per-voxel state for subsequent icet_b200_register calls. */
int icet_b200_set_dump(icet_b200_ctx* ctx, int32_t enable);
int icet_b200_get_dump(icet_b200_ctx* ctx, icet_b200_voxel_dump* out);

/* The reference's public member `points2` (include/icet.h:80) for the most recent icet_b200_register call: scan 2
 * as transformed by the LAST iteration, i.e. with the X that iteration started from (src/icet.cpp:375-378 runs
 * before :433), in the caller's point order (the reference leaves it in its internal permuted order).
 * out: HOST buffer of 3*n2 floats (planes), n2 must equal the registered size. */
int icet_b200_get_points2(icet_b200_ctx* ctx, float* out, int32_t n2);

/* Parity-test entry: the class the per-point pipeline (transform, cartesianToSpherical, sortSphericalCoordinates,
 * filterPointsInsideCluster; src/icet.cpp:375-388, :290-300) gives every point of scan 2 of the most recent DUMPED
 * icet_b200_register call in iteration `iter`, in the caller's point order: cell[n2] = bins_theta*phi + theta,
 * in[n2] = 1 if the point is inside the cluster box of a voxel that has a scan-1 Gaussian and passes the scan-1 gates
 * of fitCells2 (`indices1.size() > n`, `outer > 1`).  HOST buffers, blocking. */
int icet_b200_classify_scan2(icet_b200_ctx* ctx, int32_t iter, int32_t* cell, uint8_t* in, int32_t n2);

/* Stage outputs used by the parity tests (HOST buffers, blocking):
 * spherical coordinates [3*n] (r | theta | phi) and the cell index of each point,
 * utils::cartesianToSpherical (src/utils.cpp:93-119) + ICET::sortSphericalCoordinates (src/icet.cpp:545-546). */
int icet_b200_spherical_bins(icet_b200_ctx* ctx, const icet_b200_params* p, const float* scan, int32_t n,
                             int32_t ld, float* sph, int32_t* cell);

/* -- callers either side of the path (SURVEY.md 8f rows N1, N2) --------------------------------------------------
 * The two ROS nodes of the reference wrap the constructor in the same few steps; these entry points keep those steps
 * on the device so that filtered clouds, their data-dependent sizes, the seed of the next registration and the
 * accumulated pose never visit the host:
 *   OdometryNode::pointcloudCallback   src/odometry.cpp:38-168        (min_range 2, runlen 7, chain_x0 1, no guard)
 *   MapMakerNode::pointcloudCallback   src/simpleMapMaker.cpp:78-240  (min_range 0.2, runlen 12, chain_x0 0, guard 0.3)
 */
typedef struct {
  float min_range;     /* keep rows with ||p|| > min_range (odometry.cpp:57-70: 2.0; simpleMapMaker.cpp:100-112: 0.2);
                          < 0: keep every row                                                                      */
  int32_t chain_x0;    /* 1: X0 of the next registration = X of this one (odometry.cpp:82);
                          0: X0 = 0 every time (simpleMapMaker.cpp:124)                                            */
  float rate_hz;       /* twist = rate_hz * X (odometry.cpp:134-139 assumes a 10 Hz sensor)                        */
  float guard_trans;   /* divergence guard (simpleMapMaker.cpp:128-137, :241-242: 0.3 / 0.3): if any |X| exceeds    */
  float guard_rot;     /* its threshold the pose update uses X = 0;  <= 0: no guard (odometry.cpp has none)         */
  int32_t reserved[3];
} icet_b200_odometry_params;

/* what the nodes publish per registration (nav_msgs::Odometry of odometry.cpp:104-140, the tf of both nodes) */
typedef struct {
  float X_homo[16];         /* accumulated transform, row-major 4x4 (X_homo = X_homo * X_homo_i, odometry.cpp:87-98)  */
  float position[3];        /* X_homo(0..2, 3)                                              odometry.cpp:110-112      */
  float orientation[4];     /* Eigen::Quaternionf(X_homo.topLeftCorner(3,3)) as x, y, z, w  odometry.cpp:114-119      */
  float covariance_diag[6]; /* pose.covariance[0,7,14,21,28,35] = pred_stds                 odometry.cpp:126-131      */
  float twist[6];           /* rate_hz * X                                                  odometry.cpp:134-139      */
  float X[6];               /* the registration result the pose update used (after the guard)                         */
  int32_t n_points;         /* rows of the current scan that passed the min-range filter                              */
  int32_t guarded;          /* 1: the divergence guard replaced X by 0                                                */
  int32_t frame;            /* registrations so far (frameCount - 1)                                                  */
  int32_t reserved;
} icet_b200_pose;           /* 45 x 4 bytes */

typedef struct icet_b200_node icet_b200_node; /* state of one node: prev_pcl_matrix, X0, X_homo (all device resident) */

/* max_points: capacity per scan.  X_homo0 (16 floats, row-major) / x0 (6 floats): HOST, NULL = identity / zeros. */
int icet_b200_node_create(icet_b200_ctx* ctx, const icet_b200_params* p, const icet_b200_odometry_params* op,
                          int32_t max_points, const float* X_homo0, const float* x0, icet_b200_node** node);
int icet_b200_node_destroy(icet_b200_node* node);
/* The callback for `nscans` consecutive scans in DEVICE memory ([nscans][3][n] planes), asynchronous on the context's
 * stream.  The very first scan a node sees only becomes prev_pcl_matrix, unfiltered (odometry.cpp:47-52); every other
 * scan is filtered and registered against its predecessor.  res / poses: DEVICE arrays with room for nscans entries.
 * Returns the number of registrations enqueued (nscans, or nscans - 1 on the first call) or a negative status.
 * With chain_x0 the registrations run as ONE persistent kernel in chain order (ICET_B200_FLAG_CHAIN_X0). */
int icet_b200_node_push_device(icet_b200_node* node, int32_t nscans, const float* scans, int32_t n,
                               icet_b200_result* res, icet_b200_pose* poses);
/* The callback for one scan in HOST memory (planes, leading dimension ld), blocking.  Returns 0 when the scan only
 * initialised the node, 1 when *res / *pose were written. */
int icet_b200_node_push(icet_b200_node* node, const float* scan, int32_t n, int32_t ld, icet_b200_result* res,
                        icet_b200_pose* pose);
/* The filtered current scan (= prev_pcl_matrix for the next callback): device planes, leading dimension *ld, row count
 * in device memory at *n_dev.  Valid until the next push. */
int icet_b200_node_current_scan(icet_b200_node* node, const float** scan, const int32_t** n_dev, int32_t* ld);
/* The device-resident result of the most recent registration (NULL before the first one). */
int icet_b200_node_last_result(icet_b200_node* node, const icet_b200_result** res_dev);

/* The rigid re-expressions the nodes apply to whole clouds, with trans / rot_mat taken from X = (x y z phi theta psi) in
 * DEVICE memory (e.g. &result->X), rot_mat.inverse() by cofactors like Eigen's 3x3 inverse:
 *   mode 0:  out = (cloud * rot_mat.inverse()).rowwise() - trans   scan 2 in the frame of scan 1, scanMatcher.cpp:73;
 *                                                                   the snail trails, scanMatcher.cpp:76, simpleMapMaker.cpp:222
 *   mode 1:  out = (cloud.rowwise() - trans) * rot_mat.inverse()   EigenQueue::add_new_scan, simpleMapMaker.cpp:41
 * cloud / out: DEVICE planes (leading dimensions ld / ld_out; out may alias cloud), n rows or *n_dev rows when n_dev is
 * given (device-resident count, clipped to n).  Asynchronous on the context's stream. */
int icet_b200_transform_cloud_device(icet_b200_ctx* ctx, const float* cloud, int32_t n, int32_t ld, const int32_t* n_dev,
                                     const float* X, int32_t mode, float* out, int32_t ld_out);
/* Same with the result in HOST memory (planes, leading dimension ld_out >= n), blocking: what a node publishes. */
int icet_b200_transform_cloud(icet_b200_ctx* ctx, const float* cloud, int32_t n, int32_t ld, const float* X, int32_t mode,
                              float* out, int32_t ld_out);

/* EigenQueue (simpleMapMaker.cpp:18-58): FIFO of map points (600 000 in the reference, :62), re-expressed in the
 * newest sensor frame at every insertion. */
typedef struct icet_b200_map icet_b200_map;
int icet_b200_map_create(icet_b200_ctx* ctx, int32_t capacity, icet_b200_map** map);
int icet_b200_map_destroy(icet_b200_map* map);
/* EigenQueue::add_new_scan(newScan, trans, rot_mat) (:34-42): append rows of the DEVICE cloud `scan` (n rows, leading
 * dimension ld; n_dev: optional device-resident row count, e.g. from icet_b200_node_current_scan) and re-express every
 * stored row, `(matrix.rowwise() - trans) * rot_mat.inverse()`, with trans / rot_mat from X (6 floats, DEVICE memory,
 * e.g. &result->X) after the divergence guard (<= 0: none).  idx: HOST list of `count` row numbers to append in that
 * order -- the shuffled prefix of simpleMapMaker.cpp:150-159 -- or NULL for rows 0 .. count-1.  Asynchronous. */
int icet_b200_map_add_scan_device(icet_b200_map* map, const float* scan, int32_t n, int32_t ld, const int32_t* n_dev,
                                  const int32_t* idx, int32_t count, const float* X, float guard_trans,
                                  float guard_rot);
/* EigenQueue::getQueue (:44-51): rows oldest first.  out: planes with leading dimension ld_out (>= capacity unless the
 * caller knows better), HOST memory, blocking / DEVICE memory, asynchronous (n_out then device memory too). */
int icet_b200_map_get(icet_b200_map* map, float* out, int32_t ld_out, int32_t* n_out);
int icet_b200_map_get_device(icet_b200_map* map, float* out, int32_t ld_out, int32_t* n_out);

/* -- ingest (SURVEY.md 8f row N3) ----------------------------------------------------------------------------------
 * The reference's callers all convert what they hold into an N x 3 Eigen::MatrixXf on the host, one element at a time:
 * convertPCLtoEigen (odometry.cpp:186-192) from the PointCloud2 records, loadPointCloudCSV (src/utils.cpp:19-61) from
 * integer millimetres, the notebooks from float64 .npy arrays.  These entry points take the caller's buffer as it is:
 * the raw bytes cross PCIe once and one kernel writes the x | y | z planes the path reads. */
enum { ICET_B200_F32 = 0, ICET_B200_F64 = 1, ICET_B200_I32 = 2 };
typedef struct {
  const void* data;    /* HOST: n records of point_step bytes                                                          */
  int32_t n;
  int32_t point_step;  /* bytes per record: 12 numpy float32 N x 3, 24 float64 N x 3, 16 pcl::PointXYZ, PointCloud2.point_step */
  int32_t off[3];      /* byte offsets of x, y, z inside a record (PointCloud2.fields[k].offset); multiples of the
                          element size, like point_step                                                                */
  int32_t dtype;       /* ICET_B200_F32 | ICET_B200_F64 (rounded to float like Eigen's cast<float>()) | ICET_B200_I32  */
  float divide;        /* value = float(raw) / divide when != 0 and != 1 (src/utils.cpp:51: integer mm `/ 1000`)        */
  int32_t plane_stride; /* 0: records (array of structures).  > 0: the buffer holds three planes of n elements,
                           plane k starting plane_stride elements after plane k-1 (numpy Fortran order: n)             */
} icet_b200_cloud;
/* Converts one HOST cloud into DEVICE planes (out: 3 planes, leading dimension ld >= n).  Asynchronous on the context's
 * stream once the raw bytes are staged (the call returns after the host buffer has been read). */
int icet_b200_ingest(icet_b200_ctx* ctx, const icet_b200_cloud* cloud, float* out, int32_t ld);
/* icet_b200_register for two clouds in their native layout (blocking). */
int icet_b200_register_clouds(icet_b200_ctx* ctx, const icet_b200_params* p, const icet_b200_cloud* scan1,
                              const icet_b200_cloud* scan2, const float x0[6], icet_b200_result* out);
/* icet_b200_node_push for a cloud in its native layout, e.g. straight from a sensor_msgs::PointCloud2 (blocking). */
int icet_b200_node_push_cloud(icet_b200_node* node, const icet_b200_cloud* cloud, icet_b200_result* res,
                              icet_b200_pose* pose);

/* -- keyframe odometry (DESIGN.md §13) --------------------------------------------------------------------------------
 * An odometry node that registers every filtered scan against its current KEYFRAME instead of its predecessor, so
 * that the registration errors of the scans between two keyframes do not add up.  Per scan k (after the first):
 *   - min-range filter as in icet_b200_node_push_device; the very first scan is stored unfiltered and is keyframe 0,
 *     with pose X_homo0;
 *   - registration against keyframe f seeded with x0_k; its X is X_rel, scan k relative to keyframe f;
 *   - pose X_homo_k = X_homo_f * Hi(X_rel), Hi = [R(X3,X4,X5) t; 0 1], the float product of icet_b200_node_push_device
 *     (quaternion, covariance diagonal = pred_stds as there; twist = rate_hz * step_k; pose.X = X_rel);
 *   - frame step step_k = X_rel verbatim when f = k-1, else params(Hi(X_rel,k-1)^-1 Hi(X_rel,k)) (both share f);
 *     params(H) = translation column verbatim, angles from the inverse of R(), evaluated in double;
 *   - next seed with chain_x0 = 1: params(Hi(X_rel,k) Hi(step_k)) (constant velocity), or step_k when scan k was
 *     promoted; with chain_x0 = 0 always 0;
 *   - promotion: scan k becomes the keyframe of scan k+1 when any enabled test of the policy fires (below) or
 *     result.status != ICET_B200_OK.
 * A policy that promotes every scan (max_interval = 1, other tests off) reproduces icet_b200_node_push_device bit for
 * bit.  Filtered clouds, their sizes, the keyframe's scan-1 fit, seeds and poses stay on the device. */
typedef struct {
  float max_trans;      /* promote when ||X_rel[0..2]|| > max_trans (m)                                    */
  float max_rot;        /* promote when max |X_rel[3..5]| > max_rot (rad)                                  */
  float min_overlap;    /* promote when result.n_used < min_overlap * n_gauss1 of the keyframe             */
  int32_t max_interval; /* promote when max_interval scans have been registered against the keyframe       */
  int32_t reserved[4];  /* must be 0;  a threshold <= 0 turns its test off                                 */
} icet_b200_keyframe_policy;

enum { /* icet_b200_kf_info.reason: one bit per test that fired */
  ICET_B200_KF_TRANS = 1,
  ICET_B200_KF_ROT = 2,
  ICET_B200_KF_OVERLAP = 4,
  ICET_B200_KF_INTERVAL = 8,
  ICET_B200_KF_STATUS = 16
};

typedef struct {
  int32_t keyframe;  /* frame index of the keyframe the scan was registered against (0 = the first scan) */
  int32_t promoted;  /* 1: this scan is the keyframe of the next one                                    */
  int32_t reason;    /* ICET_B200_KF_* bits                                                             */
  float x0[6];       /* the seed the registration started from                                          */
  int32_t reserved;
} icet_b200_kf_info; /* 10 x 4 bytes */

typedef struct icet_b200_kfnode icet_b200_kfnode;

/* op: min_range, chain_x0 and rate_hz as for icet_b200_node_create; guard_trans / guard_rot must be <= 0.  p must not
 * carry ICET_B200_FLAG_CHAIN_X0 (the node seeds every registration itself) or ICET_B200_FLAG_SHIPPED_ORDER (its scan-1
 * fit needs a host round trip).  max_points: capacity per scan (the huge-cell path of the scan-1 fit stays off below
 * 262 144).  X_homo0 (16 floats) / x0 (6 floats, the seed of the first registration with chain_x0): HOST or NULL. */
int icet_b200_kfnode_create(icet_b200_ctx* ctx, const icet_b200_params* p, const icet_b200_odometry_params* op,
                            const icet_b200_keyframe_policy* kp, int32_t max_points, const float* X_homo0,
                            const float* x0, icet_b200_kfnode** node);
int icet_b200_kfnode_destroy(icet_b200_kfnode* node);
/* `nscans` consecutive scans in DEVICE memory ([nscans][3][n] planes), asynchronous on the context's stream.
 * res / poses / info: DEVICE arrays with room for nscans entries (info may be NULL).  Returns the number of
 * registrations enqueued (nscans, or nscans - 1 on the node's first call).  Equals nscans blocking pushes byte for
 * byte: a promotion takes effect for the very next scan. */
int icet_b200_kfnode_push_device(icet_b200_kfnode* node, int32_t nscans, const float* scans, int32_t n,
                                 icet_b200_result* res, icet_b200_pose* poses, icet_b200_kf_info* info);
/* One scan in HOST memory (planes, leading dimension ld), blocking.  Returns 0 for the first scan, else 1. */
int icet_b200_kfnode_push(icet_b200_kfnode* node, const float* scan, int32_t n, int32_t ld, icet_b200_result* res,
                          icet_b200_pose* pose, icet_b200_kf_info* info);
/* icet_b200_kfnode_push for a cloud in its native layout (blocking). */
int icet_b200_kfnode_push_cloud(icet_b200_kfnode* node, const icet_b200_cloud* cloud, icet_b200_result* res,
                                icet_b200_pose* pose, icet_b200_kf_info* info);
/* The current keyframe's filtered cloud: device planes, leading dimension *ld, row count in device memory at *n_dev.
 * Valid until the next push. */
int icet_b200_kfnode_keyframe(icet_b200_kfnode* node, const float** scan, const int32_t** n_dev, int32_t* ld);

/* Local-map keyframe odometry (DESIGN.md §14): a keyframe odometry node whose scan 1 is the LOCAL MAP, the filtered
 * clouds of its last map_keyframes = M keyframes (1 <= M <= 16) expressed in the frame of the newest keyframe f.
 * Pose, frame step, seeds, promotion policy, icet_b200_kf_info and the rejections are those above; the overlap test
 * uses the map's n_gauss1 (the result's).  The map:
 *   - rows of f first, bit for bit as icet_b200_kfnode_keyframe holds them; then the older keyframes, newest to
 *     oldest; no gaps; row count = the sum of the window's kept counts, in device memory.  (Results do not depend on
 *     the row order; it is fixed so that maps compare byte for byte.)
 *   - Re-expression: registering scan k against f maps p of k into f as (p + t) R(X) (row vectors), so on promotion of
 *     k a point q of f's frame is q R^-1 - t in k's frame (icet_b200_transform_cloud_device mode 0).  Each window
 *     keyframe keeps its original filtered cloud and its transform into the current keyframe frame, composed in double
 *     on the device and applied in float to that original cloud (never to an already re-expressed map).  These
 *     transforms are not derived from the published pose X_homo.
 *   - The window slides: after the (M+1)-th keyframe the oldest leaves it; before M keyframes it holds those there are.
 * M = 1 is icet_b200_kfnode_create byte for byte.  max_points: capacity per scan; M * max_points must not exceed 2^28
 * (the huge-cell path of the candidate fit is on once M * max_points exceeds 262 144).  Everything else as
 * icet_b200_kfnode_create; push / keyframe / destroy take the node as they are. */
int icet_b200_kfnode_create_local_map(icet_b200_ctx* ctx, const icet_b200_params* p, const icet_b200_odometry_params* op,
                                      const icet_b200_keyframe_policy* kp, int32_t map_keyframes, int32_t max_points,
                                      const float* X_homo0, const float* x0, icet_b200_kfnode** node);
/* The current local map (scan 1 of the next registration): device planes, leading dimension *ld, row count in device
 * memory at *n_dev.  Valid until the next push.  For a node of icet_b200_kfnode_create: its keyframe cloud. */
int icet_b200_kfnode_local_map(icet_b200_kfnode* node, const float** cloud, const int32_t** n_dev, int32_t* ld);
/* The same in HOST memory, blocking: *n_out = its row count; with out != NULL the x | y | z planes (leading dimension
 * ld_out >= *n_out) as well.  Call with out = NULL to size the buffer. */
int icet_b200_kfnode_local_map_host(icet_b200_kfnode* node, float* out, int32_t ld_out, int32_t* n_out);

/* -- multi-GPU (SURVEY.md 8e) ---------------------------------------------------------------------------------------
 * The reference's registrations are independent objects ("run multiple ICETs at once", include/icet.h:43), so a batch
 * shards by scan pair: ONE process, one context per device, device d of G registers the contiguous pair range
 * [P d / G, P (d+1) / G); nothing is exchanged during the registration; ONE ncclAllGather of 48 floats per pair
 * (X 6 | pred_stds 6 | Q 36) closes the call, after which every device holds every result.  NCCL is loaded at run time
 * (libnccl.so.2); creation fails without it. */
typedef struct icet_b200_multi icet_b200_multi;
/* devices: ndev distinct CUDA device indices (NULL: 0 .. ndev-1).  Creates one context per device and the communicator
 * (ncclCommInitAll). */
int icet_b200_multi_create(const int32_t* devices, int32_t ndev, icet_b200_multi** multi);
int icet_b200_multi_destroy(icet_b200_multi* multi);
int icet_b200_multi_devices(icet_b200_multi* multi);
/* the context of device slot d (to configure chunks / lanes / streams per device) */
icet_b200_ctx* icet_b200_multi_context(icet_b200_multi* multi, int32_t d);
/* icet_b200_register_batch over all devices: HOST buffers, blocking; `out` (HOST, npairs records) is written by the
 * devices' own downloads; the gathered rows stay on every device (icet_b200_multi_gathered). */
int icet_b200_register_batch_multi(icet_b200_multi* multi, const icet_b200_params* p, int32_t npairs,
                                   const float* const* scan1, const int32_t* n1, const float* const* scan2,
                                   const int32_t* n2, const float* x0, icet_b200_result* out);
/* icet_b200_register_sequence_device over all devices: a sequence of nscans clouds of n points whose consecutive pairs
 * are sharded as above; shard_scans[d] is DEVICE memory on device d holding the scans lo_d .. hi_d of its pair range
 * ([hi_d - lo_d + 1][3][n], one boundary scan is duplicated on the next device).  Blocking. */
int icet_b200_register_sequence_multi_device(icet_b200_multi* multi, const icet_b200_params* p, int32_t nscans,
                                             const float* const* shard_scans, int32_t n);
/* The all-gathered results on device slot d: DEVICE pointer to [ndev][rows_per_shard][48] floats (shard s holds the pairs
 * of device s in order; shards shorter than rows_per_shard are zero padded). */
int icet_b200_multi_gathered(icet_b200_multi* multi, int32_t d, const float** rows, int32_t* rows_per_shard);
/* The same rows copied to HOST memory (`out`: ndev * rows_per_shard * 48 floats), blocking. */
int icet_b200_multi_gathered_host(icet_b200_multi* multi, int32_t d, float* out);

/* -- synthetic 64-channel scans (bench / test utility, SURVEY.md 8d) --------------------------- */
/* Writes nscans consecutive scans (index first_scan ...) of rings x azim points each to DEVICE memory
 * `out` ([nscans][3][rings*azim] float32 planes).  Asynchronous on the context's stream. */
int icet_b200_synth_scans_device(icet_b200_ctx* ctx, uint64_t seed, int32_t first_scan, int32_t nscans,
                                 int32_t rings, int32_t azim, float* out);

/* -- instrumentation ---------------------------------------------------------------------------- */
/* Number of kernels this library has launched on the context since creation. */
int64_t icet_b200_kernel_launches(icet_b200_ctx* ctx);

/* Per-kernel device time: when enabled every kernel launch is bracketed by CUDA events on the context's
 * stream (small overhead -- use a separate pass, not the throughput measurement).  Enabling resets the
 * sums.  get_profile synchronises and returns, per kernel id, the summed milliseconds and launch count. */
#define ICET_B200_NKERNELS 11
int icet_b200_set_profile(icet_b200_ctx* ctx, int32_t enable);
int icet_b200_get_profile(icet_b200_ctx* ctx, double ms[ICET_B200_NKERNELS], int64_t launches[ICET_B200_NKERNELS]);
const char* icet_b200_kernel_name(int id);
/* Debug: %globaltimer stamps [runlen][16] of the persistent loop kernel for the most recent dumped single-pair call
 * (0 last vox task arrived, 1 / 2 begin / end of the latest vox task, 3 partial sums added, 4 solve done,
 * 5 iteration published, 6 / 7 begin / end of tile 0 of the iteration, 8 / 9 algebra / partial sums of the latest
 * vox task done), followed by begin / end stamps of up to 2048 tiles of iteration 3.
 * HOST buffer of runlen*16 + 4096 values. */
int icet_b200_debug_timeline(icet_b200_ctx* ctx, uint64_t* out, int32_t runlen);

#ifdef __cplusplus
}
#endif
#endif /* ICET_B200_H */

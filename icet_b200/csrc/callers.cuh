// icet_b200/csrc/callers.cuh -- device side of the callers either side of the registration path
// (SURVEY.md 8f rows N1 and N2), included by icet_b200.cu inside its anonymous namespace:
//
//   N1  OdometryNode::pointcloudCallback  (reference src/odometry.cpp:38-168)
//         min-range filter :57-70, ICET(prev, cur, ...) :73-76, X0 <- X :82, X_homo accumulation :87-98,
//         pose / covariance diagonal / twist of the nav_msgs::Odometry message :104-140
//   N2  MapMakerNode::pointcloudCallback + EigenQueue  (reference src/simpleMapMaker.cpp:18-58, :78-240)
//         min-range filter :100-112, divergence guard :128-137, down-sample :150-159,
//         EigenQueue::add_new_scan :34-42, EigenQueue::getQueue :44-51
//
// Everything stays on the device: the filtered clouds, their (data dependent) sizes, the pair descriptors built
// from them, the seed of the next registration and the accumulated pose never visit the host.
#pragma once

// ----------------------------------------------------------------------------------------------
// Min-range filter (odometry.cpp:57-70, simpleMapMaker.cpp:100-112): keep row i iff row(i).norm() > minD,
// order preserved.  Two kernels: per-tile counts, then a stable scatter (every tile adds up the counts of the
// tiles before it -- at most a few thousand values).  min_d < 0 keeps every row (also NaN rows).
// ----------------------------------------------------------------------------------------------
constexpr int FILT_THREADS = 256;
constexpr int FILT_ROUNDS = 4;
constexpr int FILT_TILE = FILT_THREADS * FILT_ROUNDS;

struct FilterJob {        // one cloud to filter
  const float* src;       // planes x | y | z, leading dimension ld
  float* dst;             // planes, leading dimension ld_dst
  int32_t* kept;          // [1] number of rows kept
  const int32_t* n_dev;   // number of rows, device resident (or null: n)
  int n, ld, ld_dst;
  float min_d;            // < 0: copy
};

__device__ __forceinline__ bool range_keep(float x, float y, float z, float min_d) {
  if (min_d < 0.f) return true;
  const float s = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  return __fsqrt_rn(s) > min_d;  // `distance > minD` (false for NaN)
}

__global__ void __launch_bounds__(FILT_THREADS) k_range_count(const FilterJob* jobs, int ntile, int32_t* tile_cnt) {
  const FilterJob j = jobs[blockIdx.y];
  const int n = j.n_dev ? min(j.n, *j.n_dev) : j.n;
  const int base = blockIdx.x * FILT_TILE;
  int cnt = 0;
  if (base < n) {
#pragma unroll
    for (int r = 0; r < FILT_ROUNDS; r++) {
      const int i = base + r * FILT_THREADS + threadIdx.x;
      if (i < n) cnt += range_keep(__ldg(j.src + i), __ldg(j.src + j.ld + i), __ldg(j.src + 2 * (size_t)j.ld + i), j.min_d) ? 1 : 0;
    }
  }
  __shared__ int s_w[FILT_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(FULL, cnt, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < FILT_THREADS / 32; w++) t += s_w[w];
    tile_cnt[(size_t)blockIdx.y * ntile + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(FILT_THREADS) k_range_scatter(const FilterJob* jobs, int ntile, const int32_t* tile_cnt) {
  const FilterJob j = jobs[blockIdx.y];
  const int n = j.n_dev ? min(j.n, *j.n_dev) : j.n;
  const int base = blockIdx.x * FILT_TILE;
  __shared__ int s_w[FILT_THREADS / 32];
  __shared__ int s_base;
  // rows kept by the tiles before this one
  {
    int part = 0;
    const int32_t* tc = tile_cnt + (size_t)blockIdx.y * ntile;
    for (int t = threadIdx.x; t < (int)blockIdx.x; t += FILT_THREADS) part += tc[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < FILT_THREADS / 32; w++) t += s_w[w];
      s_base = t;
    }
    __syncthreads();
  }
  int run = s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = 0; r < FILT_ROUNDS; r++) {
    const int i = base + r * FILT_THREADS + threadIdx.x;
    float x = 0.f, y = 0.f, z = 0.f;
    bool keep = false;
    if (i < n) {
      x = __ldg(j.src + i); y = __ldg(j.src + j.ld + i); z = __ldg(j.src + 2 * (size_t)j.ld + i);
      keep = range_keep(x, y, z, j.min_d);
    }
    const unsigned m = __ballot_sync(FULL, keep);
    __syncthreads();  // s_w of the previous round has been read
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < FILT_THREADS / 32; w++) {
      const int c = s_w[w];
      before += (w < warp) ? c : 0;
      total += c;
    }
    if (keep) {
      const int o = run + before + __popc(m & ((1u << lane) - 1u));
      j.dst[o] = x;
      j.dst[j.ld_dst + o] = y;
      j.dst[2 * (size_t)j.ld_dst + o] = z;
    }
    run += total;
  }
  if (blockIdx.x == (unsigned)ntile - 1 && threadIdx.x == 0) *j.kept = run;
}

// prev_pcl_matrix = pcl_matrix (odometry.cpp:89): the rows that exist (device-resident count), not the whole capacity
__global__ void __launch_bounds__(256) k_copy_cloud(const float* src, float* dst, int ld, const int32_t* n_dev) {
  const int n = min(*n_dev, ld);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    dst[i] = src[i];
    dst[ld + i] = src[ld + i];
    dst[2 * (size_t)ld + i] = src[2 * (size_t)ld + i];
  }
}

// Pair descriptors of a sequence of filtered clouds held back to back: slot k at slots + k*3*cap, kept[k] rows.
__global__ void k_seq_desc(PairDesc* desc, int npairs, const float* slots, int cap, const int32_t* kept) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= npairs) return;
  PairDesc d;
  d.s1 = slots + (size_t)k * 3 * cap;
  d.s2 = slots + (size_t)(k + 1) * 3 * cap;
  d.n1 = kept[k]; d.ld1 = cap;
  d.n2 = kept[k + 1]; d.ld2 = cap;
  desc[k] = d;
}

// ----------------------------------------------------------------------------------------------
// Pose bookkeeping of the two nodes, one thread walking the pairs in order (it is a chain of 4x4 products).
// ----------------------------------------------------------------------------------------------
struct NodeState {       // device resident members of OdometryNode / MapMakerNode
  float X_homo[16];      // Matrix4f X_homo, row-major              (odometry.cpp:184, simpleMapMaker.cpp:260)
  float X0[6];           // VectorXf X0                              (odometry.cpp:170, simpleMapMaker.cpp:238)
  int32_t prev_n;        // rows of prev_pcl_matrix
  int32_t frames;        // registrations done so far
};

// Eigen::Quaternionf(Matrix3f) as called at odometry.cpp:115-116 / simpleMapMaker.cpp:182-183 (Eigen 3.3
// Geometry/Quaternion.h, quaternionbase_assign_impl<Other,3,3>: the trace / largest-diagonal-entry method).
// m row-major 3x3; q = (x, y, z, w).
__device__ inline void quat_from_rot(const float* m, float* q) {
  float t = m[0] + m[4] + m[8];
  if (t > 0.f) {
    t = sqrtf(t + 1.0f);
    q[3] = 0.5f * t;
    t = 0.5f / t;
    q[0] = (m[7] - m[5]) * t;  // (m(2,1) - m(1,2)) * t
    q[1] = (m[2] - m[6]) * t;  // (m(0,2) - m(2,0)) * t
    q[2] = (m[3] - m[1]) * t;  // (m(1,0) - m(0,1)) * t
  } else {
    int i = 0;
    if (m[4] > m[0]) i = 1;
    if (m[8] > m[4 * i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrtf(m[4 * i] - m[4 * j] - m[4 * k] + 1.0f);
    q[i] = 0.5f * t;
    t = 0.5f / t;
    q[3] = (m[3 * k + j] - m[3 * j + k]) * t;
    q[j] = (m[3 * j + i] + m[3 * i + j]) * t;
    q[k] = (m[3 * k + i] + m[3 * i + k]) * t;
  }
}

__global__ void k_node_poses(NodeState* st, const icet_b200_result* res, int npairs, const int32_t* kept /* per slot */,
                             icet_b200_odometry_params op, icet_b200_pose* out) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  float H[16];
  for (int k = 0; k < 16; k++) H[k] = st->X_homo[k];
  float Xl[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int p = 0; p < npairs; p++) {
    float X[6];
    for (int k = 0; k < 6; k++) X[k] = res[p].X[k];
    for (int k = 0; k < 6; k++) Xl[k] = X[k];  // the chain seed is the solution itself (odometry.cpp:82)
    // divergence guard, simpleMapMaker.cpp:128-137
    int guarded = 0;
    if (op.guard_trans > 0.f || op.guard_rot > 0.f) {
      const float tt = op.guard_trans > 0.f ? op.guard_trans : INFINITY;
      const float rt = op.guard_rot > 0.f ? op.guard_rot : INFINITY;
      if (fabsf(X[0]) > tt || fabsf(X[1]) > tt || fabsf(X[2]) > tt || fabsf(X[3]) > rt || fabsf(X[4]) > rt ||
          fabsf(X[5]) > rt) {
        guarded = 1;
        for (int k = 0; k < 6; k++) X[k] = 0.f;
      }
    }
    // X_homo_i = [R(X3,X4,X5) t; 0 1]; X_homo = X_homo * X_homo_i   (odometry.cpp:87-98)
    float R[9];
    icet::rotR(X[3], X[4], X[5], R);
    float Hi[16] = {R[0], R[1], R[2], X[0], R[3], R[4], R[5], X[1], R[6], R[7], R[8], X[2], 0.f, 0.f, 0.f, 1.f};
    float Hn[16];
    for (int a = 0; a < 4; a++)
      for (int b = 0; b < 4; b++) {
        float s = H[4 * a] * Hi[b];
        for (int c = 1; c < 4; c++) s += H[4 * a + c] * Hi[4 * c + b];
        Hn[4 * a + b] = s;
      }
    for (int k = 0; k < 16; k++) H[k] = Hn[k];
    icet_b200_pose* o = out + p;
    for (int k = 0; k < 16; k++) o->X_homo[k] = H[k];
    o->position[0] = H[3]; o->position[1] = H[7]; o->position[2] = H[11];  // odometry.cpp:110-112
    const float Rm[9] = {H[0], H[1], H[2], H[4], H[5], H[6], H[8], H[9], H[10]};
    quat_from_rot(Rm, o->orientation);                                       // :114-119
    for (int k = 0; k < 6; k++) {
      o->covariance_diag[k] = res[p].pred_stds[k];                           // :126-131 (stds, as the reference)
      o->twist[k] = op.rate_hz * X[k];                                       // :134-139
      o->X[k] = X[k];
    }
    o->n_points = kept ? kept[p + 1] : 0;
    o->guarded = guarded;
    o->frame = st->frames + p + 1;
    o->reserved = 0;
  }
  for (int k = 0; k < 16; k++) st->X_homo[k] = H[k];
  if (npairs > 0) {
    for (int k = 0; k < 6; k++) st->X0[k] = op.chain_x0 ? Xl[k] : 0.f;       // odometry.cpp:82 / simpleMapMaker.cpp:124
    st->frames += npairs;
  }
}

__global__ void k_node_init(NodeState* st, const float* X_homo0, const float* x0) {
  if (threadIdx.x < 16) st->X_homo[threadIdx.x] = X_homo0 ? X_homo0[threadIdx.x] : ((threadIdx.x % 5 == 0) ? 1.f : 0.f);
  if (threadIdx.x < 6) st->X0[threadIdx.x] = x0 ? x0[threadIdx.x] : 0.f;
  if (threadIdx.x == 0) { st->prev_n = 0; st->frames = 0; }
}

// ----------------------------------------------------------------------------------------------
// EigenQueue (simpleMapMaker.cpp:18-58): FIFO ring of map points, re-expressed in the newest sensor frame on
// every insertion.
// ----------------------------------------------------------------------------------------------
struct MapState {
  int32_t pos;     // next slot to write
  int32_t filled;  // the ring has wrapped at least once
  float t[3];      // translation and inverse rotation of the pending re-expression
  float Rinv[9];
  int32_t added;   // rows the last insertion appended
  int32_t guarded;
};

// Matrix3f::inverse() (Eigen 3.3 LU/InverseImpl.h, compute_inverse<Matrix3f>: cofactors / determinant)
__device__ inline void inv3_cofactor(const float* m, float* r) {
  const float c00 = m[4] * m[8] - m[5] * m[7];
  const float c10 = m[5] * m[6] - m[3] * m[8];
  const float c20 = m[3] * m[7] - m[4] * m[6];
  const float det = c00 * m[0] + c10 * m[1] + c20 * m[2];
  const float id = 1.0f / det;
  r[0] = c00 * id; r[3] = c10 * id; r[6] = c20 * id;
  r[1] = (m[2] * m[7] - m[1] * m[8]) * id;
  r[4] = (m[0] * m[8] - m[2] * m[6]) * id;
  r[7] = (m[1] * m[6] - m[0] * m[7]) * id;
  r[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  r[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  r[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// Appends `count` rows (gathered through idx when given, else rows 0..count-1 of the source) at the write cursor
// -- EigenQueue::enqueue per row, :24-32 -- and prepares the re-expression (trans, rot_mat.inverse()) from the
// registration result (after the divergence guard, simpleMapMaker.cpp:128-143).  One block.
__global__ void __launch_bounds__(256) k_map_enqueue(MapState* ms, float* ring, int cap, int ldr, const float* src, int ld,
                                                     const int32_t* n_dev, int n, const int32_t* idx, int count,
                                                     const float* X /* 6, device */, float guard_trans, float guard_rot) {
  const int nsrc = n_dev ? min(n, *n_dev) : n;
  // rows available: min(downsampleSize, rows) -- the reference sizes the matrix that way (:155) but then indexes
  // past it when the scan is shorter than the sample (:156-158); here the sample is simply clipped
  const int m = idx ? count : min(count, nsrc);
  const int pos0 = ms->pos;
  __syncthreads();
  for (int k = threadIdx.x; k < m; k += blockDim.x) {
    int s = idx ? idx[k] : k;
    if (s < 0 || s >= nsrc) continue;  // cannot happen for a valid sample of an nsrc-row cloud; never write garbage
    const int o = (int)(((long long)pos0 + k) % cap);
    ring[o] = src[s];
    ring[ldr + o] = src[ld + s];
    ring[2 * (size_t)ldr + o] = src[2 * (size_t)ld + s];
  }
  if (threadIdx.x == 0) {
    const long long np = (long long)pos0 + m;
    if (np >= cap) ms->filled = 1;
    ms->pos = (int)(np % cap);
    ms->added = m;
    float Xg[6];
    for (int k = 0; k < 6; k++) Xg[k] = X[k];
    int guarded = 0;
    const float tt = guard_trans > 0.f ? guard_trans : INFINITY, rt = guard_rot > 0.f ? guard_rot : INFINITY;
    if (fabsf(Xg[0]) > tt || fabsf(Xg[1]) > tt || fabsf(Xg[2]) > tt || fabsf(Xg[3]) > rt || fabsf(Xg[4]) > rt ||
        fabsf(Xg[5]) > rt) {
      guarded = 1;
      for (int k = 0; k < 6; k++) Xg[k] = 0.f;
    }
    ms->guarded = guarded;
    float R[9];
    icet::rotR(Xg[3], Xg[4], Xg[5], R);
    inv3_cofactor(R, ms->Rinv);
    ms->t[0] = Xg[0]; ms->t[1] = Xg[1]; ms->t[2] = Xg[2];
  }
}

// matrix = (matrix.rowwise() - trans) * rot_mat.inverse()   (EigenQueue::add_new_scan, simpleMapMaker.cpp:41) over
// every stored row.  HBM-bound streaming kernel: 12 B read + 12 B written per map point, float4 accesses
// (the planes of the ring are ldr apart, a multiple of 4 floats).
__global__ void __launch_bounds__(256) k_map_reexpress(const MapState* ms, float* ring, int cap, int ldr) {
  const int rows = ms->filled ? cap : ms->pos;
  const float tx = ms->t[0], ty = ms->t[1], tz = ms->t[2];
  float R[9];
#pragma unroll
  for (int k = 0; k < 9; k++) R[k] = ms->Rinv[k];
  const int nv = (rows + 3) >> 2;
  float4* px = reinterpret_cast<float4*>(ring);
  float4* py = reinterpret_cast<float4*>(ring + ldr);
  float4* pz = reinterpret_cast<float4*>(ring + 2 * (size_t)ldr);
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += gridDim.x * blockDim.x) {
    float4 x = px[v], y = py[v], z = pz[v];
    float* xs = &x.x; float* ys = &y.x; float* zs = &z.x;
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const float ax = __fsub_rn(xs[e], tx), ay = __fsub_rn(ys[e], ty), az = __fsub_rn(zs[e], tz);
      xs[e] = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[0]), __fmul_rn(ay, R[3])), __fmul_rn(az, R[6]));
      ys[e] = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[1]), __fmul_rn(ay, R[4])), __fmul_rn(az, R[7]));
      zs[e] = __fadd_rn(__fadd_rn(__fmul_rn(ax, R[2]), __fmul_rn(ay, R[5])), __fmul_rn(az, R[8]));
    }
    px[v] = x; py[v] = y; pz[v] = z;  // rows beyond `rows` in the last vector are unused slots (overwritten on enqueue)
  }
}

// EigenQueue::getQueue (:44-51): oldest row first.  out: planes with leading dimension ld_out; n_out[0] = rows.
__global__ void __launch_bounds__(256) k_map_get(const MapState* ms, const float* ring, int cap, int ldr, float* out,
                                                 int ld_out, int32_t* n_out) {
  const int rows = ms->filled ? cap : ms->pos;
  const int first = ms->filled ? ms->pos : 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += gridDim.x * blockDim.x) {
    int s = first + i;
    if (s >= cap) s -= cap;
    out[i] = ring[s];
    out[ld_out + i] = ring[ldr + s];
    out[2 * (size_t)ld_out + i] = ring[2 * (size_t)ldr + s];
  }
  if (n_out && blockIdx.x == 0 && threadIdx.x == 0) *n_out = rows;
}

// ----------------------------------------------------------------------------------------------
// Ingest (SURVEY.md 8f N3): caller's records -> x | y | z float planes.  Replaces the host loops of
// convertPCLtoEigen (odometry.cpp:186-192) and of loadPointCloudCSV's `rows[i] / 1000` (src/utils.cpp:42-52).
// ----------------------------------------------------------------------------------------------
struct IngestDesc {
  const unsigned char* raw;  // device copy of the caller's bytes
  int n, step, off[3], dtype, plane_stride;
  float divide;
};

__device__ __forceinline__ float ingest_elem(const unsigned char* p, int dtype, float divide) {
  float v;
  if (dtype == ICET_B200_F32) v = *reinterpret_cast<const float*>(p);
  else if (dtype == ICET_B200_F64) v = (float)*reinterpret_cast<const double*>(p);  // round to nearest, like cast<float>()
  else v = (float)*reinterpret_cast<const int32_t*>(p);                             // static_cast<float>(int)
  if (divide != 0.f && divide != 1.f) v = __fdiv_rn(v, divide);
  return v;
}

__global__ void __launch_bounds__(256) k_ingest(const IngestDesc d, float* out, int ld) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d.n) return;
  const int es = d.dtype == ICET_B200_F64 ? 8 : 4;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const unsigned char* p = d.plane_stride > 0 ? d.raw + ((size_t)k * d.plane_stride + i) * es
                                                : d.raw + (size_t)i * d.step + d.off[k];
    out[(size_t)k * ld + i] = ingest_elem(p, d.dtype, d.divide);
  }
}

// ----------------------------------------------------------------------------------------------
// Whole-cloud re-expressions of the nodes (scanMatcher.cpp:73,76; simpleMapMaker.cpp:41,222), X read on the device.
// ----------------------------------------------------------------------------------------------
// One row of a re-expression: m = rot_mat.inverse() (row-major), t = trans; mode 0 `row * m - t`, mode 1 `(row - t) * m`,
// every product and sum rounded separately (no contraction), as Eigen's float expressions are evaluated.
__device__ __forceinline__ void xform_row(float& x, float& y, float& z, const float* m, float tx, float ty, float tz,
                                          int mode) {
  if (mode == 1) { x = __fsub_rn(x, tx); y = __fsub_rn(y, ty); z = __fsub_rn(z, tz); }
  float ox = __fadd_rn(__fadd_rn(__fmul_rn(x, m[0]), __fmul_rn(y, m[3])), __fmul_rn(z, m[6]));
  float oy = __fadd_rn(__fadd_rn(__fmul_rn(x, m[1]), __fmul_rn(y, m[4])), __fmul_rn(z, m[7]));
  float oz = __fadd_rn(__fadd_rn(__fmul_rn(x, m[2]), __fmul_rn(y, m[5])), __fmul_rn(z, m[8]));
  if (mode == 0) { ox = __fsub_rn(ox, tx); oy = __fsub_rn(oy, ty); oz = __fsub_rn(oz, tz); }
  x = ox; y = oy; z = oz;
}

__global__ void __launch_bounds__(256) k_transform_cloud(const float* src, int n, int ld, const int32_t* n_dev,
                                                         const float* X, int mode, float* dst, int ld_out) {
  __shared__ float s_m[12];
  if (threadIdx.x == 0) {
    float R[9];
    icet::rotR(X[3], X[4], X[5], R);
    inv3_cofactor(R, s_m);
    s_m[9] = X[0]; s_m[10] = X[1]; s_m[11] = X[2];
  }
  __syncthreads();
  const int rows = n_dev ? min(n, *n_dev) : n;
  const float tx = s_m[9], ty = s_m[10], tz = s_m[11];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += gridDim.x * blockDim.x) {
    float ox = src[i], oy = src[ld + i], oz = src[2 * (size_t)ld + i];
    xform_row(ox, oy, oz, s_m, tx, ty, tz, mode);
    dst[i] = ox;
    dst[ld_out + i] = oy;
    dst[2 * (size_t)ld_out + i] = oz;
  }
}

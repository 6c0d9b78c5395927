// icet_b200/csrc/kernels_kfnode.cuh -- device side of the keyframe odometry node (include/icet_b200.h "keyframe
// odometry", DESIGN.md §13), included by icet_b200.cu inside its anonymous namespace after callers.cuh.
//
// Per scan k (all on the context's stream, nothing returns to the host):
//   registration of slot k against the node's keyframe (k_kf_attach<const int32_t*> + the loop), seed from the state
//   k_kfnode_step    policy, pose, frame step, next seed, info; writes the descriptor of the candidate fit
//   candidate fit    chunk_setup + chunk_scan1 on that descriptor (n1 = 0 unless scan k was promoted)
//   k_kf_commit      promoted: the candidate's CellRec / Vox1 and n_gauss1 become the node's keyframe
//   k_copy_cloud     promoted: the filtered cloud becomes the node's keyframe cloud (0 rows otherwise)
// A local-map node (icet_b200_kfnode_create_local_map, DESIGN.md §14) fits the merged clouds of its last M keyframes
// instead of the promoted scan alone: k_lmap_window and k_lmap_assemble run between k_kfnode_step and the candidate
// fit, which then reads the map (n1max = M * cap).
#pragma once

struct KfNodeState {        // device-resident members of the keyframe odometry node
  float H_f[16];            // pose of the current keyframe, row-major (X_homo of that scan)
  float x0[6];              // seed of the next registration
  float X_prev[6];          // X_rel of the previous registration (frame step when both share a keyframe)
  int32_t kf_frame;         // frame index of the current keyframe (0 = the first scan)
  int32_t interval;         // registrations against the current keyframe so far
  int32_t frames;           // registrations done so far
  int32_t n_gauss1;         // Gaussians of the current keyframe (read by k_kf_attach<const int32_t*>)
  int32_t kf_n;             // rows of the keyframe cloud
  int32_t commit;           // 1: the candidate fit of the scan just stepped becomes the keyframe
};

// params(H): the translation column verbatim, the angles of icet::rotR inverted (R[6] = sin theta,
// R[7] = -sin phi cos theta, R[8] = cos phi cos theta, R[3] = -sin psi cos theta, R[0] = cos theta cos psi), |theta| < pi/2.
__device__ inline void kf_params(const double* H, float* X) {
  X[0] = (float)H[3]; X[1] = (float)H[7]; X[2] = (float)H[11];
  X[3] = (float)atan2(-H[9], H[10]);
  X[4] = (float)asin(fmin(1.0, fmax(-1.0, H[8])));
  X[5] = (float)atan2(-H[4], H[0]);
}

// Hi(X) = [R(X3,X4,X5) t; 0 1] with the float arithmetic of k_node_poses, widened to double
__device__ inline void kf_homo(const float* X, double* H) {
  float R[9];
  icet::rotR(X[3], X[4], X[5], R);
  const float Hf[16] = {R[0], R[1], R[2], X[0], R[3], R[4], R[5], X[1], R[6], R[7], R[8], X[2], 0.f, 0.f, 0.f, 1.f};
  for (int k = 0; k < 16; k++) H[k] = Hf[k];
}

__device__ inline void kf_mul(const double* A, const double* B, double* C) {
  for (int a = 0; a < 4; a++)
    for (int b = 0; b < 4; b++) {
      double s = A[4 * a] * B[b];
      for (int c = 1; c < 4; c++) s += A[4 * a + c] * B[4 * c + b];
      C[4 * a + b] = s;
    }
}

// inverse of a rigid [R t; 0 1]: [R^T  -R^T t; 0 1]
__device__ inline void kf_rigid_inv(const double* A, double* B) {
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) B[4 * i + j] = A[4 * j + i];
    B[4 * i + 3] = -(A[i] * A[3] + A[4 + i] * A[7] + A[8 + i] * A[11]);
  }
  B[12] = 0.0; B[13] = 0.0; B[14] = 0.0; B[15] = 1.0;
}

// One scan after its registration (res != null) or the first scan of the node (res == null: it becomes keyframe 0).
// One warp; lane 0 does the work.
__global__ void __launch_bounds__(32) k_kfnode_step(KfNodeState* st, const icet_b200_result* res, const int32_t* kept,
                                                    const float* slot, int cap, icet_b200_odometry_params op,
                                                    icet_b200_keyframe_policy pol, icet_b200_pose* pose,
                                                    icet_b200_kf_info* info, PairDesc* fit) {
  if (threadIdx.x != 0) return;
  PairDesc d;
  d.s1 = slot; d.ld1 = cap; d.s2 = nullptr; d.n2 = 0; d.ld2 = 0;
  if (!res) {
    st->commit = 1;
    d.n1 = *kept;
    *fit = d;
    return;
  }
  const int frame = st->frames + 1;
  float X[6];
  for (int k = 0; k < 6; k++) X[k] = res->X[k];
  // frame step: X verbatim when the keyframe is the predecessor, else Hi(X_rel,k-1)^-1 Hi(X_rel,k)
  float step[6];
  if (st->kf_frame == frame - 1) {
    for (int k = 0; k < 6; k++) step[k] = X[k];
  } else {
    double Hp[16], Hpi[16], Hk[16], Hs[16];
    kf_homo(st->X_prev, Hp);
    kf_rigid_inv(Hp, Hpi);
    kf_homo(X, Hk);
    kf_mul(Hpi, Hk, Hs);
    kf_params(Hs, step);
  }
  // promotion policy
  int reason = 0;
  const float tn = sqrtf(X[0] * X[0] + X[1] * X[1] + X[2] * X[2]);
  const float rm = fmaxf(fabsf(X[3]), fmaxf(fabsf(X[4]), fabsf(X[5])));
  if (pol.max_trans > 0.f && tn > pol.max_trans) reason |= ICET_B200_KF_TRANS;
  if (pol.max_rot > 0.f && rm > pol.max_rot) reason |= ICET_B200_KF_ROT;
  if (pol.min_overlap > 0.f && (float)res->n_used < pol.min_overlap * (float)res->n_gauss1) reason |= ICET_B200_KF_OVERLAP;
  if (pol.max_interval > 0 && st->interval + 1 >= pol.max_interval) reason |= ICET_B200_KF_INTERVAL;
  if (res->status != ICET_B200_OK) reason |= ICET_B200_KF_STATUS;
  const int promoted = reason != 0;
  // X_homo_k = X_homo_f * Hi(X_rel): the float product of k_node_poses
  float R[9];
  icet::rotR(X[3], X[4], X[5], R);
  const float Hi[16] = {R[0], R[1], R[2], X[0], R[3], R[4], R[5], X[1], R[6], R[7], R[8], X[2], 0.f, 0.f, 0.f, 1.f};
  float H[16];
  for (int a = 0; a < 4; a++)
    for (int b = 0; b < 4; b++) {
      float s = st->H_f[4 * a] * Hi[b];
      for (int c = 1; c < 4; c++) s += st->H_f[4 * a + c] * Hi[4 * c + b];
      H[4 * a + b] = s;
    }
  for (int k = 0; k < 16; k++) pose->X_homo[k] = H[k];
  pose->position[0] = H[3]; pose->position[1] = H[7]; pose->position[2] = H[11];
  const float Rm[9] = {H[0], H[1], H[2], H[4], H[5], H[6], H[8], H[9], H[10]};
  quat_from_rot(Rm, pose->orientation);
  for (int k = 0; k < 6; k++) {
    pose->covariance_diag[k] = res->pred_stds[k];
    pose->twist[k] = op.rate_hz * step[k];
    pose->X[k] = X[k];
  }
  pose->n_points = *kept;
  pose->guarded = 0;
  pose->frame = frame;
  pose->reserved = 0;
  info->keyframe = st->kf_frame;
  info->promoted = promoted;
  info->reason = reason;
  for (int k = 0; k < 6; k++) info->x0[k] = st->x0[k];
  info->reserved = 0;
  // seed of the next registration: constant velocity, relative to the keyframe it will be registered against
  float xn[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (op.chain_x0) {
    if (promoted) {
      for (int k = 0; k < 6; k++) xn[k] = step[k];
    } else {
      double Hk[16], Hs[16], Hn[16];
      kf_homo(X, Hk);
      kf_homo(step, Hs);
      kf_mul(Hk, Hs, Hn);
      kf_params(Hn, xn);
    }
  }
  for (int k = 0; k < 6; k++) { st->x0[k] = xn[k]; st->X_prev[k] = X[k]; }
  if (promoted) {
    for (int k = 0; k < 16; k++) st->H_f[k] = H[k];
    st->kf_frame = frame;
    st->interval = 0;
  } else {
    st->interval += 1;
  }
  st->frames = frame;
  st->commit = promoted;
  d.n1 = promoted ? *kept : 0;
  *fit = d;
}

// The candidate fit becomes the keyframe (when the step kernel promoted its scan): flat 16-byte copies of its CellRec
// and Vox1 records (one 8-byte tail word when ncell * sizeof(Vox1) is not a multiple of 16) and its Gaussian count.
static_assert(sizeof(CellRec) % 16 == 0 && sizeof(Vox1) % 8 == 0, "k_kf_commit copies 16-byte words (+ one 8-byte tail)");
// kf_rows: rows of the promoted keyframe's own cloud (the fit's n1 for a plain node; a local-map node fits more rows).
__global__ void __launch_bounds__(256) k_kf_commit(KfNodeState* st, const CellRec* __restrict__ crec,
                                                   const Vox1* __restrict__ cvox, const icet_b200_result* cres,
                                                   const int32_t* kf_rows, CellRec* krec, Vox1* kvox, int ncell) {
  if (!st->commit) return;
  const int nr = ncell * (int)(sizeof(CellRec) / 16);
  const size_t vb = (size_t)ncell * sizeof(Vox1);
  const int nv = (int)(vb / 16);
  const float4* rs = reinterpret_cast<const float4*>(crec);
  float4* rd = reinterpret_cast<float4*>(krec);
  const float4* vs = reinterpret_cast<const float4*>(cvox);
  float4* vd = reinterpret_cast<float4*>(kvox);
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < nr + nv; w += gridDim.x * blockDim.x) {
    if (w < nr) rd[w] = __ldg(rs + w);
    else vd[w - nr] = __ldg(vs + (w - nr));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (vb % 16) reinterpret_cast<uint2*>(kvox)[vb / 8 - 1] = reinterpret_cast<const uint2*>(cvox)[vb / 8 - 1];
    st->n_gauss1 = cres->n_gauss1;
    st->kf_n = *kf_rows;
  }
}

// -- local map (DESIGN.md §14) ---------------------------------------------------------------------------------------
// A ring of M keyframe slots: the original filtered cloud of each keyframe ([M][3][cap], owned by the host struct),
// its row count and its transform into the frame of the newest keyframe.  The map lists the slots newest first.
constexpr int LMAP_MAX = 16;
constexpr long long LMAP_MAX_ROWS = 1LL << 28;  // map capacity M * cap: int32 row offsets and tile grids stay far from 2^31

struct LmapState {
  double T[LMAP_MAX][16];     // ring slot -> current keyframe frame, on column vectors: p_cur = T p_slot (row-major)
  float m[LMAP_MAX][12];      // map block b: T of its slot as k_transform_cloud mode 0 takes it, `row * m[0..8] - m[9..11]`
  int32_t n[LMAP_MAX];        // rows of each ring slot
  int32_t src[LMAP_MAX];      // map block b -> ring slot
  int32_t off[LMAP_MAX + 1];  // map block b -> its first map row; off[count] = map_n
  int32_t head;               // ring slot of the newest keyframe
  int32_t count;              // keyframes in the window (<= M)
  int32_t nblk;               // blocks k_lmap_assemble writes for the scan just stepped (0: it was not promoted)
  int32_t newest_n;           // rows of the keyframe promoted by that scan (0: none)
  int32_t map_n;              // rows of the map
};

// After k_kfnode_step: when it promoted scan k, re-express the window in k's frame and give k the next ring slot.
// The registration of k against keyframe f maps a point p of k into f as (p + t) R(X) (row vectors), so a point q of
// f is q R^-1 - t in k's frame (k_transform_cloud mode 0): F = [R t'; 0 1] with t' = -t on column vectors (R^-T = R
// for a rotation), and every slot's T becomes F T, composed in double.  Lane j composes the j-th newest slot.
__global__ void __launch_bounds__(32) k_lmap_window(const KfNodeState* st, LmapState* lm, const icet_b200_result* res,
                                                    const int32_t* kept, int M) {
  const int lane = threadIdx.x;
  if (!st->commit) {
    if (lane == 0) { lm->nblk = 0; lm->newest_n = 0; }
    return;
  }
  const int head = lm->head, count = lm->count;
  if (res && lane < count) {
    double F[16], T[16];
    kf_homo(res->X, F);
    F[3] = -F[3]; F[7] = -F[7]; F[11] = -F[11];
    double* Ts = lm->T[(head - lane + M) % M];
    kf_mul(F, Ts, T);
    for (int k = 0; k < 16; k++) Ts[k] = T[k];
  }
  __syncwarp();
  if (lane != 0) return;
  const int h = (head + 1) % M, cnt = min(count + 1, M);  // a full ring retires its oldest slot, h
  for (int k = 0; k < 16; k++) lm->T[h][k] = (k % 5 == 0) ? 1.0 : 0.0;
  lm->n[h] = *kept;
  int off = 0;
  for (int b = 0; b < cnt; b++) {
    const int s = (h - b + M) % M;
    const double* T = lm->T[s];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) lm->m[b][3 * r + c] = (float)T[4 * c + r];
    lm->m[b][9] = (float)-T[3]; lm->m[b][10] = (float)-T[7]; lm->m[b][11] = (float)-T[11];
    lm->src[b] = s;
    lm->off[b] = off;
    off += lm->n[s];
  }
  lm->off[cnt] = off;
  lm->head = h; lm->count = cnt; lm->nblk = cnt; lm->newest_n = *kept; lm->map_n = off;
}

// The map, one block row per window slot (blockIdx.y = b, newest first, no gaps): block 0 is the promoted scan's
// filtered cloud, copied verbatim into the map and into its ring slot; the others are their slot's stored cloud through
// the mode-0 arithmetic of k_transform_cloud.  Writes the candidate-fit descriptor (scan 1 = the map).  Nothing when
// the scan was not promoted: k_kfnode_step's descriptor (n1 = 0) stands.
__global__ void __launch_bounds__(256) k_lmap_assemble(const LmapState* lm, const float* slot, int cap, float* ring,
                                                       float* map, int ldm, PairDesc* fit) {
  const int b = blockIdx.y;
  if (b >= lm->nblk) return;
  const int s = lm->src[b], n = lm->n[s], o = lm->off[b];
  float m[12];
  for (int k = 0; k < 12; k++) m[k] = lm->m[b][k];
  const float* src = b == 0 ? slot : ring + (size_t)s * 3 * cap;
  float* keep = ring + (size_t)s * 3 * cap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float x = src[i], y = src[cap + i], z = src[2 * (size_t)cap + i];
    if (b == 0) {
      keep[i] = x; keep[cap + i] = y; keep[2 * (size_t)cap + i] = z;
    } else {
      xform_row(x, y, z, m, m[9], m[10], m[11], 0);
    }
    map[o + i] = x; map[ldm + o + i] = y; map[2 * (size_t)ldm + o + i] = z;
  }
  if (b == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    PairDesc d;
    d.s1 = map; d.n1 = lm->map_n; d.ld1 = ldm; d.s2 = nullptr; d.n2 = 0; d.ld2 = 0;
    *fit = d;
  }
}

__global__ void k_lmap_init(LmapState* lm, int M) {
  if (threadIdx.x == 0) {
    lm->head = M - 1; lm->count = 0; lm->nblk = 0; lm->newest_n = 0; lm->map_n = 0;
  }
}

__global__ void k_kfnode_init(KfNodeState* st, const float* X_homo0, const float* x0, int chain) {
  if (threadIdx.x < 16) st->H_f[threadIdx.x] = X_homo0 ? X_homo0[threadIdx.x] : ((threadIdx.x % 5 == 0) ? 1.f : 0.f);
  if (threadIdx.x < 6) {
    st->x0[threadIdx.x] = (chain && x0) ? x0[threadIdx.x] : 0.f;
    st->X_prev[threadIdx.x] = 0.f;
  }
  if (threadIdx.x == 0) {
    st->kf_frame = 0; st->interval = 0; st->frames = 0; st->n_gauss1 = 0; st->kf_n = 0; st->commit = 0;
  }
}

// Registration descriptors of a call: scan 1 is the node's keyframe, scan 2 the filtered slot k (kept[k] rows).
__global__ void k_kfnode_desc(PairDesc* desc, int nscans, const float* slots, int cap, const int32_t* kept) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nscans) return;
  PairDesc d;
  d.s1 = nullptr; d.n1 = 0; d.ld1 = 0;
  d.s2 = slots + (size_t)k * 3 * cap;
  d.n2 = kept[k]; d.ld2 = cap;
  desc[k] = d;
}

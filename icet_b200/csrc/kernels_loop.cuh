// icet_b200/csrc/kernels_loop.cuh -- the Gauss-Newton iteration: per-voxel algebra of fitCells2 (K5b), the 6x6 solve
// with checkCondition (K6), the persistent loop kernel k_loop and the split-loop kernels k_vox2 / k_solve6, plus the
// small utility kernels (points2, spherical bins test hook, synthetic scans).  Included by icet_b200.cu inside its
// anonymous namespace.
#pragma once
// ----------------------------------------------------------------------------------------------
// K5b: per voxel.  Scan-2 mean / covariance, R_noise, W, H_z and the voxel's contributions
// H^T W H_j (upper triangle, 21) and H^T W dz_j (6)  (fitCells2 src/icet.cpp:302-338), ADDED to acc[].
// Takes the voxel's integer accumulators (L2 reads: other SMs produced them) and clears them for the next
// iteration.
// ----------------------------------------------------------------------------------------------
constexpr int VOX_THREADS = 64;
// a0 b0 + a1 b1 + a2 b2 with fused multiply-adds.  The translation unit is compiled with -fmad=false for the point-wise
// fp32 geometry (which must round like the reference's scalar code); the per-voxel double algebra has no such
// constraint, and it is a serial chain on the critical path of every iteration: explicit fma halves its arithmetic
// instructions and shortens the dependency chains.
__device__ __forceinline__ double dot3(double a0, double b0, double a1, double b1, double a2, double b2) {
  return fma(a2, b2, fma(a1, b1, a0 * b0));
}
constexpr int NRED = 28;  // 21 (upper triangle of H^T W H) + 6 (H^T W dz) + 1 (voxels used)

// Sum over the 32 lanes of each of the NRED (28) per-lane values; lane k < NRED returns the total of value k.
// Transposing butterfly: at distance o the lanes with bit o set keep the upper half of the remaining values and the
// others the lower half, so 16 + 8 + 4 + 2 + 1 shuffles replace 28 x 5.  The pairing of the additions is that of the
// plain xor butterfly (lanes L and L ^ o at every level), so the sums are bit-identical to it.
__device__ __forceinline__ double warp_sum_transposed(const double (&acc)[NRED], int lane) {
  double v[16];
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const double hi = (i + 16 < NRED) ? acc[i + 16] : 0.0;
      const double send = up ? acc[i] : hi;
      const double keep = up ? hi : acc[i];
      v[i] = keep + __shfl_xor_sync(FULL, send, 16);
    }
  }
#pragma unroll
  for (int o = 8; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; i++) {
      const double send = up ? v[i] : v[i + o];
      const double keep = up ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(FULL, send, o);
    }
  }
  return v[0];
}

// Gate of fitCells2 for one voxel (`indices2.size() > n` :290, `rows > n` :302).  Returns true if the voxel
// contributes; its accumulators are then left in place for vox_algebra, otherwise they are cleared here.
__device__ __forceinline__ bool vox_gate(const Chunk& ck, int pair, int cell, int iter) {
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const uint32_t flags = ck.rec[ci].flags;
  if (!(flags & F_ACTIVE2)) {
    if (ck.dump_on) {
      ck.dump.cnt2[(size_t)iter * ck.ncell + cell] = -1;
      ck.dump.nin2[(size_t)iter * ck.ncell + cell] = -1;
      ck.dump.used2[(size_t)iter * ck.ncell + cell] = 0;
    }
    return false;
  }
  unsigned long long* qp = ck.acc + ci * NQ;
  const ulonglong2 q01 = __ldcg(reinterpret_cast<const ulonglong2*>(qp));
  const long long nbin = (long long)q01.x, nin = (long long)q01.y;
  const bool use = nbin > ck.n && nin > ck.n;
  if (ck.dump_on) {
    ck.dump.cnt2[(size_t)iter * ck.ncell + cell] = (int)nbin;
    ck.dump.nin2[(size_t)iter * ck.ncell + cell] = (nbin > ck.n) ? (int)nin : -1;
    ck.dump.used2[(size_t)iter * ck.ncell + cell] = use ? 1 : 0;
  }
  if (!use && nbin != 0) {
#pragma unroll
    for (int k = 0; k < NQ; k++) qp[k] = 0ull;
  }
  return use;
}

__device__ __forceinline__ void vox_algebra_core(const Chunk& ck, int pair, int cell, int iter, const float* Jm,
                                                 long long nbin, const double mean[3], const double cov[6], double acc[NRED],
                                                 const Vox1* vp = nullptr);

// The algebra of one contributing voxel; takes (and clears) its accumulators.
__device__ __forceinline__ void vox_algebra(const Chunk& ck, int pair, int cell, int iter, const float* Jm /* 27 */,
                                            double acc[NRED]) {
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const CellRec rc = ck.rec[ci];
  unsigned long long q[NQ];
  unsigned long long* qp = ck.acc + ci * NQ;
#pragma unroll
  for (int k = 0; k < NQ; k += 2) {
    const ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(qp + k));
    q[k] = t.x;
    q[k + 1] = t.y;
  }
#pragma unroll
  for (int k = 0; k < NQ; k++) qp[k] = 0ull;
  double mean[3], cov[6];
  stats_from_acc(q, rc, fix_point(__ldg(&ck.desc[pair].n2)).fs, mean, cov);
  vox_algebra_core(ck, pair, cell, iter, Jm, (long long)q[0], mean, cov, acc);
}

// from the scan-2 mean / covariance of a voxel to its contributions H^T W H_j, H^T W dz_j (src/icet.cpp:308-338)
__device__ __forceinline__ void vox_algebra_core(const Chunk& ck, int pair, int cell, int iter, const float* Jm,
                                                 long long nbin, const double mean[3], const double cov[6],
                                                 double acc[NRED], const Vox1* vp) {
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const Vox1 v = vp ? *vp : ck.vox[ci];  // (vp: the cluster loop keeps the records of its voxels in shared memory)
  if (ck.dump_on) {
    float* m2 = ck.dump.mu2 + ((size_t)iter * ck.ncell + cell) * 3;
    float* s2 = ck.dump.sigma2 + ((size_t)iter * ck.ncell + cell) * 9;
    for (int k = 0; k < 3; k++) m2[k] = (float)mean[k];
    s2[0] = (float)cov[0]; s2[1] = (float)cov[1]; s2[2] = (float)cov[2];
    s2[3] = (float)cov[1]; s2[4] = (float)cov[3]; s2[5] = (float)cov[4];
    s2[6] = (float)cov[2]; s2[7] = (float)cov[4]; s2[8] = (float)cov[5];
  }
  // R_noise = sigma1/(|idx1|-1) + sigma2/(|idx2|-1)   (:315)
  const double id2 = 1.0 / (double)(nbin - 1);
  double Rn[9];
  {
    double r6[6];
#pragma unroll
    for (int k = 0; k < 6; k++) r6[k] = v.S1n[k] + cov[k] * id2;
    Rn[0] = r6[0]; Rn[1] = r6[1]; Rn[2] = r6[2]; Rn[3] = r6[1]; Rn[4] = r6[3]; Rn[5] = r6[4];
    Rn[6] = r6[2]; Rn[7] = r6[4]; Rn[8] = r6[5];
  }
  // M = (L U^T) R_noise (L U^T)^T   (:317)
  double T[9], M[9];
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = 0; b < 3; b++)
      T[3 * a + b] = dot3(v.LV[3 * a], Rn[b], v.LV[3 * a + 1], Rn[3 + b], v.LV[3 * a + 2], Rn[6 + b]);
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = 0; b < 3; b++)
      M[3 * a + b] = dot3(T[3 * a], v.LV[3 * b], T[3 * a + 1], v.LV[3 * b + 1], T[3 * a + 2], v.LV[3 * b + 2]);
  // W = pinv(M)  (:320-321)
  double W[9];
  if (!icet::masked_inv3(M, v.lmask, W)) {  // (rare; the copies keep M / W of the common path out of local memory)
    double Mc[9], Wc[9];
#pragma unroll
    for (int k = 0; k < 9; k++) Mc[k] = M[k];
    icet::cod_pinv(Mc, 3, 3, Wc);
#pragma unroll
    for (int k = 0; k < 9; k++) W[k] = Wc[k];
  }
  // H_z = L U^T [ -I | Jx mu | Jy mu | Jz mu ]  (:324-329)
  double H[18];
#pragma unroll
  for (int a = 0; a < 3; a++) {
    H[6 * a + 0] = (a == 0) ? -1.0 : 0.0;
    H[6 * a + 1] = (a == 1) ? -1.0 : 0.0;
    H[6 * a + 2] = (a == 2) ? -1.0 : 0.0;
#pragma unroll
    for (int j = 0; j < 3; j++)
      H[6 * a + 3 + j] = dot3((double)Jm[9 * j + 3 * a], mean[0], (double)Jm[9 * j + 3 * a + 1], mean[1],
                              (double)Jm[9 * j + 3 * a + 2], mean[2]);
  }
  double Hz[18];
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int c = 0; c < 6; c++)
      Hz[6 * a + c] = dot3(v.LV[3 * a], H[c], v.LV[3 * a + 1], H[6 + c], v.LV[3 * a + 2], H[12 + c]);
  // dz = L U^T (mean2 - mu1)   (:335-337)
  const double dm[3] = {mean[0] - v.mu[0], mean[1] - v.mu[1], mean[2] - v.mu[2]};
  double dz[3];
#pragma unroll
  for (int a = 0; a < 3; a++) dz[a] = dot3(v.LV[3 * a], dm[0], v.LV[3 * a + 1], dm[1], v.LV[3 * a + 2], dm[2]);
  double WH[18], Wdz[3];
#pragma unroll
  for (int a = 0; a < 3; a++) {
#pragma unroll
    for (int c = 0; c < 6; c++)
      WH[6 * a + c] = dot3(W[3 * a], Hz[c], W[3 * a + 1], Hz[6 + c], W[3 * a + 2], Hz[12 + c]);
    Wdz[a] = dot3(W[3 * a], dz[0], W[3 * a + 1], dz[1], W[3 * a + 2], dz[2]);
  }
  int t = 0;
#pragma unroll
  for (int a = 0; a < 6; a++)
#pragma unroll
    for (int b = a; b < 6; b++) acc[t++] += dot3(Hz[a], WH[b], Hz[6 + a], WH[6 + b], Hz[12 + a], WH[12 + b]);
#pragma unroll
  for (int a = 0; a < 6; a++) acc[21 + a] += dot3(Hz[a], Wdz[0], Hz[6 + a], Wdz[1], Hz[12 + a], Wdz[2]);
  acc[27] += 1.0;
}

// ---- incremental loop (kernels_pass2.cuh): the accumulators hold exact moments of the UNTRANSFORMED members of the
// voxel, in the set the pair currently uses; nothing is cleared except, right after a rebuild, the other set.
struct VoxMode {
  int set, rebuild;
  float fs2;
  float trb[12], tr[12];
};
__device__ __forceinline__ void load_vox_mode(const Chunk& ck, int pair, VoxMode& vm) {
  const PairMode* pm = ck.pm + pair;
  const int2 h = __ldcg(reinterpret_cast<const int2*>(pm));
  vm.set = h.x;
  vm.rebuild = h.y;
  vm.fs2 = fix_point(__ldg(&ck.desc[pair].n2)).fs;
  const float4* tb = reinterpret_cast<const float4*>(pm->TRb);
  const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float4 a = __ldcg(tb + k), b = __ldcg(tp + k);
    vm.trb[4 * k] = a.x; vm.trb[4 * k + 1] = a.y; vm.trb[4 * k + 2] = a.z; vm.trb[4 * k + 3] = a.w;
    vm.tr[4 * k] = b.x; vm.tr[4 * k + 1] = b.y; vm.tr[4 * k + 2] = b.z; vm.tr[4 * k + 3] = b.w;
  }
}

__device__ __forceinline__ bool vox_gate2(const Chunk& ck, int pair, int cell, int iter, const VoxMode& vm) {
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const uint32_t flags = ck.rec[ci].flags;
  if (!(flags & F_ACTIVE2)) {
    if (ck.dump_on) {
      ck.dump.cnt2[(size_t)iter * ck.ncell + cell] = -1;
      ck.dump.nin2[(size_t)iter * ck.ncell + cell] = -1;
      ck.dump.used2[(size_t)iter * ck.ncell + cell] = 0;
    }
    return false;
  }
  if (vm.rebuild) {  // the set the pair has just left becomes the clean target of the next rebuild
    unsigned long long* sp = ck.acc + ((size_t)(vm.set ^ 1) * ck.npairs * ck.ncell + ci) * NQ;
#pragma unroll
    for (int k = 0; k < NQ; k += 2) *reinterpret_cast<ulonglong2*>(sp + k) = make_ulonglong2(0ull, 0ull);
  }
  const unsigned long long* qp = ck.acc + ((size_t)vm.set * ck.npairs * ck.ncell + ci) * NQ;
  const ulonglong2 q01 = __ldcg(reinterpret_cast<const ulonglong2*>(qp));
  const long long nbin = (long long)q01.x, nin = (long long)q01.y;
  const bool use = nbin > ck.n && nin > ck.n;
  if (ck.dump_on) {
    ck.dump.cnt2[(size_t)iter * ck.ncell + cell] = (int)nbin;
    ck.dump.nin2[(size_t)iter * ck.ncell + cell] = (nbin > ck.n) ? (int)nin : -1;
    ck.dump.used2[(size_t)iter * ck.ncell + cell] = use ? 1 : 0;
  }
  return use;
}

// mean / covariance of the voxel's scan-2 members at the current transform, from the moments of the untransformed
// points:  mu2 = (mean_OG + t) R,  Sigma2 = R^T Cov_OG R   (what src/icet.cpp:375-378 + :303-306 compute point by point)
__device__ __forceinline__ void stats2_from_moments_rec(const unsigned long long* q, float4 ra, float4 rb, const VoxMode& vm,
                                                        double mean[3], double cov[6]);
__device__ __forceinline__ void stats2_from_moments(const unsigned long long* q, const CellRec* recs, int cell,
                                                    const VoxMode& vm, double mean[3], double cov[6]) {
  const float4* rp = reinterpret_cast<const float4*>(recs + cell);
  stats2_from_moments_rec(q, __ldg(rp), __ldg(rp + 1), vm, mean, cov);
}
__device__ __forceinline__ void stats2_from_moments_rec(const unsigned long long* q, float4 ra, float4 rb, const VoxMode& vm,
                                                        double mean[3], double cov[6]) {
  float ax, ay, az, sc;
  vox_anchor2_rec(ra, rb, vm.trb, vm.fs2, ax, ay, az, sc);
  const double nin = (double)(long long)q[1];
  const double inv = 1.0 / (double)sc;  // exact: the scale is a power of two
  const double in_ = 1.0 / nin;
  const double sx = (double)(long long)q[2], sy = (double)(long long)q[3], sz = (double)(long long)q[4];
  const double mx = sx * in_, my = sy * in_, mz = sz * in_;
  const double po[3] = {((double)ax + mx * inv) + (double)vm.tr[0], ((double)ay + my * inv) + (double)vm.tr[1],
                        ((double)az + mz * inv) + (double)vm.tr[2]};
  const double f = inv * inv / (nin - 1.0);
  double co[9];
  co[0] = ((double)(long long)q[5] - sx * mx) * f;
  co[1] = co[3] = ((double)(long long)q[6] - sx * my) * f;
  co[2] = co[6] = ((double)(long long)q[7] - sx * mz) * f;
  co[4] = ((double)(long long)q[8] - sy * my) * f;
  co[5] = co[7] = ((double)(long long)q[9] - sy * mz) * f;
  co[8] = ((double)(long long)q[10] - sz * mz) * f;
  double R[9];
#pragma unroll
  for (int k = 0; k < 9; k++) R[k] = (double)vm.tr[3 + k];
#pragma unroll
  for (int i = 0; i < 3; i++) mean[i] = dot3(po[0], R[i], po[1], R[3 + i], po[2], R[6 + i]);
  double T[9];  // T = Cov_OG R
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int j = 0; j < 3; j++) T[3 * a + j] = dot3(co[3 * a], R[j], co[3 * a + 1], R[3 + j], co[3 * a + 2], R[6 + j]);
  int t = 0;
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = i; j < 3; j++) cov[t++] = dot3(R[i], T[j], R[3 + i], T[3 + j], R[6 + i], T[6 + j]);
}

__device__ __forceinline__ void vox_algebra2(const Chunk& ck, int pair, int cell, int iter, const float* Jm, const VoxMode& vm,
                                             double acc[NRED]) {
  const size_t ci = (size_t)pair * ck.ncell + cell;
  unsigned long long q[NQ];
  const unsigned long long* qp = ck.acc + ((size_t)vm.set * ck.npairs * ck.ncell + ci) * NQ;
#pragma unroll
  for (int k = 0; k < NQ; k += 2) {
    const ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(qp + k));
    q[k] = t.x;
    q[k + 1] = t.y;
  }
  double mean[3], cov[6];
  stats2_from_moments(q, ck.rec + (size_t)pair * ck.ncell, cell, vm, mean, cov);
  vox_algebra_core(ck, pair, cell, iter, Jm, (long long)q[0], mean, cov, acc);
}

__device__ __forceinline__ bool loop_incremental(const Chunk& ck) { return !(ck.flags & ICET_B200_FLAG_EXACT_PASS); }

__device__ __forceinline__ void vox_contrib(const Chunk& ck, int pair, int cell, int iter, const float* Jm,
                                            double acc[NRED]) {
  if (loop_incremental(ck)) {
    VoxMode vm;
    load_vox_mode(ck, pair, vm);
    if (vox_gate2(ck, pair, cell, iter, vm)) vox_algebra2(ck, pair, cell, iter, Jm, vm, acc);
  } else if (vox_gate(ck, pair, cell, iter)) {
    vox_algebra(ck, pair, cell, iter, Jm, acc);
  }
}

// ----------------------------------------------------------------------------------------------
// K6: one thread per pair: Q = pinv(H^T W H), pred_stds, checkCondition, dx, X += dx (src/icet.cpp:410-433,
// :443-492) and the transform / get_H trigonometry of the next iteration.  tot = the 28 sums over the voxels.
// ----------------------------------------------------------------------------------------------
// Odometry chaining (odometry.cpp:82 `X0 << X[0], ...`): the registration of pair k+1 starts from the solution of
// pair k.  Called by the thread that has just written X / TR / J of `pair` in the LAST iteration, before that
// iteration is published.
__device__ __forceinline__ void chain_seed_next(const Chunk& ck, int pair, const float* Xn) {
  if (!(ck.flags & ICET_B200_FLAG_CHAIN_X0) || pair + 1 >= ck.npairs) return;
  const int q = pair + 1;
  for (int k = 0; k < 6; k++) { ck.X[q * 6 + k] = Xn[k]; ck.res[q].X[k] = Xn[k]; }
  for (int k = 0; k < 12; k++) {
    const float v = ck.TR[(size_t)pair * 12 + k];
    ck.TR[(size_t)q * 12 + k] = v;
    ck.TRprev[(size_t)q * 12 + k] = v;
  }
  for (int k = 0; k < 27; k++) ck.J[(size_t)q * 27 + k] = ck.J[(size_t)pair * 27 + k];
  for (int k = 0; k < 12; k++) ck.pm[q].TRb[k] = ck.TR[(size_t)pair * 12 + k];  // its first iteration rebuilds at this transform
}

// Incremental loop: after the solve of an iteration, decide how the next one runs (see kernels_pass2.cuh).  tro / trn:
// the transform this iteration used / the next one will use.
// cur (optional): {SA, SB, set} of the iteration that has just run, when the caller already holds them in registers (the
// cluster loop) -- saves three dependent L2 round trips on the critical path.
struct ModeNow { float SA, SB; int set; };
__device__ __forceinline__ void mode_after_solve(const Chunk& ck, int pair, const float* tro, const float* trn,
                                                 const ModeNow* cur = nullptr) {
  PairMode* pm = ck.pm + pair;
  float a2 = 0.f, b2 = 0.f;
  for (int k = 0; k < 3; k++) b2 += (trn[k] - tro[k]) * (trn[k] - tro[k]);
  for (int k = 3; k < 12; k++) a2 += (trn[k] - tro[k]) * (trn[k] - tro[k]);
  const float SA = (cur ? cur->SA : __ldcg(&pm->SA)) + 1.001f * sqrtf(a2);
  const float SB = (cur ? cur->SB : __ldcg(&pm->SB)) + 1.001f * sqrtf(b2);
  const bool delta = !(ck.flags & ICET_B200_FLAG_FULL_REBUILD) && SA <= ck.inc_max_sa && SB <= ck.inc_max_sb;  // false for NaN
  if (delta) {
    pm->rebuild = 0;
    pm->SA = SA;
    pm->SB = SB;
    pm->C = (SB + SA * SB) * 1.0001f;
  } else {
    pm->set = (cur ? cur->set : __ldcg(&pm->set)) ^ 1;
    pm->rebuild = 1;
    pm->SA = 0.f;
    pm->SB = 0.f;
    pm->C = 0.f;
    for (int k = 0; k < 12; k++) pm->TRb[k] = trn[k];
  }
}

__device__ __noinline__ void solve_pair(const Chunk& ck, int pair, int iter, const double* tot, const ModeNow* cur = nullptr) {
  float* X = ck.X + pair * 6;
  double A[36], b[6];
  {
    int t = 0;
#pragma unroll
    for (int a = 0; a < 6; a++)
#pragma unroll
      for (int c = a; c < 6; c++) {
        A[a * 6 + c] = tot[t];
        A[c * 6 + a] = tot[t];
        t++;
      }
#pragma unroll
    for (int a = 0; a < 6; a++) b[a] = tot[21 + a];
  }
  icet_b200_result* R = ck.res + pair;
  double Q[36], dx[6], stds[6];
  int dropped = 0, status = 0;
  double cond_out = 0.0;
  bool fast = false;
  if (!(ck.flags & ICET_B200_FLAG_FULL_EIG) && icet::chol_inv6(A, Q)) {
    double trA = 0.0, trQ = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) { trA += A[k * 6 + k]; trQ += Q[k * 6 + k]; }
    // cond <= trace(A) * trace(A^-1); comfortably below the 1e6 cutoff => no axis is dropped and
    // pinv == inverse, so dx = A^-1 b  (src/icet.cpp:410-433 with an empty while-loop at :469)
    if (trA * trQ < 0.999e6) {
      fast = true;
      cond_out = -(trA * trQ);
    }
  }
  if (fast) {
#pragma unroll
    for (int k = 0; k < 6; k++) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < 6; j++) s += Q[k * 6 + j] * b[j];
      dx[k] = s;
      stds[k] = sqrt(fabs(Q[k * 6 + k]));
    }
  } else {
    double ev[6], U[36];
    icet::jacobi6(A, ev, U);
    // noise_mat = pinv(H^T W H) (:410-411) from the eigen-decomposition, with the rank rule of the COD
    // (pivot > FLT_EPSILON * 6 * largest pivot) applied to the spectrum
    {
      double lm = 0.0;
      for (int k = 0; k < 6; k++) lm = fmax(lm, fabs(ev[k]));
      const double thr = (double)FLT_EPSILON * 6.0 * lm;
      for (int i = 0; i < 36; i++) Q[i] = 0.0;
      for (int k = 0; k < 6; k++) {
        if (!(fabs(ev[k]) > thr)) continue;
        const double il = 1.0 / ev[k];
        for (int i = 0; i < 6; i++)
          for (int j = 0; j < 6; j++) Q[i * 6 + j] += U[i * 6 + k] * U[j * 6 + k] * il;
      }
    }
    for (int k = 0; k < 6; k++) stds[k] = sqrt(fabs(Q[k * 6 + k]));
    const double cutoff = 1e6;
    double condition = ev[5] / ev[0];
    cond_out = condition;
    int eyecount = 1;
    while (fabs(condition) > cutoff) {  // checkCondition :469-486
      if (eyecount > 5) { status = ICET_B200_COND_OVERFLOW; break; }
      for (int k = 0; k < 6; k++) stds[k] += U[k * 6 + (eyecount - 1)];  // :479
      dropped++;
      condition = ev[5] / ev[eyecount];
      eyecount++;
    }
    // dx = pinv(L2 lam U2^T) L2 U2^T b = sum over kept k of u_k (u_k . b) / lam_k, with the rank
    // rule of the COD applied to the kept spectrum (:427-430)
    double lmax = 0.0;
    for (int k = dropped; k < 6; k++) lmax = fmax(lmax, fabs(ev[k]));
    const double tiny = (double)FLT_EPSILON * (double)(6 - dropped) * lmax;
    for (int k = 0; k < 6; k++) dx[k] = 0.0;
    for (int k = dropped; k < 6; k++) {
      if (!(fabs(ev[k]) > tiny)) continue;
      double ub = 0.0;
      for (int j = 0; j < 6; j++) ub += U[j * 6 + k] * b[j];
      for (int j = 0; j < 6; j++) dx[j] += U[j * 6 + k] * (ub / ev[k]);
    }
  }
  float Xn[6];
  for (int k = 0; k < 6; k++) Xn[k] = (float)((double)__ldcg(X + k) + dx[k]);  // X += dx (:433), X is fp32
  for (int k = 0; k < 6; k++) X[k] = Xn[k];
  {  // trigonometry of the next iteration: utils::R (src/icet.cpp:375-376) and get_H (:507-527)
    float* TR = ck.TR + (size_t)pair * 12;
    float tro[12];
    for (int k = 0; k < 12; k++) tro[k] = __ldcg(TR + k);
    if (iter == ck.runlen - 1)
      for (int k = 0; k < 12; k++) ck.TRprev[(size_t)pair * 12 + k] = tro[k];
    if (ck.dump_on)
      for (int k = 0; k < 12; k++) ck.dump.TRit[iter * 12 + k] = tro[k];
    TR[0] = Xn[0]; TR[1] = Xn[1]; TR[2] = Xn[2];
    icet::rotR(Xn[3], Xn[4], Xn[5], TR + 3);
    icet::getH_J(Xn[3], Xn[4], Xn[5], ck.J + (size_t)pair * 27);
    if (loop_incremental(ck) && iter < ck.runlen - 1) mode_after_solve(ck, pair, tro, TR, cur);
    if (iter == ck.runlen - 1) chain_seed_next(ck, pair, Xn);
  }
  if (ck.dump_on) {
    for (int k = 0; k < 6; k++) { ck.dump.Xit[iter * 6 + k] = Xn[k]; ck.dump.HTWdz[iter * 6 + k] = (float)b[k]; }
    for (int k = 0; k < 36; k++) ck.dump.HTWH[iter * 36 + k] = (float)A[k];
  }
  if (iter == ck.runlen - 1) {
    for (int k = 0; k < 6; k++) { R->X[k] = Xn[k]; R->pred_stds[k] = (float)stds[k]; }
    for (int k = 0; k < 36; k++) R->Q[k] = (float)Q[k];
    R->n_used = (int)(tot[27] + 0.5);
    R->n_dropped = dropped;
    R->cond = (float)cond_out;
  }
  if (status) R->status = status;
}

// Warp-parallel form of the common case of solve_pair: Gauss-Jordan elimination of [A | I | b] (13 columns, one
// per lane, no pivoting: A = H^T W H is symmetric positive definite whenever this path is valid).  Returns (warp
// uniform) false when a pivot is not positive or the bound trace(A) trace(A^-1) cannot prove cond <= 1e6; the caller
// then runs solve_pair (eigen-decomposition + the reference's truncation loop) on one thread.
__device__ __forceinline__ bool solve_pair_warp(const Chunk& ck, int pair, int iter, const double* tot,
                                                const ModeNow* cur = nullptr) {
  const int lane = threadIdx.x & 31;
  // requested now, used after the elimination: the current X and (last iteration) the transform it started from
  const float x_old = lane < 6 ? __ldcg(ck.X + pair * 6 + lane) : 0.f;
  const float tr_old = lane < 12 ? __ldcg(ck.TR + (size_t)pair * 12 + lane) : 0.f;
  double col[6];
  {
    // lane j < 6: column j of A; lane 6 + j: column j of I; lane 12: b
    const int j = lane < 6 ? lane : 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const int lo = i < j ? i : j, hi = i < j ? j : i;
      const double a = tot[lo * 6 - lo * (lo - 1) / 2 + (hi - lo)];  // packed upper triangle
      col[i] = lane < 6 ? a : (lane < 12 ? (lane - 6 == i ? 1.0 : 0.0) : (lane == 12 ? tot[21 + i] : 0.0));
    }
  }
  double trA = 0.0;
#pragma unroll
  for (int i = 0; i < 6; i++) trA += tot[i * 6 - i * (i - 1) / 2];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 6; k++) {
    const double piv = __shfl_sync(FULL, col[k], k);
    ok = ok && (piv > 0.0);
    const double ip = 1.0 / piv;
    col[k] *= ip;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      if (i == k) continue;
      const double f = __shfl_sync(FULL, col[i], k);
      col[i] -= f * col[k];
    }
  }
  double trQ = 0.0;
#pragma unroll
  for (int k = 0; k < 6; k++) trQ += __shfl_sync(FULL, col[k], 6 + k);
  // cond <= trace(A) * trace(A^-1); comfortably below the 1e6 cutoff => checkCondition drops nothing and
  // pinv == inverse, so dx = A^-1 b  (src/icet.cpp:410-433 with an empty while-loop at :469)
  if (!(ok && trA * trQ < 0.999e6)) return false;
  icet_b200_result* R = ck.res + pair;
  const bool last = iter == ck.runlen - 1;
  // ---- the update, warp-wide (one lane doing all of it serially was the longest stretch of the iteration)
  // X += dx (:433), X is fp32: lane k < 6 owns component k (dx_k lives in lane 12's col[k])
  double dxk = 0.0;
#pragma unroll
  for (int k = 0; k < 6; k++) {
    const double v = __shfl_sync(FULL, col[k], 12);
    dxk = (lane == k) ? v : dxk;
  }
  const float xn = (float)((double)x_old + dxk);
  // sines / cosines of the three angles on lanes 0..2, then every lane forms all of R(X) and the get_H matrices
  // (~100 flops, same expressions as utils::R / get_H) and stores the entries it owns
  float sv, cv;
  sincosf(__shfl_sync(FULL, xn, 3 + (lane % 3)), &sv, &cv);
  const float sph = __shfl_sync(FULL, sv, 0), cph = __shfl_sync(FULL, cv, 0);
  const float sth = __shfl_sync(FULL, sv, 1), cth = __shfl_sync(FULL, cv, 1);
  const float sps = __shfl_sync(FULL, sv, 2), cps = __shfl_sync(FULL, cv, 2);
  float Rm[9], Jm[27];
  icet::rotR_sc(sph, cph, sth, cth, sps, cps, Rm);
  icet::getH_J_sc(sph, cph, sth, cth, sps, cps, Jm);
  const float t_k = __shfl_sync(FULL, xn, lane < 3 ? lane : 0);
  float trv = t_k, jv = 0.f;
#pragma unroll
  for (int e = 0; e < 9; e++) trv = (lane == 3 + e) ? Rm[e] : trv;
#pragma unroll
  for (int e = 0; e < 27; e++) jv = (lane == e) ? Jm[e] : jv;
  const bool seed = last && (ck.flags & ICET_B200_FLAG_CHAIN_X0) && pair + 1 < ck.npairs;  // odometry.cpp:82
  if (lane < 6) {
    ck.X[pair * 6 + lane] = xn;
    if (last) R->X[lane] = xn;
    if (seed) { ck.X[(pair + 1) * 6 + lane] = xn; ck.res[pair + 1].X[lane] = xn; }
    if (ck.dump_on) { ck.dump.Xit[iter * 6 + lane] = xn; ck.dump.HTWdz[iter * 6 + lane] = (float)tot[21 + lane]; }
  }
  if (lane < 12) {
    if (last) ck.TRprev[(size_t)pair * 12 + lane] = tr_old;  // the transform the LAST iteration used (`points2`)
    if (ck.dump_on) ck.dump.TRit[iter * 12 + lane] = tr_old;
    ck.TR[(size_t)pair * 12 + lane] = trv;
    if (seed) {
      ck.TR[(size_t)(pair + 1) * 12 + lane] = trv;
      ck.TRprev[(size_t)(pair + 1) * 12 + lane] = trv;
      ck.pm[pair + 1].TRb[lane] = trv;  // its first iteration rebuilds at this transform
    }
  }
  if (loop_incremental(ck) && !last) {  // how the next iteration runs (same arithmetic as mode_after_solve)
    float tro[12], trn[12];
#pragma unroll
    for (int k = 0; k < 12; k++) { tro[k] = __shfl_sync(FULL, tr_old, k); trn[k] = __shfl_sync(FULL, trv, k); }
    if (lane == 0) mode_after_solve(ck, pair, tro, trn, cur);
  }
  if (lane < 27) {
    ck.J[(size_t)pair * 27 + lane] = jv;
    if (seed) ck.J[(size_t)(pair + 1) * 27 + lane] = jv;
  }
  if (last && lane == 12) {
    R->n_used = (int)(tot[27] + 0.5);
    R->n_dropped = 0;
    R->cond = (float)(-(trA * trQ));
  }
  if (ck.dump_on && lane < 6) {
    for (int i = 0; i < 6; i++) {
      const int lo = i < lane ? i : lane, hi = i < lane ? lane : i;
      ck.dump.HTWH[iter * 36 + i * 6 + lane] = (float)tot[lo * 6 - lo * (lo - 1) / 2 + (hi - lo)];
    }
  }
  if (last && lane >= 6 && lane < 12) {
    const int j = lane - 6;
#pragma unroll
    for (int i = 0; i < 6; i++) R->Q[i * 6 + j] = (float)col[i];
    // pred_stds = sqrt|diag noise_mat| (:414-417)
    double d = col[0];
#pragma unroll
    for (int i = 1; i < 6; i++) d = (j == i) ? col[i] : d;
    R->pred_stds[j] = (float)sqrt(fabs(d));
  }
  return true;
}

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TL(slot)                                                                         \
  do {                                                                                   \
    if (ck.dump_on && (threadIdx.x & 31) == 0) ck.dump.tl[(size_t)iter * 16 + (slot)] = gtime(); \
  } while (0)

__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Spin until *p >= need.  A protocol failure must not hang the GPU: after ck.loop_timeout_ns (default 20 s of
// %globaltimer, ICET_B200_LOOP_TIMEOUT_MS overrides: long enough for compute-sanitizer / time-sliced GPUs) the wait gives
// up, records what it was waiting for in ck.dbg and marks EVERY pair of the chunk (the host reports an error).
// The polling itself uses RELAXED loads: an acquire load is followed by an invalidation of the SM's whole L1
// (CCTL.IVALL), and thousands of spinning warps would keep every L1 of the GPU empty for the warps that do the work.
// One acquire load after the condition has been seen orders the reads that follow.
__device__ __forceinline__ int ld_relaxed(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __noinline__ void loop_wait(const Chunk& ck, const int* p, int need, int kind, int pair, int iter, unsigned ticket) {
  if (ld_acquire(p) >= need) return;
  const unsigned long long t0 = gtime();
  unsigned spins = 0;
  for (;;) {
    __nanosleep(40);
    const int seen = ld_relaxed(p);
    if (seen >= need) {
      ld_acquire(p);
      return;
    }
    if ((++spins & 1023u) == 0 && (gtime() - t0 > ck.loop_timeout_ns || ld_relaxed(ck.dbg) != 0)) {
      // give up (or another warp already has): every result of the chunk is poisoned, not only the waiting pair's --
      // tasks that proceed past a failed wait work on unfinished accumulators
      if ((threadIdx.x & 31) == 0 && atomicCAS(ck.dbg, 0, 1) == 0) {
        ck.dbg[1] = kind; ck.dbg[2] = pair; ck.dbg[3] = iter; ck.dbg[4] = seen; ck.dbg[5] = need; ck.dbg[6] = (int)ticket;
        for (int q = 0; q < ck.npairs; q++) ck.res[q].status = ICET_B200_LOOP_TIMEOUT;
      }
      return;
    }
  }
}

__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// warp tiles of a pair that are counted in tiles_done per iteration: those that hold points, at least tile 0
__device__ __forceinline__ int loop_tiles_of(int n2c, int tile_points) { return max(1, (n2c + tile_points - 1) / tile_points); }

// One vox task of k_loop (see there): the fitCells2 algebra of 32 consecutive cells, and, for the task that
// arrives last, the end of the iteration of the pair.
__device__ __noinline__ void vox_task(const Chunk& ck, int iter, int pair, int grp, int tpt, int vt, double* w_tot,
                                      float* w_J) {
  const int lane = threadIdx.x & 31;
  const int cell = grp * 32 + lane;
  const bool active = cell < ck.ncell && (ck.rec[(size_t)pair * ck.ncell + cell].flags & F_ACTIVE2) != 0;
  const bool any = __any_sync(FULL, active);
  if (any) {
    loop_wait(ck, reinterpret_cast<const int*>(ck.tiles_done + pair), (iter + 1) * loop_tiles_of(__ldg(ck.n2c + pair), tpt),
              1, pair, iter, 0u);
    if (lane < 27) w_J[lane] = __ldcg(ck.J + (size_t)pair * 27 + lane);
    __syncwarp();
    TL(1);
    double acc[NRED];
#pragma unroll
    for (int k = 0; k < NRED; k++) acc[k] = 0.0;
    if (cell < ck.ncell) vox_contrib(ck, pair, cell, iter, w_J, acc);
    TL(8);
    if (__any_sync(FULL, acc[27] != 0.0)) {
      double* out = ck.part + ((size_t)pair * vt + grp) * NRED;
      const double tot = warp_sum_transposed(acc, lane);
      if (lane < NRED) out[lane] = tot;
      TL(9);
      // (the fence below, executed by every lane before vox_done is bumped, also covers these stores and the mask bit)
      if (lane == 0) {
        red_or(ck.vmask + (size_t)pair * ((vt + 31) / 32) + (grp >> 5), 1u << (grp & 31));
      }
    }
    TL(2);
  } else if (ck.dump_on && cell < ck.ncell) {
    double none[NRED];
    vox_contrib(ck, pair, cell, iter, w_J, none);  // records the "inactive" markers (no voxel of the group is active)
  }
  __threadfence();  // every lane: partial sums, cleared accumulators, the group's vmask bit
  __syncwarp();
  unsigned prev = 0;
  if (lane == 0) {
    prev = atom_add(ck.vox_done + (size_t)pair * ck.runlen + iter, 1u);
  }
  prev = __shfl_sync(FULL, prev, 0);
  if (prev + 1u == (unsigned)vt) {
    // -------------------------------------------------------------- end of the iteration of this pair
    // Iterations of a pair are strictly ordered: groups without an active voxel do not wait for the tiles, so when
    // NO group of the pair has one (degenerate inputs) nothing else would keep iteration k+1 from being closed
    // before iteration k.
    if (iter > 0) loop_wait(ck, ck.iter_done + pair, iter, 2, pair, iter, 0u);
    else if ((ck.flags & ICET_B200_FLAG_CHAIN_X0) && pair > 0)
      loop_wait(ck, ck.iter_done + pair - 1, ck.runlen, 3, pair, iter, 0u);  // X of this pair comes from pair - 1
    __threadfence();
    TL(0);
    double tot = 0.0;
    const int nw = (vt + 31) / 32;
    for (int w = 0; w < nw; w++) {
      unsigned* mp = ck.vmask + (size_t)pair * nw + w;
      unsigned m = __ldcg(mp);
      if (lane == 0 && m) *mp = 0u;
      const double* pp = ck.part + ((size_t)pair * vt + (size_t)w * 32) * NRED + (lane < NRED ? lane : 0);
      while (m) {  // group order; four loads in flight
        int g[4];
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          g[u] = m ? __ffs(m) - 1 : -1;
          m = m ? (m & (m - 1)) : 0u;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) v[u] = (g[u] >= 0) ? __ldcg(pp + (size_t)g[u] * NRED) : 0.0;
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (g[u] >= 0) tot += v[u];
      }
    }
    __syncwarp();
    if (lane < NRED) w_tot[lane] = tot;
    __syncwarp();
    TL(3);
    bool done = false;
    if (!(ck.flags & ICET_B200_FLAG_FULL_EIG)) done = solve_pair_warp(ck, pair, iter, w_tot);
    if (!done && lane == 0) solve_pair(ck, pair, iter, w_tot);
    __threadfence();  // every lane: X, TR, J, result fields
    __syncwarp();
    TL(4);
    if (lane == 0) st_release(ck.iter_done + pair, iter + 1);
    TL(5);
  }
}

// ----------------------------------------------------------------------------------------------
// The Gauss-Newton loop of every pair of the chunk in ONE persistent launch (fitScan2 x runlen,
// src/icet.cpp:47, :372-436): nothing returns to the host between iterations.
//
// The worker is the WARP.  Work is a stream of tasks, ordered
//     for it in 0..runlen:  [ (it, pair, tile) for every pair, tile ]  then  [ (it, pair, vox group) for every pair, group ]
// and warps draw tickets from one counter.
//   * tile task: one warp tile of scan 2 through pass_warp_tile (transform ... integer accumulation), then
//     tiles_done[pair] += 1.  Needs X of iteration it: waits until iter_done[pair] >= it.
//   * vox task: the fitCells2 algebra of 32 consecutive cells (one per lane), a fixed-order warp reduction of the
//     28 sums into part[pair][group][28].  Needs all tiles of (pair, it): waits on tiles_done[pair].  The vox task
//     that arrives last (vox_done[pair][it]) adds the partials in group order, solves the 6x6 system on the warp
//     (solve_pair_warp), writes the next transform and publishes iter_done[pair] = it + 1.
// Every task only ever waits for tasks with SMALLER tickets, which are held by warps that are already running, so
// the scheme cannot deadlock whatever the number of resident warps.  With many pairs in flight nobody waits (the
// solve of one pair overlaps the tiles of the others); with one pair the waits ARE the latency-critical path and
// the vox groups / tiles of the pair spread over the whole GPU.
// ----------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(PASS_THREADS, 3) k_loop(const Chunk ck, int tiles, int vt) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* tab = reinterpret_cast<float*>(smem_raw + PASS_WARPS * pass_wslots(K) * 16);
  __shared__ unsigned long long s_mbar[PASS_WARPS];  // one mbarrier per warp: completion of its staged scan-2 tiles
  {
    const int ntab = pass_tab_floats(ck.nT, ck.nP);
    for (int k = threadIdx.x; k < ntab; k += PASS_THREADS) tab[k] = __ldg(ck.binrec + k);
  }
  __syncthreads();  // the only block-wide barrier: from here on warps are independent workers
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) mbar_init(&s_mbar[warp], 1);
  __syncwarp();
  unsigned mphase = 0u;
  int4* went = reinterpret_cast<int4*>(smem_raw) + warp * pass_wslots(K);
  static_assert(pass_wslots(K) * 16 >= 512, "warp scratch too small");
  double* w_tot = reinterpret_cast<double*>(went);                          // [28]   (vox tasks only)
  float* w_J = reinterpret_cast<float*>(reinterpret_cast<char*>(went) + 256);  // [27]
  const unsigned ntile = (unsigned)ck.npairs * (unsigned)tiles;
  const unsigned per_iter = ntile + (unsigned)ck.npairs * (unsigned)vt;
  const unsigned total = per_iter * (unsigned)ck.runlen;
  const bool chain = (ck.flags & ICET_B200_FLAG_CHAIN_X0) != 0;
  unsigned t = 0;
  if (lane == 0) t = atom_add(ck.ticket, 1u);
  t = __shfl_sync(FULL, t, 0);
  while (t < total) {
    // Throughput shape: the next ticket is drawn now, its round trip to L2 hides behind this task.  Latency shape
    // (small tiles, more resident warps than tasks per iteration): one ticket per warp -- a warp that holds two
    // tiles of the same iteration starts the second one a whole tile late, while idle warps could have taken it.
    unsigned t_next = 0;
    if (K > PASS_K_SMALL && lane == 0) t_next = atom_add(ck.ticket, 1u);
    // ticket -> task.  Independent pairs: iteration-major (see above).  Chained pairs (ICET_B200_FLAG_CHAIN_X0): pair-
    // major, i.e. all iterations of pair k before any task of pair k + 1, whose first tiles wait for the last solve
    // of pair k (it seeds X / TR / J of pair k + 1) -- still only waits on smaller tickets.
    int iter, pair_t, sub;
    bool is_tile;
    if (chain) {
      const unsigned per_it1 = (unsigned)(tiles + vt);
      const unsigned per_pair = per_it1 * (unsigned)ck.runlen;
      pair_t = (int)(t / per_pair);
      const unsigned r1 = t - (unsigned)pair_t * per_pair;
      iter = (int)(r1 / per_it1);
      const unsigned r2 = r1 - (unsigned)iter * per_it1;
      is_tile = r2 < (unsigned)tiles;
      sub = is_tile ? (int)r2 : (int)(r2 - (unsigned)tiles);
    } else {
      iter = (int)(t / per_iter);
      const unsigned rem = t - (unsigned)iter * per_iter;
      is_tile = rem < ntile;
      if (is_tile) {
        pair_t = (int)(rem / (unsigned)tiles);
        sub = (int)(rem - (unsigned)pair_t * (unsigned)tiles);
      } else {
        pair_t = (int)((rem - ntile) / (unsigned)vt);
        sub = (int)((rem - ntile) - (unsigned)pair_t * (unsigned)vt);
      }
    }
    if (is_tile) {
      // ------------------------------------------------------------------ tile task
      const int pair = pair_t;
      const int tile = sub;
      const int n = __ldg(ck.n2c + pair);
      const int w0 = tile * 32 * K;
      if (w0 < n || tile == 0) {
        if (iter > 0) loop_wait(ck, ck.iter_done + pair, iter, 0, pair, iter, t);
        else if (chain && pair > 0) loop_wait(ck, ck.iter_done + pair - 1, ck.runlen, 4, pair, iter, t);
        float tr[12];
        {
          const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
          const float4 a = __ldcg(tp), b = __ldcg(tp + 1), c = __ldcg(tp + 2);
          tr[0] = a.x; tr[1] = a.y; tr[2] = a.z; tr[3] = a.w; tr[4] = b.x; tr[5] = b.y; tr[6] = b.z; tr[7] = b.w;
          tr[8] = c.x; tr[9] = c.y; tr[10] = c.z; tr[11] = c.w;
        }
        const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
        unsigned long long* accp = ck.acc + (size_t)pair * ck.ncell * NQ;
        if (tile == 0) TL(6);
        if (ck.dump_on && iter == 3 && tile < 2048 && lane == 0) ck.dump.tl[(size_t)ck.runlen * 16 + 2 * tile] = gtime();
        if (loop_incremental(ck)) {
          Pass2Mode md;
          load_pass2_mode(ck, pair, md);
          pass2_warp_tile<K>(ck, went, &s_mbar[warp], mphase, false, tab, recs, tr, md, ck.pog + (size_t)pair * 3 * ck.n2max,
                             (size_t)ck.n2max, n, w0, ck.mrec + (size_t)pair * ck.n2max,
                             (ck.flags & ICET_B200_FLAG_VERIFY_INCREMENTAL) ? &ck.res[pair].reserved[0] : nullptr);
          if (tile == 0 && lane == 0)
            pass2_dropped_returns(ck, reinterpret_cast<const float4*>(tab), reinterpret_cast<const float4*>(tab) + ck.nT + 2,
                                  recs, tr, md, pair, __ldg(ck.nz2 + pair));
        } else {
        const int n2 = __ldg(&ck.desc[pair].n2);
        pass_warp_tile<true, K, 2, (K <= 4 ? K : 1)>(ck, went, tab, recs, tr, ck.pog + (size_t)pair * 3 * ck.n2max, (size_t)ck.n2max, n, w0,
                                fix_point(n2), accp, (ck.dump_on && iter == 3 && tile < 2048) ? ck.dump.tl + (size_t)ck.runlen * 16 + 4096 + tile : nullptr);
        if (tile == 0 && lane == 0)
          pass_dropped_returns(ck, reinterpret_cast<const float4*>(tab), reinterpret_cast<const float4*>(tab) + ck.nT + 2,
                               recs, tr, accp, __ldg(ck.nz2 + pair), n2);
        }
        if (tile == 0) TL(7);
        if (ck.dump_on && iter == 3 && tile < 2048 && lane == 0) ck.dump.tl[(size_t)ck.runlen * 16 + 2 * tile + 1] = gtime();
        __threadfence();  // every lane: its accumulator updates are visible before the tile is counted
        __syncwarp();
        if (lane == 0) red_add(ck.tiles_done + pair, 1u);
      }  // tiles beyond the compacted point count of the pair are not counted (see loop_tiles_of)
    } else {
      // ------------------------------------------------------------------ vox task
      vox_task(ck, iter, pair_t, sub, 32 * K, vt, w_tot, w_J);
    }
    if (K <= PASS_K_SMALL && lane == 0) t_next = atom_add(ck.ticket, 1u);
    t = __shfl_sync(FULL, t_next, 0);
  }
}

// Split form of the loop (chunks of more than one pair): k_pass2 / k_pass<true>, then these two, per iteration.
constexpr int VOX_GRID = 8;  // blocks per pair of k_vox2 (each strides over the pair's active voxels)

// the pair's active voxels in ascending cell order (once per chunk, after k_fit1 has set F_ACTIVE2)
__global__ void __launch_bounds__(256) k_vox_list(const Chunk ck) {
  const int pair = blockIdx.x;
  __shared__ int s_w[8];
  const int per = (ck.ncell + 255) / 256;
  const int c0 = threadIdx.x * per, c1 = min(ck.ncell, c0 + per);
  const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int mine = 0;
  for (int c = c0; c < c1; c++) mine += (recs[c].flags & F_ACTIVE2) ? 1 : 0;
  int inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(FULL, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  int base = inc - mine;
  for (int w = 0; w < warp; w++) base += s_w[w];
  int32_t* out = ck.vlist + (size_t)pair * ck.ncell;
  for (int c = c0; c < c1; c++)
    if (recs[c].flags & F_ACTIVE2) out[base++] = c;
  if (threadIdx.x == 255) ck.nvox[pair] = base;
}

__global__ void __launch_bounds__(VOX_THREADS) k_vox2(const Chunk ck, int iter) {
  const int pair = blockIdx.y;
  __shared__ double s_red[NRED];
  double acc[NRED];
#pragma unroll
  for (int k = 0; k < NRED; k++) acc[k] = 0.0;
  if (ck.dump_on) {  // every cell (grid: one block per VOX_THREADS cells)
    const int cell = blockIdx.x * VOX_THREADS + threadIdx.x;
    if (cell < ck.ncell) vox_contrib(ck, pair, cell, iter, ck.J + (size_t)pair * 27, acc);
  } else {
    const int nv = ck.nvox[pair];
    const int32_t* vl = ck.vlist + (size_t)pair * ck.ncell;
    for (int k = blockIdx.x * VOX_THREADS + threadIdx.x; k < nv; k += gridDim.x * VOX_THREADS)
      vox_contrib(ck, pair, __ldg(vl + k), iter, ck.J + (size_t)pair * 27, acc);
  }
  // fixed-order reduction: xor butterfly inside each warp, then warp 1 + warp 0
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const bool any = __syncthreads_or(acc[27] != 0.0);
  double* out = ck.part + ((size_t)pair * gridDim.x + blockIdx.x) * NRED;
  if (!any) {  // block-uniform: nothing to add
    if (threadIdx.x < NRED) out[threadIdx.x] = 0.0;
    return;
  }
  const double tot = warp_sum_transposed(acc, lane);
  if (wid == 1 && lane < NRED) s_red[lane] = tot;
  __syncthreads();
  if (wid == 0 && lane < NRED) out[lane] = tot + s_red[lane];
}

constexpr int SOLVE_THREADS = 128;
__global__ void __launch_bounds__(SOLVE_THREADS) k_solve6(const Chunk ck, int iter, int nblk) {
  const int pair = blockIdx.x;
  const int lane = threadIdx.x;
  __shared__ double s_tot[NRED];
  __shared__ float s_trb[12];
  __shared__ int s_rebuild;
  if (lane < NRED) {
    double mine = 0.0;
    const double* pp = ck.part + (size_t)pair * nblk * NRED + lane;
    for (int b = 0; b < nblk; b++) mine += pp[(size_t)b * NRED];
    s_tot[lane] = mine;
  }
  __syncwarp();
  // (one thread: this kernel is bound by instruction fetch of once-executed code, the warp-parallel solve of
  // k_loop is not faster here)
  if (lane == 0) {
    solve_pair(ck, pair, iter, s_tot);
    s_rebuild = 0;
    if (loop_incremental(ck) && iter < ck.runlen - 1) {
      s_rebuild = ck.pm[pair].rebuild;  // (written by this thread a moment ago)
      for (int k = 0; k < 12; k++) s_trb[k] = ck.pm[pair].TRb[k];
    }
  }
  __syncthreads();
  // the next iteration rebuilds: the anchors of the voxel frames at ITS transform, for k_pass2 (all threads)
  if (s_rebuild) {
    float trb[12];
    for (int k = 0; k < 12; k++) trb[k] = s_trb[k];
    anchors_update(ck, pair, trb, threadIdx.x, SOLVE_THREADS);
  }
}

// public member `points2` of the reference: scan 2 as transformed by the last iteration
// ((points2_OG + t) * R with the X that iteration STARTED from, src/icet.cpp:375-378), pair 0 of the chunk
__global__ void k_points2(const Chunk ck, int n2, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n2) return;
  const PairDesc d = ck.desc[0];
  float x = d.s2[i], y = d.s2[d.ld2 + i], z = d.s2[2 * (size_t)d.ld2 + i];
  if (ck.runlen > 0) {  // without an iteration the member is still the constructor's copy of scan 2 (src/icet.cpp:30)
    float r, th, ph;
    icet::c2s(x, y, z, r, th, ph);   // points2_OG (prepScan2, src/icet.cpp:263-275), recomputed: the workspace
    icet::s2c(r, th, ph, x, y, z);   // copy is compacted
    icet::transform(x, y, z, ck.TRprev, ck.TRprev + 3, x, y, z);
  }
  out[i] = x;
  out[n2 + i] = y;
  out[2 * (size_t)n2 + i] = z;
}

// parity-test entry (icet_b200_classify_scan2): class of every point of scan 2 of pair 0 under the transform `tr`
__global__ void k_classify2(const Chunk ck, int n2, const float* trp, int32_t* cell, uint8_t* in) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n2) return;
  const PairDesc d = ck.desc[0];
  float tr[12];
  for (int k = 0; k < 12; k++) tr[k] = trp[k];
  float x = d.s2[i], y = d.s2[d.ld2 + i], z = d.s2[2 * (size_t)d.ld2 + i];
  float r, th, ph;
  icet::c2s(x, y, z, r, th, ph);   // points2_OG (prepScan2, src/icet.cpp:263-275)
  icet::s2c(r, th, ph, x, y, z);
  const float4* tth = reinterpret_cast<const float4*>(ck.binrec);
  int c;
  bool active, inb;
  point_stage1<true>(ck, tth, tth + ck.nT + 2, ck.rec, tr, x, y, z, c, active, inb, r, th, ph);
  cell[i] = c;
  in[i] = inb ? 1 : 0;
}

// spherical coordinates + cell index of a cloud (parity-test entry point)
__global__ void k_sph_bins(const float* s, int n, int ld, int nT, int nP, icet::BinTable bth, icet::BinTable bph,
                           float* sph, int32_t* cell) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r, th, ph;
  icet::c2s(s[i], s[ld + i], s[2 * (size_t)ld + i], r, th, ph);
  int bt, bp;
  bt = icet::bin_lookup(th, bth, 2 * M_PI);
  bp = icet::bin_lookup(ph, bph, M_PI);
  sph[i] = r; sph[n + i] = th; sph[2 * (size_t)n + i] = ph;
  cell[i] = nT * bp + bt;
}

// synthetic scans
__global__ void k_synth(uint64_t seed, int first_scan, int nscans, int rings, int azim, const synth::Pose* poses,
                        float* out) {
  const int npts = rings * azim;
  const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (size_t)nscans * npts) return;
  const int s = (int)(gid / npts), i = (int)(gid % npts);
  const int ring = i / azim, az = i % azim;
  float x, y, z;
  synth::ray(seed, first_scan + s, poses[s], ring, rings, az, azim, x, y, z);
  float* o = out + (size_t)s * 3 * npts;
  o[i] = x; o[npts + i] = y; o[2 * (size_t)npts + i] = z;
}


// icet_b200/csrc/kernels_pass2.cuh -- K5i: the INCREMENTAL pass over scan 2 (default form of the Gauss-Newton loop).
// Included by icet_b200.cu inside its anonymous namespace.
//
// What the reference does per iteration (src/icet.cpp:372-403): transform every point of scan 2, convert it to spherical
// coordinates, bin it, test it against the cluster box of its cell, convert the survivors back (sphericalToCartesian)
// and take mean / covariance per voxel.  From the second or third iteration on the transform moves the points by
// millimetres and almost none of them changes its voxel or its side of a cluster box.  This pass therefore keeps, per
// voxel, EXACT integer moments (count, sum, sum of products) of the UNTRANSFORMED members (points2_OG, prepScan2) and,
// per point, ONE 64-bit margin record: the class (cell | in-box) of its last evaluation together with a margin, a bound
// on how far the point can move before ANY comparison that decided its class can change.  A warp works on a tile of
// 32*K consecutive stored points whose coordinates the TMA engine stages in shared memory (three bulk asynchronous
// copies issued by one lane, completion on the warp's mbarrier).  An iteration then
//   * REBUILD (first iteration, or when the transform has moved by more than INC_MAX_SA / INC_MAX_SB since the last
//     rebuild): evaluates every point like the per-point pass (transform, spherical, bin + box look-up, range test),
//     records class and margin, and accumulates the moments of the inside points from zero;
//   * DELTA: re-evaluates only the points whose margin is used up by the motion since their evaluation (one 8-byte
//     load, one FMA, one compare for all the others) and moves the few points whose class changed from one voxel's
//     moments to another's.
// The per-voxel algebra (vox_algebra2, kernels_loop.cuh) transforms the moments analytically:
//     mu2 = (mean_OG + t) R,   Sigma2 = R^T Cov_OG R        (src/icet.cpp:375-378 applied to the moments).
//
// Parity (DESIGN.md "incremental scan-2 loop"): the CLASS of every point in every iteration is the one the per-point
// fp32 pipeline computes (the margins are conservative bounds that include the fp32 rounding of that pipeline; tested
// against the forced-rebuild form and against the per-point form ICET_B200_FLAG_EXACT_PASS), so voxel indices, bin
// counts and in-box counts are unchanged.  Mean / covariance of scan 2 no longer go through the per-point fp32 round
// trip: they differ from the reference's by that round trip's own rounding noise (<= a few ulp of the coordinates per
// point, averaged over the voxel) and are closer to the exact statistics of the transformed points.
#pragma once

// Delta iterations while the motion since the last rebuild stays below these bounds.  A delta iteration costs ~20
// instructions and 8 bytes per point plus a full evaluation for the points whose margin is used up (from a staged tile
// when more than one point in eight is listed, gathered otherwise).  Measured on the bench pairs (256-pair launches, 7
// iterations, r02j): bounds 1e-3 / 5 cm: 24.3 ms per 4096 pairs; 2e-3 / 8 cm: 24.4; 4e-3 / 12 cm: 25.4 -- the heavy
// delta iterations that wider bounds create cost what the rebuilds they replace did (ICET_B200_INC_SA / _SB: A/B runs).
constexpr float INC_MAX_SA = 1.0e-3f;         // sum |dR|_F   (x 30 m = 3 cm)
constexpr float INC_MAX_SB = 0.05f;           // sum |dt|     (metres)
// (The members of a voxel sit within one box diameter D of its anchor when they are evaluated and the anchor drifts by
// at most r * INC_MAX_SA + INC_MAX_SB < D (D >= 0.2 r + 0.2 m) before the next rebuild re-anchors it: the +-2 D range of
// the fixed-point frame (FixPt::fl) is never left.)

struct Pass2Mode {  // block-uniform copy of the pair's PairMode + accumulator set
  bool rebuild;
  int set;
  float fs2;
  int fl2;
  float SA, SB, C;
  const float* trbp;  // PairMode::TRb (global): transform of the last rebuild, loaded only where a class changes --
                      // in a rebuild iteration it IS the current transform
  unsigned long long* accp;
};

// ---- margin record of a stored point: 64 bits {u | class low byte, r_e | class high 16 bits}.
//   r_e is rounded UP to bf16 (<= 0.8 % more motion charged to the point: < 1 mm at 30 m for the SA bounds used) and u,
//   which is computed with that rounded r_e, is rounded DOWN to 24 significant bits (< 2^-16 relative) and clamped at
//   0: both make the stability test r_e * SA + C < u more conservative, never less.  u = 0 (also for NaN): the point is
//   evaluated in every iteration.
__device__ __forceinline__ float rec2_round_re(float r) {
  return __uint_as_float((__float_as_uint(r * 1.000001f) + 0xffffu) & 0xffff0000u);
}
__device__ __forceinline__ uint2 rec2_pack(float u, float re /* rec2_round_re */, uint32_t cls) {
  return make_uint2((__float_as_uint(fmaxf(u, 0.f)) & 0xffffff00u) | (cls & 0xffu), __float_as_uint(re) | (cls >> 8));
}
__device__ __forceinline__ float rec2_u(uint2 v) { return __uint_as_float(v.x & 0xffffff00u); }
__device__ __forceinline__ float rec2_re(uint2 v) { return __uint_as_float(v.y & 0xffff0000u); }
__device__ __forceinline__ uint32_t rec2_cls(uint2 v) { return (v.x & 0xffu) | ((v.y & 0xffffu) << 8); }

// bin + box look-up (see bin_box) that also returns the distance of the angle to the nearest threshold that decided it
__device__ __forceinline__ int bin_box_m(float a, const float4* rec, const icet::BinTable& bt, bool& inbox, float& dist) {
  int k = __float2int_rz(fminf(a, bt.acap) * bt.scale);
  float4 e = rec[k];
  if (a < e.x || a >= e.y) {
    k += (a < e.x) ? -1 : 1;
    e = rec[k];
  }
  inbox = a >= e.z && a <= e.w;
  dist = fminf(fminf(fabsf(a - e.x), fabsf(e.y - a)), fminf(fabsf(a - e.z), fabsf(e.w - a)));
  return k < bt.nb ? k : (k == bt.nb ? 0 : bt.sbin);
}

// Full evaluation of one point of scan 2: class word and {u, r_e}.
//   The class can only change when the computed theta / phi / r crosses one of the thresholds it was compared with.
//   A displacement delta of the transformed point changes theta by <= asin(delta / rho), phi by <= asin(delta / r) and
//   r by <= delta; the fp32 evaluation itself is within (2e-6 rad * rho + 3e-6 r) / (4e-6 rad * r / rho) / 4e-6 r of
//   exact for theta / phi / r (transform: 3 roundings per coordinate; own atan2 / acos within 1 ulp; IEEE sqrt, div),
//   counted twice (evaluation now, evaluation then).  m = the smallest distance to a threshold in metres minus that
//   slop, capped at rho / 4 (asin(x) <= 1.011 x there); the class is safe while delta < 0.9 m.
//   delta(e -> k) <= r_e (SA_k - SA_e) + SB_k SA_k + (SB_k - SB_e), hence the stored u = 0.9 m + r_e SA_e + SB_e and the
//   test r_e SA_k + C_k < u with C_k = SB_k + SA_k SB_k.
__device__ __forceinline__ void point_eval2(const Chunk& ck, const float4* tth, const float4* tph, const CellRec* recs,
                                            const float* tr, float SA, float SB, float px, float py, float pz,
                                            uint32_t& cls, float2& mg) {
  float x, y, z;
  icet::transform(px, py, pz, tr, tr + 3, x, y, z);
  const float sxy = __fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y));
  float r, th, ph;
  icet::c2s(x, y, z, r, th, ph);
  bool bt_in, bp_in;
  float dth, dph;
  const int bt = bin_box_m(th, tth, ck.bth, bt_in, dth);
  const int bp = bin_box_m(ph, tph, ck.bph, bp_in, dph);
  const int c = ck.nT * bp + bt;
  const float4 ra = __ldg(reinterpret_cast<const float4*>(recs + c));  // inner, outer, flags, scale
  const bool active = (__float_as_uint(ra.z) & F_ACTIVE2) != 0;
  const bool in = active && bt_in && bp_in && r >= ra.x && r <= ra.y;
  cls = (uint32_t)c | (in ? CLS_IN : 0u) | (active ? CLS_ACTIVE : 0u);
  float irho;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(irho) : "f"(sxy));
  const float rho = sxy * irho * 0.999f;
  const float k = r * irho * 1.001f;
  float m = fminf((dth - 2e-6f) * rho - 3e-6f * r, (dph - 4e-6f * k) * r);
  m = fminf(m, 0.25f * rho);
  if (active) m = fminf(m, fminf(fabsf(r - ra.x), fabsf(ra.y - r)) - 4e-6f * r);
  const float re = rec2_round_re(r);
  float u = fmaf(0.9f, m, -1e-6f) + fmaf(re, SA, SB);
  // non-finite coordinates (NaN rows take the 1000.0 sentinels, :116): evaluated every time
  if (!(__fadd_rn(sxy, __fmul_rn(z, z)) < 3e38f) || !(sxy > 1e-30f) || !(u == u)) u = 0.f;
  mg = make_float2(u, re);
}

// ---- Filtered evaluation.  The incremental loop needs the CLASS of a point and a conservative margin, not the values
// of theta / phi / r themselves.  Approximate angles (reciprocal / rsqrt approximations, fp32 octant fix-up; each
// within TAU of the exactly evaluated fp32 pipeline) decide the class whenever they are further than TAU from every
// threshold they are compared with -- then the exact pipeline cannot decide differently -- and only the remaining
// points (a few in 10^4) go through the exact evaluation point_eval2.  Less than half the instructions per point.
constexpr float TAU_TH = 3.0e-6f;  // |theta_fast - theta_exact| < 2e-6 (rcp.approx 1e-7 rel, polynomial 1e-7, three fp32
                                   // subtractions <= 6e-7, constants 2e-7; exact side: own atan2 within 1 ulp = 4.8e-7)
constexpr float TAU_PH = 1.5e-6f;  // |phi_fast - phi_exact| < 1e-6 for |z/r| <= 0.5 (rsqrt.approx 2e-7 rel, polynomial 1e-7)
constexpr float TAU_R = 1.0e-6f;   // |r_fast - r_exact| < 5e-7 r (rsqrt.approx; the exact side is IEEE sqrt)

__device__ __forceinline__ float fast_theta(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const bool steep = ay > ax;
  const float mx = steep ? ay : ax, mn = steep ? ax : ay;
  float rc;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(mx));
  const float t = mn * rc;  // NaN for (0, 0): every comparison below fails and the point takes the exact path
  const float s = t * t;
  float p = -0.0019267977913841605f;
  p = fmaf(p, s, 0.01150327268987894f);
  p = fmaf(p, s, -0.03226083889603615f);
  p = fmaf(p, s, 0.059030335396528244f);
  p = fmaf(p, s, -0.08465225994586945f);
  p = fmaf(p, s, 0.10972991585731506f);
  p = fmaf(p, s, -0.14268141984939575f);
  p = fmaf(p, s, 0.19998906552791595f);
  p = fmaf(p, s, -0.3333331048488617f);
  float v = fmaf(t * s, p, t);
  v = steep ? (1.57079632679489662f - v) : v;
  v = (x < 0.0f) ? (3.14159265358979324f - v) : v;
  v = (y < 0.0f) ? (6.28318530717958648f - v) : v;
  return v;
}

__device__ __forceinline__ void point_eval2_fast(const Chunk& ck, const float4* tth, const float4* tph, const CellRec* recs,
                                                 const float* tr, float SA, float SB, float px, float py, float pz,
                                                 uint32_t& cls, float2& mg) {
  float x, y, z;
  icet::transform(px, py, pz, tr, tr + 3, x, y, z);
  const float sxy = fmaf(y, y, x * x);
  const float s = fmaf(z, z, sxy);
  float irs, irho;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(irs) : "f"(s));
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(irho) : "f"(sxy));
  const float r = s * irs;
  const float q = z * irs;
  const float th = fast_theta(y, x);
  const float q2 = q * q;
  float pp = 0.0435001514852047f;
  pp = fmaf(pp, q2, 0.023313719779253006f);
  pp = fmaf(pp, q2, 0.045668356120586395f);
  pp = fmaf(pp, q2, 0.07493448257446289f);
  pp = fmaf(pp, q2, 0.166668102145195f);
  const float ph = 1.57079632679489662f - fmaf(q * q2, pp, q);
  // "sure" intervals (host: ensure_edges): strictly inside (lo + TAU, hi - TAU) of record k the exact pipeline finds
  // bin k and passes the bin's fp32 box test as well.  NaN indexes record 0 and fails every comparison.
  const float2* sth = reinterpret_cast<const float2*>(tth + ck.nT + ck.nP + 4);
  const float2* sph = sth + ck.nT + 2;
  const int bt = min(__float2int_rz(th * ck.bth.scale), ck.nT + 1);
  const int bp = min(__float2int_rz(ph * ck.bph.scale), ck.nP + 1);
  const float2 et = sth[bt], ep = sph[bp];
  const float dth = fminf(th - et.x, et.y - th), dph = fminf(ph - ep.x, ep.y - ph);
  const int c = ck.nT * min(bp, ck.nP - 1) + min(bt, ck.nT - 1);  // (clamped only so that the load below is in range)
  const float4 ra = __ldg(reinterpret_cast<const float4*>(recs + c));  // inner, outer, flags, scale
  const bool active = (__float_as_uint(ra.z) & F_ACTIVE2) != 0;
  const float dr = fminf(fabsf(r - ra.x), fabsf(ra.y - r));
  // (written so that NaN / inf anywhere fails the test)
  const bool sure = dth > 0.f && dph > 0.f && fabsf(q) <= 0.5f && s < 3e38f && sxy > 1e-30f && (!active || dr > TAU_R * r);
  if (!sure) {
    point_eval2(ck, tth, tph, recs, tr, SA, SB, px, py, pz, cls, mg);
    return;
  }
  const bool in = active && r >= ra.x && r <= ra.y;
  cls = (uint32_t)c | (in ? CLS_IN : 0u) | (active ? CLS_ACTIVE : 0u);
  // margin as in point_eval2, every distance reduced by the approximation error as well (TAU is in the table already)
  const float rho = sxy * irho * 0.999f;
  const float k = r * irho * 1.001f;
  float m = fminf((dth - 2e-6f) * rho - 3e-6f * r, (dph - 4e-6f * k) * r);
  m = fminf(m, 0.25f * rho);
  if (active) m = fminf(m, dr - (TAU_R + 4e-6f) * r);
  const float re = rec2_round_re(r);
  mg = make_float2(fmaf(0.9f, m, -1e-6f) + fmaf(re, SA, SB), re);
}

// anchor of a voxel's scan-2 fixed-point frame: the centre of its box, taken back through the transform of the last
// rebuild (p = q R^T - t), and the scale
__device__ __forceinline__ void vox_anchor2_rec(float4 ra /* inner outer flags scale */, float4 rb /* ref xyz, cnt1 */,
                                                const float* trb, float fs2, float& ax, float& ay, float& az, float& sc);
__device__ __forceinline__ void vox_anchor2(const CellRec* recs, int cell, const float* trb, float fs2, float& ax, float& ay,
                                            float& az, float& sc) {
  const float4* rp = reinterpret_cast<const float4*>(recs + cell);
  vox_anchor2_rec(__ldg(rp), __ldg(rp + 1), trb, fs2, ax, ay, az, sc);
}
__device__ __forceinline__ void vox_anchor2_rec(float4 ra, float4 rb, const float* trb, float fs2, float& ax, float& ay,
                                                float& az, float& sc) {
  const float* R = trb + 3;
  sc = ra.w * fs2;
  ax = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(rb.x, R[0]), __fmul_rn(rb.y, R[1])), __fmul_rn(rb.z, R[2])), -trb[0]);
  ay = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(rb.x, R[3]), __fmul_rn(rb.y, R[4])), __fmul_rn(rb.z, R[5])), -trb[1]);
  az = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(rb.x, R[6]), __fmul_rn(rb.y, R[7])), __fmul_rn(rb.z, R[8])), -trb[2]);
}
// Anchor table of a pair (Chunk::anch) at the transform `trb` of the rebuild that comes next: the threads of a block,
// `nth` of them, cell by cell.  Same function and inputs as the per-voxel algebra uses (stats2_from_moments): bit-identical.
__device__ __forceinline__ void anchors_update(const Chunk& ck, int pair, const float* trb, int tid, int nth) {
  const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
  float4* an = ck.anch + (size_t)pair * ck.ncell;
  const float fs2 = fix_point(ck.desc[pair].n2).fs;
  for (int c = tid; c < ck.ncell; c += nth) {
    const float4* rp = reinterpret_cast<const float4*>(recs + c);
    const float4 ra = __ldcg(rp);
    if (!(__float_as_uint(ra.z) & F_ACTIVE2)) continue;
    float ax, ay, az, sc;
    vox_anchor2_rec(ra, __ldcg(rp + 1), trb, fs2, ax, ay, az, sc);
    an[c] = make_float4(ax, ay, az, sc);
  }
}
__device__ __forceinline__ void fix2(float px, float py, float pz, float ax, float ay, float az, float sc, int lim, int& fx,
                                     int& fy, int& fz) {
  fx = max(-lim, min(lim, __float2int_rn(__fmul_rn(__fadd_rn(px, -ax), sc))));
  fy = max(-lim, min(lim, __float2int_rn(__fmul_rn(__fadd_rn(py, -ay), sc))));
  fz = max(-lim, min(lim, __float2int_rn(__fmul_rn(__fadd_rn(pz, -az), sc))));
}

// adds (w = +n) or removes (w = -n) n copies of an inside point to / from the moments of its voxel (rare: only where the
// class of a point changed in a delta iteration; the anchor transform comes straight from global memory)
__device__ __forceinline__ void moments_add(unsigned long long* accp, const CellRec* recs, int cell, const Pass2Mode& md,
                                            float px, float py, float pz, long long w) {
  float trb[12];
  {
    const float4* tb = reinterpret_cast<const float4*>(md.trbp);
    const float4 a = __ldcg(tb), b = __ldcg(tb + 1), c = __ldcg(tb + 2);
    trb[0] = a.x; trb[1] = a.y; trb[2] = a.z; trb[3] = a.w; trb[4] = b.x; trb[5] = b.y; trb[6] = b.z; trb[7] = b.w;
    trb[8] = c.x; trb[9] = c.y; trb[10] = c.z; trb[11] = c.w;
  }
  float ax, ay, az, sc;
  vox_anchor2(recs, cell, trb, md.fs2, ax, ay, az, sc);
  int ix, iy, iz;
  fix2(px, py, pz, ax, ay, az, sc, md.fl2, ix, iy, iz);
  const long long fx = ix, fy = iy, fz = iz;
  unsigned long long* q = accp + (size_t)cell * NQ;
  red_add(q + 1, (unsigned long long)w);
  red_add(q + 2, (unsigned long long)(w * fx));
  red_add(q + 3, (unsigned long long)(w * fy));
  red_add(q + 4, (unsigned long long)(w * fz));
  red_add(q + 5, (unsigned long long)(w * fx * fx));
  red_add(q + 6, (unsigned long long)(w * fx * fy));
  red_add(q + 7, (unsigned long long)(w * fx * fz));
  red_add(q + 8, (unsigned long long)(w * fy * fy));
  red_add(q + 9, (unsigned long long)(w * fy * fz));
  red_add(q + 10, (unsigned long long)(w * fz * fz));
}

// moves `w` copies of a point from class `oc` to class `nc` (either may be CLS_NONE / inactive)
__device__ __forceinline__ void class_move(unsigned long long* accp, const CellRec* recs, const Pass2Mode& md, uint32_t oc,
                                           uint32_t nc, float px, float py, float pz, long long w) {
  if (oc == nc) return;
  const int ocell = (int)(oc & CLS_CELL), ncell_ = (int)(nc & CLS_CELL);
  const bool oact = (oc & CLS_ACTIVE) != 0, nact = (nc & CLS_ACTIVE) != 0;
  if (ocell != ncell_) {
    if (oact) red_add(accp + (size_t)ocell * NQ, (unsigned long long)(-w));
    if (nact) red_add(accp + (size_t)ncell_ * NQ, (unsigned long long)w);
  }
  if (oc & CLS_IN) moments_add(accp, recs, ocell, md, px, py, pz, -w);
  if (nc & CLS_IN) moments_add(accp, recs, ncell_, md, px, py, pz, w);
}

// The dropped returns of scan 2 (points2_OG == (0,0,0) for all nz of them, SURVEY.md A.12): one point with weight nz,
// evaluated every iteration by one thread.
__device__ inline void pass2_dropped_returns(const Chunk& ck, const float4* tth, const float4* tph, const CellRec* recs,
                                             const float* tr, const Pass2Mode& md, int pair, long long nz) {
  if (nz <= 0) return;
  uint32_t cls;
  float2 mg;
  point_eval2(ck, tth, tph, recs, tr, 0.f, 0.f, 0.f, 0.f, 0.f, cls, mg);
  const uint32_t old = md.rebuild ? CLS_NONE : (uint32_t)__ldcg(&ck.pm[pair].zcls);
  class_move(md.accp, recs, md, old, cls, 0.f, 0.f, 0.f, nz);
  ck.pm[pair].zcls = (int)cls;
}

// publishes what one lane collected over a run of consecutive ACTIVE points of one cell: the bin count, and the sums of
// the inside points among them
__device__ __forceinline__ void flush_run2(unsigned long long* accp, int cell, int nb, int nin, int sx, int sy, int sz,
                                           long long pxx, long long pxy, long long pxz, long long pyy, long long pyz,
                                           long long pzz) {
  if (cell < 0) return;
  unsigned long long* q = accp + (size_t)cell * NQ;
  red_add(q, (unsigned long long)nb);
  if (nin == 0) return;
  red_add(q + 1, (unsigned long long)nin);
  red_add(q + 2, (unsigned long long)(long long)sx);
  red_add(q + 3, (unsigned long long)(long long)sy);
  red_add(q + 4, (unsigned long long)(long long)sz);
  red_add(q + 5, (unsigned long long)pxx);
  red_add(q + 6, (unsigned long long)pxy);
  red_add(q + 7, (unsigned long long)pxz);
  red_add(q + 8, (unsigned long long)pyy);
  red_add(q + 9, (unsigned long long)pyz);
  red_add(q + 10, (unsigned long long)pzz);
}

// ---- staging of a warp tile.  The warp's scratch (pass_wslots(K) 16-byte slots = 16 bytes per point) holds the three
// coordinate planes of the tile (12 bytes per point, filled by the TMA engine: three bulk copies issued by one lane,
// completion on the warp's mbarrier) and a 4-byte list entry per point.
// src: first point of the tile in the x plane of pog (16-byte aligned: Chunk::pog), ld: plane stride, cnt: points.
template <int K>
__device__ __forceinline__ void pass2_request_tile(int4* went, const float* src, size_t ld, int cnt, unsigned long long* mbar) {
  float* tx = reinterpret_cast<float*>(went);
  const unsigned bytes = (unsigned)((cnt + 3) & ~3) * 4u;  // (the planes are padded to a multiple of 4 points)
  mbar_expect_tx(mbar, 3u * bytes);
  bulk_g2s(tx, src, bytes, mbar);
  bulk_g2s(tx + 32 * K, src + ld, bytes, mbar);
  bulk_g2s(tx + 64 * K, src + 2 * ld, bytes, mbar);
}

// One warp tile of 32*K consecutive stored points of scan 2.
//   went / mbar / mphase: the warp's scratch, its mbarrier and the parity of the barrier's next completion (the caller
//   keeps it across calls); requested: the caller has already issued pass2_request_tile for this tile (k_pass2 does so
//   before it stages the tables).
// RD: rows whose margin records a lane requests together in a delta iteration.  All K of them: a delta iteration is
// latency-bound (ncu r02g: issue slots 49 % busy, DRAM 28 %), what it needs is bytes in flight, not fewer instructions.
// anch: table of the voxels' anchors at the transform of this rebuild (k_pass2), or null: computed per run (loop kernels)
template <int K, int RD = K, bool ANCH = false>
__device__ __forceinline__ void pass2_warp_tile(const Chunk& ck, int4* went, unsigned long long* mbar, unsigned& mphase,
                                                bool requested, const float* tab, const CellRec* recs, const float* tr,
                                                const Pass2Mode& md, const float* pog, size_t ld, int n, int w0, uint2* mrec,
                                                int* violations, const float4* anch = nullptr) {
  static_assert(K <= 16, "list entries keep the point's index within the tile in 9 bits");
  const int lane = threadIdx.x & 31;
  if (w0 >= n) return;
  const int cnt = min(n - w0, 32 * K);
  const float4* tth = reinterpret_cast<const float4*>(tab);
  const float4* tph = tth + ck.nT + 2;
  const unsigned lt = (1u << lane) - 1u;
  unsigned long long* accp = md.accp;
  // shared addresses (bytes) of the warp's scratch: planes x | y | z of the tile (32*K floats each), then the list
  const uint32_t sb = opaque_u32(smem_u32(went));
  const uint32_t sbl = sb + 4u * lane;
  constexpr uint32_t PL = 128u * K;   // bytes per plane
  constexpr uint32_t LO = 3u * PL;    // offset of the list
  uint2* rp = mrec + w0;
  if (md.rebuild) {
    if (!requested) {
      __syncwarp();  // (every lane is done with the scratch of the previous tile)
      if (lane == 0) pass2_request_tile<K>(went, pog + w0, ld, cnt, mbar);
    }
    mbar_wait(mbar, mphase);
    mphase ^= 1u;
    // ---- phase A: every point, lane per point, coordinates from the staged tile.  ACTIVE points (their cell takes
    // part in the loop) are listed as {index in tile, in-box flag, cell}.
    int nact = 0;
#pragma unroll(K % 4 == 0 ? 4 : 2)
    for (int j = 0; j < K; j++) {
      const int li = j * 32 + lane;
      uint32_t cls = 0u;
      if (li < cnt) {
        const float x = lds_f32(sbl + 128u * j), y = lds_f32(sbl + 128u * j + PL), z = lds_f32(sbl + 128u * j + 2u * PL);
        float2 mg;
        point_eval2_fast(ck, tth, tph, recs, tr, 0.f, 0.f, x, y, z, cls, mg);
        if (violations) {  // self-check: the filtered evaluation must give the class of the exact pipeline
          uint32_t cx;
          float2 mx;
          point_eval2(ck, tth, tph, recs, tr, 0.f, 0.f, x, y, z, cx, mx);
          if (cx != cls) atomicAdd(violations + 1, 1);
        }
        rp[li] = rec2_pack(mg.x, mg.y, cls);
      }
      const bool act = (cls & CLS_ACTIVE) != 0;
      const unsigned am = __ballot_sync(FULL, act);
      if (act) sts_u32(sb + LO + 4u * (nact + __popc(am & lt)), ((uint32_t)li << 23) | (cls & (CLS_CELL | CLS_IN)));
      nact += __popc(am);
    }
    __syncwarp();
    // ---- phase B: lane takes entries [lane*q, lane*q + q); q odd => conflict-free shared loads of the entries.  A run
    // of equal cell stays in the lane's registers: one flush (bin count + moments) per run.  In a rebuild iteration the
    // anchor transform of the voxel frames IS the current transform.
    const int q = ((nact + 31) >> 5) | 1;
    const int e0 = lane * q, e1 = min(nact, e0 + q);
    int cur = -1, nb = 0, nin = 0, sx = 0, sy = 0, sz = 0;
    long long pxx = 0, pxy = 0, pxz = 0, pyy = 0, pyz = 0, pzz = 0;
    float ax = 0.f, ay = 0.f, az = 0.f, sc = 0.f;
#pragma unroll 2
    for (int e = e0; e < e1; e++) {
      const unsigned v = lds_u32(sb + LO + 4u * e);
      const int c = (int)(v & CLS_CELL);
      if (c != cur) {
        flush_run2(accp, cur, nb, nin, sx, sy, sz, pxx, pxy, pxz, pyy, pyz, pzz);
        cur = c;
        nb = nin = sx = sy = sz = 0;
        pxx = pxy = pxz = pyy = pyz = pzz = 0;
        if (ANCH) {
          const float4 an = __ldg(anch + cur);
          ax = an.x; ay = an.y; az = an.z; sc = an.w;
        } else {
          vox_anchor2(recs, cur, tr, md.fs2, ax, ay, az, sc);
        }
      }
      nb++;
      if (v & CLS_IN) {
        const uint32_t pa = sb + 4u * (v >> 23);
        int fx, fy, fz;
        fix2(lds_f32(pa), lds_f32(pa + PL), lds_f32(pa + 2u * PL), ax, ay, az, sc, md.fl2, fx, fy, fz);
        nin++;
        sx += fx; sy += fy; sz += fz;
        pxx += (long long)fx * fx; pxy += (long long)fx * fy; pxz += (long long)fx * fz;
        pyy += (long long)fy * fy; pyz += (long long)fy * fz; pzz += (long long)fz * fz;
      }
    }
    flush_run2(accp, cur, nb, nin, sx, sy, sz, pxx, pxy, pxz, pyy, pyz, pzz);
    __syncwarp();
    return;
  }
  // ---- DELTA, phase T: which points have used up their margin?  (8 bytes per point, all rows requested up front)
  int nre = 0;
  constexpr int R = RD;  // rows whose margin records are requested together (latency shape: all of them)
  static_assert(K % RD == 0, "rows per load group must divide the tile");
#pragma unroll 1
  for (int j0 = 0; j0 < K; j0 += R) {
    uint2 rv[R];
#pragma unroll
    for (int g = 0; g < R; g++) {
      const int li = (j0 + g) * 32 + lane;
      rv[g] = make_uint2(0x7f000000u, 0u);  // (huge u, r_e = 0: stable)
      if (li < cnt) rv[g] = __ldcg(rp + li);  // (L2: written by another SM in the previous iteration)
    }
#pragma unroll
    for (int g = 0; g < R; g++) {
      const int li = (j0 + g) * 32 + lane;
      const bool stable = fmaf(rec2_re(rv[g]), md.SA, md.C) < rec2_u(rv[g]);
      // ICET_B200_FLAG_VERIFY_INCREMENTAL: evaluate the stable points as well and count those whose class changed
      const bool redo = li < cnt && (!stable || violations != nullptr);
      const unsigned rm = __ballot_sync(FULL, redo);
      if (redo) sts_u32(sb + LO + 4u * (nre + __popc(rm & lt)), stable ? ((uint32_t)li | 0x80000000u) : (uint32_t)li);
      nre += __popc(rm);
    }
  }
  if (nre == 0) return;
  // ---- phase E: full evaluation of the listed points, lane per point.  With more than one point in eight listed the
  // whole tile is staged (12 bytes per point, coalesced) instead of gathering three 32-byte sectors per listed point.
  const bool staged = nre * 8 > cnt;  // warp-uniform
  __syncwarp();
  if (staged) {
    if (lane == 0) pass2_request_tile<K>(went, pog + w0, ld, cnt, mbar);
    mbar_wait(mbar, mphase);
    mphase ^= 1u;
  }
  for (int e0 = 0; e0 < nre; e0 += 32) {
    const int e = e0 + lane;
    if (e < nre) {
      const uint32_t le = lds_u32(sb + LO + 4u * e);
      const bool was_stable = (le & 0x80000000u) != 0;
      const int li = (int)(le & 0x7fffffffu);
      float x, y, z;
      if (staged) {
        x = lds_f32(sb + 4u * li); y = lds_f32(sb + 4u * li + PL); z = lds_f32(sb + 4u * li + 2u * PL);
      } else {
        const float* pp = pog + w0 + li;
        x = __ldg(pp); y = __ldg(pp + ld); z = __ldg(pp + 2 * ld);
      }
      const uint32_t old = rec2_cls(__ldcg(rp + li));
      uint32_t cls;
      float2 mg;
      point_eval2_fast(ck, tth, tph, recs, tr, md.SA, md.SB, x, y, z, cls, mg);
      if (violations) {
        uint32_t cx;
        float2 mx;
        point_eval2(ck, tth, tph, recs, tr, md.SA, md.SB, x, y, z, cx, mx);
        if (cx != cls) atomicAdd(violations + 1, 1);
      }
      rp[li] = rec2_pack(mg.x, mg.y, cls);
      if (cls != old) {
        if (was_stable) atomicAdd(violations, 1);
        class_move(accp, recs, md, old, cls, x, y, z, 1);
      }
    }
  }
  __syncwarp();
}

__device__ __forceinline__ void load_pass2_mode(const Chunk& ck, int pair, Pass2Mode& md) {
  const PairMode* pm = ck.pm + pair;
  const int4 h = __ldcg(reinterpret_cast<const int4*>(pm));             // set, rebuild, SA, C
  md.rebuild = h.y != 0;
  md.set = h.x;
  const FixPt fp = fix_point(__ldg(&ck.desc[pair].n2));
  md.fs2 = fp.fs;
  md.fl2 = fp.fl;
  md.SA = __int_as_float(h.z);
  md.C = __int_as_float(h.w);
  md.SB = __ldcg(&pm->SB);
  md.trbp = pm->TRb;
  md.accp = ck.acc + ((size_t)h.x * ck.npairs + pair) * ck.ncell * NQ;
}

// (Measured and dropped, r02: several warp tiles per warp without double buffering (-4 %); requesting the margin records
// before the pair's mode is known (no gain, more registers).)
template <int K = PASS_K, int MINB = PASS_MINB>
__global__ void __launch_bounds__(PASS_THREADS, MINB) k_pass2(const Chunk ck) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long s_mbar[PASS_WARPS];
  int4* ent = reinterpret_cast<int4*>(smem_raw);
  float* tab = reinterpret_cast<float*>(smem_raw + PASS_WARPS * pass_wslots(K) * 16);
  const int pair = blockIdx.y;
  const int n = ck.n2c[pair];
  const int tile0 = blockIdx.x * pass_tile_points(K);
  if (tile0 >= n && blockIdx.x != 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int4* went = ent + warp * pass_wslots(K);
  const int w0 = tile0 + warp * 32 * K;
  const float* pog = ck.pog + (size_t)pair * 3 * ck.n2max;
  Pass2Mode md;
  load_pass2_mode(ck, pair, md);
  if (lane == 0) mbar_init(&s_mbar[warp], 1);
  __syncwarp();
  // a rebuild iteration reads every coordinate of the tile: request it before anything else
  const bool requested = md.rebuild && w0 < n;
  if (requested && lane == 0) pass2_request_tile<K>(went, pog + w0, (size_t)ck.n2max, min(n - w0, 32 * K), &s_mbar[warp]);
  // delta iterations only read the look-up tables for the few points they re-evaluate: straight from global memory
  const float* tabp = ck.binrec;
  if (md.rebuild) {
    const int ntab = pass_tab_floats(ck.nT, ck.nP);
    for (int k = threadIdx.x; k < ntab; k += PASS_THREADS) tab[k] = __ldg(ck.binrec + k);
    tabp = tab;
    __syncthreads();
  }
  float tr[12];
  {
    const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
    const float4 a = __ldcg(tp), b = __ldcg(tp + 1), c = __ldcg(tp + 2);
    tr[0] = a.x; tr[1] = a.y; tr[2] = a.z; tr[3] = a.w; tr[4] = b.x; tr[5] = b.y; tr[6] = b.z; tr[7] = b.w;
    tr[8] = c.x; tr[9] = c.y; tr[10] = c.z; tr[11] = c.w;
  }
  const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
  unsigned mphase = 0u;
  pass2_warp_tile<K, K, true>(ck, went, &s_mbar[warp], mphase, requested, tabp, recs, tr, md, pog, (size_t)ck.n2max, n, w0,
                              ck.mrec + (size_t)pair * ck.n2max,
                              (ck.flags & ICET_B200_FLAG_VERIFY_INCREMENTAL) ? &ck.res[pair].reserved[0] : nullptr,
                              ck.anch + (size_t)pair * ck.ncell);
  if (blockIdx.x == 0 && threadIdx.x == 0)
    pass2_dropped_returns(ck, reinterpret_cast<const float4*>(tabp), reinterpret_cast<const float4*>(tabp) + ck.nT + 2, recs,
                          tr, md, pair, ck.nz2[pair]);
}

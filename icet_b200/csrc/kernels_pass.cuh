// icet_b200/csrc/kernels_pass.cuh -- K3 / K5a (the pass over the points of a scan: cluster-box test, round trip,
// exact integer accumulation), K4 (scan-1 Gaussians, eigen-decomposition, ambiguity mask) and K0 (prepScan2).
// Included by icet_b200.cu inside its anonymous namespace.
#pragma once
// ----------------------------------------------------------------------------------------------
// K3 / K5a: one pass over the points of a scan: [transform,] spherical, cell, cluster-box test,
// sph->cart round trip, fixed-point accumulation of count / sum / sum of products per voxel.
//   SCAN2 = false: scan 1 (filterPointsInsideCluster + mean/cov of fitCells1, src/icet.cpp:155-162)
//   SCAN2 = true : scan 2, one Gauss-Newton iteration (src/icet.cpp:375-388 + fitCells2 :290-306)
// ----------------------------------------------------------------------------------------------
constexpr int PASS_THREADS = 256;
constexpr int PASS_WARPS = PASS_THREADS / 32;
constexpr int PASS_K = 12;       // rows of 32 points per warp tile (throughput shape): 48 KB of entry tiles per CTA,
constexpr int PASS_MINB = 4;     // so that four CTAs (32 warps, 64 registers per thread) fit an SM (r01g: +3 % over 16 / 3)
constexpr int PASS_K_SMALL = 4;  // same for small batches (latency shape: more, smaller tiles; 2 rows: the same
                                 // single-pair latency within 1 %, with twice the tasks)

__host__ __device__ constexpr int pass_wslots(int K) { return 32 * K; }  // 16-byte entry slots per warp tile
__host__ __device__ constexpr int pass_tile_points(int K) { return PASS_WARPS * 32 * K; }
// shared memory: entry tiles, then the angular tables: (nT + 2) + (nP + 2) records {T[k], T[k+1], lo[k], hi[k]}
// (+ the "sure" intervals of the filtered evaluation of the incremental loop: {lo, hi} per record)
__host__ __device__ inline int pass_tab_floats(int nT, int nP) { return 6 * (nT + nP + 4); }
__host__ __device__ inline int pass_smem_bytes(int nT, int nP, int K) {
  return PASS_WARPS * pass_wslots(K) * 16 + pass_tab_floats(nT, nP) * 4;
}

// Angular bin + box test in one table look-up.  rec[k] = {T[k], T[k+1], lo[k], hi[k]}:
//   T    exact thresholds of int((double(a)/period)*nb) (src/icet.cpp:545-546): bin k  <=>  T[k] <= a < T[k+1]
//   lo/hi the part of the bin that also passes the reference's inclusive fp32 box test against the bin edges
//        (src/icet.cpp:136-139, :632-633): lo = max(T[k], E[k]), hi = min(pred(T[k+1]), E[k+1]).
// Record nb (a == fp32(period), bin index nb % nb = 0) and record nb + 1 (everything beyond the period, i.e. the
// NaN sentinel 1000.0, whose bin `sbin` comes from the double formula on the host) have an empty [lo, hi].
// The fp32 estimate of k is off by at most one (checked against T).
__device__ __forceinline__ int bin_box(float a, const float4* rec, const icet::BinTable& bt, bool& inbox) {
  int k = __float2int_rz(fminf(a, bt.acap) * bt.scale);
  float4 e = rec[k];
  if (a < e.x || a >= e.y) {
    k += (a < e.x) ? -1 : 1;
    e = rec[k];
  }
  inbox = a >= e.z && a <= e.w;
  return k < bt.nb ? k : (k == bt.nb ? 0 : bt.sbin);
}

// Stage 1 of a point: [transform,] spherical coordinates, cell, gates.  active = the cell takes part
// (has a cluster / an active voxel); in = the point passes ICET::filterPointsInsideCluster (src/icet.cpp:632-634).
template <bool SCAN2>
__device__ __forceinline__ void point_stage1(const Chunk& ck, const float4* tth, const float4* tph, const CellRec* recs,
                                             const float* tr, float x, float y, float z, int& c, bool& active,
                                             bool& in, float& r, float& th, float& ph) {
  if (SCAN2) icet::transform(x, y, z, tr, tr + 3, x, y, z);
  icet::c2s(x, y, z, r, th, ph);
  bool bt_in, bp_in;
  const int bt = bin_box(th, tth, ck.bth, bt_in);
  const int bp = bin_box(ph, tph, ck.bph, bp_in);
  c = ck.nT * bp + bt;
  const float4 ra = __ldg(reinterpret_cast<const float4*>(recs + c));  // inner, outer, flags, scale
  active = (__float_as_uint(ra.z) & (SCAN2 ? F_ACTIVE2 : F_STAT1)) != 0;
  in = active && bt_in && bp_in && r >= ra.x && r <= ra.y;
}

// Stage 2 of an inside point: sph->cart round trip (statistics use round-tripped points, src/icet.cpp:159 / :303)
// and conversion to the voxel's fixed-point frame.
__device__ __forceinline__ void point_stage2(float r, float th, float ph, float refx, float refy, float refz, float sc,
                                             int lim, int& fx, int& fy, int& fz) {
  float cx, cy, cz;
  icet::s2c(r, th, ph, cx, cy, cz);
  fx = max(-lim, min(lim, __float2int_rn((cx - refx) * sc)));
  fy = max(-lim, min(lim, __float2int_rn((cy - refy) * sc)));
  fz = max(-lim, min(lim, __float2int_rn((cz - refz) * sc)));
}

// The dropped returns of scan 2: points2_OG == (0,0,0) for all of them, so they all land on t * R
// (src/icet.cpp:377-378; SURVEY.md A.12) -- evaluated once per iteration, weighted with their number.
__device__ inline void pass_dropped_returns(const Chunk& ck, const float4* tth, const float4* tph, const CellRec* recs,
                                            const float* tr, unsigned long long* accp, long long nz, int n2) {
  if (nz <= 0) return;
  int c;
  bool active, in;
  float r, th, ph;
  point_stage1<true>(ck, tth, tph, recs, tr, 0.0f, 0.0f, 0.0f, c, active, in, r, th, ph);
  if (!active) return;
  unsigned long long* q = accp + (size_t)c * NQ;
  red_add(q, (unsigned long long)nz);
  if (in) {
    const CellRec rc = recs[c];
    const FixPt fp = fix_point(n2);
    int ix, iy, iz;
    point_stage2(r, th, ph, rc.refx, rc.refy, rc.refz, rc.scale * fp.fs, fp.fl, ix, iy, iz);
    const long long fx = ix, fy = iy, fz = iz;
    red_add(q + 1, (unsigned long long)nz);
    red_add(q + 2, (unsigned long long)(nz * fx));
    red_add(q + 3, (unsigned long long)(nz * fy));
    red_add(q + 4, (unsigned long long)(nz * fz));
    red_add(q + 5, (unsigned long long)(nz * fx * fx));
    red_add(q + 6, (unsigned long long)(nz * fx * fy));
    red_add(q + 7, (unsigned long long)(nz * fx * fz));
    red_add(q + 8, (unsigned long long)(nz * fy * fy));
    red_add(q + 9, (unsigned long long)(nz * fy * fz));
    red_add(q + 10, (unsigned long long)(nz * fz * fz));
  }
}

// publishes the sums one lane collected over a run of consecutive inside points of one cell
__device__ __forceinline__ void flush_in_run(unsigned long long* accp, int cell, int nin, int sx, int sy, int sz,
                                             long long pxx, long long pxy, long long pxz, long long pyy, long long pyz,
                                             long long pzz) {
  if (cell < 0) return;
  unsigned long long* q = accp + (size_t)cell * NQ;
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

// One warp tile of 32*K consecutive points.
//  Phase A (lane per point, K rows, coalesced loads): stage 1 of every point.  Points of one cell that are
//    neighbours in the row form runs (LiDAR scans list points ring by ring: ~27 per run at 2048 azimuth steps /
//    75 bins); the head lane of a run adds the run length to the cell's bin count (one RED per run).  Inside points
//    are COMPACTED into the warp's shared-memory tile as {cell, r, theta, phi} -- typically 40 % of the points.
//  Phase B (lane per contiguous slice of the compacted list): stage 2 (the expensive round trip) only for inside
//    points and with all lanes busy; sums of a run of equal cell stay in registers, one flush per run.
// Only warp-level synchronisation inside.
//  G > 1 (latency shape): stage 1 of G rows is evaluated back to back before the warp-synchronous bookkeeping of
//    those rows, so that G independent dependency chains (each with a look-up of the cell record in the middle)
//    overlap inside one warp; the tile's latency, not its instruction count, is what a single pair waits for.
template <bool SCAN2, int K, int PF = 2, int G = 1>
__device__ __forceinline__ void pass_warp_tile(const Chunk& ck, int4* went /* the warp's pass_wslots(K) slots */,
                                               const float* tab, const CellRec* recs, const float* tr,
                                               const float* px_, size_t ld, int n, int w0, FixPt fp,
                                               unsigned long long* accp, unsigned long long* dbg_stamp = nullptr,
                                               const int32_t* s1_cell = nullptr, const float* s1_th = nullptr,
                                               const float* s1_ph = nullptr) {
  const int lane = threadIdx.x & 31;
  if (w0 >= n) return;
  const float4* tth = reinterpret_cast<const float4*>(tab);
  const float4* tph = tth + ck.nT + 2;
  const unsigned lt = (1u << lane) - 1u;
  int nin_tile = 0;
  if (!SCAN2) {
    // ---- phase A, scan 1: K1 already stored cell (+ box flag), r, theta, phi of every point; only the range test
    // against the cluster bounds (known since K2c) is left.  px_ = r1 of the pair; th / ph are read for inside points.
    // Rows in groups of R: every load of the group is requested before the first use, so that the only dependent
    // look-up left (the cell record) overlaps across the rows of the group.
    constexpr int R = (K % 4 == 0) ? 4 : ((K % 2 == 0) ? 2 : 1);
#pragma unroll 1
    for (int j0 = 0; j0 < K; j0 += R) {
      int cid[R];
      float rr[R], tt[R], pp[R];
#pragma unroll
      for (int g = 0; g < R; g++) {
        const int i = w0 + (j0 + g) * 32 + lane;
        cid[g] = -1; rr[g] = 0.f; tt[g] = 0.f; pp[g] = 0.f;
        if (i < n) { cid[g] = __ldg(s1_cell + i); rr[g] = __ldg(px_ + i); tt[g] = __ldg(s1_th + i); pp[g] = __ldg(s1_ph + i); }
      }
      float4 ra[R];
#pragma unroll
      for (int g = 0; g < R; g++) {
        ra[g] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cid[g] >= 0) ra[g] = __ldg(reinterpret_cast<const float4*>(recs + (cid[g] & ~CELL_INBOX)));  // inner, outer, flags, scale
      }
#pragma unroll
      for (int g = 0; g < R; g++) {
        const bool in = cid[g] >= 0 && (cid[g] & CELL_INBOX) && (__float_as_uint(ra[g].z) & F_STAT1) && rr[g] >= ra[g].x &&
                        rr[g] <= ra[g].y;
        const unsigned im = __ballot_sync(FULL, in);
        if (in)
          went[nin_tile + __popc(im & lt)] = make_int4(cid[g] & ~CELL_INBOX, __float_as_int(rr[g]), __float_as_int(tt[g]), __float_as_int(pp[g]));
        nin_tile += __popc(im);
      }
    }
  } else if (G > 1) {
    static_assert(G == 1 || K % G == 0, "rows per group must divide the tile");
    // ---- phase A, grouped: all coordinates of the group in flight, then G stage-1 chains, then the bookkeeping
#pragma unroll 1
    for (int j0 = 0; j0 < K; j0 += G) {
      float gx[G], gy[G], gz[G];
#pragma unroll
      for (int g = 0; g < G; g++) {
        const int i = w0 + (j0 + g) * 32 + lane;
        gx[g] = gy[g] = gz[g] = 0.f;
        if (i < n) { gx[g] = __ldg(px_ + i); gy[g] = __ldg(px_ + ld + i); gz[g] = __ldg(px_ + 2 * ld + i); }
      }
      int gc[G];
      bool gact[G], gin[G];
      float gr[G], gth[G], gph[G];
#pragma unroll
      for (int g = 0; g < G; g++) {
        const int i = w0 + (j0 + g) * 32 + lane;
        gc[g] = -1; gact[g] = false; gin[g] = false; gr[g] = 0.f; gth[g] = 0.f; gph[g] = 0.f;
        if (i < n) point_stage1<SCAN2>(ck, tth, tph, recs, tr, gx[g], gy[g], gz[g], gc[g], gact[g], gin[g], gr[g], gth[g], gph[g]);
      }
#pragma unroll
      for (int g = 0; g < G; g++) {
        const int key = gact[g] ? gc[g] : -1;
        const int prev = __shfl_up_sync(FULL, key, 1);
        const bool head = (lane == 0) || (key != prev);
        const unsigned hm = __ballot_sync(FULL, head);
        if (head && key >= 0) {
          const unsigned nh = (lane == 31) ? 0u : (hm >> (lane + 1));
          const int len = nh ? __ffs(nh) : 32 - lane;
          red_add(accp + (size_t)key * NQ, (unsigned long long)len);
        }
        const unsigned im = __ballot_sync(FULL, gin[g]);
        if (gin[g])
          went[nin_tile + __popc(im & lt)] = make_int4(gc[g], __float_as_int(gr[g]), __float_as_int(gth[g]), __float_as_int(gph[g]));
        nin_tile += __popc(im);
      }
    }
  } else {
  // ---- phase A (the coordinates of row j + PF are requested before row j is worked on)
  float bx[PF > 0 ? PF : 1], by[PF > 0 ? PF : 1], bz[PF > 0 ? PF : 1];
#pragma unroll
  for (int p = 0; p < PF; p++) {
    const int i = w0 + p * 32 + lane;
    bx[p] = by[p] = bz[p] = 0.f;
    if (p < K && i < n) { bx[p] = __ldg(px_ + i); by[p] = __ldg(px_ + ld + i); bz[p] = __ldg(px_ + 2 * ld + i); }
  }
#pragma unroll(PF > 0 ? (K % (2 * PF) == 0 ? 2 * PF : PF) : 2)
  for (int j = 0; j < K; j++) {
    const int i = w0 + j * 32 + lane;
    int c = -1;
    bool active = false, in = false;
    float r = 0.f, th = 0.f, ph = 0.f;
    float x = 0.f, y = 0.f, z = 0.f;
    if (PF > 0) {
      constexpr int PFm = PF > 0 ? PF : 1;
      x = bx[j % PFm]; y = by[j % PFm]; z = bz[j % PFm];
      const int ip = i + PF * 32;
      if (j + PF < K && ip < n) {
        bx[j % PFm] = __ldg(px_ + ip); by[j % PFm] = __ldg(px_ + ld + ip); bz[j % PFm] = __ldg(px_ + 2 * ld + ip);
      }
    } else if (i < n) {
      x = __ldg(px_ + i); y = __ldg(px_ + ld + i); z = __ldg(px_ + 2 * ld + i);
    }
    if (i < n) point_stage1<SCAN2>(ck, tth, tph, recs, tr, x, y, z, c, active, in, r, th, ph);
    // bin counts: one RED per run of equal (participating) cell in this row
    const int key = active ? c : -1;
    const int prev = __shfl_up_sync(FULL, key, 1);
    const bool head = (lane == 0) || (key != prev);
    const unsigned hm = __ballot_sync(FULL, head);
    if (head && key >= 0) {
      const unsigned nh = (lane == 31) ? 0u : (hm >> (lane + 1));
      const int len = nh ? __ffs(nh) : 32 - lane;
      red_add(accp + (size_t)key * NQ, (unsigned long long)len);
    }
    // compaction of the inside points
    const unsigned im = __ballot_sync(FULL, in);
    if (in) went[nin_tile + __popc(im & lt)] = make_int4(c, __float_as_int(r), __float_as_int(th), __float_as_int(ph));
    nin_tile += __popc(im);
  }
  }  // G == 1
  __syncwarp();
  if (dbg_stamp && lane == 0) {  // debug timeline: end of phase A
    unsigned long long t_;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
    *dbg_stamp = t_;
  }
  // ---- phase B: lane takes entries [lane*q, lane*q + q); q odd => conflict-free 16-byte shared loads
  const int q = ((nin_tile + 31) >> 5) | 1;
  const int e0 = lane * q, e1 = min(nin_tile, e0 + q);
  int cur = -1, nin = 0, sx = 0, sy = 0, sz = 0;
  long long pxx = 0, pxy = 0, pxz = 0, pyy = 0, pyz = 0, pzz = 0;
  float refx = 0.f, refy = 0.f, refz = 0.f, sc = 0.f;
  bool flushed = false;  // this lane has published a run already (its slice spans more than one cell)
#pragma unroll 2
  for (int e = e0; e < e1; e++) {
    const int4 v = went[e];
    if (v.x != cur) {
      if (cur >= 0) flushed = true;
      flush_in_run(accp, cur, nin, sx, sy, sz, pxx, pxy, pxz, pyy, pyz, pzz);
      cur = v.x;
      nin = sx = sy = sz = 0;
      pxx = pxy = pxz = pyy = pyz = pzz = 0;
      const float4* rp = reinterpret_cast<const float4*>(recs + cur);
      const float4 ra = __ldg(rp), rb = __ldg(rp + 1);
      sc = ra.w * fp.fs; refx = rb.x; refy = rb.y; refz = rb.z;
    }
    int fx, fy, fz;
    point_stage2(__int_as_float(v.y), __int_as_float(v.z), __int_as_float(v.w), refx, refy, refz, sc, fp.fl, fx, fy, fz);
    nin++;
    sx += fx; sy += fy; sz += fz;
    pxx += (long long)fx * fx; pxy += (long long)fx * fy; pxz += (long long)fx * fz;
    pyy += (long long)fy * fy; pyz += (long long)fy * fz; pzz += (long long)fz * fz;
  }
  if (!SCAN2) {
    // Scan 1 walks its points cell by cell: usually every lane of the tile has collected sums of ONE and the same cell.
    // Then the warp adds them up (shuffles) and publishes them once -- 11 REDs per tile instead of 11 per lane, which is
    // what keeps the few hot voxels of an accumulated map (10^5 points each) from serialising in the L2 atomic units.
    const int c0 = __shfl_sync(FULL, cur, 0);
    if (__all_sync(FULL, !flushed && (cur == c0 || cur < 0))) {
      long long v[9] = {(long long)sx, (long long)sy, (long long)sz, pxx, pxy, pxz, pyy, pyz, pzz};
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        nin += __shfl_xor_sync(FULL, nin, o);
#pragma unroll
        for (int k = 0; k < 9; k++) v[k] += __shfl_xor_sync(FULL, v[k], o);
      }
      if (lane == 0 && c0 >= 0 && nin > 0) {
        unsigned long long* q = accp + (size_t)c0 * NQ;
        red_add(q + 1, (unsigned long long)nin);
#pragma unroll
        for (int k = 0; k < 9; k++) red_add(q + 2 + k, (unsigned long long)v[k]);
      }
      __syncwarp();
      return;
    }
  }
  flush_in_run(accp, cur, nin, sx, sy, sz, pxx, pxy, pxz, pyy, pyz, pzz);
  __syncwarp();
}

template <bool SCAN2, int K = PASS_K, int MINB = PASS_MINB, int PF = 2, int G = 1>
__global__ void __launch_bounds__(PASS_THREADS, MINB) k_pass(const Chunk ck) {
  pdl_prologue();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int4* ent = reinterpret_cast<int4*>(smem_raw);
  float* tab = reinterpret_cast<float*>(smem_raw + PASS_WARPS * pass_wslots(K) * 16);
  const int pair = blockIdx.y;
  const PairDesc d = ck.desc[pair];
  // scan 1: the points grouped by cell (k_scatter) unless the chunk runs in shipped-order mode
  const bool grouped = !SCAN2 && ck.cellg != nullptr;
  const int n = SCAN2 ? ck.n2c[pair] : (grouped ? ck.n1g[pair] : d.n1);
  const int tile0 = blockIdx.x * pass_tile_points(K);
  if (tile0 >= n && !(SCAN2 && blockIdx.x == 0)) return;
  {
    const int ntab = pass_tab_floats(ck.nT, ck.nP);
    for (int k = threadIdx.x; k < ntab; k += PASS_THREADS) tab[k] = __ldg(ck.binrec + k);
  }
  float tr[12];
  if (SCAN2) {
    const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
    const float4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
    tr[0] = a.x; tr[1] = a.y; tr[2] = a.z; tr[3] = a.w; tr[4] = b.x; tr[5] = b.y; tr[6] = b.z; tr[7] = b.w;
    tr[8] = c.x; tr[9] = c.y; tr[10] = c.z; tr[11] = c.w;
  }
  const size_t o1 = (size_t)pair * ck.n1max;
  const float* px_ = SCAN2 ? ck.pog + (size_t)pair * 3 * ck.n2max : (grouped ? ck.rbuf : ck.r1) + o1;
  const size_t ld = SCAN2 ? (size_t)ck.n2max : (size_t)d.ld1;
  const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
  unsigned long long* accp = ck.acc + (size_t)pair * ck.ncell * NQ;
  __syncthreads();
  pass_warp_tile<SCAN2, K, PF, G>(ck, ent + (threadIdx.x >> 5) * pass_wslots(K), tab, recs, tr, px_, ld, n,
                           tile0 + (threadIdx.x >> 5) * 32 * K, fix_point(SCAN2 ? d.n2 : d.n1), accp, nullptr,
                           SCAN2 ? nullptr : (grouped ? ck.cellg : ck.cellid1) + o1,
                           SCAN2 ? nullptr : (grouped ? ck.thg : ck.th1) + o1, SCAN2 ? nullptr : (grouped ? ck.phg : ck.ph1) + o1);
  if (SCAN2 && blockIdx.x == 0 && threadIdx.x == 0)
    pass_dropped_returns(ck, reinterpret_cast<const float4*>(tab), reinterpret_cast<const float4*>(tab) + ck.nT + 2, recs, tr,
                         accp, ck.nz2[pair], d.n2);
}

// exact-sum -> mean / covariance (double) of a voxel
__device__ __forceinline__ void stats_from_acc(const unsigned long long* q, const CellRec& rc, float fs, double mean[3],
                                               double cov[6]) {
  const double nin = (double)(long long)q[1];
  const double inv = 1.0 / ((double)rc.scale * (double)fs);  // exact: both are powers of two
  const double in_ = 1.0 / nin;
  const double sx = (double)(long long)q[2], sy = (double)(long long)q[3], sz = (double)(long long)q[4];
  const double mx = sx * in_, my = sy * in_, mz = sz * in_;
  mean[0] = (double)rc.refx + mx * inv;
  mean[1] = (double)rc.refy + my * inv;
  mean[2] = (double)rc.refz + mz * inv;
  const double f = inv * inv / (nin - 1.0);
  cov[0] = ((double)(long long)q[5] - sx * mx) * f;
  cov[1] = ((double)(long long)q[6] - sx * my) * f;
  cov[2] = ((double)(long long)q[7] - sx * mz) * f;
  cov[3] = ((double)(long long)q[8] - sy * my) * f;
  cov[4] = ((double)(long long)q[9] - sy * mz) * f;
  cov[5] = ((double)(long long)q[10] - sz * mz) * f;
}

// ----------------------------------------------------------------------------------------------
// K4: per voxel of scan 1: mean / covariance, 3x3 eigen-decomposition, sigma points, L mask
// (fitCells1 src/icet.cpp:158-232, testSigmaPoints :654-696); constants for the iteration loop.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void vox_anchor2_rec(float4 ra, float4 rb, const float* trb, float fs2, float& ax, float& ay, float& az,
                                                float& sc);  // kernels_pass2.cuh
__global__ void __launch_bounds__(128) k_fit1(const Chunk ck) {
  pdl_prologue();
  const int pair = blockIdx.y;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= ck.ncell) return;
  const size_t ci = (size_t)pair * ck.ncell + cell;
  CellRec rc = ck.rec[ci];
  unsigned long long* q = ck.acc + ci * NQ;
  const PairDesc d = ck.desc[pair];
  bool has = false;
  if (rc.flags & F_STAT1) {
    const long long nin = (long long)q[1];
    if (ck.dump_on) ck.dump.nin1[cell] = (int)nin;
    // `filteredPoints.size() >= n` with size() = 3 * rows  (src/icet.cpp:158)
    if (3 * nin >= ck.n && nin >= 2) {
      has = true;
      double mean[3], cov[6];
      stats_from_acc(q, rc, fix_point(d.n1).fs, mean, cov);
      Vox1 v;
      for (int k = 0; k < 3; k++) v.mu[k] = mean[k];
      const double d1 = (double)(rc.cnt1 - 1);  // `indices1.size() - 1` (:315)
      for (int k = 0; k < 6; k++) v.S1n[k] = cov[k] / d1;
      float A[9] = {(float)cov[0], (float)cov[1], (float)cov[2], (float)cov[1], (float)cov[3],
                    (float)cov[4], (float)cov[2], (float)cov[4], (float)cov[5]};
      float ev[3], V[9];
      icet::eig3f(A, ev, V);
      // sigma points mu +- 2 sqrt(ev_k) * V.row(k)   (:187-202), tested in order 0+,0-,1+,1-,2+,2-
      const float mu[3] = {(float)mean[0], (float)mean[1], (float)mean[2]};
      const int bt = cell % ck.nT, bp = cell / ck.nT;
      const float azl = ck.azE[bt], azh = ck.azE[bt + 1], ell = ck.elE[bp], elh = ck.elE[bp + 1];
      bool inside[6] = {false, false, false, false, false, false};
      float sp[6][3];
      for (int j = 0; j < 6; j++) {
        const int k = j >> 1;
        const float al = 2.0f * sqrtf(ev[k]);
        for (int c = 0; c < 3; c++) {
          float rot = al * V[3 * k + c];
          sp[j][c] = (j & 1) ? mu[c] - rot : mu[c] + rot;
        }
      }
      for (int j = 0; j < 6; j++) {
        const float* p = sp[j];
        float r, th, ph;
        icet::c2s(p[0], p[1], p[2], r, th, ph);
        if (th >= azl && th <= azh && ph >= ell && ph <= elh && r >= rc.inner && r <= rc.outer) inside[j] = true;
        if (r > rc.outer) break;  // the early break of testSigmaPoints (:683-685)
      }
      int lm = 0;
      for (int k = 0; k < 3; k++)
        if (inside[2 * k] || inside[2 * k + 1]) lm |= (1 << k);
      v.lmask = lm;
      v.pad = 0;
      for (int k = 0; k < 3; k++)
        for (int c = 0; c < 3; c++) v.LV[3 * k + c] = (lm >> k & 1) ? (double)V[3 * k + c] : 0.0;
      ck.vox[ci] = v;
      if (ck.dump_on) {
        for (int k = 0; k < 3; k++) { ck.dump.mu1[3 * cell + k] = (float)mean[k]; ck.dump.eval1[3 * cell + k] = ev[k]; }
        for (int k = 0; k < 9; k++) { ck.dump.sigma1[9 * cell + k] = A[k]; ck.dump.evec1[9 * cell + k] = V[k]; }
        for (int k = 0; k < 3; k++) ck.dump.lmask[3 * cell + k] = (lm >> k) & 1;
        // public member testPoints (src/icet.cpp:214-232): the sigma points of the axes found extended
        for (int j = 0; j < 6; j++)
          if (!((lm >> (j >> 1)) & 1))
            for (int c = 0; c < 3; c++) ck.dump.testpts[(size_t)(6 * cell + j) * 3 + c] = sp[j][c];
      }
    }
  }
  if (ck.dump_on) ck.dump.has1[cell] = has ? 1 : 0;
  // gates of fitCells2 that do not depend on scan 2: `indices1.size() > n && bounds[5] > 1`
  // (src/icet.cpp:290); a voxel without a scan-1 Gaussian is skipped (SURVEY.md H9).
  uint32_t fl = rc.flags & ~F_ACTIVE2;
  if (has && rc.cnt1 > ck.n && rc.outer > 1.0f) fl |= F_ACTIVE2;
  if (fl != rc.flags) ck.rec[ci].flags = fl;
  if (fl & F_ACTIVE2) {  // anchor of the voxel's scan-2 frame at the transform of the first rebuild (k_cell_scan: TRb = R(X0))
    float trb[12], ax, ay, az, sc;
    for (int k = 0; k < 12; k++) trb[k] = ck.pm[pair].TRb[k];
    vox_anchor2_rec(make_float4(rc.inner, rc.outer, __uint_as_float(fl), rc.scale),
                    make_float4(rc.refx, rc.refy, rc.refz, __int_as_float(rc.cnt1)), trb, fix_point(d.n2).fs, ax, ay, az, sc);
    ck.anch[ci] = make_float4(ax, ay, az, sc);
  }
  if (rc.flags & F_STAT1)
    for (int k = 0; k < NQ; k++) q[k] = 0ull;  // hand the accumulators to the scan-2 loop
  if (has) atomicAdd(&ck.res[pair].n_gauss1, 1);
}

// ----------------------------------------------------------------------------------------------
// Keyframe chunks (icet_b200_register_keyframe*): K1-K4 ran once, when the keyframe was created, and left its CellRec /
// Vox1 records (after k_fit1) in krec / kvox.  This kernel puts them into the slots of every pair of the chunk, anchors
// the scan-2 frames of the active voxels at R(X0) with the pair's fixed-point scale as k_fit1 does, and starts the pair like
// k_cell_scan.  After it the scan-2 kernels see the same state as after k_fit1.  Grid: (ceil(ncell / 128), P).
// ----------------------------------------------------------------------------------------------
// NG: int (the keyframe's Gaussian count, known on the host) or const int32_t* (a device word: the keyframe odometry node
// replaces its keyframe on the device, kernels_kfnode.cuh).
static_assert(sizeof(CellRec) == 32 && sizeof(Vox1) % 8 == 0, "k_kf_attach copies CellRec as 2 float4, Vox1 as 8-byte words");
__device__ __forceinline__ int kf_gaussians(int n) { return n; }
__device__ __forceinline__ int kf_gaussians(const int32_t* n) { return *n; }
template <class NG>
__global__ void __launch_bounds__(128) k_kf_attach(const Chunk ck, const CellRec* __restrict__ krec,
                                                   const Vox1* __restrict__ kvox, NG n_gauss1) {
  pdl_prologue();
  __shared__ float s_tr[12];
  const int pair = blockIdx.y;
  pair_start(ck, pair, kf_gaussians(n_gauss1), s_tr, blockIdx.x == 0);
  const int c0 = blockIdx.x * 128, nc = min(128, ck.ncell - c0);
  const size_t pc = (size_t)pair * ck.ncell + c0;
  {  // flat copies of the block's cells, consecutive threads on consecutive words
    const uint2* vs = reinterpret_cast<const uint2*>(kvox + c0);
    uint2* vd = reinterpret_cast<uint2*>(ck.vox + pc);
    for (int w = threadIdx.x; w < nc * (int)(sizeof(Vox1) / 8); w += 128) vd[w] = __ldg(vs + w);
    const float4* rs = reinterpret_cast<const float4*>(krec + c0);
    float4* rd = reinterpret_cast<float4*>(ck.rec + pc);
    for (int w = threadIdx.x; w < 2 * nc; w += 128) rd[w] = __ldg(rs + w);
  }
  __syncthreads();  // s_tr
  if ((int)threadIdx.x < nc) {
    const float4* rp = reinterpret_cast<const float4*>(krec + c0 + threadIdx.x);
    const float4 ra = __ldg(rp);
    if (__float_as_uint(ra.z) & F_ACTIVE2) {
      float ax, ay, az, sc;
      vox_anchor2_rec(ra, __ldg(rp + 1), s_tr, fix_point(ck.desc[pair].n2).fs, ax, ay, az, sc);
      ck.anch[pc + threadIdx.x] = make_float4(ax, ay, az, sc);
    }
  }
}

// ----------------------------------------------------------------------------------------------
// prepScan2 (src/icet.cpp:254-277): points2_OG = sphericalToCartesian(cartesianToSpherical(scan2)).
// (The radial re-ordering of scan 2 only changes the reference's summation order.)
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_prep2(const Chunk ck) {
  const int pair = blockIdx.y;
  const PairDesc d = ck.desc[pair];
  // scan 2 of this pair is scan 1 of the next one (sequences): k_scan1_bin of that pair has done this work already
  if (pair + 1 < ck.npairs) {
    const PairDesc nx = ck.desc[pair + 1];
    if (nx.s1 == d.s2 && nx.n1 == d.n2 && nx.ld1 == d.ld2) return;
  }
  // (few blocks per pair in big chunks, where most pairs return above: the grid stays small)
  for (int b0 = blockIdx.x * blockDim.x; b0 < d.n2; b0 += gridDim.x * blockDim.x) {  // block-uniform
    const int i = b0 + threadIdx.x;
    float x = 0.f, y = 0.f, z = 0.f;
    bool keep = false, zero = false;
    if (i < d.n2) {
      x = __ldg(d.s2 + i); y = __ldg(d.s2 + d.ld2 + i); z = __ldg(d.s2 + 2 * (size_t)d.ld2 + i);
      if ((__float_as_uint(x) | __float_as_uint(y) | __float_as_uint(z)) != 0u) {  // (+0,+0,+0) round-trips to itself, see k_scan1_bin
        float r, th, ph;
        icet::c2s(x, y, z, r, th, ph);
        icet::s2c(r, th, ph, x, y, z);
      }
      // Dropped returns: (0,0,0) stays (+0,+0,+0).  They are all the same point in every iteration, so they are
      // counted here and evaluated once per iteration by k_pass<true> instead of being stored.
      zero = (__float_as_uint(x) | __float_as_uint(y) | __float_as_uint(z)) == 0u;
      keep = !zero;
    }
    prep2_compact(ck, pair, x, y, z, keep, zero);
    __syncthreads();  // the shared scratch of prep2_compact is reused by the next round
  }
}


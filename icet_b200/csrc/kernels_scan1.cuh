// icet_b200/csrc/kernels_scan1.cuh -- K1, K2a, K2b, K2c: spherical coordinates and voxel indices of scan 1, cell
// bookkeeping, grouping of the ranges by cell, radial clustering (fitScan1 up to findCluster, src/icet.cpp:68-107,
// :557-607), and the shipped-row-order validation kernels.  Included by icet_b200.cu inside its anonymous namespace.
#pragma once
// ----------------------------------------------------------------------------------------------
// Fixed-point accumulators acc[cell][NQ] (64-bit integers, RED.64 to L2):
//   q[0] += points in the angular bin, q[1] += points inside the cluster box,
//   q[2..4] += sum d, q[5..10] += sum d d^T (xx xy xz yy yz zz),   d = round((p - ref) * scale)
// Exact integer arithmetic => the sums do not depend on the order or grouping of the additions.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void cell_of(const Chunk& ck, float th, float ph, int& bt, int& bp) {
  bt = icet::bin_lookup(th, ck.bth, 2 * M_PI);
  bp = icet::bin_lookup(ph, ck.bph, M_PI);
}
// ----------------------------------------------------------------------------------------------
// K1: scan 1 -> spherical, cell index, per-cell histogram.
// utils::cartesianToSpherical (src/utils.cpp:93-119) + sortSphericalCoordinates (src/icet.cpp:534-554)
// ----------------------------------------------------------------------------------------------
// Block-level compaction of points2_OG into pog[pair] (the order of points2_OG is irrelevant: all sums over it are
// exact integers); dropped returns are counted, not stored.  Called by every thread of a 256-thread block.
__device__ __forceinline__ void prep2_compact(const Chunk& ck, int pair, float x, float y, float z, bool keep, bool zero) {
  __shared__ int s_cnt[8], s_zero[8], s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned mk = __ballot_sync(FULL, keep), mz = __ballot_sync(FULL, zero);
  if (lane == 0) { s_cnt[warp] = __popc(mk); s_zero[warp] = __popc(mz); }
  __syncthreads();
  if (threadIdx.x == 0) {
    int tot = 0, totz = 0;
    for (int w = 0; w < 8; w++) { const int c = s_cnt[w]; s_cnt[w] = tot; tot += c; totz += s_zero[w]; }
    s_base = tot ? atomicAdd(&ck.n2c[pair], tot) : 0;
    if (totz) atomicAdd(&ck.nz2[pair], totz);
  }
  __syncthreads();
  if (keep) {
    const int o = s_base + s_cnt[warp] + __popc(mk & ((1u << lane) - 1));
    float* pg = ck.pog + (size_t)pair * 3 * ck.n2max;
    pg[o] = x;
    pg[ck.n2max + o] = y;
    pg[2 * (size_t)ck.n2max + o] = z;
  }
}

// Cells with up to this many non-zero ranges are clustered by one warp (k_cluster): WSORT_MAX with the bucket form; when
// the threshold is too small / too large for buckets, only what the small register sort holds -- bigger cells then take
// the CTA path (its own bucket windows or a block sort).  Chunk-uniform: k_cell_scan counts the others into nbig.
constexpr int WB_SORT_MAX = 128;  // cells up to this many ranges use the register sort (cheaper than buckets there)
__device__ __forceinline__ bool warp_buckets_ok(float thresh) { return thresh > 1e-3f && thresh < 1e30f; }
__device__ __forceinline__ int warp_cell_max(float thresh) { return warp_buckets_ok(thresh) ? WSORT_MAX : WB_SORT_MAX; }

constexpr int32_t CELL_INBOX = 0x40000000;  // cellid1 flag: the point passes the fp32 az / el box test of its own bin
__device__ __forceinline__ int bin_box(float a, const float4* rec, const icet::BinTable& bt, bool& inbox);

__global__ void __launch_bounds__(256) k_scan1_bin(const Chunk ck) {
  pdl_prologue();
  const int pair = blockIdx.y;
  const PairDesc d = ck.desc[pair];
  if ((int)(blockIdx.x * blockDim.x) >= d.n1) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int cell = -1;
  bool zero = false;
  // Consecutive pairs of a sequence share a scan: scan 1 of this pair is scan 2 of the previous one.  Its spherical
  // coordinates are computed here anyway, so prepScan2 of the previous pair (round trip + compaction, see k_prep2)
  // is done in the same pass and k_prep2 skips that pair.
  bool prev_shares = false;
  if (pair > 0) {
    const PairDesc pv = ck.desc[pair - 1];
    prev_shares = pv.s2 == d.s1 && pv.n2 == d.n1 && pv.ld2 == d.ld1;
  }
  float px = 0.f, py = 0.f, pz = 0.f;
  bool pkeep = false, pzero = false;
  if (i < d.n1) {
    float x = __ldg(d.s1 + i), y = __ldg(d.s1 + d.ld1 + i), z = __ldg(d.s1 + 2 * (size_t)d.ld1 + i);
    float r, th, ph;
    // Dropped returns are stored as (+0,+0,+0): a tenth of a scan, spread over every warp, and each of them takes the
    // slow paths of the IEEE square root / division and the library atan2f / acosf.  Their result is known:
    // cartesianToSpherical gives r = sqrt(0) = 0, theta = atan2f(+0,+0) = +0, phi = acosf(0/0) = NaN -> 1000.0
    // (src/utils.cpp:98-116), and sphericalToCartesian of that is (+0,+0,+0) again (sin 1000 > 0, cos 1000 > 0).
    const bool origin = (__float_as_uint(x) | __float_as_uint(y) | __float_as_uint(z)) == 0u;
    if (origin) {
      r = 0.0f; th = 0.0f; ph = 1000.0f;
    } else {
      icet::c2s(x, y, z, r, th, ph);
    }
    if (prev_shares) {
      if (!origin) icet::s2c(r, th, ph, px, py, pz);
      pzero = (__float_as_uint(px) | __float_as_uint(py) | __float_as_uint(pz)) == 0u;
      pkeep = !pzero;
    }
    // bin and box test in one look-up (same records as the pass kernels, read through L1 here)
    const float4* tth = reinterpret_cast<const float4*>(ck.binrec);
    const float4* tph = tth + ck.nT + 2;
    bool bt_in, bp_in;
    const int bt = bin_box(th, tth, ck.bth, bt_in);
    const int bp = bin_box(ph, tph, ck.bph, bp_in);
    cell = ck.nT * bp + bt;
    zero = (r == 0.0f);
    const size_t o = (size_t)pair * ck.n1max + i;
    ck.cellid1[o] = cell | ((bt_in && bp_in) ? CELL_INBOX : 0);
    ck.r1[o] = r;
    ck.th1[o] = th;
    ck.ph1[o] = ph;
  }
  // warp-aggregated histogram.  Every lane takes part in the match and in the vote (rows beyond the cloud form their
  // own group with cell -1): collectives under a divergent mask cost a WARPSYNC round per group.
  const int lane = threadIdx.x & 31;
  {
    const unsigned m = __match_any_sync(FULL, cell);
    const unsigned mz = __ballot_sync(FULL, zero) & m;
    if (cell >= 0 && lane == __ffs(m) - 1) {
      atomicAdd(&ck.cnt1[(size_t)pair * ck.ncell + cell], __popc(m));
      if (mz) atomicAdd(&ck.cntz[(size_t)pair * ck.ncell + cell], __popc(mz));
    }
  }
  if (prev_shares) prep2_compact(ck, pair - 1, px, py, pz, pkeep, pzero);  // block-uniform
}

// Per-pair state at the start of a registration: X = X0, its transform TR (= TRprev), the get_H derivatives J, the control
// block of the incremental loop and the result record (n_gauss1 = `n_gauss1`).  Called by every thread of a block of at
// least 64 threads: warp 1 owns the result record, thread 0 the transform.  write = false: nothing global is written.
// tr (or null): thread 0 also stores the transform there (the keyframe path anchors its voxels at it, k_kf_attach).
__device__ __forceinline__ void pair_start(const Chunk& ck, int pair, int n_gauss1, float* tr, bool write) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 1 && write) {
    icet_b200_result* R = ck.res + pair;
    // chained pairs (ICET_B200_FLAG_CHAIN_X0, odometry.cpp:82): x0 holds ONE seed, that of pair 0; the later pairs are
    // seeded by the last solve of their predecessor (chain_seed_next).  Without iterations the seed is the answer.
    const bool chain = (ck.flags & ICET_B200_FLAG_CHAIN_X0) != 0;
    const bool seeded = ck.x0 && (!chain || pair == 0 || ck.runlen == 0);
    if (lane < 6) {
      const float x = seeded ? ck.x0[(chain ? 0 : pair * 6) + lane] : 0.f;
      ck.X[pair * 6 + lane] = x;
      R->X[lane] = x;
      R->pred_stds[lane] = 0.f;
    }
    for (int k = lane; k < 36; k += 32) R->Q[k] = 0.f;
    if (lane == 6) { R->status = 0; R->n_gauss1 = n_gauss1; R->n_used = 0; R->n_dropped = 0; R->cond = 0.f; }
    if (lane >= 7 && lane < 10) R->reserved[lane - 7] = 0;
  }
  if (threadIdx.x == 0) {
    const bool chain = (ck.flags & ICET_B200_FLAG_CHAIN_X0) != 0;
    const bool seeded = ck.x0 && (!chain || pair == 0 || ck.runlen == 0);
    float X[6];
    for (int k = 0; k < 6; k++) X[k] = seeded ? ck.x0[(chain ? 0 : pair * 6) + k] : 0.f;
    float* TR = write ? ck.TR + (size_t)pair * 12 : tr;
    TR[0] = X[0]; TR[1] = X[1]; TR[2] = X[2];
    icet::rotR(X[3], X[4], X[5], TR + 3);
    if (write) {
      icet::getH_J(X[3], X[4], X[5], ck.J + (size_t)pair * 27);
      for (int k = 0; k < 12; k++) ck.TRprev[(size_t)pair * 12 + k] = TR[k];
      // incremental scan-2 loop: the first iteration builds the moments from zero in set 0, anchored at this transform
      PairMode* pm = ck.pm + pair;
      pm->set = 0; pm->rebuild = 1; pm->SA = 0.f; pm->C = 0.f; pm->SB = 0.f; pm->zcls = (int)CLS_NONE;
      for (int k = 0; k < 12; k++) pm->TRb[k] = TR[k];
      if (tr)
        for (int k = 0; k < 12; k++) tr[k] = TR[k];
    }
  }
}

// ----------------------------------------------------------------------------------------------
// K2a: per pair: exclusive scan of the non-zero counts (offsets into rbuf), work list of cells with
// cnt1 >= n (src/icet.cpp:115), default cell records (the else-branch :243-251: inner = outer = 0).
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cell_scan(const Chunk ck) {
  pdl_prologue();
  const int pair = blockIdx.x;
  __shared__ int s_ws[8], s_ww[8];
  const int per = (ck.ncell + 255) / 256;
  const int c0 = threadIdx.x * per, c1 = min(ck.ncell, c0 + per);
  const int32_t* cnt1 = ck.cnt1 + (size_t)pair * ck.ncell;
  const int32_t* cntz = ck.cntz + (size_t)pair * ck.ncell;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int s = 0, w = 0, big = 0;
  for (int c = c0; c < c1; c++) {
    const int m = cnt1[c] - cntz[c];
    s += m;
    w += (cnt1[c] >= ck.n) ? 1 : 0;
    big += (cnt1[c] >= ck.n && m > warp_cell_max(ck.thresh)) ? 1 : 0;
  }
  {
    const int anybig = __syncthreads_count(big > 0);  // (number of threads that own a big cell: only zero / non-zero matters)
    if (threadIdx.x == 0) ck.nbig[pair] = anybig;
  }
  // exclusive block scan of (s, w): inclusive warp scans, then the warp totals
  int is = s, iw = w;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int ts = __shfl_up_sync(FULL, is, o), tw = __shfl_up_sync(FULL, iw, o);
    if (lane >= o) { is += ts; iw += tw; }
  }
  if (lane == 31) { s_ws[warp] = is; s_ww[warp] = iw; }
  pair_start(ck, pair, 0, nullptr, true);  // meanwhile: the per-pair state
  __syncthreads();
  int a = is - s, b = iw - w;
  for (int q = 0; q < warp; q++) { a += s_ws[q]; b += s_ww[q]; }
  if (threadIdx.x == 255) {
    ck.nwork[pair] = b + w;
    ck.n1g[pair] = a + s;  // every non-zero range of the pair
  }
  for (int c = c0; c < c1; c++) {
    ck.off[(size_t)pair * ck.ncell + c] = a;
    a += cnt1[c] - cntz[c];
    if (cnt1[c] >= ck.n) ck.work[(size_t)pair * ck.ncell + (b++)] = c;
    if (ck.hbkt && cnt1[c] >= ck.n && cnt1[c] - cntz[c] > HUGE_MIN) {
      const int slot = atomicAdd(ck.nhuge, 1);
      if (slot < HUGE_SLOTS) {
        ck.hslot[(size_t)pair * ck.ncell + c] = slot + 1;
        ck.hpair[slot] = pair;
        ck.hcell[slot] = c;
      }
    }
    CellRec rc;
    rc.inner = 0.f; rc.outer = 0.f; rc.refx = rc.refy = rc.refz = 0.f; rc.scale = 0.f;
    rc.flags = 0; rc.cnt1 = cnt1[c];
    ck.rec[(size_t)pair * ck.ncell + c] = rc;
  }
}

// K2b: group the non-zero ranges by cell
__global__ void __launch_bounds__(256) k_scatter(const Chunk ck) {
  pdl_prologue();
  const int pair = blockIdx.y;
  const PairDesc d = ck.desc[pair];
  if ((int)(blockIdx.x * blockDim.x) >= d.n1) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int cell = -1, cid = 0;
  float r = 0.f, th = 0.f, ph = 0.f;
  if (i < d.n1) {
    const size_t o = (size_t)pair * ck.n1max + i;
    r = ck.r1[o];
    cid = ck.cellid1[o];
    if (ck.cellg) { th = ck.th1[o]; ph = ck.ph1[o]; }
    if (r != 0.0f) cell = cid & ~CELL_INBOX;
  }
  const int lane = threadIdx.x & 31;
  // (every lane takes part in the match and the shuffle; zero ranges / rows beyond the cloud: group of cell -1)
  const unsigned m = __match_any_sync(FULL, cell);
  const int leader = __ffs(m) - 1;
  int base = 0, off = 0;
  if (cell >= 0) off = __ldg(&ck.off[(size_t)pair * ck.ncell + cell]);  // (requested beside the atomic)
  if (cell >= 0 && lane == leader) base = atomicAdd(&ck.cursor[(size_t)pair * ck.ncell + cell], __popc(m));
  base = __shfl_sync(FULL, base, leader);
  if (cell >= 0) {
    const int rank = __popc(m & ((1u << lane) - 1));
    const size_t g = (size_t)pair * ck.n1max + off + base + rank;
    ck.rbuf[g] = r;
    if (ck.cellg) { ck.cellg[g] = cid; ck.thg[g] = th; ck.phg[g] = ph; }
  }
}

// ----------------------------------------------------------------------------------------------
// K2c: per cell with cnt1 >= n: sort the ranges ascending (what src/icet.cpp:71-83 intends) and run
// ICET::findCluster (src/icet.cpp:557-607) on them; write the cell record.
// ----------------------------------------------------------------------------------------------
// Bitonic-style network with all comparators ascending ("mirror" first step): works for any m,
// indices >= m behave as +inf and are never touched.
template <class Ptr>
__device__ inline void block_sort_asc(Ptr a, int m) {
  int p2 = 1;
  while (p2 < m) p2 <<= 1;
  for (int k = 2; k <= p2; k <<= 1) {
    // mirror step: i with partner i ^ (k-1)
    for (int t = threadIdx.x; t < p2 / 2; t += blockDim.x) {
      int blk = t / (k / 2), o = t % (k / 2);
      int i = blk * k + o, j = blk * k + (k - 1 - o);
      if (j < m) {
        auto x = a[i];
        auto y = a[j];
        if (y < x) { a[i] = y; a[j] = x; }
      }
    }
    __syncthreads();
    for (int j2 = k / 4; j2 >= 1; j2 >>= 1) {
      for (int t = threadIdx.x; t < p2 / 2; t += blockDim.x) {
        int i = (t / j2) * (2 * j2) + (t % j2), j = i + j2;
        if (j < m) {
          auto x = a[i];
          auto y = a[j];
          if (y < x) { a[i] = y; a[j] = x; }
        }
      }
      __syncthreads();
    }
  }
}

// findCluster over the virtual sequence seq = [0 x nz, a[0..m)] (ascending); executed by warp 0,
// every lane computes the same result.  A "break" at position i means seq[i] does not extend the
// current run (reference :572); the run before a break is returned if it has >= n points (:577-582,
// no zero check), the run that reaches the end of the data goes through the zero check (:592-603).
template <class Ptr>
__device__ inline void find_cluster_warp(Ptr a, int m, int nz, int n, float thresh, float buff, float& inner,
                                         float& outer) {
  const int lane = threadIdx.x & 31;
  const int total = nz + m;
  auto seq = [&](int i) -> float { return i < nz ? 0.0f : a[i - nz]; };
  int start = 0;  // first element of the current run; the nz leading zeros never break (thresh >= 0)
  bool found = false;
  float fi = 0.f, fo = 0.f;
  for (int base = nz; base < total && !found; base += 32) {
    const int i = base + lane;
    bool brk = false;
    if (i < total && i > 0) brk = !(fabsf(seq(i - 1) - seq(i)) <= thresh);
    unsigned mask = __ballot_sync(FULL, brk);
    while (mask && !found) {
      const int pos = base + __ffs(mask) - 1;
      mask &= mask - 1;
      if (pos - start >= n) {
        fi = seq(start) - buff;
        fo = seq(pos - 1) + buff;
        found = true;
      } else {
        start = pos;
      }
    }
  }
  if (!found && total > 0 && total - start >= n) {
    if (seq(start) != 0.0f) {
      fi = seq(start) - buff;
      fo = seq(total - 1) + buff;
    }
  }
  inner = fi;
  outer = fo;
}

// writes the cell record of a clustered cell (clusterBounds columns 4,5 + the voxel's fixed-point frame)
__device__ inline void write_cluster_rec(const Chunk& ck, int pair, int cell, int cnt, float inner, float outer) {
  const int bt = cell % ck.nT, bp = cell / ck.nT;
  CellRec rc;
  rc.inner = inner;
  rc.outer = outer;
  rc.cnt1 = cnt;
  rc.flags = ((double)outer > 0.1) ? F_STAT1 : 0u;  // `outerDistance > 0.1` src/icet.cpp:158
  // fixed-point frame of the voxel: reference point = centre of the spherical box, scale from
  // a bound on the box diameter
  const float azl = ck.azE[bt], azh = ck.azE[bt + 1], ell = ck.elE[bp], elh = ck.elE[bp + 1];
  const float rm = 0.5f * (inner + outer), tm = 0.5f * (azl + azh), pm = 0.5f * (ell + elh);
  icet::s2c(rm, tm, pm, rc.refx, rc.refy, rc.refz);
  float D = (outer - inner) + fabsf(outer) * ((azh - azl) + (elh - ell));
  int e;
  frexpf(fmaxf(D, 1e-20f), &e);          // D < 2^e
  rc.scale = ldexpf(1.0f, FPB - e - 1);  // |d| <= D  =>  |d*scale| < 2^(FPB-1)
  ck.rec[(size_t)pair * ck.ncell + cell] = rc;
}

// Bitonic sort of 32*EPL floats held EPL per lane; element index = lane*EPL + j.  Compare-exchange distances
// below EPL stay inside a lane (registers), larger ones are one shuffle per element.  Fully unrolled.
template <int EPL>
__device__ __forceinline__ void warp_sort_regs(float (&v)[EPL]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 2; k <= 32 * EPL; k <<= 1) {
#pragma unroll
    for (int d = k >> 1; d > 0; d >>= 1) {
      if (d >= EPL) {
        const int ld = d / EPL;                                             // partner lane distance
        const bool asc = (k >= 32 * EPL) || ((lane & (k / EPL)) == 0);
        const bool keep_min = (((lane & ld) == 0) == asc);
#pragma unroll
        for (int j = 0; j < EPL; j++) {
          const float o = __shfl_xor_sync(FULL, v[j], ld);
          v[j] = keep_min ? fminf(v[j], o) : fmaxf(v[j], o);
        }
      } else {
#pragma unroll
        for (int j = 0; j < EPL; j++) {
          if ((j & d) == 0) {
            // direction bit k of the element index: in the register index for k < EPL, in the lane above
            const bool asc = (k >= 32 * EPL) || (k < EPL ? ((j & k) == 0) : ((lane & (k / EPL)) == 0));
            const float lo = fminf(v[j], v[j ^ d]), hi = fmaxf(v[j], v[j ^ d]);
            v[j] = asc ? lo : hi;
            v[j ^ d] = asc ? hi : lo;
          }
        }
      }
    }
  }
}

// loads the m ranges of a cell (any order), sorts them in registers and leaves them ascending in the warp's
// shared-memory row (index i stored at i + i/32: conflict-free for the blocked write and for consecutive reads)
template <int EPL>
__device__ __forceinline__ void warp_sort_cell(const float* __restrict__ g, int m, float* srow) {
  const int lane = threadIdx.x & 31;
  float v[EPL];
#pragma unroll
  for (int j = 0; j < EPL; j++) {
    const int i = j * 32 + lane;  // coalesced; which register an unsorted value lands in is irrelevant
    v[j] = i < m ? __ldg(g + i) : INFINITY;
  }
  warp_sort_regs<EPL>(v);
#pragma unroll
  for (int j = 0; j < EPL; j++) {
    const int i = lane * EPL + j;
    srow[i + (i >> 5)] = v[j];
  }
  __syncwarp();
}

struct PaddedRow {  // view of a shared-memory row written by warp_sort_cell
  const float* p;
  __device__ __forceinline__ float operator[](int i) const { return p[i + (i >> 5)]; }
};

// ---- findCluster of one cell by one warp WITHOUT a sort (cells with more than WB_SORT_MAX ranges).  As in the CTA and
// multi-CTA paths below, ranges are dropped into buckets half a threshold wide (count / min / max per bucket in shared
// memory; two ranges of one bucket are closer than the threshold by construction) and the non-empty buckets are walked
// in ascending order -- here a window of WB buckets at a time, starting at the cell's smallest range.  The walk is
// data-parallel: the non-empty buckets of the window are compacted (ballot) into a list, and 32 list entries at a
// time, one per lane, find their breaks (neighbour's max by shuffle), the elements in front of them (warp scan), the
// break that opened their run (bit tricks on the ballot of the breaks) and whether their run holds >= n elements; the
// first such break wins.  Bit-identical bounds to the sorted form (tests); ~550 warp instructions for a 260-range cell
// against ~2500 for the 512-element bitonic network it replaces.
constexpr int WB = 512;           // buckets per window (25.6 m at the default threshold of 0.1 m)

// Exact but slow form for a cell whose ranges the buckets cannot index (a range that is inf or beyond 10^7 m: garbage
// input): the distinct ranges in ascending order by repeated selection (one pass over the cell per distinct value),
// fed to the sequential walk.  NaN never reaches a cell list (cartesianToSpherical replaces it, src/utils.cpp:116).
__device__ inline void find_cluster_select_warp(const float* __restrict__ g, int m, int nz, int n, float thresh, float buff,
                                                float& inner, float& outer) {
  const int lane = threadIdx.x & 31;
  int idx = nz, start = 0;
  float start_val = 0.f, prev_val = 0.f;
  int curb = -1;  // bit pattern of the last value taken (ranges are > 0)
  inner = 0.f;
  outer = 0.f;
  while (idx < nz + m) {
    int nb = 0x7fffffff;
    for (int i = lane; i < m; i += 32) {
      const int b = __float_as_int(__ldg(g + i));
      if (b > curb) nb = min(nb, b);
    }
    nb = __reduce_min_sync(FULL, nb);
    if (nb == 0x7fffffff) break;  // (only NaN payloads left)
    int mult = 0;
    for (int i = lane; i < m; i += 32) mult += (__float_as_int(__ldg(g + i)) == nb) ? 1 : 0;
    mult = __reduce_add_sync(FULL, mult);
    const float v = __int_as_float(nb);
    if (idx > 0) {
      if (!(fabsf(prev_val - v) <= thresh)) {  // reference :572
        if (idx - start >= n) {                // :577-582
          inner = start_val - buff;
          outer = prev_val + buff;
          return;
        }
        start = idx;
        start_val = v;
      }
    } else {
      start_val = v;
    }
    // (equal values: |v - v| <= thresh unless v is inf, where the reference breaks between every two of them)
    if (mult > 1 && !(fabsf(v - v) <= thresh)) {
      for (int k = 1; k < mult; k++) {
        if (idx + k - start >= n) { inner = start_val - buff; outer = v + buff; return; }
        start = idx + k;
        start_val = v;
      }
    }
    idx += mult;
    prev_val = v;
    curb = nb;
  }
  if (nz + m - start >= n && start_val != 0.0f) {  // :592-603
    inner = start_val - buff;
    outer = prev_val + buff;
  }
}

// Returns false (warp-uniform) without a result when a range is not finite / absurdly large: the caller takes the
// selection form instead.
__device__ inline bool find_cluster_buckets_warp(const float* __restrict__ g, int m, int nz, int n, float thresh, float buff,
                                                 int* sb /* [3 * WB] */, float& inner, float& outer) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  int* b_cnt = sb;
  int* b_min = sb + WB;
  int* b_max = sb + 2 * WB;
  const float wdt = 0.5f * thresh, inv_w = 1.0f / wdt;
  // smallest / largest range of the cell (ranges are > 0: their bit patterns order like the values)
  int rmin_b = 0x7f800000, rmax_b = 0;
  for (int i = lane; i < m; i += 32) {
    const int b = __float_as_int(__ldg(g + i));
    rmin_b = min(rmin_b, b);
    rmax_b = max(rmax_b, b);
  }
  rmin_b = __reduce_min_sync(FULL, rmin_b);
  rmax_b = __reduce_max_sync(FULL, rmax_b);
  const float rmin = __int_as_float(rmin_b);
  if (!(__int_as_float(rmax_b) * inv_w < 1.0e9f)) return false;  // inf / NaN / bucket index beyond an int
  int lo = __float2int_rd(rmin * inv_w);  // first bucket of the current window
  // state of the walk (uniform across the lanes)
  int idx = nz;                                // elements in front of the next list entry (the zeros come first)
  int start = 0;                               // elements in front of the last break
  float start_val = nz > 0 ? 0.0f : rmin;      // first value of the current run
  float prev_val = 0.0f;                       // max of the last non-empty bucket (0.0: the zeros / nothing yet)
  bool any_before = nz > 0;
  int seen = 0;
  bool found = false;
  inner = 0.f;
  outer = 0.f;
  while (seen < m && !found) {
    {
      int4* c4 = reinterpret_cast<int4*>(b_cnt);
      int4* n4 = reinterpret_cast<int4*>(b_min);
      int4* x4 = reinterpret_cast<int4*>(b_max);
#pragma unroll
      for (int k = 0; k < WB / 128; k++) {
        c4[k * 32 + lane] = make_int4(0, 0, 0, 0);
        n4[k * 32 + lane] = make_int4(0x7f800000, 0x7f800000, 0x7f800000, 0x7f800000);
        x4[k * 32 + lane] = make_int4(0, 0, 0, 0);
      }
    }
    __syncwarp();
    int nxt = 0x7f800000;  // smallest range behind this window: the next window starts at its bucket
    for (int i = lane; i < m; i += 32) {
      const float r = __ldg(g + i);
      const int k = __float2int_rd(r * inv_w) - lo;
      if (k >= 0 && k < WB) {
        atomicAdd(&b_cnt[k], 1);
        atomicMin(&b_min[k], __float_as_int(r));
        atomicMax(&b_max[k], __float_as_int(r));
      } else if (k >= WB) {
        nxt = min(nxt, __float_as_int(r));
      }
    }
    nxt = __reduce_min_sync(FULL, nxt);
    __syncwarp();
    // compaction of the non-empty buckets, in place (an entry never moves behind the bucket it came from)
    int L = 0;
#pragma unroll 4
    for (int k0 = 0; k0 < WB; k0 += 32) {
      const int c = b_cnt[k0 + lane];
      const unsigned ne = __ballot_sync(FULL, c > 0);
      if (ne == 0u) continue;  // (most 32-bucket groups of a window are empty)
      int mn = 0, mx = 0;
      if (c > 0) { mn = b_min[k0 + lane]; mx = b_max[k0 + lane]; }
      __syncwarp();
      if (c > 0) {
        const int p = L + __popc(ne & lt);
        b_cnt[p] = c; b_min[p] = mn; b_max[p] = mx;
      }
      L += __popc(ne);
    }
    __syncwarp();
    // the walk, 32 list entries at a time
    for (int e0 = 0; e0 < L && !found; e0 += 32) {
      const int e = e0 + lane;
      const bool valid = e < L;
      const int c = valid ? b_cnt[e] : 0;
      const float mn = valid ? __int_as_float(b_min[e]) : 0.f, mx = valid ? __int_as_float(b_max[e]) : 0.f;
      float pmx = __shfl_up_sync(FULL, mx, 1);
      if (lane == 0) pmx = prev_val;
      const bool brk = valid && (lane > 0 || any_before) && !(fabsf(pmx - mn) <= thresh);  // reference :572
      int pc = c;  // inclusive prefix of the counts
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(FULL, pc, o);
        if (lane >= o) pc += u;
      }
      const int ie = idx + pc - c;  // elements in front of this entry
      const unsigned bm = __ballot_sync(FULL, brk);
      const unsigned below = bm & lt;
      const int pb = below ? 31 - __clz(below) : 0;  // the break that opened the run which ends in front of this entry
      const int pb_idx = __shfl_sync(FULL, ie, pb);
      const float pb_mn = __shfl_sync(FULL, mn, pb);
      const int run_start = below ? pb_idx : start;
      const float run_val = below ? pb_mn : start_val;
      const unsigned qm = __ballot_sync(FULL, brk && ie - run_start >= n);  // (:577-582, no zero check)
      if (qm) {
        const int w = __ffs(qm) - 1;
        inner = __shfl_sync(FULL, run_val, w) - buff;
        outer = __shfl_sync(FULL, pmx, w) + buff;
        found = true;
      } else {
        const int nv = min(32, L - e0);
        idx += __shfl_sync(FULL, pc, nv - 1);
        if (bm) {
          const int lb = 31 - __clz(bm);
          start = __shfl_sync(FULL, ie, lb);
          start_val = __shfl_sync(FULL, mn, lb);
        }
        prev_val = __shfl_sync(FULL, mx, nv - 1);
        any_before = true;
      }
    }
    if (!found) {
      seen = idx - nz;
      lo = __float2int_rd(__int_as_float(nxt) * inv_w);  // (only used while ranges are left: nxt is one of them)
    }
    __syncwarp();
  }
  if (!found && nz + m - start >= n && start_val != 0.0f) {  // end of the data (:592-603)
    inner = start_val - buff;
    outer = prev_val + buff;
  }
  return true;
}

// K2c: ONE WARP per cell with cnt1 >= n (a cell of a 64-ring scan holds ~260 ranges): register bitonic sort, then
// ICET::findCluster on the sorted row.  Cells with more than WSORT_MAX ranges take the CTA path at the end of the kernel.
__global__ void __launch_bounds__(CLUSTER_WARPS * 32) k_cluster(const Chunk ck) {
  pdl_prologue();
  const int pair = blockIdx.y;
  constexpr int ROW = WSORT_MAX + WSORT_MAX / 32;
  constexpr int SM_FLOATS = CLUSTER_WARPS * ROW > SORT_SMEM ? CLUSTER_WARPS * ROW : SORT_SMEM;
  // (the bucket tables of the warp path and the tables / sort buffer of the CTA path share the block's shared memory:
  // the CTA path starts after a block-wide barrier)
  constexpr int SM_WORDS = SM_FLOATS > CLUSTER_WARPS * 3 * WB ? SM_FLOATS : CLUSTER_WARPS * 3 * WB;
  __shared__ __align__(16) float s_all[SM_WORDS];
  int* s_bkt = reinterpret_cast<int*>(s_all);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int ROW4 = WB_SORT_MAX + WB_SORT_MAX / 32;  // row of the small register sort
  float* srow = s_all + warp * 3 * WB;                  // (inside the warp's own bucket region)
  const bool buckets_ok = warp_buckets_ok(ck.thresh);
  const int wmax = warp_cell_max(ck.thresh);
  const int nw = ck.nwork[pair];
  for (int w = blockIdx.x * CLUSTER_WARPS + warp; w < nw; w += gridDim.x * CLUSTER_WARPS) {
    const int cell = ck.work[(size_t)pair * ck.ncell + w];
    const int cnt = ck.cnt1[(size_t)pair * ck.ncell + cell];
    const int nz = ck.cntz[(size_t)pair * ck.ncell + cell];
    const int m = cnt - nz;
    if (m > wmax) continue;
    const float* g = ck.rbuf + (size_t)pair * ck.n1max + ck.off[(size_t)pair * ck.ncell + cell];
    float inner, outer;
    if (m <= WB_SORT_MAX) {
      static_assert(ROW4 <= 3 * WB, "sort row inside the bucket region");
      warp_sort_cell<4>(g, m, srow);
      find_cluster_warp(PaddedRow{srow}, m, nz, ck.n, ck.thresh, ck.buff, inner, outer);
    } else if (!(buckets_ok && find_cluster_buckets_warp(g, m, nz, ck.n, ck.thresh, ck.buff, s_bkt + warp * 3 * WB, inner, outer))) {
      find_cluster_select_warp(g, m, nz, ck.n, ck.thresh, ck.buff, inner, outer);
    }
    if (lane == 0) write_cluster_rec(ck, pair, cell, cnt, inner, outer);
    __syncwarp();
  }
  // The big cells (more than WSORT_MAX ranges: an accumulated map as scan 1; k_cell_scan counted them), the whole CTA per
  // cell.  findCluster only needs to know where consecutive SORTED ranges are more than `thresh` apart, so no sort:
  // the ranges are dropped into buckets half a threshold wide (count, min, max per bucket; ranges inside one bucket
  // are closer than the threshold by construction), windows of NBKT buckets are walked in ascending order, and the
  // walk stops at the first run that qualifies.  O(m) per window instead of the O(m log^2 m) of a bitonic network
  // (a 2 M-point map: 217 ms -> well under 1 ms).  Fallback for thresholds / ranges the buckets cannot cover: sort.
  if (ck.nbig[pair] == 0) return;  // block-uniform
  __syncthreads();
  constexpr int NBKT = (SM_FLOATS - 8) / 3;
  int* b_cnt = reinterpret_cast<int*>(s_all);
  int* b_min = b_cnt + NBKT;
  int* b_max = b_min + NBKT;
  int* s_ctl = b_max + NBKT;  // [0] points seen so far, [1] done, [2..3] result bits
  for (int w = blockIdx.x; w < nw; w += gridDim.x) {
    const int cell = ck.work[(size_t)pair * ck.ncell + w];
    const int cnt = ck.cnt1[(size_t)pair * ck.ncell + cell];
    const int nz = ck.cntz[(size_t)pair * ck.ncell + cell];
    const int m = cnt - nz;
    if (m <= wmax) continue;  // block-uniform
    if (ck.hbkt) {  // clustered by k_huge_* already (unless a range fell outside its table)
      const int hs = ck.hslot[(size_t)pair * ck.ncell + cell];
      if (hs > 0 && ck.hflag[hs - 1] == 0) continue;  // block-uniform
    }
    float* g = ck.rbuf + (size_t)pair * ck.n1max + ck.off[(size_t)pair * ck.ncell + cell];
    // largest range of the cell (the ranges are >= 0: their bit patterns order like the values)
    __syncthreads();
    if (threadIdx.x == 0) s_ctl[0] = 0;
    __syncthreads();
    {
      int mx = 0;
      for (int i0 = threadIdx.x; i0 < m; i0 += 8 * blockDim.x) {  // eight loads in flight per thread
        int v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const int i = i0 + u * blockDim.x;
          v[u] = i < m ? __float_as_int(g[i]) : 0;
        }
#pragma unroll
        for (int u = 0; u < 8; u++) mx = max(mx, v[u]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(FULL, mx, o));
      if (lane == 0) atomicMax(&s_ctl[0], mx);
    }
    __syncthreads();
    const float rmax = __int_as_float(s_ctl[0]);
    const float wdt = 0.5f * ck.thresh, inv_w = 1.0f / wdt;
    const bool buckets_ok = ck.thresh > 1e-6f && rmax * inv_w < 64.0f * NBKT;  // false for inf / NaN as well
    float inner = 0.f, outer = 0.f;
    if (buckets_ok) {
      // state of the walk (warp 0, uniform across its lanes)
      int idx = nz, start = 0;
      float start_val = 0.f, prev_val = 0.f;
      bool found = false;
      __syncthreads();
      if (threadIdx.x == 0) { s_ctl[0] = 0; s_ctl[1] = 0; }
      for (int win = 0;; win++) {
        for (int k = threadIdx.x; k < NBKT; k += blockDim.x) { b_cnt[k] = 0; b_min[k] = 0x7f800000; b_max[k] = 0; }
        __syncthreads();
        if (s_ctl[1]) break;  // found, or every range has been walked
        const int lo = win * NBKT;
        for (int i0 = threadIdx.x; i0 < m; i0 += 8 * blockDim.x) {  // eight loads in flight per thread
          float rv[8];
#pragma unroll
          for (int u = 0; u < 8; u++) {
            const int i = i0 + u * blockDim.x;
            rv[u] = i < m ? g[i] : -1.0f;
          }
#pragma unroll
          for (int u = 0; u < 8; u++) {
            const float r = rv[u];
            const int k = __float2int_rd(r * inv_w) - lo;
            if (r >= 0.0f && k >= 0 && k < NBKT) {
              atomicAdd(&b_cnt[k], 1);
              atomicMin(&b_min[k], __float_as_int(r));
              atomicMax(&b_max[k], __float_as_int(r));
            }
          }
        }
        __syncthreads();
        if (warp == 0) {
          int seen = 0;
          for (int base = 0; base < NBKT && !found; base += 32) {
            const int k = base + lane;
            const int c = k < NBKT ? b_cnt[k] : 0;
            unsigned mask = __ballot_sync(FULL, c > 0);
            while (mask && !found) {
              const int kb = base + __ffs(mask) - 1;
              mask &= mask - 1;
              const int bc = b_cnt[kb];
              const float mn = __int_as_float(b_min[kb]), mxv = __int_as_float(b_max[kb]);
              if (idx > 0) {
                if (!(fabsf(prev_val - mn) <= ck.thresh)) {  // a break in front of this bucket (reference :572)
                  if (idx - start >= ck.n) {
                    inner = start_val - ck.buff;             // :577-582, no zero check
                    outer = prev_val + ck.buff;
                    found = true;
                    break;
                  }
                  start = idx;
                  start_val = mn;
                }
              } else {
                start_val = mn;
              }
              idx += bc;
              seen += bc;
              prev_val = mxv;
            }
          }
          if (lane == 0) {
            s_ctl[0] += seen;
            if (found || s_ctl[0] >= m) s_ctl[1] = 1;
          }
        }
        __syncthreads();
      }
      if (warp == 0 && !found && nz + m - start >= ck.n && start_val != 0.0f) {  // end of the data (:592-603)
        inner = start_val - ck.buff;
        outer = prev_val + ck.buff;
      }
    } else {
      float* s_r = s_all;
      if (m <= SORT_SMEM) {
        for (int i = threadIdx.x; i < m; i += blockDim.x) s_r[i] = g[i];
        __syncthreads();
        block_sort_asc(s_r, m);
        if (threadIdx.x < 32) find_cluster_warp(s_r, m, nz, ck.n, ck.thresh, ck.buff, inner, outer);
      } else {
        __syncthreads();
        block_sort_asc(g, m);
        if (threadIdx.x < 32) find_cluster_warp(g, m, nz, ck.n, ck.thresh, ck.buff, inner, outer);
      }
    }
    if (threadIdx.x == 0) write_cluster_rec(ck, pair, cell, cnt, inner, outer);
    __syncthreads();
  }
}

// ----------------------------------------------------------------------------------------------
// Huge cells (more than HUGE_MIN non-zero ranges: an accumulated map as scan 1 puts 10^5..10^6 ranges into the cells
// along the street).  Same bucket form of findCluster as the CTA path of k_cluster, but the table of half-threshold
// buckets (count, min, max) lives in global memory and is filled by HUGE_SPLIT CTAs per cell with warp-aggregated
// atomics; one warp then walks the 32 768 buckets in ascending order.  Bit-identical bounds.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_huge_init(const Chunk ck) {
  const int slot = blockIdx.y;
  if (slot >= min(*ck.nhuge, HUGE_SLOTS)) return;
  int32_t* t = ck.hbkt + (size_t)slot * 3 * HUGE_NB;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < HUGE_NB; k += gridDim.x * blockDim.x) {
    t[k] = 0;
    t[HUGE_NB + k] = 0x7f800000;
    t[2 * HUGE_NB + k] = 0;
  }
}

__global__ void __launch_bounds__(256) k_huge_hist(const Chunk ck) {
  const int slot = blockIdx.y;
  if (slot >= min(*ck.nhuge, HUGE_SLOTS)) return;
  const int pair = ck.hpair[slot], cell = ck.hcell[slot];
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const int m = ck.cnt1[ci] - ck.cntz[ci];
  const float* g = ck.rbuf + (size_t)pair * ck.n1max + ck.off[ci];
  int32_t* t = ck.hbkt + (size_t)slot * 3 * HUGE_NB;
  const float inv_w = 1.0f / (0.5f * ck.thresh);
  const bool usable = ck.thresh > 1e-6f;
  const int lane = threadIdx.x & 31;
  bool overflow = !usable;
  for (int b0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31; b0 < m; b0 += gridDim.x * blockDim.x) {  // warp-uniform
    const int i = b0 + lane;
    int k = -1;
    float r = 0.f;
    if (i < m && usable) {
      r = __ldg(g + i);
      const float kf = floorf(r * inv_w);
      if (r >= 0.0f && kf < (float)HUGE_NB) k = (int)kf;   // false for NaN / inf as well
      else overflow = true;
    }
    const unsigned act = __ballot_sync(FULL, k >= 0);
    if (k >= 0) {
      // lanes that hit the same bucket combine: count by popc, min / max over the group
      const unsigned grp = __match_any_sync(act, k);
      int mn = __float_as_int(r), mx = mn;
      for (unsigned rest = grp & ~(1u << lane); rest; rest &= rest - 1) {
        const int o = __shfl_sync(grp, __float_as_int(r), __ffs(rest) - 1);
        mn = min(mn, o);
        mx = max(mx, o);
      }
      if (lane == __ffs(grp) - 1) {
        atomicAdd(&t[k], __popc(grp));
        atomicMin(&t[HUGE_NB + k], mn);
        atomicMax(&t[2 * HUGE_NB + k], mx);
      }
    }
  }
  if (__any_sync(FULL, overflow) && lane == 0) atomicOr(&ck.hflag[slot], 1);
}

// The walk over the bucket table of one huge cell, by one CTA.  The sequential walk (see the CTA path of k_cluster) is
//     for every non-empty bucket j in ascending order:  a BREAK in front of j  <=>  something precedes j and
//     !(|max of the previous non-empty bucket - min of j| <= thresh);  the run that ends at the first break whose run
//     holds >= n elements is the cluster (src/icet.cpp:572-582); else the last run, with the zero check (:592-603)
// i.e. a segmented scan: thread t owns HW_PER consecutive buckets; three block scans carry (elements so far, max of the
// last non-empty bucket so far, position / min of the last break so far) across the threads.  One serial warp over
// 32 768 buckets with dependent loads took 1.39 ms for a 2 M-point map; this form takes microseconds.
constexpr int HW_THREADS = 1024;
constexpr int HW_PER = HUGE_NB / HW_THREADS;  // 32 buckets per thread
static_assert(HUGE_NB % HW_THREADS == 0 && HW_PER % 4 == 0, "bucket table / walk shape");

struct HwCarry {     // "last one wins" summaries of a range of buckets
  int cnt;           // elements in the range
  int has;           // the range has a non-empty bucket
  int lastmax;       // ... max (bits) of its last non-empty bucket
  int hasbrk;        // the range has a break
  int brkidx;        // ... elements in front of its last break (within the range: relative, made absolute by the caller)
  int brkmin;        // ... min (bits) of the bucket behind that break
};

// inclusive block scan of a value with an associative operator; returns the EXCLUSIVE prefix of the calling thread
template <class T, class Op>
__device__ __forceinline__ T block_scan_excl(T v, T ident, Op op, T* s_w /* [32] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    T u;
    unsigned char* pu = reinterpret_cast<unsigned char*>(&u);
    const unsigned char* pi = reinterpret_cast<const unsigned char*>(&inc);
    static_assert(sizeof(T) % 4 == 0, "word-sized scan values");
    for (int k = 0; k < (int)sizeof(T) / 4; k++)
      reinterpret_cast<int*>(pu)[k] = __shfl_up_sync(FULL, reinterpret_cast<const int*>(pi)[k], o);
    if (lane >= o) inc = op(u, inc);
  }
  __syncthreads();  // (s_w may still be read from a previous scan)
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  T pre = ident;
  for (int w = 0; w < warp; w++) pre = op(pre, s_w[w]);
  // exclusive within the warp
  T exw;
  {
    unsigned char* pu = reinterpret_cast<unsigned char*>(&exw);
    const unsigned char* pi = reinterpret_cast<const unsigned char*>(&inc);
    for (int k = 0; k < (int)sizeof(T) / 4; k++)
      reinterpret_cast<int*>(pu)[k] = __shfl_up_sync(FULL, reinterpret_cast<const int*>(pi)[k], 1);
  }
  return lane == 0 ? pre : op(pre, exw);
}

__global__ void __launch_bounds__(HW_THREADS) k_huge_walk(const Chunk ck) {
  const int slot = blockIdx.x;
  if (slot >= min(*ck.nhuge, HUGE_SLOTS) || ck.hflag[slot] != 0) return;
  const int pair = ck.hpair[slot], cell = ck.hcell[slot];
  const size_t ci = (size_t)pair * ck.ncell + cell;
  const int cnt = ck.cnt1[ci], nz = ck.cntz[ci], m = cnt - nz;
  const int32_t* t = ck.hbkt + (size_t)slot * 3 * HUGE_NB;
  const int b0 = threadIdx.x * HW_PER;
  __shared__ int2 s_a[32];
  __shared__ int4 s_b[32];
  __shared__ int s_best;
  __shared__ float s_res[2];
  if (threadIdx.x == 0) s_best = 0x7fffffff;
  // the thread's buckets: counts, mins, maxs (vector loads; the table is L2-resident, k_huge_hist has just filled it)
  int c[HW_PER], mn[HW_PER], mx[HW_PER];
#pragma unroll
  for (int k = 0; k < HW_PER; k += 4) {
    const int4 a = *reinterpret_cast<const int4*>(t + b0 + k);
    const int4 b = *reinterpret_cast<const int4*>(t + HUGE_NB + b0 + k);
    const int4 d = *reinterpret_cast<const int4*>(t + 2 * HUGE_NB + b0 + k);
    c[k] = a.x; c[k + 1] = a.y; c[k + 2] = a.z; c[k + 3] = a.w;
    mn[k] = b.x; mn[k + 1] = b.y; mn[k + 2] = b.z; mn[k + 3] = b.w;
    mx[k] = d.x; mx[k + 1] = d.y; mx[k + 2] = d.z; mx[k + 3] = d.w;
  }
  // scan 1: elements in front of the thread's buckets, max of the last non-empty bucket in front of them
  int2 mine = make_int2(0, -1);  // {count, last max bits or -1}
#pragma unroll
  for (int k = 0; k < HW_PER; k++)
    if (c[k] > 0) { mine.x += c[k]; mine.y = mx[k]; }
  const int2 pre = block_scan_excl(mine, make_int2(0, -1),
                                   [](int2 a, int2 b) { return make_int2(a.x + b.x, b.y >= 0 ? b.y : a.y); }, s_a);
  // local pass: breaks.  idx = elements in front of bucket k (the nz zeros first); prev = max of the previous non-empty
  // bucket, 0.0 for the zeros / the start
  int idx = nz + pre.x;
  float prev = pre.y >= 0 ? __int_as_float(pre.y) : 0.0f;
  bool any_before = nz > 0 || pre.y >= 0;  // (idx > 0 in the sequential walk)
  // the thread's breaks: {first: position, idx}, {last: idx, min}; run lengths between its own breaks are checked here
  int first_brk_idx = -1, last_brk_idx = -1, last_brk_min = 0;
  int found_k = -1;          // first bucket of this thread whose break ends a run of >= n that STARTED in this thread
  float found_in = 0.f, found_out = 0.f;
  int first_brk_k = -1;
  float first_brk_prev = 0.f;  // max in front of the thread's first break (the run that ends there began earlier)
#pragma unroll
  for (int k = 0; k < HW_PER; k++) {
    if (c[k] > 0) {
      const float mnv = __int_as_float(mn[k]);
      if (any_before && !(fabsf(prev - mnv) <= ck.thresh)) {
        if (first_brk_idx < 0) {
          first_brk_idx = idx; first_brk_k = k; first_brk_prev = prev;
        } else if (found_k < 0 && idx - last_brk_idx >= ck.n) {
          found_k = k; found_in = __int_as_float(last_brk_min) - ck.buff; found_out = prev + ck.buff;
        }
        last_brk_idx = idx; last_brk_min = mn[k];
      }
      idx += c[k];
      prev = __int_as_float(mx[k]);
      any_before = true;
    }
  }
  // scan 2: the last break in front of the thread: {has, idx, min bits}
  const int4 lb = block_scan_excl(make_int4(last_brk_idx >= 0 ? 1 : 0, last_brk_idx, last_brk_min, 0), make_int4(0, 0, 0, 0),
                                  [](int4 a, int4 b) { return b.x ? b : a; }, s_b);
  // the run that ends at the thread's FIRST break started at the last break in front of the thread, or at element 0
  // (then its first value is 0.0 if there are zeros, else the min of the very first non-empty bucket: thread-uniform
  // quantity found below)
  int cand = 0x7fffffff;  // global bucket index of the thread's first qualifying break
  bool cand_first = false;
  if (first_brk_idx >= 0 && first_brk_idx - (lb.x ? lb.y : 0) >= ck.n) { cand = b0 + first_brk_k; cand_first = true; }
  else if (found_k >= 0) cand = b0 + found_k;
  __syncthreads();
  if (cand != 0x7fffffff) atomicMin(&s_best, cand);
  // min of the very first non-empty bucket of the table (start value of the first run when there are no zeros)
  __shared__ int s_firstmin_k, s_firstmin;
  if (threadIdx.x == 0) s_firstmin_k = 0x7fffffff;
  __syncthreads();
  int fk = -1, fmn = 0;
#pragma unroll
  for (int k = HW_PER - 1; k >= 0; k--)
    if (c[k] > 0) { fk = k; fmn = mn[k]; }
  if (fk >= 0) atomicMin(&s_firstmin_k, b0 + fk);
  __syncthreads();
  if (fk >= 0 && s_firstmin_k == b0 + fk) s_firstmin = fmn;
  __syncthreads();
  const float first_val = (nz > 0 || s_firstmin_k == 0x7fffffff) ? 0.0f : __int_as_float(s_firstmin);
  if (cand != 0x7fffffff && cand == s_best) {  // exactly one thread
    if (cand_first) {
      s_res[0] = (lb.x ? __int_as_float(lb.z) : first_val) - ck.buff;
      s_res[1] = first_brk_prev + ck.buff;
    } else {
      s_res[0] = found_in;
      s_res[1] = found_out;
    }
  }
  __syncthreads();
  float inner = 0.f, outer = 0.f;
  if (s_best != 0x7fffffff) {
    inner = s_res[0];
    outer = s_res[1];
  } else if (threadIdx.x == HW_THREADS - 1) {
    // end of the data (:592-603): the run behind the last break of the whole table (inclusive of this thread's)
    const int st = last_brk_idx >= 0 ? last_brk_idx : (lb.x ? lb.y : 0);
    const float sv = last_brk_idx >= 0 ? __int_as_float(last_brk_min) : (lb.x ? __int_as_float(lb.z) : first_val);
    if (nz + m - st >= ck.n && sv != 0.0f) {
      inner = sv - ck.buff;
      outer = prev + ck.buff;  // max of the last non-empty bucket of the table
    }
    s_res[0] = inner;
    s_res[1] = outer;
  }
  __syncthreads();
  if (threadIdx.x == 0) write_cluster_rec(ck, pair, cell, cnt, s_res[0], s_res[1]);
}

// ----------------------------------------------------------------------------------------------
// ICET_B200_FLAG_SHIPPED_ORDER (single pair, validation): clustering in the row order the reference ends up with
// after its broken permutation loop (src/icet.cpp:72-83); ck.pos1 holds that position for every row of scan 1.
// Zero ranges are ordinary members of the sequence here.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_off_shipped(const Chunk ck) {  // offsets of ALL points per cell
  const int pair = blockIdx.x;
  __shared__ int s_part[256];
  const int per = (ck.ncell + 255) / 256;
  const int c0 = threadIdx.x * per, c1 = min(ck.ncell, c0 + per);
  const int32_t* cnt1 = ck.cnt1 + (size_t)pair * ck.ncell;
  int s = 0;
  for (int c = c0; c < c1; c++) s += cnt1[c];
  s_part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int a = 0;
    for (int t = 0; t < 256; t++) { const int v = s_part[t]; s_part[t] = a; a += v; }
  }
  __syncthreads();
  int a = s_part[threadIdx.x];
  for (int c = c0; c < c1; c++) {
    ck.off[(size_t)pair * ck.ncell + c] = a;
    ck.cursor[(size_t)pair * ck.ncell + c] = 0;
    a += cnt1[c];
  }
}

__global__ void __launch_bounds__(256) k_scatter_shipped(const Chunk ck) {
  const int pair = blockIdx.y;
  const PairDesc d = ck.desc[pair];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d.n1) return;
  const size_t o = (size_t)pair * ck.n1max + i;
  const int cell = ck.cellid1[o] & ~CELL_INBOX;
  const int slot = atomicAdd(&ck.cursor[(size_t)pair * ck.ncell + cell], 1);
  const unsigned long long key = ((unsigned long long)(unsigned)ck.pos1[o] << 32) | (unsigned)__float_as_uint(ck.r1[o]);
  ck.kbuf[(size_t)pair * ck.n1max + ck.off[(size_t)pair * ck.ncell + cell] + slot] = key;
}

struct KeyRanges {  // the ranges of a cell in row order: low words of the keys sorted by position
  const unsigned long long* k;
  __device__ __forceinline__ float operator[](int i) const { return __uint_as_float((unsigned)(k[i] & 0xffffffffull)); }
};

__global__ void __launch_bounds__(128) k_cluster_shipped(const Chunk ck) {
  const int pair = blockIdx.y;
  const int nw = ck.nwork[pair];
  for (int w = blockIdx.x; w < nw; w += gridDim.x) {
    const int cell = ck.work[(size_t)pair * ck.ncell + w];
    const int m = ck.cnt1[(size_t)pair * ck.ncell + cell];
    unsigned long long* g = ck.kbuf + (size_t)pair * ck.n1max + ck.off[(size_t)pair * ck.ncell + cell];
    __syncthreads();
    block_sort_asc(g, m);  // by row position (the high word is unique)
    float inner = 0.f, outer = 0.f;
    if (threadIdx.x < 32) find_cluster_warp(KeyRanges{g}, m, 0, ck.n, ck.thresh, ck.buff, inner, outer);
    if (threadIdx.x == 0) write_cluster_rec(ck, pair, cell, m, inner, outer);
    __syncthreads();
  }
}


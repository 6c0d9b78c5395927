// icet_b200/csrc/kernels_cluster.cuh -- the Gauss-Newton loop of a pair inside ONE THREAD-BLOCK CLUSTER (latency shape:
// single pairs, small batches, chained odometry).  Included by icet_b200.cu inside its anonymous namespace.
//
// The persistent kernel k_loop spreads the ~1100 tasks of an iteration over the whole GPU and orders them with flags
// in global memory (tickets, per-pair counters, polling): with one pair in flight the flag round trips ARE the
// iteration (33 us per iteration for ~1 us of issue, VERDICT r01).  With the incremental scan-2 pass an iteration is
// small enough for a handful of SMs, so this form gives a pair to one cluster of CS CTAs (16 where the device allows
// the non-portable size, else 8) and replaces every flag by the hardware cluster barrier:
//     phase 1  all warps of the cluster walk the pair's scan-2 tiles (pass2_warp_tile: margin test / re-evaluation /
//              rebuild), integer moments go to the L2-resident accumulators            -> barrier.cluster
//     phase 2  one thread per voxel: fitCells2 algebra; 28 partial sums per CTA in ITS shared memory, fixed order
//                                                                                       -> barrier.cluster
//     phase 3  warp 0 of CTA 0 adds the CS partial sums through DISTRIBUTED SHARED MEMORY (rank order), solves the
//              6x6 system on the warp, publishes X / R(X) / get_H / the mode of the next iteration -> barrier.cluster
// Independent pairs of a small batch run in different clusters of the same launch; chained pairs (odometry.cpp:82)
// run back to back in one cluster.  Same per-point / per-voxel arithmetic as the other loop forms.
#pragma once
// (icet_b200.cu includes <cooperative_groups.h> at global scope)

constexpr int CL_THREADS = 256;
constexpr int CL_WARPS = CL_THREADS / 32;
constexpr int CL_K = PASS_K_SMALL;  // rows per warp tile (128 points: ~4 tiles per warp of a 16-CTA cluster at 64 channels)

__host__ __device__ inline int cluster_smem_bytes(int nT, int nP, int /*cs*/) {
  return CL_WARPS * pass_wslots(CL_K) * 16 + pass_tab_floats(nT, nP) * 4 + (CL_WARPS + 1) * NRED * 8 + 64 * 4;
}

// phase 2 of an iteration (inlined: a non-inlined callee would read the Chunk through local memory instead of the
// constant bank, which costs more than the spills it saves -- measured)
__device__ __forceinline__ void cluster_vox_phase(const Chunk& ck, int pair, int iter, int rank, int cs, const float* s_J,
                                               double* wpart, double* cpart) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc[NRED];
#pragma unroll
  for (int k = 0; k < NRED; k++) acc[k] = 0.0;
  // cell c -> CTA c % cs, thread c / cs: the occupied rows of the grid spread over all CTAs
  for (int c = rank + cs * (int)threadIdx.x; c < ck.ncell; c += cs * CL_THREADS) vox_contrib(ck, pair, c, iter, s_J, acc);
  // debug timeline (per-voxel dumps only): when the LAST thread of CTA 0 is through its voxel / the warp reduction
  if (ck.dump_on && rank == 0) atomicMax(&ck.dump.tl[(size_t)iter * 16 + 8], gtime());
  const double tot = warp_sum_transposed(acc, lane);
  if (lane < NRED) wpart[warp * NRED + lane] = tot;
  if (ck.dump_on && rank == 0) atomicMax(&ck.dump.tl[(size_t)iter * 16 + 9], gtime());
  __syncthreads();
  if (threadIdx.x < NRED) {
    double s = 0.0;
    for (int w = 0; w < CL_WARPS; w++) s += wpart[w * NRED + threadIdx.x];
    cpart[threadIdx.x] = s;
  }
}

// phase 3 (warp 0 of CTA 0): the partial sums of all CTAs through distributed shared memory, then the 6x6 solve
__device__ __noinline__ void cluster_solve_phase(const Chunk& ck, int pair, int iter, int cs, double* cpart, double* w_tot,
                                                 const ModeNow* cur) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int lane = threadIdx.x & 31;
  // every remote load is requested before the first addition (a rolled loop would pay the ~200-cycle DSMEM latency 16
  // times in a row); the additions are in rank order
  double pv[16];
#pragma unroll
  for (int r = 0; r < 16; r++) pv[r] = (lane < NRED && r < cs) ? cluster.map_shared_rank(cpart, r)[lane] : 0.0;
  double tot = 0.0;
#pragma unroll
  for (int r = 0; r < 16; r++) tot += pv[r];
  if (lane < NRED) w_tot[lane] = tot;  // (phase 2 is over: its scratch is reused)
  __syncwarp();
  if (ck.dump_on && lane == 0) ck.dump.tl[(size_t)iter * 16 + 11] = gtime();  // (debug timeline: partial sums gathered)
  bool done = false;
  if (!(ck.flags & ICET_B200_FLAG_FULL_EIG)) done = solve_pair_warp(ck, pair, iter, w_tot, cur);
  if (!done && lane == 0) solve_pair(ck, pair, iter, w_tot, cur);
}

// first_tiles_done: the tiles of iteration 0 of every pair have been processed by a GPU-wide k_pass2 launch already
// (single pairs: the first rebuild then runs on 148 SMs instead of the cluster's 16)
// nhelp > 0 (single pair / chained pairs): the launch has 1 + nhelp clusters.  Cluster 0 is the pair's cluster as
// described above; the others are HELPERS that take their share of the scan-2 tiles of every iteration (a rebuild
// evaluates every point: 21 us on the 16 SMs of one cluster; the delta iterations right after it re-evaluate a good
// part of them) and do nothing else.  Two words
// in global memory order them: `go` = (sequence number of the iteration << 1 | shared rebuild), published by the solve
// warp of the master as soon as it has written the transform and the mode of that iteration (the helpers start on the
// tiles while the master is still in the barrier that ends the previous one); `done` = helper warps through with their
// tiles, awaited by the master before its first cluster barrier.  A helper that finds `go` beyond the iteration it
// waits for knows that iteration was not shared.  An iteration is shared only if every helper cluster has reported
// itself RESIDENT (`alive`) when the solve warp decides: the master never waits for a cluster that is not running, so
// the scheme cannot deadlock however the clusters of concurrent launches are placed.
__device__ __forceinline__ int cluster_spin_ge(const int* p, int need) {  // value >= need, by one lane; traps after 20 s
  // (relaxed polling: an acquire load invalidates the SM's L1 every time; one acquire load once the value is there)
  int v = ld_relaxed(p);
  unsigned long long t0 = 0;
  for (unsigned spin = 1; v < need; spin++) {
    __nanosleep(32);
    v = ld_relaxed(p);
    if ((spin & 1023u) == 0u) {
      const unsigned long long t = gtime();
      if (t0 == 0) t0 = t;
      else if (t - t0 > 20000000000ull) __trap();
    }
  }
  return ld_acquire(p);
}

__global__ void __launch_bounds__(CL_THREADS, 1) k_loop_cluster(const Chunk ck, int first_tiles_done, int nhelp) {
  pdl_prologue();
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int4* ent = reinterpret_cast<int4*>(smem_raw);
  float* tab = reinterpret_cast<float*>(smem_raw + CL_WARPS * pass_wslots(CL_K) * 16);
  double* wpart = reinterpret_cast<double*>(tab + pass_tab_floats(ck.nT, ck.nP));  // [CL_WARPS][NRED]
  double* cpart = wpart + CL_WARPS * NRED;                                         // [NRED]  this CTA's partial sums
  float* s_J = reinterpret_cast<float*>(cpart + NRED);                             // [27]
  __shared__ unsigned long long s_mbar[CL_WARPS];  // one mbarrier per warp: completion of its staged scan-2 tiles
  const unsigned cs = cluster.num_blocks(), rank = cluster.block_rank();
  {
    const int ntab = pass_tab_floats(ck.nT, ck.nP);
    for (int k = threadIdx.x; k < ntab; k += CL_THREADS) tab[k] = __ldg(ck.binrec + k);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ncl = gridDim.x / cs, cl = blockIdx.x / cs;  // clusters of the launch, this cluster
  int4* went = ent + warp * pass_wslots(CL_K);
  if (lane == 0) mbar_init(&s_mbar[warp], 1);
  __syncwarp();
  unsigned mphase = 0u;
  const bool chain = (ck.flags & ICET_B200_FLAG_CHAIN_X0) != 0;
  const bool inc = loop_incremental(ck);
  const int gwarp = (int)rank * CL_WARPS + warp, nwarp = (int)cs * CL_WARPS;
  int* go = ck.iter_done;                                  // (words of the persistent kernel, unused in this form)
  int* done = reinterpret_cast<int*>(ck.tiles_done);
  int* alive = reinterpret_cast<int*>(ck.vox_done);
  const int gw_all = cl * nwarp + gwarp, nw_all = (1 + nhelp) * nwarp;  // this warp among those of all clusters
  if (nhelp > 0 && cl > 0) {
    // ------------------------------------------------------------------ helper cluster
    if (rank == 0 && threadIdx.x == 0) red_add(reinterpret_cast<unsigned*>(alive), 1u);  // (a cluster is co-scheduled)
    for (int pair = 0; pair < ck.npairs; pair++) {
      const int n = __ldg(ck.n2c + pair);
      const int tiles = max(1, (n + 32 * CL_K - 1) / (32 * CL_K));
      const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
      for (int iter = 0; iter < ck.runlen; iter++) {
        const int seq = pair * ck.runlen + iter + 1;
        int g = 0;
        if (lane == 0) g = cluster_spin_ge(go, seq << 1);
        g = __shfl_sync(FULL, g, 0);
        if ((g >> 1) != seq || !(g & 1)) continue;  // not shared (or the master is past it already: it was not)
        float tr[12];
        {
          const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
          const float4 a = __ldcg(tp), b = __ldcg(tp + 1), c = __ldcg(tp + 2);
          tr[0] = a.x; tr[1] = a.y; tr[2] = a.z; tr[3] = a.w; tr[4] = b.x; tr[5] = b.y; tr[6] = b.z; tr[7] = b.w;
          tr[8] = c.x; tr[9] = c.y; tr[10] = c.z; tr[11] = c.w;
        }
        Pass2Mode md;
        load_pass2_mode(ck, pair, md);
        for (int tile = gw_all; tile < tiles; tile += nw_all)
          pass2_warp_tile<CL_K>(ck, went, &s_mbar[warp], mphase, false, tab, recs, tr, md,
                                ck.pog + (size_t)pair * 3 * ck.n2max, (size_t)ck.n2max, n, tile * 32 * CL_K,
                                ck.mrec + (size_t)pair * ck.n2max,
                                (ck.flags & ICET_B200_FLAG_VERIFY_INCREMENTAL) ? &ck.res[pair].reserved[0] : nullptr);
        __threadfence();  // every lane: its records and moment updates before the warp is counted
        __syncwarp();
        if (lane == 0) red_add(reinterpret_cast<unsigned*>(done), 1u);
      }
    }
    return;
  }
  int nshared = 0;  // rebuild iterations shared with the helpers so far
  // chained pairs: one cluster walks them in order; independent pairs: round robin over the clusters of the launch
  const int pstride = (chain || nhelp > 0) ? 1 : ncl;
  for (int pair = (chain || nhelp > 0) ? 0 : cl; pair < ck.npairs; pair += pstride) {
    const int n = __ldg(ck.n2c + pair);
    const int tiles = max(1, (n + 32 * CL_K - 1) / (32 * CL_K));
    const CellRec* recs = ck.rec + (size_t)pair * ck.ncell;
    for (int iter = 0; iter < ck.runlen; iter++) {
#define CTL(slot)                                                                                           \
  do {                                                                                                      \
    if (ck.dump_on && rank == 0 && threadIdx.x == 0) ck.dump.tl[(size_t)iter * 16 + (slot)] = gtime();      \
  } while (0)
      CTL(0);
      // ------------------------------------------------------------------ phase 1: scan-2 tiles
      float tr[12];
      {
        const float4* tp = reinterpret_cast<const float4*>(ck.TR + (size_t)pair * 12);
        const float4 a = __ldcg(tp), b = __ldcg(tp + 1), c = __ldcg(tp + 2);
        tr[0] = a.x; tr[1] = a.y; tr[2] = a.z; tr[3] = a.w; tr[4] = b.x; tr[5] = b.y; tr[6] = b.z; tr[7] = b.w;
        tr[8] = c.x; tr[9] = c.y; tr[10] = c.z; tr[11] = c.w;
      }
      if (threadIdx.x < 27) s_J[threadIdx.x] = __ldcg(ck.J + (size_t)pair * 27 + threadIdx.x);
      Pass2Mode md;
      if (inc) load_pass2_mode(ck, pair, md);
      const bool skip_tiles = first_tiles_done && iter == 0 && !(chain && pair > 0);
      // a rebuild iteration is shared with the helper clusters (the mode is what the last solve published: uniform)
      const bool first_iter = pair == 0 && iter == 0;  // (no solve of this launch in front of it: never shared)
      const bool share = nhelp > 0 && inc && !skip_tiles && !first_iter && __ldcg(&ck.pm[pair].pad[0]) != 0;
      if (nhelp > 0 && first_iter && rank == 0 && threadIdx.x == 0) st_release(go, 1 << 1);
      if (!skip_tiles) {
        if (inc) {
          for (int tile = share ? gw_all : gwarp; tile < tiles; tile += share ? nw_all : nwarp)
            pass2_warp_tile<CL_K>(ck, went, &s_mbar[warp], mphase, false, tab, recs, tr, md,
                                        ck.pog + (size_t)pair * 3 * ck.n2max, (size_t)ck.n2max, n, tile * 32 * CL_K,
                                        ck.mrec + (size_t)pair * ck.n2max,
                                        (ck.flags & ICET_B200_FLAG_VERIFY_INCREMENTAL) ? &ck.res[pair].reserved[0] : nullptr);
          if (gwarp == nwarp - 1 && lane == 0)  // (the last warp has the fewest tiles)
            pass2_dropped_returns(ck, reinterpret_cast<const float4*>(tab), reinterpret_cast<const float4*>(tab) + ck.nT + 2,
                                  recs, tr, md, pair, __ldg(ck.nz2 + pair));
        } else {
          unsigned long long* accp = ck.acc + (size_t)pair * ck.ncell * NQ;
          const int n2 = __ldg(&ck.desc[pair].n2);
          for (int tile = gwarp; tile < tiles; tile += nwarp)
            pass_warp_tile<true, CL_K, 2, 4>(ck, went, tab, recs, tr, ck.pog + (size_t)pair * 3 * ck.n2max,
                                             (size_t)ck.n2max, n, tile * 32 * CL_K, fix_point(n2), accp);
          if (gwarp == nwarp - 1 && lane == 0)
            pass_dropped_returns(ck, reinterpret_cast<const float4*>(tab), reinterpret_cast<const float4*>(tab) + ck.nT + 2,
                                 recs, tr, accp, __ldg(ck.nz2 + pair), n2);
        }
      }
      if (share) {  // (uniform) the helpers' tiles before the voxel phase
        nshared++;
        if (rank == 0 && threadIdx.x == 0) cluster_spin_ge(done, nshared * nhelp * nwarp);
      }
      CTL(1);
      // (barrier.cluster has release / acquire semantics at cluster scope: the moments -- RED to L2 -- and the records
      // written above are visible to every thread of the cluster after it; no GPU-wide fence is needed)
      cluster.sync();
      CTL(2);
      // ------------------------------------------------------------------ phase 2: one thread per voxel
      cluster_vox_phase(ck, pair, iter, (int)rank, (int)cs, s_J, wpart, cpart);
      CTL(3);
      cluster.sync();
      CTL(4);
      // ------------------------------------------------------------------ phase 3: DSMEM reduction + solve
      if (rank == 0 && warp == 0) {
        int nalive = 0;
        if (nhelp > 0 && lane == 0) nalive = ld_relaxed(alive);  // (requested now, needed after the solve)
        ModeNow now = {md.SA, md.SB, md.set};
        cluster_solve_phase(ck, pair, iter, (int)cs, cpart, wpart, inc ? &now : nullptr);
        if (ck.dump_on && lane == 0) ck.dump.tl[(size_t)iter * 16 + 12] = gtime();  // (debug timeline: solved)
        // the NEXT iteration (of this pair, or the first one of the next chained pair) is announced right here
        if (nhelp > 0) {
          int npair = pair, niter = iter + 1;
          if (niter == ck.runlen) { npair = pair + 1; niter = 0; }
          if (npair < ck.npairs) {
            __syncwarp();  // (the lanes' stores of X / TR / J / mode before lane 0 publishes)
            if (lane == 0) {
              // every iteration is shared when the helpers are there (measured: sharing only rebuilds 0.2015 ms /
              // 6.3 k chained pairs/s; rebuilds + deltas after a step of millimetres 0.196 / 6.5 k; everything 0.188 / 7.0 k)
              const int sh = (inc && nalive == nhelp) ? 1 : 0;
              ck.pm[npair].pad[0] = sh;
              st_release(go, ((npair * ck.runlen + niter + 1) << 1) | sh);
            }
          }
        }
      }
      CTL(5);
      cluster.sync();
      CTL(6);
#undef CTL
    }
  }
}

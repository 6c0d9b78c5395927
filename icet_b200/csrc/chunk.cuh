// icet_b200/csrc/chunk.cuh -- error reporting helpers, per-chunk device state (Chunk and its records), constants and
// the explicit-address-space atomics.  Included by icet_b200.cu inside its anonymous namespace.
#pragma once

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(ICET_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));      \
  } while (0)

constexpr int FPB = 21;                 // fixed-point basis: CellRec::scale maps the voxel's box diameter D to 2^(FPB-1)
constexpr int FP_LIM = (1 << FPB);      // (the per-pair multiplier FixPt::fs refines it, see fp_bits below)
constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t F_STAT1 = 1u;        // scan-1 statistics wanted for this cell
constexpr uint32_t F_ACTIVE2 = 2u;      // voxel takes part in the scan-2 loop
constexpr int SORT_SMEM = 4096;         // cells up to this many points are sorted in shared memory
constexpr int NQ = 12;                  // accumulator words per cell
constexpr int CLUSTER_WARPS = 4;
constexpr int WSORT_MAX = 1024;         // cells up to this many non-zero ranges are sorted by one warp in registers
constexpr int HUGE_MIN = 32768;         // cells with more non-zero ranges (accumulated maps) are clustered by many CTAs
constexpr int HUGE_SLOTS = 64;          //   ... at most this many per chunk (the rest take the one-CTA path)
constexpr int HUGE_NB = 32768;          //   ... through a global table of this many half-threshold buckets per cell
constexpr int HUGE_SPLIT = 128;         //   ... filled by this many CTAs per cell
// class word of a stored point of scan 2 (incremental loop, kernels_pass2.cuh): 24 bits, packed into its margin record
constexpr uint32_t CLS_CELL = 0x003fffffu;    // cell index (validate(): bins_phi * bins_theta <= 2^20)
constexpr uint32_t CLS_IN = 0x00400000u;      // the point passes filterPointsInsideCluster of its cell
constexpr uint32_t CLS_ACTIVE = 0x00800000u;  // its cell takes part in the loop (F_ACTIVE2)
constexpr uint32_t CLS_NONE = 0x003fffffu;    // "no class yet"

struct PairDesc {
  const float* s1;
  const float* s2;
  int n1, ld1, n2, ld2;
};

// Fixed-point refinement of the per-voxel accumulators of a cloud of n points: offsets are quantised to
// round(d * CellRec::scale * fs), clamped to +-fl, with fs = 2^(bits - FPB) and fl = 2^bits.  Offsets up to 2^bits,
// products up to 2^(2 bits), 64-bit sums over at most n points: 2 bits + ceil(log2 n) <= 62.  As fine as that allows
// (131 072 points: 2^22 levels per box diameter, i.e. ~2 um at 50 m -- below the fp32 ulp of the coordinates
// themselves).  A function of the pair's own cloud (PairDesc::n1 for scan 1, n2 for scan 2), never of the other pairs
// of its chunk: the result of a pair does not depend on how a batch is cut into chunks or ordered.
__host__ __device__ __forceinline__ int fp_bits(int n) {
  const unsigned m = (unsigned)(n > 2 ? n : 2) - 1u;  // ceil(log2(max(n, 2))) = bit length of m
#ifdef __CUDA_ARCH__
  const int lg = 32 - __clz(m);
#else
  const int lg = 32 - __builtin_clz(m);
#endif
  const int b = (62 - lg) / 2;
  return b < 12 ? 12 : (b > 23 ? 23 : b);
}
struct FixPt {
  float fs;  // multiplier of CellRec::scale (a power of two)
  int fl;    // clamp of the offsets
};
__host__ __device__ __forceinline__ FixPt fix_point(int n) {
  const int b = fp_bits(n);
#ifdef __CUDA_ARCH__
  return FixPt{__int_as_float((127 + b - FPB) << 23), 1 << b};
#else
  return FixPt{ldexpf(1.0f, b - FPB), 1 << b};
#endif
}

struct __align__(16) CellRec {  // read by the pass kernels: first half by every point, second half per run of inside points
  float inner, outer;           // clusterBounds columns 4,5 (src/icet.cpp:149)
  uint32_t flags;
  float scale;                  // power-of-two scale of the voxel's fixed-point frame
  float refx, refy, refz;       // reference point of the fixed-point frame
  int32_t cnt1;                 // points of scan 1 in this angular bin
};

struct Vox1 {     // scan-1 Gaussian, constants of the iteration loop (sigma1/mu1/U/L, include/icet.h:89-94)
  double mu[3];
  double S1n[6];  // sigma1 / (cnt1 - 1), upper triangle xx xy xz yy yz zz
  double LV[9];   // L * U^T = L * V  (rows of V, zeroed where L is 0)
  int lmask;      // bit k: L(k,k) == 1
  int pad;
};

// Per-pair control block of the incremental scan-2 loop (kernels_pass2.cuh): written by k_cell_scan (first iteration:
// rebuild) and by the 6x6 solve for the iteration that follows it.
struct __align__(16) PairMode {
  int set;        // accumulator set (0 / 1) the current iteration reads and updates
  int rebuild;    // 1: every point is evaluated and the set is built from zero; 0: only points whose margin is used up
  float SA, C;    // motion odometers since the last rebuild: SA = sum |R_j+1 - R_j|_F, C = SB + SA * SB, SB = sum |t_j+1 - t_j|
  float SB;
  int zcls;       // class word of the dropped-return point (0,0,0) in the previous iteration
  int pad[2];
  float TRb[12];  // transform of the last rebuild: the voxels' fixed-point frames of scan 2 are anchored to it
  int pad2[4];
};

struct Dump {  // optional per-voxel recording (device memory), single-pair debugging only
  int32_t* nin1; uint8_t* has1; float* mu1; float* sigma1; float* evec1; float* eval1; uint8_t* lmask;
  int32_t* cnt2; int32_t* nin2; uint8_t* used2; float* mu2; float* sigma2; float* Xit; float* HTWH; float* HTWdz;
  float* TRit;      // [runlen][12] t | R(X) every iteration used (src/icet.cpp:375-376)
  float* testpts;   // [ncell*6][3] the reference's public `testPoints` (src/icet.cpp:214-232): sigma points of suppressed axes
  unsigned long long* tl;  // [runlen][16] globaltimer stamps of the loop kernel (debug) + per-tile stamps of iteration 3
};

struct Chunk {  // everything a kernel needs, passed by value
  const PairDesc* desc;
  int npairs, ncell, nT, nP, n, runlen, flags;
  float thresh, buff;
  int n1max, n2max;  // capacities of the per-pair arrays below (the fixed-point precision of a pair: fix_point)
  // scan 1
  int32_t* cellid1;  // [P][n1max]
  float* r1;         // [P][n1max]
  float* th1;        // [P][n1max]  theta, phi of scan 1 (K1 -> K3: the second pass over scan 1 does not redo the
  float* ph1;        // [P][n1max]  spherical conversion)
  float* rbuf;       // [P][n1max]  non-zero ranges grouped by cell
  int32_t* cellg;    // [P][n1max]  ... and, in the same grouped order, cell | CELL_INBOX, theta, phi of those points: the
  float* thg;        // [P][n1max]  second pass over scan 1 (K3) walks the points cell by cell (long runs of equal cell,
  float* phg;        // [P][n1max]  also for an unordered cloud such as an accumulated map).  Null in shipped-order mode.
  int32_t* n1g;      // [P]         number of grouped (non-zero) points
  unsigned long long* kbuf;  // [n1max]  ICET_B200_FLAG_SHIPPED_ORDER: (row position << 32 | range bits) grouped by cell
  int32_t* pos1;     // [n1max]  ... position of every row of scan 1 in the reference's shipped row order
  int32_t* cnt1;     // [P][ncell]
  int32_t* cntz;     // [P][ncell]  zero-range points
  int32_t* off;      // [P][ncell]
  int32_t* cursor;   // [P][ncell]
  int32_t* work;     // [P][ncell]  cells with cnt1 >= n
  int32_t* nwork;    // [P]
  int32_t* nbig;     // [P]  cells of the work list with more than WSORT_MAX non-zero ranges
  int32_t* hslot;    // [P][ncell]  huge cells: slot + 1 in the tables below (0: none)
  int32_t* nhuge;    // [1]
  int32_t* hpair;    // [HUGE_SLOTS]
  int32_t* hcell;    // [HUGE_SLOTS]
  int32_t* hflag;    // [HUGE_SLOTS]  1: a range fell outside the table -> the cell takes the one-CTA path after all
  int32_t* hbkt;     // [HUGE_SLOTS][3][HUGE_NB]  count | min bits | max bits per bucket (null: path disabled for the chunk)
  CellRec* rec;      // [P][ncell]
  unsigned long long* acc;  // [2][P][ncell][NQ]  (set 1 is used by the incremental scan-2 loop only)
  Vox1* vox;         // [P][ncell]
  int32_t* vlist;    // [P][ncell]  split loop: the pair's active voxels (F_ACTIVE2) in ascending cell order (k_vox_list)
  int32_t* nvox;     // [P]         ... and their number
  const float* azE;  // [nT+1] float azimuth bin edges  (src/icet.cpp:136-137)
  const float* elE;  // [nP+1] float elevation bin edges (src/icet.cpp:138-139)
  icet::BinTable bth, bph;  // exact bin lookup tables (src/icet.cpp:545-546)
  const float* binrec;      // [(nT+1) + (nP+1)][4] bin + box records of the pass kernels (see bin_box)
  float* TR;         // [P][12] translation (3) and rotation R(X) (9) of the current iteration
  float* TRprev;     // [P][12] transform the LAST iteration used (the reference's public `points2`)
  float* J;          // [P][27] get_H derivative matrices Jx | Jy | Jz of the current iteration
  double* part;      // [P][nblk][NRED] per-block partial sums of the voxel contributions
  // scan 2
  float* pog;        // [P][3][n2max]  points2_OG without the dropped returns (compacted, any order); n2max is a multiple
                     //               of 4 so that every plane (and every 32-point row of it) starts on a 16-byte boundary:
                     //               the pass kernels stage their tiles with bulk async copies (cp.async.bulk)
  int32_t* n2c;      // [P] points stored in pog
  int32_t* nz2;      // [P] dropped returns of scan 2 (points2_OG == 0)
  uint2* mrec;       // [P][n2max]  incremental loop: one 64-bit margin record per stored point (rec2_pack, kernels_pass2.cuh):
                     //               {u (24 significant bits, rounded down), r_e (bf16, rounded up), class word (24 bits)};
                     //               the class of the point's last evaluation cannot have changed while r_e * SA + C < u
  float4* anch;      // [P][ncell]  {anchor xyz, scale} of the scan-2 fixed-point frame of every active voxel at the transform
                     //               of the pair's last rebuild (written by k_fit1 / k_solve6, read by k_pass2)
  float inc_max_sa, inc_max_sb;  // a pair rebuilds when its motion odometers exceed these (INC_MAX_SA / INC_MAX_SB)
  PairMode* pm;      // [P]
  float* X;          // [P][6]
  const float* x0;   // [P][6] or null
  icet_b200_result* res;  // [P] device
  // control words of the persistent Gauss-Newton kernel (k_loop)
  unsigned* ticket;      // [1]  next task
  unsigned* tiles_done;  // [P]  scan-2 tiles finished so far (all iterations)
  int* iter_done;        // [P]  iterations whose solve has been published
  unsigned* vox_done;    // [P][runlen] vox tasks finished per iteration
  unsigned* vmask;       // [P][ceil(vt/32)] vox groups that wrote a partial sum (current iteration)
  int* dbg;              // [8] watchdog record of k_loop: {tripped, kind, pair, iter, seen, need, ticket, -}
  unsigned long long loop_timeout_ns;  // a wait inside k_loop gives up after this long
  Dump dump;
  int dump_on;
};

// Atomics on Chunk memory, with the address space spelled out.  Kernels that hand the Chunk to non-inlined device
// functions by reference (k_loop) keep it in local memory, and the compiler then no longer knows which address space
// the pointers it loads from there refer to: atomicAdd() becomes a GENERIC atomic that waits for a predicate from the
// memory system (one L2 round trip each instead of a fire-and-forget RED) plus a shared-memory CAS fallback.
__device__ __forceinline__ void red_add(unsigned long long* p, unsigned long long v) {
  asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void red_add(unsigned* p, unsigned v) {
  asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_or(unsigned* p, unsigned v) {
  asm volatile("red.global.or.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned atom_add(unsigned* p, unsigned v) {
  unsigned r;
  asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "r"(v) : "memory");
  return r;
}


// Programmatic dependent launch (sm_90+): the kernels of the single-pair (latency) path are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so that the launch of kernel k+1 overlaps the tail of kernel k.
// Every kernel of that path starts with pdl_prologue(): it lets ITS dependent launch right away and then waits until
// the grid it depends on has completed and flushed (griddepcontrol.wait is a no-op for a normally launched kernel).
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---- bulk asynchronous copies global -> shared (TMA engine, sm_90+ / sm_100a; SASS UBLKCP) completing on an mbarrier.
// The scan-2 pass stages the coordinates of a warp tile with three of them (one per plane) issued by one lane: no
// per-lane address arithmetic, no registers held across the load latency.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // visible to the async proxy before the first copy
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// dst / src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// (try_wait suspends the thread in hardware for a bounded time per call.  A copy that never completes -- a bug, not a
// slow device: the limit is 20 s of %globaltimer, far beyond compute-sanitizer / time-sliced GPUs -- traps instead of
// hanging the device.)
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  if (mbar_try_wait(bar, parity)) return;
  unsigned long long t0 = 0;
  for (unsigned spin = 1; !mbar_try_wait(bar, parity); spin++) {
    if ((spin & 1023u) == 0u) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 20000000000ull) __trap();
    }
  }
}

// Shared-memory accesses through explicit 32-bit shared addresses.  The pass kernels run at 64 registers per thread;
// left to itself the compiler REMATERIALISES the address of a warp's scratch (S2R tid, shifts, the CTA's shared window
// base: six instructions, two of them with S2R latency) at every use instead of keeping it in a register.  An address
// that comes out of an opaque asm cannot be recomputed.
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) {
  uint32_t r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

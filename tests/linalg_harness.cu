// tests/linalg_harness.cu -- test kernels around the dense linear algebra of the Gauss-Newton loop.
//
// The library's translation unit is included whole, so the routines under test (icet::eig3f, icet::masked_inv3,
// icet::cod_pinv, icet::jacobi6, solve_pair_warp, k_solve6, vox_algebra_core) are the library's own source text,
// compiled with the library's flags.  tests/test_gpu_linalg.py builds this file into a private shared object and
// calls the extern "C" launchers below through ctypes.  Every launcher takes host arrays, copies them to the device,
// runs one case per thread (per block for the solves), copies the results back and returns a cudaError_t.
#include "../icet_b200/csrc/icet_b200.cu"

namespace {

__global__ void k_t_eig3(const float* A, int n, float* ev, float* V) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) icet::eig3f(A + 9 * i, ev + 3 * i, V + 9 * i);
}

// W = pinv(M) exactly as vox_algebra_core forms it; branch: 1 = closed form (masked_inv3), 0 = cod_pinv
__global__ void k_t_wpinv(const double* M, const int* mask, int n, double* W, int* branch) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double m[9], w[9];
  for (int k = 0; k < 9; k++) m[k] = M[9 * i + k];
  const bool closed = icet::masked_inv3(m, mask[i], w);
  if (!closed) icet::cod_pinv(m, 3, 3, w);
  for (int k = 0; k < 9; k++) W[9 * i + k] = w[k];
  branch[i] = closed ? 1 : 0;
}

__global__ void k_t_cod(const double* A, int rows, int cols, int n, double* P, int* rank) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) rank[i] = icet::cod_pinv(A + 36 * i, rows, cols, P + 36 * i);
}

__global__ void k_t_jacobi(const double* A, int n, double* ev, double* U) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) icet::jacobi6(A + 36 * i, ev + 6 * i, U + 36 * i);
}

// the tail of cluster_solve_phase (kernels_cluster.cuh): the warp solve, one thread's solve_pair when it declines
__global__ void k_t_solve_cluster(const Chunk ck, const double* tot) {
  const int pair = blockIdx.x;
  const double* t = tot + (size_t)NRED * pair;
  bool done = false;
  if (!(ck.flags & ICET_B200_FLAG_FULL_EIG)) done = solve_pair_warp(ck, pair, 0, t);
  if (!done && threadIdx.x == 0) solve_pair(ck, pair, 0, t);
}

__global__ void k_t_vox(const Vox1* vox, const double* mean, const double* cov, const long long* nbin, const float* Jm,
                        int n, double* acc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Chunk ck{};  // dump_on = 0: vox_algebra_core reads nothing else of the chunk when the voxel record is passed in
  double a[NRED];
  for (int k = 0; k < NRED; k++) a[k] = 0.0;
  vox_algebra_core(ck, 0, i, 0, Jm + 27 * i, nbin[i], mean + 3 * i, cov + 6 * i, a, vox + i);
  for (int k = 0; k < NRED; k++) acc[(size_t)NRED * i + k] = a[k];
}

// device copies of the launchers' arguments, freed on every return path
struct Dev {
  std::vector<void*> ptrs;
  ~Dev() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T>
  T* in(const T* host, size_t count) {
    void* p = nullptr;
    if (cudaMalloc(&p, count * sizeof(T) + 16) != cudaSuccess) return nullptr;
    ptrs.push_back(p);
    if (host && cudaMemcpy(p, host, count * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
    if (!host && cudaMemset(p, 0, count * sizeof(T)) != cudaSuccess) return nullptr;
    return static_cast<T*>(p);
  }
};
template <class T>
int out(T* host, const T* dev, size_t count) {
  return (int)cudaMemcpy(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost);
}
int finish() {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  return (int)cudaDeviceSynchronize();
}
#define NEED(p) \
  if (!(p)) return (int)cudaErrorMemoryAllocation
int blocks(int n) { return (n + 127) / 128; }

// k_solve6 (split loop) or the cluster form on npairs independent 1-iteration chunks: tot [npairs][28] are the
// voxel sums, X [npairs][6] the transform each solve starts from.  Returns the result records, TR and J.
int run_solve(int cluster, const double* tot, const float* X, int flags, int npairs, void* res, float* TR, float* J) {
  if (npairs <= 0) return 0;
  Dev d;
  Chunk ck{};
  ck.npairs = npairs;
  ck.runlen = 1;
  ck.flags = flags;
  ck.dump_on = 0;
  double* dtot = d.in(tot, (size_t)npairs * NRED);
  NEED(dtot);
  NEED(ck.X = d.in(X, (size_t)npairs * 6));
  NEED(ck.TR = d.in<float>(nullptr, (size_t)npairs * 12));
  NEED(ck.TRprev = d.in<float>(nullptr, (size_t)npairs * 12));
  NEED(ck.J = d.in<float>(nullptr, (size_t)npairs * 27));
  NEED(ck.pm = d.in<PairMode>(nullptr, (size_t)npairs));
  NEED(ck.res = d.in<icet_b200_result>(nullptr, (size_t)npairs));
  if (cluster) {
    k_t_solve_cluster<<<npairs, 32>>>(ck, dtot);
  } else {
    ck.part = dtot;  // one partial block per pair: k_solve6 adds it to 0.0
    k_solve6<<<npairs, SOLVE_THREADS>>>(ck, 0, 1);
  }
  int e = finish();
  if (e) return e;
  if ((e = out(static_cast<icet_b200_result*>(res), ck.res, (size_t)npairs))) return e;
  if ((e = out(TR, ck.TR, (size_t)npairs * 12))) return e;
  return out(J, ck.J, (size_t)npairs * 27);
}

}  // namespace

extern "C" {

int lh_result_size(void) { return (int)sizeof(icet_b200_result); }
int lh_vox1_size(void) { return (int)sizeof(Vox1); }

int lh_eig3(const float* A, int n, float* ev, float* V) {
  if (n <= 0) return 0;
  Dev d;
  const float* dA = d.in(A, 9 * (size_t)n);
  float* dev = d.in<float>(nullptr, 3 * (size_t)n);
  float* dV = d.in<float>(nullptr, 9 * (size_t)n);
  NEED(dA && dev && dV);
  k_t_eig3<<<blocks(n), 128>>>(dA, n, dev, dV);
  int e = finish();
  if (e || (e = out(ev, dev, 3 * (size_t)n))) return e;
  return out(V, dV, 9 * (size_t)n);
}

int lh_wpinv(const double* M, const int* mask, int n, double* W, int* branch) {
  if (n <= 0) return 0;
  Dev d;
  const double* dM = d.in(M, 9 * (size_t)n);
  const int* dmask = d.in(mask, (size_t)n);
  double* dW = d.in<double>(nullptr, 9 * (size_t)n);
  int* db = d.in<int>(nullptr, (size_t)n);
  NEED(dM && dmask && dW && db);
  k_t_wpinv<<<blocks(n), 128>>>(dM, dmask, n, dW, db);
  int e = finish();
  if (e || (e = out(W, dW, 9 * (size_t)n))) return e;
  return out(branch, db, (size_t)n);
}

int lh_cod(const double* A, int rows, int cols, int n, double* P, int* rank) {
  if (n <= 0) return 0;
  if (rows < 1 || cols < 1 || rows > 6 || cols > 6) return (int)cudaErrorInvalidValue;
  Dev d;
  const double* dA = d.in(A, 36 * (size_t)n);
  double* dP = d.in<double>(nullptr, 36 * (size_t)n);
  int* dr = d.in<int>(nullptr, (size_t)n);
  NEED(dA && dP && dr);
  k_t_cod<<<blocks(n), 128>>>(dA, rows, cols, n, dP, dr);
  int e = finish();
  if (e || (e = out(P, dP, 36 * (size_t)n))) return e;
  return out(rank, dr, (size_t)n);
}

int lh_jacobi(const double* A, int n, double* ev, double* U) {
  if (n <= 0) return 0;
  Dev d;
  const double* dA = d.in(A, 36 * (size_t)n);
  double* dev = d.in<double>(nullptr, 6 * (size_t)n);
  double* dU = d.in<double>(nullptr, 36 * (size_t)n);
  NEED(dA && dev && dU);
  k_t_jacobi<<<blocks(n), 128>>>(dA, n, dev, dU);
  int e = finish();
  if (e || (e = out(ev, dev, 6 * (size_t)n))) return e;
  return out(U, dU, 36 * (size_t)n);
}

int lh_solve_split(const double* tot, const float* X, int flags, int npairs, void* res, float* TR, float* J) {
  return run_solve(0, tot, X, flags, npairs, res, TR, J);
}

int lh_solve_cluster(const double* tot, const float* X, int flags, int npairs, void* res, float* TR, float* J) {
  return run_solve(1, tot, X, flags, npairs, res, TR, J);
}

int lh_vox(const void* vox, const double* mean, const double* cov, const long long* nbin, const float* Jm, int n,
           double* acc) {
  if (n <= 0) return 0;
  Dev d;
  const Vox1* dv = d.in(static_cast<const Vox1*>(vox), (size_t)n);
  const double* dm = d.in(mean, 3 * (size_t)n);
  const double* dc = d.in(cov, 6 * (size_t)n);
  const long long* dn = d.in(nbin, (size_t)n);
  const float* dJ = d.in(Jm, 27 * (size_t)n);
  double* da = d.in<double>(nullptr, (size_t)NRED * n);
  NEED(dv && dm && dc && dn && dJ && da);
  k_t_vox<<<blocks(n), 128>>>(dv, dm, dc, dn, dJ, n, da);
  const int e = finish();
  if (e) return e;
  return out(acc, da, (size_t)NRED * n);
}

}  // extern "C"

// icet_b200/csrc/icet_b200.cu -- sm_100a kernels and the C ABI (include/icet_b200.h) of the
// B200-native ICET registration hot path.
//
// Replaces the work of the reference constructor ICET::ICET (src/icet.cpp:29-63):
//   fitScan1  (:68-107)  -> k_scan1_bin, k_cell_scan, k_scatter, k_cluster, k_pass<false>, k_fit1
//   prepScan2 (:254-277) -> k_prep2
//   fitScan2  (:372-436) -> per iteration: k_pass<true>, k_vox2, k_solve6 (batches), or all iterations in the
//                           persistent k_loop (single pairs, chained pairs)
// All pairs of a chunk advance together through these kernels (bulk-synchronous over the batch),
// everything stays on the device between iterations; the host only enqueues.
// callers.cuh / callers_abi.inl (included below) hold the thin callers around the path: range filter, pose
// bookkeeping, FIFO map, cloud re-expression, ingest.
//
// Determinism: per-voxel statistics are accumulated as 64-bit fixed-point integers (run sums in registers, then
// RED.64 to L2), so results do not depend on thread / block / GPU partitioning or on atomic ordering.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/icet_b200.h"
#include "icet_math.cuh"
#include "synth.h"

namespace {

#include "chunk.cuh"
#include "kernels_scan1.cuh"
#include "kernels_pass.cuh"
#include "kernels_pass2.cuh"
#include "kernels_loop.cuh"
#include "kernels_cluster.cuh"
#include "runtime.inl"
#include "callers.cuh"
#include "kernels_kfnode.cuh"

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int icet_b200_version(void) { return ICET_B200_VERSION; }
const char* icet_b200_last_error(void) { return g_err.c_str(); }

int icet_b200_create(int device, icet_b200_ctx** out) {
  if (!out) return fail(ICET_B200_E_INVALID, "ctx out-pointer is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail(ICET_B200_E_NODEVICE, std::string("no CUDA device available (") +
                                          (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                                          "); icet_b200 has no CPU fallback");
  }
  if (device < 0) CK(cudaGetDevice(&device));
  if (device >= ndev) return fail(ICET_B200_E_INVALID, "device index out of range");
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(ICET_B200_E_NODEVICE, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                                          std::to_string(prop.minor) + "; this library is built for sm_100a only");
  CK(cudaSetDevice(device));
  Building<icet_b200_ctx> c(new icet_b200_ctx(), icet_b200_destroy);
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("ICET_B200_LOOP_TIMEOUT_MS")) {
    const long long ms = atoll(e);
    if (ms > 0) c->loop_timeout_ns = (unsigned long long)ms * 1000000ull;
  }
  if (const char* e = getenv("ICET_B200_FIRST_TILES")) c->first_tiles_wide = atoi(e) != 0;
  if (const char* e = getenv("ICET_B200_CLUSTER_HELPERS")) { const int v = atoi(e); if (v >= 0 && v <= 8) c->cluster_helpers = v; }
  if (const char* e = getenv("ICET_B200_INC_SA")) { const double v = atof(e); if (v > 0 && v <= 4e-3) c->inc_max_sa = (float)v; }
  if (const char* e = getenv("ICET_B200_INC_SB")) { const double v = atof(e); if (v > 0 && v <= 0.15) c->inc_max_sb = (float)v; }
  CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (int l = 1; l < ICET_NLANE; l++) {
    CK(cudaStreamCreateWithFlags(&c->lanes[l], cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&c->ev_join[l], cudaEventDisableTiming));
  }
  for (int l = 0; l < ICET_NLANE; l++) CK(cudaEventCreateWithFlags(&c->ev_lane[l], cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  for (int k = 0; k < 2; k++) CK(cudaEventCreateWithFlags(&c->ev_aux[k], cudaEventDisableTiming));
  for (int i = 0; i < ICET_NSLOT; i++) {
    CK(cudaEventCreateWithFlags(&c->ev_copy[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
  }
  *out = c.release();
  return 0;
}

int icet_b200_destroy(icet_b200_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  for (int l = 1; l < ICET_NLANE; l++)
    if (c->lanes[l]) cudaStreamSynchronize(c->lanes[l]);
  for (int i = 0; i < ICET_NSLOT; i++) {
    if (c->ev_copy[i]) cudaEventDestroy(c->ev_copy[i]);
    if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
  }
  for (cudaEvent_t e : c->prof_ev) cudaEventDestroy(e);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (int l = 1; l < ICET_NLANE; l++) {
    if (c->lanes[l]) cudaStreamDestroy(c->lanes[l]);
    if (c->ev_join[l]) cudaEventDestroy(c->ev_join[l]);
  }
  for (int l = 0; l < ICET_NLANE; l++)
    if (c->ev_lane[l]) cudaEventDestroy(c->ev_lane[l]);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  for (int k = 0; k < 2; k++)
    if (c->ev_aux[k]) cudaEventDestroy(c->ev_aux[k]);
  delete c;
  return 0;
}

int icet_b200_set_stream(icet_b200_ctx* c, void* stream) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)stream;
  c->own_stream = false;
  return 0;
}

int icet_b200_set_chunk(icet_b200_ctx* c, int32_t m) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (m < 0) return fail(ICET_B200_E_INVALID, "chunk must be >= 0");
  c->chunk_pairs = m == 0 ? ICET_DEFAULT_CHUNK : std::min(m, 65535);
  return 0;
}

int icet_b200_set_host_chunk(icet_b200_ctx* c, int32_t m) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (m < 0) return fail(ICET_B200_E_INVALID, "chunk must be >= 0");
  c->host_chunk = m == 0 ? 64 : std::min(m, 65535);
  return 0;
}

int icet_b200_synchronize(icet_b200_ctx* c) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  for (int l = 1; l < ICET_NLANE; l++) CK(cudaStreamSynchronize(c->lanes[l]));
  return 0;
}

int icet_b200_set_lanes(icet_b200_ctx* c, int32_t n) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (n < 0 || n > ICET_NLANE) return fail(ICET_B200_E_INVALID, "lanes must be 0 (default) .. 8");
  c->nlanes = n == 0 ? c->nlanes_default : n;
  return 0;
}

int64_t icet_b200_kernel_launches(icet_b200_ctx* c) { return c ? c->launches : 0; }

// (k_kf_attach, the scan-1 set-up of a keyframe chunk, is counted under id 1: it does k_cell_scan's per-pair
// initialisation)
static const char* const k_names[ICET_B200_NKERNELS] = {"k_scan1_bin", "k_cell_scan", "k_scatter", "k_cluster",
                                                        "k_pass<scan1>", "k_fit1", "k_prep2", "k_pass<scan2>",
                                                        "k_vox2", "k_solve6", "k_loop"};
const char* icet_b200_kernel_name(int id) { return (id >= 0 && id < ICET_B200_NKERNELS) ? k_names[id] : ""; }

static int prof_collect(icet_b200_ctx* c) {
  CK(cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i < c->prof_id.size(); i++) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, c->prof_ev[2 * i], c->prof_ev[2 * i + 1]));
    c->prof_ms[c->prof_id[i]] += ms;
    c->prof_n[c->prof_id[i]]++;
  }
  c->prof_id.clear();
  c->prof_used = 0;
  return 0;
}

int icet_b200_set_profile(icet_b200_ctx* c, int32_t enable) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  CK(cudaSetDevice(c->device));
  int rc = prof_collect(c);
  if (rc) return rc;
  if (enable && !c->profile_on)
    for (int k = 0; k < ICET_B200_NKERNELS; k++) { c->prof_ms[k] = 0.0; c->prof_n[k] = 0; }
  c->profile_on = enable ? 1 : 0;
  return 0;
}

int icet_b200_get_profile(icet_b200_ctx* c, double* ms, int64_t* launches) {
  if (!c || !ms || !launches) return fail(ICET_B200_E_INVALID, "NULL argument");
  CK(cudaSetDevice(c->device));
  int rc = prof_collect(c);
  if (rc) return rc;
  for (int k = 0; k < ICET_B200_NKERNELS; k++) { ms[k] = c->prof_ms[k]; launches[k] = c->prof_n[k]; }
  return 0;
}

int icet_b200_set_dump(icet_b200_ctx* c, int32_t enable) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  c->dump_on = enable ? 1 : 0;
  if (!enable) c->dump_valid = false;
  return 0;
}

// -- device-resident batch --------------------------------------------------------------------
// The pair arrays of a batch: present, and every pair with sizes >= 0 and a scan wherever it has points.  Without
// scan 1 (with_scan1 false: a batch against a keyframe) scan1 and n1 are not read.
static int check_pairs(int32_t npairs, bool with_scan1, const float* const* scan1, const int32_t* n1,
                       const float* const* scan2, const int32_t* n2, const icet_b200_result* out) {
  if (npairs < 0 || (npairs > 0 && ((with_scan1 && (!scan1 || !n1)) || !scan2 || !n2 || !out)))
    return fail(ICET_B200_E_INVALID, "NULL argument");
  for (int i = 0; i < npairs; i++)
    if ((with_scan1 && (n1[i] < 0 || (n1[i] > 0 && !scan1[i]))) || n2[i] < 0 || (n2[i] > 0 && !scan2[i]))
      return fail(ICET_B200_E_INVALID, "bad scan pointer / size in pair " + std::to_string(i));
  return 0;
}

static int batch_device_impl(icet_b200_ctx* c, const icet_b200_params* p, int32_t npairs, const PairDesc* h_desc,
                             const float* d_x0, icet_b200_result* d_out, bool dump, const PairDesc* d_desc_all = nullptr,
                             int nmax_dev = 0, const icet_b200_keyframe* kf = nullptr) {
  // h_desc lives in host memory; descriptors are uploaded per chunk through the pinned bounce buffer.
  // d_desc_all (callers layer): the descriptors are already on the device -- built there, with data-dependent
  // sizes no larger than nmax_dev -- and h_desc is not read.
  // kf: scan 1 of every pair is this keyframe (the descriptors hold no scan 1).
  int rc = c->pinned.ensure((size_t)std::min(npairs, c->chunk_pairs) * sizeof(PairDesc) * ICET_NLANE + 4096);
  if (rc) return rc;
  // consecutive chunks alternate between the two compute lanes (own stream + workspace each); lane 1 starts after
  // everything already queued on the caller's stream and the caller's stream resumes after lane 1
  const bool chain = (p->flags & ICET_B200_FLAG_CHAIN_X0) != 0;  // chunks depend on each other: one lane, in order
  // Chunk size: the configured bound, but small enough that every lane gets a chunk (not below 64 pairs): with all
  // lanes busy the latency-bound kernels at the end of each iteration of one chunk hide behind the pass kernels of
  // the others (measured at 512 pairs: 2 x 256 -> 66.9 k pairs/s, 4 x 128 -> 69.1 k).
  // (Chunks as large as four lanes allow -- 512-pair launches run 1.3 % faster than 256-pair ones -- and only then more
  // lanes: a 4096-pair batch runs as 8 chunks on 8 lanes, a 2048-pair batch as 4 chunks on 4.)
  const int lane_div = std::min(c->nlanes, 4);
  const int chunk_pairs = (c->nlanes > 1 && !dump && !chain)
                              ? std::min(c->chunk_pairs, std::max(64, (npairs + lane_div - 1) / lane_div))
                              : c->chunk_pairs;
  const int nchunks = (npairs + chunk_pairs - 1) / chunk_pairs;
  const int nl = (c->nlanes > 1 && nchunks > 1 && !dump && !chain) ? std::min(c->nlanes, nchunks) : 1;
  if (nl > 1) {
    CK(cudaEventRecord(c->ev_fork, c->stream));
    for (int l = 1; l < nl; l++) CK(cudaStreamWaitEvent(c->lanes[l], c->ev_fork, 0));
  }
  int chunk_no = 0;
  for (int base = 0; base < npairs; base += chunk_pairs, chunk_no++) {
    const int P = std::min(chunk_pairs, npairs - base);
    const int lane = chunk_no % nl;
    const int slot = lane;  // descriptors of a lane are reused in stream order
    cudaStream_t st = lane == 0 ? c->stream : c->lanes[lane];
    int n1max = nmax_dev, n2max = nmax_dev;
    const PairDesc* d_desc = d_desc_all ? d_desc_all + base : nullptr;
    if (!d_desc) {
      for (int i = 0; i < P; i++) {
        n1max = std::max(n1max, h_desc[base + i].n1);
        n2max = std::max(n2max, h_desc[base + i].n2);
      }
      // (the device buffer may grow: everything the lane has queued must be done with the old one first)
      if ((size_t)P * sizeof(PairDesc) > c->lane_desc[slot].cap) CK(cudaStreamSynchronize(st));
      rc = c->lane_desc[slot].ensure((size_t)P * sizeof(PairDesc));
      if (rc) return rc;
      // the pinned part of this lane may still be in flight from its previous chunk
      CK(cudaEventSynchronize(c->ev_lane[slot]));
      PairDesc* hp = (PairDesc*)c->pinned.p + (size_t)slot * std::min(npairs, c->chunk_pairs);
      memcpy(hp, h_desc + base, (size_t)P * sizeof(PairDesc));
      CK(cudaMemcpyAsync(c->lane_desc[slot].p, hp, (size_t)P * sizeof(PairDesc), cudaMemcpyHostToDevice, st));
      CK(cudaEventRecord(c->ev_lane[slot], st));
      d_desc = (const PairDesc*)c->lane_desc[slot].p;
    }
    const float* x0c = d_x0 ? d_x0 + (chain ? 0 : (size_t)base * 6) : nullptr;
    if (chain && base > 0) x0c = d_out[base - 1].X;  // stream order: the previous chunk has finished by then
    rc = run_chunk(c, p, P, d_desc, n1max, n2max, x0c, d_out + base, dump, lane, kf);
    if (rc) return rc;
  }
  for (int l = 1; l < nl; l++) {
    CK(cudaEventRecord(c->ev_join[l], c->lanes[l]));
    CK(cudaStreamWaitEvent(c->stream, c->ev_join[l], 0));
  }
  return 0;
}

int icet_b200_register_batch_device(icet_b200_ctx* c, const icet_b200_params* p, int32_t npairs,
                                    const float* const* scan1, const int32_t* n1, const float* const* scan2,
                                    const int32_t* n2, const float* x0, icet_b200_result* out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  int rc = validate(p);
  if (!rc) rc = check_pairs(npairs, true, scan1, n1, scan2, n2, out);
  if (rc) return rc;
  if (npairs == 0) return 0;
  CK(cudaSetDevice(c->device));
  std::vector<PairDesc> d(npairs);
  for (int i = 0; i < npairs; i++) d[i] = PairDesc{scan1[i], scan2[i], n1[i], n1[i], n2[i], n2[i]};
  return batch_device_impl(c, p, npairs, d.data(), x0, out, false);
}

int icet_b200_register_sequence_device(icet_b200_ctx* c, const icet_b200_params* p, int32_t nscans,
                                       const float* scans, int32_t n, icet_b200_result* out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  int rc = validate(p);
  if (rc) return rc;
  if (nscans < 1 || n < 0 || !scans || (nscans > 1 && !out)) return fail(ICET_B200_E_INVALID, "bad argument");
  if (nscans == 1) return 0;
  CK(cudaSetDevice(c->device));
  std::vector<PairDesc> d(nscans - 1);
  for (int i = 0; i < nscans - 1; i++)
    d[i] = PairDesc{scans + (size_t)i * 3 * n, scans + (size_t)(i + 1) * 3 * n, n, n, n, n};
  return batch_device_impl(c, p, nscans - 1, d.data(), nullptr, out, false);
}

// -- host-buffer entry points ------------------------------------------------------------------
int icet_b200_register_batch(icet_b200_ctx* c, const icet_b200_params* p, int32_t npairs,
                             const float* const* scan1, const int32_t* n1, const float* const* scan2,
                             const int32_t* n2, const float* x0, icet_b200_result* out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  int rc = validate(p);
  if (!rc) rc = check_pairs(npairs, true, scan1, n1, scan2, n2, out);
  if (rc) return rc;
  if (npairs == 0) return 0;
  CK(cudaSetDevice(c->device));
  rc = c->resbuf.ensure((size_t)npairs * sizeof(icet_b200_result));
  if (rc) return rc;
  icet_b200_result* d_res = (icet_b200_result*)c->resbuf.p;
  // Upload/compute pipeline: the batch is cut into chunks; chunk k+1 is uploaded (copy stream) while chunk k is
  // registered (compute stream).  The link is the bottleneck at 64-channel size (1.5 MB per scan over PCIe against
  // ~25 us of GPU time per pair), so the chunks are small (host_chunk pairs) and ramp up from / down to an eighth of
  // that: the first upload and the last registration are the only parts that nothing overlaps.
  const int CH = std::max(1, std::min(c->chunk_pairs, c->host_chunk));
  std::vector<int> sizes;
  {
    int left = npairs;
    std::vector<int> head, tail;
    for (int s = std::max(1, CH / 8); s < CH && left > 2 * CH; s *= 2) {
      head.push_back(s);
      tail.push_back(s);
      left -= 2 * s;
    }
    sizes = head;
    while (left > 0) {
      const int s = std::min(CH, left);
      sizes.push_back(s);
      left -= s;
    }
    for (size_t k = tail.size(); k-- > 0;) sizes.push_back(tail[k]);
  }
  const size_t pin_slot = (size_t)CH * (sizeof(PairDesc) + 6 * sizeof(float)) + 2048;
  rc = c->pinned.ensure(pin_slot * ICET_NSLOT + 4096);
  if (rc) return rc;
  auto pad = [](size_t f) { return (f + 63) & ~(size_t)63; };
  int base = 0;
  const float* prev_scan2_dev = nullptr;  // device copy of the previous chunk's last scan 2
  const bool chain = (p->flags & ICET_B200_FLAG_CHAIN_X0) != 0;  // chunks depend on each other: one lane, in order
  // (the host pipeline is bound by the link, two lanes are plenty)
  const bool two = c->nlanes > 1 && sizes.size() > 1 && !(c->dump_on && npairs == 1) && !chain;
  if (two) {
    CK(cudaEventRecord(c->ev_fork, c->stream));
    CK(cudaStreamWaitEvent(c->lanes[1], c->ev_fork, 0));
  }
  for (size_t k = 0; k < sizes.size(); base += sizes[k], k++) {
    const int P = sizes[k];
    const int slot = (int)(k % ICET_NSLOT);
    // plan the staging area: a scan shared by consecutive pairs (scan2[g-1] == scan1[g]) is uploaded once, also
    // across the chunk boundary (the previous chunk's staging slot is still intact, see the waits below)
    std::vector<PairDesc> d(P);
    std::vector<size_t> off1(P), off2(P);
    std::vector<char> up1(P);
    size_t floats = 0;
    int n1max = 0, n2max = 0;
    for (int i = 0; i < P; i++) {
      const int g = base + i;
      const bool shared = g > 0 && scan1[g] == scan2[g - 1] && n1[g] == n2[g - 1] && (i > 0 || prev_scan2_dev);
      up1[i] = !shared;
      if (shared) {
        off1[i] = (i > 0) ? off2[i - 1] : (size_t)-1;
      } else {
        off1[i] = floats;
        floats += pad((size_t)3 * n1[g]);
      }
      off2[i] = floats;
      floats += pad((size_t)3 * n2[g]);
      n1max = std::max(n1max, n1[g]);
      n2max = std::max(n2max, n2[g]);
    }
    // Slot reuse: this slot last held chunk k - NSLOT; chunk k - NSLOT + 1 may still read its last scan (shared
    // across the boundary), so wait for THAT chunk's registration before overwriting.
    CK(cudaEventSynchronize(c->ev_done[slot]));
    CK(cudaEventSynchronize(c->ev_done[(slot + 1) % ICET_NSLOT]));
    rc = c->stage[slot].ensure(floats * sizeof(float));
    if (rc) return rc;
    rc = c->descbuf[slot].ensure((size_t)CH * sizeof(PairDesc));
    if (rc) return rc;
    rc = c->x0buf[slot].ensure((size_t)CH * 6 * sizeof(float));
    if (rc) return rc;
    float* sbase = (float*)c->stage[slot].p;
    // uploads; runs that are contiguous on both sides are merged into one copy
    const float* run_src = nullptr;
    float* run_dst = nullptr;
    size_t run_floats = 0;
    auto flush = [&]() -> int {
      if (run_floats)
        CK(cudaMemcpyAsync(run_dst, run_src, run_floats * sizeof(float), cudaMemcpyHostToDevice, c->copy_stream));
      run_floats = 0;
      return 0;
    };
    auto upload = [&](const float* src, float* dst, size_t nf) -> int {
      if (nf == 0) return 0;
      if (run_floats && src == run_src + run_floats && dst == run_dst + run_floats) {
        run_floats += nf;
        return 0;
      }
      int r = flush();
      if (r) return r;
      run_src = src;
      run_dst = dst;
      run_floats = nf;
      return 0;
    };
    for (int i = 0; i < P; i++) {
      const int g = base + i;
      if (up1[i]) {
        rc = upload(scan1[g], sbase + off1[i], (size_t)3 * n1[g]);
        if (rc) return rc;
      }
      rc = upload(scan2[g], sbase + off2[i], (size_t)3 * n2[g]);
      if (rc) return rc;
      const float* s1p = up1[i] ? sbase + off1[i] : (i > 0 ? sbase + off2[i - 1] : prev_scan2_dev);
      d[i] = PairDesc{s1p, sbase + off2[i], n1[g], n1[g], n2[g], n2[g]};
    }
    rc = flush();
    if (rc) return rc;
    prev_scan2_dev = sbase + off2[P - 1];
    char* hp = (char*)c->pinned.p + (size_t)slot * pin_slot;
    memcpy(hp, d.data(), (size_t)P * sizeof(PairDesc));
    CK(cudaMemcpyAsync(c->descbuf[slot].p, hp, (size_t)P * sizeof(PairDesc), cudaMemcpyHostToDevice, c->copy_stream));
    const float* d_x0 = nullptr;
    if (chain && base > 0) {
      d_x0 = d_res[base - 1].X;  // the previous chunk's last solution (same stream, already ordered)
    } else if (x0) {
      const size_t nx = chain ? 6 : (size_t)P * 6;  // chained: one seed, that of pair 0
      float* hx = (float*)(hp + (size_t)CH * sizeof(PairDesc));
      memcpy(hx, x0 + (size_t)base * 6, nx * sizeof(float));
      CK(cudaMemcpyAsync(c->x0buf[slot].p, hx, nx * sizeof(float), cudaMemcpyHostToDevice, c->copy_stream));
      d_x0 = (const float*)c->x0buf[slot].p;
    }
    CK(cudaEventRecord(c->ev_copy[slot], c->copy_stream));
    const int lane = two ? (int)(k & 1) : 0;
    cudaStream_t lst = lane == 0 ? c->stream : c->lanes[1];
    CK(cudaStreamWaitEvent(lst, c->ev_copy[slot], 0));
    const bool dump = c->dump_on && npairs == 1;
    if (dump) {
      rc = ensure_dump(c, p);
      if (rc) return rc;
    }
    rc = run_chunk(c, p, P, (const PairDesc*)c->descbuf[slot].p, n1max, n2max, d_x0, d_res + base, dump, lane);
    if (rc) return rc;
    CK(cudaEventRecord(c->ev_done[slot], lst));
    if (dump) {
      c->dump_params = *p;
      c->dump_valid = true;
    }
    if (npairs == 1) {
      c->last_n2 = n2[0];
      c->last_valid = true;
    }
  }
  if (two) {
    CK(cudaEventRecord(c->ev_join[1], c->lanes[1]));
    CK(cudaStreamWaitEvent(c->stream, c->ev_join[1], 0));
  }
  CK(cudaMemcpyAsync(out, d_res, (size_t)npairs * sizeof(icet_b200_result), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return check_loop_watchdog(c);
}

int icet_b200_register(icet_b200_ctx* c, const icet_b200_params* p, const float* scan1, int32_t n1, int32_t ld1,
                       const float* scan2, int32_t n2, int32_t ld2, const float x0[6], icet_b200_result* out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (!out) return fail(ICET_B200_E_INVALID, "out is NULL");
  if (n1 < 0 || n2 < 0 || ld1 < n1 || ld2 < n2) return fail(ICET_B200_E_INVALID, "bad n / ld");
  if (ld1 == n1 && ld2 == n2) return icet_b200_register_batch(c, p, 1, &scan1, &n1, &scan2, &n2, x0, out);
  // general leading dimension: pack the three planes on the host side of the copy
  std::vector<float> a((size_t)3 * n1), b((size_t)3 * n2);
  for (int k = 0; k < 3; k++) {
    if (n1) memcpy(a.data() + (size_t)k * n1, scan1 + (size_t)k * ld1, (size_t)n1 * sizeof(float));
    if (n2) memcpy(b.data() + (size_t)k * n2, scan2 + (size_t)k * ld2, (size_t)n2 * sizeof(float));
  }
  const float* pa = a.data();
  const float* pb = b.data();
  return icet_b200_register_batch(c, p, 1, &pa, &n1, &pb, &n2, x0, out);
}

// -- keyframes -----------------------------------------------------------------------------------
// A registration's params must describe the keyframe's scan-1 fit.
static int keyframe_params(const icet_b200_keyframe* kf, const icet_b200_params* p) {
  if (!kf) return fail(ICET_B200_E_INVALID, "keyframe is NULL");
  int rc = validate(p);
  if (rc) return rc;
  const icet_b200_params& k = kf->p;
  if (p->bins_phi != k.bins_phi) return fail(ICET_B200_E_INVALID, "bins_phi differs from the keyframe's");
  if (p->bins_theta != k.bins_theta) return fail(ICET_B200_E_INVALID, "bins_theta differs from the keyframe's");
  if (p->n != k.n) return fail(ICET_B200_E_INVALID, "n differs from the keyframe's");
  if (p->thresh != k.thresh) return fail(ICET_B200_E_INVALID, "thresh differs from the keyframe's");
  if (p->buff != k.buff) return fail(ICET_B200_E_INVALID, "buff differs from the keyframe's");
  if ((p->flags ^ k.flags) & ICET_B200_FLAG_SHIPPED_ORDER)
    return fail(ICET_B200_E_INVALID, "ICET_B200_FLAG_SHIPPED_ORDER differs from the keyframe's");
  if (p->flags & ICET_B200_FLAG_CHAIN_X0)
    return fail(ICET_B200_E_INVALID, "ICET_B200_FLAG_CHAIN_X0 is not supported against a keyframe");
  return 0;
}

// Copies a HOST cloud (planes, leading dimension ld) into n-strided DEVICE planes at dst, on the context's stream.
static int upload_cloud(icet_b200_ctx* c, float* dst, const float* src, int32_t n, int32_t ld) {
  if (n == 0) return 0;
  if (ld == n)
    CK(cudaMemcpyAsync(dst, src, (size_t)3 * n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  else
    CK(cudaMemcpy2DAsync(dst, (size_t)n * sizeof(float), src, (size_t)ld * sizeof(float), (size_t)n * sizeof(float), 3,
                         cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int icet_b200_keyframe_create_device(icet_b200_ctx* c, const icet_b200_params* p, const float* scan1, int32_t n1,
                                     int32_t ld1, icet_b200_keyframe** out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (!out) return fail(ICET_B200_E_INVALID, "keyframe out-pointer is NULL");
  *out = nullptr;
  int rc = validate(p);
  if (rc) return rc;
  if (n1 < 0 || ld1 < n1 || (n1 > 0 && !scan1)) return fail(ICET_B200_E_INVALID, "bad scan1 / n1 / ld1");
  CK(cudaSetDevice(c->device));
  // the scan-1 set-up of one pair without scan 2 or iterations (it also starts the pair's result record)
  icet_b200_params q = *p;
  q.runlen = 0;
  q.flags = p->flags & ICET_B200_FLAG_SHIPPED_ORDER;
  rc = c->pinned.ensure(4096);
  if (rc) return rc;
  rc = c->descbuf[0].ensure(sizeof(PairDesc));
  if (rc) return rc;
  rc = c->resbuf.ensure(sizeof(icet_b200_result));
  if (rc) return rc;
  CK(cudaStreamSynchronize(c->stream));  // the pinned bounce buffer may still feed an earlier upload
  PairDesc* hd = (PairDesc*)c->pinned.p;
  *hd = PairDesc{scan1, nullptr, n1, ld1, 0, 0};
  CK(cudaMemcpyAsync(c->descbuf[0].p, hd, sizeof(PairDesc), cudaMemcpyHostToDevice, c->stream));
  icet_b200_result* d_res = (icet_b200_result*)c->resbuf.p;
  ChunkRun r;
  rc = chunk_setup(c, &q, 1, (const PairDesc*)c->descbuf[0].p, n1, 0, nullptr, d_res, false, 0, r);
  if (!rc) rc = chunk_scan1(r);
  c->last_valid = false;  // lane 0's workspace now holds this chunk
  if (rc) return rc;
  CK(cudaGetLastError());
  Building<icet_b200_keyframe> kf(new icet_b200_keyframe(), icet_b200_keyframe_destroy);
  kf->ctx = c;
  kf->p = q;
  const size_t ncell = (size_t)p->bins_phi * p->bins_theta;
  if ((rc = kf->rec.ensure(ncell * sizeof(CellRec))) || (rc = kf->vox.ensure(ncell * sizeof(Vox1)))) return rc;
  int32_t* h_ng = (int32_t*)((char*)c->pinned.p + 1024);
  cudaError_t e = cudaMemcpyAsync(kf->rec.p, r.ck.rec, ncell * sizeof(CellRec), cudaMemcpyDeviceToDevice, c->stream);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(kf->vox.p, r.ck.vox, ncell * sizeof(Vox1), cudaMemcpyDeviceToDevice, c->stream);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(h_ng, &d_res->n_gauss1, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess) return fail(ICET_B200_E_CUDA, std::string("keyframe copy: ") + cudaGetErrorString(e));
  kf->n_gauss1 = *h_ng;
  *out = kf.release();
  return 0;
}

int icet_b200_keyframe_create(icet_b200_ctx* c, const icet_b200_params* p, const float* scan1, int32_t n1, int32_t ld1,
                              icet_b200_keyframe** out) {
  if (!c) return fail(ICET_B200_E_INVALID, "ctx is NULL");
  if (!out) return fail(ICET_B200_E_INVALID, "keyframe out-pointer is NULL");
  *out = nullptr;
  int rc = validate(p);
  if (rc) return rc;
  if (n1 < 0 || ld1 < n1 || (n1 > 0 && !scan1)) return fail(ICET_B200_E_INVALID, "bad scan1 / n1 / ld1");
  CK(cudaSetDevice(c->device));
  CK(cudaEventSynchronize(c->ev_done[0]));
  rc = c->stage[0].ensure(std::max<size_t>(1, (size_t)3 * n1) * sizeof(float));
  if (rc) return rc;
  float* d_s1 = (float*)c->stage[0].p;
  rc = upload_cloud(c, d_s1, scan1, n1, ld1);
  if (rc) return rc;
  return icet_b200_keyframe_create_device(c, p, d_s1, n1, n1, out);
}

int icet_b200_keyframe_destroy(icet_b200_keyframe* kf) {
  if (!kf) return 0;
  icet_b200_ctx* c = kf->ctx;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (int l = 1; l < ICET_NLANE; l++)
    if (c->lanes[l]) cudaStreamSynchronize(c->lanes[l]);
  delete kf;
  return 0;
}

int icet_b200_keyframe_gaussians(icet_b200_keyframe* kf) {
  if (!kf) return fail(ICET_B200_E_INVALID, "keyframe is NULL");
  return kf->n_gauss1;
}

int icet_b200_register_keyframe(icet_b200_keyframe* kf, const icet_b200_params* p, const float* scan2, int32_t n2,
                                int32_t ld2, const float x0[6], icet_b200_result* out) {
  int rc = keyframe_params(kf, p);
  if (rc) return rc;
  if (!out) return fail(ICET_B200_E_INVALID, "out is NULL");
  if (n2 < 0 || ld2 < n2 || (n2 > 0 && !scan2)) return fail(ICET_B200_E_INVALID, "bad scan2 / n2 / ld2");
  icet_b200_ctx* c = kf->ctx;
  CK(cudaSetDevice(c->device));
  CK(cudaEventSynchronize(c->ev_done[0]));
  rc = c->stage[0].ensure(std::max<size_t>(1, (size_t)3 * n2) * sizeof(float));
  if (rc) return rc;
  rc = c->x0buf[0].ensure(6 * sizeof(float));
  if (rc) return rc;
  rc = c->resbuf.ensure(sizeof(icet_b200_result));
  if (rc) return rc;
  float* d_s2 = (float*)c->stage[0].p;
  rc = upload_cloud(c, d_s2, scan2, n2, ld2);
  if (rc) return rc;
  const float* d_x0 = nullptr;
  if (x0) {  // (straight from the caller's array: the pinned bounce buffer is batch_device_impl's, which may grow it)
    CK(cudaMemcpyAsync(c->x0buf[0].p, x0, 6 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    d_x0 = (const float*)c->x0buf[0].p;
  }
  const PairDesc desc{nullptr, d_s2, 0, 0, n2, n2};
  icet_b200_result* d_res = (icet_b200_result*)c->resbuf.p;
  rc = batch_device_impl(c, p, 1, &desc, d_x0, d_res, false, nullptr, 0, kf);
  if (rc) return rc;
  CK(cudaMemcpyAsync(out, d_res, sizeof(icet_b200_result), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return check_loop_watchdog(c);
}

int icet_b200_register_keyframe_batch_device(icet_b200_keyframe* kf, const icet_b200_params* p, int32_t npairs,
                                             const float* const* scan2, const int32_t* n2, const float* x0,
                                             icet_b200_result* out) {
  int rc = keyframe_params(kf, p);
  if (!rc) rc = check_pairs(npairs, false, nullptr, nullptr, scan2, n2, out);
  if (rc) return rc;
  if (npairs == 0) return 0;
  icet_b200_ctx* c = kf->ctx;
  CK(cudaSetDevice(c->device));
  std::vector<PairDesc> d(npairs);
  for (int i = 0; i < npairs; i++) d[i] = PairDesc{nullptr, scan2[i], 0, 0, n2[i], n2[i]};
  return batch_device_impl(c, p, npairs, d.data(), x0, out, false, nullptr, 0, kf);
}

int icet_b200_get_dump(icet_b200_ctx* c, icet_b200_voxel_dump* o) {
  if (!c || !o) return fail(ICET_B200_E_INVALID, "NULL argument");
  if (!c->dump_valid) return fail(ICET_B200_E_INVALID, "no dump recorded: call icet_b200_set_dump(ctx,1) before icet_b200_register");
  CK(cudaSetDevice(c->device));
  const icet_b200_params& p = c->dump_params;
  const size_t ncell = (size_t)p.bins_phi * p.bins_theta, rl = (size_t)p.runlen;
  const Dump& d = c->dump_ptrs;
  // workspace-resident pieces: cnt1 and the cell records of pair 0
  Chunk ck;
  memset(&ck, 0, sizeof(ck));
  size_t zb;
  // NOTE: the workspace layout of the last (single-pair) chunk
  cudaStream_t st = c->stream;
  CK(cudaStreamSynchronize(st));
  // n1max/n2max only affect arrays behind rec/cnt1, which are carved first
  carve_chunk(c->ws[0].p, 1, (int)ncell, 0, 0, p.runlen, ck, &zb);
  if (o->cnt1) CK(cudaMemcpy(o->cnt1, ck.cnt1, ncell * 4, cudaMemcpyDeviceToHost));
  if (o->bounds) {
    std::vector<CellRec> rec(ncell);
    CK(cudaMemcpy(rec.data(), ck.rec, ncell * sizeof(CellRec), cudaMemcpyDeviceToHost));
    const int nT = p.bins_theta, nP = p.bins_phi;
    for (size_t cidx = 0; cidx < ncell; cidx++) {
      const int t = (int)(cidx % nT), q = (int)(cidx / nT);
      float* b = o->bounds + cidx * 6;
      b[0] = (static_cast<float>(t) / nT) * (2 * M_PI);
      b[1] = (static_cast<float>(t + 1) / nT) * (2 * M_PI);
      b[2] = (static_cast<float>(q) / nP) * (M_PI);
      b[3] = (static_cast<float>(q + 1) / nP) * (M_PI);
      b[4] = rec[cidx].inner;
      b[5] = rec[cidx].outer;
    }
  }
#define CP(dst, src, bytes) if (o->dst) CK(cudaMemcpy(o->dst, d.src, (bytes), cudaMemcpyDeviceToHost))
  CP(nin1, nin1, ncell * 4); CP(has1, has1, ncell); CP(mu1, mu1, ncell * 12); CP(sigma1, sigma1, ncell * 36);
  CP(evec1, evec1, ncell * 36); CP(eval1, eval1, ncell * 12); CP(lmask, lmask, ncell * 3);
  CP(cnt2, cnt2, rl * ncell * 4); CP(nin2, nin2, rl * ncell * 4); CP(used2, used2, rl * ncell);
  CP(mu2, mu2, rl * ncell * 12); CP(sigma2, sigma2, rl * ncell * 36); CP(Xit, Xit, rl * 24);
  CP(HTWH, HTWH, rl * 144); CP(HTWdz, HTWdz, rl * 24); CP(TRit, TRit, rl * 48); CP(testPoints, testpts, ncell * 72);
#undef CP
  return 0;
}

int icet_b200_debug_timeline(icet_b200_ctx* c, uint64_t* out, int32_t runlen) {
  if (!c || !out) return fail(ICET_B200_E_INVALID, "NULL argument");
  if (!c->dump_valid || runlen != c->dump_params.runlen) return fail(ICET_B200_E_INVALID, "no dump recorded");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaMemcpy(out, c->dump_ptrs.tl, ((size_t)runlen * 16 + 6144) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return 0;
}

int icet_b200_get_points2(icet_b200_ctx* c, float* out, int32_t n2) {
  if (!c || !out) return fail(ICET_B200_E_INVALID, "NULL argument");
  if (!c->last_valid) return fail(ICET_B200_E_INVALID, "no single-pair registration to take points2 from");
  if (n2 != c->last_n2) return fail(ICET_B200_E_INVALID, "n2 does not match the last registration");
  if (n2 == 0) return 0;
  CK(cudaSetDevice(c->device));
  Chunk ck;
  memcpy(&ck, c->last_ck, sizeof(Chunk));
  // the staging buffers are idle here: use one for the device-side output
  CK(cudaStreamSynchronize(c->stream));
  int rc = c->resbuf.ensure((size_t)3 * n2 * sizeof(float) + 1024);
  if (rc) return rc;
  float* d_out = (float*)c->resbuf.p;
  k_points2<<<(n2 + 255) / 256, 256, 0, c->stream>>>(ck, n2, d_out);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, d_out, (size_t)3 * n2 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int icet_b200_classify_scan2(icet_b200_ctx* c, int32_t iter, int32_t* cell, uint8_t* in, int32_t n2) {
  if (!c || !cell || !in) return fail(ICET_B200_E_INVALID, "NULL argument");
  if (!c->last_valid || !c->dump_valid) return fail(ICET_B200_E_INVALID, "no dumped single-pair registration to classify");
  if (n2 != c->last_n2) return fail(ICET_B200_E_INVALID, "n2 does not match the last registration");
  if (iter < 0 || iter >= c->dump_params.runlen) return fail(ICET_B200_E_INVALID, "iteration out of range");
  if (n2 == 0) return 0;
  CK(cudaSetDevice(c->device));
  Chunk ck;
  memcpy(&ck, c->last_ck, sizeof(Chunk));
  CK(cudaStreamSynchronize(c->stream));
  int rc = c->resbuf.ensure((size_t)5 * n2 + 1024);
  if (rc) return rc;
  int32_t* d_cell = (int32_t*)c->resbuf.p;
  uint8_t* d_in = (uint8_t*)(d_cell + n2);
  k_classify2<<<(n2 + 255) / 256, 256, 0, c->stream>>>(ck, n2, c->dump_ptrs.TRit + (size_t)iter * 12, d_cell, d_in);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(cell, d_cell, (size_t)n2 * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(in, d_in, (size_t)n2, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int icet_b200_spherical_bins(icet_b200_ctx* c, const icet_b200_params* p, const float* scan, int32_t n, int32_t ld,
                             float* sph, int32_t* cell) {
  if (!c || !scan || !sph || !cell) return fail(ICET_B200_E_INVALID, "NULL argument");
  int rc = validate(p);
  if (rc) return rc;
  if (n <= 0 || ld < n) return fail(ICET_B200_E_INVALID, "bad n / ld");
  CK(cudaSetDevice(c->device));
  rc = c->stage[0].ensure(((size_t)3 * ld + 3 * (size_t)n + n) * 4);
  if (rc) return rc;
  CK(cudaEventSynchronize(c->ev_done[0]));
  float* d_s = (float*)c->stage[0].p;
  float* d_sph = d_s + (size_t)3 * ld;
  int32_t* d_cell = (int32_t*)(d_sph + (size_t)3 * n);
  CK(cudaMemcpyAsync(d_s, scan, (size_t)3 * ld * 4, cudaMemcpyHostToDevice, c->stream));
  rc = ensure_edges(c, p->bins_theta, p->bins_phi);
  if (rc) return rc;
  const float *azE, *elE;
  icet::BinTable bth, bph;
  fill_tables(c, p->bins_theta, p->bins_phi, &azE, &elE, &bth, &bph);
  k_sph_bins<<<(n + 255) / 256, 256, 0, c->stream>>>(d_s, n, ld, p->bins_theta, p->bins_phi, bth, bph, d_sph, d_cell);
  c->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(sph, d_sph, (size_t)3 * n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(cell, d_cell, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int icet_b200_synth_scans_device(icet_b200_ctx* c, uint64_t seed, int32_t first_scan, int32_t nscans, int32_t rings,
                                 int32_t azim, float* out) {
  if (!c || !out) return fail(ICET_B200_E_INVALID, "NULL argument");
  if (first_scan < 0 || nscans < 1 || rings < 1 || azim < 1) return fail(ICET_B200_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  // poses of scans first_scan .. first_scan+nscans-1 (composition of the per-step motions)
  std::vector<synth::Pose> poses(nscans);
  synth::Pose P;
  synth::pose_identity(P);
  for (int k = 0; k < first_scan + nscans; k++) {
    if (k >= first_scan) poses[k - first_scan] = P;
    double d[6];
    synth::drive_step(seed, k, P, d);
    synth::advance(P, d);
  }
  int rc = c->posebuf.ensure(poses.size() * sizeof(synth::Pose));
  if (rc) return rc;
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaMemcpyAsync(c->posebuf.p, poses.data(), poses.size() * sizeof(synth::Pose), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const size_t total = (size_t)nscans * rings * azim;
  k_synth<<<(unsigned)((total + 127) / 128), 128, 0, c->stream>>>(seed, first_scan, nscans, rings, azim,
                                                                  (const synth::Pose*)c->posebuf.p, out);
  c->launches++;
  CK(cudaGetLastError());
  return 0;
}

#include "callers_abi.inl"
#include "kfnode_abi.inl"
#include "multi_abi.inl"

}  // extern "C"

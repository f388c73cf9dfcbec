// Whole hot path, device resident: DAISY x2 -> per direction {kNN proposals, random proposals, BCD sweeps,
// label->flow} -> forward/backward check.  This is what `daisy i flann.py` + `python bcd.py` (run once per
// direction) + postprocessing.postProcessing compute between them, without the .npy round trips.
// Also: error strings and the host-buffer context used by the drop-in scripts and the e2e benchmark.
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace flowb200 {

static thread_local std::string g_last_cuda_error;

void set_cuda_error(cudaError_t e, const char* where) {
  g_last_cuda_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e) + " at " + where;
}

static std::atomic<long long> g_launches{0};
void count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// Auxiliary streams (+ fork/join events) for the backward direction: a process-wide pool per device.  A call takes one
// for its duration and gives it back, so that concurrent calls from any number of host threads (bench.py --inflight)
// reuse a handful of streams instead of creating one per thread; they live until the process ends.
struct AuxStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
struct AuxPool {
  std::mutex m;
  std::vector<AuxStream*> idle[64];
};
static AuxPool& aux_pool() {
  static AuxPool* p = new AuxPool();   // (never destroyed: CUDA may already be shut down at static destruction)
  return *p;
}
static AuxStream* aux_acquire(int* dev_out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  *dev_out = dev;
  {
    std::lock_guard<std::mutex> lock(aux_pool().m);
    auto& v = aux_pool().idle[dev];
    if (!v.empty()) {
      AuxStream* a = v.back();
      v.pop_back();
      return a;
    }
  }
  AuxStream* a = new AuxStream();
  if (cudaStreamCreateWithFlags(&a->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&a->fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&a->join, cudaEventDisableTiming) != cudaSuccess) {
    if (a->stream) cudaStreamDestroy(a->stream);
    if (a->fork) cudaEventDestroy(a->fork);
    delete a;
    return nullptr;
  }
  return a;
}
static void aux_release(int dev, AuxStream* a) {
  std::lock_guard<std::mutex> lock(aux_pool().m);
  aux_pool().idle[dev].push_back(a);
}

struct PairLayout {
  size_t desc[2], daisy_ws, pvec[2], lcost[2], nprop[2], labels[2], uvv[2], bcd_ws[2], knn_ws[2], total;
};

static PairLayout pair_layout(const flowb200_params* p) {
  PairLayout L{};
  const size_t n = (size_t)p->H * p->W, K = (size_t)p->maxnprop;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += align_up(bytes);
    return o;
  };
  L.desc[0] = take(n * kDescDim * sizeof(float));
  L.desc[1] = take(n * kDescDim * sizeof(float));
  L.daisy_ws = take(flowb200_daisy_workspace_bytes(p->H, p->W));
  for (int d = 0; d < 2; ++d) {
    L.pvec[d] = take(n * K * sizeof(int32_t));
    L.lcost[d] = take(n * K * sizeof(float));
    L.nprop[d] = take(n * sizeof(int32_t));
    L.labels[d] = take(n * sizeof(int32_t));
    L.uvv[d] = take(n * 3 * sizeof(float));
    L.bcd_ws[d] = take(flowb200_bcd_workspace_bytes(p->H, p->W, p->maxnprop));
    L.knn_ws[d] = take(flowb200_knn_workspace_bytes(p));
  }
  L.total = off;
  return L;
}

}  // namespace flowb200

using namespace flowb200;

extern "C" int flowb200_version(void) { return FLOWB200_VERSION; }

extern "C" const char* flowb200_error_string(int code) {
  switch (code) {
    case FLOWB200_OK: return "ok";
    case FLOWB200_EINVAL: return "invalid argument";
    case FLOWB200_EWORKSPACE: return "workspace too small";
    case FLOWB200_ECUDA: return "CUDA error";
    case FLOWB200_EUNSUPPORTED: return "unsupported parameter combination";
    default: return "unknown error";
  }
}

extern "C" long long flowb200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" const char* flowb200_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

extern "C" size_t flowb200_pair_workspace_bytes(const flowb200_params* p) {
  if (!p || p->H <= 0 || p->W <= 0 || p->maxnprop <= 0) return 0;
  return pair_layout(p).total;
}

// one direction = proposals (search + random), then BCD + flow field (integer, or sub-pixel with p->flow_refine)
static int run_proposals(const flowb200_params* p, const PairLayout& L, char* ws, int d, uint64_t seed,
                         cudaStream_t stream) {
  const float* src = reinterpret_cast<const float*>(ws + L.desc[d]);
  const float* tgt = reinterpret_cast<const float*>(ws + L.desc[1 - d]);
  int32_t* pvec = reinterpret_cast<int32_t*>(ws + L.pvec[d]);
  float* lcost = reinterpret_cast<float*>(ws + L.lcost[d]);
  int32_t* nprop = reinterpret_cast<int32_t*>(ws + L.nprop[d]);
  int32_t* labels = reinterpret_cast<int32_t*>(ws + L.labels[d]);
  int rc = flowb200_knn_proposals(src, tgt, p, pvec, lcost, nprop, labels, nullptr, nullptr, ws + L.knn_ws[d],
                                  flowb200_knn_workspace_bytes(p), stream);
  if (rc) return rc;
  return flowb200_random_proposals(src, tgt, p, pvec, lcost, nprop, labels, nullptr, seed + (uint64_t)d, stream);
}

static int run_bcd(const flowb200_params* p, const PairLayout& L, char* ws, int d, int sweeps, cudaStream_t stream) {
  int32_t* pvec = reinterpret_cast<int32_t*>(ws + L.pvec[d]);
  float* lcost = reinterpret_cast<float*>(ws + L.lcost[d]);
  int32_t* nprop = reinterpret_cast<int32_t*>(ws + L.nprop[d]);
  int32_t* labels = reinterpret_cast<int32_t*>(ws + L.labels[d]);
  // the pipeline produces float32 costs: the int32 programme quantises them on the fly
  // (FLOWB200_BCD_MRF passes through to the chains)
  const int mrf = p->bcd_mode & FLOWB200_BCD_MRF;
  int mode = p->bcd_mode & ~FLOWB200_BCD_MRF;
  if (mode == FLOWB200_BCD_INT32) mode = FLOWB200_BCD_INT32_F32COST;
  if (mode != FLOWB200_BCD_INT32_F32COST && mode != FLOWB200_BCD_FP64_F32COST) return FLOWB200_EINVAL;
  int rc = flowb200_bcd(pvec, lcost, nprop, labels, p->H, p->W, p->maxnprop, mode | mrf, p->lamda, p->tpsi,
                        p->cost_shift, sweeps, nullptr, ws + L.bcd_ws[d],
                        flowb200_bcd_workspace_bytes(p->H, p->W, p->maxnprop), stream);
  if (rc) return rc;
  float* uvv = reinterpret_cast<float*>(ws + L.uvv[d]);
  if (p->flow_refine)   // both directions' descriptors stay in the workspace until the call returns
    return flowb200_flow_subpixel(reinterpret_cast<const float*>(ws + L.desc[d]),
                                  reinterpret_cast<const float*>(ws + L.desc[1 - d]), pvec, nprop, labels, p->H, p->W,
                                  p->maxnprop, uvv, stream);
  return flowb200_flow_from_labels(pvec, labels, p->H, p->W, p->maxnprop, nullptr, uvv, stream);
}

static int run_direction(const flowb200_params* p, const PairLayout& L, char* ws, int d, int sweeps, uint64_t seed,
                         cudaStream_t stream) {
  const int rc = run_proposals(p, L, ws, d, seed, stream);
  return rc ? rc : run_bcd(p, L, ws, d, sweeps, stream);
}

extern "C" int flowb200_flow_pair(const uint8_t* bgr0, const uint8_t* bgr1, const flowb200_params* p, int sweeps,
                                  int directions, uint64_t seed, float* out_fwd, float* out_fwd_raw, float* out_bwd_raw,
                                  void* workspace, size_t workspace_bytes, flowb200_stream_t stream) {
  if (!bgr0 || !bgr1 || !p || !out_fwd || !workspace) return FLOWB200_EINVAL;
  if (directions != 1 && directions != 2) return FLOWB200_EINVAL;
  if (sweeps < 0) return FLOWB200_EINVAL;
  if (p->flow_refine != 0 && p->flow_refine != 1) return FLOWB200_EINVAL;
  const PairLayout L = pair_layout(p);
  if (workspace_bytes < L.total) return FLOWB200_EWORKSPACE;
  char* ws = static_cast<char*>(workspace);
  const size_t n = (size_t)p->H * p->W;
  const size_t dws = flowb200_daisy_workspace_bytes(p->H, p->W);
  int rc = flowb200_daisy(bgr0, p->H, p->W, reinterpret_cast<float*>(ws + L.desc[0]), ws + L.daisy_ws, dws, stream);
  if (rc) return rc;
  rc = flowb200_daisy(bgr1, p->H, p->W, reinterpret_cast<float*>(ws + L.desc[1]), ws + L.daisy_ws, dws, stream);
  if (rc) return rc;
  // forward and backward are independent (README.md:40): the backward direction runs on an auxiliary stream
  // so that the small launches of one direction (BCD row phases have only H/2 chains) fill the SMs the other
  // leaves idle.  fork: aux waits for the DAISYs; join: `stream` waits for aux before the consistency check.
  int aux_dev = 0;
  AuxStream* aux = directions == 2 ? aux_acquire(&aux_dev) : nullptr;
  if (aux) {
    // whatever happens after the fork, `stream` waits for the auxiliary stream before this call returns: the caller
    // may reuse the workspace as soon as `stream` is done
    // (Both directions start together.  Starting the backward search only when the forward BCD begins, so that
    // unlike kernels overlap, was measured slower, 71.7 against 68.8 ms per pair: the persistent selection CTAs hold
    // the shared memory the chain kernels need.)
    int rc1 = FLOWB200_OK, rc0 = FLOWB200_OK;
    cudaError_t e = cudaEventRecord(aux->fork, stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(aux->stream, aux->fork, 0);
    if (e == cudaSuccess) {
      rc1 = run_direction(p, L, ws, 1, sweeps, seed, aux->stream);
      rc0 = run_direction(p, L, ws, 0, sweeps, seed, stream);
      e = cudaEventRecord(aux->join, aux->stream);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, aux->join, 0);
    }
    aux_release(aux_dev, aux);
    if (e != cudaSuccess) {
      set_cuda_error(e, "flowb200_flow_pair (fork / join of the backward direction)");
      return FLOWB200_ECUDA;
    }
    if (rc0 || rc1) return rc0 ? rc0 : rc1;
  } else {
    rc = run_direction(p, L, ws, 0, sweeps, seed, stream);
    if (rc) return rc;
    if (directions == 2) {
      rc = run_direction(p, L, ws, 1, sweeps, seed, stream);
      if (rc) return rc;
    }
  }
  const size_t fbytes = n * 3 * sizeof(float);
  FB_CUDA_CHECK(cudaMemcpyAsync(out_fwd, ws + L.uvv[0], fbytes, cudaMemcpyDeviceToDevice, stream));
  if (out_fwd_raw) FB_CUDA_CHECK(cudaMemcpyAsync(out_fwd_raw, ws + L.uvv[0], fbytes, cudaMemcpyDeviceToDevice, stream));
  if (directions == 2) {
    if (out_bwd_raw)
      FB_CUDA_CHECK(cudaMemcpyAsync(out_bwd_raw, ws + L.uvv[1], fbytes, cudaMemcpyDeviceToDevice, stream));
    rc = flowb200_consistency(out_fwd, reinterpret_cast<const float*>(ws + L.uvv[1]), p->H, p->W, p->con_tresh, 0,
                              p->H, 0, p->W, stream);
    if (rc) return rc;
  }
  return FLOWB200_OK;
}

// ---------------------------------------------------------------------------------------------
// host-buffer context
// ---------------------------------------------------------------------------------------------
struct flowb200_ctx {
  flowb200_params p;
  cudaStream_t stream = nullptr;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  uint8_t* d_img[2] = {nullptr, nullptr};
  float* d_out = nullptr;
  uint8_t* h_img[2] = {nullptr, nullptr};   // pinned staging
  float* h_out = nullptr;
  // second set of image / output buffers, a copy stream and events: flowb200_ctx_flow_pairs_host moves pair i+1 in
  // and result i-1 out while pair i is computed (created on first use)
  cudaStream_t copy = nullptr;
  uint8_t* d_img2[2] = {nullptr, nullptr};
  float* d_out2 = nullptr;
  uint8_t* h_img2[2] = {nullptr, nullptr};
  float* h_out2 = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
};

extern "C" void flowb200_ctx_destroy(flowb200_ctx* c) {
  if (!c) return;
  if (c->stream) cudaStreamSynchronize(c->stream);
  cudaFree(c->ws);
  cudaFree(c->d_img[0]);
  cudaFree(c->d_img[1]);
  cudaFree(c->d_out);
  cudaFreeHost(c->h_img[0]);
  cudaFreeHost(c->h_img[1]);
  cudaFreeHost(c->h_out);
  if (c->copy) cudaStreamSynchronize(c->copy);
  cudaFree(c->d_img2[0]);
  cudaFree(c->d_img2[1]);
  cudaFree(c->d_out2);
  cudaFreeHost(c->h_img2[0]);
  cudaFreeHost(c->h_img2[1]);
  cudaFreeHost(c->h_out2);
  for (int i = 0; i < 2; ++i) {
    if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
    if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
    if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
  }
  if (c->copy) cudaStreamDestroy(c->copy);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" flowb200_ctx* flowb200_ctx_create(const flowb200_params* p) {
  if (!p || p->H <= 0 || p->W <= 0) return nullptr;
  flowb200_ctx* c = new flowb200_ctx();
  c->p = *p;
  const size_t n = (size_t)p->H * p->W;
  c->ws_bytes = flowb200_pair_workspace_bytes(p);
  bool ok = c->ws_bytes > 0;
  auto chk = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess) {
      set_cuda_error(e, what);
      ok = false;
    }
  };
  if (ok) chk(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), "cudaStreamCreate");
  if (ok) chk(cudaMalloc(&c->ws, c->ws_bytes), "cudaMalloc(workspace)");
  for (int i = 0; i < 2 && ok; ++i) {
    chk(cudaMalloc(reinterpret_cast<void**>(&c->d_img[i]), n * 3), "cudaMalloc(image)");
    if (ok) chk(cudaHostAlloc(reinterpret_cast<void**>(&c->h_img[i]), n * 3, cudaHostAllocDefault), "cudaHostAlloc");
  }
  if (ok) chk(cudaMalloc(reinterpret_cast<void**>(&c->d_out), n * 3 * sizeof(float)), "cudaMalloc(out)");
  if (ok) chk(cudaHostAlloc(reinterpret_cast<void**>(&c->h_out), n * 3 * sizeof(float), cudaHostAllocDefault), "cudaHostAlloc");
  if (!ok) {
    flowb200_ctx_destroy(c);
    return nullptr;
  }
  return c;
}

extern "C" int flowb200_ctx_flow_pair_host(flowb200_ctx* c, const uint8_t* bgr0_host, const uint8_t* bgr1_host,
                                           int sweeps, int directions, uint64_t seed, float* out_fwd_host) {
  if (!c || !bgr0_host || !bgr1_host || !out_fwd_host) return FLOWB200_EINVAL;
  const size_t n = (size_t)c->p.H * c->p.W;
  memcpy(c->h_img[0], bgr0_host, n * 3);
  memcpy(c->h_img[1], bgr1_host, n * 3);
  FB_CUDA_CHECK(cudaMemcpyAsync(c->d_img[0], c->h_img[0], n * 3, cudaMemcpyHostToDevice, c->stream));
  FB_CUDA_CHECK(cudaMemcpyAsync(c->d_img[1], c->h_img[1], n * 3, cudaMemcpyHostToDevice, c->stream));
  int rc = flowb200_flow_pair(c->d_img[0], c->d_img[1], &c->p, sweeps, directions, seed, c->d_out, nullptr, nullptr,
                              c->ws, c->ws_bytes, c->stream);
  if (rc) return rc;
  FB_CUDA_CHECK(cudaMemcpyAsync(c->h_out, c->d_out, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  FB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  memcpy(out_fwd_host, c->h_out, n * 3 * sizeof(float));
  return FLOWB200_OK;
}

// A batch of host-resident pairs (BASELINE.json configs[3]: a rank's share of the 99 pairs), one after the other on the
// context's stream, with the copies of the neighbouring pairs overlapped: while pair i is computed, pair i+1 travels to
// the device and result i-1 back, on a second stream (two buffer sets).
extern "C" int flowb200_ctx_flow_pairs_host(flowb200_ctx* c, const uint8_t* const* bgr0_host, const uint8_t* const* bgr1_host,
                                            int n_pairs, int sweeps, int directions, uint64_t seed0,
                                            float* const* out_fwd_host) {
  if (!c || !bgr0_host || !bgr1_host || !out_fwd_host || n_pairs < 0) return FLOWB200_EINVAL;
  if (n_pairs == 0) return FLOWB200_OK;
  const size_t n = (size_t)c->p.H * c->p.W, ibytes = n * 3, obytes = n * 3 * sizeof(float);
  if (!c->copy) {   // second buffer set, copy stream, events
    FB_CUDA_CHECK(cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&c->d_img2[i]), ibytes));
      FB_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&c->h_img2[i]), ibytes, cudaHostAllocDefault));
      FB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
      FB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
      FB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming));
    }
    FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&c->d_out2), obytes));
    FB_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&c->h_out2), obytes, cudaHostAllocDefault));
  }
  uint8_t* d_img[2][2] = {{c->d_img[0], c->d_img[1]}, {c->d_img2[0], c->d_img2[1]}};
  uint8_t* h_img[2][2] = {{c->h_img[0], c->h_img[1]}, {c->h_img2[0], c->h_img2[1]}};
  float* d_out[2] = {c->d_out, c->d_out2};
  float* h_out[2] = {c->h_out, c->h_out2};
  // pair i uses buffer set i & 1.  Copy stream, in this order: in(0), [in(i+1), out(i)] for every i.
  auto copy_in = [&](int i) -> int {
    const int s = i & 1;
    if (i >= 2) FB_CUDA_CHECK(cudaEventSynchronize(c->ev_in[s]));   // staging buffer of pair i-2 has left the host
    memcpy(h_img[s][0], bgr0_host[i], ibytes);
    memcpy(h_img[s][1], bgr1_host[i], ibytes);
    if (i >= 2) FB_CUDA_CHECK(cudaStreamWaitEvent(c->copy, c->ev_done[s], 0));   // pair i-2 no longer reads the images
    FB_CUDA_CHECK(cudaMemcpyAsync(d_img[s][0], h_img[s][0], ibytes, cudaMemcpyHostToDevice, c->copy));
    FB_CUDA_CHECK(cudaMemcpyAsync(d_img[s][1], h_img[s][1], ibytes, cudaMemcpyHostToDevice, c->copy));
    FB_CUDA_CHECK(cudaEventRecord(c->ev_in[s], c->copy));
    return FLOWB200_OK;
  };
  auto fetch_out = [&](int i) -> int {   // result i: pinned staging -> the caller's array
    FB_CUDA_CHECK(cudaEventSynchronize(c->ev_out[i & 1]));
    memcpy(out_fwd_host[i], h_out[i & 1], obytes);
    return FLOWB200_OK;
  };
  int rc = copy_in(0);
  if (rc) return rc;
  for (int i = 0; i < n_pairs; ++i) {
    const int s = i & 1;
    if (i + 1 < n_pairs && (rc = copy_in(i + 1))) return rc;
    FB_CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->ev_in[s], 0));
    if (i >= 2) FB_CUDA_CHECK(cudaStreamWaitEvent(c->stream, c->ev_out[s], 0));   // result i-2 has left d_out[s]
    rc = flowb200_flow_pair(d_img[s][0], d_img[s][1], &c->p, sweeps, directions, seed0 + (uint64_t)i, d_out[s], nullptr,
                            nullptr, c->ws, c->ws_bytes, c->stream);
    if (rc) return rc;
    FB_CUDA_CHECK(cudaEventRecord(c->ev_done[s], c->stream));
    if (i >= 2 && (rc = fetch_out(i - 2))) return rc;             // frees h_out[s] for result i
    FB_CUDA_CHECK(cudaStreamWaitEvent(c->copy, c->ev_done[s], 0));
    FB_CUDA_CHECK(cudaMemcpyAsync(h_out[s], d_out[s], obytes, cudaMemcpyDeviceToHost, c->copy));
    FB_CUDA_CHECK(cudaEventRecord(c->ev_out[s], c->copy));
  }
  for (int i = n_pairs >= 2 ? n_pairs - 2 : 0; i < n_pairs; ++i)
    if ((rc = fetch_out(i))) return rc;
  FB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return FLOWB200_OK;
}

extern "C" int flowb200_consistency_host(float* flow1_host, const float* flow2_host, int A, int B, float tresh, int a0,
                                         int a1, int b0, int b1) {
  if (!flow1_host || !flow2_host || A <= 0 || B <= 0) return FLOWB200_EINVAL;
  const size_t bytes = (size_t)A * B * 3 * sizeof(float);
  float *d1 = nullptr, *d2 = nullptr;
  int rc = FLOWB200_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d1), bytes);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d2), bytes);
  if (e == cudaSuccess) e = cudaMemcpy(d1, flow1_host, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d2, flow2_host, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    rc = flowb200_consistency(d1, d2, A, B, tresh, a0, a1, b0, b1, nullptr);
    if (rc == FLOWB200_OK) e = cudaMemcpy(flow1_host, d1, bytes, cudaMemcpyDeviceToHost);
  }
  cudaFree(d1);
  cudaFree(d2);
  if (e != cudaSuccess) {
    set_cuda_error(e, "flowb200_consistency_host");
    return FLOWB200_ECUDA;
  }
  return rc;
}

// removeSmallSegments (postprocessing.py:29-76) on the device; SURVEY section 8(f) row 1.
//
// Disabled in the reference's own postProcessing (:132) but part of its module, and Menze's second post-processing
// step.  Why it is split into a parallel and a sequential part, and what exactly is replayed, is explained in
// segments_core.cuh.  Kernels:
//   seg_init_kernel     transposes the field into scan order (float2 per pixel), one singleton set per valid pixel
//   seg_union_kernel    union-find over "valid 4-neighbours whose float32 L1 flow difference is <= tresh"
//                       (lock-free: atomicMin on the larger root, roots are minimal scan indices)
//   seg_flatten_kernel  root per pixel, pixels per root
//   seg_prefilter_*     settle the seed events that cannot have an effect (segments_core.cuh)
//   seg_replay_kernel   ONE warp walks the reference's scan: 32 pixels of a column per step (coalesced, ballot for
//                       the unvisited ones), lane 0 handles the seed events in order (seg_process_seed)
// HBM bound in the first three (36 B/pixel), latency bound in the replay (two dependent loads per 32 pixels and per
// seed event); the replay is what the reference's semantics leave sequential.
#include "common.cuh"
#include "segments_core.cuh"
#include "unionfind.cuh"

namespace flowb200 {
namespace {

struct SegLayout {
  size_t fT, root, size, cchk, vis, touch, queue, total;
};

SegLayout seg_layout(int A, int B) {
  const size_t n = (size_t)A * B;
  SegLayout L;
  size_t o = 0;
  L.fT = o;    o = align_up(o + n * sizeof(float2));
  L.root = o;  o = align_up(o + n * sizeof(int32_t));
  L.size = o;  o = align_up(o + n * sizeof(int32_t));
  L.queue = o; o = align_up(o + n * sizeof(int32_t));
  L.cchk = o;  o = align_up(o + n);
  L.vis = o;   o = align_up(o + n);
  L.touch = o; o = align_up(o + n);
  L.total = o;
  return L;
}

__global__ void seg_init_kernel(const float* __restrict__ flow, int A, int B, float2* __restrict__ fT,
                                int32_t* __restrict__ root, int32_t* __restrict__ size, uint8_t* __restrict__ cchk,
                                uint8_t* __restrict__ vis) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A * B) return;
  const float* p = flow + ((size_t)(s % A) * B + s / A) * 3;
  fT[s] = make_float2(p[0], p[1]);
  root[s] = p[2] > 0.5f ? s : kSegInvalid;
  size[s] = 0;
  cchk[s] = 0;
  vis[s] = 0;
}

__global__ void seg_union_kernel(const float2* __restrict__ fT, int A, int B, float tresh, int32_t* parent) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A * B) return;
  if (parent[s] < 0) return;
  const float2 f = fT[s];
  const int a = s % A, b = s / A;
  if (a + 1 < A && parent[s + 1] >= 0 && seg_near(f, fT[s + 1], tresh)) uf_merge(parent, s, s + 1);
  if (b + 1 < B && parent[s + A] >= 0 && seg_near(f, fT[s + A], tresh)) uf_merge(parent, s, s + A);
}

__global__ void seg_flatten_kernel(int n, int32_t* parent, int32_t* __restrict__ size) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  if (parent[s] < 0) return;
  const int r = uf_find(parent, s);
  parent[s] = r;   // a root keeps pointing at itself, so concurrent finds through s still end at r
  atomicAdd(&size[r], 1);
}

// Settle the seed events that cannot have an effect before the replay (segments_core.cuh): 8.4 instead of 29.7 ms on
// the bench workload's checked field, same valid flags (profiles/r02_segments_prefilter{0,1}.json).
__global__ void seg_prefilter_invalid_kernel(SegState S) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S.A * S.B) return;
  if (S.root[s] >= 0) return;
  if (!seg_invalid_touches(S, s)) S.root[s] = kSegInvalidChecked;
}

__global__ void seg_prefilter_component_kernel(SegState S) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S.A * S.B) return;
  if (S.root[s] != s) return;
  if (seg_component_inert(S, s)) S.cchk[s] = 1;
}

// 32 pixels of the column per step: one ballot marks the unvisited ones.  The mask may be stale by the time a bit is
// reached (an earlier seed of the same step took that pixel's component), so lane 0 re-tests every candidate - pixels
// only ever go from unvisited to visited, so a pixel absent from the mask stays skipped rightly.  A removal that moves
// the scan to another column restarts the step there.  The seed events, not the scan, bound the replay: 128 pixels
// per step measured the same time (profiles/r01_segments_time.json).
__global__ void __launch_bounds__(32, 1) seg_replay_kernel(SegState S) {
  const unsigned lane = threadIdx.x;
  for (int bo = 0; bo < S.B; ++bo) {
    int b = bo;      // :36; may be rebound by a removal until the column scan ends (:74)
    int a = 0;       // :37
    while (a < S.A) {
      const int pa = a + (int)lane;
      const bool open = pa < S.A && seg_unchecked(S, b * S.A + pa);
      unsigned m = __ballot_sync(0xffffffffu, open);
      int next_a = a + 32;
      bool moved = false;
      while (m != 0 && !moved) {
        const int sa = a + __ffs(m) - 1;
        m &= m - 1;
        int nb = b;
        if (lane == 0 && seg_unchecked(S, b * S.A + sa)) nb = seg_process_seed(S, b * S.A + sa, b);
        __syncwarp();   // lane 0's flag updates are ordered before the next loads of all lanes
        nb = __shfl_sync(0xffffffffu, nb, 0);
        if (nb != b) {
          b = nb;
          next_a = sa + 1;
          moved = true;
        }
      }
      a = next_a;
    }
  }
}

}  // namespace
}  // namespace flowb200

using namespace flowb200;

extern "C" size_t flowb200_segments_workspace_bytes(int A, int B) {
  if (A <= 0 || B <= 0) return 0;
  return seg_layout(A, B).total;
}

extern "C" int flowb200_remove_small_segments(float* flow, int A, int B, float tresh, int min_segment_size,
                                              void* workspace, size_t workspace_bytes, flowb200_stream_t stream) {
  if (!flow || A <= 0 || B <= 0 || (long long)A * B > 0x7fffffffLL) return FLOWB200_EINVAL;
  if (!workspace) return FLOWB200_EINVAL;
  const SegLayout L = seg_layout(A, B);
  if (workspace_bytes < L.total) return FLOWB200_EWORKSPACE;
  if (min_segment_size <= 2) return FLOWB200_OK;   // 1 < count < min_segment_size (:73) has no solution
  char* ws = static_cast<char*>(workspace);
  const int n = A * B;
  SegState S;
  S.A = A;
  S.B = B;
  S.tresh = tresh;
  S.min_size = min_segment_size;
  S.fT = reinterpret_cast<const float2*>(ws + L.fT);
  S.root = reinterpret_cast<int32_t*>(ws + L.root);
  S.size = reinterpret_cast<const int32_t*>(ws + L.size);
  S.cchk = reinterpret_cast<uint8_t*>(ws + L.cchk);
  S.vis = reinterpret_cast<uint8_t*>(ws + L.vis);
  S.touch = reinterpret_cast<uint8_t*>(ws + L.touch);
  S.queue = reinterpret_cast<int32_t*>(ws + L.queue);
  S.flow = flow;
  float2* fT = reinterpret_cast<float2*>(ws + L.fT);
  int32_t* root = reinterpret_cast<int32_t*>(ws + L.root);
  int32_t* size = reinterpret_cast<int32_t*>(ws + L.size);
  const int T = 256, G = (n + T - 1) / T;
  seg_init_kernel<<<G, T, 0, stream>>>(flow, A, B, fT, root, size, reinterpret_cast<uint8_t*>(ws + L.cchk), S.vis);
  seg_union_kernel<<<G, T, 0, stream>>>(fT, A, B, tresh, root);
  seg_flatten_kernel<<<G, T, 0, stream>>>(n, root, size);
  FB_CUDA_CHECK(cudaMemsetAsync(S.touch, 0, (size_t)n, stream));
  seg_prefilter_invalid_kernel<<<G, T, 0, stream>>>(S);
  seg_prefilter_component_kernel<<<G, T, 0, stream>>>(S);
  seg_replay_kernel<<<1, 32, 0, stream>>>(S);
  FB_LAUNCH_CHECK_N(6);
  return FLOWB200_OK;
}

extern "C" int flowb200_remove_small_segments_host(float* flow_host, int A, int B, float tresh, int min_segment_size) {
  if (!flow_host || A <= 0 || B <= 0 || (long long)A * B > 0x7fffffffLL) return FLOWB200_EINVAL;
  const size_t bytes = (size_t)A * B * 3 * sizeof(float);
  const size_t wsb = flowb200_segments_workspace_bytes(A, B);
  float* d = nullptr;
  void* ws = nullptr;
  int rc = FLOWB200_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d), bytes);
  if (e == cudaSuccess) e = cudaMalloc(&ws, wsb);
  if (e == cudaSuccess) e = cudaMemcpy(d, flow_host, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    rc = flowb200_remove_small_segments(d, A, B, tresh, min_segment_size, ws, wsb, nullptr);
    if (rc == FLOWB200_OK) e = cudaMemcpy(flow_host, d, bytes, cudaMemcpyDeviceToHost);
  }
  cudaFree(d);
  cudaFree(ws);
  if (e != cudaSuccess) {
    set_cuda_error(e, "flowb200_remove_small_segments_host");
    return FLOWB200_ECUDA;
  }
  return rc;
}

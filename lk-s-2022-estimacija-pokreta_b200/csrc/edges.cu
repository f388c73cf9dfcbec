// edge.canny_ivice (edge.py:19-35) on the device: the Canny edge map EpicFlow takes as its edge input.
// SURVEY section 8(f) row 4.  gray -> 3x3 Gaussian -> Sobel -> non-maximum suppression + double threshold ->
// hysteresis, bit-identical to OpenCV's 8-bit integer path (arithmetic in edges_core.cuh, pinned against cv2 by
// the oracle tests).  Kernels, one thread per pixel, HBM bound (3 B in, 4 B out per pixel; intermediates stay in L2
// at the sizes of the path):
//   edge_blur_kernel   uint8 BGR -> blurred gray uint8
//   edge_sobel_kernel  -> packed int16 (dx, dy)
//   edge_nms_kernel    -> survivor map {1 none, 0 weak, 2 strong}; one singleton set per survivor
//   edge_link_kernel   union of 8-connected survivors (E, SW, S, SE of every survivor; lock-free union-find)
//   edge_mark_kernel   the root of every strong survivor is flagged
//   edge_out_kernel    0.0f where the survivor's root is flagged, 1.0f elsewhere (`(255 - edges) / 255`, edge.py:29)
// cv::Canny floods from the strong pixels with a stack; "8-connected to a strong survivor" is the same set.
#include "common.cuh"
#include "edges_core.cuh"
#include "unionfind.cuh"

namespace flowb200 {
namespace {

struct EdgeLayout {
  size_t blur, grad, parent, pmap, strong, total;
};

EdgeLayout edge_layout(int H, int W) {
  const size_t n = (size_t)H * W;
  EdgeLayout L;
  size_t o = 0;
  L.grad = o;   o = align_up(o + n * sizeof(int32_t));
  L.parent = o; o = align_up(o + n * sizeof(int32_t));
  L.blur = o;   o = align_up(o + n);
  L.pmap = o;   o = align_up(o + n);
  L.strong = o; o = align_up(o + n);
  L.total = o;
  return L;
}

__global__ void edge_blur_kernel(const uint8_t* __restrict__ bgr, int H, int W, uint8_t* __restrict__ blur) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  blur[i] = edge_gray_blur_at(bgr, H, W, i / W, i % W);
}

__global__ void edge_sobel_kernel(const uint8_t* __restrict__ blur, int H, int W, int32_t* __restrict__ grad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  grad[i] = edge_sobel_at(blur, H, W, i / W, i % W);
}

__global__ void edge_nms_kernel(const int32_t* __restrict__ grad, int H, int W, int low, int high,
                                uint8_t* __restrict__ pmap, int32_t* __restrict__ parent,
                                uint8_t* __restrict__ strong) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const uint8_t v = edge_nms_at(grad, H, W, i / W, i % W, low, high);
  pmap[i] = v;
  parent[i] = v != 1 ? i : -1;
  strong[i] = 0;
}

__global__ void edge_link_kernel(const uint8_t* __restrict__ pmap, int H, int W, int32_t* parent) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  if (pmap[i] == 1) return;
  const int y = i / W, x = i % W;
  if (x + 1 < W && pmap[i + 1] != 1) uf_merge(parent, i, i + 1);
  if (y + 1 < H) {
    if (x > 0 && pmap[i + W - 1] != 1) uf_merge(parent, i, i + W - 1);
    if (pmap[i + W] != 1) uf_merge(parent, i, i + W);
    if (x + 1 < W && pmap[i + W + 1] != 1) uf_merge(parent, i, i + W + 1);
  }
}

__global__ void edge_mark_kernel(const uint8_t* __restrict__ pmap, int n, int32_t* parent, uint8_t* strong) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (pmap[i] == 2) strong[uf_find(parent, i)] = 1;
}

__global__ void edge_out_kernel(const uint8_t* __restrict__ pmap, int n, int32_t* parent,
                                const uint8_t* __restrict__ strong, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = (pmap[i] != 1 && strong[uf_find(parent, i)]) ? 0.f : 1.f;
}

}  // namespace
}  // namespace flowb200

using namespace flowb200;

extern "C" size_t flowb200_edges_workspace_bytes(int H, int W) {
  if (H <= 0 || W <= 0) return 0;
  return edge_layout(H, W).total;
}

extern "C" int flowb200_canny_edges(const uint8_t* bgr, int H, int W, int low, int high, float* inverted_edges,
                                    void* workspace, size_t workspace_bytes, flowb200_stream_t stream) {
  if (!bgr || !inverted_edges || !workspace || H <= 0 || W <= 0 || (long long)H * W > 0x7fffffffLL)
    return FLOWB200_EINVAL;
  const EdgeLayout L = edge_layout(H, W);
  if (workspace_bytes < L.total) return FLOWB200_EWORKSPACE;
  if (low > high) {   // cv::Canny swaps its thresholds when threshold1 > threshold2
    const int t = low;
    low = high;
    high = t;
  }
  char* ws = static_cast<char*>(workspace);
  uint8_t* blur = reinterpret_cast<uint8_t*>(ws + L.blur);
  uint8_t* pmap = reinterpret_cast<uint8_t*>(ws + L.pmap);
  uint8_t* strong = reinterpret_cast<uint8_t*>(ws + L.strong);
  int32_t* grad = reinterpret_cast<int32_t*>(ws + L.grad);
  int32_t* parent = reinterpret_cast<int32_t*>(ws + L.parent);
  const int n = H * W, T = 256, G = (n + T - 1) / T;
  edge_blur_kernel<<<G, T, 0, stream>>>(bgr, H, W, blur);
  edge_sobel_kernel<<<G, T, 0, stream>>>(blur, H, W, grad);
  edge_nms_kernel<<<G, T, 0, stream>>>(grad, H, W, low, high, pmap, parent, strong);
  edge_link_kernel<<<G, T, 0, stream>>>(pmap, H, W, parent);
  edge_mark_kernel<<<G, T, 0, stream>>>(pmap, n, parent, strong);
  edge_out_kernel<<<G, T, 0, stream>>>(pmap, n, parent, strong, inverted_edges);
  FB_LAUNCH_CHECK_N(6);
  return FLOWB200_OK;
}

extern "C" int flowb200_canny_edges_host(const uint8_t* bgr_host, int H, int W, int low, int high,
                                         float* inverted_edges_host) {
  if (!bgr_host || !inverted_edges_host || H <= 0 || W <= 0 || (long long)H * W > 0x7fffffffLL)
    return FLOWB200_EINVAL;
  const size_t n = (size_t)H * W;
  const size_t wsb = flowb200_edges_workspace_bytes(H, W);
  uint8_t* d_in = nullptr;
  float* d_out = nullptr;
  void* ws = nullptr;
  int rc = FLOWB200_OK;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&d_in), n * 3);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d_out), n * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&ws, wsb);
  if (e == cudaSuccess) e = cudaMemcpy(d_in, bgr_host, n * 3, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    rc = flowb200_canny_edges(d_in, H, W, low, high, d_out, ws, wsb, nullptr);
    if (rc == FLOWB200_OK) e = cudaMemcpy(inverted_edges_host, d_out, n * sizeof(float), cudaMemcpyDeviceToHost);
  }
  cudaFree(d_in);
  cudaFree(d_out);
  cudaFree(ws);
  if (e != cudaSuccess) {
    set_cuda_error(e, "flowb200_canny_edges_host");
    return FLOWB200_ECUDA;
  }
  return rc;
}

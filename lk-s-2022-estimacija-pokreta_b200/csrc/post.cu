// Label -> flow gather and the forward/backward consistency check.
//   flow_from_labels : vratiKonacniFlow (daisy i flann.py:192-197 / python bcd.py:90-95) fused with
//                      FlowImage.ucitajFlow's (dx, dy, valid=1) float32 layout (postprocessing.py:7-17)
//   flow_subpixel    : flow_from_labels with each vector refined to sub-pixel precision (DESIGN section 4.8;
//                      no reference counterpart)
//   consistency      : consistencyCheck / fowardBackwardConsistency (postprocessing.py:79-117)
// flow_from_labels and consistency are HBM-bound streaming kernels: 28 B/pixel algorithmic (SURVEY.md section 8d);
// flow_subpixel reads six descriptor rows per pixel: 1652 B/pixel, mostly from L2 (DESIGN section 4.8).
#include <climits>

#include "common.cuh"

namespace flowb200 {

__global__ void flow_from_labels_kernel(const int32_t* __restrict__ pvec, const int32_t* __restrict__ labels,
                                        int n_pix, int K, double* __restrict__ flow_yx, float* __restrict__ uvv) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pix) return;
  int32_t v = pvec[(size_t)i * K + labels[i]];
  int dy = vec_dy(v), dx = vec_dx(v);
  if (flow_yx) {
    flow_yx[2 * (size_t)i] = (double)dy;
    flow_yx[2 * (size_t)i + 1] = (double)dx;
  }
  if (uvv) {
    uvv[3 * (size_t)i] = (float)dx;
    uvv[3 * (size_t)i + 1] = (float)dy;
    uvv[3 * (size_t)i + 2] = 1.0f;
  }
}

// Sub-pixel refinement (DESIGN section 4.8): per axis, the vertex of the parabola through the data costs of the chosen
// target and its two neighbours along that axis.  One thread per pixel; the source row stays in registers and each
// target row is read as 17 float4 loads (rows are 272 B: 16-byte aligned when the base is).  Every float32 operation
// is an explicit round-to-nearest intrinsic, so that tests/subpixel_oracle.py restates it bit for bit.
__device__ __forceinline__ float subpixel_cost(const float (&s)[kDescDim], const float* __restrict__ row) {
  float t[kDescDim];
  const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
  for (int k = 0; k < kDescDim / 4; ++k) {
    const float4 v = __ldg(r4 + k);
    t[4 * k] = v.x;
    t[4 * k + 1] = v.y;
    t[4 * k + 2] = v.z;
    t[4 * k + 3] = v.w;
  }
  return sum68_numpy_order([&](int d) { return fabsf(__fsub_rn(s[d], t[d])); });
}

// (c- - c+) / (2 (c- - 2 c0 + c+)) where c0 is a strict minimum, clamped to [-0.5, 0.5]; 0 otherwise
__device__ __forceinline__ float subpixel_offset(float cm, float c0, float cp) {
  if (!(c0 < cm && c0 < cp)) return 0.f;
  const float num = __fsub_rn(cm, cp);
  const float den = __fmul_rn(2.f, __fadd_rn(__fsub_rn(cm, __fmul_rn(2.f, c0)), cp));
  return fminf(fmaxf(__fdiv_rn(num, den), -0.5f), 0.5f);
}

__global__ void __launch_bounds__(128) subpixel_kernel(const float* __restrict__ desc_src,
                                                       const float* __restrict__ desc_tgt,
                                                       const int32_t* __restrict__ pvec,
                                                       const int32_t* __restrict__ nprop,
                                                       const int32_t* __restrict__ labels, int H, int W, int K,
                                                       float* __restrict__ uvv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  float* o = uvv + 3 * (size_t)i;
  const int l = labels[i];
  if (l < 0 || l >= K) {   // names no slot: no vector
    o[0] = 0.f;
    o[1] = 0.f;
    o[2] = 0.f;
    return;
  }
  const int32_t v = pvec[(size_t)i * K + l];
  const int dy = vec_dy(v), dx = vec_dx(v);
  const int y = i / W, x = i - y * W, ty = y + dy, tx = x + dx;
  float ox = 0.f, oy = 0.f;
  if (l < nprop[i] && v != -1 && ty >= 0 && ty < H && tx >= 0 && tx < W) {
    float s[kDescDim];
    const float4* s4 = reinterpret_cast<const float4*>(desc_src + (size_t)i * kDescDim);
#pragma unroll
    for (int k = 0; k < kDescDim / 4; ++k) {
      const float4 a = __ldg(s4 + k);
      s[4 * k] = a.x;
      s[4 * k + 1] = a.y;
      s[4 * k + 2] = a.z;
      s[4 * k + 3] = a.w;
    }
    const float* t = desc_tgt + ((size_t)ty * W + tx) * kDescDim;
    const float c0 = subpixel_cost(s, t);
    if (tx >= 1 && tx + 1 < W)
      ox = subpixel_offset(subpixel_cost(s, t - kDescDim), c0, subpixel_cost(s, t + kDescDim));
    if (ty >= 1 && ty + 1 < H)
      oy = subpixel_offset(subpixel_cost(s, t - (size_t)W * kDescDim), c0, subpixel_cost(s, t + (size_t)W * kDescDim));
  }
  o[0] = __fadd_rn((float)dx, ox);
  o[1] = __fadd_rn((float)dy, oy);
  o[2] = 1.0f;
}

// One thread per checked pixel (a, b) = (row, col) of flow1.  float32 arithmetic with explicit
// round-to-nearest ops so that nothing is contracted into an FMA: the reference evaluates
// du*du and dv*dv as separately rounded numpy float32 products (postprocessing.py:102-104).
// Quirk Q5: channel 0 (dx) is added to the row index and tested against shape[0]; channel 1 (dy)
// to the column index (postprocessing.py:80, 87-90).
__global__ void consistency_kernel(float* __restrict__ f1, const float* __restrict__ f2, int A, int B,
                                   float tresh, int a0, int a1, int b0, int b1) {
  int nb = b1 - b0;
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (a1 - a0) * nb) return;
  int a = a0 + t / nb, b = b0 + t % nb;
  size_t o = 3 * ((size_t)a * B + b);
  float u = f1[o], v = f1[o + 1], val = f1[o + 2];
  if (!(val > 0.5f)) return;
  const float fa = __fadd_rn(u, (float)a), fb = __fadd_rn(v, (float)b);
  int a2 = (int)fa;   // int() truncates toward zero; +-inf saturates to INT_MAX / INT_MIN: out of range
  int b2 = (int)fb;
  // The conversion turns NaN into 0, a valid row / column.  The reference's int() raises on NaN and the oracle's cast
  // gives INT64_MIN: a NaN coordinate is out of range, so the pixel is zeroed (deliberate difference, DESIGN section 1).
  bool bad = (isnan(fa) || isnan(fb) || a2 < 0 || b2 < 0 || a2 >= A || b2 >= B);
  if (!bad) {
    size_t o2 = 3 * ((size_t)a2 * B + b2);
    float u2 = f2[o2], v2 = f2[o2 + 1], val2 = f2[o2 + 2];
    if (!(val2 > 0.5f)) {
      bad = true;
    } else {
      float du = __fadd_rn(u, u2), dv = __fadd_rn(v, v2);
      float err = __fsqrt_rn(__fadd_rn(__fmul_rn(dv, dv), __fmul_rn(du, du)));
      bad = err > tresh;
    }
  }
  if (bad) {
    f1[o] = 0.f;
    f1[o + 1] = 0.f;
    f1[o + 2] = 0.f;
  }
}

// visualization.errorImage (visualization.py:128-152): over pixels valid in both fields, f_err = sqrt(dfu^2 + dfv^2)
// in float32; accumulates sum(f_err), #(f_err > abs_thresh), #valid in float64.
__global__ void epe_kernel(const float* __restrict__ test, const float* __restrict__ gt, int n_pix, float abs_thresh,
                           double* __restrict__ out) {
  double s = 0.0, no = 0.0, nv = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pix; i += gridDim.x * blockDim.x) {
    const float* t = test + 3 * (size_t)i;
    const float* g = gt + 3 * (size_t)i;
    if (t[2] > 0.5f && g[2] > 0.5f) {
      const float dfu = __fsub_rn(t[0], g[0]), dfv = __fsub_rn(t[1], g[1]);
      const float e = __fsqrt_rn(__fadd_rn(__fmul_rn(dfu, dfu), __fmul_rn(dfv, dfv)));
      s += (double)e;
      no += e > abs_thresh ? 1.0 : 0.0;
      nv += 1.0;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, off);
    no += __shfl_xor_sync(0xffffffffu, no, off);
    nv += __shfl_xor_sync(0xffffffffu, nv, off);
  }
  if ((threadIdx.x & 31) == 0 && nv > 0.0) {
    atomicAdd(out, s);
    atomicAdd(out + 1, no);
    atomicAdd(out + 2, nv);
  }
}

}  // namespace flowb200

using namespace flowb200;

extern "C" int flowb200_epe(const float* test_uvv, const float* gt_uvv, int H, int W, float abs_thresh, double* out3,
                            flowb200_stream_t stream) {
  if (!test_uvv || !gt_uvv || !out3 || H <= 0 || W <= 0) return FLOWB200_EINVAL;
  FB_CUDA_CHECK(cudaMemsetAsync(out3, 0, 3 * sizeof(double), stream));
  epe_kernel<<<kNumSMs * 4, 256, 0, stream>>>(test_uvv, gt_uvv, H * W, abs_thresh, out3);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

// bestlabels of generisi (daisy i flann.py:181-184): the first strict minimum of the data costs of the first nprop
// slots.  One warp per pixel; costs are >= 0, so (float bits << 32 | slot) orders like (cost, slot).
__global__ void best_labels_kernel(const float* __restrict__ lcost, const int32_t* __restrict__ nprop, int n, int K,
                                   int32_t* __restrict__ labels) {
  const int pix = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (pix >= n) return;
  const int np = min(nprop[pix], K);
  const float* c = lcost + (size_t)pix * K;
  unsigned long long best = ~0ull;
  for (int s = lane; s < np; s += 32) {
    const unsigned long long key = ((unsigned long long)__float_as_uint(c[s]) << 32) | (uint32_t)s;
    best = key < best ? key : best;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, off);
    best = o < best ? o : best;
  }
  if (lane == 0) labels[pix] = np > 0 ? (int32_t)(best & 0xffffffffu) : 0;
}

extern "C" int flowb200_best_labels(const float* lcost, const int32_t* nprop, int H, int W, int K, int32_t* labels,
                                    flowb200_stream_t stream) {
  if (!lcost || !nprop || !labels || H <= 0 || W <= 0 || K <= 0) return FLOWB200_EINVAL;
  const int n = H * W;
  best_labels_kernel<<<(unsigned)(((size_t)n * 32 + 255) / 256), 256, 0, stream>>>(lcost, nprop, n, K, labels);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

// Slot-range copies of the single-huge-image merge (huge.py: pack_band / unpack_band as ONE launch instead of one
// strided copy per range).  blockIdx.y = table entry, one warp per pixel of the entry, lanes over the slots: both
// sides of the copy are contiguous runs of n slots.
__global__ void slot_copy_kernel(const long long* __restrict__ table, int32_t* __restrict__ vec,
                                 int32_t* __restrict__ cost, int width, int K, int32_t* __restrict__ flat, int to_flat) {
  const long long* e = table + 8 * (size_t)blockIdx.y;
  const int y0 = (int)e[0], y1 = (int)e[1], x0 = (int)e[2], x1 = (int)e[3], slot0 = (int)e[4], n = (int)e[5];
  const long long off_vec = e[6], off_cost = e[7];
  const int cols = x1 - x0, npix = (y1 - y0) * cols;
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int i = blockIdx.x * wpb + (threadIdx.x >> 5); i < npix; i += gridDim.x * wpb) {
    const int r = i / cols, c = i - r * cols;
    const size_t a = ((size_t)(y0 + r) * width + (x0 + c)) * K + slot0;
    const size_t f = (size_t)i * n;
    for (int s = lane; s < n; s += 32) {
      if (to_flat) {
        flat[off_vec + f + s] = vec[a + s];
        flat[off_cost + f + s] = cost[a + s];
      } else {
        vec[a + s] = flat[off_vec + f + s];
        cost[a + s] = flat[off_cost + f + s];
      }
    }
  }
}

extern "C" int flowb200_slot_copy(const int64_t* table, int n_entries, int32_t* vec, float* cost, int width, int K,
                                  int32_t* flat, int to_flat, flowb200_stream_t stream) {
  if (n_entries < 0 || width <= 0 || K <= 0) return FLOWB200_EINVAL;
  if (n_entries == 0) return FLOWB200_OK;
  if (!table || !vec || !cost || !flat || n_entries > 65535) return FLOWB200_EINVAL;
  static_assert(sizeof(long long) == sizeof(int64_t), "table entries are 64-bit");
  slot_copy_kernel<<<dim3(64, (unsigned)n_entries), 256, 0, stream>>>(
      reinterpret_cast<const long long*>(table), vec, reinterpret_cast<int32_t*>(cost), width, K, flat, to_flat);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

extern "C" int flowb200_flow_from_labels(const int32_t* pvec, const int32_t* labels, int H, int W, int K,
                                         double* flow_yx, float* uvv, flowb200_stream_t stream) {
  if (!pvec || !labels || H <= 0 || W <= 0 || K <= 0) return FLOWB200_EINVAL;
  int n = H * W;
  flow_from_labels_kernel<<<(n + 255) / 256, 256, 0, stream>>>(pvec, labels, n, K, flow_yx, uvv);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

extern "C" int flowb200_flow_subpixel(const float* desc_src, const float* desc_tgt, const int32_t* pvec,
                                      const int32_t* nprop, const int32_t* labels, int H, int W, int K, float* uvv,
                                      flowb200_stream_t stream) {
  if (!desc_src || !desc_tgt || !pvec || !nprop || !labels || !uvv) return FLOWB200_EINVAL;
  if (H < 1 || W < 1 || K < 1 || K > 512 || (long long)H * W > INT_MAX) return FLOWB200_EINVAL;
  // descriptor rows are read as float4
  if ((reinterpret_cast<uintptr_t>(desc_src) | reinterpret_cast<uintptr_t>(desc_tgt)) & 15) return FLOWB200_EINVAL;
  const int n = H * W;
  subpixel_kernel<<<(n + 127) / 128, 128, 0, stream>>>(desc_src, desc_tgt, pvec, nprop, labels, H, W, K, uvv);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

extern "C" int flowb200_consistency(float* flow1, const float* flow2, int A, int B, float tresh, int a0, int a1,
                                    int b0, int b1, flowb200_stream_t stream) {
  if (!flow1 || !flow2 || A <= 0 || B <= 0) return FLOWB200_EINVAL;
  if (a0 < 0 || b0 < 0 || a1 > A || b1 > B || a0 > a1 || b0 > b1) return FLOWB200_EINVAL;
  // In place on flow1 while gathering flow2: when both alias, behaviour would be order dependent.
  if (flow1 == flow2) return FLOWB200_EINVAL;
  int n = (a1 - a0) * (b1 - b0);
  if (n == 0) return FLOWB200_OK;
  consistency_kernel<<<(n + 255) / 256, 256, 0, stream>>>(flow1, flow2, A, B, tresh, a0, a1, b0, b1);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

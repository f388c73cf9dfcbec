// Label -> flow gather and the forward/backward consistency check.
//   flow_from_labels : vratiKonacniFlow (daisy i flann.py:192-197 / python bcd.py:90-95) fused with
//                      FlowImage.ucitajFlow's (dx, dy, valid=1) float32 layout (postprocessing.py:7-17)
//   consistency      : consistencyCheck / fowardBackwardConsistency (postprocessing.py:79-117)
// Both are HBM-bound streaming kernels: 28 B/pixel algorithmic (SURVEY.md section 8d).
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

// Flow proposals: per-cell exact nearest neighbours (generisi), random-neighbour proposals (nasumicni)
// and the legacy K-set export (pakovanje).  Reference: `daisy i flann.py` :144-148, :157-189, :205-233,
// :256-309.  FLANN's approximate kd-forest (:164, :171-172) is replaced by an exact search.
#include <math_constants.h>

#include "common.cuh"

namespace flowb200 {

// ----------------------------------------------------------------------------------------------
// Exact brute-force k-NN on CUDA cores in float64 (FLOWB200_KNN_EXACT_FP64; also the certified
// fallback of the tcgen05 path).  distance(q,t) = sum_d (diff*diff), every product and every add rounded
// separately (no FMA), diff = double(q_d) - double(t_d), d ascending; ties -> lowest target index.
//
// grid = (query blocks of 128, cells); one thread per source pixel of the cell's +-r band; the cell's
// targets stream through shared memory as doubles in tiles of TT; every thread keeps its own sorted
// top-KC list in registers.  FP64-pipe bound: 2 DP ops per (query, target, dim).
// ----------------------------------------------------------------------------------------------
constexpr int kKnnThreads = 128;
constexpr int kKnnTT = 32;

struct KnnGeom {
  int H, W, cellw, cellh, ncellx, ncelly, R, K;
  float tphi;
};

template <int KC>
__device__ __forceinline__ void topk_insert(double (&bd)[KC], int (&bi)[KC], double d, int idx) {
  // list sorted ascending by (distance, index); idx is larger than every stored index, so the new
  // entry goes after all entries with distance <= d
  if (!(d < bd[KC - 1])) return;
#pragma unroll
  for (int j = KC - 1; j > 0; --j) {
    if (d < bd[j - 1]) {
      bd[j] = bd[j - 1];
      bi[j] = bi[j - 1];
    } else if (d < bd[j]) {
      bd[j] = d;
      bi[j] = idx;
    }
  }
  if (d < bd[0]) {
    bd[0] = d;
    bi[0] = idx;
  }
}

template <int KC>
__global__ void __launch_bounds__(kKnnThreads)
knn_exact_kernel(const float* __restrict__ desc_src, const float* __restrict__ desc_tgt, KnnGeom g,
                 int32_t* __restrict__ pvec, float* __restrict__ lcost, int32_t* __restrict__ knn_idx) {
  __shared__ __align__(16) double ts[kKnnTT][kDescDim];
  const int cell = blockIdx.y;
  const int ci = cell % g.ncellx, cj = cell / g.ncellx;
  const int x0 = max(0, g.cellw * (ci - g.R)), x1 = min(g.W, g.cellw * (ci + g.R + 1));
  const int y0 = max(0, g.cellh * (cj - g.R)), y1 = min(g.H, g.cellh * (cj + g.R + 1));
  const int bw = x1 - x0, nq = bw * (y1 - y0);
  if ((int)blockIdx.x * kKnnThreads >= nq) return;
  const int qi = blockIdx.x * kKnnThreads + threadIdx.x;
  const bool active = qi < nq;
  const int qy = y0 + (active ? qi / bw : 0), qx = x0 + (active ? qi % bw : 0);
  const float* qptr = desc_src + ((size_t)qy * g.W + qx) * kDescDim;

  double q[kDescDim];
#pragma unroll
  for (int d = 0; d < kDescDim; d += 4) {
    float4 v = *reinterpret_cast<const float4*>(qptr + d);
    q[d] = v.x; q[d + 1] = v.y; q[d + 2] = v.z; q[d + 3] = v.w;
  }
  double bd[KC];
  int bi[KC];
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    bd[j] = CUDART_INF;
    bi[j] = 0x7fffffff;
  }

  const int T = g.cellw * g.cellh;
  const int ty0 = cj * g.cellh, tx0 = ci * g.cellw;
  for (int tb = 0; tb < T; tb += kKnnTT) {
    __syncthreads();
    for (int e = threadIdx.x; e < kKnnTT * kDescDim; e += kKnnThreads) {
      int tt = e / kDescDim, d = e - tt * kDescDim;
      int idx = tb + tt;
      double v = 0.0;
      if (idx < T) {
        int r = idx / g.cellw, c = idx - r * g.cellw;
        v = (double)desc_tgt[((size_t)(ty0 + r) * g.W + (tx0 + c)) * kDescDim + d];
      }
      ts[tt][d] = v;
    }
    __syncthreads();
    const int nt = min(kKnnTT, T - tb);
    for (int tt = 0; tt < nt; tt += 4) {
      double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
      for (int d = 0; d < kDescDim; d += 2) {
        double2 t0 = *reinterpret_cast<const double2*>(&ts[tt][d]);
        double2 t1 = *reinterpret_cast<const double2*>(&ts[tt + 1][d]);
        double2 t2 = *reinterpret_cast<const double2*>(&ts[tt + 2][d]);
        double2 t3 = *reinterpret_cast<const double2*>(&ts[tt + 3][d]);
        double e;   // separately rounded multiply and add (no FMA): the oracle's `d += diff * diff`
        e = q[d] - t0.x; a0 = __dadd_rn(a0, __dmul_rn(e, e));
        e = q[d] - t1.x; a1 = __dadd_rn(a1, __dmul_rn(e, e));
        e = q[d] - t2.x; a2 = __dadd_rn(a2, __dmul_rn(e, e));
        e = q[d] - t3.x; a3 = __dadd_rn(a3, __dmul_rn(e, e));
        e = q[d + 1] - t0.y; a0 = __dadd_rn(a0, __dmul_rn(e, e));
        e = q[d + 1] - t1.y; a1 = __dadd_rn(a1, __dmul_rn(e, e));
        e = q[d + 1] - t2.y; a2 = __dadd_rn(a2, __dmul_rn(e, e));
        e = q[d + 1] - t3.y; a3 = __dadd_rn(a3, __dmul_rn(e, e));
      }
      topk_insert<KC>(bd, bi, a0, tb + tt);
      if (tt + 1 < nt) topk_insert<KC>(bd, bi, a1, tb + tt + 1);
      if (tt + 2 < nt) topk_insert<KC>(bd, bi, a2, tb + tt + 2);
      if (tt + 3 < nt) topk_insert<KC>(bd, bi, a3, tb + tt + 3);
    }
  }
  if (!active) return;

  // generisi bookkeeping (:173-189): slot order is ci-major, cj-minor, then rank
  int cimin, cimax, cjmin, cjmax;
  cell_range(qx, g.cellw, g.ncellx, g.R, &cimin, &cimax);
  cell_range(qy, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
  const int ncj = cjmax - cjmin + 1;
  const int blk = (ci - cimin) * ncj + (cj - cjmin);
  const size_t pix = (size_t)qy * g.W + qx;
  const int nblk = (2 * g.R + 1) * (2 * g.R + 1);
#pragma unroll
  for (int r = 0; r < KC; ++r) {
    const int idx = bi[r];
    const int tr = idx / g.cellw, tc = idx - tr * g.cellw;
    const int ty = ty0 + tr, tx = tx0 + tc;
    const float* tptr = desc_tgt + ((size_t)ty * g.W + tx) * kDescDim;
    float s = sum68_numpy_order([&](int d) { return fabsf(__fsub_rn((float)q[d], tptr[d])); });
    const int slot = KC * blk + r;
    pvec[pix * g.K + slot] = pack_vec(ty - qy, tx - qx);
    lcost[pix * g.K + slot] = s < g.tphi ? s : g.tphi;      // min(tphi, sum) (:178-180)
    if (knn_idx) knn_idx[(pix * nblk + blk) * KC + r] = idx;
  }
}

// nprop, unused-slot fill, and bestlabels = first strict argmin of the NN costs (:93, :181-184, :189)
__global__ void finish_nn_kernel(KnnGeom g, int KC, int32_t* __restrict__ pvec, float* __restrict__ lcost,
                                 int32_t* __restrict__ nprop, int32_t* __restrict__ labels,
                                 int32_t* __restrict__ knn_idx) {
  const int pix = blockIdx.x;
  const int qy = pix / g.W, qx = pix - qy * g.W;
  int cimin, cimax, cjmin, cjmax;
  cell_range(qx, g.cellw, g.ncellx, g.R, &cimin, &cimax);
  cell_range(qy, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
  const int nci = max(0, cimax - cimin + 1), ncj = max(0, cjmax - cjmin + 1);
  const int nn = KC * nci * ncj;
  for (int s = nn + threadIdx.x; s < g.K; s += blockDim.x) {
    pvec[(size_t)pix * g.K + s] = -1;
    lcost[(size_t)pix * g.K + s] = FLOWB200_UNUSED_COST;
  }
  if (knn_idx) {
    const int tot = (2 * g.R + 1) * (2 * g.R + 1) * KC;
    for (int s = nn + threadIdx.x; s < tot; s += blockDim.x) knn_idx[(size_t)pix * tot + s] = -1;
  }
  if (threadIdx.x == 0) {
    nprop[pix] = nn;
    float best = FLOWB200_UNUSED_COST;
    int lab = 0;
    for (int s = 0; s < nn; ++s) {
      float c = lcost[(size_t)pix * g.K + s];
      if (c < best) {
        best = c;
        lab = s;
      }
    }
    labels[pix] = lab;
  }
}

// ----------------------------------------------------------------------------------------------
// nasumicni (:205-233).  One thread per pixel; the 25 draws of a pixel are sequential because each
// accepted proposal changes the duplicate test of the next one.  Reads only NN slots of other
// pixels (never rewritten here), so pixels are independent.  The one exception, refused by
// flowb200_random_proposals: radius 0 on a frame that is no whole multiple of the cell, where the
// remainder pixels have no NN slot and publish their first random proposal in slot 0, which the
// reference's x-major scan shows to the pixels after them and not to those before.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mulhilo(uint32_t a, uint32_t b, uint32_t* hi) {
  uint64_t p = (uint64_t)a * b;
  *hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
}

__device__ inline uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0, hi1;
    uint32_t lo0 = mulhilo(0xD2511F53u, ctr.x, &hi0);
    uint32_t lo1 = mulhilo(0xCD9E8D57u, ctr.z, &hi1);
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// `tv in arr[a:b]` with Python slice semantics on the pixel's K proposal rows (quirk Q4):
// true when either component equals the same component of any row in the slice.
__device__ __forceinline__ bool in_slice(const int32_t* rows, int K, int a, int b, int tdy, int tdx) {
  a = a < 0 ? max(a + K, 0) : min(a, K);
  b = b < 0 ? max(b + K, 0) : min(b, K);
  bool hit = false;
  for (int r = a; r < b; ++r) {
    int32_t v = rows[r];
    hit |= (vec_dy(v) == tdy) | (vec_dx(v) == tdx);
  }
  return hit;
}

__global__ void random_proposals_kernel(const float* __restrict__ desc_src, const float* __restrict__ desc_tgt,
                                        KnnGeom g, int KC, int n_gauss, float sigma, int32_t* pvec, float* lcost,
                                        int32_t* nprop, const int32_t* __restrict__ labels,
                                        const int16_t* __restrict__ draws, uint64_t seed) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= g.H * g.W) return;
  const int y = pix / g.W, x = pix - y * g.W;
  const int mincellyl = max(0, y / g.cellh - 2);
  const int ncellyl = min(g.ncelly, y / g.cellh + 2) - mincellyl;   // :211, one too small (Q4)
  const int mincellxl = max(0, x / g.cellw - 2);
  int32_t* rows = pvec + (size_t)pix * g.K;
  float* crow = lcost + (size_t)pix * g.K;
  const float* d1 = desc_src + (size_t)pix * kDescDim;
  int n = nprop[pix];
  int ng = 0;
  uint32_t ctr = 0;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  for (int i = 0; i < n_gauss; ++i) {
    int tgy, tgx;
    if (draws) {
      tgy = draws[((size_t)pix * n_gauss + i) * 2];
      tgx = draws[((size_t)pix * n_gauss + i) * 2 + 1];
    } else {
      // int(np.random.normal(y, sigma)) then int(np.random.normal(x, sigma)); a sample outside the
      // image restarts the pair without counting (:216-222, :233)
      for (;;) {
        uint4 r = philox4x32_10(make_uint4((uint32_t)pix, ctr++, 0u, 0u), key);
        double u1 = ((double)r.x + 0.5) * (1.0 / 4294967296.0), u2 = ((double)r.y + 0.5) * (1.0 / 4294967296.0);
        double u3 = ((double)r.z + 0.5) * (1.0 / 4294967296.0), u4 = ((double)r.w + 0.5) * (1.0 / 4294967296.0);
        double zy = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        tgy = (int)((double)y + (double)sigma * zy);
        if (tgy < 0 || tgy >= g.H) continue;
        double zx = sqrt(-2.0 * log(u3)) * cospi(2.0 * u4);
        tgx = (int)((double)x + (double)sigma * zx);
        if (tgx < 0 || tgx >= g.W) continue;
        break;
      }
    }
    const int broj = KC * ((tgy / g.cellh - mincellyl) + (tgx / g.cellw - mincellxl) * ncellyl);
    const int tpix = tgy * g.W + tgx;
    const int32_t tv = pvec[(size_t)tpix * g.K + labels[tpix]];     // neighbour's pre-random best vector (:225)
    const int tdy = vec_dy(tv), tdx = vec_dx(tv);
    if (!in_slice(rows, g.K, broj, broj + KC, tdy, tdx) && !in_slice(rows, g.K, n - ng, n, tdy, tdx)) {
      const float* d2 = desc_tgt + (size_t)tpix * kDescDim;
      float s = sum68_numpy_order([&](int d) { return __fsub_rn(d1[d], d2[d]); });
      s = fabsf(s);                                                  // quirk Q6 (:228-229)
      rows[n] = tv;
      crow[n] = s < g.tphi ? s : g.tphi;
      ++n;
      ++ng;
    }
  }
  nprop[pix] = n;
}

// ----------------------------------------------------------------------------------------------
// pakovanje (:256-309): one thread per output byte of packedksets (np.packbits: MSB first).
// ----------------------------------------------------------------------------------------------
__global__ void ksets_pack_kernel(const int32_t* __restrict__ pvec, const int32_t* __restrict__ nprop, int H, int W,
                                  int K, int tpsi, int kdim, uint8_t* __restrict__ packed) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)H * W * 2 * kdim;
  if (t >= total) return;
  const int j = (int)(t % kdim);
  const size_t ps = t / kdim;
  const int slot = (int)(ps & 1);
  const int pix = (int)(ps >> 1);
  const int y = pix / W, x = pix - y * W;
  const int ny = slot == 0 ? y + 1 : y, nx = slot == 0 ? x : x + 1;
  uint8_t byte = 0;
  if (ny < H && nx < W) {
    const int np_ = nprop[pix], nq = nprop[ny * W + nx];
    const int32_t* vp = pvec + (size_t)pix * K;
    const int32_t* vq = pvec + (size_t)(ny * W + nx) * K;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int bit = j * 8 + b;
      if (bit >= K * K) break;
      const int l = bit / K, k = bit - l * K;
      if (l < np_ && k < nq) {
        const int32_t a = vp[l];
        if (l1_vec(vec_dy(a), vec_dx(a), vq[k]) < tpsi) byte |= (uint8_t)(0x80u >> b);
      }
    }
  }
  packed[t] = byte;
}

static KnnGeom make_geom(const flowb200_params* p) {
  KnnGeom g;
  g.H = p->H; g.W = p->W; g.cellw = p->cellw; g.cellh = p->cellh;
  g.ncellx = p->W / p->cellw; g.ncelly = p->H / p->cellh;
  g.R = p->cell_radius; g.K = p->maxnprop; g.tphi = p->tphi;
  return g;
}

static int check_params(const flowb200_params* p) {
  if (!p) return FLOWB200_EINVAL;
  if (p->H <= 0 || p->W <= 0 || p->cellw <= 0 || p->cellh <= 0 || p->cell_radius < 0) return FLOWB200_EINVAL;
  if (p->W / p->cellw < 1 || p->H / p->cellh < 1) return FLOWB200_EINVAL;
  if (p->H > 16384 || p->W > 16384) return FLOWB200_EINVAL;
  const int r = 2 * p->cell_radius + 1;
  if (p->k_cell < 1 || p->k_cell > p->cellw * p->cellh) return FLOWB200_EINVAL;
  if (p->n_gauss < 0 || p->maxnprop < r * r * p->k_cell + p->n_gauss || p->maxnprop > 512) return FLOWB200_EINVAL;
  return FLOWB200_OK;
}

template <int KC>
static int launch_knn_exact(const float* desc_src, const float* desc_tgt, const KnnGeom& g, int32_t* pvec, float* lcost,
                            int32_t* knn_idx, cudaStream_t stream) {
  const int r = 2 * g.R + 1;
  const int maxq = min(g.W, r * g.cellw) * min(g.H, r * g.cellh);
  dim3 grid((maxq + kKnnThreads - 1) / kKnnThreads, g.ncellx * g.ncelly);
  knn_exact_kernel<KC><<<grid, kKnnThreads, 0, stream>>>(desc_src, desc_tgt, g, pvec, lcost, knn_idx);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

int knn_exact_dispatch(const float* desc_src, const float* desc_tgt, const flowb200_params* p, int32_t* pvec,
                       float* lcost, int32_t* knn_idx, cudaStream_t stream) {
  const KnnGeom g = make_geom(p);
  switch (p->k_cell) {
    case 1: return launch_knn_exact<1>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 2: return launch_knn_exact<2>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 3: return launch_knn_exact<3>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 4: return launch_knn_exact<4>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 5: return launch_knn_exact<5>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 8: return launch_knn_exact<8>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 10: return launch_knn_exact<10>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 12: return launch_knn_exact<12>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    case 16: return launch_knn_exact<16>(desc_src, desc_tgt, g, pvec, lcost, knn_idx, stream);
    default: return FLOWB200_EUNSUPPORTED;
  }
}

int finish_nn(const flowb200_params* p, int32_t* pvec, float* lcost, int32_t* nprop, int32_t* labels, int32_t* knn_idx,
              cudaStream_t stream) {
  const KnnGeom g = make_geom(p);
  finish_nn_kernel<<<g.H * g.W, 64, 0, stream>>>(g, p->k_cell, pvec, lcost, nprop, labels, knn_idx);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

// knn_tc.cu
size_t knn_tc_workspace_bytes(const flowb200_params* p);
bool knn_tc_supported(const flowb200_params* p);
int knn_tc_dispatch(const float* desc_src, const float* desc_tgt, const flowb200_params* p, int32_t* pvec, float* lcost,
                    int32_t* nprop, int32_t* labels, int32_t* knn_idx, int32_t* stats, float* dbg_scores, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream);
int knn_tc_debug_scores(const float* desc_src, const float* desc_tgt, const flowb200_params* p, float* scores,
                        int32_t* geom_out_host, void* workspace, size_t workspace_bytes, cudaStream_t stream);

}  // namespace flowb200

using namespace flowb200;

extern "C" size_t flowb200_knn_workspace_bytes(const flowb200_params* p) {
  if (!p || check_params(p)) return 0;
  if (p->knn_mode == FLOWB200_KNN_TCGEN05 && knn_tc_supported(p)) return knn_tc_workspace_bytes(p);
  return 256;   // the exact float64 search needs no scratch
}

extern "C" int flowb200_knn_debug_scores(const float* desc_src, const float* desc_tgt, const flowb200_params* p,
                                         float* scores, int32_t* geom_out_host, void* workspace,
                                         size_t workspace_bytes, flowb200_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  return knn_tc_debug_scores(desc_src, desc_tgt, p, scores, geom_out_host, workspace, workspace_bytes, stream);
}

extern "C" int flowb200_knn_proposals(const float* desc_src, const float* desc_tgt, const flowb200_params* p,
                                      int32_t* pvec, float* lcost, int32_t* nprop, int32_t* labels, int32_t* knn_idx,
                                      int32_t* stats, void* workspace, size_t workspace_bytes,
                                      flowb200_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!desc_src || !desc_tgt || !pvec || !lcost || !nprop || !labels) return FLOWB200_EINVAL;
  if (p->knn_mode == FLOWB200_KNN_TCGEN05) {
    if (!workspace) return FLOWB200_EINVAL;
    // the tensor-core path also writes nprop, the unused-slot fills and bestlabels
    return knn_tc_dispatch(desc_src, desc_tgt, p, pvec, lcost, nprop, labels, knn_idx, stats, nullptr, workspace,
                           workspace_bytes, stream);
  } else if (p->knn_mode == FLOWB200_KNN_EXACT_FP64) {
    rc = knn_exact_dispatch(desc_src, desc_tgt, p, pvec, lcost, knn_idx, stream);
  } else {
    return FLOWB200_EINVAL;
  }
  if (rc) return rc;
  return finish_nn(p, pvec, lcost, nprop, labels, knn_idx, stream);
}

extern "C" int flowb200_random_proposals(const float* desc_src, const float* desc_tgt, const flowb200_params* p,
                                         int32_t* pvec, float* lcost, int32_t* nprop, const int32_t* labels,
                                         const int16_t* draws, uint64_t seed, flowb200_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!desc_src || !desc_tgt || !pvec || !lcost || !nprop || !labels) return FLOWB200_EINVAL;
  if (p->n_gauss == 0) return FLOWB200_OK;
  // radius 0, ragged frame: the result depends on the reference's scan order (see random_proposals_kernel)
  if (p->cell_radius == 0 && (p->H % p->cellh || p->W % p->cellw)) return FLOWB200_EUNSUPPORTED;
  const KnnGeom g = make_geom(p);
  const int n = g.H * g.W;
  random_proposals_kernel<<<(n + 127) / 128, 128, 0, stream>>>(desc_src, desc_tgt, g, p->k_cell, p->n_gauss, p->sigma,
                                                               pvec, lcost, nprop, labels, draws, seed);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

extern "C" int flowb200_ksets_pack(const int32_t* pvec, const int32_t* nprop, int H, int W, int K, int tpsi,
                                   uint8_t* packed, flowb200_stream_t stream) {
  if (!pvec || !nprop || !packed || H <= 0 || W <= 0 || K <= 0 || K > 512) return FLOWB200_EINVAL;
  const int kdim = K * K / 8 + 1;
  const size_t total = (size_t)H * W * 2 * kdim;
  if (total > ((size_t)1 << 38)) return FLOWB200_EINVAL;
  ksets_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(pvec, nprop, H, W, K, tpsi, kdim, packed);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

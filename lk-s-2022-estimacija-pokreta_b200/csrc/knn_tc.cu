// Per-cell exact k-NN, tensor-core path (FLOWB200_KNN_TCGEN05).  Replaces generisi's FLANN search
// (daisy i flann.py:157-189) with an exact one in three steps:
//
//  1. knn_prep_*      descriptors -> fp16 GEMM operands (scaled by 64), K = 68 -> 80:
//                       query row  q' = [ q~(68) | 1 1 1 | m_hi m_mid m_lo | 0.. ]   image layout [H][W][80]
//                       target row t' = [-t~(68) | n_hi n_mid n_lo | 1 1 1 | 0.. ]   cell-major   [cell][Tpad][80]
//                     with n = |t~|^2/2 and m = |q~|^2/2 split into three halves each, so that
//                     q'.t' = |q~|^2/2 + |t~|^2/2 - q~.t~ = |q~-t~|^2/2 =: a(q,t) >= 0: the accumulator IS the
//                     ranking score (m only shifts a row; it cancels in every comparison).
//                     Targets of a cell are stored in a decimating permutation (pos -> idx = pos*s mod T) so that
//                     every run of 32 columns is a spread-out sample of the cell.
//  2. knn_select_kernel  tcgen05 GEMM (TMA -> smem -> tcgen05.mma -> TMEM, M=128 queries x N=128 targets per MMA
//                     chunk, fp32 accumulate) with a fused selection epilogue read back with tcgen05.ld: every thread
//                     owns one query row.  A cell's targets are streamed twice: pass 0 keeps the k smallest
//                     32-column group minima (an upper bound tau on the k-th smallest score), pass 1 writes every
//                     column with score <= tau + 2*eps to the candidate array.  eps bounds |a - exact score|
//                     rigorously (fp16 rounding residual norms by Cauchy-Schwarz + fp32 accumulation slack), so the
//                     surviving candidate set provably contains the exact k nearest neighbours (ties included).
//  3. knn_rerank_kernel  exact float64 distances of the candidates (same arithmetic as the float64 brute force and
//                     the CPU oracle), rank by (distance, index), write the k proposals + float32 L1 data costs.
//     knn_fallback_kernel  (query, cell) pairs whose lists overflowed are redone by brute force.
//
// One CTA = one 16x8-pixel query tile x one target cell at a time (persistent over a static work list), 6 warps:
// warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue (one TMEM lane quadrant each).
// Three CTAs are resident per SM (128 TMEM columns each) so that one CTA's selection overlaps the others' MMAs.
// Measured in round 1 with the epilogue switched off: the TMA stream alone takes 1.8 ms and TMA + tcgen05.mma 2.8 ms
// per direction (tensor pipe 53 % busy); the selection epilogue is what bounds the kernel.
#include <cuda.h>
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace flowb200 {

constexpr int kKP = 80;            // padded contraction depth (5 x k16)
constexpr int kKB = 5;             // k16 blocks
constexpr float kScale = 64.0f;    // descriptors are < ~0.5: keeps fp16 values far from subnormals
constexpr int kTileW = 16, kTileH = 8, kTileM = 128;   // one MMA tile = one work item: 16 x 8 query pixels (two
                                                         // tiles per item halve the target stream but leave one CTA
                                                         // per SM: measured slower, the selection epilogue, not the
                                                         // stream, bounds the kernel)
constexpr int kChunkN = 128;       // targets per accumulator stage
// Two passes over a cell's targets (the GEMM is recomputed; the tensor pipe is mostly idle anyway): pass 0 only
// tracks the k smallest group minima (tau), pass 1 compares every score with the FINAL bound tau + 2 eps and
// writes the few survivors straight to the candidate array.  No shared-memory lists, no compaction; per 32 scores
// pass 0 issues ~36 instructions (group minimum + list insert) and pass 1 ~54 (16 packed subtractions, 32 sign-bit
// shifts, the mask assembly, one hit test per 128 columns) (a single-pass streaming selection with per-row lists in
// shared memory was built first: ~6.5 issue slots per score).
constexpr int kPasses = 2;
// The two-pass selection needs no shared-memory lists, so more CTAs fit an SM: with ONE accumulator stage (128 TMEM
// columns) three CTAs are resident and it is the other CTAs' epilogues, not a second accumulator stage of the same
// CTA, that overlap a CTA's MMAs (four CTAs per SM measured slower, DESIGN section 4.2).
constexpr int kCtasPerSM = 3;
constexpr int kBStages = 2;                              // target chunk stages in shared memory
constexpr int kTmemCols = kChunkN;                       // the one accumulator stage: 128 columns
constexpr int kSlabBytes = kTileM * 32;                  // one k16 block of 128 rows: 4096 B
constexpr int kTileBytes = kKB * kSlabBytes;             // 20480 B
constexpr int kCand = 32;          // candidates handed to the exact re-rank per (query, cell)
constexpr int kSelThreads = 64 + 128;                    // TMA warp, MMA warp, 4 epilogue warps
constexpr float kPadNorm = 60000.0f;   // n_hi of padding target rows: their score can never be selected

struct KnnTcGeom {
  int H, W, cellw, cellh, ncellx, ncelly, R, K, T, Tpad, stride_s, tiles_x, tiles_y, nblk;
  int cx0, cx1;   // target cell columns searched (flowb200_params.cell_x0 / cell_x1; all: 0, ncellx)
  uint32_t rcp_T, rcp_cellw;   // floor(2^32 / T), floor(2^32 / cellw): divisions by multiply-high + one fix-up step
  float tphi;
};

// ------------------------------------------------------------------------------------------------
// 1. operand preparation
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float up(float x) { return __fmul_ru(x, 1.0001f); }   // slack for fp32 rounding in the bounds

// one warp per pixel.  qinfo[pix] = (rq, Nq): rq >= |64 q - q~|_2, Nq >= |q~|_2
__global__ void knn_prep_query_kernel(const float* __restrict__ desc, int npix, __half* __restrict__ out,
                                      float2* __restrict__ qinfo) {
  const int pix = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pix >= npix) return;
  const float* d = desc + (size_t)pix * kDescDim;
  __half* o = out + (size_t)pix * kKP;
  float r2 = 0.f, n2 = 0.f;
  for (int j = lane; j < kKP; j += 32) {
    __half h = __float2half_rn(0.f);
    if (j < kDescDim) {
      const float v = d[j] * kScale;          // exact (power of two)
      h = __float2half_rn(v);
      const float hv = __half2float(h);
      const float e = v - hv;                 // exact (Sterbenz-like: hv is v rounded to 11 bits)
      r2 = fmaf(e, e, r2);
      n2 = fmaf(hv, hv, n2);
    } else if (j < kDescDim + 3) {
      h = __float2half_rn(1.0f);
    }
    if (j < kDescDim + 3 || j >= kDescDim + 6) o[j] = h;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    r2 += __shfl_xor_sync(0xffffffffu, r2, off);
    n2 += __shfl_xor_sync(0xffffffffu, n2, off);
  }
  if (lane == 0) {
    qinfo[pix] = make_float2(up(sqrtf(up(r2))), up(sqrtf(up(n2))));
    // slots 71..73: |q~|^2/2 in three halves (times the target's 1s): shifts every score of this row by the
    // same amount, which makes a = |q~ - t~|^2 / 2 >= 0 without changing the ranking
    const float nq = 0.5f * n2;
    const __half h0 = __float2half_rn(nq);
    const float r0 = nq - __half2float(h0);
    const __half h1 = __float2half_rn(r0);
    o[kDescDim + 3] = h0;
    o[kDescDim + 4] = h1;
    o[kDescDim + 5] = __float2half_rn(r0 - __half2float(h1));
  }
}

// Target operand layout: [cell][chunk of kChunkN targets][k16 block][row][16 halves], every (chunk, k16 block) slab
// already in the 32-byte-swizzled form the UMMA descriptor expects (byte-offset bit 4 ^= bit 7, i.e. the two
// 16-byte halves of rows 4-7 of every 8-row group are exchanged).  One chunk is then ONE contiguous 20 KB bulk
// copy instead of 5 x 128 strided 32-byte rows, which is what the L2 -> shared-memory path needs to run fast.
__device__ __forceinline__ size_t tgt_off(int cell, int nchunks, int pos, int j) {
  const int chunk = pos / kChunkN, row = pos - chunk * kChunkN;
  const int kb = j >> 4, jj = j & 15;
  const int h16 = (jj >> 3) ^ ((row >> 2) & 1);
  return (((size_t)cell * nchunks + chunk) * kKB + kb) * (size_t)(kChunkN * 16) + row * 16 + h16 * 8 + (jj & 7);
}

// one warp per (cell, pos).  cellinfo[cell] = (max rt, max Nt, max n) as float bit patterns (atomicMax on ints)
__global__ void knn_prep_target_kernel(const float* __restrict__ desc, KnnTcGeom g, __half* __restrict__ out,
                                       int* __restrict__ cellinfo) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int ncell = g.ncellx * g.ncelly;
  if (w >= ncell * g.Tpad) return;
  const int cell = w / g.Tpad, pos = w - cell * g.Tpad;
  const int nchunks = g.Tpad / kChunkN;
  if (pos >= g.T) {   // padding row
    for (int j = lane; j < kKP; j += 32) out[tgt_off(cell, nchunks, pos, j)] = __float2half_rn(j == kDescDim ? kPadNorm : 0.f);
    return;
  }
  const int idx = (int)(((long long)pos * g.stride_s) % g.T);
  const int ci = cell % g.ncellx, cj = cell / g.ncellx;
  const int ty = cj * g.cellh + idx / g.cellw, tx = ci * g.cellw + idx % g.cellw;
  const float* d = desc + ((size_t)ty * g.W + tx) * kDescDim;
  float r2 = 0.f, n2 = 0.f, s2 = 0.f;
  for (int j = lane; j < kDescDim; j += 32) {
    const float v = d[j] * kScale;
    const __half h = __float2half_rn(v);
    const float hv = __half2float(h);
    const float e = v - hv;
    r2 = fmaf(e, e, r2);
    n2 = fmaf(hv, hv, n2);
    s2 = fmaf(v, v, s2);
    out[tgt_off(cell, nchunks, pos, j)] = __float2half_rn(-hv);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    r2 += __shfl_xor_sync(0xffffffffu, r2, off);
    n2 += __shfl_xor_sync(0xffffffffu, n2, off);
    s2 += __shfl_xor_sync(0xffffffffu, s2, off);
  }
  // n = |t~|^2 / 2 as three halves (residual below 2^-30 n, covered by the accumulation slack in eps)
  const float n = 0.5f * n2;
  const __half h0 = __float2half_rn(n);
  const float r0 = n - __half2float(h0);
  const __half h1 = __float2half_rn(r0);
  const float r1 = r0 - __half2float(h1);
  const __half h2 = __float2half_rn(r1);
  for (int j = kDescDim + lane; j < kKP; j += 32) {
    out[tgt_off(cell, nchunks, pos, j)] = j == kDescDim ? h0 : j == kDescDim + 1 ? h1 : j == kDescDim + 2 ? h2
                                          : j < kDescDim + 6 ? __float2half_rn(1.0f) : __float2half_rn(0.f);
  }
  if (lane == 0) {
    // n as computed here differs from the exact |t~|^2/2 by fp32 rounding of n2: folded into rt's slack
    atomicMax(cellinfo + 4 * cell + 0, __float_as_int(up(sqrtf(up(r2)))));
    atomicMax(cellinfo + 4 * cell + 1, __float_as_int(up(sqrtf(up(fmaxf(s2, n2))))));
    atomicMax(cellinfo + 4 * cell + 2, __float_as_int(up(n)));
  }
}

// ------------------------------------------------------------------------------------------------
// 2. tcgen05 GEMM + streaming selection
// ------------------------------------------------------------------------------------------------
struct SelSmem {
  uint64_t a_full, a_empty;
  uint64_t b_full[kBStages], b_empty[kBStages];
  uint64_t t_full, t_empty;   // the accumulator stage
  uint32_t tmem_base;
};

__device__ __forceinline__ float fmin3(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// insert v into the ascending list (branch free): list keeps its KC smallest values
template <int KC>
__device__ __forceinline__ void list_insert(float (&lst)[KC], float v) {
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    const float lo = fminf(lst[j], v);
    v = fmaxf(lst[j], v);
    lst[j] = lo;
  }
}

// bb - {x0, x1} as one packed fp32 subtraction (FADD2 on sm_100); bb holds the bound twice
__device__ __forceinline__ void sub_f32x2(uint64_t bb, uint32_t x0, uint32_t x1, uint32_t& d0, uint32_t& d1) {
  asm("{\n\t.reg .b64 x, d;\n\tmov.b64 x, {%2, %3};\n\tsub.rn.f32x2 d, %4, x;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=r"(d0), "=r"(d1) : "r"(x0), "r"(x1), "l"(bb));
}

// decode a work item; returns false when the tile lies outside the cell's query band
__device__ __forceinline__ bool decode_item(const KnnTcGeom& g, int item, int& cell, int& qx0, int& qy0, int& x1,
                                            int& y1) {
  // cell-minor order: CTAs running at the same time stream DIFFERENT cells' targets, which spreads the L2 load
  // over all slices (with cell-major order every SM hammered the same 300 KB and the L2 slices holding it)
  const int ncell = g.ncellx * g.ncelly;
  const int t = item / ncell;
  cell = item - t * ncell;
  const int tyi = t / g.tiles_x, txi = t - tyi * g.tiles_x;
  const int ci = cell % g.ncellx, cj = cell / g.ncellx;
  if (ci < g.cx0 || ci >= g.cx1) return false;   // not this caller's band of target cells
  const int x0 = max(0, g.cellw * (ci - g.R)), y0 = max(0, g.cellh * (cj - g.R));
  x1 = min(g.W, g.cellw * (ci + g.R + 1));
  y1 = min(g.H, g.cellh * (cj + g.R + 1));
  qx0 = x0 + txi * kTileW;
  qy0 = y0 + tyi * kTileH;
  return qx0 < x1 && qy0 < y1;
}

template <int KC, bool DBG>
__global__ void __launch_bounds__(kSelThreads, kCtasPerSM)
knn_select_kernel(const __grid_constant__ CUtensorMap tmap_q, const __half* __restrict__ t16, KnnTcGeom g,
                  int n_items, const float2* __restrict__ qinfo, const int* __restrict__ cellinfo,
                  uint16_t* __restrict__ cand, uint8_t* __restrict__ cand_cnt, int32_t* __restrict__ counters,
                  int counters_on, float* __restrict__ dbg_scores) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                                                                     // [5 slabs]
  uint8_t* sB = smem + kTileBytes;                                                         // [stage][5 slabs]
  SelSmem* ss = reinterpret_cast<SelSmem*>(smem + kTileBytes * (1 + kBStages));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunks = g.Tpad / kChunkN;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_q);
    ptx::mbar_init(&ss->a_full, 1);
    ptx::mbar_init(&ss->a_empty, 1);
    for (int i = 0; i < kBStages; ++i) {
      ptx::mbar_init(&ss->b_full[i], 1);
      ptx::mbar_init(&ss->b_empty[i], 1);
    }
    ptx::mbar_init(&ss->t_full, 1);
    ptx::mbar_init(&ss->t_empty, 4);      // one arrival per epilogue warp
    ptx::fence_barrier_init();
  }
  if (warp == 1) ptx::tmem_alloc<kTmemCols>(&ss->tmem_base);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ss->tmem_base;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0, bcount = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        int cell, qx0, qy0, x1, y1;
        if (!decode_item(g, item, cell, qx0, qy0, x1, y1)) continue;
        ptx::mbar_wait_backoff(&ss->a_empty, (it & 1) ^ 1, 2000);
        ptx::mbar_arrive_expect_tx(&ss->a_full, kTileBytes);
#pragma unroll
        for (int kb = 0; kb < kKB; ++kb)
          ptx::tma_load_3d(sA + kb * kSlabBytes, &tmap_q, &ss->a_full, kb * 16, qx0, qy0);
        for (int cc = 0; cc < kPasses * nchunks; ++cc, ++bcount) {
          const int c = cc % nchunks;
          const uint32_t st = bcount % kBStages, ph = (bcount / kBStages) & 1;
          ptx::mbar_wait_backoff(&ss->b_empty[st], ph ^ 1, 100);
          ptx::mbar_arrive_expect_tx(&ss->b_full[st], kTileBytes);
          ptx::bulk_load(sB + st * kTileBytes, t16 + ((size_t)cell * nchunks + c) * (kTileBytes / 2), kTileBytes,
                         &ss->b_full[st]);
        }
        ++it;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = ptx::umma_idesc_f16(kTileM, kChunkN);
      uint32_t it = 0, bcount = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        int cell, qx0, qy0, x1, y1;
        if (!decode_item(g, item, cell, qx0, qy0, x1, y1)) continue;
        ptx::mbar_wait_backoff(&ss->a_full, it & 1, 1000);
        for (int cc = 0; cc < kPasses * nchunks; ++cc, ++bcount) {
          const uint32_t st = bcount % kBStages, ph = (bcount / kBStages) & 1;
          ptx::mbar_wait_backoff(&ss->b_full[st], ph, 100);
          ptx::mbar_wait_backoff(&ss->t_empty, (bcount & 1) ^ 1, 100);
          ptx::tc_fence_after();
#pragma unroll
          for (int kb = 0; kb < kKB; ++kb) {
            const uint64_t da = ptx::umma_desc_k_sw32(ptx::smem_u32(sA + kb * kSlabBytes));
            const uint64_t db = ptx::umma_desc_k_sw32(ptx::smem_u32(sB + st * kTileBytes + kb * kSlabBytes));
            ptx::mma_f16_ss(tmem_base, da, db, idesc, kb > 0 ? 1u : 0u);
          }
          ptx::mma_commit(&ss->b_empty[st]);     // B stage reusable once these MMAs have read it
          ptx::mma_commit(&ss->t_full);          // accumulator stage complete
        }
        ptx::mma_commit(&ss->a_empty);           // A tile reusable
        ++it;
      }
    }
  } else {
    // ===================== selection epilogue =====================
    {
      const int quad = warp & 3;                   // TMEM lane quadrant this warp may access
      const int row = quad * 32 + lane;            // query row of the tile = TMEM lane
      uint32_t bcount = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        int cell, qx0, qy0, x1, y1;
        if (!decode_item(g, item, cell, qx0, qy0, x1, y1)) continue;
        const int px = qx0 + (row & (kTileW - 1)), py = qy0 + (row >> 4);
        const bool valid = px < x1 && py < y1;
        const int pix = valid ? py * g.W + px : 0;
        // eps >= |a - exact score| for every target of the cell (see file header)
        const float2 qi = qinfo[pix];
        const float rt = __int_as_float(cellinfo[4 * cell + 0]), nt = __int_as_float(cellinfo[4 * cell + 1]);
        const float nmax = __int_as_float(cellinfo[4 * cell + 2]);
        const float eps = qi.x * nt + qi.y * rt + rt * (nt + rt) + 2.0e-5f * (qi.y * nt + nmax) + 1.0e-5f * nmax;
        const float eps2 = 2.0f * up(eps);
        size_t task = 0;
        if (valid) {
          const int ci = cell % g.ncellx, cj = cell / g.ncellx;
          int cimin, cimax, cjmin, cjmax;
          cell_range(px, g.cellw, g.ncellx, g.R, &cimin, &cimax);
          cell_range(py, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
          task = (size_t)pix * g.nblk + (ci - cimin) * (cjmax - cjmin + 1) + (cj - cjmin);
        }
        uint16_t* cand_row = cand + task * kCand;

        float lst[KC];
#pragma unroll
        for (int j = 0; j < KC; ++j) lst[j] = CUDART_INF_F;
        uint64_t bound2 = 0;   // the pass-1 bound, twice
        int ns = 0;

        // pass 0: one group = 32 consecutive score columns of this row; the k smallest group minima are k distinct
        // targets' scores, so the largest of them bounds the k-th smallest score of the cell from above
        auto track = [&](const uint32_t (&r)[32], int pos0, bool first) {
          if constexpr (DBG) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              dbg_scores[((size_t)item * kTileM + row) * g.Tpad + pos0 + j] = __uint_as_float(r[j]);
          }
          if (first) {   // first group of the cell: 16 pair minima (distinct elements) seed the list
#pragma unroll
            for (int j = 0; j < 16; ++j)
              list_insert<KC>(lst, fminf(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])));
          } else {
            float m[11];
#pragma unroll
            for (int j = 0; j < 10; ++j)
              m[j] = fmin3(__uint_as_float(r[3 * j]), __uint_as_float(r[3 * j + 1]), __uint_as_float(r[3 * j + 2]));
            m[10] = fminf(__uint_as_float(r[30]), __uint_as_float(r[31]));
            const float gm = fmin3(fmin3(m[0], m[1], m[2]), fmin3(m[3], m[4], m[5]),
                                   fmin3(fmin3(m[6], m[7], m[8]), m[9], m[10]));
            list_insert<KC>(lst, gm);
          }
        };
        // pass 1: every score x <= the final bound b is a candidate for the exact re-rank.  b is finite and not -0
        // (the list is seeded with 16 pair minima of the first group, T >= 32 >= KC, scores are finite: padding rows
        // score ~6e4, and eps2 >= +0), so x <= b exactly when the sign bit of RN(b - x) is clear: b - x = +0 when
        // they are equal, rounding and overflow to +-inf keep the sign, and without .ftz nothing is flushed (the
        // difference of two floats is never rounded to zero).  Returns bit 31 - j set when column j is ABOVE b.
        // Four independent chains of funnel shifts gather the sign bits of 8 consecutive columns each.
        auto above = [&](const uint32_t (&r)[32]) -> uint32_t {
          uint32_t m[4] = {0u, 0u, 0u, 0u};
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            uint32_t d0, d1;
            sub_f32x2(bound2, r[j], r[j + 1], d0, d1);
            m[j >> 3] = __funnelshift_l(d0, m[j >> 3], 1);
            m[j >> 3] = __funnelshift_l(d1, m[j >> 3], 1);
          }
          return (m[0] << 24) | (m[1] << 16) | (m[2] << 8) | m[3];
        };
        // the candidates of one 128-column chunk, in ascending position
        auto pick = [&](const uint32_t (&ab)[4], int cpos) {
          if ((ab[0] & ab[1] & ab[2] & ab[3]) == 0xffffffffu) return;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint32_t mask = __brev(~ab[q]);
            while (mask) {
              const int j = __ffs((int)mask) - 1;
              mask &= mask - 1;
              if (valid && ns < kCand) cand_row[ns] = (uint16_t)(cpos + 32 * q + j);   // position; knn_rerank maps
              ++ns;                                                                    // it to the index
            }
          }
        };

#pragma unroll 1
        for (int pass = 0; pass < kPasses; ++pass) {
#pragma unroll 1
          for (int c = 0; c < nchunks; ++c, ++bcount) {
            ptx::mbar_wait_backoff(&ss->t_full, bcount & 1, 100);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
            const int cpos = c * kChunkN;
            uint32_t r0[32], r1[32], ab[4];
            ptx::tmem_ld_32x32(taddr, r0);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int h = 0; h < kChunkN / 64; ++h) {
              ptx::tmem_ld_32x32(taddr + 64 * h + 32, r1);      // in flight while r0 is processed
              if (pass == 0) track(r0, cpos + 64 * h, c == 0 && h == 0);
              else ab[2 * h] = above(r0);
              ptx::tmem_ld_wait();
              if (h + 1 < kChunkN / 64) {
                ptx::tmem_ld_32x32(taddr + 64 * h + 64, r0);
              } else {
                ptx::tc_fence_before();                          // all TMEM reads of this stage are done
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&ss->t_empty);
              }
              if (pass == 0) track(r1, cpos + 64 * h + 32, false);
              else ab[2 * h + 1] = above(r1);
              ptx::tmem_ld_wait();
            }
            if (pass == 1) pick(ab, cpos);
          }
          const float bound = lst[KC - 1] + eps2;
          asm("mov.b64 %0, {%1, %1};" : "=l"(bound2) : "f"(bound));
        }
        int ns_stat = 0;
        if (valid) {
          cand_cnt[task] = ns > kCand ? 255 : (uint8_t)ns;
          if (ns > kCand) atomicAdd(counters + 2, 1);          // diagnostics (rare)
          else ns_stat = ns;
        }
        if (counters_on) {   // diagnostics: one atomic per warp and cell
          const int tot = __reduce_add_sync(0xffffffffu, ns_stat);
          if (lane == 0) atomicAdd(reinterpret_cast<unsigned long long*>(counters + 4), (unsigned long long)tot);
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<kTmemCols>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// 3. exact re-rank + data cost.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double exact_dist(const float* __restrict__ q, const float* __restrict__ t) {
  double acc = 0.0;
#pragma unroll
  for (int d = 0; d < kDescDim; d += 4) {
    const float4 a = *reinterpret_cast<const float4*>(q + d);
    const float4 b = *reinterpret_cast<const float4*>(t + d);
    double e;
    e = (double)a.x - (double)b.x; acc = __dadd_rn(acc, __dmul_rn(e, e));
    e = (double)a.y - (double)b.y; acc = __dadd_rn(acc, __dmul_rn(e, e));
    e = (double)a.z - (double)b.z; acc = __dadd_rn(acc, __dmul_rn(e, e));
    e = (double)a.w - (double)b.w; acc = __dadd_rn(acc, __dmul_rn(e, e));
  }
  return acc;
}

// candidate array entry -> target index inside the cell: the two-pass selection stores the POSITION in the cell's
// permuted target order (the modulo is cheaper here, one lane per candidate, than in the selection's hit loop)
// x / d and x % d for a divisor known on the host: q = mulhi(x, floor(2^32 / d)) is short of the quotient by at
// most one for every 32-bit x
__device__ __forceinline__ uint32_t divmod_rcp(uint32_t x, uint32_t d, uint32_t rcp, uint32_t& rem) {
  uint32_t q = __umulhi(x, rcp);
  uint32_t r = x - q * d;
  if (r >= d) { ++q; r -= d; }
  rem = r;
  return q;
}

__device__ __forceinline__ int cand_index(const KnnTcGeom& g, uint32_t c) {
  uint32_t rem;
  divmod_rcp(c * (uint32_t)g.stride_s, (uint32_t)g.T, g.rcp_T, rem);
  return (int)rem;
}

template <int KC>
__device__ __forceinline__ void emit_proposal(const KnnTcGeom& g, const float* __restrict__ q, const float* __restrict__ desc_tgt,
                                              int qx, int qy, int ci, int cj, int blk, int rank, int idx,
                                              int32_t* __restrict__ pvec, float* __restrict__ lcost,
                                              int32_t* __restrict__ knn_idx, unsigned long long* __restrict__ best64) {
  const int ty = cj * g.cellh + idx / g.cellw, tx = ci * g.cellw + idx % g.cellw;
  const float* t = desc_tgt + ((size_t)ty * g.W + tx) * kDescDim;
  const float s = sum68_numpy_order([&](int d) { return fabsf(__fsub_rn(q[d], t[d])); });
  const size_t pix = (size_t)qy * g.W + qx;
  const int slot = KC * blk + rank;
  pvec[pix * g.K + slot] = pack_vec(ty - qy, tx - qx);
  const float c = s < g.tphi ? s : g.tphi;
  lcost[pix * g.K + slot] = c;
  if (knn_idx) knn_idx[(pix * g.nblk + blk) * KC + rank] = idx;
  atomicMin(best64 + pix, ((unsigned long long)__float_as_uint(c) << 32) | (uint32_t)slot);
}

// One pass over a (query, target) descriptor pair:
//   ds   float32 screening distance, sum of fl(q-t)^2 with FMA.  All terms are >= 0, so it is within a relative
//        70 * 2^-24 = 4.2e-6 of the real-valued distance (and the float64 oracle value within 1e-14 of it);
//   cost the float32 L1 data cost sum |fl(q-t)| in numpy's pairwise order (daisy i flann.py:178-180), exactly as
//        sum68_numpy_order evaluates it.
// Every lane reads a DIFFERENT target row, and the L1 data pipe serves such a request one 32-byte sector per lane
// and pass: with 16-byte loads the kernel ran at 98 % of that pipe (17 passes per row).  The row is therefore read as
// its nine 32-byte sectors with 256-bit loads (sm_100).  Rows are 272 bytes apart, so every other row starts in the
// middle of a sector: the lane then works on the 72-float window that starts 4 floats before the row.  Window
// position k is dimension k - 4*odd, and k & 7 is a compile-time register index: accumulator r[k & 7] collects the
// dimensions numpy's r[(k - 4*odd) & 7] does, in the same order, and the final ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7))
// only exchanges its two halves (a commutative add).  Masked positions add +0, which changes no partial sum.
__device__ __forceinline__ void ldg256(const float* p, float (&v)[8]) {
  asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
      : "l"(p));
}

__device__ __forceinline__ void screen_and_cost(const float* __restrict__ q, const float* __restrict__ t, float& ds,
                                                float& cost) {
  const bool odd = (reinterpret_cast<uintptr_t>(t) & 16) != 0;
  const float* tb = t - (odd ? 4 : 0);          // 32-byte aligned
  const float* qb = q - (odd ? 4 : 0);          // same window over the query row (only its in-row part is read)
  float acc = 0.f, r[8], tail[4];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float w[8];
    ldg256(tb + 8 * i, w);
    const float4 a0 = *reinterpret_cast<const float4*>(i == 0 ? q : qb + 8 * i);   // (i = 0, odd: masked below)
    const float4 a1 = *reinterpret_cast<const float4*>(qb + 8 * i + 4);
    float e[8] = {__fsub_rn(a0.x, w[0]), __fsub_rn(a0.y, w[1]), __fsub_rn(a0.z, w[2]), __fsub_rn(a0.w, w[3]),
                  __fsub_rn(a1.x, w[4]), __fsub_rn(a1.y, w[5]), __fsub_rn(a1.z, w[6]), __fsub_rn(a1.w, w[7])};
    if (i == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) e[j] = odd ? 0.f : e[j];   // the four floats in front of an odd row
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc = fmaf(e[j], e[j], acc);
      r[j] = __fadd_rn(r[j], fabsf(e[j]));
    }
  }
  // last sector: window positions 64..67 (dimensions 64..67 of an even row, 60..63 of an odd one) and, for odd rows
  // only, 68..71 (their dimensions 64..67); an even row's second half belongs to the next pixel and is not read
  {
    const float4 x = *reinterpret_cast<const float4*>(tb + 64);
    const float4 a = *reinterpret_cast<const float4*>(qb + 64);
    float4 y = make_float4(0.f, 0.f, 0.f, 0.f), b = y;
    if (odd) {
      y = *reinterpret_cast<const float4*>(tb + 68);
      b = *reinterpret_cast<const float4*>(qb + 68);
    }
    const float ex[4] = {__fsub_rn(a.x, x.x), __fsub_rn(a.y, x.y), __fsub_rn(a.z, x.z), __fsub_rn(a.w, x.w)};
    const float ey[4] = {__fsub_rn(b.x, y.x), __fsub_rn(b.y, y.y), __fsub_rn(b.z, y.z), __fsub_rn(b.w, y.w)};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc = fmaf(ex[j], ex[j], acc);
      acc = fmaf(ey[j], ey[j], acc);
      r[j] = __fadd_rn(r[j], odd ? fabsf(ex[j]) : 0.f);
      tail[j] = odd ? fabsf(ey[j]) : fabsf(ex[j]);
    }
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
#pragma unroll
  for (int i = 0; i < 4; ++i) res = __fadd_rn(res, tail[i]);
  ds = acc;
  cost = res;
}

// Interval [screen_lo(ds), screen_hi(ds)] that certainly holds the real-valued distance of a screening distance ds.
// Relative part: 70 roundings of at most 2^-24 each (4.2e-6) for normal floats.  Absolute part: once partial sums are
// subnormal, every fma rounds by up to half a subnormal ulp (2^-150) whatever the size of its result, so 68 of them
// plus the rounding of the bound itself stay below 2^-142.  It matters at the rim of flat image regions, where
// descriptors of ~1e-20 give squared distances below 2^-126 that the fma chain cannot order.
__device__ __forceinline__ float screen_lo(float ds) { return ds * (1.0f - 1.0e-5f) - 0x1p-142f; }
__device__ __forceinline__ float screen_hi(float ds) { return ds * (1.0f + 1.0e-5f) + 0x1p-142f; }

__device__ __noinline__ double exact_dist_call(const float* __restrict__ q, const float* __restrict__ t) {
  return exact_dist(q, t);
}

// One half-warp per source pixel, looping over the pixel's cells (= blocks of the slot order); lane = candidate.
// Ranking uses the float32 screening distance wherever it decides the order with certainty (relative gap > 2e-5 and
// absolute gap > 2^-141, see screen_lo / screen_hi);
// candidates involved in an uncertain pair get the exact float64 distance of the oracle, so the final order is
// always the oracle's (distance, index) order.
template <int KC>
__global__ void __launch_bounds__(256, 4)
knn_rerank_kernel(const float* __restrict__ desc_src, const float* __restrict__ desc_tgt, KnnTcGeom g,
                  const uint16_t* __restrict__ cand, const uint8_t* __restrict__ cand_cnt, int32_t* __restrict__ pvec,
                  float* __restrict__ lcost, int32_t* __restrict__ knn_idx, int32_t* __restrict__ nprop,
                  unsigned long long* __restrict__ best64, int32_t* __restrict__ fb_list,
                  int32_t* __restrict__ fb_count, int fb_cap) {
  const int sub = threadIdx.x & 15;
  const size_t pix = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  if (pix >= (size_t)g.H * g.W) return;
  const unsigned gmask = 0xFFFFu << (threadIdx.x & 16);
  const int qy = (int)(pix / g.W), qx = (int)(pix - (size_t)qy * g.W);
  int cimin, cimax, cjmin, cjmax;
  cell_range(qx, g.cellw, g.ncellx, g.R, &cimin, &cimax);
  cell_range(qy, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
  const float* qp = desc_src + pix * kDescDim;
  // running (cost, slot) minimum of this lane's proposals: bestlabels = first strict argmin (:181-184) = the
  // lexicographic minimum; costs are >= 0, so their float bit patterns order like the values
  unsigned long long bkey = ((unsigned long long)__float_as_uint(FLOWB200_UNUSED_COST) << 32);
  int blk = 0;
  for (int ci = cimin; ci <= cimax; ++ci) {
    for (int cj = cjmin; cj <= cjmax; ++cj, ++blk) {
      const size_t task = pix * g.nblk + blk;
      if (ci < g.cx0 || ci >= g.cx1) continue;   // (uniform over the half-warp) another caller's band: slots left unwritten
      const int n = cand_cnt[task];
      if (n == 255) {
        if (sub == 0) {   // (past fb_cap the fallback finds the overflowed tasks in cand_cnt instead)
          const int at = atomicAdd(fb_count, 1);
          if (at < fb_cap) {
            fb_list[2 * at] = (int)pix;
            fb_list[2 * at + 1] = ci + cj * g.ncellx;
          }
        }
        continue;
      }
      const int ty0 = cj * g.cellh, tx0 = ci * g.cellw;
      // candidates 0..15 in round 0, 16..31 in round 1 (rare: only when more than 16 survived the prefilter)
      float ds0 = CUDART_INF_F, ds1 = CUDART_INF_F, co0 = 0.f, co1 = 0.f;
      int id0 = 0x7fffffff, id1 = 0x7fffffff;
      const float* tp0 = nullptr;
      const float* tp1 = nullptr;
      if (sub < n) {
        id0 = cand_index(g, cand[task * kCand + sub]);
        uint32_t cc;
        const int r = (int)divmod_rcp((uint32_t)id0, (uint32_t)g.cellw, g.rcp_cellw, cc);
        tp0 = desc_tgt + ((size_t)(ty0 + r) * g.W + tx0 + (int)cc) * kDescDim;
        screen_and_cost(qp, tp0, ds0, co0);
      }
      const bool two = n > 16;
      if (two && 16 + sub < n) {
        id1 = cand_index(g, cand[task * kCand + 16 + sub]);
        uint32_t cc;
        const int r = (int)divmod_rcp((uint32_t)id1, (uint32_t)g.cellw, g.rcp_cellw, cc);
        tp1 = desc_tgt + ((size_t)(ty0 + r) * g.W + tx0 + (int)cc) * kDescDim;
        screen_and_cost(qp, tp1, ds1, co1);
      }
      // rank by the screening distance; note every pair it cannot order with certainty
      const float lo0 = screen_lo(ds0), hi0 = screen_hi(ds0);
      const float lo1 = screen_lo(ds1), hi1 = screen_hi(ds1);
      int rank0 = 0, rank1 = 0;
      bool amb0 = false, amb1 = false;
      const int nl = n < 16 ? n : 16;   // (lanes >= n hold infinity: "certainly larger", they change nothing)
      if (!two) {   // (uniform over the half-warp) the common case: one round, candidates 0..n-1
        for (int l = 0; l < nl; ++l) {
          const float od = __shfl_sync(gmask, ds0, l, 16);     // (a shuffle is a pass of the L1 data pipe: send one value)
          const float ol = screen_lo(od), oh = screen_hi(od);
          rank0 += oh < lo0;                                   // certainly smaller
          amb0 |= (l != sub) && !(oh < lo0) && !(hi0 < ol);    // intervals overlap
        }
      } else {
        // (raw od < ds ranks like the intervals wherever they are disjoint, as lo <= ds <= hi; every pair where they
        // overlap is ambiguous and re-ranked below)
        for (int l = 0; l < 16; ++l) {
          const float od = __shfl_sync(gmask, ds0, l, 16);
          const float ol = screen_lo(od), oh = screen_hi(od);
          rank0 += od < ds0;
          amb0 |= (l != sub) && !(oh < lo0) && !(hi0 < ol);
          rank1 += od < ds1;
          amb1 |= !(oh < lo1) && !(hi1 < ol);
        }
        for (int l = 0; l < 16; ++l) {
          const float od = __shfl_sync(gmask, ds1, l, 16);
          const float ol = screen_lo(od), oh = screen_hi(od);
          rank0 += od < ds0;
          amb0 |= !(oh < lo0) && !(hi0 < ol);
          rank1 += od < ds1;
          amb1 |= (l != sub) && !(oh < lo1) && !(hi1 < ol);
        }
      }
      amb0 &= ds0 < CUDART_INF_F;      // (inf is "certainly larger" than every finite distance: hi < inf)
      amb1 &= ds1 < CUDART_INF_F;
      if (__any_sync(gmask, amb0 || amb1)) {
        // exact float64 distances for the uncertain candidates, then the oracle's (distance, index) order
        double dx0 = 0.0, dx1 = 0.0;
        if (amb0) dx0 = exact_dist_call(qp, tp0);
        if (amb1) dx1 = exact_dist_call(qp, tp1);
        rank0 = rank1 = 0;
        for (int o = 0; o < (two ? 2 : 1); ++o)
          for (int l = 0; l < 16; ++l) {
            const float od = __shfl_sync(gmask, o ? ds1 : ds0, l, 16);
            const int oi = __shfl_sync(gmask, o ? id1 : id0, l, 16);
            const bool oa = __shfl_sync(gmask, (int)(o ? amb1 : amb0), l, 16) != 0;
            const double ox = __shfl_sync(gmask, o ? dx1 : dx0, l, 16);
            rank0 += ((oa && amb0) ? (ox < dx0 || (ox == dx0 && oi < id0)) : (od < ds0)) ? 1 : 0;
            rank1 += ((oa && amb1) ? (ox < dx1 || (ox == dx1 && oi < id1)) : (od < ds1)) ? 1 : 0;
          }
      }
      const size_t obase = pix * g.K + (size_t)KC * blk;
      if (sub < n && rank0 < KC) {
        uint32_t cc;
        const int r = (int)divmod_rcp((uint32_t)id0, (uint32_t)g.cellw, g.rcp_cellw, cc);
        pvec[obase + rank0] = pack_vec(ty0 + r - qy, tx0 + (int)cc - qx);
        const float cc0 = co0 < g.tphi ? co0 : g.tphi;            // min(tphi, sum) (:178-180)
        lcost[obase + rank0] = cc0;
        const unsigned long long k0 = ((unsigned long long)__float_as_uint(cc0) << 32) | (uint32_t)(KC * blk + rank0);
        if (k0 < bkey) bkey = k0;
        if (knn_idx) knn_idx[(pix * g.nblk + blk) * KC + rank0] = id0;
      }
      if (two && 16 + sub < n && rank1 < KC) {
        uint32_t cc;
        const int r = (int)divmod_rcp((uint32_t)id1, (uint32_t)g.cellw, g.rcp_cellw, cc);
        pvec[obase + rank1] = pack_vec(ty0 + r - qy, tx0 + (int)cc - qx);
        const float cc1 = co1 < g.tphi ? co1 : g.tphi;
        lcost[obase + rank1] = cc1;
        const unsigned long long k1 = ((unsigned long long)__float_as_uint(cc1) << 32) | (uint32_t)(KC * blk + rank1);
        if (k1 < bkey) bkey = k1;
        if (knn_idx) knn_idx[(pix * g.nblk + blk) * KC + rank1] = id1;
      }
    }
  }
  // what finish_nn does for the float64 path: nprop, fills of the unused slots, and the pre-BCD best label
#pragma unroll
  for (int off = 8; off > 0; off >>= 1) {
    const unsigned long long o = __shfl_xor_sync(gmask, bkey, off, 16);
    if (o < bkey) bkey = o;
  }
  const int nn = KC * blk;
  if (sub == 0) {
    nprop[pix] = nn;
    best64[pix] = bkey;      // brute-forced tasks fold their proposals in with atomicMin (knn_fallback_kernel)
  }
  for (int sl = nn + sub; sl < g.K; sl += 16) {
    pvec[pix * g.K + sl] = -1;
    lcost[pix * g.K + sl] = FLOWB200_UNUSED_COST;
  }
  if (knn_idx)
    for (int sl = nn + sub; sl < g.nblk * KC; sl += 16) knn_idx[pix * (size_t)(g.nblk * KC) + sl] = -1;
}

__global__ void labels_from_best_kernel(const unsigned long long* __restrict__ best64, int32_t* __restrict__ labels, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) labels[i] = (int32_t)(best64[i] & 0xffffffffu);
}

// brute force of one (query, cell) task by the whole block (128 threads); fb_d: [T] doubles of shared memory
template <int KC>
__device__ void fallback_task(const float* __restrict__ desc_src, const float* __restrict__ desc_tgt, const KnnTcGeom& g,
                              int pix, int ci, int cj, double* fb_d, int32_t* __restrict__ pvec, float* __restrict__ lcost,
                              int32_t* __restrict__ knn_idx, unsigned long long* __restrict__ best64) {
  __shared__ double red_d[4];
  __shared__ int red_i[4];
  const int qy = pix / g.W, qx = pix - qy * g.W;
  const float* q = desc_src + (size_t)pix * kDescDim;
  const int ty0 = cj * g.cellh, tx0 = ci * g.cellw;
  __syncthreads();
  for (int i = threadIdx.x; i < g.T; i += blockDim.x) {
    const int r = i / g.cellw, c = i - r * g.cellw;
    fb_d[i] = exact_dist(q, desc_tgt + ((size_t)(ty0 + r) * g.W + tx0 + c) * kDescDim);
  }
  __syncthreads();
  int cimin, cimax, cjmin, cjmax;
  cell_range(qx, g.cellw, g.ncellx, g.R, &cimin, &cimax);
  cell_range(qy, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
  const int blk = (ci - cimin) * (cjmax - cjmin + 1) + (cj - cjmin);
  for (int rank = 0; rank < KC; ++rank) {
    double bd = CUDART_INF;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < g.T; i += blockDim.x)
      if (fb_d[i] < bd) {     // ascending i: strict < keeps the lowest index
        bd = fb_d[i];
        bi = i;
      }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, bd, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (od < bd || (od == bd && oi < bi)) {
        bd = od;
        bi = oi;
      }
    }
    if ((threadIdx.x & 31) == 0) {
      red_d[threadIdx.x >> 5] = bd;
      red_i[threadIdx.x >> 5] = bi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < 4; ++w)
        if (red_d[w] < bd || (red_d[w] == bd && red_i[w] < bi)) {
          bd = red_d[w];
          bi = red_i[w];
        }
      fb_d[bi] = CUDART_INF;
      emit_proposal<KC>(g, q, desc_tgt, qx, qy, ci, cj, blk, rank, bi, pvec, lcost, knn_idx, best64);
    }
    __syncthreads();
  }
}

// Brute force for the (rare) tasks whose candidate lists overflowed (cand_cnt == 255), one block per task.  The
// re-rank lists up to fb_cap of them.  When more overflowed (*fb_count > fb_cap: large flat regions, where every query
// ties with every target of a flat cell), the list is incomplete, and the blocks find every overflowed task by scanning
// cand_cnt instead: no task is dropped, and the workspace does not grow with the worst case.
template <int KC>
__global__ void __launch_bounds__(128)
knn_fallback_kernel(const float* __restrict__ desc_src, const float* __restrict__ desc_tgt, KnnTcGeom g,
                    const uint8_t* __restrict__ cand_cnt, const int32_t* __restrict__ fb_list,
                    const int32_t* __restrict__ fb_count, int fb_cap, int32_t* __restrict__ pvec,
                    float* __restrict__ lcost, int32_t* __restrict__ knn_idx, unsigned long long* __restrict__ best64) {
  extern __shared__ double fb_d[];       // [T]
  const int count = *fb_count;
  if (count <= fb_cap) {
    for (int t = blockIdx.x; t < count; t += gridDim.x) {
      const int cell = fb_list[2 * t + 1];
      fallback_task<KC>(desc_src, desc_tgt, g, fb_list[2 * t], cell % g.ncellx, cell / g.ncellx, fb_d, pvec, lcost,
                        knn_idx, best64);
    }
    return;
  }
  __shared__ int hit_pix[128], hit_ci[128], hit_cj[128];
  __shared__ int nhit;
  const size_t ntask = (size_t)g.H * g.W * g.nblk;
  for (size_t base = (size_t)blockIdx.x * blockDim.x; base < ntask; base += (size_t)gridDim.x * blockDim.x) {
    const size_t task = base + threadIdx.x;
    __syncthreads();                     // the previous chunk's hits are consumed
    if (threadIdx.x == 0) nhit = 0;
    __syncthreads();
    // cand_cnt holds no value for tasks past a pixel's cell window (which is empty for a pixel of the remainder strip
    // when R = 0) or of cells outside [cx0, cx1): those are skipped before their block number is decoded
    if (task < ntask && cand_cnt[task] == 255) {
      const int pix = (int)(task / g.nblk), blk = (int)(task - (size_t)pix * g.nblk);
      const int qy = pix / g.W, qx = pix - qy * g.W;
      int cimin, cimax, cjmin, cjmax;
      cell_range(qx, g.cellw, g.ncellx, g.R, &cimin, &cimax);
      cell_range(qy, g.cellh, g.ncelly, g.R, &cjmin, &cjmax);
      const int nbx = cimax - cimin + 1, nby = cjmax - cjmin + 1;
      if (nbx > 0 && nby > 0 && blk < nbx * nby) {
        const int ci = cimin + blk / nby, cj = cjmin + blk % nby;
        if (ci >= g.cx0 && ci < g.cx1) {
          const int h = atomicAdd(&nhit, 1);
          hit_pix[h] = pix;
          hit_ci[h] = ci;
          hit_cj[h] = cj;
        }
      }
    }
    __syncthreads();
    const int nh = nhit;
    for (int h = 0; h < nh; ++h)           // (tasks write disjoint slots; best64 is an atomic minimum: any order)
      fallback_task<KC>(desc_src, desc_tgt, g, hit_pix[h], hit_ci[h], hit_cj[h], fb_d, pvec, lcost, knn_idx, best64);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 3-D fp16 tensor map {80 halves, d1, d2}, box {16, b1, b2}, 32-byte swizzle
static bool make_map(CUtensorMap* m, void* base, uint64_t d1, uint64_t d2, uint32_t b1, uint32_t b2) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)kKP, d1, d2};
  cuuint64_t strides[2] = {(cuuint64_t)kKP * 2, (cuuint64_t)kKP * 2 * d1};
  cuuint32_t box[3] = {16, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
         CUDA_SUCCESS;
}

static int gcd_i(int a, int b) { return b ? gcd_i(b, a % b) : a; }

static KnnTcGeom make_tc_geom(const flowb200_params* p) {
  KnnTcGeom g;
  g.H = p->H; g.W = p->W; g.cellw = p->cellw; g.cellh = p->cellh;
  g.ncellx = p->W / p->cellw; g.ncelly = p->H / p->cellh;
  g.R = p->cell_radius; g.K = p->maxnprop; g.tphi = p->tphi;
  g.T = p->cellw * p->cellh;
  g.Tpad = (g.T + kChunkN - 1) / kChunkN * kChunkN;
  int s = (int)(0.41421356 * g.T);
  if (s < 1) s = 1;
  while (gcd_i(s, g.T) != 1) ++s;
  g.stride_s = s;
  g.rcp_T = g.T > 1 ? (uint32_t)((1ull << 32) / (uint64_t)g.T) : 0xffffffffu;
  g.rcp_cellw = g.cellw > 1 ? (uint32_t)((1ull << 32) / (uint64_t)g.cellw) : 0xffffffffu;
  const int r = 2 * g.R + 1;
  g.tiles_x = (min(g.W, r * g.cellw) + kTileW - 1) / kTileW;
  g.tiles_y = (min(g.H, r * g.cellh) + kTileH - 1) / kTileH;
  g.nblk = r * r;
  g.cx0 = 0;
  g.cx1 = g.ncellx;
  if (p->cell_x1 > p->cell_x0) {
    g.cx0 = max(0, p->cell_x0);
    g.cx1 = min(g.ncellx, p->cell_x1);
  }
  return g;
}

struct TcLayout {
  size_t q16, t16, qinfo, cellinfo, cand, cnt, best, fb_list, fb_count, total;
  int grid, fb_cap;
};

static TcLayout tc_layout(const flowb200_params* p) {
  const KnnTcGeom g = make_tc_geom(p);
  TcLayout L{};
  const size_t n = (size_t)g.H * g.W, ncell = (size_t)g.ncellx * g.ncelly;
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off += align_up(b, 1024); return o; };
  L.grid = kCtasPerSM * kNumSMs;
  L.fb_cap = 1 << 20;
  L.q16 = take(n * kKP * 2);
  L.t16 = take(ncell * g.Tpad * kKP * 2);
  L.qinfo = take(n * sizeof(float2));
  L.cellinfo = take(ncell * 4 * sizeof(int));
  L.cand = take(n * g.nblk * kCand * sizeof(uint16_t));
  L.cnt = take(n * g.nblk);
  L.best = take(n * sizeof(unsigned long long));
  L.fb_list = take((size_t)L.fb_cap * 2 * sizeof(int32_t));
  L.fb_count = take(256);
  L.total = off;
  return L;
}

size_t knn_tc_workspace_bytes(const flowb200_params* p) { return tc_layout(p).total; }

bool knn_tc_supported(const flowb200_params* p) {
  const int T = p->cellw * p->cellh;
  return T >= 32 && T <= 2048 && (p->k_cell == 5 || p->k_cell == 10 || p->k_cell == 12) && p->k_cell <= 16 &&
         T >= p->k_cell;
}

template <int KC>
static int run_tc(const float* desc_src, const float* desc_tgt, const flowb200_params* p, const KnnTcGeom& g,
                  const TcLayout& L, char* ws, int32_t* pvec, float* lcost, int32_t* nprop, int32_t* labels,
                  int32_t* knn_idx, int32_t* stats,
                  float* dbg_scores, cudaStream_t stream) {
  const size_t n = (size_t)g.H * g.W;
  const int ncell = g.ncellx * g.ncelly;
  __half* q16 = reinterpret_cast<__half*>(ws + L.q16);
  __half* t16 = reinterpret_cast<__half*>(ws + L.t16);
  float2* qinfo = reinterpret_cast<float2*>(ws + L.qinfo);
  int* cellinfo = reinterpret_cast<int*>(ws + L.cellinfo);
  uint16_t* cand = reinterpret_cast<uint16_t*>(ws + L.cand);
  uint8_t* cnt = reinterpret_cast<uint8_t*>(ws + L.cnt);
  int32_t* fb_list = reinterpret_cast<int32_t*>(ws + L.fb_list);
  int32_t* fb_count = reinterpret_cast<int32_t*>(ws + L.fb_count);
  unsigned long long* best64 = reinterpret_cast<unsigned long long*>(ws + L.best);

  FB_CUDA_CHECK(cudaMemsetAsync(cellinfo, 0, (size_t)ncell * 4 * sizeof(int), stream));
  FB_CUDA_CHECK(cudaMemsetAsync(fb_count, 0, 8 * sizeof(int32_t), stream));
  knn_prep_query_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, stream>>>(desc_src, (int)n, q16, qinfo);
  FB_LAUNCH_CHECK();
  const size_t tw = (size_t)ncell * g.Tpad;
  knn_prep_target_kernel<<<(unsigned)((tw * 32 + 255) / 256), 256, 0, stream>>>(desc_tgt, g, t16, cellinfo);
  FB_LAUNCH_CHECK();

  CUtensorMap mq;
  if (!make_map(&mq, q16, (uint64_t)g.W, (uint64_t)g.H, kTileW, kTileH)) return FLOWB200_ECUDA;
  const int n_items = ncell * g.tiles_x * g.tiles_y;
  const size_t smem = (size_t)kTileBytes * (1 + kBStages) + sizeof(SelSmem) + 1024;
  auto kern = dbg_scores ? knn_select_kernel<KC, true> : knn_select_kernel<KC, false>;
  FB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = min(L.grid, n_items);
  kern<<<grid, kSelThreads, smem, stream>>>(mq, t16, g, n_items, qinfo, cellinfo, cand, cnt, fb_count, stats != nullptr, dbg_scores);
  FB_LAUNCH_CHECK();

  const unsigned rgrid = (unsigned)((n * 16 + 255) / 256);
  knn_rerank_kernel<KC><<<rgrid, 256, 0, stream>>>(desc_src, desc_tgt, g, cand, cnt, pvec, lcost, knn_idx, nprop, best64,
                                                    fb_list, fb_count, L.fb_cap);
  FB_LAUNCH_CHECK();
  auto fkern = knn_fallback_kernel<KC>;
  const size_t fsmem = (size_t)g.T * sizeof(double);
  if (fsmem > 48 * 1024) FB_CUDA_CHECK(cudaFuncSetAttribute(fkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
  fkern<<<4 * kNumSMs, 128, fsmem, stream>>>(desc_src, desc_tgt, g, cnt, fb_list, fb_count, L.fb_cap, pvec, lcost,
                                             knn_idx, best64);
  FB_LAUNCH_CHECK();
  labels_from_best_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(best64, labels, (int)n);
  FB_LAUNCH_CHECK();
  // stats: {fallback tasks, 0, candidate-list overflows, 0, sum of candidates as one uint64 in slots 4-5}
  if (stats) FB_CUDA_CHECK(cudaMemcpyAsync(stats, fb_count, 6 * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
  (void)p;
  return FLOWB200_OK;
}

int knn_tc_dispatch(const float* desc_src, const float* desc_tgt, const flowb200_params* p, int32_t* pvec, float* lcost,
                    int32_t* nprop, int32_t* labels, int32_t* knn_idx, int32_t* stats, float* dbg_scores, void* workspace, size_t workspace_bytes,
                    cudaStream_t stream) {
  if (!knn_tc_supported(p)) return FLOWB200_EUNSUPPORTED;
  const TcLayout L = tc_layout(p);
  if (workspace_bytes < L.total) return FLOWB200_EWORKSPACE;
  const KnnTcGeom g = make_tc_geom(p);
  char* ws = static_cast<char*>(workspace);
  switch (p->k_cell) {
    case 5: return run_tc<5>(desc_src, desc_tgt, p, g, L, ws, pvec, lcost, nprop, labels, knn_idx, stats, dbg_scores,
                               stream);
    case 10: return run_tc<10>(desc_src, desc_tgt, p, g, L, ws, pvec, lcost, nprop, labels, knn_idx, stats, dbg_scores,
                               stream);
    case 12: return run_tc<12>(desc_src, desc_tgt, p, g, L, ws, pvec, lcost, nprop, labels, knn_idx, stats, dbg_scores,
                               stream);
    default: return FLOWB200_EUNSUPPORTED;
  }
}

int knn_tc_debug_scores(const float* desc_src, const float* desc_tgt, const flowb200_params* p, float* scores,
                        int32_t* geom_out_host, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!knn_tc_supported(p)) return FLOWB200_EUNSUPPORTED;
  const TcLayout L = tc_layout(p);
  const KnnTcGeom g = make_tc_geom(p);
  if (geom_out_host) {
    geom_out_host[0] = g.Tpad; geom_out_host[1] = g.stride_s; geom_out_host[2] = g.tiles_x;
    geom_out_host[3] = g.tiles_y; geom_out_host[4] = g.ncellx * g.ncelly * g.tiles_x * g.tiles_y;
    geom_out_host[5] = kTileW; geom_out_host[6] = kTileH; geom_out_host[7] = kCand;
  }
  if (!scores) return FLOWB200_OK;
  if (workspace_bytes < L.total) return FLOWB200_EWORKSPACE;
  const size_t n = (size_t)g.H * g.W;   // the proposals of this diagnostic run go to a throw-away allocation
  int32_t *pvec = nullptr, *np_ = nullptr, *lb_ = nullptr;
  float* lcost = nullptr;
  FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&pvec), n * g.K * sizeof(int32_t)));
  FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&lcost), n * g.K * sizeof(float)));
  FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&np_), n * sizeof(int32_t)));
  FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&lb_), n * sizeof(int32_t)));
  int rc = knn_tc_dispatch(desc_src, desc_tgt, p, pvec, lcost, np_, lb_, nullptr, nullptr, scores, workspace,
                           workspace_bytes, stream);
  cudaStreamSynchronize(stream);
  cudaFree(pvec);
  cudaFree(lcost);
  cudaFree(np_);
  cudaFree(lb_);
  return rc;
}

}  // namespace flowb200

// Block-coordinate-descent MRF inference: row/column chain Viterbi over the K proposal labels.
// Reference: `python bcd.py` bcd() :101-257 (one chain), ceoBCD() :261-284 (phase order), sidepsi :84-88; see
// oracle/bcd.py for the recurrence in words.  Arithmetic modes (include/flowb200.h): float64 with the reference's
// operation order, or uint32 in units of 2^-S.
//
// It is organised around what the reference itself does -- it evaluates the K-sets S_l = {k : L1(v_l, u_k) < tpsi}
// ONCE per proposal set (pakovanje, daisy i flann.py:256-309, the 2.6 GB packedksets cache) and only reads them inside
// bcd() (python bcd.py:131-142).  Here the cache is sparse:
//
//   kset_sort_kernel   per pixel: label indices (and vectors) ordered by the spatial-hash bucket of the flow vector
//   kset_build_kernel  per (pixel, chain orientation): one RECORD = everything a chain step needs, contiguous (layout
//                      at the kernel).  Only pairs with L1 < tpsi are stored, as uint16 entries (k << 3 | L1 << 12),
//                      labels ordered by decreasing list length, every list padded to whole groups of four entries.
//                      Records are carved from an arena with one atomic cursor; a 64-bit descriptor per record
//                      (offset | size) is the only index.  All (pixel, orientation) pairs are independent, so this
//                      kernel is throughput bound, unlike the chains.
//   kset_chain32_kernel  one CTA per chain, one thread per label position.  One thread streams the chain's records
//                      into a ring of shared-memory slots with bulk asynchronous copies (TMA engine, mbarrier
//                      completion) four steps ahead; a step is: wait for the slot, lexicographic minimum over the
//                      label's entry list of (dp[k] + (L1 << S), k), add the unary term, publish the new dp, one block
//                      barrier.  dp is a uint32 in units of 2^-S; (dp, label) pairs order like np.argmin does
//                      (python bcd.py:155/:175/:234: smallest value, lowest index on ties).
//   kset_chainf64_kernel  the float64 programme (FLOWB200_BCD_FP64_*) on the same records, steps without a stored
//                      record evaluated densely.  Its integer variant runs the int32 programme, exactly, on the chains
//                      the 32-bit kernel cannot (a step without a stored record, K = 512), which it flags.
//
// A record that does not fit (arena exhausted, staging or slot too small, list longer than 124, data cost out of 16
// bits) gets descriptor 0 and
// its step is evaluated densely from pvec/cost inside the chain kernel, so any workspace size gives the exact result.
// Records are built for tpsi 1..8 (an entry holds L1 in 3 bits) and, in the int32 modes, cost shifts 4..14.  Other
// inputs (tpsi 0 or 9..32, cost shift 0..3) get no records: every descriptor is 0 and every step is evaluated densely.
// Precondition of the int32 modes: 0 <= m < 65536 for every used slot (the uint32 dp bound of make_plan assumes it).
#include <math_constants.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace flowb200 {

namespace {

struct ChainGeom {
  int sy, sx, ystep, xstep, len;
};

__device__ __forceinline__ ChainGeom chain_geom(int phase, int c, int H, int W) {
  ChainGeom g;
  switch (phase) {
    case 0: g = {0, 2 * c, 1, 0, H}; break;           // even columns, downwards   (:265-266)
    case 1: g = {2 * c, W - 1, 0, -1, W}; break;      // even rows, right to left  (:270-271)
    case 2: g = {H - 1, 2 * c + 1, -1, 0, H}; break;  // odd columns, upwards      (:273-274)
    default: g = {2 * c + 1, 0, 0, 1, W}; break;      // odd rows, left to right   (:276-277)
  }
  return g;
}

int phase_chains(int phase, int H, int W) {
  switch (phase) {
    case 0: return (W + 1) / 2;
    case 1: return (H + 1) / 2;
    case 2: return W / 2;
    default: return H / 2;
  }
}

// Spatial hash of flow vectors: bucket edge 2^bshift >= tpsi, 16 x 64 buckets (offset and clamped), so that every
// u with L1(v, u) < tpsi lies in the 3 x 3 buckets around v's bucket.
constexpr int kHashY = 16, kHashX = 64, kHashSize = kHashY * kHashX;
// bucket coordinates are offset and clamped (not wrapped) so that buckets adjacent in x have consecutive keys:
// the labels of three x-adjacent buckets form ONE contiguous range.  Clamping merges far-away buckets into the
// border ones, which is harmless because membership is always decided by the exact L1 test.
__device__ __forceinline__ int bkt_y(int b) { return min(max(b + kHashY / 2, 0), kHashY - 1); }
__device__ __forceinline__ int bkt_x(int b) { return min(max(b + kHashX / 2, 0), kHashX - 1); }
__device__ __forceinline__ int bucket_key(int32_t v, int bshift) {
  return (bkt_y(vec_dy(v) >> bshift) << 6) | bkt_x(vec_dx(v) >> bshift);
}

constexpr uint32_t kRngEmpty = 0x0000FFFFu;   // first = 0xFFFF, last+1 = 0
constexpr int kRecHeader = 16;

__device__ __forceinline__ int cidx(int k) { return k + (k >> 5); }

template <typename CostT>
__device__ __forceinline__ int32_t quant_cost(CostT c, double lamda, int shift) {
  if constexpr (std::is_integral<CostT>::value) return (int32_t)c;
  else return (int32_t)rint(__dmul_rn(__dmul_rn(lamda, (double)c), (double)(1 << shift)));
}

// ------------------------------------------------------------------------------------------------
// energy (SURVEY 8a): E = lamda * sum_p lcost(p, l_p) + sum over 4-connected pairs of min(L1(v_p, v_q), tpsi), in the
// arithmetic of the mode: QUANT (int32 modes) sums quant_cost and min(L1, tpsi) << shift as integers (exact);
// otherwise the data term is a float64 sum of lamda * lcost.  One CTA: every thread sums a fixed set of pixels, then
// a fixed tree, so that repeated calls give the same bits.  Pixels whose label is outside [0, nprop) are counted and
// left out, with every pair they belong to.
// ------------------------------------------------------------------------------------------------
constexpr int kEnergyThreads = 1024;

template <typename CostT, bool QUANT>
__global__ void __launch_bounds__(kEnergyThreads)
energy_kernel(const int32_t* __restrict__ pvec, const CostT* __restrict__ cost, const int32_t* __restrict__ nprop,
              const int32_t* __restrict__ labels, int H, int W, int K, double lamda, int tpsi, int shift,
              double* __restrict__ out4) {
  __shared__ double fd_s[kEnergyThreads];
  __shared__ long long qd_s[kEnergyThreads], pw_s[kEnergyThreads], bad_s[kEnergyThreads];
  const int t = threadIdx.x;
  const int npix = H * W;
  auto valid = [&](int p, int l) { return l >= 0 && l < nprop[p]; };
  double fd = 0.0;
  long long qd = 0, pw = 0, bad = 0;
  for (int p = t; p < npix; p += kEnergyThreads) {
    const int l = labels[p];
    if (!valid(p, l)) {
      ++bad;
      continue;
    }
    const CostT c = cost[(size_t)p * K + l];
    if constexpr (QUANT) qd += quant_cost<CostT>(c, lamda, shift);
    else fd = __dadd_rn(fd, __dmul_rn(lamda, (double)c));
    const int32_t v = pvec[(size_t)p * K + l];
    const int y = p / W, x = p - y * W;
    if (x + 1 < W && valid(p + 1, labels[p + 1]))
      pw += min(tpsi, l1_vec(vec_dy(v), vec_dx(v), pvec[(size_t)(p + 1) * K + labels[p + 1]]));
    if (y + 1 < H && valid(p + W, labels[p + W]))
      pw += min(tpsi, l1_vec(vec_dy(v), vec_dx(v), pvec[(size_t)(p + W) * K + labels[p + W]]));
  }
  fd_s[t] = fd;
  qd_s[t] = qd;
  pw_s[t] = pw;
  bad_s[t] = bad;
  __syncthreads();
  for (int s = kEnergyThreads / 2; s > 0; s >>= 1) {
    if (t < s) {
      fd_s[t] = __dadd_rn(fd_s[t], fd_s[t + s]);
      qd_s[t] += qd_s[t + s];
      pw_s[t] += pw_s[t + s];
      bad_s[t] += bad_s[t + s];
    }
    __syncthreads();
  }
  if (t == 0) {
    const double pair = (double)pw_s[0];
    if constexpr (QUANT) {   // in units of 2^-shift: every sum below 2^53, so exact
      const double unit = 1.0 / (double)(1 << shift);
      out4[0] = (double)qd_s[0] * unit;
      out4[1] = pair;
      out4[2] = (double)(qd_s[0] + (pw_s[0] << shift)) * unit;
    } else {
      out4[0] = fd_s[0];
      out4[1] = pair;
      out4[2] = __dadd_rn(fd_s[0], pair);
    }
    out4[3] = (double)bad_s[0];
  }
}

// ------------------------------------------------------------------------------------------------
// sort: one warp per pixel, counting sort of the label indices by bucket key (order inside a bucket is arbitrary)
// ------------------------------------------------------------------------------------------------
constexpr int kSortWarps = 8;
constexpr int kCntSize = kHashSize + kHashSize / 32;   // 1056, a multiple of 4

// single-huge-image mode: line (column x or row y) `line` of `nlines` belongs to chain line >> 1 of its parity's
// phase; part `part` of `nparts` runs a contiguous share of every phase's chains (the range of ksets_phase on the host)
__device__ __forceinline__ bool owns_line(int line, int nlines, int part, int nparts) {
  const long long nch = (line & 1) ? nlines / 2 : (nlines + 1) / 2;
  const int c = line >> 1;
  return c >= (int)(nch * part / nparts) && c < (int)(nch * (part + 1) / nparts);
}

__global__ void __launch_bounds__(kSortWarps * 32)
kset_sort_kernel(const int32_t* __restrict__ pvec, const int32_t* __restrict__ nprop, int npix, int K, int Kst,
                 int bshift, uint16_t* __restrict__ sorig, int32_t* __restrict__ svec, int H, int W, int part,
                 int nparts) {
  __shared__ __align__(16) int cnt_s[kSortWarps][kCntSize];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* cnt = cnt_s[warp];
  for (int pix = blockIdx.x * kSortWarps + warp; pix < npix; pix += gridDim.x * kSortWarps) {
    if (nparts > 1) {   // only pixels on a column or row chain this part runs (their records are the ones built)
      const int y = pix / W, x = pix - y * W;
      if (!owns_line(x, W, part, nparts) && !owns_line(y, H, part, nparts)) continue;
    }
    const int n = nprop[pix];
    const int32_t* v = pvec + (size_t)pix * K;
    uint16_t* o = sorig + (size_t)pix * Kst;
    int32_t* ov = svec + (size_t)pix * Kst;
    for (int i = lane; i < kCntSize / 4; i += 32) reinterpret_cast<int4*>(cnt)[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    for (int j = lane; j < n; j += 32) atomicAdd(&cnt[cidx(bucket_key(v[j], bshift))], 1);
    __syncwarp();
    // exclusive scan: lane owns counters [32*lane, 32*lane+32), stored at 33*lane + i (conflict free)
    int sum = 0;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) sum += cnt[lane * 33 + i];
    int pre = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, pre, off);
      if (lane >= off) pre += t;
    }
    pre -= sum;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const int c = cnt[lane * 33 + i];
      cnt[lane * 33 + i] = pre;
      pre += c;
    }
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
      const int32_t vj = v[j];
      const int pos = atomicAdd(&cnt[cidx(bucket_key(vj, bshift))], 1);
      o[pos] = (uint16_t)j;
      ov[pos] = vj;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// build: one CTA (kBuildThreads threads) per record
//
// Record layout (16-byte aligned, at most one chain-kernel slot).  Labels are stored in order of DECREASING list
// length (position t = thread t of the chain kernel), so that the lanes of a warp have (almost) equal trip counts:
//   [0,16)   uint32 n, number of entry groups, struct byte offset, entry byte offset
//   [16,..)  uint16 goff[n, padded to 8]: first entry group of position t
//   structs  n x {int32 vector; uint32 data cost (16) | original label (9) << 16 | entry groups (7) << 25}
//   entries  groups of four uint16 (8 bytes, one shared-memory load): (k << 3) | (L1 << 12) = previous-pixel label k
//            (original index; << 3 = byte offset of its key pair in the chain kernel) and L1(v_l, u_k) < tpsi; a list
//            is padded to whole groups with kNullEntry.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxList = 124;                  // 31 groups of four
constexpr uint32_t kNullEntry = 0x8FF8u;       // bit 15 = "no entry"; its label field is 511, whose key slot the 32-bit
                                               // chain kernel keeps infinite (it runs proposal sets of K <= 511 labels)
constexpr uint32_t kCostLimit16 = 1u << 16;    // data cost field: 16 bits
constexpr int kStagePerLabel = 16;             // staging capacity of the build kernel: candidates per label of Kpad
constexpr int kSlotPerLabel = 12;              // chain-kernel slot capacity: stored entries per label of Kpad

// previous pixel of `p` in the chain of orientation `orient` (0 = column chain, 1 = row chain) that visits it, or -1
// at the start of the chain (python bcd.py:265-277: even columns run down, even rows right to left, odd columns up,
// odd rows left to right)
__device__ __forceinline__ int prev_pixel(int y, int x, int orient, int H, int W) {
  if (orient == 0) {
    const int yq = (x & 1) ? y + 1 : y - 1;
    return (yq < 0 || yq >= H) ? -1 : yq * W + x;
  }
  const int xq = (y & 1) ? x - 1 : x + 1;
  return (xq < 0 || xq >= W) ? -1 : y * W + xq;
}

// candidate ranges of vector v in the previous pixel's sorted label array: up to three [t0, t1) (one per bucket row)
struct Ranges {
  int t0[3], t1[3];
};
__device__ __forceinline__ Ranges lookup_ranges(const uint32_t* rng, int32_t v, int bshift) {
  Ranges R;
  const int by = vec_dy(v) >> bshift, bx = vec_dx(v) >> bshift;
  const int kx0 = bkt_x(bx - 1), kx1 = bkt_x(bx), kx2 = bkt_x(bx + 1);
  int last_row = -1;
#pragma unroll
  for (int oy = 0; oy < 3; ++oy) {
    const int ky = bkt_y(by + oy - 1);
    R.t0[oy] = R.t1[oy] = 0;
    if (ky != last_row) {   // clamped rows can coincide: scan each bucket row once
      const uint32_t* row = rng + (ky << 6);
      const uint32_t r0 = row[kx0], r1 = row[kx1], r2 = row[kx2];
      const int a = (int)min(min(r0 & 0xFFFFu, r1 & 0xFFFFu), r2 & 0xFFFFu);
      const int b = (int)max(max(r0 >> 16, r1 >> 16), r2 >> 16);
      if (b > a) {
        R.t0[oy] = a;
        R.t1[oy] = b;
      }
    }
    last_row = ky;
  }
  return R;
}

// Shared memory of one build CTA (one record at a time):
// rng u32[kHashSize] | hist u32[128] | start u32[128] | gstart u32[128] | misc u32[16] | vq2 int2[Kpad] |
// ln, so, rk, inv, cq u16[Kpad] | stage u16[kStagePerLabel * Kpad]
__host__ __device__ inline size_t build_smem_bytes(int Kpad) {
  return (size_t)kHashSize * 4 + 128 * 4 * 3 + 64 + (size_t)Kpad * 8 + (size_t)Kpad * 2 * 5 +
         (size_t)kStagePerLabel * Kpad * 2;
}

constexpr int kBuildThreads = 128;   // 256 threads per record measured slower (DESIGN section 6)

template <typename CostT>
__global__ void __launch_bounds__(kBuildThreads)
kset_build_kernel(const int32_t* __restrict__ pvec, const CostT* __restrict__ cost, const int32_t* __restrict__ nprop,
                  const uint16_t* __restrict__ sorig, const int32_t* __restrict__ svec, int H, int W, int K, int Kst,
                  int Kpad, int tpsi, int bshift, int shift, double lamda, uint32_t slot_bytes,
                  unsigned char* __restrict__ arena, unsigned long long arena_bytes,
                  unsigned long long* __restrict__ cursor, unsigned long long* __restrict__ desc, int part,
                  int nparts) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int t = threadIdx.x, lane = t & 31;
  uint32_t* rng = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t* hist = rng + kHashSize;
  uint32_t* start = hist + 128;
  uint32_t* gstart = start + 128;        // first entry group of the labels with list length m
  uint32_t* misc = gstart + 128;         // [0] staged entries, [1] failure flag, [3] ok, [4..5] arena offset,
                                         // [6] struct offset, [7] entry offset
  int2* vq2 = reinterpret_cast<int2*>(misc + 16);   // previous pixel's labels: {dy, dx << 16 | label << 3}: one 8-byte load
  uint16_t* ln = reinterpret_cast<uint16_t*>(vq2 + Kpad);
  uint16_t* so = ln + Kpad;
  uint16_t* rk = so + Kpad;
  uint16_t* inv = rk + Kpad;
  uint16_t* cq = inv + Kpad;
  uint16_t* stage = cq + Kpad;
  const uint32_t stage_cap = (uint32_t)kStagePerLabel * Kpad;
  for (int i = t; i < kHashSize; i += kBuildThreads) rng[i] = kRngEmpty;
  if (t < 16) misc[t] = 0;
  __syncthreads();

  const int npix = H * W;
  const int ntask = 2 * npix;
  for (int task = blockIdx.x; task < ntask; task += gridDim.x) {
    const int orient = task >= npix ? 1 : 0;
    const int p = task - orient * npix;
    const int y = p / W, x = p - y * W;
    if (nparts > 1) {   // only the records of the chains this part runs (column x: chain x/2 of phase 0 or 2; row y alike)
      if (!owns_line(orient ? y : x, orient ? H : W, part, nparts)) {
        if (t == 0) desc[task] = 0ull;
        continue;
      }
    }
    const int q = prev_pixel(y, x, orient, H, W);
    const int n = nprop[p];
    const int nq = q >= 0 ? nprop[q] : 0;
    const int32_t* vp = pvec + (size_t)p * K;
    const CostT* cp = cost + (size_t)p * K;
    const uint16_t* sp = sorig + (size_t)p * Kst;
    const int32_t* svp = svec + (size_t)p * Kst;

    // 1. previous pixel's labels in bucket order
    if (q >= 0) {
      const uint16_t* sq = sorig + (size_t)q * Kst;
      const int32_t* svq = svec + (size_t)q * Kst;
      for (int s = t; s < nq; s += kBuildThreads) {
        const int32_t v = svq[s];
        vq2[s] = make_int2(vec_dy(v), (int)(((uint32_t)vec_dx(v) << 16) | ((uint32_t)sq[s] << 3)));
        inv[s] = (uint16_t)bucket_key(v, bshift);
      }
    }
    for (int i = t; i < 128; i += kBuildThreads) hist[i] = 0;
    __syncthreads();
    // 2. every bucket's [first, last+1) range (the bucket keys were left in `inv`, which is free until step 5)
    for (int s = t; s < nq; s += kBuildThreads) {
      const int key = inv[s];
      uint16_t* half = reinterpret_cast<uint16_t*>(rng + key);
      if (s == 0 || inv[s - 1] != key) half[0] = (uint16_t)s;
      if (s == nq - 1 || inv[s + 1] != key) half[1] = (uint16_t)(s + 1);
    }
    __syncthreads();

    // 3. evaluate: this pixel's labels in bucket order too (neighbouring lanes scan the same or adjacent ranges, so
    // their trip counts are similar); members are staged in shared memory, lists allocated by candidate count
    for (int s0 = 0; s0 < n; s0 += kBuildThreads) {
      const int s = s0 + t;
      const bool act = s < n;
      const int j = act ? (int)sp[s] : 0;
      int dy = 0, dx = 0;
      uint32_t c = 0, c0 = 0, c01 = 0;
      int o0 = 0, o1 = 0, o2 = 0;
      if (act) {
        const int32_t v = svp[s];
        dy = vec_dy(v);
        dx = vec_dx(v);
        const int32_t m = quant_cost<CostT>(cp[j], lamda, shift);
        if (m < 0 || (uint32_t)m >= kCostLimit16) misc[1] = 1;
        cq[j] = (uint16_t)m;
        if (q >= 0) {
          const Ranges R = lookup_ranges(rng, v, bshift);
          c0 = (uint32_t)(R.t1[0] - R.t0[0]);
          c01 = c0 + (uint32_t)(R.t1[1] - R.t0[1]);
          c = c01 + (uint32_t)(R.t1[2] - R.t0[2]);
          o0 = R.t0[0];
          o1 = R.t0[1] - (int)c0;
          o2 = R.t0[2] - (int)c01;
        }
      }
      uint32_t inc = c;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        uint32_t u = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += u;
      }
      const uint32_t warp_total = __shfl_sync(0xffffffffu, inc, 31);
      uint32_t wbase = 0;
      if (lane == 0) wbase = atomicAdd(&misc[0], warp_total);
      wbase = __shfl_sync(0xffffffffu, wbase, 0);
      if (wbase + warp_total > stage_cap) {   // warp-uniform
        if (lane == 0) misc[1] = 1;
      } else if (act) {
        const uint32_t sbase = wbase + inc - c;
        uint16_t* e = stage + sbase;
        uint32_t m = 0;
        for (uint32_t xx = 0; xx < c; ++xx) {   // the three ranges as one index space
          const int tt = (int)xx + (xx < c0 ? o0 : (xx < c01 ? o1 : o2));
          const int2 u = vq2[tt];
          const int l1 = (int)__sad(dy, u.x, __sad(dx, u.y >> 16, 0u));
          if (l1 < tpsi) e[m++] = (uint16_t)(((uint32_t)u.y & 0xFFFFu) | ((uint32_t)l1 << 12));
        }
        if (m > (uint32_t)kMaxList) {
          misc[1] = 1;
          m = kMaxList;
        }
        ln[j] = (uint16_t)m;
        so[j] = (uint16_t)sbase;
        rk[j] = (uint16_t)atomicAdd(&hist[m], 1u);
      }
    }
    __syncthreads();

    // 4. labels in order of decreasing list length (warp 0): start[m] = number of labels with a longer list,
    //    gstart[m] = number of entry groups those labels take (a list of m entries takes ceil(m / 4));  arena allocation
    if (t < 32) {
      bool ok = misc[1] == 0;
      const uint32_t h0 = hist[4 * lane], h1 = hist[4 * lane + 1], h2 = hist[4 * lane + 2], h3 = hist[4 * lane + 3];
      const uint32_t hs = h0 + h1 + h2 + h3;
      const uint32_t gl = (uint32_t)lane + 1u;                      // groups of a list of 4*lane+1 .. 4*lane+4 entries
      const uint32_t ws = h0 * (uint32_t)lane + (h1 + h2 + h3) * gl;  // groups of this lane's four bins (bin 4*lane: lane)
      uint32_t suf = hs, sufw = ws;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_down_sync(0xffffffffu, suf, o), uw = __shfl_down_sync(0xffffffffu, sufw, o);
        if (lane + o < 32) {
          suf += u;
          sufw += uw;
        }
      }
      const uint32_t total = __shfl_sync(0xffffffffu, sufw, 0);     // entry groups of the record
      const uint32_t s3 = suf - hs, s2 = s3 + h3, s1 = s2 + h2, s0_ = s1 + h1;   // start of bins 4*lane+3 .. 4*lane
      start[4 * lane] = s0_;
      start[4 * lane + 1] = s1;
      start[4 * lane + 2] = s2;
      start[4 * lane + 3] = s3;
      const uint32_t g3 = sufw - ws, g2 = g3 + h3 * gl, g1 = g2 + h2 * gl, g0 = g1 + h1 * gl;
      gstart[4 * lane] = g0;
      gstart[4 * lane + 1] = g1;
      gstart[4 * lane + 2] = g2;
      gstart[4 * lane + 3] = g3;
      const uint32_t so_b = (uint32_t)(kRecHeader + 2 * ((n + 7) & ~7));
      const uint32_t eo_b = so_b + 8u * (uint32_t)n;
      const unsigned long long bytes = ((unsigned long long)eo_b + 8ull * total + 15ull) & ~15ull;
      unsigned long long off = 0;
      ok = ok && bytes <= slot_bytes;
      if (ok) {
        if (lane == 0) off = atomicAdd(cursor, bytes);
        off = __shfl_sync(0xffffffffu, off, 0);
        ok = off + bytes <= arena_bytes;
      }
      if (lane == 0) {
        misc[3] = ok ? 1u : 0u;
        misc[4] = (uint32_t)off;
        misc[5] = (uint32_t)(off >> 32);
        misc[6] = so_b;
        misc[7] = eo_b;
        desc[task] = ok ? ((off >> 4) | ((bytes >> 4) << 40)) : 0ull;
        if (ok) {
          uint32_t* h = reinterpret_cast<uint32_t*>(arena + off);
          h[0] = (uint32_t)n;
          h[1] = total;
          h[2] = so_b;
          h[3] = eo_b;
        }
      }
    }
    __syncthreads();
    const bool ok = misc[3] != 0;
    if (ok) {
      // 5. position of every label
      for (int j = t; j < n; j += kBuildThreads) inv[start[ln[j]] + rk[j]] = (uint16_t)j;
      __syncthreads();
      // 6. write the record
      unsigned char* rec = arena + (((unsigned long long)misc[5] << 32) | misc[4]);
      uint16_t* go_g = reinterpret_cast<uint16_t*>(rec + kRecHeader);
      uint2* st = reinterpret_cast<uint2*>(rec + misc[6]);
      uint2* ents = reinterpret_cast<uint2*>(rec + misc[7]);
      for (int pos = t; pos < n; pos += kBuildThreads) {
        const int j = inv[pos];
        const int len = ln[j];
        const int ng = (len + 3) >> 2;
        const uint32_t g0 = gstart[len] + (uint32_t)rk[j] * (uint32_t)ng;
        const uint16_t* src = stage + so[j];
        st[pos] = make_uint2((uint32_t)vp[j], (uint32_t)cq[j] | ((uint32_t)j << 16) | ((uint32_t)ng << 25));
        go_g[pos] = (uint16_t)g0;
        for (int g = 0; g < ng; ++g) {
          const int r = 4 * g;
          const uint32_t e0 = src[r];
          const uint32_t e1 = r + 1 < len ? (uint32_t)src[r + 1] : kNullEntry;
          const uint32_t e2 = r + 2 < len ? (uint32_t)src[r + 2] : kNullEntry;
          const uint32_t e3 = r + 3 < len ? (uint32_t)src[r + 3] : kNullEntry;
          ents[g0 + g] = make_uint2(e0 | (e1 << 16), e2 | (e3 << 16));
        }
      }
    }
    // 7. empty the bucket table (4 KB: two 16-byte stores per thread) and the per-record state for the next record
    if (q >= 0)
      for (int i = t; i < kHashSize / 4; i += kBuildThreads)
        reinterpret_cast<uint4*>(rng)[i] = make_uint4(kRngEmpty, kRngEmpty, kRngEmpty, kRngEmpty);
    if (t < 2) misc[t] = 0;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// chains
// ------------------------------------------------------------------------------------------------
struct ChainArgs {
  const int32_t* pvec;
  const void* cost;
  const int32_t* nprop;
  int32_t* labels;
  uint16_t* bp;
  const unsigned long long* desc;
  const unsigned char* arena;
  int32_t* flags;     // per chain of the launch: the 32-bit kernel sets 1 when it leaves the chain to the fallback
  int H, W, K, Kpad, phase, chain0, tpsi, shift, slot_shift;   // chain = chain0 + blockIdx.x; 1 << slot_shift slots
  uint32_t slot_bytes;
  int force_generic;  // (tests) leave every chain to the fallback, the integer variant of the float64 kernel
  double lamda;
};

constexpr int kMaxWarps = 16;   // T <= 512

// a record slot of the chain kernels holds header, group offsets, n structs and kSlotPerLabel entries per label of
// Kpad; larger records are not stored (their steps are evaluated densely)
__host__ __device__ inline uint32_t kset_slot_bytes(int Kpad) {
  return (uint32_t)((kRecHeader + 2 * (size_t)Kpad + 8 * (size_t)Kpad + 2 * (size_t)kSlotPerLabel * Kpad + 127) & ~(size_t)127);
}
// dynamic shared memory of the float64 kernel: side vectors int32[nside * len] | vprev int32[Kpad] | path uint16[len] |
// the record slots, 128-aligned.  nside = 1: the reference's side terms read the chain's own old vectors (oldvec);
// nside = 2 (FLOWB200_BCD_MRF): the labels' vectors of the two across-chain neighbours of every step
__host__ __device__ inline size_t chain_fixed_smem(int Kpad, int len, int nside = 1) {
  return (4 * (size_t)nside * len + 4 * (size_t)Kpad + 2 * (size_t)len + 127) & ~(size_t)127;
}
// ... of the 32-bit kernel, behind the (run-time) pad that aligns it to 4 KB: dp 4 KB | control 384 B |
// side vectors int32[nside * len] | path uint16[len] | the record slots, 128-aligned
__host__ __device__ inline size_t chain32_fixed_smem(int len, int nside = 1) {
  return (4096 + 384 + 4 * (size_t)nside * len + 2 * (size_t)len + 127) & ~(size_t)127;
}

// FLOWB200_BCD_MRF: the side neighbours of a chain step lie ACROSS the chain axis -- (y, x + 1) and (y, x - 1) of a
// column chain, (y + 1, x) and (y - 1, x) of a row chain, in that order.  They belong to lines of the other parity,
// which no chain of the phase writes, so their labels are read once when the chain starts.  Whether they exist
// depends on the chain's line only.
struct AcrossChain {
  bool has_p, has_m;
  int off;   // pixel index offset of the + neighbour (the - neighbour is at -off)
};
__device__ __forceinline__ AcrossChain across_chain(const ChainGeom& g, int H, int W) {
  if (g.ystep != 0) return {g.sx + 1 < W, g.sx > 0, 1};
  return {g.sy + 1 < H, g.sy > 0, W};
}
// side[i] / side[len + i]: vector of the label of the + / - neighbour of step i (0 where it does not exist)
template <int T>
__device__ __forceinline__ void load_across(const ChainArgs& a, const ChainGeom& g, int32_t* side) {
  const AcrossChain ac = across_chain(g, a.H, a.W);
  for (int i = threadIdx.x; i < g.len; i += T) {
    const int p = (g.sy + i * g.ystep) * a.W + (g.sx + i * g.xstep);
    const int pp = p + ac.off, pm = p - ac.off;
    side[i] = ac.has_p ? a.pvec[(size_t)pp * a.K + a.labels[pp]] : 0;
    side[g.len + i] = ac.has_m ? a.pvec[(size_t)pm * a.K + a.labels[pm]] : 0;
  }
}

// backtrack (:238-253) through the back-pointers of the chain of this block, staged through shared memory (the record
// slots, free by now) a segment of rows at a time; the labels are written once the whole path is known
template <int T>
__device__ __forceinline__ void backtrack(const ChainArgs& a, const ChainGeom& g, int lab, uint16_t* path,
                                          unsigned char* slots, int S) {
  const int t = threadIdx.x, Kpad = a.Kpad;
  const int rows_cap = max(1, (int)(((size_t)S * a.slot_bytes) / ((size_t)Kpad * 2)));
  uint16_t* seg = reinterpret_cast<uint16_t*>(slots);
  const int vec_per_row = Kpad / 8;   // uint4 = 8 back-pointers
  const uint16_t* bp_chain = a.bp + (size_t)blockIdx.x * g.len * Kpad;
  for (int hi = g.len - 1; hi >= 1; hi -= rows_cap) {
    const int lo = max(1, hi - rows_cap + 1);
    const int nrow = hi - lo + 1;
    const uint4* src = reinterpret_cast<const uint4*>(bp_chain + (size_t)lo * Kpad);
    uint4* dst = reinterpret_cast<uint4*>(seg);
    for (int x = t; x < nrow * vec_per_row; x += T) dst[x] = src[x];
    __syncthreads();
    if (t == 0) {
      for (int i = hi; i >= lo; --i) {
        path[i] = (uint16_t)lab;
        lab = seg[(size_t)(i - lo) * Kpad + lab];
      }
    }
    __syncthreads();   // (uniform: lab is only meaningful in thread 0)
  }
  if (t == 0) path[0] = (uint16_t)lab;
  __syncthreads();
  for (int i = t; i < g.len; i += T) a.labels[(g.sy + i * g.ystep) * a.W + (g.sx + i * g.xstep)] = (int)path[i];
}

// The float64 programme on the same records (FLOWB200_BCD_FP64_*: arbitrary data costs, the reference's own arithmetic
// and operation order, python bcd.py:118-120, :152-176): dp is a double per label, candidates are compared as
// (value, label) pairs -- np.argmin takes the lowest label among equal values --, and the data cost comes from the
// cost array (the record's 16-bit cost field is unused).  One thread per label position, every chain of the launch.
// QUANT: the int32 modes' programme on the chains the 32-bit kernel flagged (its other blocks return at once).  Every
// term is then an integer in units of 2^-shift -- the quantised data cost (what a record's cost field holds), L1 << shift,
// min(tpsi, L1) << shift, tpsi << shift -- and make_plan keeps dp below 2^32, so the double arithmetic is exact in any
// order and the (value, label) compares order as the 32-bit kernel's lexicographic ones do.
__device__ __forceinline__ void warp_argmin_f64(double& val, int& idx) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, val, off);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, off);
    if (ov < val || (ov == val && oi < idx)) {
      val = ov;
      idx = oi;
    }
  }
}

// MRF (FLOWB200_BCD_MRF): side terms across the chain (AcrossChain) and, at every step, the smaller of the K-set
// candidate and the truncation candidate (DESIGN 4.4).
template <typename CostT, int T, bool QUANT, bool MRF>
__device__ __forceinline__ void chainf64_body(const ChainArgs& a) {
  constexpr int NW = T / 32;
  constexpr int kNone = 0x7fffffff;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(16) double rep_s[2 * 512];   // [2 * k + b]: dp of label k at a step of parity b
  __shared__ double red_val[2][kMaxWarps];          // per warp: min of (tpsi + dp, label) of a step, lowest label on ties
  __shared__ int red_idx[2][kMaxWarps];             // (the sum is what the reference minimises, :152-157: it can tie where dp does not)
  __shared__ uint32_t present_s[4];
  __shared__ __align__(8) uint64_t mbar[4];
  if constexpr (QUANT) {
    if (a.flags[blockIdx.x] == 0) return;   // (uniform) done by the 32-bit kernel
  }
  // an L1 distance or tpsi in the units of dp
  auto units = [&](auto x) {
    if constexpr (QUANT) return x << a.shift;
    else return x;
  };

  const ChainGeom g = chain_geom(a.phase, a.chain0 + (int)blockIdx.x, a.H, a.W);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int K = a.K, Kpad = a.Kpad, tpsi = a.tpsi;
  const int S = 1 << a.slot_shift, smask = S - 1;
  const unsigned long long* dsc = a.desc + (size_t)(a.phase & 1) * a.H * a.W;
  const CostT* cost = static_cast<const CostT*>(a.cost);
  const double lamda = a.lamda;

  constexpr int kSide = MRF ? 2 : 1;
  int32_t* oldvec = reinterpret_cast<int32_t*>(smem_raw);   // MRF: the across-chain vectors, 2 x len
  int32_t* vprev = oldvec + kSide * g.len;
  uint16_t* path = reinterpret_cast<uint16_t*>(vprev + Kpad);
  unsigned char* slots = smem_raw + chain_fixed_smem(Kpad, g.len, kSide);
  auto pixel = [&](int i) { return (g.sy + i * g.ystep) * a.W + (g.sx + i * g.xstep); };

  if constexpr (MRF) {
    load_across<T>(a, g, oldvec);
  } else {
    for (int i = t; i < g.len; i += T) {
      const int p = pixel(i);
      oldvec[i] = a.pvec[(size_t)p * K + a.labels[p]];
    }
  }
  if (t == 0) {
    for (int s = 0; s < S; ++s) ptx::mbar_init(&mbar[s], 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();

  unsigned long long d_next = 0;
  auto issue = [&](int i, unsigned long long d) {
    const int slot = i & smask;
    const uint32_t bytes = (uint32_t)(d >> 40) << 4;
    present_s[slot] = bytes;
    if (bytes) {
      ptx::mbar_arrive_expect_tx(&mbar[slot], bytes);
      ptx::bulk_load(slots + (size_t)slot * a.slot_bytes, a.arena + ((d & ((1ull << 40) - 1)) << 4), bytes, &mbar[slot]);
    } else {
      ptx::mbar_arrive(&mbar[slot]);
    }
  };
  if (t == 0) {
    for (int i = 0; i < S && i < g.len; ++i) issue(i, dsc[pixel(i)]);
    if (S < g.len) d_next = dsc[pixel(S)];
  }

  // block argmin of what the warps left in red_val / red_idx[step & 1]
  auto block_argmin = [&](int step, double& v, int& k) {
    v = red_val[step & 1][0];
    k = red_idx[step & 1][0];
#pragma unroll
    for (int w = 1; w < NW; ++w) {
      const double ov = red_val[step & 1][w];
      const int oi = red_idx[step & 1][w];
      if (ov < v || (ov == v && oi < k)) {
        v = ov;
        k = oi;
      }
    }
  };
  const int sgn = g.ystep + g.xstep;   // +1: the image coordinate grows with the step index
  uint16_t* bp_row = a.bp + (size_t)blockIdx.x * g.len * Kpad;
  double last_dp = CUDART_INF;
  int last_label = kNone;

  for (int i = 0; i < g.len; ++i, bp_row += Kpad) {
    const int slot = i & smask;
    ptx::mbar_wait(&mbar[slot], (uint32_t)(i >> a.slot_shift) & 1u);
    const uint32_t present = present_s[slot];
    const int prv = (i & 1) ^ 1;
    double dpv = CUDART_INF;
    int mine = kNone;
    // side terms (sidepsi :84-88): the neighbour on the +1 side of the chain axis first, as the reference adds them
    bool has_p, has_m;
    int32_t ov_p, ov_m;
    if constexpr (MRF) {
      const AcrossChain ac = across_chain(g, a.H, a.W);
      has_p = ac.has_p;
      has_m = ac.has_m;
      ov_p = oldvec[i];
      ov_m = oldvec[g.len + i];
    } else {
      const int ip = i + sgn, im = i - sgn;
      has_p = ip >= 0 && ip < g.len;
      has_m = im >= 0 && im < g.len;
      ov_p = has_p ? oldvec[ip] : 0;
      ov_m = has_m ? oldvec[im] : 0;
    }
    // dp of label `orig` (vector dy, dx) from the minimum (best, arg) over the previous step's candidates
    auto finish = [&](int dy, int dx, int orig, double best, int arg, const int p) {
      const int psi_p = has_p ? units(min(tpsi, l1_vec(dy, dx, ov_p))) : 0;
      const int psi_m = has_m ? units(min(tpsi, l1_vec(dy, dx, ov_m))) : 0;
      double lc;
      if constexpr (QUANT) lc = (double)quant_cost<CostT>(cost[(size_t)p * K + orig], lamda, a.shift);
      else lc = __dmul_rn(lamda, (double)cost[(size_t)p * K + orig]);
      if (i == 0) {   // (psi+ + psi-) + lamda*lcost   (:118-120)
        dpv = __dadd_rn((double)(psi_p + psi_m), lc);
      } else {        // (lamda*lcost + psi+) + psi-, then m + that   (:161-162, :176)
        if constexpr (MRF) {   // the truncation candidate at every step: the smaller (value, label) of the two
          double tv;
          int tk;
          block_argmin(i - 1, tv, tk);
          if (tv < best || (tv == best && tk < arg)) {
            best = tv;
            arg = tk;
          }
        } else if (arg == kNone) {
          block_argmin(i - 1, best, arg);   // quirk Q1: min_k (tpsi + dp_prev[k]), lowest k (:152-157), only for an
                                            // empty K-set
        }
        dpv = __dadd_rn(best, __dadd_rn(__dadd_rn(lc, (double)psi_p), (double)psi_m));
        bp_row[orig] = (uint16_t)arg;
      }
      mine = orig;
      rep_s[2 * orig + (i & 1)] = dpv;
    };
    if (present) {
      const unsigned char* rec = slots + (size_t)slot * a.slot_bytes;
      const uint4 hdr = *reinterpret_cast<const uint4*>(rec);
      if (t < (int)hdr.x) {
        const uint2 st = *reinterpret_cast<const uint2*>(rec + hdr.z + 8 * t);
        double best = CUDART_INF;
        int arg = kNone;
        if (i > 0) {
          const int ng = (int)(st.y >> 25);
          const uint32_t g0 = *reinterpret_cast<const uint16_t*>(rec + kRecHeader + 2 * t);
          const uint2* eg = reinterpret_cast<const uint2*>(rec + hdr.w) + g0;
          for (int gi = 0; gi < ng; ++gi) {
            const uint2 w = eg[gi];
            const uint32_t e[4] = {w.x & 0xFFFFu, w.x >> 16, w.y & 0xFFFFu, w.y >> 16};
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (!(e[j] & 0x8000u)) {   // (not a padding entry)
                const int k = (int)((e[j] >> 3) & 511u);
                const double cand = __dadd_rn(rep_s[2 * k + prv], (double)units((e[j] >> 12) & 7u));
                if (cand < best || (cand == best && k < arg)) {   // np.argmin: lowest k wins ties
                  best = cand;
                  arg = k;
                }
              }
          }
        }
        finish(vec_dy((int32_t)st.x), vec_dx((int32_t)st.x), (int)((st.y >> 16) & 511u), best, arg, pixel(i));
      }
    } else {
      // dense step: the record was not stored; evaluate the K-set from the proposal arrays
      const int p = pixel(i);
      const int n = a.nprop[p];
      int nq = 0;
      if (i > 0) {
        const int q = pixel(i - 1);
        nq = a.nprop[q];
        for (int k = t; k < nq; k += T) vprev[k] = a.pvec[(size_t)q * K + k];
      }
      __syncthreads();
      if (t < n) {
        const int32_t v = a.pvec[(size_t)p * K + t];
        const int dy = vec_dy(v), dx = vec_dx(v);
        double best = CUDART_INF;
        int arg = kNone;
        for (int k = 0; k < nq; ++k) {
          const int l1 = l1_vec(dy, dx, vprev[k]);
          if (l1 < tpsi) {
            const double cand = __dadd_rn(rep_s[2 * k + prv], (double)units(l1));
            if (cand < best) {   // (k ascending: the first minimum is the lowest k)
              best = cand;
              arg = k;
            }
          }
        }
        finish(dy, dx, t, best, arg, p);
      }
    }
    last_dp = dpv;
    last_label = mine;
    {
      double wv = __dadd_rn((double)units(tpsi), dpv);
      int wi = mine;
      warp_argmin_f64(wv, wi);
      if (lane == 0) {
        red_val[i & 1][warp] = wv;
        red_idx[i & 1][warp] = wi;
      }
    }
    __syncthreads();
    if (t == 0 && i + S < g.len) {
      issue(i + S, d_next);
      if (i + S + 1 < g.len) d_next = dsc[pixel(i + S + 1)];
    }
  }

  // final label: lowest-index argmin of dp_last (:231-237)
  warp_argmin_f64(last_dp, last_label);
  const int fin = g.len & 1;   // the buffer the last step's reduction did not use
  if (lane == 0) {
    red_val[fin][warp] = last_dp;
    red_idx[fin][warp] = last_label;
  }
  __syncthreads();
  double bv;
  int lab;
  block_argmin(fin, bv, lab);
  backtrack<T>(a, g, lab, path, slots, S);
}

// ------------------------------------------------------------------------------------------------
// The 32-bit chain kernel proper: one thread per label position, as few instructions per step as possible.  Measured
// (ncu, profiles/): a chain step is bound by the NUMBER of warp instructions it issues -- an SM holds ~3 chains whose
// warps each run one dependent instruction stream at ~7 cycles per instruction -- so what counts is: dp is a plain
// uint32 in units of 2^-shift (make_plan bounds a whole chain below 2^32: no rebasing); "smallest dp, lowest label
// on ties" (np.argmin, python bcd.py:155/:175/:234) is the lexicographic minimum of (dp, label field of the entry) --
// two compares on 32-bit registers; warps without labels go straight to the barrier; the dp array is 4 KB aligned, so
// that the shared-memory address of an entry's dp is one logic operation on the packed entry word (mask | base |
// buffer); the cost shift is a template parameter (12 is what the scripts and the benchmark use; 0 = run time); the
// last warp, which has no labels or the shortest lists, streams the records.  Chains with a record that was not stored
// are left to the integer variant of kset_chainf64_kernel (flags[chain] = 1), which evaluates such steps densely.
// (Keys of (dp relative to the running minimum) << 9 | label, one unsigned minimum per entry, were built first and are
// NOT exact: because of quirk Q1 -- no truncation candidate for a non-empty K-set, :170-176 -- whole families of labels
// fall behind the minimum by ~16 units per step, overflow any 22-bit field within ~64 steps, and now and then catch up
// again: one column chain in 512 went wrong at 1024x436.)
// ------------------------------------------------------------------------------------------------
constexpr int kKeyBytes = 4096;   // dp of labels 0..510 in two buffers; the slot of label 511 stays infinite (null entries)
constexpr int kCtlBytes = 384;    // warp minima [2][16] x 2, four mbarriers

template <typename CostT, int T, int SHIFT, bool MRF>
__device__ __forceinline__ void chain32_body(const ChainArgs& a) {
  constexpr int NW = T / 32;
  constexpr uint32_t kInf = 0xFFFFFFFFu;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ int absent_s;

  const ChainGeom g = chain_geom(a.phase, a.chain0 + (int)blockIdx.x, a.H, a.W);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, wfirst = t & ~31;
  const int K = a.K, Kpad = a.Kpad, tpsi = a.tpsi;
  const int shift = SHIFT ? SHIFT : a.shift;
  const int S = 1 << a.slot_shift, smask = S - 1;
  const unsigned long long* dsc = a.desc + (size_t)(a.phase & 1) * a.H * a.W;
  const int len = g.len;

  // dynamic shared memory: [pad] dp (4 KB aligned) | warp minima, mbarriers (kCtlBytes) | oldvec | path | record slots.
  // Everything hangs off ONE base pointer held in a register (static shared arrays cost an address computation from
  // the cluster CTA id at every use on sm_100).
  const uint32_t dyn0 = ptx::smem_u32(smem_raw);
  const uint32_t pad = (0u - dyn0) & (uint32_t)(kKeyBytes - 1);
  uint32_t* rep_s = reinterpret_cast<uint32_t*>(smem_raw + pad);   // [2 * k + parity]
  const uint32_t rep_u32 = dyn0 + pad;
  uint32_t (*wred_v)[kMaxWarps] = reinterpret_cast<uint32_t (*)[kMaxWarps]>(smem_raw + pad + kKeyBytes);         // [2][16]: per warp,
  uint32_t (*wred_l)[kMaxWarps] = reinterpret_cast<uint32_t (*)[kMaxWarps]>(smem_raw + pad + kKeyBytes + 128);   // min dp of a step and the lowest label that has it
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + pad + kKeyBytes + 256);                                // [4]
  constexpr int kSide = MRF ? 2 : 1;
  int32_t* oldvec = reinterpret_cast<int32_t*>(smem_raw + pad + kKeyBytes + kCtlBytes);   // MRF: across-chain, 2 x len
  uint16_t* path = reinterpret_cast<uint16_t*>(oldvec + kSide * len);
  unsigned char* slots = smem_raw + pad + chain32_fixed_smem(len, kSide);
  auto pixel = [&](int i) { return (g.sy + i * g.ystep) * a.W + (g.sx + i * g.xstep); };

  if (t == 0) absent_s = 0;
  __syncthreads();
  {
    bool absent = false;
    if constexpr (MRF) load_across<T>(a, g, oldvec);
    for (int i = t; i < len; i += T) {
      const int p = pixel(i);
      if constexpr (!MRF) oldvec[i] = a.pvec[(size_t)p * K + a.labels[p]];
      absent |= (dsc[p] >> 40) == 0;
    }
    if (absent || K > 511 || a.force_generic) absent_s = 1;   // (label 511's slot is the padding entries' infinity)
  }
  if (t < 2) rep_s[2 * 511 + t] = kInf;
  if (t == 0) {
    for (int s = 0; s < S; ++s) ptx::mbar_init(&mbar[s], 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();
  if (absent_s) {   // (uniform)
    if (t == 0) a.flags[blockIdx.x] = 1;
    return;
  }
  if (t == 0) a.flags[blockIdx.x] = 0;

  const bool producer = t == T - 32;
  unsigned long long d_next = 0;
  auto issue = [&](int i, unsigned long long d) {
    const int slot = i & smask;
    const uint32_t bytes = (uint32_t)(d >> 40) << 4;
    ptx::mbar_arrive_expect_tx(&mbar[slot], bytes);
    ptx::bulk_load(slots + (size_t)slot * a.slot_bytes, a.arena + ((d & ((1ull << 40) - 1)) << 4), bytes, &mbar[slot]);
  };
  if (producer) {
    for (int i = 0; i < S && i < len; ++i) issue(i, dsc[pixel(i)]);
    if (S < len) d_next = dsc[pixel(S)];
  }

  const uint32_t tpsi_dp = (uint32_t)tpsi << shift;
  uint16_t* bp_row = a.bp + (size_t)blockIdx.x * len * Kpad;   // row of step i (advanced every step)
  const uint32_t mbar_u32 = ptx::smem_u32(mbar);
  // (value, label field) pairs: lexicographic minimum with two compares on the 32-bit halves
  auto lex_min = [](uint32_t& bv, uint32_t& bk, uint32_t v, uint32_t k) {
    const unsigned long long x = ((unsigned long long)v << 32) | k, y = ((unsigned long long)bv << 32) | bk;
    const bool lt = x < y;
    bv = lt ? v : bv;
    bk = lt ? k : bk;
  };

  for (int i = 0; i < len; ++i, bp_row += Kpad) {
    const int slot = i & smask;
    ptx::mbar_wait_u32(mbar_u32 + 8u * (uint32_t)slot, (uint32_t)(i >> a.slot_shift) & 1u);
    const unsigned char* rec = slots + (size_t)slot * a.slot_bytes;
    const uint4 hdr = *reinterpret_cast<const uint4*>(rec);   // n, entry groups, struct offset, entry offset
    const int n = (int)hdr.x;
    uint32_t dp = kInf, mine = kInf;
    if (t < n) {
      const uint2 st = *reinterpret_cast<const uint2*>(rec + hdr.z + 8 * t);
      const uint32_t orig = (st.y >> 16) & 511u;
      // unary term: data cost + the two side terms (sidepsi :84-88: the chain's own neighbours with their labels from
      // before this call), in units of 2^-shift
      const int dy = vec_dy((int32_t)st.x), dx = vec_dx((int32_t)st.x);
      uint32_t psi = 0;
      if constexpr (MRF) {
        const AcrossChain ac = across_chain(g, a.H, a.W);
        if (ac.has_p) psi += (uint32_t)min(tpsi, l1_vec(dy, dx, oldvec[i]));
        if (ac.has_m) psi += (uint32_t)min(tpsi, l1_vec(dy, dx, oldvec[len + i]));
      } else {
        if (i + 1 < len) psi += (uint32_t)min(tpsi, l1_vec(dy, dx, oldvec[i + 1]));
        if (i > 0) psi += (uint32_t)min(tpsi, l1_vec(dy, dx, oldvec[i - 1]));
      }
      dp = (st.y & 0xFFFFu) + (psi << shift);   // dp_0 = unary (:118-120)
      if (i > 0) {
        const uint32_t ng = st.y >> 25;
        const uint32_t g0 = *reinterpret_cast<const uint16_t*>(rec + kRecHeader + 2 * t);
        const uint2* eg = reinterpret_cast<const uint2*>(rec + hdr.w) + g0;
        const uint32_t base = rep_u32 | ((uint32_t)((i & 1) ^ 1) << 2);   // previous step's buffer
        uint32_t v0 = kInf, k0 = kInf, v1 = kInf, k1 = kInf;   // two independent running minima
#pragma unroll 1
        for (uint32_t gi = 0; gi < ng; ++gi) {
          const uint2 w = eg[gi];
          // an entry: bits 3..11 = previous-pixel label << 3 (= offset of its dp pair), bits 12..14 = L1 (with the usual
          // shift of 12 the pairwise cost L1 << 12 is one mask of the entry)
          const uint32_t hx = w.x >> 16, hy = w.y >> 16;
          const uint32_t ka = w.x & 0xFF8u, kb = hx & 0xFF8u, kc = w.y & 0xFF8u, kd = hy & 0xFF8u;
          uint32_t ca = ptx::lds_u32(ka | base), cb = ptx::lds_u32(kb | base);
          uint32_t cc = ptx::lds_u32(kc | base), cd = ptx::lds_u32(kd | base);
          if constexpr (SHIFT == 12) {
            ca += w.x & 0x7000u;
            cb += hx & 0x7000u;
            cc += w.y & 0x7000u;
            cd += hy & 0x7000u;
          } else {
            ca += ((w.x >> 12) & 7u) << shift;
            cb += ((hx >> 12) & 7u) << shift;
            cc += ((w.y >> 12) & 7u) << shift;
            cd += ((hy >> 12) & 7u) << shift;
          }
          lex_min(v0, k0, ca, ka);
          lex_min(v1, k1, cb, kb);
          lex_min(v0, k0, cc, kc);
          lex_min(v1, k1, cd, kd);
        }
        lex_min(v0, k0, v1, k1);
        if constexpr (MRF) {   // the truncation candidate at every step, label field << 3 like the entries'
          uint32_t tv = kInf, tk = kInf;
#pragma unroll
          for (int k = 0; k < NW; ++k) lex_min(tv, tk, wred_v[(i - 1) & 1][k], wred_l[(i - 1) & 1][k]);
          lex_min(v0, k0, tv + tpsi_dp, tk << 3);
        }
        uint32_t arg = k0 >> 3;
        if (!MRF && ng == 0) {   // quirk Q1: the truncation candidate min_k (tpsi + dp_prev[k]), lowest k (:152-157), only for an
                         // empty K-set (last warps: labels are stored by decreasing list length)
          v0 = kInf;
          arg = kInf;
#pragma unroll
          for (int k = 0; k < NW; ++k) lex_min(v0, arg, wred_v[(i - 1) & 1][k], wred_l[(i - 1) & 1][k]);
          v0 += tpsi_dp;
        }
        dp += v0;
        bp_row[orig] = (uint16_t)arg;
      }
      mine = orig;
      rep_s[2 * orig + (i & 1)] = dp;
    }
    if (wfirst < n) {   // (warp uniform) minimum dp of the warp's labels and the lowest label that has it
      const uint32_t m = __reduce_min_sync(0xffffffffu, dp);
      mine = __reduce_min_sync(0xffffffffu, dp == m ? mine : kInf);
      dp = m;
    }
    if (lane == 0) {
      wred_v[i & 1][warp] = dp;
      wred_l[i & 1][warp] = mine;
    }
    __syncthreads();
    if (producer && i + S < len) {
      issue(i + S, d_next);
      if (i + S + 1 < len) d_next = dsc[pixel(i + S + 1)];
    }
  }

  // final label: lowest-index argmin of dp_last (:231-237)
  uint32_t bv = kInf, lab = kInf;
#pragma unroll
  for (int k = 0; k < NW; ++k) lex_min(bv, lab, wred_v[(len - 1) & 1][k], wred_l[(len - 1) & 1][k]);
  backtrack<T>(a, g, (int)lab, path, slots, S);
}

template <typename CostT, int T, int MINB, bool QUANT>
__global__ void __launch_bounds__(T, MINB) kset_chainf64_kernel(const ChainArgs a) {
  chainf64_body<CostT, T, QUANT, false>(a);
}

template <typename CostT, int T, int MINB, int SHIFT>
__global__ void __launch_bounds__(T, MINB) kset_chain32_kernel(const ChainArgs a) {
  chain32_body<CostT, T, SHIFT, false>(a);
}

// the FLOWB200_BCD_MRF programme: kernels of their own, so that the reference programme's stay as they are
template <typename CostT, int T, int MINB, bool QUANT>
__global__ void __launch_bounds__(T, MINB) kset_chainf64_mrf_kernel(const ChainArgs a) {
  chainf64_body<CostT, T, QUANT, true>(a);
}

template <typename CostT, int T, int MINB, int SHIFT>
__global__ void __launch_bounds__(T, MINB) kset_chain32_mrf_kernel(const ChainArgs a) {
  chain32_body<CostT, T, SHIFT, true>(a);
}

// the kernels a mode runs.  Only variants a mode can run are compiled: int32 costs come only with the int32 modes,
// double costs only with the float64 modes (no 32-bit kernel)
template <typename CostT, int T, int MINB, bool MRF>
auto chain32_kernel(int shift) {
  if constexpr (std::is_same<CostT, double>::value) return (void (*)(const ChainArgs)) nullptr;
  else if constexpr (MRF) return shift == 12 ? kset_chain32_mrf_kernel<CostT, T, MINB, 12> : kset_chain32_mrf_kernel<CostT, T, MINB, 0>;
  else return shift == 12 ? kset_chain32_kernel<CostT, T, MINB, 12> : kset_chain32_kernel<CostT, T, MINB, 0>;
}
// the float64 kernel runs the float64 programme, or (QUANT) the integer one: int32 costs, and float costs in the int32
// modes (shift >= 0)
template <typename CostT, int T, bool MRF, bool QUANT = !std::is_same<CostT, double>::value>
auto chainf64_kernel(int shift) {
  if constexpr (std::is_same<CostT, float>::value && QUANT)
    if (shift < 0) return chainf64_kernel<CostT, T, MRF, false>(shift);
  if constexpr (MRF) return kset_chainf64_mrf_kernel<CostT, T, 1, QUANT>;
  else return kset_chainf64_kernel<CostT, T, 1, QUANT>;
}

struct KsetLayout {
  size_t bp, sorig, svec, desc, cursor, flags, arena, arena_bytes, total;
  int Kst, Kpad;
};

KsetLayout kset_layout(int H, int W, int K, size_t workspace_bytes) {
  KsetLayout L{};
  L.Kpad = (K + 31) / 32 * 32;
  L.Kst = (K + 7) / 8 * 8;
  const size_t n = (size_t)H * W;
  const size_t col = (size_t)((W + 1) / 2) * H, row = (size_t)((H + 1) / 2) * W;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += align_up(bytes);
    return o;
  };
  L.bp = take((col > row ? col : row) * L.Kpad * sizeof(uint16_t));
  L.sorig = take(n * L.Kst * sizeof(uint16_t));
  L.svec = take(n * L.Kst * sizeof(int32_t));
  L.desc = take(2 * n * sizeof(unsigned long long));
  L.cursor = take(256);
  L.flags = take((size_t)(((W > H ? W : H) + 1) / 2) * sizeof(int32_t));
  L.arena = off;
  if (workspace_bytes == 0) {
    // default budget: header + 10 B per label + ~9 entries per label (whole groups of four), per record
    L.arena_bytes = 2 * n * (size_t)(kRecHeader + 16 + 10 * K + 18 * K);
  } else {
    L.arena_bytes = workspace_bytes > off ? (workspace_bytes - off) & ~(size_t)15 : 0;
  }
  L.total = off + align_up(L.arena_bytes);
  return L;
}

struct KsetPlan {
  KsetLayout L;
  void (*kern32)(const ChainArgs) = nullptr;   // int32 modes: every chain, 32-bit dp; nullptr in the float64 modes
  void (*kern32_lo)(const ChainArgs) = nullptr;  // the same compiled for one chain per SM fewer (more registers): used
                                                 // for the orientation whose shared memory does not admit more anyway
  void (*kernf64)(const ChainArgs) = nullptr;  // float64 modes: every chain; int32 modes: the chains kern32 flagged
  int T = 0, bshift = 0, slot_shift = 2, minb = 1;
  bool records = false;   // false: no record is built, every step is evaluated densely
  uint32_t slot_bytes = 0;
  size_t smem32[2] = {0, 0}, smem64 = 0;   // smem32: by chain orientation (column chains are H long, row chains W)
};

template <typename CostT>
struct BcdProblem {   // the problem a BCD call solves, as the entry points receive it (cost typed for the mode)
  const int32_t* pvec;
  const CostT* cost;
  const int32_t* nprop;
  int H, W, K;
  double lamda;
  int tpsi, shift;   // shift -1: the float64 programme
  bool mrf;          // FLOWB200_BCD_MRF
};

// the chain widths: T threads, one per label position, and the chains per SM aimed at (registers and shared memory)
constexpr int kWidths[][2] = {{64, 8}, {128, 6}, {192, 5}, {256, 4}, {320, 4}, {384, 3}, {512, 2}};

// the kernels of the first width that holds K; returns the chains per SM aimed at, 0 if no width holds K
template <bool MRF, size_t I = 0, typename CostT>
int pick_kernels(const BcdProblem<CostT>& pb, KsetPlan* P) {
  constexpr int T = kWidths[I][0], MB = kWidths[I][1];
  const int K = pb.K, shift = pb.shift;
  if constexpr (I + 1 < sizeof(kWidths) / sizeof(kWidths[0]))
    if (K > T) return pick_kernels<MRF, I + 1>(pb, P);
  if (K > T) return 0;
  constexpr int mb = MB > 4 ? 4 : MB;
  constexpr int mb_lo = MRF ? mb : mb - (MB >= 4 ? 1 : 0);   // MRF: no variant for fewer chains per SM
  if (shift >= 0) {
    P->kern32 = chain32_kernel<CostT, T, mb, MRF>(shift);
    P->kern32_lo = chain32_kernel<CostT, T, mb_lo, MRF>(shift);
  }
  P->minb = mb;
  P->kernf64 = chainf64_kernel<CostT, T, MRF>(shift);
  P->T = T;
  return MB;
}

// shift < 0 selects the float64 programme (kset_chainf64_kernel): the records then carry no data costs, and no 32-bit
// chain kernel is compiled (double costs) or set up.  Dropping the 32-bit kernel's shared-memory check there changes
// nothing: the float64 kernel's check is stricter, its left side is 4*Kpad + 128 bytes larger at every chain length
// mrf: the FLOWB200_BCD_MRF kernels, whose side vectors take 2 x len int32 of shared memory instead of len (the dp
// bound holds as it is: a step adds at most the smaller of the two candidates, so at most tpsi over the minimum)
template <typename CostT>
static int make_plan(const BcdProblem<CostT>& pb, size_t workspace_bytes, KsetPlan* P) {
  const int H = pb.H, W = pb.W, K = pb.K, tpsi = pb.tpsi, shift = pb.shift, nside = pb.mrf ? 2 : 1;
  if (K > 512 || tpsi < 0 || tpsi > 32) return FLOWB200_EUNSUPPORTED;
  P->records = tpsi >= 1 && tpsi <= 8 && (shift < 0 || shift >= 4);
  if (shift >= 0) {   // dp is a uint32
    const unsigned long long per_step = ((unsigned long long)(3 * tpsi) << shift) + 65535ull;
    if ((unsigned long long)(H > W ? H : W) * per_step >= 0xFFFF0000ull) return FLOWB200_EUNSUPPORTED;
  }
  P->L = kset_layout(H, W, K, workspace_bytes);
  if (workspace_bytes < P->L.arena) return FLOWB200_EWORKSPACE;
  const int Kpad = P->L.Kpad;
  while ((1 << P->bshift) < tpsi) ++P->bshift;
  const int minb = pb.mrf ? pick_kernels<true>(pb, P) : pick_kernels<false>(pb, P);
  if (!P->kernf64) return FLOWB200_EUNSUPPORTED;
  // ring of record slots: as many (<= 4) as keep `minb` chains per SM resident
  const int maxlen = H > W ? H : W;
  P->slot_bytes = kset_slot_bytes(Kpad);
  // + static shared memory (32-bit kernel 0.2 KB, float64 kernel 8.5 KB) + the driver's 1 KB per CTA
  const size_t budget = (size_t)(227 * 1024) / minb - 1024 - 512;
  if (4096 + chain32_fixed_smem(H < W ? H : W, nside) + 4 * (size_t)P->slot_bytes > budget) P->slot_shift = 1;
  // long chains (large images): fewer resident chains rather than smaller slots
  const size_t slots = (size_t)P->slot_bytes << P->slot_shift;
  P->smem32[0] = 4096 + chain32_fixed_smem(H, nside) + slots;
  P->smem32[1] = 4096 + chain32_fixed_smem(W, nside) + slots;
  P->smem64 = chain_fixed_smem(Kpad, maxlen, nside) + slots;
  if (P->smem64 + 1024 + 9216 > (size_t)227 * 1024) return FLOWB200_EUNSUPPORTED;
  if (P->kern32) {   // int32 modes
    const size_t smem32 = 4096 + chain32_fixed_smem(maxlen, nside) + slots;   // (4096: worst case of the run-time pad)
    if (smem32 + 1536 > (size_t)227 * 1024) return FLOWB200_EUNSUPPORTED;
    FB_CUDA_CHECK(cudaFuncSetAttribute(P->kern32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem32));
    FB_CUDA_CHECK(cudaFuncSetAttribute(P->kern32_lo, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem32));
  }
  FB_CUDA_CHECK(cudaFuncSetAttribute(P->kernf64, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P->smem64));
  return FLOWB200_OK;
}

// sort + record build for the chains this part owns
template <typename CostT>
int ksets_prepare(const BcdProblem<CostT>& pb, int part, int nparts, void* workspace, size_t workspace_bytes,
                  cudaStream_t stream) {
  if (nparts < 1 || part < 0 || part >= nparts) return FLOWB200_EINVAL;
  KsetPlan P;
  const int rc = make_plan(pb, workspace_bytes, &P);
  if (rc) return rc;
  const KsetLayout& L = P.L;
  char* ws = static_cast<char*>(workspace);
  const int H = pb.H, W = pb.W, K = pb.K, shift = pb.shift, npix = H * W;
  if (!P.records) {   // every descriptor 0: the chain kernels evaluate every step densely
    FB_CUDA_CHECK(cudaMemsetAsync(ws + L.desc, 0, 2 * (size_t)npix * sizeof(unsigned long long), stream));
    return FLOWB200_OK;
  }
  uint16_t* sorig = reinterpret_cast<uint16_t*>(ws + L.sorig);
  unsigned long long* cursor = reinterpret_cast<unsigned long long*>(ws + L.cursor);
  FB_CUDA_CHECK(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long), stream));
  int32_t* svec = reinterpret_cast<int32_t*>(ws + L.svec);
  kset_sort_kernel<<<min((npix + kSortWarps - 1) / kSortWarps, 8 * kNumSMs), kSortWarps * 32, 0, stream>>>(
      pb.pvec, pb.nprop, npix, K, L.Kst, P.bshift, sorig, svec, H, W, part, nparts);
  FB_LAUNCH_CHECK();
  const size_t bsmem = build_smem_bytes(L.Kpad);
  auto bk = kset_build_kernel<CostT>;
  FB_CUDA_CHECK(cudaFuncSetAttribute(bk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
  const int bctas = std::min(16, (int)(227 * 1024 / (bsmem + 1024)));
  bk<<<min(2 * npix, max(1, bctas) * kNumSMs), kBuildThreads, bsmem, stream>>>(
      pb.pvec, pb.cost, pb.nprop, sorig, svec, H, W, K, L.Kst, L.Kpad, pb.tpsi, P.bshift, shift < 0 ? 0 : shift,
      shift < 0 ? 0.0 : pb.lamda, P.slot_bytes, reinterpret_cast<unsigned char*>(ws + L.arena),
      (unsigned long long)L.arena_bytes, cursor, reinterpret_cast<unsigned long long*>(ws + L.desc), part, nparts);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

// one phase, the chains this part owns, in place on labels
template <typename CostT>
int ksets_phase(const BcdProblem<CostT>& pb, int32_t* labels, int phase, int part, int nparts, void* workspace,
                size_t workspace_bytes, cudaStream_t stream) {
  if (nparts < 1 || part < 0 || part >= nparts || phase < 0 || phase > 3) return FLOWB200_EINVAL;
  KsetPlan P;
  const int rc = make_plan(pb, workspace_bytes, &P);
  if (rc) return rc;
  const KsetLayout& L = P.L;
  char* ws = static_cast<char*>(workspace);
  // this part's chains [c0, c1) (single-huge-image mode; the chains of a phase are independent, python bcd.py:265-277)
  const long long nch = phase_chains(phase, pb.H, pb.W);
  const int c0 = (int)(nch * part / nparts), c1 = (int)(nch * (part + 1) / nparts);
  if (c1 <= c0) return FLOWB200_OK;
  ChainArgs a{};
  a.pvec = pb.pvec; a.cost = pb.cost; a.nprop = pb.nprop; a.labels = labels;
  a.bp = reinterpret_cast<uint16_t*>(ws + L.bp);
  a.desc = reinterpret_cast<const unsigned long long*>(ws + L.desc);
  a.arena = reinterpret_cast<const unsigned char*>(ws + L.arena);
  a.H = pb.H; a.W = pb.W; a.K = pb.K; a.Kpad = L.Kpad; a.tpsi = pb.tpsi; a.shift = pb.shift;
  a.slot_shift = P.slot_shift; a.slot_bytes = P.slot_bytes;
  a.lamda = pb.lamda; a.phase = phase; a.chain0 = c0;
  a.flags = reinterpret_cast<int32_t*>(ws + L.flags);
  a.force_generic = getenv("FLOWB200_KSET_FORCE_GENERIC") != nullptr;   // read at every call (tests)
  if (pb.shift >= 0) {
    // (1300: static shared memory + the driver's 1 KB per CTA)
    const bool fits = (size_t)P.minb * (P.smem32[phase & 1] + 1300) <= (size_t)227 * 1024;
    (fits ? P.kern32 : P.kern32_lo)<<<c1 - c0, P.T, P.smem32[phase & 1], stream>>>(a);
    FB_LAUNCH_CHECK();
  }
  // int32 modes: the blocks of the chains kern32 did not flag return at once
  P.kernf64<<<c1 - c0, P.T, P.smem64, stream>>>(a);
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

template <typename CostT>
int launch_sweeps_ksets(const BcdProblem<CostT>& pb, int32_t* labels, int sweeps, int32_t* labels_per_sweep,
                        void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (sweeps <= 0) {   // the plan only
    KsetPlan P;
    return make_plan(pb, workspace_bytes, &P);
  }
  int rc = ksets_prepare(pb, 0, 1, workspace, workspace_bytes, stream);
  if (rc) return rc;
  for (int w = 0; w < sweeps; ++w) {
    for (int phase = 0; phase < 4; ++phase) {
      rc = ksets_phase(pb, labels, phase, 0, 1, workspace, workspace_bytes, stream);
      if (rc) return rc;
    }
    if (labels_per_sweep)
      FB_CUDA_CHECK(cudaMemcpyAsync(labels_per_sweep + (size_t)w * pb.H * pb.W, labels, sizeof(int32_t) * pb.H * pb.W,
                                    cudaMemcpyDeviceToDevice, stream));
  }
  return FLOWB200_OK;
}

// The checks the entry points share, after their null-pointer checks; splits the FLOWB200_BCD_MRF flag off *bcd_mode.
// chains: K <= 512 and H, W <= 16384.  int_modes_only (prepare / phase): the cost shift checked in every mode, then
// every other mode (stray bits too) unsupported; else the shift checked in the int32 modes, the mode by with_mode.
int check_args(int H, int W, int K, int cost_shift, int* bcd_mode, bool* mrf, bool chains, bool int_modes_only) {
  if (H <= 0 || W <= 0 || K <= 0) return FLOWB200_EINVAL;
  if (chains && (K > 512 || H > 16384 || W > 16384)) return FLOWB200_EINVAL;
  *mrf = (*bcd_mode & FLOWB200_BCD_MRF) != 0;
  *bcd_mode &= ~FLOWB200_BCD_MRF;
  const bool int_mode = *bcd_mode == FLOWB200_BCD_INT32 || *bcd_mode == FLOWB200_BCD_INT32_F32COST;
  if ((int_mode || int_modes_only) && (cost_shift < 0 || cost_shift > 14)) return FLOWB200_EINVAL;
  return int_modes_only && !int_mode ? FLOWB200_EUNSUPPORTED : FLOWB200_OK;
}

// run(cost, shift) with the cost array typed for bcd_mode; shift -1 selects the float64 programme
template <typename Run>
int with_mode(int bcd_mode, const void* cost, int cost_shift, Run run) {
  switch (bcd_mode) {
    case FLOWB200_BCD_FP64_F32COST: return run(static_cast<const float*>(cost), -1);
    case FLOWB200_BCD_FP64_F64COST: return run(static_cast<const double*>(cost), -1);
    case FLOWB200_BCD_INT32: return run(static_cast<const int32_t*>(cost), cost_shift);
    case FLOWB200_BCD_INT32_F32COST: return run(static_cast<const float*>(cost), cost_shift);
    default: return FLOWB200_EINVAL;
  }
}

}  // namespace

__global__ void quantise_costs_kernel(const float* __restrict__ lcost, int32_t* __restrict__ m, size_t n, double lamda,
                                      double scale) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float c = lcost[i];
  m[i] = (c == FLOWB200_UNUSED_COST) ? 0 : (int32_t)rint(__dmul_rn(__dmul_rn(lamda, (double)c), scale));
}

}  // namespace flowb200

using namespace flowb200;

extern "C" size_t flowb200_bcd_workspace_bytes(int H, int W, int K) {
  if (H <= 0 || W <= 0 || K <= 0) return 0;
  return kset_layout(H, W, K, 0).total;
}

// fixed part only: every K-set is then evaluated densely
extern "C" size_t flowb200_bcd_min_workspace_bytes(int H, int W, int K) {
  if (H <= 0 || W <= 0 || K <= 0) return 0;
  return kset_layout(H, W, K, 0).arena;
}

extern "C" int flowb200_bcd(const int32_t* pvec, const void* cost, const int32_t* nprop, int32_t* labels, int H, int W,
                            int K, int bcd_mode, double lamda, int tpsi, int cost_shift, int sweeps,
                            int32_t* labels_per_sweep, void* workspace, size_t workspace_bytes,
                            flowb200_stream_t stream) {
  if (!pvec || !cost || !nprop || !labels || !workspace) return FLOWB200_EINVAL;
  if (sweeps < 0 || tpsi < 0) return FLOWB200_EINVAL;   // (tpsi > 32: make_plan)
  bool mrf;
  if (const int rc = check_args(H, W, K, cost_shift, &bcd_mode, &mrf, true, false)) return rc;
  // any workspace that holds the fixed part is accepted: records that do not fit are evaluated densely
  return with_mode(bcd_mode, cost, cost_shift, [&](auto c, int shift) {
    const BcdProblem<std::decay_t<decltype(*c)>> pb{pvec, c, nprop, H, W, K, lamda, tpsi, shift, mrf};
    return launch_sweeps_ksets(pb, labels, sweeps, labels_per_sweep, workspace, workspace_bytes, stream);
  });
}

// ---- the K-set programme in pieces: one part of every phase's chains (single-huge-image mode) ----
extern "C" int flowb200_bcd_prepare(const int32_t* pvec, const void* cost, const int32_t* nprop, int H, int W, int K,
                                    int bcd_mode, double lamda, int tpsi, int cost_shift, int part, int nparts,
                                    void* workspace, size_t workspace_bytes, flowb200_stream_t stream) {
  if (!pvec || !cost || !nprop || !workspace) return FLOWB200_EINVAL;
  bool mrf;
  if (const int rc = check_args(H, W, K, cost_shift, &bcd_mode, &mrf, true, true)) return rc;
  return with_mode(bcd_mode, cost, cost_shift, [&](auto c, int shift) {
    const BcdProblem<std::decay_t<decltype(*c)>> pb{pvec, c, nprop, H, W, K, lamda, tpsi, shift, mrf};
    return ksets_prepare(pb, part, nparts, workspace, workspace_bytes, stream);
  });
}

extern "C" int flowb200_bcd_phase(const int32_t* pvec, const void* cost, const int32_t* nprop, int32_t* labels, int H,
                                  int W, int K, int bcd_mode, double lamda, int tpsi, int cost_shift, int phase, int part,
                                  int nparts, void* workspace, size_t workspace_bytes, flowb200_stream_t stream) {
  if (!pvec || !cost || !nprop || !labels || !workspace) return FLOWB200_EINVAL;
  bool mrf;
  if (const int rc = check_args(H, W, K, cost_shift, &bcd_mode, &mrf, true, true)) return rc;
  return with_mode(bcd_mode, cost, cost_shift, [&](auto c, int shift) {
    const BcdProblem<std::decay_t<decltype(*c)>> pb{pvec, c, nprop, H, W, K, lamda, tpsi, shift, mrf};
    return ksets_phase(pb, labels, phase, part, nparts, workspace, workspace_bytes, stream);
  });
}

extern "C" int flowb200_energy(const int32_t* pvec, const void* cost, const int32_t* nprop, const int32_t* labels,
                               int H, int W, int K, int bcd_mode, double lamda, int tpsi, int cost_shift, double* out4,
                               flowb200_stream_t stream) {
  if (!pvec || !cost || !nprop || !labels || !out4) return FLOWB200_EINVAL;
  if (tpsi < 0 || (long long)H * W > 0x7FFFFFFFll) return FLOWB200_EINVAL;
  bool mrf;   // (the energy does not depend on the optimiser)
  if (const int rc = check_args(H, W, K, cost_shift, &bcd_mode, &mrf, false, false)) return rc;
  return with_mode(bcd_mode, cost, cost_shift, [&](auto c, int shift) {
    using CostT = std::remove_const_t<std::remove_pointer_t<decltype(c)>>;
    // (only the variants a mode can run, as for the chain kernels)
    auto kern = energy_kernel<CostT, !std::is_same<CostT, double>::value>;
    if constexpr (std::is_same<CostT, float>::value) kern = shift >= 0 ? energy_kernel<float, true> : energy_kernel<float, false>;
    kern<<<1, kEnergyThreads, 0, stream>>>(pvec, c, nprop, labels, H, W, K, lamda, tpsi, shift < 0 ? 0 : shift, out4);
    FB_LAUNCH_CHECK();
    return FLOWB200_OK;
  });
}

extern "C" int flowb200_quantise_costs(const float* lcost, int32_t* m, size_t n, double lamda, int shift,
                                       flowb200_stream_t stream) {
  if (shift < 0 || shift > 14) return FLOWB200_EINVAL;
  if (n == 0) return FLOWB200_OK;          // (an empty tensor's pointers are null)
  if (!lcost || !m) return FLOWB200_EINVAL;
  quantise_costs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(lcost, m, n, lamda, (double)(1 << shift));
  FB_LAUNCH_CHECK();
  return FLOWB200_OK;
}

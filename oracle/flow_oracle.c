/* CPU oracle, C part.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): it is the checker and the
 * timed CPU baseline, never part of the product path.
 *
 * Restates, in plain C with the reference's operation order (compiled with -ffp-contract=off):
 *   fo_generisi     daisy i flann.py:144-148 (napraviCD2), :157-189 (generisi) with FLANN replaced by
 *                   exact float64 brute force (ties -> lowest index), the search the north star prescribes
 *   fo_bcd          python bcd.py:84-88 (sidepsi), :98-99 (purepsi), :101-257 (bcd), :261-284 (ceoBCD)
 *   fo_consistency  postprocessing.py:79-117 (consistencyCheck / fowardBackwardConsistency)
 *   fo_remove_small_segments  postprocessing.py:29-76 (removeSmallSegments, scan-order quirks included)
 * It is pinned by tests/test_oracle_c.py against tests/golden/ (outputs of the reference's own source).
 * OpenMP parallelises over independent units only (cells' query bands, chains of one phase, pixels),
 * so results do not depend on the thread count.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define DESC 68

int fo_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

void fo_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}

/* float32 sum of 68 terms in numpy's pairwise_sum order for n < 128 (8 strided accumulators, tree, tail) */
static float sum68(const float* a) {
  float r[8];
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  for (int i = 8; i < 64; i += 8)
    for (int j = 0; j < 8; ++j) r[j] = r[j] + a[i + j];
  float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (int i = 64; i < DESC; ++i) res = res + a[i];
  return res;
}

/* generisi.  desc1/desc2: float32 [H][W][68].  Outputs: proposals int32 [H][W][K][2] (dy,dx) fill -1,
 * lcosts float64 [H][W][K] fill 1000, nprop int32 [H][W], bestlabels int32 [H][W],
 * knn_idx (optional) int32 [H][W][(2R+1)^2][kc] fill -1. */
int fo_generisi(const float* desc1, const float* desc2, int H, int W, int cellw, int cellh, int R, int kc, int K,
                double tphi, int32_t* proposals, double* lcosts, int32_t* nprop, int32_t* bestlabels,
                int32_t* knn_idx) {
  const int ncx = W / cellw, ncy = H / cellh, T = cellw * cellh;
  const int nblk = (2 * R + 1) * (2 * R + 1);
  if (ncx < 1 || ncy < 1 || kc < 1 || kc > T || kc > 64) return -1;
  const size_t n = (size_t)H * W;
  for (size_t i = 0; i < n * K * 2; ++i) proposals[i] = -1;
  for (size_t i = 0; i < n * K; ++i) lcosts[i] = 1000.0;
  memset(nprop, 0, n * sizeof(int32_t));
  memset(bestlabels, 0, n * sizeof(int32_t));
  if (knn_idx) for (size_t i = 0; i < n * nblk * kc; ++i) knn_idx[i] = -1;
  double* mind = (double*)malloc(n * sizeof(double));
  double* tg = (double*)malloc((size_t)T * DESC * sizeof(double));
  if (!mind || !tg) return -2;
  for (size_t i = 0; i < n; ++i) mind[i] = 1000.0;
  for (int ci = 0; ci < ncx; ++ci) {          /* ci-major, cj-minor: the slot order (:162-163) */
    for (int cj = 0; cj < ncy; ++cj) {
      for (int r = 0; r < cellh; ++r)         /* napraviCD2 (:144-148) */
        for (int c = 0; c < cellw; ++c) {
          const float* s = desc2 + ((size_t)(cj * cellh + r) * W + ci * cellw + c) * DESC;
          double* d = tg + (size_t)(r * cellw + c) * DESC;
          for (int k = 0; k < DESC; ++k) d[k] = (double)s[k];
        }
      const int x0 = cellw * (ci - R) < 0 ? 0 : cellw * (ci - R);
      const int x1 = cellw * (ci + R + 1) > W ? W : cellw * (ci + R + 1);
      const int y0 = cellh * (cj - R) < 0 ? 0 : cellh * (cj - R);
      const int y1 = cellh * (cj + R + 1) > H ? H : cellh * (cj + R + 1);
#pragma omp parallel for collapse(2) schedule(static)
      for (int y = y0; y < y1; ++y) {
        for (int x = x0; x < x1; ++x) {
          const size_t pix = (size_t)y * W + x;
          const float* qf = desc1 + pix * DESC;
          double q[DESC];
          for (int k = 0; k < DESC; ++k) q[k] = (double)qf[k];
          double bd[64];
          int bi[64];
          for (int j = 0; j < kc; ++j) { bd[j] = INFINITY; bi[j] = 0x7fffffff; }
          for (int t = 0; t < T; ++t) {
            const double* tt = tg + (size_t)t * DESC;
            double d = 0.0;
            for (int k = 0; k < DESC; ++k) { double e = q[k] - tt[k]; d += e * e; }
            if (d < bd[kc - 1]) {             /* strict: an equal distance with a higher index loses */
              int j = kc - 1;
              while (j > 0 && d < bd[j - 1]) { bd[j] = bd[j - 1]; bi[j] = bi[j - 1]; --j; }
              bd[j] = d; bi[j] = t;
            }
          }
          const int base = nprop[pix];
          const int blk = base / kc;
          for (int r = 0; r < kc; ++r) {      /* :173-189 */
            const int idx = bi[r];
            const int ty = cj * cellh + idx / cellw, tx = ci * cellw + idx % cellw;
            const float* tf = desc2 + ((size_t)ty * W + tx) * DESC;
            float ad[DESC];
            for (int k = 0; k < DESC; ++k) ad[k] = fabsf(qf[k] - tf[k]);
            double cost = (double)sum68(ad);
            if (tphi < cost) cost = tphi;
            const int slot = base + r;
            proposals[(pix * K + slot) * 2] = ty - y;
            proposals[(pix * K + slot) * 2 + 1] = tx - x;
            lcosts[pix * K + slot] = cost;
            if (cost < mind[pix]) { mind[pix] = cost; bestlabels[pix] = slot; }
            if (knn_idx) knn_idx[(pix * nblk + blk) * kc + r] = idx;
          }
          nprop[pix] = base + kc;
        }
      }
    }
  }
  free(mind);
  free(tg);
  return 0;
}

/* ---------------------------------------------------------------------------------------------------- */
static inline int l1i(const int32_t* a, const int32_t* b) { return abs(a[0] - b[0]) + abs(a[1] - b[1]); }

/* one chain (bcd(), :101-257).  old = labels of the chain before the call */
static void bcd_chain(const int32_t* prop, const double* lc, const int32_t* nprop, int32_t* labels, int H, int W, int K,
                      double lamda, int tpsi, int sy, int sx, int ystep, int xstep, double* dp, int16_t* back,
                      int32_t* oldv) {
  const int len = ystep != 0 ? H : W;
  const int s = ystep + xstep;
#define PIX(i) ((size_t)(sy + (i)*ystep) * W + (sx + (i)*xstep))
  for (int i = 0; i < len; ++i) {
    const size_t p = PIX(i);
    oldv[2 * i] = prop[(p * K + labels[p]) * 2];
    oldv[2 * i + 1] = prop[(p * K + labels[p]) * 2 + 1];
  }
  int nprev = 0;
  for (int i = 0; i < len; ++i) {
    const size_t p = PIX(i);
    const int n = nprop[p];
    double* cur = dp + (size_t)(i & 1) * K;
    const double* prv = dp + (size_t)((i & 1) ^ 1) * K;
    const int ip = i + s, im = i - s;         /* side neighbours lie ALONG the chain (:108-113) */
    double permmin = 800000.0;
    int permlab = -8;
    if (i > 0)
      for (int k = 0; k < nprev; ++k)
        if ((double)tpsi + prv[k] < permmin) { permmin = (double)tpsi + prv[k]; permlab = k; }
    const size_t pp = i > 0 ? PIX(i - 1) : 0;
    for (int l = 0; l < n; ++l) {
      const int32_t* v = prop + (p * K + l) * 2;
      int psi_p = 0, psi_m = 0;
      if (ip >= 0 && ip < len) { int d = l1i(v, oldv + 2 * ip); psi_p = d < tpsi ? d : tpsi; }
      if (im >= 0 && im < len) { int d = l1i(v, oldv + 2 * im); psi_m = d < tpsi ? d : tpsi; }
      if (i == 0) {
        cur[l] = (double)(psi_p + psi_m) + lamda * lc[p * K + l];        /* :118-120 */
      } else {
        const double small = (lamda * lc[p * K + l] + (double)psi_p) + (double)psi_m;   /* :161-162 */
        double m = INFINITY;
        int arg = -1;
        for (int k = 0; k < nprev; ++k) {
          const int d = l1i(v, prop + (pp * K + k) * 2);
          if (d < tpsi) {
            const double c = prv[k] + (double)d;
            if (c < m) { m = c; arg = k; }
          }
        }
        if (arg < 0) { m = permmin; arg = permlab; }                      /* quirk Q1 */
        cur[l] = m + small;
        back[(size_t)i * K + l] = (int16_t)arg;
      }
    }
    nprev = n;
  }
  const double* last = dp + (size_t)((len - 1) & 1) * K;
  double best = 800000.0;
  int lab = 0;
  for (int l = 0; l < nprev; ++l)
    if (last[l] < best) { best = last[l]; lab = l; }
  for (int i = len - 1; i >= 0; --i) {
    labels[PIX(i)] = lab;
    if (i > 0) lab = back[(size_t)i * K + lab];
  }
#undef PIX
}

/* ceoBCD: `sweeps` sweeps, labels in place; snaps (optional) int32 [sweeps][H][W]. */
int fo_bcd(const int32_t* prop, const double* lc, const int32_t* nprop, int32_t* labels, int H, int W, int K,
           double lamda, int tpsi, int sweeps, int32_t* snaps) {
  const int maxlen = H > W ? H : W;
  int err = 0;
  for (int w = 0; w < sweeps; ++w) {
    for (int phase = 0; phase < 4; ++phase) {
      const int nch = phase == 0 ? (W + 1) / 2 : phase == 1 ? (H + 1) / 2 : phase == 2 ? W / 2 : H / 2;
#pragma omp parallel
      {
        double* dp = (double*)malloc((size_t)2 * K * sizeof(double));
        int16_t* back = (int16_t*)malloc((size_t)maxlen * K * sizeof(int16_t));
        int32_t* oldv = (int32_t*)malloc((size_t)maxlen * 2 * sizeof(int32_t));
        if (!dp || !back || !oldv) {
#pragma omp atomic write
          err = 1;
        } else {
#pragma omp for schedule(dynamic, 1)
          for (int c = 0; c < nch; ++c) {
            switch (phase) {
              case 0: bcd_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 0, 2 * c, 1, 0, dp, back, oldv); break;
              case 1: bcd_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 2 * c, W - 1, 0, -1, dp, back, oldv); break;
              case 2: bcd_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, H - 1, 2 * c + 1, -1, 0, dp, back, oldv); break;
              default: bcd_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 2 * c + 1, 0, 0, 1, dp, back, oldv); break;
            }
          }
        }
        free(dp);
        free(back);
        free(oldv);
      }
      if (err) return -2;
    }
    if (snaps) memcpy(snaps + (size_t)w * H * W, labels, (size_t)H * W * sizeof(int32_t));
  }
  return 0;
}

/* fowardBackwardConsistency: f1 (in place), f2: float32 [A][B][3] = (dx, dy, valid).  Quirk Q5 kept. */
int fo_consistency(float* f1, const float* f2, int A, int B, float tresh) {
#pragma omp parallel for schedule(static)
  for (int a = 0; a < A; ++a) {
    for (int b = 0; b < B; ++b) {
      float* p = f1 + ((size_t)a * B + b) * 3;
      if (!(p[2] > 0.5f)) continue;
      const int a2 = (int)(p[0] + (float)a), b2 = (int)(p[1] + (float)b);
      int bad = a2 < 0 || b2 < 0 || a2 >= A || b2 >= B;
      if (!bad) {
        const float* g = f2 + ((size_t)a2 * B + b2) * 3;
        if (!(g[2] > 0.5f)) {
          bad = 1;
        } else {
          const float du = p[0] + g[0], dv = p[1] + g[1];
          const float e = sqrtf(dv * dv + du * du);
          bad = e > tresh;
        }
      }
      if (bad) p[0] = p[1] = p[2] = 0.f;
    }
  }
  return 0;
}

/* removeSmallSegments (postprocessing.py:29-76), in place on f: float32 [A][B][3] = (dx, dy, valid).
 * A = shape[0] (the reference calls it `width`), B = shape[1] (`height`).  Sequential by nature; what is kept:
 *  - seeds are visited column by column (outer index b, inner index a, :36-37) and a seed need not be valid (:41-43);
 *  - a neighbour joins when it is unvisited, valid and its float32 L1 flow difference to the CURRENT pixel is
 *    <= tresh (:62-65); neighbour order a-1, a+1, b-1, b+1 (:50-58);
 *  - a segment with 1 < count < min_size loses its valid flags (:73-75), the flow components stay;
 *  - the removal loop `for u, v in zip(...)` (:74) rebinds the scan's own `v`: the rest of the current column scan
 *    reads column b = (second index of the segment's LAST pixel) until the outer loop advances.
 * n_removed (optional): number of segments removed. */
int fo_remove_small_segments(float* f, int A, int B, float tresh, int min_size, int32_t* n_removed) {
  const size_t n = (size_t)A * B;
  uint8_t* check = (uint8_t*)calloc(n, 1);
  int32_t* q = (int32_t*)malloc(n * sizeof(int32_t));
  if (!check || !q) { free(check); free(q); return -1; }
  int removed = 0;
  for (int bo = 0; bo < B; ++bo) {
    int b = bo;
    for (int a = 0; a < A; ++a) {
      if (check[(size_t)a * B + b]) continue;
      int count = 1, curr = 0;
      q[0] = a * B + b;
      while (curr < count) {
        const int c = q[curr], ca = c / B, cb = c % B;
        const float* fc = f + (size_t)c * 3;
        const int na[4] = {ca - 1, ca + 1, ca, ca}, nb[4] = {cb, cb, cb - 1, cb + 1};
        for (int t = 0; t < 4; ++t) {
          if (na[t] < 0 || nb[t] < 0 || na[t] >= A || nb[t] >= B) continue;
          const int m = na[t] * B + nb[t];
          const float* fm = f + (size_t)m * 3;
          if (check[m] || !(fm[2] > 0.5f)) continue;
          const float d = fabsf(fc[0] - fm[0]) + fabsf(fc[1] - fm[1]);
          if (d <= tresh) { q[count++] = m; check[m] = 1; }
        }
        ++curr;
        check[c] = 1;
      }
      if (count > 1 && count < min_size) {
        for (int i = 0; i < count; ++i) f[(size_t)q[i] * 3 + 2] = 0.f;
        b = q[count - 1] % B;
        ++removed;
      }
    }
  }
  if (n_removed) *n_removed = removed;
  free(check);
  free(q);
  return 0;
}

/* ---------------------------------------------------------------------------------------------------- */
/* `tv in arr[a:b]` with Python slice semantics on the (K,2) rows of one pixel (quirk Q4) */
static int in_slice(const int32_t* rows, int K, int a, int b, const int32_t* tv) {
  if (a < 0) { a += K; if (a < 0) a = 0; } else if (a > K) a = K;
  if (b < 0) { b += K; if (b < 0) b = 0; } else if (b > K) b = K;
  for (int r = a; r < b; ++r)
    if (rows[2 * r] == tv[0] || rows[2 * r + 1] == tv[1]) return 1;
  return 0;
}

static inline uint64_t splitmix64(uint64_t* s) {
  uint64_t z = (*s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
static inline double gauss(uint64_t* s) {
  const double u1 = ((double)(splitmix64(s) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  const double u2 = ((double)(splitmix64(s) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}

/* nasumicni (daisy i flann.py:205-233).  proposals int32 [H][W][K][2], lcosts f64, nprop int32 are updated
 * in place; bestlabels is read only.  draws: optional int16 [H][W][n_gauss][2] accepted in-bounds (tgy,tgx)
 * to replay; NULL -> Gaussian draws from `seed` with the reference's rejection rules (:216-222, :233).
 * Pixels are independent: only NN slots of other pixels are read, and those are never rewritten.  The exception is
 * radius 0 on a frame that is no whole multiple of the cell (flowb200_random_proposals refuses it): a remainder pixel
 * has no NN slot, its first random proposal lands in slot 0 (its bestlabels), and the reference's x-major scan shows
 * it to the pixels after it only; this row-major parallel loop does not reproduce that. */
int fo_nasumicni(const float* desc1, const float* desc2, int H, int W, int cellw, int cellh, int kc, int K,
                 int n_gauss, double sigma, double tphi, int32_t* proposals, double* lcosts, int32_t* nprop,
                 const int32_t* bestlabels, const int16_t* draws, uint64_t seed) {
  const int ncy = H / cellh;
#pragma omp parallel for schedule(static)
  for (int y = 0; y < H; ++y) {
    for (int x = 0; x < W; ++x) {
      const size_t pix = (size_t)y * W + x;
      uint64_t st = seed * 0x100000001B3ull + pix;
      const int mincellyl = y / cellh - 2 > 0 ? y / cellh - 2 : 0;
      const int ncellyl = (ncy < y / cellh + 2 ? ncy : y / cellh + 2) - mincellyl;   /* :211 (Q4) */
      const int mincellxl = x / cellw - 2 > 0 ? x / cellw - 2 : 0;
      int32_t* rows = proposals + pix * K * 2;
      int n = nprop[pix], ng = 0;
      for (int i = 0; i < n_gauss; ++i) {
        int tgy, tgx;
        if (draws) {
          tgy = draws[(pix * n_gauss + i) * 2];
          tgx = draws[(pix * n_gauss + i) * 2 + 1];
        } else {
          for (;;) {
            tgy = (int)((double)y + sigma * gauss(&st));
            if (tgy < 0 || tgy >= H) continue;
            tgx = (int)((double)x + sigma * gauss(&st));
            if (tgx < 0 || tgx >= W) continue;
            break;
          }
        }
        const int broj = kc * ((tgy / cellh - mincellyl) + (tgx / cellw - mincellxl) * ncellyl);
        const size_t tp = (size_t)tgy * W + tgx;
        const int32_t* tv = proposals + (tp * K + bestlabels[tp]) * 2;
        if (!in_slice(rows, K, broj, broj + kc, tv) && !in_slice(rows, K, n - ng, n, tv)) {
          float df[DESC];
          const float* a = desc1 + pix * DESC;
          const float* b = desc2 + tp * DESC;
          for (int k = 0; k < DESC; ++k) df[k] = a[k] - b[k];
          double c = fabs((double)sum68(df));                       /* quirk Q6 */
          rows[2 * n] = tv[0];
          rows[2 * n + 1] = tv[1];
          lcosts[pix * K + n] = tphi < c ? tphi : c;
          ++n;
          ++ng;
        }
      }
      nprop[pix] = n;
    }
  }
  return 0;
}

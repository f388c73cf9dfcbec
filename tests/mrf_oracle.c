/* CPU oracle of FLOWB200_BCD_MRF (block coordinate descent on the MRF energy), C part.  TEST INFRASTRUCTURE: compiled
 * and bound by tests/mrf_oracle.py, never part of the product path.
 *
 * The phases of ceoBCD (python bcd.py:261-284, as oracle/flow_oracle.c fo_bcd runs them), each chain an exact
 * minimisation of E(l) = lamda * sum_p lcost(p, l_p) + sum over 4-connected pairs of min(L1(v_p, v_q), tpsi) over its
 * pixels, the rest fixed, written directly rather than as the kernels' two candidates:
 *   side terms: the two neighbours ACROSS the chain -- (y, x+1), (y, x-1) of a column chain, (y+1, x), (y-1, x) of a
 *     row chain -- with their current labels (lines of the other parity, which the phase does not write);
 *   dp0(l) = (psi+ + psi-) + lamda*lcost,  U(l) = (lamda*lcost + psi+) + psi-   (the reference's operation order);
 *   transition: first minimum over every k < nprop[prev] of dp(k) + min(L1, tpsi);
 *   end: lowest-index argmin of the last dp, backtrack.
 * Compiled with -ffp-contract=off, like flow_oracle.c.  OpenMP over the chains of a phase only: results do not depend
 * on the thread count. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static inline int l1i(const int32_t* a, const int32_t* b) { return abs(a[0] - b[0]) + abs(a[1] - b[1]); }

/* one chain; acc: 4 * len int32 (vectors of the + and - across-chain neighbours of every step) */
static void mrf_chain(const int32_t* prop, const double* lc, const int32_t* nprop, int32_t* labels, int H, int W, int K,
                      double lamda, int tpsi, int sy, int sx, int ystep, int xstep, double* dp, int16_t* back,
                      int32_t* acc) {
  const int len = ystep != 0 ? H : W;
#define PIX(i) ((size_t)(sy + (i)*ystep) * W + (sx + (i)*xstep))
  const int aoff = ystep != 0 ? 1 : W;
  const int a_p = ystep != 0 ? sx + 1 < W : sy + 1 < H, a_m = ystep != 0 ? sx > 0 : sy > 0;
  for (int i = 0; i < len; ++i) {
    const size_t p = PIX(i), pp = p + aoff, pm = p - aoff;
    if (a_p) { acc[4 * i] = prop[(pp * K + labels[pp]) * 2]; acc[4 * i + 1] = prop[(pp * K + labels[pp]) * 2 + 1]; }
    if (a_m) { acc[4 * i + 2] = prop[(pm * K + labels[pm]) * 2]; acc[4 * i + 3] = prop[(pm * K + labels[pm]) * 2 + 1]; }
  }
  int nprev = 0;
  for (int i = 0; i < len; ++i) {
    const size_t p = PIX(i);
    const int n = nprop[p];
    double* cur = dp + (size_t)(i & 1) * K;
    const double* prv = dp + (size_t)((i & 1) ^ 1) * K;
    const size_t pq = i > 0 ? PIX(i - 1) : 0;
    for (int l = 0; l < n; ++l) {
      const int32_t* v = prop + (p * K + l) * 2;
      int psi_p = 0, psi_m = 0;
      if (a_p) { int d = l1i(v, acc + 4 * i); psi_p = d < tpsi ? d : tpsi; }
      if (a_m) { int d = l1i(v, acc + 4 * i + 2); psi_m = d < tpsi ? d : tpsi; }
      if (i == 0) {
        cur[l] = (double)(psi_p + psi_m) + lamda * lc[p * K + l];
      } else {
        const double small = (lamda * lc[p * K + l] + (double)psi_p) + (double)psi_m;
        double m = INFINITY;
        int arg = 0;
        for (int k = 0; k < nprev; ++k) {
          const int d = l1i(v, prop + (pq * K + k) * 2);
          const double c = prv[k] + (double)(d < tpsi ? d : tpsi);
          if (c < m) { m = c; arg = k; }
        }
        cur[l] = m + small;
        back[(size_t)i * K + l] = (int16_t)arg;
      }
    }
    nprev = n;
  }
  const double* last = dp + (size_t)((len - 1) & 1) * K;
  double best = INFINITY;
  int lab = 0;
  for (int l = 0; l < nprev; ++l)
    if (last[l] < best) { best = last[l]; lab = l; }
  for (int i = len - 1; i >= 0; --i) {
    labels[PIX(i)] = lab;
    if (i > 0) lab = back[(size_t)i * K + lab];
  }
#undef PIX
}

/* `sweeps` sweeps of the four phases, labels in place; snaps (optional) int32 [sweeps][H][W]; phases: run only the
 * first `phases` phases of the last sweep (4 = whole sweeps) */
int mrf_bcd(const int32_t* prop, const double* lc, const int32_t* nprop, int32_t* labels, int H, int W, int K,
            double lamda, int tpsi, int sweeps, int phases, int32_t* snaps) {
  const int maxlen = H > W ? H : W;
  int err = 0;
  for (int w = 0; w < sweeps; ++w) {
    const int nph = w == sweeps - 1 ? phases : 4;
    for (int phase = 0; phase < nph; ++phase) {
      const int nch = phase == 0 ? (W + 1) / 2 : phase == 1 ? (H + 1) / 2 : phase == 2 ? W / 2 : H / 2;
#pragma omp parallel
      {
        double* dp = (double*)malloc((size_t)2 * K * sizeof(double));
        int16_t* back = (int16_t*)malloc((size_t)maxlen * K * sizeof(int16_t));
        int32_t* acc = (int32_t*)malloc((size_t)maxlen * 4 * sizeof(int32_t));
        if (!dp || !back || !acc) {
#pragma omp atomic write
          err = 1;
        } else {
#pragma omp for schedule(dynamic, 1)
          for (int c = 0; c < nch; ++c) {
            switch (phase) {
              case 0: mrf_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 0, 2 * c, 1, 0, dp, back, acc); break;
              case 1: mrf_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 2 * c, W - 1, 0, -1, dp, back, acc); break;
              case 2: mrf_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, H - 1, 2 * c + 1, -1, 0, dp, back, acc); break;
              default: mrf_chain(prop, lc, nprop, labels, H, W, K, lamda, tpsi, 2 * c + 1, 0, 0, 1, dp, back, acc); break;
            }
          }
        }
        free(dp);
        free(back);
        free(acc);
      }
      if (err) return -2;
    }
    if (snaps) memcpy(snaps + (size_t)w * H * W, labels, (size_t)H * W * sizeof(int32_t));
  }
  return 0;
}

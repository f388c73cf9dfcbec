// removeSmallSegments (postprocessing.py:29-76): the part of the algorithm that is sequential by definition.
//
// The reference flood-fills the flow field seed by seed in a fixed scan order; three things make the result depend
// on that order: (1) a seed need not be valid, and an invalid seed absorbs every not yet visited neighbouring
// segment whose flow is within `tresh` of the seed's own (stale) flow; (2) the removal loop rebinds the scan's
// column variable (`for u, v in zip(...)`, :74), so after a removal the rest of the column scan runs in another
// column; (3) that column is the second index of the LAST pixel the flood fill appended.
//
// What does not depend on the order: among VALID pixels "L1 flow difference <= tresh between 4-neighbours" is a
// symmetric relation, so a flood fill always takes whole connected components of it.  The device code therefore
// labels those components in parallel (segments.cu) and only REPLAYS the scan at component granularity: a seed
// event is O(1) (valid seed: its component; invalid seed: itself + the unvisited components its four neighbours
// belong to), and the actual breadth-first order is reproduced only for the segments that are removed
// (fewer than min_segment_size pixels each), because only their last pixel matters.
//
// All arrays are indexed in SCAN order s = b*A + a (a = first index of flow[a][b], the inner loop of the scan),
// so a column of the scan is contiguous.  This file is plain C++ (no CUDA intrinsics): tests/seg_host_emul.cpp
// compiles the same functions for the host to check the replay against the oracle without a GPU.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define SEG_HD __host__ __device__ __forceinline__
#else
#define SEG_HD static inline
struct float2 { float x, y; };   // host emulation build only
#endif

namespace flowb200 {

constexpr int32_t kSegInvalid = -1;         // root[] of an invalid pixel that has not been a seed yet
constexpr int32_t kSegInvalidChecked = -2;  // ... that has

struct SegState {
  int A, B;               // flow is [A][B][3]
  float tresh;
  int min_size;
  const float2* fT;       // (dx, dy) in scan order
  volatile int32_t* root; // component root (scan index of its first pixel) of a valid pixel, or kSegInvalid*
  const int32_t* size;    // pixels per component, at the root
  volatile uint8_t* cchk; // component already taken by a flood fill (at the root)
  uint8_t* vis;           // pixel already appended by the breadth-first replay of a removed segment
  uint8_t* touch;         // prefilter: component has a near invalid 4-neighbour (at the root)
  int32_t* queue;         // A*B scan indices
  float* flow;            // the caller's field: valid flags are cleared here
};

// :62-63, float32: |dx - dx'| + |dy - dy'| <= tresh (no products, nothing to contract)
SEG_HD bool seg_near(float2 p, float2 q, float tresh) { return fabsf(p.x - q.x) + fabsf(p.y - q.y) <= tresh; }

SEG_HD bool seg_unchecked(const SegState& S, int s) {
  const int32_t r = S.root[s];
  return r >= 0 ? !S.cchk[r] : r == kSegInvalid;
}

// scan-order neighbours of s in the reference's order a-1, a+1, b-1, b+1 (:50-58); -1 where off the image
SEG_HD void seg_neighbours(const SegState& S, int s, int nb[4]) {
  const int a = s % S.A, b = s / S.A;
  nb[0] = a > 0 ? s - 1 : -1;
  nb[1] = a + 1 < S.A ? s + 1 : -1;
  nb[2] = b > 0 ? s - S.A : -1;
  nb[3] = b + 1 < S.B ? s + S.A : -1;
}

// ---- prefilter: seed events that cannot have any effect are settled before the replay ----
// An invalid pixel none of whose valid 4-neighbours is near can never absorb anything: its event only marks itself.
// A component that no invalid pixel can absorb (no near invalid 4-neighbour) and that is not removable (one pixel, or
// min_size and more) has an event that only sets its own flag, which nobody else ever reads.  Both are marked visited
// up front; neither the order of the remaining events nor what they see changes.
// Step 1, per invalid pixel s: flag the components it could absorb; returns whether there is any.
SEG_HD bool seg_invalid_touches(const SegState& S, int s) {
  int nb[4];
  seg_neighbours(S, s, nb);
  const float2 fs = S.fT[s];
  bool any = false;
  for (int t = 0; t < 4; ++t) {
    if (nb[t] < 0) continue;
    const int32_t r = S.root[nb[t]];
    if (r < 0 || !seg_near(fs, S.fT[nb[t]], S.tresh)) continue;
    S.touch[r] = 1;
    any = true;
  }
  return any;
}
// Step 2 (after step 1 has finished everywhere), per component root r
SEG_HD bool seg_component_inert(const SegState& S, int r) {
  const int32_t n = S.size[r];
  return !S.touch[r] && (n == 1 || n >= S.min_size);
}

// One seed event of the scan (:40-75) for the unvisited pixel `seed`.  Returns the column the scan continues in:
// b itself, or the rebound column after a removal.
SEG_HD int seg_process_seed(const SegState& S, int seed, int b) {
  int nb[4];
  seg_neighbours(S, seed, nb);
  const float2 fs = S.fT[seed];
  const int32_t rs = S.root[seed];
  int32_t first[4];   // per direction: root of the neighbour the seed itself appends (:60-70), else -1
  int32_t count;
  if (rs >= 0) {
    // valid seed: the fill takes exactly its component, which is unvisited as a whole
    count = S.size[rs];
    S.cchk[rs] = 1;
    for (int t = 0; t < 4; ++t) first[t] = -1;   // recomputed below if the order is needed
  } else {
    // invalid seed: itself + every unvisited component one of its neighbours belongs to and is near enough
    S.root[seed] = kSegInvalidChecked;
    count = 1;
    for (int t = 0; t < 4; ++t) {
      first[t] = -1;
      if (nb[t] < 0) continue;
      const int32_t r = S.root[nb[t]];
      if (r < 0 || S.cchk[r] || !seg_near(fs, S.fT[nb[t]], S.tresh)) continue;
      first[t] = r;
    }
    for (int t = 0; t < 4; ++t) {
      if (first[t] < 0) continue;
      bool seen = false;
      for (int j = 0; j < t; ++j) seen = seen || first[j] == first[t];
      if (!seen) count += S.size[first[t]];
    }
    for (int t = 0; t < 4; ++t)
      if (first[t] >= 0) S.cchk[first[t]] = 1;
  }
  if (!(count > 1 && count < S.min_size)) return b;

  // removed segment: replay the breadth-first order (:45-72) to find its last pixel
  int n = 1, curr = 0;
  S.queue[0] = seed;
  S.vis[seed] = 1;
  while (curr < n) {
    const int c = S.queue[curr];
    const float2 fc = S.fT[c];
    int cn[4];
    seg_neighbours(S, c, cn);
    for (int t = 0; t < 4; ++t) {
      const int m = cn[t];
      if (m < 0 || S.vis[m]) continue;
      bool take;
      if (curr == 0 && rs < 0) {
        take = first[t] >= 0;                       // decided above, before the components were marked
      } else {
        take = S.root[m] >= 0 && seg_near(fc, S.fT[m], S.tresh);   // valid and near => same (taken) component
      }
      if (take) {
        S.queue[n++] = m;
        S.vis[m] = 1;
      }
    }
    ++curr;
  }
  for (int i = 0; i < n; ++i) {
    const int s = S.queue[i];
    S.flow[((size_t)(s % S.A) * S.B + s / S.A) * 3 + 2] = 0.f;   // :75, the flow components stay
  }
  return S.queue[n - 1] / S.A;                      // :74 leaves `v` at the last pixel's second index
}

}  // namespace flowb200

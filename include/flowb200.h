/* flowb200 — C ABI of the B200-native discrete-optical-flow hot path.
 *
 * The reference (pfe-rs/lk-s-2022-estimacija-pokreta) has no FFI: its boundary is process CLI +
 * .npy files + one importable module (SURVEY.md section 8b).  This header is the C boundary the
 * drop-in scripts in this repository bind with ctypes; each entry point names the reference
 * function (file:line under /root/reference) whose work it performs.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - images are row-major, index [y][x]; flow vectors are (dy, dx) = (rows, cols) as in the
 *     reference (daisy i flann.py:173), packed on the device as one int32:
 *         pvec = (uint16)dy | ((uint16)dx << 16)          (two's complement int16 halves);
 *     an unused proposal slot is (-1,-1) = 0xFFFFFFFF with data cost 1000.0f, as the reference
 *     fills them (daisy i flann.py:89-90);
 *   - no global state, no allocation inside the per-stage calls: the caller owns all memory and
 *     passes a workspace whose size the matching *_workspace_bytes() call returns;
 *   - every call enqueues on `stream` and returns without synchronising; it returns 0 or a
 *     negative FLOWB200_E* code (flowb200_error_string()).
 */
#ifndef FLOWB200_H
#define FLOWB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* flowb200_stream_t;

#define FLOWB200_DESC_DIM 68        /* DAISY(5,4,4,4): 17 regions x 4 bins (daisy i flann.py:66)   */
#define FLOWB200_UNUSED_COST 1000.0f /* lcosts fill (daisy i flann.py:90)                           */

enum {
  FLOWB200_OK = 0,
  FLOWB200_EINVAL = -1,      /* bad argument / unsupported parameter combination */
  FLOWB200_EWORKSPACE = -2,  /* workspace too small                              */
  FLOWB200_ECUDA = -3,       /* a CUDA runtime call failed (see flowb200_last_cuda_error) */
  FLOWB200_EUNSUPPORTED = -4
};

/* BCD arithmetic (python bcd.py:101-257).
 *   FP64_F32COST / FP64_F64COST: float64 dynamic programme with the reference's operation order,
 *       bit-exact labels for arbitrary data costs (cost array float32 resp. float64);
 *   INT32: int32 dynamic programme in units of 2^-cost_shift on integer data costs m
 *       (lamda*lcost*2^S == m, 0 <= m < 65536, 0 <= cost_shift <= 14); bit-exact with the reference whenever
 *       lcost == 20*m/2^S;
 *   INT32_F32COST: the same int32 programme fed with float32 costs, m = rint(lamda*lcost*2^S) on the fly
 *       (what flowb200_quantise_costs computes, without the extra array). */
enum { FLOWB200_BCD_FP64_F32COST = 0, FLOWB200_BCD_FP64_F64COST = 1, FLOWB200_BCD_INT32 = 2,
       FLOWB200_BCD_INT32_F32COST = 3 };

/* how the per-cell nearest-neighbour search is carried out (all give the exact answer) */
enum { FLOWB200_KNN_EXACT_FP64 = 0,   /* brute force, float64 CUDA cores                              */
       FLOWB200_KNN_TCGEN05 = 1 };    /* fp16 tcgen05 GEMM prefilter + float64 re-rank + certified fallback */

typedef struct flowb200_params {
  int32_t H, W;              /* pich, picw            daisy i flann.py:34-35 */
  int32_t cellw, cellh;      /*                        :42-43                 */
  int32_t cell_radius;       /* 2                      :167-168               */
  int32_t k_cell;            /* 5 neighbours per cell  :171-172               */
  int32_t n_gauss;           /* 25                     :207                   */
  float sigma;               /* 8                      :208                   */
  int32_t maxnprop;          /* 150                    :88                    */
  float tphi;                /* 2.5                    :46                    */
  int32_t tpsi;              /* 8                      :47                    */
  double lamda;              /* 0.05                   :48                    */
  int32_t cost_shift;        /* S of the INT32 BCD mode                      */
  int32_t bcd_mode;          /* FLOWB200_BCD_*                                */
  int32_t knn_mode;          /* FLOWB200_KNN_*                                */
  float con_tresh;           /* 10   README.md:65                             */
  int32_t cell_x0, cell_x1;  /* target cell columns searched by flowb200_knn_proposals: [cell_x0, cell_x1);
                                0, 0 = all.  For callers that shard the target cells (single-huge-image mode): the
                                slots of the other columns' proposals are left unwritten, nprop / labels assume
                                the full set.  Honoured by FLOWB200_KNN_TCGEN05 (KNN_EXACT_FP64 searches all). */
} flowb200_params;

int flowb200_version(void);
const char* flowb200_error_string(int code);
const char* flowb200_last_cuda_error(void);
/* number of kernel launches this process has enqueued through the library (diagnostics for bench.py) */
long long flowb200_launch_count(void);

/* ---- A2  izracunajDaisy  (daisy i flann.py:69-77; cv2.xfeatures2d.DAISY_create(5,4,4,4), :66) ---- */
size_t flowb200_daisy_workspace_bytes(int H, int W);
/* bgr: uint8 [H][W][3];  desc: float32 [H][W][68] */
int flowb200_daisy(const uint8_t* bgr, int H, int W, float* desc, void* workspace, size_t workspace_bytes,
                   flowb200_stream_t stream);

/* ---- A3+A4  napraviCD2 + generisi  (daisy i flann.py:144-148, 157-189) ----
 * Exact k_cell nearest neighbours (squared L2 in float64, ties -> lowest target index) of every source
 * pixel in every target cell within +-cell_radius cells; writes the NN proposal slots in the reference's
 * slot order, their truncated-L1 data costs, nprop, and bestlabels (first strict argmin, :181-184);
 * slots >= nprop are filled (-1,-1) / 1000.
 *   pvec int32 [H][W][K], lcost float32 [H][W][K], nprop int32 [H][W], labels int32 [H][W]
 *   knn_idx (optional, may be NULL): int32 [H][W][(2r+1)^2][k_cell] target index inside the cell
 *       (idx = row*cellw + col, :147-148), -1 for cells out of range; block order = slot order.
 *   stats (optional): int32[8] device counters of the tcgen05 path {tasks redone by brute force, collect-list
 *       overflows, candidate-list overflows, 0, sum of candidates handed to the re-rank, sum of collected scores}. */
size_t flowb200_knn_workspace_bytes(const flowb200_params* p);
int flowb200_knn_proposals(const float* desc_src, const float* desc_tgt, const flowb200_params* p,
                           int32_t* pvec, float* lcost, int32_t* nprop, int32_t* labels, int32_t* knn_idx,
                           int32_t* stats, void* workspace, size_t workspace_bytes, flowb200_stream_t stream);

/* diagnostics of the FLOWB200_KNN_TCGEN05 path: geom_out_host (host int32[8]) = {Tpad, stride s of the target
 * permutation pos -> idx = pos*s mod T, tiles_x, tiles_y, n_items, tile_w, tile_h, max candidates};
 * scores (optional, device float32 [n_items][tile_w*tile_h][Tpad]) = raw tensor-core ranking scores of every
 * (tile_w x tile_h query pixels, cell) work item, item = tile*n_cells + cell; the rows of an item are tile_w/16
 * consecutive 16 x tile_h MMA tiles of 128 rows.  Synchronises. */
int flowb200_knn_debug_scores(const float* desc_src, const float* desc_tgt, const flowb200_params* p, float* scores,
                              int32_t* geom_out_host, void* workspace, size_t workspace_bytes,
                              flowb200_stream_t stream);

/* ---- A6  nasumicni  (daisy i flann.py:205-233), quirks Q4/Q6 reproduced ----
 * draws: optional int16 [H][W][n_gauss][2] accepted in-bounds (tgy,tgx) samples to replay (parity mode);
 * NULL -> Philox4x32-10 Gaussian draws from `seed` with the reference's rejection rules. */
int flowb200_random_proposals(const float* desc_src, const float* desc_tgt, const flowb200_params* p,
                              int32_t* pvec, float* lcost, int32_t* nprop, const int32_t* labels,
                              const int16_t* draws, uint64_t seed, flowb200_stream_t stream);

/* ---- A8  pakovanje  (daisy i flann.py:256-309): legacy packedksets export, small sizes only ----
 * packed: uint8 [H][W][2][K*K/8+1], slot 0 = down neighbour, slot 1 = right; bits outside
 * [:nprop[p], :nprop[q]] are zero. */
int flowb200_ksets_pack(const int32_t* pvec, const int32_t* nprop, int H, int W, int K, int tpsi,
                        uint8_t* packed, flowb200_stream_t stream);

/* lamda*lcost -> integer units of 2^-S (rint), unused slots -> 0.  m: int32 [n] */
int flowb200_quantise_costs(const float* lcost, int32_t* m, size_t n, double lamda, int shift,
                            flowb200_stream_t stream);

/* ---- A9-A11  bcd / ceoBCD  (python bcd.py:101-257, 261-284) ----
 * Runs `sweeps` sweeps of the four phases (even columns down, even rows right-to-left, odd columns up,
 * odd rows left-to-right) on `labels` in place.  cost: float32 / float64 / int32 [H][W][K] per bcd_mode.
 * labels_per_sweep (optional): int32 [sweeps][H][W] snapshot after every sweep (what ceoBCD saves).
 * tpsi: 0..32 (larger: FLOWB200_EUNSUPPORTED); cost_shift (int32 modes): 0..14.
 * Every mode compiles the K-sets S_l = {k : L1(v_l,u_k) < tpsi} of every (pixel, chain direction) once per call
 * into sparse records in the workspace (the reference caches them too: pakovanje, daisy i flann.py:256-309) and the
 * chains stream them; K-sets that do not fit are evaluated on the fly, so any workspace between
 * flowb200_bcd_min_workspace_bytes() and flowb200_bcd_workspace_bytes() (the recommended size) gives the same labels.
 * Inputs outside the record format (tpsi outside 1..8, or an int32 mode with cost_shift < 4) get no records: every
 * step is evaluated on the fly. */
size_t flowb200_bcd_workspace_bytes(int H, int W, int K);
size_t flowb200_bcd_min_workspace_bytes(int H, int W, int K);
int flowb200_bcd(const int32_t* pvec, const void* cost, const int32_t* nprop, int32_t* labels,
                 int H, int W, int K, int bcd_mode, double lamda, int tpsi, int cost_shift, int sweeps,
                 int32_t* labels_per_sweep, void* workspace, size_t workspace_bytes, flowb200_stream_t stream);

/* The int32 programme in pieces, for a caller that splits the (independent) chains of every phase over several
 * GPUs and exchanges the labels between phases (single-huge-image mode, SURVEY.md 8e): part `part` of `nparts` owns
 * a contiguous range of every phase's chains.  flowb200_bcd_prepare compiles the K-sets of the owned chains (once per
 * proposal set); flowb200_bcd_phase runs the owned chains of one phase (0 even columns down, 1 even rows right to
 * left, 2 odd columns up, 3 odd rows left to right; python bcd.py:265-277) in place on labels.
 * flowb200_bcd(sweeps) == prepare(0,1) + sweeps x phases 0..3 (0,1).  INT32 / INT32_F32COST modes only. */
int flowb200_bcd_prepare(const int32_t* pvec, const void* cost, const int32_t* nprop, int H, int W, int K,
                         int bcd_mode, double lamda, int tpsi, int cost_shift, int part, int nparts,
                         void* workspace, size_t workspace_bytes, flowb200_stream_t stream);
int flowb200_bcd_phase(const int32_t* pvec, const void* cost, const int32_t* nprop, int32_t* labels, int H, int W,
                       int K, int bcd_mode, double lamda, int tpsi, int cost_shift, int phase, int part, int nparts,
                       void* workspace, size_t workspace_bytes, flowb200_stream_t stream);

/* bestlabels as generisi leaves them (daisy i flann.py:181-184): first strict minimum of the data costs of the first
 * nprop slots (0 where nprop is 0).  flowb200_knn_proposals computes them itself; this entry point serves callers that
 * assemble a proposal set from pieces (single-huge-image mode: the bands of several GPUs). */
int flowb200_best_labels(const float* lcost, const int32_t* nprop, int H, int W, int K, int32_t* labels,
                         flowb200_stream_t stream);

/* Single-huge-image mode: slot ranges of proposal arrays <-> a flat exchange buffer, one launch for a whole copy plan
 * (huge.py copy_plan; the reference has no multi-GPU path, this replaces per-range strided copies).  table: n_entries
 * (at most 65535) x 8 int64 {y0, y1, x0, x1, slot0, n, off_vec, off_cost}, x relative to the array; for y0 <= y < y1,
 * x0 <= x < x1, 0 <= s < n, with i = (y - y0) * (x1 - x0) + (x - x0):
 *   flat[off_vec + i * n + s]  <->  vec [(y * width + x) * K + slot0 + s]
 *   flat[off_cost + i * n + s] <->  cost[(y * width + x) * K + slot0 + s]   (bit pattern of the float)
 * to_flat != 0 packs the arrays into flat, 0 unpacks flat into the arrays.  Ranges must lie inside the arrays. */
int flowb200_slot_copy(const int64_t* table, int n_entries, int32_t* vec, float* cost, int width, int K,
                       int32_t* flat, int to_flat, flowb200_stream_t stream);

/* ---- A5  vratiKonacniFlow (daisy i flann.py:192-197) + A12 FlowImage.ucitajFlow (postprocessing.py:7-17) ----
 * flow_yx (optional): float64 [H][W][2] = (dy,dx);  uvv (optional): float32 [H][W][3] = (dx, dy, 1). */
int flowb200_flow_from_labels(const int32_t* pvec, const int32_t* labels, int H, int W, int K,
                              double* flow_yx, float* uvv, flowb200_stream_t stream);

/* ---- A13/A14  consistencyCheck / fowardBackwardConsistency (postprocessing.py:79-117) ----
 * flow1 (in place) and flow2: float32 [A][B][3] = (dx, dy, valid).  Quirk Q5 (dx added to the row index)
 * is reproduced.  Only pixels a0<=a<a1, b0<=b<b1 are checked (whole image: 0,A,0,B). */
int flowb200_consistency(float* flow1, const float* flow2, int A, int B, float tresh,
                         int a0, int a1, int b0, int b1, flowb200_stream_t stream);

/* ---- removeSmallSegments (postprocessing.py:29-76; SURVEY 8f row 1; disabled in the reference's postProcessing, :132) ----
 * flow (in place): float32 [A][B][3] = (dx, dy, valid).  Flood fill over 4-neighbours whose float32 L1 flow difference
 * is <= tresh; a segment with 1 < pixels < min_segment_size loses its valid flags (the flow components stay).  The
 * reference's scan-order effects (invalid seeds, the column rebinding of :74) are reproduced bit for bit: connected
 * components are labelled in parallel, the scan itself is replayed by one warp (csrc/segments_core.cuh). */
size_t flowb200_segments_workspace_bytes(int A, int B);
int flowb200_remove_small_segments(float* flow, int A, int B, float tresh, int min_segment_size, void* workspace,
                                   size_t workspace_bytes, flowb200_stream_t stream);

/* ---- edge.canny_ivice (edge.py:19-35; SURVEY 8f row 4): EpicFlow's edge input ----
 * bgr: uint8 [H][W][3].  inverted_edges: float32 [H][W], 0.0f on an edge, 1.0f elsewhere (edge.py:29).
 * cvtColor(BGR2GRAY) -> GaussianBlur(3x3, sigma 0) -> Canny(low, high) (the reference passes 100, 200), L1 gradient,
 * aperture 3: OpenCV's 8-bit integer arithmetic, bit-identical (csrc/edges_core.cuh). */
size_t flowb200_edges_workspace_bytes(int H, int W);
int flowb200_canny_edges(const uint8_t* bgr, int H, int W, int low, int high, float* inverted_edges, void* workspace,
                         size_t workspace_bytes, flowb200_stream_t stream);

/* ---- metric: visualization.errorImage (visualization.py:128-152), the EPE definition of the benchmark ----
 * test/gt: float32 [H][W][3] = (u, v, valid).  out3 (device float64[3]) = {sum of end-point errors over pixels valid
 * in both, number of them with error > abs_thresh (3.0 in the reference), number of pixels valid in both}. */
int flowb200_epe(const float* test_uvv, const float* gt_uvv, int H, int W, float abs_thresh, double* out3,
                 flowb200_stream_t stream);

/* ---- whole path, device resident: two DAISYs, per direction kNN + random proposals + `sweeps` BCD
 *      sweeps, then the forward/backward check.  bgr0/bgr1: uint8 [H][W][3].
 * out_fwd: float32 [H][W][3] checked forward field (sparse_field.npy layout); out_fwd_raw / out_bwd_raw
 * (optional): unchecked (dx,dy,1) fields of both directions. directions: 1 = forward only (no check),
 * 2 = forward + backward + check. */
size_t flowb200_pair_workspace_bytes(const flowb200_params* p);
int flowb200_flow_pair(const uint8_t* bgr0, const uint8_t* bgr1, const flowb200_params* p, int sweeps,
                       int directions, uint64_t seed, float* out_fwd, float* out_fwd_raw, float* out_bwd_raw,
                       void* workspace, size_t workspace_bytes, flowb200_stream_t stream);

/* ---- host-buffer convenience context (what the drop-in scripts and the e2e benchmark call) ----
 * Owns device workspace, pinned staging buffers and a stream on the current device. */
typedef struct flowb200_ctx flowb200_ctx;
flowb200_ctx* flowb200_ctx_create(const flowb200_params* p);
void flowb200_ctx_destroy(flowb200_ctx* ctx);
/* bgr0_host/bgr1_host: uint8 [H][W][3] host memory; out_fwd_host: float32 [H][W][3] host memory.
 * Copies in, runs flowb200_flow_pair, copies out, synchronises. */
int flowb200_ctx_flow_pair_host(flowb200_ctx* ctx, const uint8_t* bgr0_host, const uint8_t* bgr1_host,
                                int sweeps, int directions, uint64_t seed, float* out_fwd_host);
/* A batch of host-resident pairs, e.g. one rank's share of the 99 pairs x 2 directions of BASELINE.json configs[3]
 * (README.md:8, :40: pairs are independent).  Pair i of bgr0_host[] / bgr1_host[] -> out_fwd_host[i], seed seed0 + i;
 * the host<->device copies of the neighbouring pairs overlap the computation of pair i (second stream, two buffer
 * sets).  Synchronises. */
int flowb200_ctx_flow_pairs_host(flowb200_ctx* ctx, const uint8_t* const* bgr0_host, const uint8_t* const* bgr1_host,
                                 int n_pairs, int sweeps, int directions, uint64_t seed0, float* const* out_fwd_host);
/* postprocessing.fowardBackwardConsistency on host arrays (flow1_host modified in place). */
int flowb200_consistency_host(float* flow1_host, const float* flow2_host, int A, int B, float tresh,
                              int a0, int a1, int b0, int b1);

/* postprocessing.removeSmallSegments on a host array (flow_host modified in place). */
int flowb200_remove_small_segments_host(float* flow_host, int A, int B, float tresh, int min_segment_size);

/* edge.canny_ivice on host arrays (bgr_host uint8 [H][W][3] -> inverted_edges_host float32 [H][W]). */
int flowb200_canny_edges_host(const uint8_t* bgr_host, int H, int W, int low, int high, float* inverted_edges_host);

#ifdef __cplusplus
}
#endif
#endif /* FLOWB200_H */

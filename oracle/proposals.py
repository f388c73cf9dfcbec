"""Proposal generation oracle (numpy).  TEST INFRASTRUCTURE — see oracle/__init__.py.

Restates `daisy i flann.py`:
  napraviCD2   :144-148   cell regrouping of the target descriptors
  generisi     :157-189   per-cell k-NN proposals, truncated-L1 data cost, running argmin
  vratiKonacniFlow :192-197
  nasumicni    :205-233   proposals borrowed from Gaussian-sampled neighbours (quirks Q4, Q6)
  pakovanje    :256-309   K-set bit packing

The FLANN kd-tree search (`flann.nn_index`, :171-172; third-party pyflann, approximate, unseeded:
PARITY UNPINNED) is replaced by exact brute force `knn_exact` as the north star prescribes.
Everything else is pinned against the reference's own code by tests/golden (exact-kNN shim).
"""
import numpy as np


class Params:
    """Reference constants (daisy i flann.py:34-48, 88, 167-172, 207-208) made parametric."""

    def __init__(self, H, W, cellw=73, cellh=25, cell_radius=2, k_cell=5, n_gauss=25, sigma=8.0,
                 maxnprop=150, tphi=2.5, tpsi=8, lamda=0.05):
        self.H, self.W = int(H), int(W)
        self.cellw, self.cellh = int(cellw), int(cellh)
        self.cell_radius = int(cell_radius)
        self.k_cell = int(k_cell)
        self.n_gauss = int(n_gauss)
        self.sigma = float(sigma)
        self.maxnprop = int(maxnprop)
        self.tphi = float(tphi)
        self.tpsi = int(tpsi)
        self.lamda = float(lamda)

    @property
    def ncellx(self):
        return self.W // self.cellw          # :85

    @property
    def ncelly(self):
        return self.H // self.cellh          # :86


def sum_f32_numpy_order(a):
    """float32 sum over the last axis in the order numpy's pairwise_sum uses for n < 128:
    8 strided accumulators, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the n%8 tail sequentially.
    This is what `np.sum(np.absolute(d1 - d2))` (:178-180) evaluates on a 68-vector."""
    a = np.asarray(a, dtype=np.float32)
    n = a.shape[-1]
    if n < 8:
        res = np.zeros(a.shape[:-1], dtype=np.float32)
        for i in range(n):
            res = (res + a[..., i]).astype(np.float32)
        return res
    assert n <= 128
    r = [a[..., j].copy() for j in range(8)]
    m = n - (n % 8)
    for i in range(8, m, 8):
        for j in range(8):
            r[j] = (r[j] + a[..., i + j]).astype(np.float32)
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    res = res.astype(np.float32)
    for i in range(m, n):
        res = (res + a[..., i]).astype(np.float32)
    return res


def knn_exact(q, t, k, chunk=2048):
    """Exact k nearest neighbours of every row of q among the rows of t.

    Distance = sum_d (double(q_d) - double(t_d))^2 accumulated in float64; ties -> lowest index.
    Returns int32 (nq, k) indices, nearest first."""
    q = np.asarray(q, dtype=np.float32)
    t64 = np.asarray(t, dtype=np.float32).astype(np.float64)
    out = np.empty((q.shape[0], k), dtype=np.int32)
    for s in range(0, q.shape[0], chunk):
        q64 = q[s:s + chunk].astype(np.float64)
        d = np.zeros((q64.shape[0], t64.shape[0]), dtype=np.float64)
        for j in range(q64.shape[1]):                 # sequential in d, like the C/CUDA kernels
            diff = q64[:, j:j + 1] - t64[None, :, j]
            d += diff * diff
        out[s:s + chunk] = np.argsort(d, axis=1, kind="stable")[:, :k]
    return out


def cell_descriptors(desc2, p):
    """napraviCD2 (:144-148): (ncellx*ncelly, cellw*cellh, 68); cell id = ci + cj*ncellx."""
    out = np.zeros((p.ncellx * p.ncelly, p.cellw * p.cellh, desc2.shape[2]), dtype=np.float32)
    for ci in range(p.ncellx):
        for cj in range(p.ncelly):
            blk = desc2[cj * p.cellh:(cj + 1) * p.cellh, ci * p.cellw:(ci + 1) * p.cellw]
            out[ci + cj * p.ncellx] = blk.reshape(p.cellw * p.cellh, -1)
    return out


def generisi(desc1, desc2, p, knn=knn_exact):
    """generisi (:157-189) with an exact search.  Returns the reference's global arrays
    (proposals int64 (H,W,K,2) fill -1, lcosts f64 fill 1000, nprop int64, bestlabels int64)."""
    H, W, K, kc, R = p.H, p.W, p.maxnprop, p.k_cell, p.cell_radius
    proposals = np.full((H, W, K, 2), -1, dtype=np.int64)
    lcosts = np.full((H, W, K), 1000.0, dtype=np.float64)
    nprop = np.zeros((H, W), dtype=np.int64)
    mindists = np.full((H, W), 1000.0)
    bestlabels = np.zeros((H, W), dtype=np.int64)
    cd2 = cell_descriptors(desc2, p)
    for ci in range(p.ncellx):
        for cj in range(p.ncelly):
            x0, x1 = max(0, p.cellw * (ci - R)), min(W, p.cellw * (ci + R + 1))
            y0, y1 = max(0, p.cellh * (cj - R)), min(H, p.cellh * (cj + R + 1))
            tgt = cd2[ci + cj * p.ncellx]
            q = desc1[y0:y1, x0:x1].reshape(-1, desc1.shape[2])
            idx = knn(q, tgt, kc).reshape(y1 - y0, x1 - x0, kc).astype(np.int64)
            ys, xs = np.meshgrid(np.arange(y0, y1), np.arange(x0, x1), indexing="ij")
            base = nprop[y0:y1, x0:x1].copy()
            cost = sum_f32_numpy_order(np.abs(q[:, None, :] - tgt[idx.reshape(-1, kc)]))
            cost = np.minimum(np.float64(p.tphi), cost.astype(np.float64)).reshape(y1 - y0, x1 - x0, kc)
            for r in range(kc):
                slot = base + r
                proposals[ys, xs, slot, 1] = ci * p.cellw + idx[..., r] % p.cellw - xs
                proposals[ys, xs, slot, 0] = cj * p.cellh + idx[..., r] // p.cellw - ys
                lcosts[ys, xs, slot] = cost[..., r]
                better = cost[..., r] < mindists[y0:y1, x0:x1]          # strict <, :181
                mindists[y0:y1, x0:x1] = np.where(better, cost[..., r], mindists[y0:y1, x0:x1])
                bestlabels[y0:y1, x0:x1] = np.where(better, slot, bestlabels[y0:y1, x0:x1])
            nprop[y0:y1, x0:x1] += kc
    return proposals, lcosts, nprop, bestlabels


def final_flow(proposals, bestlabels):
    """vratiKonacniFlow (:192-197): float64 (H,W,2) [dy,dx]."""
    H, W = bestlabels.shape
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    return proposals[ys, xs, bestlabels].astype(np.float64)


def _in_slice(tv, arr, a, b):
    """`tv in arr[a:b]` for an (n,2) int array with Python slice semantics (quirk Q4):
    True when either component equals the same component of any row of the slice."""
    sl = arr[a:b]
    return bool((sl == tv).any())


def nasumicni(desc1, desc2, proposals, lcosts, nprop, bestlabels, p, draws, snapshot=False):
    """nasumicni (:205-233) with the accepted Gaussian draws replayed from `draws`
    (int array (H,W,n_gauss,2) of in-bounds (tgy,tgx)); modifies proposals/lcosts/nprop in place.

    The reference scans x-major and reads a neighbour's best vector from the array it is filling, so a pixel that
    had no NN proposals (bestlabels 0 pointing at an unused slot) shows its first random proposal to the pixels
    scanned after it.  snapshot=True reads every neighbour's vector as it was before the pass instead."""
    H, W = p.H, p.W
    src = proposals.copy() if snapshot else proposals
    ngaussprop = np.zeros((H, W), dtype=np.int64)
    for x in range(W):
        for y in range(H):
            mincellyl = max(0, y // p.cellh - 2)
            ncellyl = min(p.ncelly, y // p.cellh + 2) - mincellyl           # :211 (one too small: Q4)
            mincellxl = max(0, x // p.cellw - 2)
            for i in range(p.n_gauss):
                tgy, tgx = int(draws[y, x, i, 0]), int(draws[y, x, i, 1])
                broj = p.k_cell * ((tgy // p.cellh - mincellyl) + (tgx // p.cellw - mincellxl) * ncellyl)
                tv = src[tgy, tgx, bestlabels[tgy, tgx]]
                n = int(nprop[y, x])
                if (not _in_slice(tv, proposals[y, x], broj, broj + p.k_cell)) and \
                        (not _in_slice(tv, proposals[y, x], n - int(ngaussprop[y, x]), n)):
                    proposals[y, x, n] = tv
                    s = sum_f32_numpy_order((desc1[y, x] - desc2[tgy, tgx])[None, :])[0]
                    lcosts[y, x, n] = min(p.tphi, abs(float(s)))             # Q6
                    nprop[y, x] += 1
                    ngaussprop[y, x] += 1
    return proposals, lcosts, nprop


def pakovanje(proposals, nprop, p):
    """pakovanje (:256-309): uint8 (H,W,2,K*K//8+1); slot 0 = down neighbour, slot 1 = right.
    Bits outside [:nprop[p], :nprop[q]] are left zero here (the reference may leave stale bits
    there in its last row / column; nothing reads them)."""
    H, W, K = p.H, p.W, p.maxnprop
    kdim = K * K // 8 + 1
    out = np.zeros((H, W, 2, kdim), dtype=np.uint8)
    for y in range(H):
        for x in range(W):
            n = int(nprop[y, x])
            v = proposals[y, x, :n]
            for slot, (ny, nx) in enumerate(((y + 1, x), (y, x + 1))):
                if ny >= H or nx >= W:
                    continue
                m = int(nprop[ny, nx])
                u = proposals[ny, nx, :m]
                near = (np.abs(u[None, :, 0] - v[:, None, 0]) + np.abs(u[None, :, 1] - v[:, None, 1])) < p.tpsi
                bits = np.zeros((K, K), dtype=bool)
                bits[:n, :m] = near
                out[y, x, slot, :K * K // 8 + (1 if (K * K) % 8 else 0)] = np.packbits(bits.reshape(-1))
    return out


def ksets_masked_equal(a, b, nprop, p):
    """Compare two packedksets arrays on the meaningful region [:nprop[p], :nprop[q]] only."""
    H, W, K = p.H, p.W, p.maxnprop
    for y in range(H):
        for x in range(W):
            for slot, (ny, nx) in enumerate(((y + 1, x), (y, x + 1))):
                if ny >= H or nx >= W:
                    continue
                n, m = int(nprop[y, x]), int(nprop[ny, nx])
                ba = np.unpackbits(a[y, x, slot])[:K * K].reshape(K, K)[:n, :m]
                bb = np.unpackbits(b[y, x, slot])[:K * K].reshape(K, K)[:n, :m]
                if not np.array_equal(ba, bb):
                    return False
    return True

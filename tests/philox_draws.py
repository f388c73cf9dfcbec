"""A numpy restatement of the seeded draws of random_proposals_kernel (csrc/proposals.cu, draws == NULL).

Per pixel `pix` and attempt `a` (counting every attempt of the pixel, accepted or not, from 0):
  r = Philox4x32-10(counter (pix, a, 0, 0), key (seed & 0xffffffff, seed >> 32))
  u_i = (r_i + 0.5) * 2^-32
  zy = sqrt(-2 log u_0) cos(2 pi u_1),  zx = sqrt(-2 log u_2) cos(2 pi u_3)
  tgy = trunc(y + sigma zy); outside [0, H): next attempt
  tgx = trunc(x + sigma zx); outside [0, W): next attempt (tgy is drawn again too)
The first n_gauss attempts that pass are the pixel's draws.

The device evaluates log and cospi in float64 with nvcc's default FMA contraction, numpy with its own libm: the two
agree to a few ulp, which decides a truncation only when a value lies that close to an integer.  `seeded_draws`
therefore also returns, per pixel, the smallest distance of any value it truncated to an integer; a pixel whose
margin is below AMBIGUOUS is not decided by this restatement.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
AMBIGUOUS = 1e-9


def philox4x32_10(ctr, key):
    """Philox4x32-10 of uint32 counters (..., 4) under uint32 keys (..., 2) (broadcast): uint32 (..., 4)."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = PHILOX_M0 * c0, PHILOX_M1 * c2          # products of two uint32 fit a uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + PHILOX_W0) & M32, (k1 + PHILOX_W1) & M32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def seed_key(seed):
    seed = int(seed)
    return np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64)


def _margin(v):
    return np.abs(v - np.rint(v))


def attempts(pix, y, x, H, W, sigma, seed, a0, n):
    """Attempts a0 .. a0+n-1 of the pixels `pix` at (y, x): (tgy, tgx, ok, margin), each (len(pix), n); margin covers
    the values the kernel truncates (tgx only where tgy is inside the frame)."""
    pix = np.asarray(pix, dtype=np.uint64)
    a = np.arange(a0, a0 + n, dtype=np.uint64)
    ctr = np.zeros(pix.shape + (n, 4), dtype=np.uint64)
    ctr[..., 0] = pix[:, None]
    ctr[..., 1] = a[None, :]
    r = philox4x32_10(ctr, seed_key(seed)).astype(np.float64)
    u = (r + 0.5) * 2.0 ** -32
    zy = np.sqrt(-2.0 * np.log(u[..., 0])) * np.cos(2.0 * np.pi * u[..., 1])
    zx = np.sqrt(-2.0 * np.log(u[..., 2])) * np.cos(2.0 * np.pi * u[..., 3])
    vy = np.asarray(y, np.float64)[:, None] + np.float64(np.float32(sigma)) * zy
    vx = np.asarray(x, np.float64)[:, None] + np.float64(np.float32(sigma)) * zx
    tgy, tgx = np.trunc(vy), np.trunc(vx)
    oky = (tgy >= 0) & (tgy < H)
    ok = oky & (tgx >= 0) & (tgx < W)
    margin = np.where(oky, np.minimum(_margin(vy), _margin(vx)), _margin(vy))
    return tgy.astype(np.int64), tgx.astype(np.int64), ok, margin


def draws_at(pix, y, x, H, W, n_gauss, sigma, seed, block=4096):
    """The accepted draws of the pixels `pix` at (y, x) of an H x W frame: int64 (n, n_gauss, 2) (tgy, tgx), the
    margin (n,) and the number of attempts each pixel used (n,)."""
    pix, y, x = (np.asarray(v, dtype=np.int64).ravel() for v in (pix, y, x))
    n = pix.size
    out = np.zeros((n, n_gauss, 2), dtype=np.int64)
    used = np.zeros(n, dtype=np.int64)
    margin = np.full(n, np.inf)
    for s in range(0, n if n_gauss > 0 else 0, block):
        sl = slice(s, min(n, s + block))
        out[sl], margin[sl], used[sl] = _draws_block(pix[sl], y[sl], x[sl], H, W, n_gauss, sigma, seed)
    return out, margin, used


def _draws_block(pix, y, x, H, W, n_gauss, sigma, seed):
    n = pix.size
    out = np.zeros((n, n_gauss, 2), dtype=np.int64)
    got = np.zeros(n, dtype=np.int64)
    used = np.zeros(n, dtype=np.int64)
    margin = np.full(n, np.inf)
    todo = np.arange(n)
    a0, chunk = 0, min(n_gauss + n_gauss // 5 + 8, 1024)
    while todo.size:
        ty, tx, ok, mg = attempts(pix[todo], y[todo], x[todo], H, W, sigma, seed, a0, chunk)
        rank = np.cumsum(ok, axis=1) + got[todo, None]          # accepted draws up to and including each attempt
        take = ok & (rank <= n_gauss)
        rows, cols = np.nonzero(take)
        out[todo[rows], rank[rows, cols] - 1, 0] = ty[rows, cols]
        out[todo[rows], rank[rows, cols] - 1, 1] = tx[rows, cols]
        last = np.where(rank[:, -1] >= n_gauss, np.argmax(rank >= n_gauss, axis=1), chunk - 1)
        live = np.arange(chunk)[None, :] <= last[:, None]      # attempts the kernel made
        margin[todo] = np.minimum(margin[todo], np.where(live, mg, np.inf).min(axis=1))
        used[todo] += last + 1
        got[todo] = np.minimum(rank[:, -1], n_gauss)
        todo = todo[got[todo] < n_gauss]
        a0 += chunk
        chunk = min(4 * chunk, 1024)
    return out, margin, used


def seeded_draws(H, W, n_gauss, sigma, seed):
    """Every pixel's accepted draws: int16 (H, W, n_gauss, 2) as `draws` of flowb200_random_proposals expects them,
    and the margin float64 (H, W)."""
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    out, margin, _ = draws_at(np.arange(H * W), yy, xx, H, W, n_gauss, sigma, seed)
    return out.reshape(H, W, n_gauss, 2).astype(np.int16), margin.reshape(H, W)

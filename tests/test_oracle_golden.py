"""The oracle restatements against outputs of the reference's own source (tests/golden, CPU only).

pair_a / pair_b keep the reference's stage-1 proposals, costs and K-set bits as SHA-256 digests only: helpers.load_case
recomputes them with the numpy oracle and checks them against the digests before any test sees them.  A regression of
the oracle's stage 1 therefore fails in load_case (naming the case, direction and array), in every test that loads the
case.  The comparisons below (and those of test_oracle_c and the GPU parity tests) use the verified arrays."""
import numpy as np
import pytest

from helpers import load_case, load_npz, oracle_params
from oracle import bcd as obcd
from oracle import consistency as ocons
from oracle import proposals as oprop


@pytest.mark.parametrize("name,dirs", [("pair_a", (0, 1)), ("pair_b", (0,))])
def test_generisi_nasumicni_pakovanje(name, dirs):
    z = load_case(name)
    p = oracle_params(z["meta"])
    for b in dirs:
        d1, d2 = (z["desc1"], z["desc2"]) if b == 0 else (z["desc2"], z["desc1"])
        P, L, N, B = oprop.generisi(d1, d2, p)
        assert np.array_equal(B, z[f"b{b}_labels00"])
        assert np.array_equal(oprop.final_flow(P, B), z[f"b{b}_flow00"])
        oprop.nasumicni(d1, d2, P, L, N, B, p, z[f"b{b}_draws"])
        assert np.array_equal(P, z[f"b{b}_proposals"])
        assert np.array_equal(L, z[f"b{b}_lcosts"])
        assert np.array_equal(N, z[f"b{b}_nprop"])
        pk = oprop.pakovanje(P, N, p)
        assert oprop.ksets_masked_equal(pk, z[f"b{b}_packedksets"], N, p)


@pytest.mark.parametrize("name,dirs", [("pair_a", (0, 1)), ("pair_b", (0,))])
def test_bcd_fp64(name, dirs):
    z = load_case(name)
    sweeps = int(z["meta"][5])
    for b in dirs:
        got = obcd.ceo_bcd(z[f"b{b}_proposals"], z[f"b{b}_lcosts"], z[f"b{b}_nprop"], z[f"b{b}_labels00"], sweeps)
        for w in range(sweeps):
            assert np.array_equal(got[w], z[f"b{b}_labels{w + 1:02d}"]), f"sweep {w + 1} dir {b}"
            assert np.array_equal(oprop.final_flow(z[f"b{b}_proposals"], got[w]), z[f"b{b}_flow{w + 1:02d}"])


def test_bcd_quantised_costs():
    z = load_npz("bcd_q12")
    sweeps, shift = int(z["meta"][5]), int(z["meta"][6])
    lq = 20.0 * z["m"].astype(np.float64) / float(1 << shift)
    got = obcd.ceo_bcd(z["proposals"].astype(np.int64), lq, z["nprop"].astype(np.int64),
                       z["labels00"].astype(np.int64), sweeps)
    for w in range(sweeps):
        assert np.array_equal(got[w], z[f"labels{w + 1:02d}"])


def test_consistency_cases():
    z = load_npz("consistency")
    for k in ("const", "randint", "real"):
        out = ocons.post_processing(z[k + "_fwd"], z[k + "_bwd"], z[k + "_thr"].item())
        assert out.dtype == np.float32
        assert np.array_equal(out, z[k + "_out"]), k
    # quirk Q5: constant dx=+3 invalidates the bottom three ROWS
    out = z["const_out"]
    assert (out[-3:, :, 2] == 0).all() and (out[:-3, :, 2] == 1).all()


def test_consistency_pipeline_outputs():
    z = load_case("pair_a")
    for thr in (10, 2):
        out = ocons.post_processing(z["b0_flow02"], z["b1_flow02"], thr)
        assert np.array_equal(out, z[f"sparse_thr{thr}"])


def zac_masks(nprop, H, W, K):
    """For every entry of the four `pakovani za c` arrays (daisy i flann.py:321-398): the (pixel, neighbour) pair it
    holds, as index arrays.  Returns a list of four (index tuple into the array, p_y, p_x, q_y, q_x)."""
    out = []
    ty, tx = np.meshgrid(np.arange(H - 1), np.arange(0, W, 2), indexing="ij")           # even columns, down
    out.append(((tx // 2, ty), ty, tx, ty + 1, tx))
    ty, tx = np.meshgrid(np.arange(0, H, 2), np.arange(W - 1), indexing="ij")           # even rows, right to left
    out.append(((ty // 2, W - 2 - tx), ty, tx, ty, tx + 1))
    ty, tx = np.meshgrid(np.arange(H - 1), np.arange(1, W, 2), indexing="ij")           # odd columns, up
    out.append((((W - 1 - tx) // 2, H - 2 - ty), ty, tx, ty + 1, tx))
    ty, tx = np.meshgrid(np.arange(1, H, 2), np.arange(W - 1), indexing="ij")           # odd rows, left to right
    out.append((((H - 1 - ty) // 2, tx), ty, tx, ty, tx + 1))
    return out


def assert_zac_equal(got, z):
    """got: the four arrays of pack_for_c; z: tests/golden/zac.npz.  Bits are compared inside [:nprop[p], :nprop[q]]
    (the reference's scratch matrix keeps stale bits outside it in the last row / column loops, :366-393); entries
    the reference never writes must be zero in both."""
    H, W, _, _, _, K = (int(v) for v in z["meta"])
    nprop = z["nprop"].astype(np.int64)
    for i, (where, py, px, qy, qx) in enumerate(zac_masks(nprop, H, W, K)):
        want, have = z[f"zac{i}"], got[i]
        assert have.shape == want.shape and have.dtype == np.uint8
        written = np.zeros(want.shape[:2], bool)
        written[where] = True
        assert not want[~written].any() and not have[~written].any()
        wb = np.unpackbits(want[where], axis=-1)[..., :K * K].reshape(py.shape + (K, K))
        hb = np.unpackbits(have[where], axis=-1)[..., :K * K].reshape(py.shape + (K, K))
        l = np.arange(K)
        mask = (l[None, None, :, None] < nprop[py, px][..., None, None]) & \
               (l[None, None, None, :] < nprop[qy, qx][..., None, None])
        assert np.array_equal(wb & mask, hb & mask), f"pakovani za c {i}"
        assert not (hb & ~mask).any()


def test_pack_for_c_contents():
    """stage1.pack_for_c (host re-layout of the K-set bits) against the reference's own pakovanjeZaC output."""
    from helpers import pkg
    z = load_npz("zac")
    H, W, cw, ch, _, K = (int(v) for v in z["meta"])
    p = oprop.Params(H, W, cw, ch, maxnprop=K)
    pk = oprop.pakovanje(z["proposals"].astype(np.int64), z["nprop"].astype(np.int64), p)
    assert_zac_equal(pkg("stage1").pack_for_c(pk, H, W), z)


def test_error_image_metric():
    """oracle.epe.error_image against visualization.errorImage itself (exec'd by tests/golden/make_golden_extra.py)."""
    from oracle import epe as oepe
    z = load_npz("epe")
    for k in range(3):
        mean, outl, n = oepe.error_image(z[f"c{k}_test"], z[f"c{k}_gt"])
        assert n == int(z[f"c{k}_nvalid"])
        # the reference prints str(np.float32 mean): equal to float32 precision; the percentage is an exact ratio
        assert np.float32(mean) == np.float32(z[f"c{k}_mean"]), (mean, z[f"c{k}_mean"])
        assert abs(outl - float(z[f"c{k}_outliers"])) < 1e-9

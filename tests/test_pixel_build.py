"""CPU checks of tests/pixel_build.py and of the forward transform's FP32 error table: the kernel's kAanErrBound covers
tools/aan_error_bound.bound() at every (i, j), the builder's tables are the reference's, and the families are reproducible
and do what they claim according to the reference encoder's own FP64 DCT values (the oracle)."""
import os
import sys

import numpy as np
import pytest

import pixel_build as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_kernel_error_table_covers_flowgraph_bound():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import aan_error_bound
    finally:
        sys.path.remove(os.path.join(ROOT, "tools"))
    B = aan_error_bound.bound().reshape(64)
    table = P.aan_err_bound()
    assert (table >= B).all(), "kAanErrBound below the flowgraph bound at %s" % np.nonzero(table < B)[0].tolist()
    assert (table - B).min() == 0.0 and table.max() < 7.5e-3     # the exact positions (0 and 0) and the (7,7) bound


def test_tables_are_the_reference_tables(oracle):
    zz, qy, qc, _, _ = oracle.tables()
    assert (P.QY == qy).all() and (P.QC == qc).all()
    assert (P.ZZ == zz).all() or (P.ZZ == np.argsort(zz)).all()


def test_colour_inverse():
    luma, cb, cr, pair = P.colour_tables()
    for tbl, want, off in ((luma, (np.arange(256) - 128, 0, 0), 128), (cb, (None, np.arange(241) - 120, 0), 120),
                           (cr, (None, 0, np.arange(241) - 120), 120)):
        r, g, b = P.unpack(tbl)
        got = (P.ref_y(r, g, b), P.ref_cb(r, g, b), P.ref_cr(r, g, b))
        for x, w in zip(got, want):
            if w is not None:
                assert (x == w).all()
    lo, hi = P.PAIR_RANGE
    cbv, crv = np.meshgrid(np.arange(lo, hi + 1), np.arange(lo, hi + 1), indexing="ij")
    r, g, b = P.unpack(pair[(cbv + 128) * 256 + crv + 128])
    assert (P.ref_cb(r, g, b) == cbv).all() and (P.ref_cr(r, g, b) == crv).all()


@pytest.fixture(scope="module")
def ties():
    return P.ties_image(11)


def test_ties_reproducible_and_certified(oracle, ties):
    r, g, b, W, H = ties
    again = P.ties_image(11)
    assert all((x == y).all() for x, y in zip(ties[:3], again[:3]))
    _, raw = oracle.coefs(r, g, b, W, H, want_raw=True)
    d = P.certify(raw)
    assert (d == P.certify(oracle.coefs(*again, want_raw=True)[1])).all()
    sure, unsure = P.queued(d)
    exact = d < 1e-6
    tie_blocks = np.zeros(exact.shape[:2], bool)
    tie_blocks[0::2, :4] = tie_blocks[1::2, 4:] = True                 # luma ties in even MCUs, chroma ties in odd ones
    assert (exact.sum(2)[tie_blocks] >= 5).all()
    assert (exact <= sure).all()
    nat = [[i * 8 + j for i, j in s] for s in P.TIE_SETS]
    for pos in nat[0] + nat[1]:
        for cls in (0, 1):
            blocks = raw[:, 4:] if cls else raw[:, :4]
            k = np.round(blocks[..., pos] / P.Q[cls][pos])
            tied = (exact & tie_blocks[..., None])[:, 4:, pos] if cls else (exact & tie_blocks[..., None])[:, :4, pos]
            assert set(k[tied].astype(int).tolist()) >= {-1, 1}, (cls, pos)     # both signs at k = +-1
            if P.Q[cls][pos] < 70:
                assert np.abs(k[tied]).max() >= 2, (cls, pos)


def mask_of(coefs):
    """bit g: zig-zag group g (group 0 without the DC) holds a non-zero coefficient"""
    c = np.asarray(coefs).reshape(-1, 64).copy()
    c[:, 0] = 0
    return (c.reshape(-1, 8, 8) != 0).any(2).astype(np.int64) @ (1 << np.arange(8))


def test_masks_cover_every_group_pattern(oracle):
    r, g, b, W, H = P.mask_image(12)
    c = oracle.coefs(r, g, b, W, H)
    for cls, blocks in ((0, c[:, :4]), (1, c[:, 4:])):
        assert set(mask_of(blocks).tolist()) == set(range(256)), cls
    # all-black and all-white MCUs (320, 321): the extreme DC values of luma
    assert (c[320, :4, 0] == c[:, :4, 0].min()).all() and (c[321, :4, 0] == c[:, :4, 0].max()).all()
    assert c[320, 0, 0] <= -63 and c[321, 0, 0] >= 63
    dconly = (mask_of(c[:, :4]) == 0) & (c[:, :4, 0].reshape(-1) != 0)
    assert dconly.sum() >= 80


def test_sweep_reproducible_and_covers_every_position(oracle):
    r, g, b, W, H = P.sweep_image(13)
    assert all((x == y).all() for x, y in zip((r, g, b), P.sweep_image(13)[:3]))
    _, raw = oracle.coefs(r, g, b, W, H, want_raw=True)
    missing = sweep_gaps(raw)
    assert not missing, missing[:8]


def sweep_gaps(raw):
    """(class, i, j) without a block at every guard-band distance of the sweep, and on both sides of |w| = 1 - 2G"""
    d = P.certify(raw)
    w = np.abs(raw) / P.Q[(np.arange(6) >= 4).astype(np.int64)][None]
    gaps = []
    for cls, blk in ((0, slice(0, 4)), (1, slice(4, 6))):
        for n in range(1, 64):
            if divmod(n, 8) in P.RATIONAL:
                continue
            x, y = d[:, blk, n].ravel(), w[:, blk, n].ravel()
            need = [(x < 0.25).any()] + [(np.abs(x - t) < 0.1).any() for t in (0.5, 1, 2, 4)]
            need += [((y < 1) & (x > 2) & (x < 3)).any(), ((y < 1) & (x < 2)).any()]
            if not all(need):
                gaps.append((cls, divmod(n, 8), need))
    return gaps

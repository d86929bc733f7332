"""The entropy decoder (dec_entropy.cuh) against a sequential restatement on adversarial DHT tables and hand-built streams.

Tables: every code length 1..16, end-of-block and DC category 0 at 16 bits (the slow lookup, nothing folded); a 1-bit
end-of-block with symbols on both sides of the fold boundary (used + eob_len = 10 / 11); nothing shorter than 11 bits (fast tables
all kEntryNone); fixed-length codes (slow self-synchronisation: repair launches, EAGAIN, the host loop); a very incomplete code
("no such code" while speculating); 27-bit symbols (16-bit DC code + category 11); the device optimiser's 16-bit tables.
Coefficients: dense full range, long zero runs and ZRL at the end of a block, DC differences at the category 10/11 boundaries,
2-bit blocks, streams that are mostly FF bytes, photographic content.  Streams come from tests/jpeg_build.py (numpy, pinned to the
oracle's encoder and to libjpeg by the CPU tests below).  Bar: the very coefficients, the very pixels of the reference decoder, and
ECORRUPT -- never a wrong result -- for malformed streams."""
import io
import os
import subprocess

import numpy as np
import pytest

import jpeg_build as B
from jpeg_build import LAYOUTS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEC = os.path.join(ROOT, "jpezy_b200", "bin", "jpezy_decode")
ECORRUPT, EAGAIN = 5, 9
OPT_SYNC_ROUNDS, OPT_SYNC_GUESSES = 3, 6
STAT_SYNC_ROUNDS, STAT_SYNC_ITERS0, STAT_SYNC_ITERS1 = 4, 5, 6
DEFAULT_ROUNDS, DEFAULT_GUESSES = 3, 0          # context.h


# ---- table families ---------------------------------------------------------------------------------------------------
def _ac_rest(first):
    return [s for s in B.AC_SYMBOLS if s not in first]


def family_tables(name):
    """{class: (DC Huff, AC Huff)}; luma and chroma differ in every family"""
    T = B.table
    if name == "annexk":
        return {k: (B.ANNEX_K[0][k], B.ANNEX_K[1][k]) for k in (0, 1)}
    if name == "chain16":
        # lengths 1..8 and 16 (AC), 1..11 and 16 (luma DC), 1..5 and 12..16 (chroma DC): every length 1..16 is used; ZRL at 1 bit,
        # end-of-block and DC category 0 at 16 bits
        acs = []
        for chain in ([0x01, 0x02, 0x11, 0x03, 0x21, 0x04, 0x12], [0x02, 0x01, 0x03, 0x11, 0x05, 0x31, 0x04]):
            pairs = [(0xF0, 1)] + [(s, 2 + i) for i, s in enumerate(chain)] + [(s, 16) for s in _ac_rest([0xF0] + chain)]
            acs.append(T(pairs if chain[0] == 0x01 else pairs[:8] + pairs[8:][::-1]))
        dc0 = T([(k, k) for k in range(1, 12)] + [(0, 16)])
        dc1 = T([(1, 1), (2, 2), (3, 3), (4, 4), (5, 5), (6, 12), (7, 13), (8, 14), (9, 15), (10, 16), (11, 16), (0, 16)])
        return {0: (dc0, acs[0]), 1: (dc1, acs[1])}
    if name == "eob1":
        # luma: ZRL and DC category 0 at 9 bits, (0,1) and DC category 1 at 8 bits -> used + 1 == 10 (folded); (0,2) at 8 bits, the
        # others at 9 / 10 -> used + 1 >= 11 (not folded).  Chroma: DC category 0 at 1 bit, so an empty block takes 2 bits.
        ac0 = T([(0x00, 1), (0x01, 8), (0x02, 8), (0xF0, 9)] + [(s, 9 if s >> 4 < 8 else 10) for s in _ac_rest([0x00, 0x01, 0x02, 0xF0])])
        ac1 = T([(0x00, 1), (0x01, 9), (0xF0, 10)] + [(s, 9 if (s >> 4) % 2 == 0 else 10) for s in _ac_rest([0x00, 0x01, 0xF0])])
        dc0 = T([(1, 8), (2, 8), (0, 9)] + [(k, 9 + k % 2) for k in range(3, 12)])
        dc1 = T([(0, 1)] + [(k, 5) for k in range(1, 12)])
        return {0: (dc0, ac0), 1: (dc1, ac1)}
    if name == "all_slow":
        ac0 = T([(s, 11 + min(5, i // 30)) for i, s in enumerate(B.AC_SYMBOLS)])
        ac1 = T([(s, 11 + min(5, i // 20)) for i, s in enumerate(B.AC_SYMBOLS[::-1])])
        return {0: (T([(k, 11 + k % 6) for k in range(12)]), ac0), 1: (T([(k, 12 + k % 5) for k in range(12)]), ac1)}
    if name == "fixed8":
        return {0: (T([(k, 4) for k in range(12)]), T([(s, 8) for s in B.AC_SYMBOLS])),
                1: (T([(k, 4) for k in range(11, -1, -1)]), T([(s, 8) for s in B.AC_SYMBOLS[::-1]]))}
    if name == "sparse":
        # Kraft sums 0.24 / 0.14 (AC) and 0.375 / 0.19 (DC): most bit positions start no code word at all
        ac0 = T([(0x00, 3)] + [(s, 8 if i < 20 else 12) for i, s in enumerate(_ac_rest([0x00]))])
        ac1 = T([(0x00, 4)] + [(s, 9 if i < 30 else 13) for i, s in enumerate(_ac_rest([0x00])[::-1])])
        return {0: (T([(k, 5) for k in range(12)]), ac0), 1: (T([(k, 6) for k in range(12)]), ac1)}
    if name == "max_consume":
        # DC category 11 at 16 bits (27-bit symbols); AC (0,10) and (15,10) at 16 bits (26-bit symbols)
        dc0 = T([(k, L) for k, L in enumerate([2, 3, 3, 3, 3, 3, 4, 5, 6, 7, 8])] + [(11, 16)])
        dc1 = T([(k, L) for k, L in enumerate([2, 2, 2, 3, 4, 5, 6, 7, 8, 9, 10])] + [(11, 16)])
        ac1 = B.ANNEX_K[1][1].lengths()
        ac1[0x0A] = 16
        return {0: (dc0, B.ANNEX_K[1][0]), 1: (dc1, T(sorted(ac1.items(), key=lambda p: (p[1], p[0] == 0x0A))))}
    if name == "optimised":
        hist, _ = B.symbol_hist(B.fibonacci_coefs()[0])
        mk = lambda counts: B.Huff(*B.gen_optimal_table(counts)[:2])   # noqa: E731
        return {k: (mk(hist[k, :16]), mk(hist[k, 16:])) for k in (0, 1)}
    if name == "ff":
        # a chain: end-of-block '0', ..., (0,10) = 1111111111111110; with every AC coefficient 1023 a block is 63 x 26 bits of
        # which one is zero, so most bytes of the segment are FF (and stuffed)
        chains = ([0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x11, 0x12, 0x13, 0x14, 0x15],
                  [0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x21, 0x22, 0x23, 0x24, 0x25])
        out = {}
        for k, ch in enumerate(chains):
            out[k] = (T([(0, 1)] + [(c, 5 + k) for c in range(1, 12)]), T([(0x00, 1)] + [(s, 2 + i) for i, s in enumerate(ch)] + [(0x0A, 16)]))
        return out
    raise KeyError(name)


TABLE_FAMILIES = ["annexk", "chain16", "eob1", "all_slow", "fixed8", "sparse", "max_consume", "optimised"]
COEF_FAMILIES = ["dense", "zrl", "dc11", "eob_only", "ff_heavy", "photo"]
LAYOUT_NAMES = ["420", "444", "422", "440", "gray1"]
GEOMS = [(200, 120), (8, 8), (264, 136), (1, 1), (96, 64), (640, 360)]


# ---- coefficient families -------------------------------------------------------------------------------------------
def coefficients(family, nblk, comp, seed, oracle=None):
    """int32 [nblk, 64]: zig-zag, scan order, absolute DC; |AC| <= 1023, |DC difference| <= 2047 in every restart interval"""
    rng = np.random.default_rng(seed)
    c = np.zeros((nblk, 64), np.int64)
    comp = np.tile(np.asarray(comp), nblk // len(comp))
    sgn = lambda n: rng.choice([-1, 1], n)          # noqa: E731
    if family == "dense":
        c[:] = rng.integers(1, 1024, (nblk, 64)) * sgn((nblk, 64))
        c[:, 0] = rng.integers(-1023, 1024, nblk)
    elif family == "zrl":
        kind = rng.integers(0, 5, nblk)
        v = lambda: rng.integers(1, 1024, nblk) * sgn(nblk)       # noqa: E731
        p = rng.integers(17, 64, nblk)
        r = np.arange(nblk)
        c[r[kind == 0], p[kind == 0]] = v()[kind == 0]           # one coefficient after a run of 16..62
        for k, (a, b) in {1: (47, 63), 2: (46, 63), 3: (1, 63)}.items():
            m = kind == k                                        # (15, s) onto 63; ZRL right before 63; ZRL, ZRL, ZRL, (13, s)
            c[m, a], c[m, b] = v()[m], v()[m]
        m = kind == 4                                            # a run, one coefficient, the end of block
        c[r[m], np.minimum(p[m], 62)] = v()[m]
        c[:, 0] = rng.integers(-40, 41, nblk)
    elif family == "dc11":
        steps = np.array([2047, 1024, 1023, 512, 511])
        for k in set(comp.tolist()):
            i = np.nonzero(comp == k)[0]
            dc, seq = 0, []
            for m in steps[rng.integers(0, 5, i.size)]:
                dc = dc - m if dc > 0 else dc + m                 # towards zero: |DC| <= 2047
                seq.append(dc)
            c[i, 0] = seq
        c[:, 1:4] = rng.integers(-3, 4, (nblk, 3))
    elif family == "eob_only":
        pass
    elif family == "ff_heavy":
        c[:, 1:] = 1023
    elif family == "photo":
        import jpezy_b200 as J
        W, H = 256, 128
        flat = np.concatenate([oracle.coefs(*J.synth.image(f, W, H, seed % 7), W, H).reshape(-1, 64) for f in (0, 1)])
        c[:] = np.resize(flat, (nblk, 64))
    else:
        raise KeyError(family)
    return c.astype(np.int32)


def case_list():
    """(table family, coefficient family, layout, W, H): tables x coefficients rotated over the layouts and sizes"""
    out = []
    for ti, t in enumerate(TABLE_FAMILIES):
        if t == "optimised":
            out.append((t, "fibonacci", "420") + B.fibonacci_coefs()[1:])
            continue
        for ci, cf in enumerate(COEF_FAMILIES):
            out.append((t, cf, LAYOUT_NAMES[(ti + ci) % 5]) + GEOMS[(ti + 2 * ci) % len(GEOMS)])
    return out


CASES = case_list()


class Stream:
    def __init__(self, tfam, cfam, layout, W, H, nimg=2, restart_interval=0, oracle=None, seed=0):
        self.tfam, self.cfam, self.layout, self.W, self.H, self.ri = tfam, cfam, layout, W, H, restart_interval
        self.tables = family_tables("ff" if cfam == "ff_heavy" else tfam)
        nmcu, self.nb, comp = B.geometry(W, H, layout)
        self.nblk = nmcu * self.nb
        if cfam == "fibonacci":
            fib = B.fibonacci_coefs()[0].reshape(-1, 64).astype(np.int32)
            self.coefs = [fib] * nimg
        else:
            base = 1000 * TABLE_FAMILIES.index(tfam) + 10 * COEF_FAMILIES.index(cfam) + seed
            self.coefs = [coefficients(cfam, self.nblk, comp, base + i, oracle) for i in range(nimg)]
        self.scans = [B.encode_scan(c, layout, self.tables, restart_interval) for c in self.coefs]

    def file(self, i=0, **kw):
        return B.jpeg_file(self.W, self.H, self.layout, self.scans[i], self.tables, restart_interval=self.ri, **kw)

    def name(self):
        return "%s/%s/%s %dx%d R%d" % (self.tfam, self.cfam, self.layout, self.W, self.H, self.ri)


@pytest.fixture(scope="module")
def streams(oracle):
    return [Stream(*c, oracle=oracle) for c in CASES]


def annexk_file(s, i=0):
    K = family_tables("annexk")
    return B.jpeg_file(s.W, s.H, s.layout, B.encode_scan(s.coefs[i], s.layout, K, s.ri), K, restart_interval=s.ri)


def oracle_coefs(oracle, f):
    return oracle.decode_coefs(f).reshape(-1, 64)


# ---- CPU: the writer itself -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("restart_interval", [0, 1, 7, 10000])
def test_writer_matches_oracle_encoder(oracle, restart_interval):
    """Annex K tables, 4:2:0: the segment is the oracle encoder's byte for byte"""
    import jpezy_b200 as J
    K = family_tables("annexk")
    for fam, (W, H) in ((0, (200, 120)), (1, (264, 136))):
        c = oracle.coefs(*J.synth.image(fam, W, H, 1), W, H).astype(np.int32)
        assert B.encode_scan(c.reshape(-1, 64), "420", K, restart_interval) == oracle.scan_from_coefs(c, restart_interval=restart_interval)
    c = coefficients("dense", 6 * 40, [0, 0, 0, 0, 1, 2], 5)
    assert B.encode_scan(c, "420", K, restart_interval) == oracle.scan_from_coefs(c.reshape(-1, 6, 64), restart_interval=restart_interval)


def test_table_families_are_valid():
    for name in TABLE_FAMILIES + ["ff"]:
        T = family_tables(name)
        assert [(h.bits, h.vals) for h in T[0]] != [(h.bits, h.vals) for h in T[1]], name
        for k in (0, 1):
            for h in T[k]:
                assert 0 < h.kraft() < 65536, name
    L = lambda n, k, t: family_tables(n)[k][t].lengths()                    # noqa: E731
    assert {l for k in (0, 1) for t in (0, 1) for l in L("chain16", k, t).values()} == set(range(1, 17))
    assert all(L("chain16", k, 1)[0x00] == 16 and L("chain16", k, 0)[0] == 16 and L("chain16", k, 1)[0xF0] == 1 for k in (0, 1))
    assert min(l for k in (0, 1) for t in (0, 1) for l in L("all_slow", k, t).values()) == 11
    assert L("max_consume", 0, 0)[11] == 16 and L("max_consume", 1, 1)[0x0A] == 16 and L("max_consume", 0, 1)[0xFA] == 16
    assert max(L("optimised", 0, 1).values()) == 16
    e = L("eob1", 0, 1)
    assert e[0x00] == 1 and {e[0xF0] + 0 + 1, e[0x01] + 1 + 1, e[0x02] + 2 + 1} == {10, 11}


def test_every_file_decodes_to_its_coefficients(oracle, streams):
    for s in streams:
        for i in range(len(s.coefs)):
            assert (oracle_coefs(oracle, s.file(i)) == s.coefs[i]).all(), s.name()
    s = next(s for s in streams if s.cfam == "ff_heavy")
    assert s.scans[0].count(b"\xff") > len(s.scans[0]) // 3          # FF + stuffed 00: most of the bytes


@pytest.mark.parametrize("tfam", TABLE_FAMILIES)
def test_libjpeg_decodes_like_annex_k(streams, tfam):
    """libjpeg (through Pillow) opens every adversarial-table file and gets the pixels of the Annex K file of the same coefficients"""
    from PIL import Image
    for s in streams:
        if s.tfam != tfam:
            continue
        a = np.asarray(Image.open(io.BytesIO(s.file(0))).convert("RGB"))
        k = np.asarray(Image.open(io.BytesIO(annexk_file(s))).convert("RGB"))
        assert a.shape == k.shape and (a == k).all(), s.name()


def test_writer_options(oracle, streams):
    """tables at ids 2 / 3, several tables per DHT segment or one each, restart intervals: the oracle reads them all"""
    s = streams[1]
    c = s.coefs[0]
    for ids, per in (((2, 0), False), ((1, 2), True)):
        extra = [(0x03, B.ANNEX_K[0][0]), (0x13, B.ANNEX_K[1][1])]
        f = B.jpeg_file(s.W, s.H, s.layout, s.scans[0], s.tables, ids=ids, extra=extra, dht_per_table=per)
        assert (oracle_coefs(oracle, f) == c).all()
    for R in (1, 3):
        f = B.jpeg_file(s.W, s.H, s.layout, B.encode_scan(c, s.layout, s.tables, R), s.tables, restart_interval=R)
        assert (oracle_coefs(oracle, f) == c).all()


# ---- device --------------------------------------------------------------------------------------------------------
def frame_for(s, ids=(0, 1), restart_interval=None, qt=None):
    import jpezy_b200 as J
    hs, vs = LAYOUTS[s.layout]
    f = J.default_frame(s.W, s.H)
    f.ncomp = len(hs)
    for i in range(len(hs)):
        f.hs[i], f.vs[i], f.tq[i] = hs[i], vs[i], min(i, 1)
        f.td[i] = f.ta[i] = ids[min(i, 1)]
    for k in (0, 1):
        for t in (0, 1):
            set_huff(f.ht[t][ids[k]], s.tables[k][t])
    q = np.ones((2, 64), np.int64) if qt is None else qt
    for k in (0, 1):
        for i in range(64):
            f.qt[k][i] = int(q[k][i])
    f.restart_interval = s.ri if restart_interval is None else restart_interval
    return f


def set_huff(dst, h):
    dst.present = 1
    for i in range(16):
        dst.bits[i] = h.bits[i]
    for i in range(256):
        dst.vals[i] = h.vals[i] if i < len(h.vals) else 0


def upload(scans):
    import torch
    slot = max(len(x) for x in scans) + 64
    buf = np.zeros((len(scans), slot), np.uint8)
    for i, x in enumerate(scans):
        buf[i, :len(x)] = np.frombuffer(x, np.uint8)
    return torch.from_numpy(buf).cuda(), slot, np.array([len(x) for x in scans], np.uint64)


def entropy(ctx, scans, frame, nblk, rounds=DEFAULT_ROUNDS, guesses=DEFAULT_GUESSES):
    """entropy_decode_dev on the segments -> (coefficients [nimg, nblk, 64], statuses, (rounds, iters0, iters1))"""
    import torch
    from gpu_util import Guarded
    d_scan, slot, nbytes = upload(scans)
    n = len(scans)
    out = Guarded(n * nblk * 64, torch.int16, fill=0x7777)
    st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    ctx.set_option(OPT_SYNC_ROUNDS, rounds)
    ctx.set_option(OPT_SYNC_GUESSES, guesses)
    try:
        torch.cuda.synchronize()
        ctx.entropy_decode_dev(d_scan, slot, nbytes, n, frame, out.view, st, stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    finally:
        ctx.set_option(OPT_SYNC_ROUNDS, DEFAULT_ROUNDS)
        ctx.set_option(OPT_SYNC_GUESSES, DEFAULT_GUESSES)
    assert out.intact(), "a guard zone of the coefficient buffer was written"
    stats = tuple(ctx.stat(k) for k in (STAT_SYNC_ROUNDS, STAT_SYNC_ITERS0, STAT_SYNC_ITERS1))
    return out.view.cpu().numpy().reshape(n, nblk, 64), st.cpu().tolist(), stats


def check_exact(ctx, scans, frame, want, what, rounds=DEFAULT_ROUNDS, guesses=DEFAULT_GUESSES):
    """the very coefficients; EAGAIN only from the enqueued rounds, and then the host loop (rounds = 0) must give them.
    -> (stats, statuses)"""
    got, st, stats = entropy(ctx, scans, frame, want[0].shape[0], rounds, guesses)
    for i, x in enumerate(st):
        assert x in ((0, EAGAIN) if rounds else (0,)), "%s image %d: status %d" % (what, i, x)
        if x == 0:
            nd = int((got[i] != want[i]).sum())
            assert nd == 0, "%s image %d: %d coefficients differ from those the segment was made from" % (what, i, nd)
    if EAGAIN in st:
        check_exact(ctx, scans, frame, want, what + " (host loop)", 0, guesses)
    return stats, st


SYNC_STATS = {}


@pytest.mark.gpu
@pytest.mark.parametrize("tfam", TABLE_FAMILIES)
def test_entropy_decode_returns_the_coefficients(ctx, streams, tfam):
    for s in streams:
        if s.tfam == tfam:
            stats, st = check_exact(ctx, s.scans, frame_for(s), s.coefs, s.name())
            SYNC_STATS.setdefault(tfam, []).append((s.cfam, s.layout, len(s.scans[0])) + stats + (EAGAIN in st,))
    for row in SYNC_STATS[tfam]:
        print("sync %-11s %-9s %-5s %8d bytes: rounds %d iters0 %d iters1 %d eagain %d" % ((tfam,) + row))


@pytest.fixture(scope="module")
def sync_streams(oracle):
    """per nb in {3, 4, 6}: dense and photographic content large enough for a few dozen CTAs"""
    return {(t, lay): Stream(t, cf, lay, 512, 256, nimg=2, oracle=oracle, seed=77)
            for t, cf in (("fixed8", "dense"), ("sparse", "photo"), ("chain16", "zrl"), ("eob1", "photo"), ("annexk", "dense"))
            for lay in ("444", "422", "420")}


@pytest.mark.gpu
@pytest.mark.parametrize("tfam", ["fixed8", "sparse", "chain16", "eob1", "annexk"])
def test_sync_options(ctx, sync_streams, tfam):
    """OPT_SYNC_ROUNDS 3, 1, 0 x OPT_SYNC_GUESSES 0, 1, 2 (the multi-guess first launch) on 3-, 4- and 6-block MCUs"""
    for lay in ("444", "422", "420"):
        s = sync_streams[(tfam, lay)]
        for rounds in (3, 1, 0):
            for guesses in (0, 1, 2):
                stats, st = check_exact(ctx, s.scans, frame_for(s), s.coefs, "%s rounds %d guesses %d" % (s.name(), rounds, guesses),
                                        rounds, guesses)
                print("sync options %-28s rounds %d guesses %d: stat rounds %d iters0 %d iters1 %d status %s" %
                      ((s.name(), rounds, guesses) + stats + (st,)))
                if tfam == "fixed8" and rounds == 3 and guesses == 0:
                    assert stats[0] > 1, "fixed-length codes did not need a repair launch (%s)" % (stats,)
                if tfam == "fixed8" and rounds == 1:
                    # dense content under fixed-length codes stays unsynchronised over whole CTAs: one repair launch is not
                    # enough, on every layout and with either first launch (deterministic: the streams are seeded)
                    assert st == [EAGAIN, EAGAIN], st


@pytest.mark.gpu
@pytest.mark.parametrize("tfam", TABLE_FAMILIES)
def test_restart_intervals(ctx, oracle, tfam):
    """k_decode_segments: R = 1, 7, and R >= nmcu, against the oracle's reading of the same file"""
    for ci, cf in enumerate(["dense", "zrl", "dc11"] if tfam != "optimised" else ["fibonacci"]):
        lay = LAYOUT_NAMES[(TABLE_FAMILIES.index(tfam) + ci) % 5] if tfam != "optimised" else "420"
        W, H = (200, 120) if tfam != "optimised" else B.fibonacci_coefs()[1:]
        nmcu = B.geometry(W, H, lay)[0]
        for R in (1, 7, nmcu, nmcu + 3):
            s = Stream(tfam, cf, lay, W, H, nimg=2, restart_interval=R, oracle=oracle, seed=R)
            assert (oracle_coefs(oracle, s.file(1)) == s.coefs[1]).all()
            got, st, _ = entropy(ctx, s.scans, frame_for(s), s.nblk)
            assert st == [0, 0], s.name()
            for i in range(2):
                assert (got[i] == s.coefs[i]).all(), s.name()


def check_pixels(got, want, what):
    for k, (a, w) in enumerate(zip(got, want)):
        a = a.cpu().numpy() if hasattr(a, "cpu") else a
        nd = int((a != w).sum())
        assert nd == 0, "%s: %d of %d samples of plane %d differ from the reference decoder" % (what, nd, w.size, k)


@pytest.mark.gpu
@pytest.mark.parametrize("tfam", TABLE_FAMILIES)
def test_fused_paths_match_oracle(ctx, oracle, streams, tfam):
    """jpezyb200_decode and decode_batch_dev2 give the oracle's pixels of the file (tables at ids 2 and 1); EAGAIN is legal from
    decode_batch_dev2 only, which has no host retry"""
    import torch
    from gpu_util import Guarded
    from jpezy_b200 import capi
    _, qy, qc, _, _ = oracle.tables()
    qt = np.stack([qy, qc]) // 4 + 1
    for s in streams:
        if s.tfam != tfam:
            continue
        frame = frame_for(s, ids=(2, 1), qt=qt)
        files = [s.file(i, ids=(2, 1), qt=qt) for i in range(len(s.scans))]
        want = [oracle.decode(f)[2:] for f in files]
        for i, f in enumerate(files):
            check_pixels(ctx.decode(s.scans[i], frame), want[i], "jpezyb200_decode %s image %d" % (s.name(), i))
        n = len(s.scans)
        d_scan, slot, nbytes = upload(s.scans)
        pl = capi.plane_bytes(frame)
        out = [Guarded(n * pl, torch.uint8, fill=0x3C) for _ in range(3)]
        st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        d_nb = torch.from_numpy(nbytes.astype(np.int64)).cuda()
        torch.cuda.synchronize()
        ctx.decode_batch_dev2(d_scan, slot, d_nb, int(nbytes.max()), n, frame, False, out[0].view, out[1].view, out[2].view, pl, st,
                              stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert all(o.intact() for o in out)
        for i, x in enumerate(st.cpu().tolist()):
            assert x in (0, EAGAIN), "decode_batch_dev2 %s image %d: status %d" % (s.name(), i, x)
            if x == 0:
                check_pixels([o.view[i * pl:(i + 1) * pl] for o in out], want[i], "decode_batch_dev2 %s image %d" % (s.name(), i))


@pytest.mark.gpu
def test_cli_decodes_adversarial_files(tmp_path, streams):
    """the host DHT parser: the CLI's PPM of an adversarial-table file equals that of the Annex K file"""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "jpezy_b200", "cli"), "-s"])
    picked = [s for s in streams if s.cfam in ("dense", "zrl", "ff_heavy", "fibonacci") and s.W * s.H > 64][:8]
    for j, s in enumerate(picked):
        outs = []
        for name, data in (("a", s.file(0, ids=(2, 0))), ("k", annexk_file(s))):
            (tmp_path / ("%d%s.jpg" % (j, name))).write_bytes(data)
            p = subprocess.run([DEC, str(tmp_path / ("%d%s.jpg" % (j, name))), str(tmp_path / ("%d%s.ppm" % (j, name)))], capture_output=True, text=True)
            assert p.returncode == 0, s.name() + p.stderr
            outs.append((tmp_path / ("%d%s.ppm" % (j, name))).read_bytes())
        assert outs[0] == outs[1], s.name()


@pytest.mark.gpu
def test_geometry(ctx, oracle):
    """one MCU; single frames (128-thread CTAs) and batches over 2 x #SM CTAs (256 threads); batches whose nimg x longest segment
    picks 128-, 256- and 512-bit subsequences (launch_entropy_decode); more than 8 images (sizes copied, not inline)"""
    for tfam in ("chain16", "fixed8", "all_slow"):
        s = Stream(tfam, "dense", "420", 16, 16, nimg=1, oracle=oracle)
        assert s.nblk == 6
        check_exact(ctx, s.scans, frame_for(s), s.coefs, "one MCU " + s.name())
    for tfam, cf, lay, (W, H), n, sub in (("fixed8", "dense", "420", (480, 320), 10, 256), ("chain16", "dense", "444", (480, 256), 10, 512),
                                          ("sparse", "dense", "422", (1920, 1088), 1, 512), ("eob1", "photo", "420", (640, 360), 12, 128)):
        s = Stream(tfam, cf, lay, W, H, nimg=n, oracle=oracle)
        big = n * max(len(x) for x in s.scans) * 8 // 131072
        assert (128 if big < 256 else 256 if big < 512 else 512) == sub, (s.name(), big)
        stats, st = check_exact(ctx, s.scans, frame_for(s), s.coefs, "%s x %d" % (s.name(), n))
        print("geometry %-32s x %2d, %d-bit subsequences: rounds %d iters0 %d iters1 %d status %s" % ((s.name(), n, sub) + stats + (st,)))


@pytest.mark.gpu
def test_adversarial_image_among_normal_ones(ctx, oracle):
    """a truncated segment among valid ones of the same batch: ECORRUPT for it, the very coefficients for the others"""
    s = Stream("fixed8", "photo", "444", 264, 136, nimg=4, oracle=oracle)
    scans = list(s.scans)
    scans[2] = scans[2][: len(scans[2]) // 2]
    for rounds in (3, 0):
        got, st, _ = entropy(ctx, scans, frame_for(s), s.nblk, rounds=rounds)
        assert st[2] == ECORRUPT or (rounds and st[2] == EAGAIN), st
        for i in (0, 1, 3):
            assert st[i] in ((0, EAGAIN) if rounds else (0,))
            if st[i] == 0:
                assert (got[i] == s.coefs[i]).all()


def corrupt_streams(oracle):
    """(Stream, malformed segments): cut in half, and a code word that no table holds (sparse tables: a run of 1 bits)"""
    out = []
    for tfam, lay, R in (("sparse", "420", 0), ("chain16", "444", 0), ("sparse", "gray1", 5), ("annexk", "422", 0)):
        s = Stream(tfam, "photo", lay, 264, 136, nimg=1, restart_interval=R, oracle=oracle)
        x = s.scans[0]
        bad = [x[: len(x) // 2]]
        if tfam == "sparse":
            k = len(x) // 3
            bad.append(x[:k] + b"\xfe" * 8 + x[k + 8:])
        out.append((s, bad))
    return out


@pytest.mark.gpu
def test_malformed_streams_are_corrupt(ctx, oracle, tmp_path):
    """every path reports ECORRUPT and never a wrong result"""
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi
    for s, bad in corrupt_streams(oracle):
        frame = frame_for(s)
        for j, x in enumerate(bad):
            what = "%s malformed %d" % (s.name(), j)
            for rounds in (3, 1, 0):
                _, st, _ = entropy(ctx, [x], frame, s.nblk, rounds=rounds)
                assert st[0] == ECORRUPT or (rounds and st[0] == EAGAIN), (what, rounds, st)
            with pytest.raises(J.JpezyError) as e:
                ctx.decode(x, frame)
            assert e.value.code == ECORRUPT, what
            d_scan, slot, nbytes = upload([x])
            pl = capi.plane_bytes(frame)
            out = [torch.zeros(pl, dtype=torch.uint8, device="cuda") for _ in range(3)]
            st = torch.full((1,), -1, dtype=torch.int32, device="cuda")
            d_nb = torch.from_numpy(nbytes.astype(np.int64)).cuda()
            torch.cuda.synchronize()
            ctx.decode_batch_dev2(d_scan, slot, d_nb, int(nbytes.max()), 1, frame, False, *out, pl, st,
                                  stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            assert st.item() in (ECORRUPT, EAGAIN), what
            path = tmp_path / "bad.jpg"
            path.write_bytes(B.jpeg_file(s.W, s.H, s.layout, x, s.tables, restart_interval=s.ri))
            p = subprocess.run([DEC, str(path), str(tmp_path / "bad.ppm")], capture_output=True, text=True)
            assert p.returncode == 1, what


@pytest.mark.gpu
def test_dc_symbol_above_15_is_refused(ctx, oracle, tmp_path):
    """a DC table holding a symbol above 15 is corrupt (huff_entry keeps 4 bits of it, the reference reads them all); categories
    12..15 stay decodable"""
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi
    s = Stream("annexk", "photo", "420", 200, 120, nimg=1, oracle=oracle)
    wide = dict(s.tables)
    wide[1] = (B.table([(k, 4) for k in range(12)] + [(k, 6) for k in (12, 13, 14, 15)]), s.tables[1][1])
    # a stream that uses categories 12..14 (differences 2048..16383) in the chroma DC
    c = s.coefs[0].copy()
    comp = np.tile([0, 0, 0, 0, 1, 2], c.shape[0] // 6)
    c[comp == 1, 0] = np.where(np.arange((comp == 1).sum()) % 2, 3000, -9000)
    s.tables, s.coefs, s.scans = wide, [c], [B.encode_scan(c, "420", wide)]
    assert (oracle_coefs(oracle, s.file()) == c).all()
    got, st, _ = entropy(ctx, s.scans, frame_for(s), s.nblk)
    assert st == [0] and (got[0] == c).all()
    bad = dict(wide)
    for sym in (16, 0x1B):
        bad[1] = (B.Huff(wide[1][0].bits, wide[1][0].vals[:-1] + [sym]), wide[1][1])
        s.tables = bad
        frame = frame_for(s)
        d_scan, slot, nbytes = upload(s.scans)
        pl = capi.plane_bytes(frame)
        out = [torch.zeros(pl, dtype=torch.uint8, device="cuda") for _ in range(3)]
        st = torch.zeros(1, dtype=torch.int32, device="cuda")
        d_nb = torch.from_numpy(nbytes.astype(np.int64)).cuda()
        calls = [lambda: ctx.decode(s.scans[0], frame),
                 lambda: ctx.entropy_decode_dev(d_scan, slot, nbytes, 1, frame, torch.zeros(s.nblk * 64, dtype=torch.int16, device="cuda"), st),
                 lambda: ctx.decode_batch_dev2(d_scan, slot, d_nb, int(nbytes.max()), 1, frame, False, *out, pl, st)]
        for call in calls:
            with pytest.raises(J.JpezyError) as e:
                call()
            assert e.value.code == ECORRUPT
        path = tmp_path / "dc16.jpg"
        path.write_bytes(s.file())
        p = subprocess.run([DEC, str(path), str(tmp_path / "dc16.ppm")], capture_output=True, text=True)
        assert p.returncode == 1

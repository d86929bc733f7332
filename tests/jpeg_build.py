"""Test-side baseline JPEG writer, independent of the device code and of the oracle: zig-zag coefficients in scan order ->
entropy-coded segment (any DHT tables, any of the device's layouts, optional restart intervals) and complete files.

Vectorised with numpy: the symbols of all blocks come from np.nonzero over the AC coefficients, every symbol and its value
field become one code word of at most 27 bits, and the words are packed at their cumulative bit offsets; no Python loop runs
per symbol, so a dense full-HD frame encodes in seconds.  Also home of the Python restatement of the optimised-table
construction (T.81 K.2) that tests/test_huffopt_gpu.py checks the device against."""
import numpy as np

# ---- tables ---------------------------------------------------------------------------------------------------------
class Huff:
    """BITS[16] + HUFFVAL of one DHT table (the attribute names of capi.Huff, so dht() takes either)"""
    def __init__(self, bits, vals):
        self.bits, self.vals = [int(b) for b in bits], [int(v) for v in vals]
        assert len(self.bits) == 16 and sum(self.bits) == len(self.vals) <= 256 and len(set(self.vals)) == len(self.vals)

    def lengths(self):
        """{symbol: code length}"""
        return dict(zip(self.vals, [L for L in range(1, 17) for _ in range(self.bits[L - 1])]))

    def kraft(self):
        """sum of 2^(16 - L) over the codes: below 65536 for a DHT that leaves the all-ones code word unused"""
        return sum(b << (16 - L) for L, b in zip(range(1, 17), self.bits))

    def codes(self):
        """(code[256], length[256]) of the canonical code (length 0: the symbol has none), T.81 C.1-C.2"""
        code, length = np.zeros(256, np.int64), np.zeros(256, np.int64)
        c, k = 0, 0
        for L in range(1, 17):
            for _ in range(self.bits[L - 1]):
                code[self.vals[k]], length[self.vals[k]] = c, L
                c, k = c + 1, k + 1
            c <<= 1
        return code, length


def table(pairs):
    """Huff from [(symbol, code length)]; codes are assigned in length order, ties in the order given"""
    pairs = sorted(pairs, key=lambda p: p[1])      # (stable)
    assert all(1 <= L <= 16 for _, L in pairs)
    h = Huff([sum(1 for _, L in pairs if L == n) for n in range(1, 17)], [s for s, _ in pairs])
    assert h.kraft() < 65536, "over-subscribed, or the all-ones code word is used"
    return h


_AC_Y = bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a"
    "434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9"
    "aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa")
_AC_C = bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a3536373839"
    "3a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7"
    "a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa")
# ITU-T T.81 tables K.3-K.6: [0 = DC, 1 = AC][0 = luma, 1 = chroma]
ANNEX_K = [[Huff([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], range(12)), Huff([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], range(12))],
           [Huff([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D], _AC_Y), Huff([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77], _AC_C)]]
AC_SYMBOLS = [0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]
DC_SYMBOLS = list(range(12))


def dht(tc_th, h, *more):
    """one DHT marker segment holding table h as Tc/Th = tc_th, followed by the further (tc_th, h) pairs in `more`"""
    body = b""
    for t, x in ((tc_th, h),) + tuple(more):
        n = sum(x.bits)
        body += bytes([t]) + bytes(x.bits) + bytes(x.vals[:n])
    return bytes([0xFF, 0xC4, (len(body) + 2) >> 8, (len(body) + 2) & 0xFF]) + body


# ---- layouts --------------------------------------------------------------------------------------------------------
LAYOUTS = {"420": ((2, 1, 1), (2, 1, 1)), "444": ((1, 1, 1), (1, 1, 1)), "422": ((2, 1, 1), (1, 1, 1)), "440": ((1, 1, 1), (2, 1, 1)),
           "gray1": ((1,), (1,))}


def geometry(W, H, layout):
    """-> (nmcu, blocks per MCU, component of every block position of the MCU)"""
    hs, vs = LAYOUTS[layout]
    hu, vu = -(-W // (8 * max(hs))), -(-H // (8 * max(vs)))
    comp = [c for c in range(len(hs)) for _ in range(hs[c] * vs[c])]
    return hu * vu, len(comp), comp


def bit_length(a):
    a = np.abs(np.asarray(a, dtype=np.int64))
    return sum((a >= (1 << i)).astype(np.int64) for i in range(16))


# ---- entropy coder --------------------------------------------------------------------------------------------------
def encode_scan(coefs, layout, tables, restart_interval=0):
    """coefs: int [nblk, 64] zig-zag, scan order, absolute DC; tables: {class: (DC Huff, AC Huff)}, class 0 = component 0,
    class 1 = the others.  -> the stuffed segment: 1-bit padding at the end of every restart interval, RSTn markers between them.
    A symbol without a code raises."""
    hs, vs = LAYOUTS[layout]
    c = np.asarray(coefs, dtype=np.int64).reshape(-1, 64)
    nb = sum(h * v for h, v in zip(hs, vs))
    nblk = c.shape[0]
    assert nblk % nb == 0
    comp = np.tile(np.array([k for k in range(len(hs)) for _ in range(hs[k] * vs[k])]), nblk // nb)
    cls = (comp > 0).astype(np.int64)
    seg = (np.arange(nblk) // nb) // restart_interval if restart_interval else np.zeros(nblk, np.int64)
    codes = [[tables[k][t].codes() for k in (0, 1)] for t in (0, 1)]    # [DC/AC][class] -> (code, length)

    def word(t, sym, k):
        code = np.where(k == 0, codes[t][0][0][sym], codes[t][1][0][sym])
        ln = np.where(k == 0, codes[t][0][1][sym], codes[t][1][1][sym])
        if (ln == 0).any():
            raise ValueError("symbol %#x has no code in the %s table" % (int(sym[ln == 0][0]), "DC" if t == 0 else "AC"))
        return code, ln

    # DC differences per component, the predictor reset at every restart
    diff = np.zeros(nblk, np.int64)
    for k in range(len(hs)):
        i = np.nonzero(comp == k)[0]
        d = c[i, 0].copy()
        same = seg[i][1:] == seg[i][:-1]
        d[1:] -= np.where(same, c[i[:-1], 0], 0)
        diff[i] = d
    cat = bit_length(diff)
    assert cat.max(initial=0) <= 15, "DC difference beyond the 15 bits of a DC category"
    items = []                                  # (block, order inside the block, code word, its length)

    def add(blk, order, code, ln, val, size):
        vbits = np.where(val < 0, val - 1, val) & ((np.int64(1) << size) - 1)
        items.append((blk, order, (code << size) | vbits, ln + size))

    code, ln = word(0, cat, cls)
    add(np.arange(nblk), np.zeros(nblk, np.int64), code, ln, diff, cat)
    ac = c[:, 1:]
    assert np.abs(ac).max(initial=0) <= 1023, "AC value beyond 1023"
    bi, pos = np.nonzero(ac)
    prev = np.full(pos.shape, -1, np.int64)
    prev[1:] = np.where(bi[1:] == bi[:-1], pos[:-1], -1)
    run = pos - prev - 1
    size = bit_length(ac[bi, pos])
    nzrl = run // 16
    if nzrl.any():                              # ZRL codes in front of the coefficient
        zb = np.repeat(bi, nzrl)
        zo = np.repeat(2 * pos, nzrl)
        code, ln = word(1, np.full(zb.shape, 0xF0), cls[zb])
        add(zb, zo, code, ln, np.zeros_like(zb), np.zeros_like(zb))
    code, ln = word(1, ((run % 16) << 4) | size, cls[bi])
    add(bi, 2 * pos + 1, code, ln, ac[bi, pos], size)
    eb = np.nonzero(ac[:, 62] == 0)[0]          # end of block unless coefficient 63 is coded
    code, ln = word(1, np.zeros(eb.shape, np.int64), cls[eb])
    add(eb, np.full(eb.shape, 200), code, ln, np.zeros_like(eb), np.zeros_like(eb))
    blk, order, w, L = (np.concatenate(x) for x in zip(*items))
    s = seg[blk]
    nseg = int(seg[-1]) + 1
    # 1-bit padding to the byte at the end of every interval
    seg_bits = np.bincount(s, weights=L, minlength=nseg).astype(np.int64)
    pad = (-seg_bits) % 8
    last = np.searchsorted(seg, np.arange(nseg), side="right") - 1
    blk = np.concatenate([blk, last])
    order = np.concatenate([order, np.full(nseg, 255)])
    w = np.concatenate([w, (np.int64(1) << pad) - 1])
    L = np.concatenate([L, pad])
    o = np.lexsort((order, blk))
    w, L = w[o], L[o]
    off = np.concatenate([[0], np.cumsum(L)[:-1]])
    nbytes = int(L.sum()) // 8
    # pack: a word of <= 27 bits at bit offset off lies in the 5 bytes from off // 8; no two words share a bit, so OR == sum
    v = w << (40 - (off & 7) - L)
    idx = np.concatenate([(off >> 3) + k for k in range(5)])
    val = np.concatenate([(v >> (32 - 8 * k)) & 0xFF for k in range(5)])
    raw = np.bincount(idx, weights=val, minlength=nbytes + 5)[:nbytes].astype(np.uint8)
    # stuffing (00 after every FF) and the markers between the intervals (FF D0 + (k mod 8) in front of interval k + 1)
    seg_end = np.cumsum(seg_bits + pad) // 8                # raw byte at which every interval ends
    ff = raw == 0xFF
    before = np.zeros(nbytes, np.int64)                     # markers in front of every raw byte
    if nseg > 1:
        np.add.at(before, seg_end[:-1], 1)
        before = np.cumsum(before)
    dst = np.arange(nbytes) + np.concatenate([[0], np.cumsum(ff)[:-1]]) + 2 * before
    out = np.zeros(nbytes + int(ff.sum()) + 2 * (nseg - 1), np.uint8)
    out[dst] = raw
    if nseg > 1:
        mpos = seg_end[:-1] + np.concatenate([[0], np.cumsum(ff)])[seg_end[:-1]] + 2 * np.arange(nseg - 1)
        out[mpos] = 0xFF
        out[mpos + 1] = 0xD0 + (np.arange(nseg - 1) & 7)
    return out.tobytes()


def jpeg_file(W, H, layout, scan, tables, ids=(0, 1), qt=None, restart_interval=0, extra=(), dht_per_table=False):
    """SOI, DQT, SOF0, DHT, [DRI], SOS, segment, EOI.  ids: DHT table ids of class 0 and class 1 (the SOS selects the same id
    for the DC and the AC table of a component); extra: further (Tc/Th, Huff) pairs written to the DHT; dht_per_table: one
    DHT segment per table instead of one for all; qt: one natural-order 8-bit table per class (default: all 1)."""
    hs, vs = LAYOUTS[layout]
    qt = np.ones((2, 64), np.int64) if qt is None else np.asarray(qt)
    from_nat = _zigzag()
    f = bytearray(b"\xFF\xD8")
    f += bytes([0xFF, 0xDB, 0, 132]) + bytes([0]) + bytes(int(qt[0][k]) for k in from_nat) + bytes([1]) + bytes(int(qt[1][k]) for k in from_nat)
    f += bytes([0xFF, 0xC0, 0, 8 + 3 * len(hs), 8, H >> 8, H & 255, W >> 8, W & 255, len(hs)])
    for k in range(len(hs)):
        f += bytes([k + 1, (hs[k] << 4) | vs[k], min(k, 1)])
    pairs = [(ids[k], tables[k][t], t) for k in (0, 1) for t in (0, 1)][: 4 if len(hs) > 1 else 2]
    pairs = [((t << 4) | i, h) for i, h, t in pairs] + list(extra)
    f += b"".join(dht(*p) for p in pairs) if dht_per_table else dht(*pairs[0], *pairs[1:])
    if restart_interval:
        f += bytes([0xFF, 0xDD, 0, 4, restart_interval >> 8, restart_interval & 255])
    f += bytes([0xFF, 0xDA, 0, 6 + 2 * len(hs), len(hs)])
    for k in range(len(hs)):
        i = ids[min(k, 1)]
        f += bytes([k + 1, (i << 4) | i])
    f += bytes([0, 63, 0])
    return bytes(f) + scan + b"\xFF\xD9"


def _zigzag():
    """natural index of every zig-zag position"""
    zz = sorted(((x + y, y if (x + y) % 2 else -y, y * 8 + x) for y in range(8) for x in range(8)))
    return [n for _, _, n in zz]


# ---- optimised tables (T.81 K.2) -------------------------------------------------------------------------------------
def symbol_hist(coefs):
    """[2 classes][16 DC categories + 256 AC symbols] counts of the symbols the encoder emits for zig-zag coefficients
    [nmcu, 6, 64] (categories and sizes clamped to 11 and 10 as the encoder clamps them), and the magnitude bits"""
    c = np.asarray(coefs, dtype=np.int64).reshape(-1, 6, 64)
    hist = np.zeros((2, 272), np.int64)
    extra = 0
    dc = c[:, :, 0]
    for cls, seq in ((0, dc[:, :4].reshape(-1)), (1, dc[:, 4]), (1, dc[:, 5])):
        cat = np.minimum(bit_length(np.diff(seq, prepend=0)), 11)
        hist[cls, :16] += np.bincount(cat, minlength=16)
        extra += int(cat.sum())
    ac = c[:, :, 1:].reshape(-1, 63)
    blk_cls = np.tile((np.arange(6) >= 4).astype(np.int64), c.shape[0])
    bi, pos = np.nonzero(ac)
    prev = np.full(pos.shape, -1, np.int64)
    prev[1:] = np.where(bi[1:] == bi[:-1], pos[:-1], -1)
    run = pos - prev - 1
    size = np.minimum(bit_length(ac[bi, pos]), 10)
    cls = blk_cls[bi]
    for k in (0, 1):
        m = cls == k
        hist[k, 16 + 0xF0] += int((run[m] // 16).sum())
        hist[k, 16:] += np.bincount(((run[m] % 16) << 4) | size[m], minlength=256)
        hist[k, 16 + 0x00] += int(((ac[:, 62] == 0) & (blk_cls == k)).sum())
    extra += int(size.sum())
    return hist, extra


def gen_optimal_table(counts):
    """T.81 K.2 (Figures K.1-K.4) line for line after libjpeg's jpeg_gen_optimal_table -> (BITS[16], HUFFVAL, codesize)"""
    MAX_CLEN = 32
    freq = [int(x) for x in counts] + [0] * (257 - len(counts))
    bits = [0] * (MAX_CLEN + 1)
    codesize = [0] * 257
    others = [-1] * 257
    freq[256] = 1
    while True:
        c1, v = -1, 1 << 62
        for i in range(257):
            if freq[i] and freq[i] <= v:
                v, c1 = freq[i], i
        c2, v = -1, 1 << 62
        for i in range(257):
            if freq[i] and freq[i] <= v and i != c1:
                v, c2 = freq[i], i
        if c2 < 0:
            break
        freq[c1] += freq[c2]
        freq[c2] = 0
        codesize[c1] += 1
        while others[c1] >= 0:
            c1 = others[c1]
            codesize[c1] += 1
        others[c1] = c2
        codesize[c2] += 1
        while others[c2] >= 0:
            c2 = others[c2]
            codesize[c2] += 1
    for i in range(257):
        if codesize[i]:
            assert codesize[i] <= MAX_CLEN
            bits[codesize[i]] += 1
    i = MAX_CLEN
    while i > 16:
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
        i -= 1
    while bits[i] == 0:
        i -= 1
    bits[i] -= 1
    huffval = [j for i in range(1, MAX_CLEN + 1) for j in range(256) if codesize[j] == i]
    return bits[1:17], huffval, codesize


def fibonacci_coefs():
    """luma AC symbols (run, size), run 0..1 and size 1..10, counted 1, 1, 3, 5, 9, 15, ... (f[k] = f[k-1] + f[k-2] + 1,
    20 symbols: with the plain Fibonacci counts the tie rule balances the tree); one symbol per luma block, so EOB (one per
    block) outweighs them all and the unconstrained code is a chain of depth 21.  -> (coefficients [nmcu, 6, 64], W, H)"""
    syms = [(r, s) for r in (0, 1) for s in range(1, 11)]
    fib = [1, 1]
    while len(fib) < len(syms):
        fib.append(fib[-1] + fib[-2] + 1)
    seq = [sym for sym, f in zip(syms, fib) for _ in range(f)]
    np.random.default_rng(7).shuffle(seq)
    HU = 64
    VU = -(-len(seq) // (4 * HU))
    coefs = np.zeros((HU * VU, 6, 64), np.int16)
    for k, (run, s) in enumerate(seq):
        coefs[k // 4, k % 4, run + 1] = (1 << (s - 1)) * (1 if k % 2 else -1)
    return coefs, HU * 16, VU * 16

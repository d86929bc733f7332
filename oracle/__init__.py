"""ctypes binding of the CPU oracle (oracle/jpezy_oracle.cpp).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under jpezy_b200/ imports this package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_u8p = C.POINTER(C.c_uint8)
_i16p = C.POINTER(C.c_int16)
_i32p = C.POINTER(C.c_int32)


def build(force=False):
    """Compile liboracle.so / liboracle_shipped.so (and oracle/_ref when /root/reference exists)."""
    so = os.path.join(_HERE, "liboracle.so")
    src = os.path.join(_HERE, "jpezy_oracle.cpp")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "all"])
    return so


def ref_dir():
    """oracle/_ref: the reference's own sources compiled against oracle/shim (None when it was never built)."""
    d = os.path.join(_HERE, "_ref")
    return d if os.path.exists(os.path.join(d, "libjpezy_ref.so")) else None


class Reference:
    """The reference's own encoder / decoder classes (oracle/ref_driver.cpp).  File based, like the reference."""

    def __init__(self):
        d = ref_dir()
        if d is None:
            raise RuntimeError("oracle/_ref is not built (needs /root/reference: `make -C oracle ref`)")
        L = self.lib = C.CDLL(os.path.join(d, "libjpezy_ref.so"))
        L.ref_encode_file.restype = C.c_longlong
        L.ref_encode_file.argtypes = [_u8p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_char_p]
        L.ref_constants.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double)]
        self.encode_exe = os.path.join(d, "jpezy_encode")
        self.decode_exe = os.path.join(d, "jpezy_decode")
        self.tool = os.path.join(d, "ref_tool")

    def encode(self, r, g, b, W, H, gray=False, path=None):
        """-> (file bytes, wrote_size()) of jpezy::encoder(...).encode<MODE>(path)"""
        import tempfile
        r, g, b = (np.ascontiguousarray(x, dtype=np.uint8).reshape(-1) for x in (r, g, b))
        with tempfile.TemporaryDirectory() as tmp:
            p = path or os.path.join(tmp, "ref.jpg")
            n = self.lib.ref_encode_file(_ptr(r), _ptr(g), _ptr(b), W, H, int(gray), p.encode())
            if n < 0:
                raise RuntimeError("reference encoder threw")
            return open(p, "rb").read(), int(n)

    def decode(self, data, gray=False):
        """-> (W, H, r, g, b) of jpezy::decoder<Release>(file).decode<MODE>(); None when decode() returns an empty optional.
        Runs in a process of its own (oracle/_ref/ref_tool): the reference's analyze_dht reads one element past a vector
        (src/decoder/jpezy_decoder.hpp:231), harmless in a fresh process, heap-corrupting inside a long-lived one."""
        import tempfile
        with tempfile.TemporaryDirectory() as tmp:
            p, out = os.path.join(tmp, "ref.jpg"), os.path.join(tmp, "ref.bin")
            open(p, "wb").write(data)
            rc = subprocess.run([self.tool, "decode", p, str(int(gray)), out], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL).returncode
            if rc:
                return None
            raw = np.fromfile(out, dtype=np.uint8)
            W, H = (int(x) for x in raw[:8].view(np.int32))
            pl = int(raw[8:16].view(np.uint64)[0])
            r, g, b = (raw[16 + k * pl: 16 + (k + 1) * pl].copy() for k in range(3))
            return W, H, r, g, b

    def time_roundtrip(self, r, g, b, W, H, gray=False, reps=1, nprocs=1):
        """nprocs concurrent instances of `ref_tool bench` (one per core), each `reps` x (encode() + decode()) of the image.
        -> (wall seconds of the slowest instance's timed region, mean encode seconds, mean decode seconds) per instance"""
        import tempfile
        r, g, b = (np.ascontiguousarray(x, dtype=np.uint8).reshape(-1) for x in (r, g, b))
        tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            src = os.path.join(tmp, "in.rgb")
            np.concatenate([r, g, b]).tofile(src)
            ps = [subprocess.Popen([self.tool, "bench", src, str(W), str(H), str(int(gray)), str(reps), os.path.join(tmp, "s%d.jpg" % i)],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL) for i in range(nprocs)]
            outs = [p.communicate()[0].split() for p in ps]
            if any(p.returncode for p in ps):
                raise RuntimeError("ref_tool bench failed")
            te = [float(o[0]) for o in outs]
            td = [float(o[1]) for o in outs]
            return max(a + c for a, c in zip(te, td)), sum(te) / nprocs, sum(td) / nprocs
        finally:
            import shutil
            shutil.rmtree(tmp, ignore_errors=True)

    def constants(self):
        cos = np.zeros(64, np.float64)
        ds = C.c_double(0)
        self.lib.ref_constants(_ptr(cos, C.POINTER(C.c_double)), C.byref(ds))
        return cos, ds.value


def _ptr(a, t=_u8p):
    return a.ctypes.data_as(t)


class Oracle:
    def __init__(self, variant="canonical"):
        name = {"canonical": "liboracle.so", "shipped": "liboracle_shipped.so"}[variant]
        path = os.path.join(_HERE, name)
        if not os.path.exists(path):
            build()
        L = self.lib = C.CDLL(path)
        L.orc_num_mcus.restype = C.c_size_t
        L.orc_num_mcus.argtypes = [C.c_int, C.c_int]
        L.orc_coefs.argtypes = [_u8p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, _i16p, C.POINTER(C.c_double)]
        L.orc_encode.argtypes = [_u8p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_size_t,
                                 C.POINTER(C.c_size_t)]
        L.orc_header.argtypes = [C.c_int, C.c_int, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.orc_scan_from_coefs.argtypes = [_i16p, C.c_size_t, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_size_t),
                                          C.POINTER(C.c_uint64)]
        L.orc_scan_from_coefs32.argtypes = [_i32p, C.c_size_t, C.c_int, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_size_t),
                                            C.POINTER(C.c_uint64)]
        L.orc_probe.argtypes = [_u8p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t), _i32p, _i32p,
                                _i32p, C.POINTER(C.c_size_t)]
        L.orc_pixels_from_coefs.argtypes = [_i32p, C.c_size_t, C.c_int, C.c_int, C.c_int, _i32p, _i32p, C.POINTER(C.c_uint16),
                                            C.c_int, _u8p, _u8p, _u8p, C.c_size_t]
        L.orc_decode.argtypes = [_u8p, C.c_size_t, C.c_int, _u8p, _u8p, _u8p, C.c_size_t]
        L.orc_decode_coefs.argtypes = [_u8p, C.c_size_t, _i16p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.orc_enc_lut.argtypes = [C.c_int] + [C.POINTER(C.c_int)] * 4
        L.orc_tables.argtypes = [C.POINTER(C.c_int)] * 3 + [C.POINTER(C.c_double)] * 2
        L.orc_time_roundtrip.restype = C.c_double
        L.orc_time_roundtrip.argtypes = [_u8p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_double), C.POINTER(C.c_double)]

    # ---- encoder side -------------------------------------------------------------------------
    def num_mcus(self, W, H):
        return int(self.lib.orc_num_mcus(W, H))

    @staticmethod
    def _planes(r, g, b):
        r, g, b = (np.ascontiguousarray(x, dtype=np.uint8).reshape(-1) for x in (r, g, b))
        return r, g, b

    def coefs(self, r, g, b, W, H, gray=False, want_raw=False):
        """-> int16 [nmcu, 6, 64] zig-zag quantised coefficients (+ float64 [nmcu,6,64] raw DCT, natural order)."""
        r, g, b = self._planes(r, g, b)
        n = self.num_mcus(W, H)
        out = np.zeros((n, 6, 64), dtype=np.int16)
        raw = np.zeros((n, 6, 64), dtype=np.float64) if want_raw else None
        rc = self.lib.orc_coefs(_ptr(r), _ptr(g), _ptr(b), W, H, int(gray), _ptr(out, _i16p),
                                _ptr(raw, C.POINTER(C.c_double)) if want_raw else None)
        if rc:
            raise RuntimeError("orc_coefs failed")
        return (out, raw) if want_raw else out

    def encode(self, r, g, b, W, H, gray=False, pad_ones=True, scan_only=False):
        """-> bytes of the complete JPEG file (or only the stuffed, padded entropy segment)."""
        r, g, b = self._planes(r, g, b)
        cap = max(W * H * 3, 10240) + 1024
        out = np.zeros(cap, dtype=np.uint8)
        n = C.c_size_t(0)
        rc = self.lib.orc_encode(_ptr(r), _ptr(g), _ptr(b), W, H, int(gray), int(pad_ones), int(scan_only), _ptr(out), cap,
                                 C.byref(n))
        if rc:
            raise RuntimeError("orc_encode failed (buffer overflow as in the reference?)")
        return out[: n.value].tobytes()

    def header(self, W, H, gray=False):
        out = np.zeros(4096, dtype=np.uint8)
        n = C.c_size_t(0)
        if self.lib.orc_header(W, H, int(gray), _ptr(out), 4096, C.byref(n)):
            raise RuntimeError("orc_header failed")
        return out[: n.value].tobytes()

    def scan_from_coefs(self, coefs, pad_ones=True, restart_interval=0):
        """4:2:0 coefficients (zig-zag, scan order; int32, so a DC may walk past the int16 range) -> entropy-coded segment,
        with RSTn markers every restart_interval MCUs when it is > 0."""
        coefs = np.ascontiguousarray(coefs, dtype=np.int32).reshape(-1, 6, 64)
        cap = coefs.size * 4 + coefs.shape[0] * 2 + 1024
        out = np.zeros(cap, dtype=np.uint8)
        n = C.c_size_t(0)
        nb = C.c_uint64(0)
        rc = self.lib.orc_scan_from_coefs32(_ptr(coefs, _i32p), coefs.shape[0], int(pad_ones), int(restart_interval), _ptr(out), cap,
                                            C.byref(n), C.byref(nb))
        if rc:
            raise RuntimeError("orc_scan_from_coefs32 failed")
        return out[: n.value].tobytes()

    # ---- decoder side -------------------------------------------------------------------------
    def probe(self, data):
        return self.layout(data)[:3]

    def layout(self, data):
        """-> (W, H, plane_len, ncomp, hs, vs, nblocks) from the file's frame header"""
        a = np.frombuffer(data, dtype=np.uint8)
        W, H, pl, nb = C.c_int(0), C.c_int(0), C.c_size_t(0), C.c_size_t(0)
        nc, hs, vs = np.zeros(1, np.int32), np.zeros(3, np.int32), np.zeros(3, np.int32)
        if self.lib.orc_probe(_ptr(a), a.size, C.byref(W), C.byref(H), C.byref(pl), _ptr(nc, _i32p), _ptr(hs, _i32p), _ptr(vs, _i32p),
                              C.byref(nb)):
            raise RuntimeError("orc_probe failed")
        n = int(nc[0])
        return W.value, H.value, pl.value, n, tuple(int(x) for x in hs[:n]), tuple(int(x) for x in vs[:n]), nb.value

    def decode(self, data, gray=False):
        """-> (W, H, r, g, b) with planes of the reference's padded length (stride W)."""
        a = np.frombuffer(data, dtype=np.uint8)
        W, H, pl = self.probe(data)
        r, g, b = (np.zeros(pl, dtype=np.uint8) for _ in range(3))
        rc = self.lib.orc_decode(_ptr(a), a.size, int(gray), _ptr(r), _ptr(g), _ptr(b), pl)
        if rc:
            raise RuntimeError("orc_decode failed rc=%d" % rc)
        return W, H, r, g, b

    def decode_coefs(self, data):
        """-> int16 zig-zag coefficients in scan order, absolute DC: [nmcu, 6, 64] for 4:2:0 frames, flat for the other layouts."""
        a = np.frombuffer(data, dtype=np.uint8)
        _, _, _, nc, hs, vs, nblk = self.layout(data)
        cap = nblk * 64
        out = np.zeros(cap, dtype=np.int16)
        n = C.c_size_t(0)
        rc = self.lib.orc_decode_coefs(_ptr(a), a.size, _ptr(out, _i16p), cap, C.byref(n))
        if rc:
            raise RuntimeError("orc_decode_coefs failed rc=%d" % rc)
        out = out[: n.value]
        return out.reshape(-1, 6, 64) if (nc, hs, vs) == (3, (2, 1, 1), (2, 1, 1)) else out

    def pixels_from_coefs(self, coefs, W, H, qt, ncomp=3, hs=(2, 1, 1), vs=(2, 1, 1), gray=False):
        """The reference decoder's pixel stage (dequant, idct, replication, make_rgb) on given coefficients: zig-zag, scan order,
        absolute DC (int32, so DC values beyond int16 can be expressed); qt: one natural-order table per component (16 bit).
        -> (r, g, b) planes of the reference's padded length (stride W)."""
        c = np.ascontiguousarray(coefs, dtype=np.int32).reshape(-1)
        q = np.ascontiguousarray(qt, dtype=np.uint16).reshape(ncomp, 64)
        hs_a, vs_a = np.array(hs[:ncomp], np.int32), np.array(vs[:ncomp], np.int32)
        hmax, vmax = int(hs_a.max()), int(vs_a.max())
        hb, vb = (W + 7) // 8, (H + 7) // 8
        pl = ((vb + vmax - 1) // vmax) * vmax * 8 * ((hb + hmax - 1) // hmax) * hmax * 8
        r, g, b = (np.zeros(pl, dtype=np.uint8) for _ in range(3))
        rc = self.lib.orc_pixels_from_coefs(_ptr(c, _i32p), c.size, W, H, ncomp, _ptr(hs_a, _i32p), _ptr(vs_a, _i32p),
                                            _ptr(q, C.POINTER(C.c_uint16)), int(gray), _ptr(r), _ptr(g), _ptr(b), pl)
        if rc:
            raise RuntimeError("orc_pixels_from_coefs failed rc=%d" % rc)
        return r, g, b

    # ---- tables -------------------------------------------------------------------------------
    def enc_lut(self, chroma):
        arrs = [np.zeros(12, np.int32), np.zeros(12, np.int32), np.zeros(162, np.int32), np.zeros(162, np.int32)]
        self.lib.orc_enc_lut(int(chroma), *[_ptr(a, C.POINTER(C.c_int)) for a in arrs])
        return arrs

    def tables(self):
        zz, qy, qc = (np.zeros(64, np.int32) for _ in range(3))
        cos = np.zeros(64, np.float64)
        ds = C.c_double(0)
        self.lib.orc_tables(*[_ptr(a, C.POINTER(C.c_int)) for a in (zz, qy, qc)], _ptr(cos, C.POINTER(C.c_double)),
                            C.byref(ds))
        return zz, qy, qc, cos, ds.value

    # ---- timing -------------------------------------------------------------------------------
    def time_roundtrip(self, r, g, b, W, H, gray=False, reps=1, nthreads=1):
        r, g, b = self._planes(r, g, b)
        te, td = C.c_double(0), C.c_double(0)
        wall = self.lib.orc_time_roundtrip(_ptr(r), _ptr(g), _ptr(b), W, H, int(gray), reps, nthreads, C.byref(te),
                                           C.byref(td))
        return wall, te.value, td.value

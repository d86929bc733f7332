"""ctypes view of include/jpezy_b200.h."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

OK, EINVAL, ECAPACITY, ECUDA, ENCCL, ECORRUPT, ENODEVICE, ENOMEM, EUNSUPPORTED, EAGAIN = range(10)
OPT_PAD_ONES, OPT_TRANSFORM, OPT_SYNC_ROUNDS, OPT_BATCH_GROUP_BYTES, OPT_SHARD_SCRATCH_BYTES, OPT_SYNC_GUESSES = 1, 2, 3, 4, 5, 6
OPT_RESTART_INTERVAL = 7   # MCUs per restart interval of the encoders (0 = none); decode with Frame.restart_interval
STAT_KERNEL_LAUNCHES, STAT_GUARD_FWD, STAT_GUARD_INV, STAT_SYNC_ROUNDS, STAT_SYNC_ITERS0, STAT_SYNC_ITERS1 = 1, 2, 3, 4, 5, 6

EXPORTS = [
    "jpezyb200_abi_version", "jpezyb200_ctx_create", "jpezyb200_ctx_destroy", "jpezyb200_strerror", "jpezyb200_last_error",
    "jpezyb200_set_option", "jpezyb200_get_stat", "jpezyb200_encode", "jpezyb200_encode_batch_dev",
    "jpezyb200_transform_fwd_dev", "jpezyb200_entropy_encode_dev", "jpezyb200_plane_bytes", "jpezyb200_default_frame",
    "jpezyb200_decode", "jpezyb200_decode_batch_dev", "jpezyb200_decode_batch_dev2", "jpezyb200_entropy_decode_dev", "jpezyb200_transform_inv_dev",
    "jpezyb200_synth_dev", "jpezyb200_synth_rows_dev", "jpezyb200_shard_encode_a", "jpezyb200_shard_encode_b",
    "jpezyb200_shard_encode_c", "jpezyb200_shard_encode_d", "jpezyb200_ipc_alloc", "jpezyb200_ipc_open", "jpezyb200_ipc_close",
    "jpezyb200_ipc_free", "jpezyb200_shard_decode_dev", "jpezyb200_encode_batch", "jpezyb200_decode_batch", "jpezyb200_read_sizes",
    "jpezyb200_group_create", "jpezyb200_group_destroy", "jpezyb200_group_size", "jpezyb200_group_last_error", "jpezyb200_group_ctx",
    "jpezyb200_group_partition", "jpezyb200_group_encode", "jpezyb200_encode_optimized", "jpezyb200_encode_batch_optimized_dev",
    "jpezyb200_entropy_encode_optimized_dev",
]


class JpezyError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("jpezy_b200 error %d: %s" % (code, msg))
        self.code = code


class Huff(C.Structure):
    _fields_ = [("present", C.c_uint8), ("bits", C.c_uint8 * 16), ("vals", C.c_uint8 * 256)]


HuffTables = (Huff * 2) * 2   # [class 0=DC,1=AC][0=luma, 1=chroma], as the optimised encoders write them
HUFF_TABLES_BYTES = C.sizeof(HuffTables)


class Frame(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("sample_precision", C.c_uint8), ("ncomp", C.c_uint8),
                ("hs", C.c_uint8 * 3), ("vs", C.c_uint8 * 3), ("tq", C.c_uint8 * 3), ("td", C.c_uint8 * 3),
                ("ta", C.c_uint8 * 3), ("restart_interval", C.c_uint16), ("qt", (C.c_uint16 * 64) * 4),
                ("ht", (Huff * 4) * 2)]


def library_path():
    return os.path.join(_HERE, "libjpezy_b200.so")


def build_library(force=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> jpezy_b200/libjpezy_b200.so (in-tree)."""
    args = ["make", "-C", os.path.join(_HERE, "csrc"), "-s"]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return library_path()


def load_library():
    """Load libjpezy_b200.so; raises (never falls back) when it is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise JpezyError(ENODEVICE, "%s not built: run __graft_entry__.build() (there is no CPU fallback)" % path)
    L = C.CDLL(path)
    vp, u8p, i16p, u64p, u32, sz = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_size_t
    L.jpezyb200_abi_version.restype = C.c_int
    L.jpezyb200_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.jpezyb200_ctx_destroy.argtypes = [vp]
    L.jpezyb200_ctx_destroy.restype = None
    L.jpezyb200_strerror.argtypes = [C.c_int]
    L.jpezyb200_strerror.restype = C.c_char_p
    L.jpezyb200_last_error.argtypes = [vp]
    L.jpezyb200_last_error.restype = C.c_char_p
    L.jpezyb200_set_option.argtypes = [vp, C.c_int, C.c_int64]
    L.jpezyb200_get_stat.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64)]
    L.jpezyb200_encode.argtypes = [vp, u8p, u8p, u8p, u32, u32, C.c_int, u8p, sz, C.POINTER(sz), C.POINTER(C.c_uint64)]
    L.jpezyb200_encode_batch_dev.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, C.c_int, u8p, sz, u64p, u64p, vp]
    L.jpezyb200_encode_optimized.argtypes = [vp, u8p, u8p, u8p, u32, u32, C.c_int, u8p, sz, C.POINTER(sz), C.POINTER(C.c_uint64),
                                             C.POINTER(HuffTables)]
    L.jpezyb200_encode_batch_optimized_dev.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, C.c_int, u8p, sz, u64p, u64p, vp, vp]
    L.jpezyb200_entropy_encode_optimized_dev.argtypes = [vp, i16p, u32, u32, u32, C.c_int, u8p, sz, u64p, u64p, vp, vp]
    L.jpezyb200_transform_fwd_dev.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, C.c_int, i16p, vp]
    L.jpezyb200_read_sizes.argtypes = [vp, u64p, u32, u64p, vp]
    L.jpezyb200_entropy_encode_dev.argtypes = [vp, i16p, u32, u32, u32, C.c_int, u8p, sz, u64p, u64p, vp]
    L.jpezyb200_plane_bytes.argtypes = [C.POINTER(Frame)]
    L.jpezyb200_plane_bytes.restype = sz
    L.jpezyb200_default_frame.argtypes = [u32, u32, C.POINTER(Frame)]
    L.jpezyb200_decode.argtypes = [vp, u8p, sz, C.POINTER(Frame), C.c_int, u8p, u8p, u8p, sz]
    L.jpezyb200_decode_batch_dev.argtypes = [vp, u8p, sz, u64p, u32, C.POINTER(Frame), C.c_int, u8p, u8p, u8p, sz, vp, vp]
    L.jpezyb200_decode_batch_dev2.argtypes = [vp, u8p, sz, vp, C.c_uint64, u32, C.POINTER(Frame), C.c_int, u8p, u8p, u8p, sz, vp, vp]
    L.jpezyb200_entropy_decode_dev.argtypes = [vp, u8p, sz, u64p, u32, C.POINTER(Frame), i16p, vp, vp]
    L.jpezyb200_transform_inv_dev.argtypes = [vp, i16p, C.POINTER(Frame), u32, C.c_int, u8p, u8p, u8p, sz, vp]
    L.jpezyb200_synth_dev.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, u32, C.c_int, vp]
    L.jpezyb200_synth_rows_dev.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, u32, C.c_int, vp]
    L.jpezyb200_shard_encode_a.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, u32, u32, C.c_int, vp, vp]
    L.jpezyb200_shard_encode_b.argtypes = [vp, vp, vp, vp]
    L.jpezyb200_shard_encode_c.argtypes = [vp, vp, u32, u32, vp, vp]
    L.jpezyb200_shard_encode_d.argtypes = [vp, vp, u8p, sz, vp, vp, vp]
    L.jpezyb200_shard_decode_dev.argtypes = [vp, u8p, sz, C.POINTER(Frame), C.c_int, u32, u32, u8p, u8p, u8p, sz, vp, vp]
    L.jpezyb200_encode_batch.argtypes = [vp, u8p, u8p, u8p, u32, u32, u32, C.c_int, u8p, sz, u64p]
    L.jpezyb200_decode_batch.argtypes = [vp, u8p, sz, u64p, u32, C.POINTER(Frame), C.c_int, u8p, u8p, u8p, sz, vp]
    L.jpezyb200_ipc_alloc.argtypes = [vp, sz, C.POINTER(vp), C.c_char_p]
    L.jpezyb200_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.jpezyb200_ipc_close.argtypes = [vp, vp]
    L.jpezyb200_ipc_free.argtypes = [vp, vp]
    _LIB = L
    return L


def abi_version():
    return load_library().jpezyb200_abi_version()


def default_frame(W, H):
    f = Frame()
    rc = load_library().jpezyb200_default_frame(W, H, C.byref(f))
    if rc:
        raise JpezyError(rc, "default_frame")
    return f


def huff_tables(data):
    """HuffTables from the HUFF_TABLES_BYTES bytes of one image's records (e.g. a slice of d_ht copied to the host)"""
    if isinstance(data, HuffTables):
        return data
    if hasattr(data, "cpu"):
        data = data.cpu().numpy()
    return HuffTables.from_buffer_copy(bytes(memoryview(data).cast("B")))


def optimized_frame(W, H, ht):
    """default_frame(W, H) with the Huffman tables an optimised encode returned (HuffTables or its bytes): the frame
    descriptor that decodes that image"""
    f = default_frame(W, H)
    ht = huff_tables(ht)
    for c in range(2):
        for i in range(2):
            f.ht[c][i] = ht[c][i]
    return f


def plane_bytes(frame):
    return int(load_library().jpezyb200_plane_bytes(C.byref(frame)))


def num_mcus(W, H):
    return ((W + 15) // 16) * ((H + 15) // 16)


def _dp(t):
    """device (or host) pointer of a torch tensor / numpy array / int / None"""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


class Context:
    """One per device (jpezyb200_ctx).  `stream` arguments are raw cudaStream_t ints
    (torch.cuda.current_stream().cuda_stream); None = the context's own stream."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.jpezyb200_ctx_create(int(device), C.byref(h))
        if rc:
            raise JpezyError(rc, self.lib.jpezyb200_strerror(rc).decode())
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.jpezyb200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc:
            raise JpezyError(rc, "%s (%s)" % (self.lib.jpezyb200_strerror(rc).decode(),
                                              self.lib.jpezyb200_last_error(self.h).decode()))

    def set_option(self, opt, value):
        self._chk(self.lib.jpezyb200_set_option(self.h, opt, int(value)))

    def stat(self, which):
        v = C.c_uint64(0)
        self._chk(self.lib.jpezyb200_get_stat(self.h, which, C.byref(v)))
        return v.value

    # ---- host-buffer entry points (numpy uint8 arrays) -----------------------------------------
    def encode(self, r, g, b, W, H, gray=False, scan_cap=None):
        import numpy as np
        r, g, b = (np.ascontiguousarray(x, dtype=np.uint8).reshape(-1) for x in (r, g, b))
        cap = int(scan_cap if scan_cap is not None else max(W * H * 3, 10240))
        out = np.empty(cap, dtype=np.uint8)
        n, nb = C.c_size_t(0), C.c_uint64(0)
        self._chk(self.lib.jpezyb200_encode(self.h, _dp(r), _dp(g), _dp(b), W, H, int(gray), _dp(out), cap, C.byref(n),
                                            C.byref(nb)))
        return out[: n.value].tobytes(), nb.value

    def encode_optimized(self, r, g, b, W, H, gray=False, scan_cap=None):
        """encode with Huffman tables fitted to the image -> (segment, bit count, HuffTables)"""
        import numpy as np
        r, g, b = (np.ascontiguousarray(x, dtype=np.uint8).reshape(-1) for x in (r, g, b))
        cap = int(scan_cap if scan_cap is not None else max(W * H * 3, 10240))
        out = np.empty(cap, dtype=np.uint8)
        n, nb, ht = C.c_size_t(0), C.c_uint64(0), HuffTables()
        self._chk(self.lib.jpezyb200_encode_optimized(self.h, _dp(r), _dp(g), _dp(b), W, H, int(gray), _dp(out), cap, C.byref(n),
                                                      C.byref(nb), C.byref(ht)))
        return out[: n.value].tobytes(), nb.value, ht

    def decode(self, scan, frame, gray=False):
        import numpy as np
        a = np.frombuffer(scan, dtype=np.uint8)
        pl = plane_bytes(frame)
        r, g, b = (np.zeros(pl, dtype=np.uint8) for _ in range(3))
        self._chk(self.lib.jpezyb200_decode(self.h, _dp(a), a.size, C.byref(frame), int(gray), _dp(r), _dp(g), _dp(b), pl))
        return r, g, b

    # ---- device-resident entry points (torch tensors or raw pointers) -------------------------
    def encode_batch_dev(self, d_r, d_g, d_b, W, H, nimg, gray, d_scan, slot_bytes, d_bytes=None, d_bits=None, stream=None):
        self._chk(self.lib.jpezyb200_encode_batch_dev(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, H, nimg, int(gray), _dp(d_scan),
                                                      slot_bytes, _dp(d_bytes), _dp(d_bits), stream))

    def encode_batch_optimized_dev(self, d_r, d_g, d_b, W, H, nimg, gray, d_scan, slot_bytes, d_ht, d_bytes=None, d_bits=None,
                                   stream=None):
        """d_ht: device buffer of nimg * HUFF_TABLES_BYTES bytes, the tables of image i at i * HUFF_TABLES_BYTES"""
        self._chk(self.lib.jpezyb200_encode_batch_optimized_dev(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, H, nimg, int(gray),
                                                                _dp(d_scan), slot_bytes, _dp(d_bytes), _dp(d_bits), _dp(d_ht), stream))

    def read_sizes(self, d_values, n, h_out, stream=None):
        """n uint64 values of a device array into the numpy uint64 array h_out; returns when `stream` has reached this point"""
        self._chk(self.lib.jpezyb200_read_sizes(self.h, _dp(d_values), n, _dp(h_out), stream))

    def transform_fwd_dev(self, d_r, d_g, d_b, W, H, nimg, gray, d_coefs, stream=None):
        self._chk(self.lib.jpezyb200_transform_fwd_dev(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, H, nimg, int(gray),
                                                       _dp(d_coefs), stream))

    def entropy_encode_dev(self, d_coefs, W, H, nimg, gray, d_scan, slot_bytes, d_bytes=None, d_bits=None, stream=None):
        self._chk(self.lib.jpezyb200_entropy_encode_dev(self.h, _dp(d_coefs), W, H, nimg, int(gray), _dp(d_scan), slot_bytes,
                                                        _dp(d_bytes), _dp(d_bits), stream))

    def entropy_encode_optimized_dev(self, d_coefs, W, H, nimg, gray, d_scan, slot_bytes, d_ht, d_bytes=None, d_bits=None,
                                     stream=None):
        self._chk(self.lib.jpezyb200_entropy_encode_optimized_dev(self.h, _dp(d_coefs), W, H, nimg, int(gray), _dp(d_scan), slot_bytes,
                                                                  _dp(d_bytes), _dp(d_bits), _dp(d_ht), stream))

    def decode_batch_dev(self, d_scan, slot_bytes, h_scan_bytes, nimg, frame, gray, d_r, d_g, d_b, plane_len, d_status=None,
                         stream=None):
        import numpy as np
        hs = np.ascontiguousarray(h_scan_bytes, dtype=np.uint64)
        self._chk(self.lib.jpezyb200_decode_batch_dev(self.h, _dp(d_scan), slot_bytes, _dp(hs), nimg, C.byref(frame), int(gray),
                                                      _dp(d_r), _dp(d_g), _dp(d_b), plane_len, _dp(d_status), stream))

    def decode_batch_dev2(self, d_scan, slot_bytes, d_scan_bytes, max_scan_bytes, nimg, frame, gray, d_r, d_g, d_b, plane_len,
                          d_status=None, stream=None):
        """segment lengths read from device memory (no host round trip behind the encoder)"""
        self._chk(self.lib.jpezyb200_decode_batch_dev2(self.h, _dp(d_scan), slot_bytes, _dp(d_scan_bytes), int(max_scan_bytes), nimg,
                                                       C.byref(frame), int(gray), _dp(d_r), _dp(d_g), _dp(d_b), plane_len,
                                                       _dp(d_status), stream))

    def entropy_decode_dev(self, d_scan, slot_bytes, h_scan_bytes, nimg, frame, d_coefs, d_status=None, stream=None):
        import numpy as np
        hs = np.ascontiguousarray(h_scan_bytes, dtype=np.uint64)
        self._chk(self.lib.jpezyb200_entropy_decode_dev(self.h, _dp(d_scan), slot_bytes, _dp(hs), nimg, C.byref(frame),
                                                        _dp(d_coefs), _dp(d_status), stream))

    def transform_inv_dev(self, d_coefs, frame, nimg, gray, d_r, d_g, d_b, plane_len, stream=None):
        self._chk(self.lib.jpezyb200_transform_inv_dev(self.h, _dp(d_coefs), C.byref(frame), nimg, int(gray), _dp(d_r),
                                                       _dp(d_g), _dp(d_b), plane_len, stream))

    def synth_dev(self, d_r, d_g, d_b, W, H, nimg=1, first_frame=0, family=0, stream=None):
        self._chk(self.lib.jpezyb200_synth_dev(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, H, nimg, first_frame, family, stream))

    def synth_rows_dev(self, d_r, d_g, d_b, W, y0, nrows, frame=0, family=0, stream=None):
        self._chk(self.lib.jpezyb200_synth_rows_dev(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, y0, nrows, frame, family, stream))

    # ---- MCU-row sharded encoder (one image, several GPUs): see jpezy_b200/shard.py for the orchestration ----
    def shard_encode_a(self, d_r, d_g, d_b, W, H, mcu_row0, mcu_rows, y_origin, gray, d_last_dc, stream=None):
        self._chk(self.lib.jpezyb200_shard_encode_a(self.h, _dp(d_r), _dp(d_g), _dp(d_b), W, H, mcu_row0, mcu_rows, y_origin, int(gray),
                                                    _dp(d_last_dc), stream))

    def shard_encode_b(self, d_dc_init, d_info, stream=None):
        self._chk(self.lib.jpezyb200_shard_encode_b(self.h, _dp(d_dc_init), _dp(d_info), stream))

    def shard_encode_c(self, d_all_info, rank, nranks, d_out_bytes, stream=None):
        self._chk(self.lib.jpezyb200_shard_encode_c(self.h, _dp(d_all_info), rank, nranks, _dp(d_out_bytes), stream))

    def shard_encode_d(self, d_all_bytes, d_dst, dst_cap, d_total_bytes=None, d_overflow=None, stream=None):
        self._chk(self.lib.jpezyb200_shard_encode_d(self.h, _dp(d_all_bytes), _dp(d_dst), dst_cap, _dp(d_total_bytes), _dp(d_overflow),
                                                    stream))

    def ipc_alloc(self, nbytes):
        """-> (device pointer, 64-byte handle) of a peer-visible buffer owned by this context"""
        p = C.c_void_p()
        h = C.create_string_buffer(64)
        self._chk(self.lib.jpezyb200_ipc_alloc(self.h, nbytes, C.byref(p), h))
        return p.value, h.raw

    def ipc_open(self, handle):
        p = C.c_void_p()
        self._chk(self.lib.jpezyb200_ipc_open(self.h, handle, C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        self._chk(self.lib.jpezyb200_ipc_close(self.h, ptr))

    def ipc_free(self, ptr):
        self._chk(self.lib.jpezyb200_ipc_free(self.h, ptr))

    def shard_decode_dev(self, d_scan, scan_bytes, frame, gray, mcu_row0, mcu_rows, d_r, d_g, d_b, plane_len, d_status=None, stream=None):
        self._chk(self.lib.jpezyb200_shard_decode_dev(self.h, _dp(d_scan), int(scan_bytes), C.byref(frame), int(gray), mcu_row0, mcu_rows,
                                                      _dp(d_r), _dp(d_g), _dp(d_b), plane_len, _dp(d_status), stream))

    # ---- pipelined host batches (numpy arrays or pinned torch tensors) ----
    def encode_batch(self, r, g, b, W, H, nimg, gray, scan_out, slot_bytes, scan_bytes):
        self._chk(self.lib.jpezyb200_encode_batch(self.h, _dp(r), _dp(g), _dp(b), W, H, nimg, int(gray), _dp(scan_out), slot_bytes, _dp(scan_bytes)))

    def decode_batch(self, scan, slot_bytes, scan_bytes, nimg, frame, gray, r, g, b, plane_len, status=None):
        self._chk(self.lib.jpezyb200_decode_batch(self.h, _dp(scan), slot_bytes, _dp(scan_bytes), nimg, C.byref(frame), int(gray), _dp(r), _dp(g),
                                                  _dp(b), plane_len, _dp(status)))

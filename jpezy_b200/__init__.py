"""jpezy_b200 -- B200-native baseline-JPEG hot path behind falgon/jpezy's encoder/decoder.

The product is `libjpezy_b200.so` (hand-written sm_100a CUDA kernels + the C ABI declared in
include/jpezy_b200.h) and the C++ host mirror of the reference classes under include/jpezy/.
This Python package is the thin ctypes view of that C ABI used by the tests and bench.py;
PyTorch only supplies device memory, streams and torch.distributed.

There is no CPU path: importing works anywhere (so the build can be checked on a CPU box), but
creating a Context without the library or without a CUDA device raises.
"""
from .capi import (Context, Frame, HuffTables, JpezyError, abi_version, build_library, default_frame, huff_tables,  # noqa: F401
                   library_path, load_library, optimized_frame, plane_bytes)
from . import synth  # noqa: F401

__all__ = ["Context", "Frame", "HuffTables", "JpezyError", "abi_version", "build_library", "default_frame", "huff_tables",
           "library_path", "load_library", "optimized_frame", "plane_bytes", "synth"]

"""Small end-to-end run for compute-sanitizer (memcheck): encode, decode, sharded encode/decode, general layouts."""
import io
import sys
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import jpezy_b200 as J
from jpezy_b200 import shard

ctx = J.Context(0)
# (the inverse transform takes the second-generation kernel -- TMA bulk copy, mbarrier --; S-noise fills the guard-band queues)
for fam, W, H, gray in ((0, 208, 128, False), (1, 64, 48, False), (2, 17, 33, True), (1, 640, 360, False), (0, 1, 1, False),
                        (0, 1920, 1080, False), (1, 320, 200, True)):
    r, g, b = J.synth.image(fam, W, H)
    scan, _ = ctx.encode(r, g, b, W, H, gray=gray)
    R, G, B = ctx.decode(scan, J.default_frame(W, H), gray=gray)
    ctxs = [J.Context(0) for _ in range(3)] if H >= 48 else []
    if ctxs:
        planes = tuple(torch.from_numpy(x).cuda() for x in (r, g, b))
        got, _ = shard.encode_sharded_local(ctxs, planes, W, H, gray=gray)
        assert got == scan
        out = shard.decode_sharded_local(ctxs, scan, J.default_frame(W, H), gray=gray)
        assert (out[0] == R).all()
        for c in ctxs:
            c.close()
print("sanitize smoke ok")
ctx.close()

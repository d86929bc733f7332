"""helpers shared by the -m gpu tests: torch supplies device memory, everything goes through the C ABI"""
import numpy as np
import torch

import jpezy_b200 as J
from jpezy_b200.capi import num_mcus

GUARD = 4096


class Guarded:
    """n bytes of `dtype` elements with GUARD poisoned bytes on either side (the payload starts `offset` bytes past a 256-byte
    boundary): a kernel that writes outside its buffer leaves a trace that intact() finds"""
    def __init__(self, nelem, dtype, fill=0, offset=0):
        self.esz = torch.empty(0, dtype=dtype).element_size()
        self.n = nelem * self.esz
        self.lo = GUARD + offset
        self.raw = torch.full((self.lo + self.n + GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        self.view = self.raw[self.lo: self.lo + self.n].view(dtype)
        self.view.fill_(fill)

    def intact(self):
        return bool((self.raw[:self.lo] == 0xA5).all().item()) and bool((self.raw[self.lo + self.n:] == 0xA5).all().item())


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_coefs(ctx, r, g, b, W, H, gray=False, nimg=1):
    dr, dg, db = to_dev(r), to_dev(g), to_dev(b)
    n = num_mcus(W, H)
    dc = torch.empty((nimg, n, 6, 64), dtype=torch.int16, device="cuda")
    dc.fill_(-12345)
    torch.cuda.synchronize()      # torch's stream and the context's own (non-blocking) stream are not ordered with each other
    ctx.transform_fwd_dev(dr, dg, db, W, H, nimg, gray, dc, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return dc.cpu().numpy()


def gpu_entropy(ctx, coefs, W, H, nimg=1, slot=None):
    dc = to_dev(np.ascontiguousarray(coefs, dtype=np.int16))
    slot = int(slot or max(W * H * 3, 10240))
    out = torch.zeros((nimg, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    nbits = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.entropy_encode_dev(dc, W, H, nimg, False, out, slot, nbytes, nbits, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    nb = nbytes.cpu().numpy()
    o = out.cpu().numpy()
    return [o[i, : nb[i]].tobytes() if nb[i] >= 0 else None for i in range(nimg)], nbits.cpu().numpy()


def planes(family, W, H, frame=0):
    return J.synth.image(family, W, H, frame)

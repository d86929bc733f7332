"""-m gpu: compute-sanitizer is closed on this pool (profiles/r02_sanitizer_closed.log), so the out-of-bounds check is our
own: every output buffer of the device-resident entry points sits between two poisoned guard zones, which must come back
untouched, and inputs sit at the very end of their allocation's used part (a read past the end lands in the next guard)."""
import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi

pytestmark = pytest.mark.gpu
GUARD = 4096


class Guarded:
    """n bytes of `dtype` elements with GUARD poisoned bytes on either side (the payload starts `offset` bytes past a 256-byte
    boundary)"""
    def __init__(self, nelem, dtype, fill=0, offset=0):
        self.esz = torch.empty(0, dtype=dtype).element_size()
        self.n = nelem * self.esz
        self.lo = GUARD + offset
        self.raw = torch.full((self.lo + self.n + GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        self.view = self.raw[self.lo: self.lo + self.n].view(dtype)
        self.view.fill_(fill)

    def intact(self):
        return bool((self.raw[:self.lo] == 0xA5).all().item()) and bool((self.raw[self.lo + self.n:] == 0xA5).all().item())


@pytest.mark.parametrize("W,H,family,gray,nimg", [(208, 128, 0, False, 1), (1920, 1080, 0, False, 2), (200, 120, 1, False, 3),
                                                   (17, 33, 2, True, 1), (3840, 2160, 1, False, 1), (16, 16, 0, False, 5),
                                                   (4080, 16, 0, False, 1), (136, 1088, 1, True, 2)])
def test_device_entry_points_stay_inside_their_buffers(ctx, W, H, family, gray, nimg):
    npx = W * H
    frame = J.default_frame(W, H)
    pl = capi.plane_bytes(frame)
    nm = capi.num_mcus(W, H)
    slot = max(3 * npx, 10240)
    planes_in = [Guarded(nimg * npx, torch.uint8) for _ in range(3)]
    coefs = Guarded(nimg * nm * 384, torch.int16, fill=0x7777)
    scan = Guarded(nimg * slot, torch.uint8)
    nbytes = Guarded(nimg, torch.int64)
    nbits = Guarded(nimg, torch.int64)
    status = Guarded(nimg, torch.int32, fill=-1)
    out = [Guarded(nimg * pl, torch.uint8, fill=0x11) for _ in range(3)]
    st = torch.cuda.Stream()
    sp = st.cuda_stream
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        ctx.synth_dev(planes_in[0].view, planes_in[1].view, planes_in[2].view, W, H, nimg=nimg, first_frame=3, family=family, stream=sp)
        # per-stage entry points ...
        ctx.transform_fwd_dev(planes_in[0].view, planes_in[1].view, planes_in[2].view, W, H, nimg, gray, coefs.view, stream=sp)
        ctx.entropy_encode_dev(coefs.view, W, H, nimg, gray, scan.view, slot, nbytes.view, nbits.view, stream=sp)
        torch.cuda.synchronize()
        h_nb = nbytes.view.cpu().numpy().astype(np.uint64)
        assert (nbytes.view > 0).all()
        coefs2 = Guarded(nimg * nm * 384, torch.int16, fill=0x7777)
        ctx.entropy_decode_dev(scan.view, slot, h_nb, nimg, frame, coefs2.view, status.view, stream=sp)
        ctx.transform_inv_dev(coefs2.view, frame, nimg, gray, out[0].view, out[1].view, out[2].view, pl, stream=sp)
        torch.cuda.synchronize()
        assert (status.view == 0).all()
        assert torch.equal(coefs.view, coefs2.view), "entropy decode does not invert entropy encode"
        first = [o.view.clone() for o in out]
        # ... and the fused ones, both length conventions
        scan.view.zero_()
        for o in out:
            o.view.fill_(0x22)
        ctx.encode_batch_dev(planes_in[0].view, planes_in[1].view, planes_in[2].view, W, H, nimg, gray, scan.view, slot, nbytes.view, nbits.view, stream=sp)
        ctx.decode_batch_dev2(scan.view, slot, nbytes.view, int(h_nb.max()), nimg, frame, gray, out[0].view, out[1].view, out[2].view, pl, status.view, stream=sp)
        torch.cuda.synchronize()
    assert (status.view == 0).all()
    for a, b in zip(first, out):
        assert torch.equal(a, b.view), "fused and per-stage paths disagree"
    for name, gbuf in [("planes_in", planes_in[0]), ("planes_in", planes_in[1]), ("planes_in", planes_in[2]), ("coefs", coefs), ("coefs2", coefs2),
                       ("scan", scan), ("nbytes", nbytes), ("nbits", nbits), ("status", status), ("out", out[0]), ("out", out[1]), ("out", out[2])]:
        assert gbuf.intact(), "guard zone around %s was written" % name


def test_unaligned_planes_take_the_first_generation_inverse_kernel(ctx):
    """4:2:0 output planes that start 1 byte past a 256-byte boundary (coefficients aligned) go to k_inv_transform, the 4:2:0
    kernel that needs no 16-byte aligned buffers: the planes equal those of the aligned call and the guard zones stay intact.
    (W is not a multiple of 16: that kernel stores whole 16-byte rows of an MCU when it is.)"""
    W, H, nimg = 200, 120, 2
    frame = J.default_frame(W, H)
    pl = capi.plane_bytes(frame)
    nm = capi.num_mcus(W, H)
    sp = torch.cuda.current_stream().cuda_stream
    planes_in = [Guarded(nimg * W * H, torch.uint8) for _ in range(3)]
    coefs = Guarded(nimg * nm * 384, torch.int16)
    ctx.synth_dev(planes_in[0].view, planes_in[1].view, planes_in[2].view, W, H, nimg=nimg, first_frame=7, family=1, stream=sp)
    ctx.transform_fwd_dev(planes_in[0].view, planes_in[1].view, planes_in[2].view, W, H, nimg, False, coefs.view, stream=sp)
    outs = []
    for offset in (0, 1):
        out = [Guarded(nimg * pl, torch.uint8, fill=0x44, offset=offset) for _ in range(3)]
        ctx.transform_inv_dev(coefs.view, frame, nimg, False, out[0].view, out[1].view, out[2].view, pl, stream=sp)
        torch.cuda.synchronize()
        for o in out:
            assert o.intact(), "guard zone around an output plane was written (offset %d)" % offset
        outs.append([o.view.clone() for o in out])
    assert coefs.intact()
    for a, b in zip(*outs):
        assert torch.equal(a, b), "%d samples differ between the unaligned and the aligned planes" % int((a != b).sum())


LAYOUTS = {"444": ((1, 1, 1), (1, 1, 1)), "422": ((2, 1, 1), (1, 1, 1)), "440": ((1, 1, 1), (2, 1, 1)), "gray1": ((1,), (1,))}


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("W,H", [(70, 45), (129, 257), (640, 368), (8, 8)])
@pytest.mark.parametrize("gray", [False, True])
def test_general_layout_inverse_equals_validation_kernel_and_stays_inside(ctx, layout, W, H, gray):
    """the fast inverse path of the sampling layouts jpezy's encoder never writes (dec_transform_g.cuh) against the FP64 validation
    kernel (JPEZYB200_OPT_TRANSFORM = 1) on random coefficients -- small ones, DC-only blocks, full-range ones that drive the
    samples far outside [0, 255] -- with guard zones around the planes."""
    hs, vs = LAYOUTS[layout]
    f = J.default_frame(W, H)
    f.ncomp = len(hs)
    for i in range(len(hs)):
        f.hs[i], f.vs[i] = hs[i], vs[i]
    if len(hs) == 3:
        f.tq[2] = 1
    hmax, vmax = max(hs), max(vs)
    hu, vu = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    nb = sum(a * b for a, b in zip(hs, vs))
    pl = capi.plane_bytes(f)
    rng = np.random.default_rng(W * 1000 + H)
    c = np.zeros((hu * vu * nb, 64), dtype=np.int16)
    c[:, 0] = rng.integers(-100, 100, size=c.shape[0])
    kind = rng.integers(0, 4, size=c.shape[0])
    m = kind == 1
    c[m, 1:6] = rng.integers(-4, 5, size=(int(m.sum()), 5))
    m = kind == 2
    c[m, :] = (rng.integers(-30, 31, size=(int(m.sum()), 64)) * (rng.random((int(m.sum()), 64)) < 0.3)).astype(np.int16)
    m = kind == 3
    c[m, :] = rng.integers(-1023, 1024, size=(int(m.sum()), 64)).astype(np.int16)
    d = Guarded(c.size, torch.int16)
    d.view.copy_(torch.from_numpy(c.reshape(-1)).cuda())
    outs = []
    for variant in (0, 1):
        ctx.set_option(capi.OPT_TRANSFORM, variant)
        try:
            out = [Guarded(pl, torch.uint8, fill=0x33) for _ in range(3)]
            ctx.transform_inv_dev(d.view, f, 1, gray, out[0].view, out[1].view, out[2].view, pl, stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        finally:
            ctx.set_option(capi.OPT_TRANSFORM, 0)
        for o in out:
            assert o.intact(), "guard zone around an output plane was written (variant %d)" % variant
        outs.append([o.view.clone() for o in out])
    assert d.intact()
    for a, b in zip(*outs):
        nd = int((a != b).sum())
        assert nd == 0, "%d samples differ from the validation kernel" % nd

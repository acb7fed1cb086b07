"""The argument checks of the seven device entry points: the six rtjgpu_decode_device* calls and rtjgpu_scan_device.  They
share one front end, so the same fault gets the same code from every call it applies to, and is refused before anything
is reserved or launched.  Every pointer is a real, small, aligned device allocation except the one a case spoils; sizes
and frame counts that a case makes too large are never backed by memory, which is safe only because they are refused
first."""
import ctypes as C

import pytest
import torch

import gmerlin_avdecoder_b200 as g
from gmerlin_avdecoder_b200 import capi
from gmerlin_avdecoder_b200 import device as D
from streams import clip

pytestmark = pytest.mark.gpu

W, H, F = 64, 48, 2
MAX_FRAMES = 65534            # RTJGPU_MAX_FRAMES_PER_BATCH
KIND = capi.CONV_RGB32
DECODES = ("decode_device", "decode_device_seq", "decode_device_select",
           "decode_device_rgb", "decode_device_rgb_seq", "decode_device_rgb_select")
ENTRY_POINTS = DECODES + ("scan_device",)
RGB = tuple(n for n in DECODES if "_rgb" in n)


def _ptrs(*p):
    return (C.c_void_p * len(p))(*p)


def _call(L, h, name, a):
    """One raw call of entry point `name` with the arguments in `a`; returns its code.  The _seq and _select calls get one
    sequence, the _select calls select frame 0; the _rgb calls get pitches that fit w and h."""
    vp = C.c_void_p
    first = (C.c_int * 2)(0, a["F"])
    sel = (C.c_int * 1)(0)
    rp = (max(a["w"], 0) * capi.CONV_BPP[KIND] + 15) // 16 * 16
    fp = rp * max(a["h"], 0)
    batch = (h, vp(a["stream"]), vp(a["desc"]), a["F"], a["w"], a["h"])
    st = vp(a["cuda_stream"])
    if name == "scan_device":
        return L.rtjgpu_scan_device(*batch, st)
    if name == "decode_device":
        return L.rtjgpu_decode_device(*batch, vp(a["out"]), vp(a["carry"]), st)
    if name == "decode_device_seq":
        return L.rtjgpu_decode_device_seq(*batch, 1, first, vp(a["out"]), _ptrs(a["carry"]), st)
    if name == "decode_device_select":
        return L.rtjgpu_decode_device_select(*batch, 1, first, _ptrs(a["carry"]), 1, sel, vp(a["out"]), st)
    if name == "decode_device_rgb":
        return L.rtjgpu_decode_device_rgb(*batch, KIND, vp(a["rgb"]), rp, fp, 0, vp(a["carry"]), vp(a["last"]), st)
    if name == "decode_device_rgb_seq":
        return L.rtjgpu_decode_device_rgb_seq(*batch, 1, first, KIND, vp(a["rgb"]), rp, fp, 0, _ptrs(a["carry"]),
                                              _ptrs(a["last"]), st)
    assert name == "decode_device_rgb_select"
    return L.rtjgpu_decode_device_rgb_select(*batch, 1, first, _ptrs(a["carry"]), 1, sel, KIND, vp(a["rgb"]), rp, fp, 0,
                                             _ptrs(a["last"]), st)


# (what is wrong, the arguments that make it so, the code, the entry points it applies to)
CASES = [
    ("NULL stream", lambda a: dict(stream=0), capi.E_ARG, ENTRY_POINTS),
    ("NULL desc", lambda a: dict(desc=0), capi.E_ARG, ENTRY_POINTS),
    ("NULL output", lambda a: dict(out=0, rgb=0), capi.E_ARG, DECODES),
    ("misaligned stream", lambda a: dict(stream=a["stream"] + 2), capi.E_ARG, ENTRY_POINTS),
    ("misaligned desc", lambda a: dict(desc=a["desc"] + 4), capi.E_ARG, ENTRY_POINTS),
    ("misaligned output", lambda a: dict(out=a["out"] + 8, rgb=a["rgb"] + 8), capi.E_ARG, DECODES),
    ("misaligned carry", lambda a: dict(carry=a["carry"] + 4), capi.E_ARG, DECODES),
    ("misaligned last_yuv", lambda a: dict(last=a["last"] + 8), capi.E_ARG, RGB),
    ("w zero", lambda a: dict(w=0), capi.E_SIZE, ENTRY_POINTS),
    ("h zero", lambda a: dict(h=0), capi.E_SIZE, ENTRY_POINTS),
    ("w not a multiple of 16", lambda a: dict(w=W + 8), capi.E_SIZE, ENTRY_POINTS),
    ("h not a multiple of 16", lambda a: dict(h=H + 8), capi.E_SIZE, ENTRY_POINTS),
    ("w above 65535", lambda a: dict(w=65536), capi.E_SIZE, ENTRY_POINTS),
    ("h above 65535", lambda a: dict(h=65536), capi.E_SIZE, ENTRY_POINTS),
    ("F over the limit", lambda a: dict(F=MAX_FRAMES + 1), capi.E_TOOBIG, ENTRY_POINTS),
    ("a frame of 4 GiB or more", lambda a: dict(F=1, w=65520, h=65520), capi.E_TOOBIG, ENTRY_POINTS),
]


@pytest.fixture(scope="module")
def batch():
    """A real two-frame batch with output, RGB, carry and last_yuv buffers for it."""
    s, o = clip(W, H, 128, F, key_rate=2, lm=2, cm=2)
    desc, _ = g.plan(s, o)
    b = D.upload(s, desc, W, H)
    fsz = W * H * 3 // 2
    bufs = dict(rgb=torch.empty((F, H, W * 4), dtype=torch.uint8, device="cuda"),
                carry=torch.zeros(fsz, dtype=torch.uint8, device="cuda"),
                last=torch.empty(fsz, dtype=torch.uint8, device="cuda"))
    args = dict(stream=b.stream.data_ptr(), desc=b.desc.data_ptr(), F=F, w=W, h=H, out=b.out.data_ptr(),
                cuda_stream=torch.cuda.current_stream().cuda_stream, **{k: t.data_ptr() for k, t in bufs.items()})
    return args, (b, bufs)


@pytest.mark.parametrize("name", ENTRY_POINTS)
def test_same_fault_same_code_nothing_launched(batch, name):
    args, _ = batch
    L = g.load_library()
    with g.BatchContext(0) as ctx:
        assert _call(L, ctx._h, name, args) == capi.OK            # the arguments the cases start from are good
        torch.cuda.synchronize()
        n0 = ctx.launch_count()
        assert n0 > 0
        for what, bad, code, applies in CASES:
            if name not in applies:
                continue
            assert _call(L, ctx._h, name, {**args, **bad(args)}) == code, what
            assert ctx.launch_count() == n0, what
        torch.cuda.synchronize()

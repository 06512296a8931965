"""libmsda_b200_amp.so without a GPU: its kernel set, its ABI version and the argument validation of its C entry point
(include/msda_b200_amp.h).

The validation sweep passes fake pointers (0 and small aligned / misaligned integers), so it only makes calls that
are rejected before anything is enqueued or that have nothing to do (rows == 0).  Like test_capi_status.py it skips
itself when a device is present, so that a validation bug cannot hand a fake pointer to a real GPU.
"""
import itertools
import math
import os
import re

import pytest
import torch

import dispatch_cases as dc
from snipper_b200 import capi
from snipper_b200.build import AMP_LIB_PATH, build_amp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64, BF16 = capi.MSDA_DTYPE_F32, capi.MSDA_DTYPE_F64, capi.MSDA_DTYPE_BF16
OK, INVALID, DTYPE = capi.MSDA_OK, capi.MSDA_ERR_INVALID_ARGUMENT, capi.MSDA_ERR_UNSUPPORTED_DTYPE
LAUNCH = "launch"                       # the call would pass validation and enqueue a kernel: never made here


@pytest.fixture(scope="module")
def amp():
    build_amp_library()
    return capi.amp_lib()


def test_kernels_are_exactly_the_16_tail_instantiations():
    missing = dc.missing_tools()
    if missing:
        pytest.skip("%s not found: cannot list the kernels of the library" % " and ".join(missing))
    want = {"layer_tail_amp_kernel<%d, %s>" % (v, r) for v in range(1, 9) for r in ("float", "__nv_bfloat16")}
    assert dc.compiled_kernels(build_amp_library()) == want


def test_abi_version_matches_the_header(amp):
    with open(os.path.join(ROOT, "include", "msda_b200_amp.h")) as f:
        header = int(re.search(r"#define MSDA_AMP_ABI_VERSION (\d+)", f.read()).group(1))
    assert amp.msda_amp_abi_version() == header == capi.MSDA_AMP_ABI_VERSION
    assert os.path.exists(AMP_LIB_PATH)
    for sym in capi.AMP_EXPORTS:
        getattr(amp, sym)


REQUIRED = ("y", "residual", "gamma", "beta", "out")
OPTIONAL = ("bias", "pos", "out_bf16", "out_pos")
BAD_PTRS = (0, 257, 260, 264)           # NULL, and 1-, 4- and 8-byte aligned
OPT_PTRS = (0, 256, 257, 260, 264)
BASE = dict(y=256, bias=512, residual=768, rdt=F32, gamma=1024, beta=1280, pos=1536, out=1792, out_bf16=2048,
            out_pos=2304, rows=9, cols=384, eps=1e-5)


def expected(a):
    """The entry point's rules, restated: dtype, then sizes and eps, then the pos pair, then rows == 0, then the
    pointers (every one 16-byte aligned, the required ones not NULL)."""
    if a["rdt"] not in (F32, BF16):
        return DTYPE
    if a["rows"] < 0 or a["cols"] <= 0 or a["cols"] % 128 or a["cols"] > 1024 or not a["eps"] >= 0:
        return INVALID
    if (a["pos"] == 0) != (a["out_pos"] == 0):
        return INVALID
    if a["rows"] == 0:
        return OK
    if any(a[k] == 0 or a[k] % 16 for k in REQUIRED) or any(a[k] % 16 for k in OPTIONAL):
        return INVALID
    return LAUNCH


def cases():
    perturb = {k: BAD_PTRS for k in REQUIRED}
    perturb.update({k: OPT_PTRS for k in OPTIONAL})
    perturb.update(rdt=(F32, BF16, F64, 7, -1), cols=(0, -128, 64, 200, 1152, 2048, 128, 1024),
                   rows=(-1, 0, 1, 1 << 40), eps=(-1e-5, float("nan"), 0.0, math.inf))
    for rows, rdt in itertools.product((0, 9), (F32, BF16)):
        for key, values in perturb.items():
            for v in values:
                yield {**BASE, "rows": rows, "rdt": rdt, key: v}
        for pos, out_pos in ((0, 0), (0, 2304), (1536, 0), (0, 257), (257, 0)):
            yield {**BASE, "rows": rows, "rdt": rdt, "pos": pos, "out_pos": out_pos}


def test_argument_validation_sweep(amp):
    if torch.cuda.is_available():
        pytest.skip("fake pointers are never handed to a machine with a device")
    made = 0
    seen = set()
    for a in cases():
        want = expected(a)
        if want == LAUNCH:
            continue
        got = amp.msda_amp_layer_tail(a["y"], a["bias"] or None, a["residual"], a["rdt"], a["gamma"], a["beta"],
                                      a["pos"] or None, a["out"], a["out_bf16"] or None, a["out_pos"] or None,
                                      a["rows"], a["cols"], a["eps"], None)
        assert got == want, a
        made += 1
        seen.add(want)
    assert made > 150 and seen == {OK, INVALID, DTYPE}

"""libmsda_b200_amp_train.so without a GPU: its kernel set, its ABI version, its workspace query and the argument
validation of its two C entry points (include/msda_b200_amp_train.h).

The validation sweep passes fake pointers (0 and small aligned / misaligned integers), so it only makes calls that
are rejected before anything is enqueued or that have nothing to do (rows == 0).  Like test_train_library.py it skips
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
from snipper_b200.build import AMP_TRAIN_LIB_PATH, build_amp_train_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64, BF16 = capi.MSDA_DTYPE_F32, capi.MSDA_DTYPE_F64, capi.MSDA_DTYPE_BF16
OK, INVALID, DTYPE = capi.MSDA_OK, capi.MSDA_ERR_INVALID_ARGUMENT, capi.MSDA_ERR_UNSUPPORTED_DTYPE
LAUNCH = "launch"                       # the call would pass validation and enqueue a kernel: never made here


@pytest.fixture(scope="module")
def lib():
    build_amp_train_library()
    return capi.amp_train_lib()


def test_kernels_are_exactly_the_forward_backward_and_sum_instantiations():
    missing = dc.missing_tools()
    if missing:
        pytest.skip("%s not found: cannot list the kernels of the library" % " and ".join(missing))
    want = {"layer_tail_amp_train_%s_kernel<%d, %s>" % (k, v, r)
            for k in ("fwd", "bwd") for v in range(1, 9) for r in ("float", "__nv_bfloat16")}
    want.add("layer_tail_param_sum_kernel")
    assert dc.compiled_kernels(build_amp_train_library()) == want


def test_abi_version_matches_the_header(lib):
    with open(os.path.join(ROOT, "include", "msda_b200_amp_train.h")) as f:
        header = int(re.search(r"#define MSDA_AMP_TRAIN_ABI_VERSION (\d+)", f.read()).group(1))
    assert lib.msda_amp_train_abi_version() == header == capi.MSDA_AMP_TRAIN_ABI_VERSION
    assert os.path.exists(AMP_TRAIN_LIB_PATH)
    for sym in capi.AMP_TRAIN_EXPORTS:
        getattr(lib, sym)


def test_exports_are_every_symbol_the_header_declares():
    with open(os.path.join(ROOT, "include", "msda_b200_amp_train.h")) as f:
        declared = set(re.findall(r"MSDA_API \w+ \*?(msda_\w+)\(", f.read()))
    assert declared == set(capi.AMP_TRAIN_EXPORTS)


def test_workspace_is_monotone_in_rows_and_empty_at_zero_rows(lib):
    for C in (128, 384, 1024):
        assert lib.msda_amp_train_layer_tail_workspace_bytes(0, C) == 0
        last = 0
        for rows in (1, 7, 8, 9, 240, 2367, 2368, 2369, 39500, 65541, 1 << 24):
            b = lib.msda_amp_train_layer_tail_workspace_bytes(rows, C)
            assert b >= last and b % 16 == 0 and b >= 3 * C * 4
            last = b
    for bad in (0, 64, 200, 1152):
        assert lib.msda_amp_train_layer_tail_workspace_bytes(9, bad) == 0
    for rows in (-1, -(1 << 40)):
        assert lib.msda_amp_train_layer_tail_workspace_bytes(rows, 384) == 0


BAD_PTRS = (0, 257, 260, 264)           # NULL, and 1-, 4- and 8-byte aligned
OPT_PTRS = (0, 256, 257, 260, 264)
SIZES = dict(cols=(0, -128, 64, 200, 1152, 2048, 128, 1024), rows=(-1, 0, 1, 1 << 40),
             scale=(0.5, 1.0, 1.25, math.inf, float("nan"), -1.0), rdt=(F32, BF16, F64, 7, -1))

FWD_REQUIRED = ("y", "residual", "gamma", "beta", "out", "h", "mean_rstd")
FWD_OPTIONAL = ("bias", "mask", "pos", "out_bf16", "out_pos")
FWD_BASE = dict(y=256, bias=512, residual=768, rdt=F32, mask=1024, scale=1.25, gamma=1280, beta=1536, pos=1792,
                out=2048, out_bf16=2304, out_pos=2560, h=2816, mean_rstd=3072, rows=9, cols=384, eps=1e-5)

BWD_REQUIRED = ("grad_out", "h", "mean_rstd", "gamma", "grad_residual", "grad_y", "param_grads", "partials")
BWD_OPTIONAL = ("grad_out_bf16", "grad_out_pos", "mask")
BWD_BASE = dict(grad_out=256, grad_out_bf16=512, grad_out_pos=768, h=1024, mean_rstd=1280, mask=1536, scale=1.25,
                gamma=1792, grad_residual=2048, rdt=F32, grad_y=2304, param_grads=2560, partials=2816, rows=9,
                cols=384)


def _sizes_ok(a):
    return (a["rows"] >= 0 and a["cols"] > 0 and a["cols"] % 128 == 0 and a["cols"] <= 1024 and
            math.isfinite(a["scale"]) and a["scale"] >= 1)


def expected_forward(a):
    """The forward's rules, restated: the residual dtype, then sizes, eps and keep_scale, then the pos pair, then
    rows == 0, then the pointers (every one 16-byte aligned, the required ones not NULL)."""
    if a["rdt"] not in (F32, BF16):
        return DTYPE
    if not _sizes_ok(a) or not a["eps"] >= 0:
        return INVALID
    if (a["pos"] == 0) != (a["out_pos"] == 0):
        return INVALID
    if a["rows"] == 0:
        return OK
    if any(a[k] == 0 or a[k] % 16 for k in FWD_REQUIRED) or any(a[k] % 16 for k in FWD_OPTIONAL):
        return INVALID
    return LAUNCH


def expected_backward(a):
    if a["rdt"] not in (F32, BF16):
        return DTYPE
    if not _sizes_ok(a):
        return INVALID
    if a["rows"] == 0:
        return OK
    if any(a[k] == 0 or a[k] % 16 for k in BWD_REQUIRED) or any(a[k] % 16 for k in BWD_OPTIONAL):
        return INVALID
    return LAUNCH


def _cases(base, required, optional, extra):
    perturb = {k: BAD_PTRS for k in required}
    perturb.update({k: OPT_PTRS for k in optional})
    perturb.update(SIZES)
    perturb.update(extra)
    for rows, rdt in itertools.product((0, 9), (F32, BF16)):
        for key, values in perturb.items():
            for v in values:
                yield {**base, "rows": rows, "rdt": rdt, key: v}


def forward_cases():
    yield from _cases(FWD_BASE, FWD_REQUIRED, FWD_OPTIONAL, {"eps": (-1e-5, float("nan"), 0.0, math.inf)})
    for rows, rdt in itertools.product((0, 9), (F32, BF16)):
        for pos, out_pos in ((0, 0), (0, 2560), (1792, 0), (0, 257), (257, 0)):
            yield {**FWD_BASE, "rows": rows, "rdt": rdt, "pos": pos, "out_pos": out_pos}


def _none(v):
    return v or None


def test_forward_argument_validation_sweep(lib):
    if torch.cuda.is_available():
        pytest.skip("fake pointers are never handed to a machine with a device")
    made, seen = 0, set()
    for a in forward_cases():
        want = expected_forward(a)
        if want == LAUNCH:
            continue
        got = lib.msda_amp_train_layer_tail_forward(
            _none(a["y"]), _none(a["bias"]), _none(a["residual"]), a["rdt"], _none(a["mask"]), a["scale"],
            _none(a["gamma"]), _none(a["beta"]), _none(a["pos"]), _none(a["out"]), _none(a["out_bf16"]),
            _none(a["out_pos"]), _none(a["h"]), _none(a["mean_rstd"]), a["rows"], a["cols"], a["eps"], None)
        assert got == want, a
        made += 1
        seen.add(want)
    assert made > 200 and seen == {OK, INVALID, DTYPE}


def test_backward_argument_validation_sweep(lib):
    if torch.cuda.is_available():
        pytest.skip("fake pointers are never handed to a machine with a device")
    made, seen = 0, set()
    for a in _cases(BWD_BASE, BWD_REQUIRED, BWD_OPTIONAL, {}):
        want = expected_backward(a)
        if want == LAUNCH:
            continue
        got = lib.msda_amp_train_layer_tail_backward(
            _none(a["grad_out"]), _none(a["grad_out_bf16"]), _none(a["grad_out_pos"]), _none(a["h"]),
            _none(a["mean_rstd"]), _none(a["mask"]), a["scale"], _none(a["gamma"]), _none(a["grad_residual"]),
            a["rdt"], _none(a["grad_y"]), _none(a["param_grads"]), _none(a["partials"]), a["rows"], a["cols"], None)
        assert got == want, a
        made += 1
        seen.add(want)
    assert made > 150 and seen == {OK, INVALID, DTYPE}

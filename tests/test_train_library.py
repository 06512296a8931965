"""libmsda_b200_train.so without a GPU: its kernel set, its ABI version, its workspace query and the argument validation
of its two C entry points (include/msda_b200_train.h).

The validation sweep passes fake pointers (0 and small aligned / misaligned integers), so it only makes calls that
are rejected before anything is enqueued or that have nothing to do (rows == 0).  Like test_amp_library.py it skips
itself when a device is present, so that a validation bug cannot hand a fake pointer to a real GPU.
"""
import math
import os
import re

import pytest
import torch

import dispatch_cases as dc
from snipper_b200 import capi
from snipper_b200.build import TRAIN_LIB_PATH, build_train_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, INVALID = capi.MSDA_OK, capi.MSDA_ERR_INVALID_ARGUMENT
LAUNCH = "launch"                       # the call would pass validation and enqueue a kernel: never made here


@pytest.fixture(scope="module")
def train():
    build_train_library()
    return capi.train_lib()


def test_kernels_are_exactly_the_forward_backward_and_sum_instantiations():
    missing = dc.missing_tools()
    if missing:
        pytest.skip("%s not found: cannot list the kernels of the library" % " and ".join(missing))
    want = {"layer_tail_train_fwd_kernel<%d>" % v for v in range(1, 9)}
    want |= {"layer_tail_train_bwd_kernel<%d>" % v for v in range(1, 9)}
    want.add("layer_tail_param_sum_kernel")
    assert dc.compiled_kernels(build_train_library()) == want


def test_abi_version_matches_the_header(train):
    with open(os.path.join(ROOT, "include", "msda_b200_train.h")) as f:
        header = int(re.search(r"#define MSDA_TRAIN_ABI_VERSION (\d+)", f.read()).group(1))
    assert train.msda_train_abi_version() == header == capi.MSDA_TRAIN_ABI_VERSION
    assert os.path.exists(TRAIN_LIB_PATH)
    for sym in capi.TRAIN_EXPORTS:
        getattr(train, sym)


def test_workspace_is_monotone_in_rows_and_empty_at_zero_rows(train):
    for C in (128, 384, 1024):
        assert train.msda_train_layer_tail_workspace_bytes(0, C) == 0
        last = 0
        for rows in (1, 7, 8, 9, 240, 2367, 2368, 2369, 39500, 65541, 1 << 24):
            b = train.msda_train_layer_tail_workspace_bytes(rows, C)
            assert b >= last and b % 16 == 0 and b >= 3 * C * 4
            last = b
    for bad in (0, 64, 200, 1152):
        assert train.msda_train_layer_tail_workspace_bytes(9, bad) == 0


BAD_PTRS = (0, 257, 260, 264)           # NULL, and 1-, 4- and 8-byte aligned
OPT_PTRS = (0, 256, 257, 260, 264)
SIZES = dict(cols=(0, -128, 64, 200, 1152, 2048, 128, 1024), rows=(-1, 0, 1, 1 << 40),
             scale=(0.5, 1.0, 1.25, math.inf, float("nan"), -1.0))

FWD_REQUIRED = ("y", "residual", "gamma", "beta", "out", "h", "mean_rstd")
FWD_OPTIONAL = ("bias", "mask", "pos", "out_pos")
FWD_BASE = dict(y=256, bias=512, residual=768, mask=1024, scale=1.25, gamma=1280, beta=1536, pos=1792, out=2048,
                out_pos=2304, h=2560, mean_rstd=2816, rows=9, cols=384, eps=1e-5)

BWD_REQUIRED = ("grad_out", "h", "mean_rstd", "gamma", "grad_residual", "grad_y", "param_grads", "partials")
BWD_OPTIONAL = ("grad_out_pos", "mask")
BWD_BASE = dict(grad_out=256, grad_out_pos=512, h=768, mean_rstd=1024, mask=1280, scale=1.25, gamma=1536,
                grad_residual=1792, grad_y=2048, param_grads=2304, partials=2560, rows=9, cols=384)


def _sizes_ok(a):
    return (a["rows"] >= 0 and a["cols"] > 0 and a["cols"] % 128 == 0 and a["cols"] <= 1024 and
            math.isfinite(a["scale"]) and a["scale"] >= 1)


def expected_forward(a):
    """The forward's rules, restated: sizes, eps and keep_scale, then the pos pair, then rows == 0, then the pointers
    (every one 16-byte aligned, the required ones not NULL)."""
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
    for rows in (0, 9):
        for key, values in perturb.items():
            for v in values:
                yield {**base, "rows": rows, key: v}


def forward_cases():
    yield from _cases(FWD_BASE, FWD_REQUIRED, FWD_OPTIONAL, {"eps": (-1e-5, float("nan"), 0.0, math.inf)})
    for rows in (0, 9):
        for pos, out_pos in ((0, 0), (0, 2304), (1792, 0), (0, 257), (257, 0)):
            yield {**FWD_BASE, "rows": rows, "pos": pos, "out_pos": out_pos}


def _none(v):
    return v or None


def test_forward_argument_validation_sweep(train):
    if torch.cuda.is_available():
        pytest.skip("fake pointers are never handed to a machine with a device")
    made, seen = 0, set()
    for a in forward_cases():
        want = expected_forward(a)
        if want == LAUNCH:
            continue
        got = train.msda_train_layer_tail_forward(
            _none(a["y"]), _none(a["bias"]), _none(a["residual"]), _none(a["mask"]), a["scale"], _none(a["gamma"]),
            _none(a["beta"]), _none(a["pos"]), _none(a["out"]), _none(a["out_pos"]), _none(a["h"]),
            _none(a["mean_rstd"]), a["rows"], a["cols"], a["eps"], None)
        assert got == want, a
        made += 1
        seen.add(want)
    assert made > 100 and seen == {OK, INVALID}


def test_backward_argument_validation_sweep(train):
    if torch.cuda.is_available():
        pytest.skip("fake pointers are never handed to a machine with a device")
    made, seen = 0, set()
    for a in _cases(BWD_BASE, BWD_REQUIRED, BWD_OPTIONAL, {}):
        want = expected_backward(a)
        if want == LAUNCH:
            continue
        got = train.msda_train_layer_tail_backward(
            _none(a["grad_out"]), _none(a["grad_out_pos"]), _none(a["h"]), _none(a["mean_rstd"]), _none(a["mask"]),
            a["scale"], _none(a["gamma"]), _none(a["grad_residual"]), _none(a["grad_y"]), _none(a["param_grads"]),
            _none(a["partials"]), a["rows"], a["cols"], None)
        assert got == want, a
        made += 1
        seen.add(want)
    assert made > 80 and seen == {OK, INVALID}


def test_keep_scale_is_torch_float_scale():
    """keep_scale(p) is 1 / (1 - p) rounded to float, the factor torch's dropout applies to kept elements."""
    from snipper_b200 import ops
    for p in (0.0, 0.1, 0.5, 0.3, 0.9):
        want = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(1.0 - p, dtype=torch.float32)
        assert ops.keep_scale(p) == float(want)

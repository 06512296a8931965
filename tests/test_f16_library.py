"""libmsda_b200_f16.so without a GPU: its kernel set, its ABI version and exports, and the rule that each of its entry
points returns what its libmsda_b200.so twin returns with MSDA_DTYPE_BF16 (include/msda_b200_f16.h).

The validation sweeps pass fake pointers (0 and small aligned / misaligned integers).  A call that the main library
accepts would enqueue work; those are never made on the fp16 library, and the sweeps skip themselves when a device is
present, so that a validation bug cannot hand a fake pointer to a real GPU (as in test_capi_status.py).
"""
import itertools
import os
import re

import pytest
import torch

import dispatch_cases as dc
import test_capi_status as cs
from snipper_b200 import capi
from snipper_b200.build import F16_LIB_PATH, build_f16_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16 = capi.MSDA_DTYPE_BF16

no_device_only = pytest.mark.skipif(torch.cuda.is_available(), reason="calls entry points with fake pointers")


@pytest.fixture(scope="module")
def f16():
    build_f16_library()
    return capi.f16_lib()


def to_f16(name):
    """The fp16 twin of a bf16 kernel instantiation: the 16-byte lane __nv_bfloat16 -> __half, the 8-byte bf16q -> halfq"""
    return name.replace("__nv_bfloat16", "__half").replace("bf16q", "halfq")


def bf16_kernels():
    """Every bf16 instantiation dispatch_cases knows of (launched by a case or listed unreachable), except the masked
    zero-fill, which the module never calls and the fp16 library does not have."""
    return {k for k in dc.covered() | set(dc.UNREACHABLE)
            if ("__nv_bfloat16" in k or "bf16q" in k) and dc.family(k) != "masked_zero_kernel"}


def test_kernels_are_the_fp16_twins_of_the_bf16_set():
    missing = dc.missing_tools()
    if missing:
        pytest.skip("%s not found: cannot list the kernels of the library" % " and ".join(missing))
    want = {to_f16(k) for k in bf16_kernels()}
    assert len(want) == len(bf16_kernels()) > 100
    assert dc.compiled_kernels(build_f16_library()) == want


def test_abi_version_and_exports_match_the_header(f16):
    with open(os.path.join(ROOT, "include", "msda_b200_f16.h")) as f:
        header = f.read()
    assert f16.msda_f16_abi_version() == int(re.search(r"#define MSDA_F16_ABI_VERSION (\d+)", header).group(1)) \
        == capi.MSDA_F16_ABI_VERSION
    assert set(re.findall(r"MSDA_API \w+ \*?(msda_f16_\w+)\(", header)) == set(capi.F16_EXPORTS)
    assert os.path.exists(F16_LIB_PATH)
    for sym in capi.F16_EXPORTS:
        getattr(f16, sym)


# ---- the fused entries and the frame passes: the argument lists of test_capi_status.ENTRIES ----
def _fwd(L, a):
    return L.msda_f16_snippet_forward(a["value"], a["shapes"], a["lsi"], a["offsets"], a["logits"], a["ref"], a["out"],
                                      a["N"], a["T2"], a["T1"], a["n_frame"], a["S"], a["M"], a["D"], a["L"], a["Lq"],
                                      a["P"], a["sn"], a["st"], a["rsn"], a["rst"], a["ors"], a["lrs"], a["ob"],
                                      a["lb"], a["vr"], a["mask"], a["mrs"], a["mcs"], a["flags"], None)


def _bwd(L, a):
    return L.msda_f16_snippet_backward(a["value"], a["shapes"], a["lsi"], a["offsets"], a["logits"], a["ref"],
                                       a["gout"], a["gvalue"], a["goffsets"], a["glogits"], a["N"], a["T2"], a["T1"],
                                       a["n_frame"], a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"], a["sn"], a["st"],
                                       a["rsn"], a["rst"], a["ors"], a["lrs"], a["ob"], a["lb"], a["vr"], a["mask"],
                                       a["mrs"], a["mcs"], a["flags"], None)


def _frame_sum(L, a):
    return L.msda_f16_frame_sum(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                                a["M"] * a["D"], a["sn"], a["st"], a["mrs"], a["mcs"], None)


def _frame_unsum(L, a):
    return L.msda_f16_frame_unsum(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                                  a["M"] * a["D"], a["mrs"], a["mcs"], None)


TWINS = {"msda_snippet_forward": _fwd, "msda_snippet_backward": _bwd, "msda_frame_sum": _frame_sum,
         "msda_frame_unsum": _frame_unsum}


@no_device_only
@pytest.mark.parametrize("name", list(TWINS))
def test_fused_and_frame_statuses_equal_the_bf16_statuses(f16, name):
    """Every bf16 argument list of the recorded sweep the main library rejects or finishes without a launch: the fp16
    entry returns the same status.  (The cases the table marks '-' would launch; they are not made.)"""
    import json
    with open(cs.TABLE) as f:
        recorded = json.load(f)[name]["status"]
    fn, cases = cs.ENTRIES[name]
    cases = list(cases())
    assert len(cases) == len(recorded)
    main = capi.lib()
    made, diff, seen = 0, [], set()
    for a, s in zip(cases, recorded):
        if a["dtype"] != BF16 or s == "-":
            continue
        want = fn(main, a)
        assert want == int(s)
        got = TWINS[name](f16, a)
        made += 1
        seen.add(want)
        if got != want:
            diff.append((a, want, got))
    assert not diff, "%d of %d cases differ, e.g. %r (bf16 %d, fp16 %d)" % ((len(diff), made) + diff[0])
    assert made > 100 and capi.MSDA_ERR_INVALID_ARGUMENT in seen and capi.MSDA_OK in seen


# ---- the per-call entries: a sweep of their own ----
PTRS_FWD = ("value", "shapes", "lsi", "loc", "attn", "out")
PTRS_BWD = ("value", "shapes", "lsi", "loc", "attn", "gout", "gvalue", "gloc", "gattn")
BASE = dict(value=256, shapes=512, lsi=768, loc=1024, attn=1280, out=1536, gout=1536, gvalue=1792, gloc=2048,
            gattn=2304, N=2, S=100, M=8, D=48, L=3, Lq=10, P=4, vbs=0, step=64, flags=0)
PERTURB = {
    "D": (0, 8, 30, 40, 144, 32, 16, 128),
    "step": (0, -1, 3, 1, 2, 4),
    ("N", "step"): ((3, 2), (4, 3), (-1, 64)),
    "S": (0, -1),
    "M": (0, -2),
    ("L", "P"): ((0, 4), (65, 1), (3, 0), (64, 1)),
    "Lq": (-1,),
    "vbs": (-16, 4, 100 * 384 + 8),
}


def percall_cases(pointers, flag_sets):
    perturb = dict(PERTURB)
    perturb.update({k: (0, 257, 260, 264) for k in pointers})
    variants = [{}] + [dict(zip(k, v)) if isinstance(k, tuple) else {k: v} for k, vs in perturb.items() for v in vs]
    for N, Lq, flags in itertools.product((2, 0), (10, 0), flag_sets):
        for v in variants:
            yield {**BASE, "N": N, "Lq": Lq, "flags": flags, **v}


def _main_fwd(L, a):
    return L.msda_forward(*(a[k] for k in PTRS_FWD), a["N"], a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"], a["vbs"],
                          a["step"], BF16, None)


def _f16_fwd(L, a):
    return L.msda_f16_forward(*(a[k] for k in PTRS_FWD), a["N"], a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"],
                              a["vbs"], a["step"], None)


def _main_bwd(L, a):
    return L.msda_backward(*(a[k] for k in PTRS_BWD), a["N"], a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"],
                           a["vbs"], a["step"], BF16, a["flags"], None, 0, None)


def _f16_bwd(L, a):
    return L.msda_f16_backward(*(a[k] for k in PTRS_BWD), a["N"], a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"],
                               a["vbs"], a["step"], a["flags"], None)


@no_device_only
@pytest.mark.parametrize("entry", ["forward", "backward"])
def test_percall_statuses_equal_the_bf16_statuses(f16, entry):
    """NULL and misaligned pointers, im2col_step, D % 16, empty and negative sizes, strides and flags: whatever the
    main library answers for MSDA_DTYPE_BF16 without reaching the device, the fp16 entry answers too."""
    if entry == "forward":
        cases, main_fn, f16_fn = percall_cases(PTRS_FWD, (0,)), _main_fwd, _f16_fwd
    else:
        cases, main_fn, f16_fn = percall_cases(PTRS_BWD, (0, 1, 2, 3, 64)), _main_bwd, _f16_bwd
    main = capi.lib()
    made, diff, seen = 0, [], set()
    for a in cases:
        want = main_fn(main, a)
        if want == capi.MSDA_ERR_CUDA:      # validated and enqueued: never made on the fp16 library
            continue
        got = f16_fn(f16, a)
        made += 1
        seen.add(want)
        if got != want:
            diff.append((a, want, got))
    assert not diff, "%d of %d cases differ, e.g. %r (bf16 %d, fp16 %d)" % ((len(diff), made) + diff[0])
    assert made > 100
    assert {capi.MSDA_OK, capi.MSDA_ERR_INVALID_ARGUMENT, capi.MSDA_ERR_IM2COL_STEP,
            capi.MSDA_ERR_UNSUPPORTED_DTYPE} <= seen

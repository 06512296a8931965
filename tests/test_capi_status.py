"""Status codes of the validating C entry points, swept over a cross product of arguments and compared with a table
recorded from a known-good build (tests/golden/capi_status.json).

Every pointer passed here is fake (0, 256, 257, 260, 264), so only calls that are rejected before anything is
enqueued, or that have nothing to do, may ever run.  Without a device, a call that gets past validation returns
MSDA_ERR_CUDA; the table marks those cases '-' and the test never makes them.  The test skips itself when a device
is present, so that a validation bug cannot hand a fake pointer to a real GPU.

    python tests/test_capi_status.py --record    # rewrite the table from the library in this tree (CPU only)
"""
import hashlib
import itertools
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from snipper_b200 import capi  # noqa: E402

TABLE = os.path.join(ROOT, "tests", "golden", "capi_status.json")
F32, F64, BF16 = capi.MSDA_DTYPE_F32, capi.MSDA_DTYPE_F64, capi.MSDA_DTYPE_BF16
DTYPES = (F32, F64, BF16, 7)
BAD_PTRS = (0, 257, 260, 264)           # NULL, and 1-, 4- and 8-byte aligned
OPT_PTRS = (256, 257, 260, 264)         # values tried for pointers that may be NULL
FLAG_SETS = tuple(sum(f for i, f in enumerate((1, 2, 4, 8)) if bits >> i & 1) for bits in range(16)) + (64,)
MASKS = ((256, 384, 1), (257, 384, 1), (256, 386, 1), (256, 384, 2), (257, 1, 0), (256, -1, 0))


def sweep(base, axes, perturb):
    """Every combination of ``axes``, each with ``base`` as it is and with one argument of ``perturb`` changed."""
    variants = [{}] + [dict(zip(keys, vals)) if isinstance(keys, tuple) else {keys: vals}
                       for keys, options in perturb.items() for vals in options]
    names = list(axes)
    for combo in itertools.product(*axes.values()):
        for v in variants:
            yield {**base, **dict(zip(names, combo)), **v}


def _snippet_perturb(pointers, optional):
    p = {k: BAD_PTRS for k in pointers}
    p.update({k: OPT_PTRS for k in optional})
    p[("mask", "mrs", "mcs")] = MASKS
    p[("sn", "st")] = ((-16, 0), (0, -16), (0, 6), (6, 0), (2 * 100 * 384 + 4, 100 * 384))
    p[("rsn", "rst")] = ((-2, 0), (0, -2), (2, 3))
    p[("ors", "lrs")] = ((288, 288), (286, 96), (289, 288), (288, 95), (-1, 0))
    p["D"] = (40, 0, 144, 32)
    p[("L", "P")] = ((9, 4), (0, 4), (3, 0), (65, 1))
    p[("T2", "n_frame")] = ((4, 5), (4, 0), (0, 4), (3, 3))
    p["T1"] = (0, 6, 2)
    p["S"] = (0, -1, 1 << 20)
    p["M"] = (0, 7)
    return p


_SNIPPET_BASE = dict(value=256, shapes=256, lsi=256, offsets=256, logits=256, ref=256, N=1, T2=4, T1=4, n_frame=4,
                     S=100, M=8, D=48, L=3, Lq=10, P=4, sn=0, st=0, rsn=0, rst=0, ors=0, lrs=0, ob=None, lb=None,
                     vr=None, mask=None, mrs=0, mcs=0)
_SNIPPET_AXES = dict(flags=FLAG_SETS, dtype=DTYPES, N=(1, 0, -1), Lq=(10, 0, 100))


def _fwd(L, a):
    return L.msda_snippet_forward(a["value"], a["shapes"], a["lsi"], a["offsets"], a["logits"], a["ref"], a["out"],
                                  a["N"], a["T2"], a["T1"], a["n_frame"], a["S"], a["M"], a["D"], a["L"], a["Lq"],
                                  a["P"], a["sn"], a["st"], a["rsn"], a["rst"], a["ors"], a["lrs"], a["ob"], a["lb"],
                                  a["vr"], a["mask"], a["mrs"], a["mcs"], a["dtype"], a["flags"], None)


def _bwd(L, a):
    ws_bytes = a["ws_bytes"]
    if ws_bytes in ("need", "need-1"):
        ws_bytes = L.msda_snippet_backward_workspace_bytes(a["N"], a["T1"], a["n_frame"], a["S"], a["M"], a["D"],
                                                           a["L"], a["Lq"], a["P"], a["dtype"], a["flags"])
        ws_bytes -= ws_bytes > 0 and a["ws_bytes"] == "need-1"
    return L.msda_snippet_backward(a["value"], a["shapes"], a["lsi"], a["offsets"], a["logits"], a["ref"], a["gout"],
                                   a["gvalue"], a["goffsets"], a["glogits"], a["N"], a["T2"], a["T1"], a["n_frame"],
                                   a["S"], a["M"], a["D"], a["L"], a["Lq"], a["P"], a["sn"], a["st"], a["rsn"],
                                   a["rst"], a["ors"], a["lrs"], a["ob"], a["lb"], a["vr"], a["mask"], a["mrs"],
                                   a["mcs"], a["dtype"], a["flags"], a["ws"], ws_bytes, None)


def _frame_sum(L, a):
    return L.msda_frame_sum(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                            a["M"] * a["D"], a["sn"], a["st"], a["mrs"], a["mcs"], a["dtype"], None)


def _frame_unsum(L, a):
    return L.msda_frame_unsum(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                              a["M"] * a["D"], a["mrs"], a["mcs"], a["dtype"], None)


def _frame_sum_planar(L, a):
    return L.msda_frame_sum_planar(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                                   a["M"], a["D"], a["sn"], a["st"], a["mrs"], a["mcs"], a["dtype"], None)


def _frame_unsum_planar(L, a):
    return L.msda_frame_unsum_planar(a["value"], a["mask"], a["out"], a["N"], a["T2"], a["T1"], a["n_frame"], a["S"],
                                     a["M"], a["D"], a["mrs"], a["mcs"], a["dtype"], None)


_FRAME_BASE = dict(value=256, mask=None, out=256, N=1, T2=4, T1=4, n_frame=4, S=100, M=8, D=48, sn=0, st=0, mrs=0,
                   mcs=0)
_FRAME_AXES = dict(dtype=DTYPES, N=(1, 0, -1), D=(48, 32, 2, 3))
_FRAME_PERTURB = {"value": BAD_PTRS, "out": BAD_PTRS, ("mask", "mrs", "mcs"): MASKS,
                  ("sn", "st"): ((-16, 0), (0, -16), (0, 6), (6, 0)), ("T2", "n_frame"): ((4, 5), (4, 0), (0, 4)),
                  "T1": (0, 6), "S": (0, -1), "M": (0, 7)}


def _masked_zero(L, a):
    return L.msda_masked_zero(a["data"], a["mask"], a["n"], a["dtype"], None)


def _layer_tail(L, a):
    return L.msda_layer_tail(a["y"], a["bias"], a["residual"], a["gamma"], a["beta"], a["pos"], a["out"], a["out2"],
                             a["rows"], a["cols"], a["eps"], a["dtype"], None)


_TAIL_PTRS = ("y", "residual", "gamma", "beta", "out")

# name -> (function, cases); statuses are compared, the two size queries compare the byte counts they return
ENTRIES = {
    "msda_snippet_forward": (_fwd, lambda: sweep(
        dict(_SNIPPET_BASE, out=256), _SNIPPET_AXES,
        _snippet_perturb(("value", "shapes", "lsi", "offsets", "logits", "ref", "out"), ("ob", "lb", "vr")))),
    "msda_snippet_backward": (_bwd, lambda: sweep(
        dict(_SNIPPET_BASE, gout=256, gvalue=256, goffsets=256, glogits=256, ws=None, ws_bytes=0), _SNIPPET_AXES,
        {**_snippet_perturb(("value", "shapes", "lsi", "offsets", "logits", "ref", "gout", "gvalue", "goffsets",
                             "glogits"), ("ob", "lb", "vr")),
         ("ws", "ws_bytes"): ((256, "need"), (256, "need-1"), (257, "need"), (None, "need"))})),
    "msda_frame_sum": (_frame_sum, lambda: sweep(_FRAME_BASE, _FRAME_AXES, _FRAME_PERTURB)),
    "msda_frame_unsum": (_frame_unsum, lambda: sweep(_FRAME_BASE, _FRAME_AXES, _FRAME_PERTURB)),
    "msda_frame_sum_planar": (_frame_sum_planar, lambda: sweep(_FRAME_BASE, _FRAME_AXES, _FRAME_PERTURB)),
    "msda_frame_unsum_planar": (_frame_unsum_planar, lambda: sweep(_FRAME_BASE, _FRAME_AXES, _FRAME_PERTURB)),
    "msda_masked_zero": (_masked_zero, lambda: (
        dict(data=d, mask=m, n=n, dtype=t) for d in (256,) + BAD_PTRS for m in (256,) + BAD_PTRS
        for n in (16, 0, -1) for t in DTYPES)),
    "msda_layer_tail": (_layer_tail, lambda: sweep(
        dict(y=256, bias=None, residual=256, gamma=256, beta=256, pos=None, out=256, out2=None, rows=4, cols=384,
             eps=1e-5),
        dict(dtype=DTYPES, rows=(4, 0, -1), cols=(384, 128, 1024, 100, 2048, 0), eps=(1e-5, 0.0, -1.0)),
        {**{k: BAD_PTRS for k in _TAIL_PTRS}, "bias": OPT_PTRS, "pos": OPT_PTRS, "out2": OPT_PTRS,
         ("pos", "out2"): ((256, 256), (256, 260), (260, 256))})),
}
SIZE_QUERIES = {
    "msda_backward_workspace_bytes": lambda L: [
        L.msda_backward_workspace_bytes(N, 100, 8, 48, 3, Lq, 4, t, f)
        for N in (0, 1, 2) for Lq in (0, 10) for t in DTYPES for f in FLAG_SETS],
    "msda_snippet_backward_workspace_bytes": lambda L: [
        L.msda_snippet_backward_workspace_bytes(N, T1, nf, 100, 8, 48, 3, Lq, 4, t, f)
        for N in (0, 1, 2, -1) for T1, nf in ((4, 4), (6, 4), (2, 4), (0, 4), (4, 0)) for Lq in (0, 10, -1)
        for t in DTYPES for f in FLAG_SETS],
}


def _fingerprint(cases):
    """Pins the case list the table was recorded for: a changed sweep must be recorded again, not compared."""
    return hashlib.sha256(json.dumps(cases, sort_keys=True).encode()).hexdigest()[:16]


def record():
    if torch.cuda.is_available():
        sys.exit("--record calls every case, including those that reach the CUDA runtime: run it without a device")
    L = capi.lib()
    table = {}
    for name, (fn, cases) in ENTRIES.items():
        cases = list(cases())
        got = [fn(L, a) for a in cases]
        table[name] = dict(cases=len(cases), fingerprint=_fingerprint(cases),
                           status="".join("-" if s == capi.MSDA_ERR_CUDA else str(s) for s in got))
    for name, query in SIZE_QUERIES.items():
        table[name] = query(L)
    with open(TABLE, "w") as f:
        json.dump(table, f, indent=0)
        f.write("\n")
    for name, entry in table.items():
        if isinstance(entry, dict):
            print("%-26s %6d cases, %6d compared" % (name, entry["cases"], entry["cases"] - entry["status"].count("-")))


no_device_only = pytest.mark.skipif(torch.cuda.is_available(), reason="calls entry points with fake pointers")


@pytest.fixture(scope="module")
def table():
    with open(TABLE) as f:
        return json.load(f)


@no_device_only
@pytest.mark.parametrize("name", list(ENTRIES))
def test_status_matches_recorded_table(table, name):
    fn, cases = ENTRIES[name]
    cases = list(cases())
    want = table[name]
    assert (len(cases), _fingerprint(cases)) == (want["cases"], want["fingerprint"]), "case list changed: re-record"
    L = capi.lib()
    diff = [(a, int(s), fn(L, a)) for a, s in zip(cases, want["status"]) if s != "-"]
    diff = [d for d in diff if d[1] != d[2]]
    assert not diff, "%d cases differ, e.g. %r (recorded %d, got %d)" % ((len(diff),) + diff[0])


@no_device_only
@pytest.mark.parametrize("name", list(SIZE_QUERIES))
def test_workspace_sizes_match_recorded_table(table, name):
    assert SIZE_QUERIES[name](capi.lib()) == table[name]


@no_device_only
def test_backward_rejects_misaligned_logits_before_launching():
    L = capi.lib()
    base = dict(_SNIPPET_BASE, gout=256, gvalue=256, goffsets=256, glogits=256, ws=None, ws_bytes=0, flags=0, dtype=F32)
    for k in ("logits", "glogits"):
        for p in (257, 258):
            assert _bwd(L, dict(base, **{k: p})) == capi.MSDA_ERR_INVALID_ARGUMENT, (k, p)
    det = dict(base, flags=capi.MSDA_FLAG_PRESUMMED | capi.MSDA_FLAG_DETERMINISTIC, ws=256, ws_bytes="need")
    assert _bwd(L, dict(det, logits=258)) == capi.MSDA_ERR_INVALID_ARGUMENT
    assert _bwd(L, dict(det, glogits=258)) == capi.MSDA_ERR_INVALID_ARGUMENT


@no_device_only
def test_backward_validates_before_zero_filling_grad_value():
    """grad_value is zero-filled on the stream only once every pointer has passed: an invalid call enqueues nothing
    (without a device, an enqueued memset would fail with MSDA_ERR_CUDA instead)."""
    L = capi.lib()
    base = dict(_SNIPPET_BASE, gout=256, gvalue=256, goffsets=256, glogits=256, ws=None, ws_bytes=0, dtype=F32)
    for flags in (0, capi.MSDA_FLAG_PRESUMMED):
        for k, p in (("value", 264), ("value", 0), ("gout", 260), ("gvalue", 264), ("goffsets", 260), ("ref", 0)):
            assert _bwd(L, dict(base, flags=flags, **{k: p})) == capi.MSDA_ERR_INVALID_ARGUMENT, (flags, k, p)


if __name__ == "__main__":
    if sys.argv[1:] != ["--record"]:
        sys.exit(__doc__)
    record()

"""Which compiled kernel each input reaches: a table of cases, each naming the exact kernel instantiations it must
launch, generated from the host dispatch rules of csrc/ (restated below in Python).

The table is checked two ways.  tests/test_kernel_inventory.py (no GPU) asserts that the cases' expected kernels plus
UNREACHABLE are exactly the kernels compiled into libmsda_b200.so, so a new instantiation without a case fails on any
machine.  tests/test_dispatch_coverage_gpu.py runs every case, asserts that the profiler saw exactly the expected
kernels and compares the results with a float64 oracle.

Kernel names are written as ``family<template args>`` in c++filt's spelling, without ``void``, namespaces or the
parameter list (``normalise``).
"""
import os
import re
import shutil
import subprocess
from dataclasses import dataclass, field

# ---- the tile-size / strategy knobs (read from the environment once per process, csrc/msda_fast.cuh:406,
# msda_percall.cu:187, msda_snippet.cu:333, msda_planar.cu:616-628) ----
DEFAULT_KNOBS = dict(pairs_d48=16, snip_pairs_d48=16, planar_pairs=32, fwd_split=True, planar_tile2d=True)
KNOB_SETS = {
    "default": ({}, DEFAULT_KNOBS),
    # 32-query tiles, 64-query planar tiles, tile kernels for few-query forwards, row-segment planar tiles
    "A": ({"MSDA_PAIRS_D48": "32", "MSDA_SNIP_PAIRS_D48": "32", "MSDA_PLANAR_PAIRS": "64", "MSDA_FWD_SPLIT": "0",
           "MSDA_PLANAR_TILE2D": "0"},
          dict(pairs_d48=32, snip_pairs_d48=32, planar_pairs=64, fwd_split=False, planar_tile2d=False)),
    # 8-query tiles on every grid, 16-query planar tiles
    "B": ({"MSDA_PAIRS_D48": "8", "MSDA_SNIP_PAIRS_D48": "8", "MSDA_PLANAR_PAIRS": "16"},
          dict(pairs_d48=8, snip_pairs_d48=8, planar_pairs=16, fwd_split=True, planar_tile2d=True)),
    # the default tile lengths without the split forwards: few-query forwards take the 8-query tile kernels
    "C": ({"MSDA_FWD_SPLIT": "0"}, dict(DEFAULT_KNOBS, fwd_split=False)),
}

SM_CTAS = 148 * 3          # grids below this many 16-query tiles count as "few CTAs" (msda_fast.cuh:418)
SNIPPET_MAX_LP = 32        # kSnippetMaxLP (msda_snippet_common.cuh)

FAMILIES = (
    "msda_fwd_fast_kernel", "msda_bwd_fast_kernel", "msda_fwd_split_kernel", "msda_fwd_generic_kernel",
    "msda_bwd_generic_kernel", "msda_snippet_fwd_kernel", "msda_snippet_bwd_kernel", "msda_snippet_fwd_split_kernel",
    "msda_planar_fwd_kernel", "msda_planar_bwd_kernel", "snippet_loc_attn_kernel", "det_count_fill_kernel",
    "scan_tiles_kernel", "scan_blocksums_kernel", "scan_add_kernel", "det_reduce_kernel", "det_reduce_long_kernel",
    "frame_sum_kernel", "frame_unsum_kernel", "frame_sum_planar_kernel", "frame_unsum_planar_kernel",
    "masked_zero_kernel", "layer_tail_kernel",
)

# the two-pass grad_value of the deterministic mode (msda_deterministic.cu launch_deterministic_grad_value_f32)
DET_KERNELS = frozenset({"det_count_fill_kernel<false>", "det_count_fill_kernel<true>", "scan_tiles_kernel",
                         "scan_blocksums_kernel", "scan_add_kernel", "det_reduce_kernel", "det_reduce_long_kernel"})

_BF16_LANES = (2, 4, 6, 8, 12, 16)       # 16-byte bf16 lanes fast_path_ok / snippet_ok accept: D in {16,32,48,64,96,128}
UNREACHABLE = {
    "msda_fwd_fast_kernel<bf16q, 12, 16, 0>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_fwd_fast_kernel<bf16q, 12, 16, 768>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_snippet_fwd_kernel<bf16q, 12, 16, 0, 0>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_snippet_fwd_kernel<bf16q, 12, 16, 0, 1>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_snippet_fwd_kernel<bf16q, 12, 16, 0, 2>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_snippet_fwd_kernel<bf16q, 12, 16, 768, 0>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
    "msda_snippet_fwd_kernel<bf16q, 12, 16, 768, 2>":
        "bf16 D=48 takes 8-byte lanes only below 444 CTAs, where pick_pairs_d48 turns the tuned 16 into 8",
}
# the bf16 8-byte-lane builds reuse the fp32 lane switch (D/4 lanes), but bf16 is validated to D/8 in _BF16_LANES:
# D = 80 and D = 112 (20 and 28 lanes of 8 bytes) are rejected before any launch
for _ln, _pr in ((20, 16), (28, 16)):
    UNREACHABLE["msda_fwd_fast_kernel<bf16q, %d, %d, 0>" % (_ln, _pr)] = \
        "bf16 needs D/8 in {2,4,6,8,12,16} (fast_path_ok): D = %d is rejected" % (4 * _ln)
    UNREACHABLE["msda_bwd_fast_kernel<bf16q, %d, %d, 0, true>" % (_ln, _pr)] = \
        "bf16 needs D/8 in {2,4,6,8,12,16} (fast_path_ok): D = %d is rejected" % (4 * _ln)
for _ln in (20, 28):
    for _mode in (0, 1, 2):
        UNREACHABLE["msda_snippet_fwd_kernel<bf16q, %d, 8, 0, %d>" % (_ln, _mode)] = \
            "bf16 needs D/8 in {2,4,6,8,12,16} (snippet_ok): D = %d is rejected" % (4 * _ln)
        UNREACHABLE["msda_snippet_bwd_kernel<bf16q, %d, 8, 0, %d, true>" % (_ln, _mode)] = \
            "bf16 needs D/8 in {2,4,6,8,12,16} (snippet_ok): D = %d is rejected" % (4 * _ln)


def normalise(name):
    """A demangled kernel name (c++filt or the profiler) -> ``family<args>``: no ``void``, namespaces or parameters."""
    name = name.strip()
    if name.startswith("void "):
        name = name[5:]
    name = name.replace("(anonymous namespace)::", "").replace("msda::", "")
    depth = 0
    for i, ch in enumerate(name):       # cut at the parameter list: the first '(' outside the template arguments
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            name = name[:i]
            break
    return re.sub(r"\s+", " ", name).strip()


def family(name):
    return name.split("<", 1)[0]


# ------------------------------------------------------------------------------------------
# the dispatch rules of csrc/, restated
# ------------------------------------------------------------------------------------------
def pick_pairs_d48(configured, Lq, M, nz):
    if configured != 16:
        return configured
    return 8 if (Lq + 15) // 16 * M * nz < SM_CTAS else 16


def few_ctas(Lq, M, nz):
    return (Lq + 15) // 16 * M * nz < SM_CTAS


def _percall_pairs(lanes, g, k):
    return pick_pairs_d48(k["pairs_d48"], g["Lq"], g["M"], g["N"]) if lanes == 12 else 16


def _snip_pairs(lanes, g, k):
    if lanes == 12:
        return pick_pairs_d48(k["snip_pairs_d48"], g["Lq"], g["M"], g["N"] * g["T1"])
    return 16 if lanes in (4, 8, 16) else 8


def _csb(vt, lanes, g, masked=False):
    """immediate cell stride: 48-channel lanes and M*D == 384 (snipper_csb / snip_csb); never with the mask"""
    n = {"float": 4, "bf16q": 4, "__nv_bfloat16": 8}[vt]
    if masked or lanes * n != 48 or g["M"] * g["D"] != 384:
        return 0
    return 384 * (4 if vt == "float" else 2)


def percall_fast_ok(g, esize):
    """fast_path_ok (msda_percall.cu:306) for the geometries the cases use (aligned, small)"""
    D = g["D"]
    epl = 16 // esize
    if D % epl:
        return False
    lanes = D // epl
    if lanes % 2 or lanes > 32 or (esize == 4 and lanes % 4) or (esize == 2 and lanes not in _BF16_LANES):
        return False
    return g["L"] * g["P"] < 4096


def _split_fwd(vt, g, k):
    """launch_fwd_split: D = 48 forwards of few CTAs -> one CTA per (query, head)"""
    LP = g["L"] * g["P"]
    if k["fwd_split"] and g["D"] == 48 and few_ctas(g["Lq"], g["M"], g["N"]):
        return "msda_fwd_split_kernel<%s, 12, %d>" % (vt, 160 if LP * 12 <= 160 else 384)
    return None


def percall_forward(dtype, g, k):
    if dtype == "f64":
        return {"msda_fwd_generic_kernel<double>"}
    if dtype == "f32":
        if not percall_fast_ok(g, 4):
            return {"msda_fwd_generic_kernel<float>"}
        s = _split_fwd("float", g, k)
        if s:
            return {s}
        lanes = g["D"] // 4
        return {"msda_fwd_fast_kernel<float, %d, %d, %d>" % (lanes, _percall_pairs(lanes, g, k), _csb("float", lanes, g))}
    assert percall_fast_ok(g, 2)
    s = _split_fwd("bf16q", g, k)
    if s:
        return {s}
    if few_ctas(g["Lq"], g["M"], g["N"]):
        lanes = g["D"] // 4
        return {"msda_fwd_fast_kernel<bf16q, %d, %d, %d>" % (lanes, _percall_pairs(lanes, g, k), _csb("bf16q", lanes, g))}
    lanes = g["D"] // 8
    return {"msda_fwd_fast_kernel<__nv_bfloat16, %d, 16, %d>" % (lanes, _csb("__nv_bfloat16", lanes, g))}


def percall_backward(dtype, g, k, deterministic=False, fast=True):
    if dtype == "f64":
        return {"msda_bwd_generic_kernel<double>"}
    vt = "float" if dtype == "f32" else "bf16q"
    if not (fast and percall_fast_ok(g, 4 if dtype == "f32" else 2)):
        assert dtype == "f32"
        return {"msda_bwd_generic_kernel<float>"} | (DET_KERNELS if deterministic else set())
    lanes = g["D"] // 4
    name = "msda_bwd_fast_kernel<%s, %d, %d, %d, %s>" % (vt, lanes, _percall_pairs(lanes, g, k), _csb(vt, lanes, g),
                                                        "false" if deterministic else "true")
    return {name} | (DET_KERNELS if deterministic else set())


def snippet_forward(dtype, mode, g, k):
    """mode: direct, masked, presummed (fp32 or bf16 cell-major value / slots)"""
    kmode = {"direct": 0, "masked": 1, "presummed": 2}[mode]
    lanes = g["D"] // 4
    LP = g["L"] * g["P"]
    if dtype == "f32":
        if (mode != "presummed" and g["D"] == 48 and k["fwd_split"] and
                pick_pairs_d48(k["snip_pairs_d48"], g["Lq"], g["M"], g["N"] * g["T1"]) == 8):
            return {"msda_snippet_fwd_split_kernel<12, %d, %d>" % (160 if LP * 12 <= 160 else 12 * SNIPPET_MAX_LP, kmode)}
        vt = "float"
    elif few_ctas(g["Lq"], g["M"], g["N"] * g["T1"]):
        vt = "bf16q"
    else:
        lanes = g["D"] // 8
        return {"msda_snippet_fwd_kernel<__nv_bfloat16, %d, %d, %d, %d>" % (
            lanes, 8 if lanes == 16 else 16, _csb("__nv_bfloat16", lanes, g, mode == "masked"), kmode)}
    return {"msda_snippet_fwd_kernel<%s, %d, %d, %d, %d>" % (vt, lanes, _snip_pairs(lanes, g, k),
                                                            _csb(vt, lanes, g, mode == "masked"), kmode)}


def snippet_backward(dtype, mode, g, k, scatter=True):
    kmode = {"direct": 0, "masked": 1, "presummed": 2}[mode]
    vt = "float" if dtype == "f32" else "bf16q"
    lanes = g["D"] // 4
    csb = _csb(vt, lanes, g, mode == "masked") if scatter else 0
    return {"msda_snippet_bwd_kernel<%s, %d, %d, %d, %d, %s>" % (vt, lanes, _snip_pairs(lanes, g, k), csb, kmode,
                                                                "true" if scatter else "false")}


def expected_kernels(case, knobs):
    """The exact set of library kernels ``case`` launches under ``knobs`` (a KNOB_SETS value)."""
    e, dt, g = case.entry, case.dtype, case.geom
    T = {"f32": "float", "bf16": "__nv_bfloat16"}.get(dt)
    if e == "fwd":
        return frozenset(percall_forward(dt, g, knobs))
    if e == "bwd":
        return frozenset(percall_backward(dt, g, knobs))
    if e == "bwd_det":
        return frozenset(percall_backward(dt, g, knobs, deterministic=True, fast=not g.get("offset_views")))
    if e in ("direct", "masked"):
        return frozenset(snippet_forward(dt, e, g, knobs) | snippet_backward(dt, e, g, knobs))
    if e == "presummed":
        return frozenset(snippet_forward(dt, e, g, knobs) | snippet_backward(dt, e, g, knobs) |
                         {"frame_sum_kernel<%s>" % T, "frame_unsum_kernel<%s>" % T})
    if e == "deterministic":
        return frozenset(snippet_forward(dt, "presummed", g, knobs) | snippet_backward(dt, "presummed", g, knobs, False) |
                         {"frame_sum_kernel<float>", "frame_unsum_kernel<float>", "snippet_loc_attn_kernel"} |
                         DET_KERNELS)
    if e == "planar":
        p = knobs["planar_pairs"]
        return frozenset({"msda_planar_fwd_kernel<%d>" % p, "msda_planar_bwd_kernel<%d>" % p,
                          "frame_sum_planar_kernel", "frame_unsum_planar_kernel"})
    if e == "masked_zero":
        return frozenset({"masked_zero_kernel<%s>" % T})
    if e == "layer_tail":
        return frozenset({"layer_tail_kernel<%d>" % (g["C"] // 128)})
    raise ValueError(e)


# ------------------------------------------------------------------------------------------
# the cases
# ------------------------------------------------------------------------------------------
@dataclass
class Case:
    id: str
    entry: str      # fwd, bwd, bwd_det (per call); direct, masked, presummed, planar, deterministic (fused fwd + bwd);
                    # masked_zero, layer_tail
    dtype: str      # f32, bf16, f64
    geom: dict = field(default_factory=dict)
    seed: int = 0

    def expected(self, knob_set="default"):
        return expected_kernels(self, KNOB_SETS[knob_set][1])


# level pyramids with the edges bilinear sampling gets wrong: one-pixel-wide and one-pixel-high levels, odd widths
_PYRAMIDS = [
    [(3, 5), (1, 7), (6, 1), (2, 3), (5, 9)],
    [(7, 1), (4, 5), (1, 1), (3, 7), (2, 9)],
    [(5, 3), (2, 1), (1, 6), (9, 5), (3, 3)],
]
# (L, P): L*P on both sides of the per-call sample chunk (32, or 16 at 32-query tiles), of the split kernels' 160-thread
# block (L*P*12 <= 160) and, per call, above 32 (several lp0 passes; the split kernels' `sp += SLOTS` loop)
_PERCALL_LP = [(2, 2), (3, 4), (4, 4), (3, 11), (1, 1), (5, 7)]
# fused ops: L*P <= 32; 32 is their limit and crosses the opt-in shared-memory size at 32-query tiles
_FUSED_LP = [(2, 2), (3, 4), (4, 8), (1, 3), (2, 7), (4, 8)]
_F32_D = (16, 32, 48, 64, 80, 96, 112, 128)
_BF16_D = (16, 32, 48, 64, 96, 128)


def _heads(D, imm):
    if imm:
        return 384 // D
    return 4 if D == 48 else (2 if D <= 96 else 1)


def _queries(M, nz, big, i):
    """few CTAs: 1 or k*32 + 1 queries (partial last tile at 8, 16 and 32 queries per tile); many: the smallest
    k*32 + 1 with at least 444 16-query tiles"""
    if not big:
        return (1, 33, 65, 17)[i % 4]
    tiles = -(-SM_CTAS // (M * nz))
    return 32 * (-(-tiles // 2)) + 1


def _geom(entry, D, imm, big, i, fused):
    M = _heads(D, imm)
    L, P = (_FUSED_LP if fused else _PERCALL_LP)[i % 6]
    if big:
        L, P = (2, 2) if i % 2 == 0 else (1, 3)     # many queries: keep the float64 oracle cheap
    if (M * L * P) % 2:                             # the packed projection row is read as float2
        P += 1
    shapes = _PYRAMIDS[i % 3][:L]
    g = dict(D=D, M=M, L=L, P=P, shapes=shapes, S=sum(h * w for h, w in shapes))
    if fused:
        n_frame, fut = ((1, 0), (2, 1), (3, 0), (2, 0))[i % 4]
        N = 1 if big else 1 + i % 2
        g.update(N=N, n_frame=n_frame, T2=n_frame + (1 if fut and i % 3 == 0 else 0), T1=n_frame + fut,
                 strided=i % 2 == 1, pixel_mask=i % 2 == 0)
        nz = N * g["T1"]
    else:
        N = 2 if i % 2 else 1
        g.update(N=N, strided=N > 1)
        nz = N
    g["Lq"] = _queries(M, nz, big, i)
    assert few_ctas(g["Lq"], M, nz) != big
    return g


def _rule_cases():
    cases = []
    i = 0
    for entry in ("fwd", "bwd", "bwd_det", "direct", "masked", "presummed", "deterministic", "planar"):
        fused = entry not in ("fwd", "bwd", "bwd_det")
        for dtype in ("f32", "bf16"):
            if dtype == "bf16" and entry in ("bwd_det", "deterministic", "planar"):
                continue
            for D in ((48,) if entry == "planar" else (_F32_D if dtype == "f32" else _BF16_D)):
                for big in (False, True):
                    for imm in ((False, True) if D == 48 else (False,)):
                        g = _geom(entry, D, imm, big, i, fused)
                        cid = "%s-%s-D%d-%s-%s" % (entry, dtype, D, "many" if big else "few", "imm" if imm else "rt")
                        cases.append(Case(cid, entry, dtype, g, seed=i))
                        i += 1
    # the generic kernels: channel counts off the vector lanes, and float64
    for entry in ("fwd", "bwd", "bwd_det"):
        g = _geom(entry, 30, False, False, i, False)
        cases.append(Case("%s-f32-D30-generic" % entry, entry, "f32", g, seed=i))
        i += 1
    for entry in ("fwd", "bwd"):
        g = _geom(entry, 48, True, False, i, False)
        cases.append(Case("%s-f64-D48" % entry, entry, "f64", g, seed=i))
        i += 1
    # deterministic per call with 4-byte (not 16-byte) aligned grad_output / grad_value views: the scalar ordered
    # reduce (det_reduce_kernel vec = 0), reached through the C ABI
    g = _geom("bwd_det", 48, True, False, i, False)
    g["offset_views"] = True
    cases.append(Case("bwd_det-f32-D48-offset-views", "bwd_det", "f32", g, seed=i))
    i += 1
    # deterministic per call adding into a non-zero grad_value (MSDA_FLAG_ACCUMULATE_VALUE)
    g = _geom("bwd_det", 48, False, False, i, False)
    g["accumulate"] = True
    cases.append(Case("bwd_det-f32-D48-accumulate", "bwd_det", "f32", g, seed=i))
    i += 1
    for dtype in ("f32", "bf16"):
        cases.append(Case("masked_zero-%s" % dtype, "masked_zero", dtype, dict(numel=4099), seed=i))
        i += 1
    for v in range(1, 9):
        cases.append(Case("layer_tail-C%d" % (128 * v), "layer_tail", "f32", dict(C=128 * v, rows=37), seed=i))
        i += 1
    return cases


CASES = _rule_cases()


def knob_cases(knob_set):
    """The cases a knob set can move: everything at 48 channels per head (the only tunable tile length) and the planar
    kernels.  Same ids, geometries and seeds as the default cases, so their outputs compare one to one."""
    return [c for c in CASES if c.geom.get("D") == 48 and c.dtype != "f64" and not c.geom.get("offset_views")
            and not c.geom.get("accumulate")]


def covered(knob_sets=KNOB_SETS):
    """Every kernel some case launches under some knob set."""
    out = set()
    for ks in knob_sets:
        for c in (CASES if ks == "default" else knob_cases(ks)):
            out |= c.expected(ks)
    return out


def missing_tools():
    """The binary tools compiled_kernels needs that are not on PATH (cuobjdump is also looked for next to nvcc)."""
    return [t for t in ("cuobjdump", "c++filt") if _tool(t) is None]


def _tool(name):
    exe = shutil.which(name)
    if exe is None and name == "cuobjdump" and os.path.exists("/usr/local/cuda/bin/cuobjdump"):
        exe = "/usr/local/cuda/bin/cuobjdump"
    return exe


def compiled_kernels(lib_path=None):
    """Normalised names of every kernel compiled into the library (cuobjdump -symbols | c++filt), or None when one of
    the two tools is missing."""
    if missing_tools():
        return None
    if lib_path is None:
        from snipper_b200.build import LIB_PATH as lib_path
    syms = subprocess.run([_tool("cuobjdump"), "-symbols", lib_path], capture_output=True, text=True, check=True).stdout
    entries = [line.split()[-1] for line in syms.splitlines() if "STT_FUNC" in line and "STO_ENTRY" in line]
    demangled = subprocess.run([_tool("c++filt")], input="\n".join(entries), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    return {normalise(n) for n in demangled}

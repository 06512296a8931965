"""The dispatch case table (tests/dispatch_cases.py) against the kernels actually compiled into libmsda_b200.so: every
instantiation is either launched by some case or listed as unreachable with a reason, and none is both.  No GPU needed:
a new instantiation without a case fails here on any machine with the CUDA binary tools."""
import pytest

import dispatch_cases as dc


@pytest.fixture(scope="module")
def inventory():
    missing = dc.missing_tools()
    if missing:
        pytest.skip("%s not found: cannot list the kernels of the library" % " and ".join(missing))
    from snipper_b200.build import build_library
    return dc.compiled_kernels(build_library())


def test_normalise_matches_both_spellings():
    assert dc.normalise("void msda::msda_fwd_fast_kernel<msda::bf16q, 12, 32, 768>(__nv_bfloat16 const*, long const*, "
                        "msda::FastArgs)") == "msda_fwd_fast_kernel<bf16q, 12, 32, 768>"
    assert dc.normalise("void msda::(anonymous namespace)::msda_planar_fwd_kernel<64>(char const*, long const*)") == \
        "msda_planar_fwd_kernel<64>"
    assert dc.normalise("msda::scan_tiles_kernel(int const*, int*, int*, long)") == "scan_tiles_kernel"


def test_every_compiled_kernel_has_a_case_or_a_reason(inventory):
    covered = dc.covered()
    unreachable = set(dc.UNREACHABLE)
    assert inventory, "no kernel symbols found in the library"
    assert not sorted(inventory - covered - unreachable), "compiled, but no case launches it and no reason says why"
    assert not sorted(covered - inventory), "a case expects a kernel the library does not contain"
    assert not sorted(unreachable - inventory), "UNREACHABLE names a kernel the library does not contain"
    assert not sorted(covered & unreachable), "listed as unreachable, yet a case launches it"
    assert {dc.family(n) for n in inventory} == set(dc.FAMILIES)


def test_every_knob_set_moves_some_kernel():
    """Each knob child reaches instantiations the default knobs do not (otherwise it tests nothing new)."""
    base = dc.covered(["default"])
    for ks in ("A", "B", "C"):
        assert dc.covered([ks]) - base, ks


def test_cases_sit_on_both_sides_of_the_thresholds():
    few = [c for c in dc.CASES if "Lq" in c.geom and dc.few_ctas(c.geom["Lq"], c.geom["M"], c.geom["N"] * c.geom.get("T1", 1))]
    many = [c for c in dc.CASES if "Lq" in c.geom and c not in few]
    assert few and many
    lqs = {c.geom["Lq"] for c in dc.CASES if "Lq" in c.geom}
    assert 1 in lqs and all(q % 8 == 1 for q in lqs)           # a partial last tile at 8, 16 and 32 queries per tile
    lp = {c.geom["L"] * c.geom["P"] for c in dc.CASES if "L" in c.geom}
    assert min(lp) * 12 <= 160 < max(lp) * 12 and max(lp) > 32   # split block sizes; several per-call sample passes
    fused_lp = {c.geom["L"] * c.geom["P"] for c in dc.CASES if c.entry in ("direct", "masked", "presummed", "planar")}
    assert max(fused_lp) == 32

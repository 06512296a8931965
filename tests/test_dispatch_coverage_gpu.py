"""Every case of tests/dispatch_cases.py on the GPU: the profiler must see exactly the kernel instantiations the case
names, and the results must match a float64 oracle.  The tile-size knobs are read once per process, so each knob set
runs in a child process of its own; the children's forward outputs are then compared with this process's.

Tolerances (rel_err = max |got - ref| / max |ref| per tensor, as in conftest.py):
  fp32 forward 1e-5, every fp32 gradient 1e-4;
  bf16 forward and bf16 grad_value (fp32 sums rounded once to bf16):  |got - ref| <= 2^-8 |ref| + 1e-5 max|ref|;
  bf16-mode fp32 gradients 1e-4 (computed in fp32 from exactly representable inputs), except on the pre-summed path,
  whose neighbour-frame slot sums are themselves stored in bf16: its output and gradients carry bf16-level error, 1e-2.
"""
import json
import os
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from conftest import level_start_index, rel_err  # noqa: E402
import dispatch_cases as dc  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f64": torch.float64}


# ------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------
def _percall_inputs(c):
    g = c.geom
    gen = torch.Generator().manual_seed(1000 + c.seed)
    shapes = torch.as_tensor(g["shapes"], dtype=torch.long)
    N, S, M, D, L, P, Lq = g["N"], g["S"], g["M"], g["D"], g["L"], g["P"], g["Lq"]
    dt = _DT[c.dtype]
    value = torch.randn(N, S, M, D, generator=gen).to(dt)
    loc = 0.5 + (torch.rand(N, Lq, M, L, P, 2, generator=gen) - 0.5) * 4.0     # a share falls outside [0,1]
    attn = torch.softmax(torch.randn(N, Lq, M, L * P, generator=gen), -1).view(N, Lq, M, L, P)
    go = torch.randn(N, Lq, M * D, generator=gen).to(dt)
    if c.dtype == "f64":
        loc, attn = loc.double(), attn.double()
    return dict(value=value, shapes=shapes, lsi=level_start_index(shapes), loc=loc, attn=attn, grad_out=go)


def _fused_inputs(c):
    g = c.geom
    gen = torch.Generator().manual_seed(2000 + c.seed)
    shapes = torch.as_tensor(g["shapes"], dtype=torch.long)
    N, T1, T2, S, M, D, L, P, Lq = g["N"], g["T1"], g["T2"], g["S"], g["M"], g["D"], g["L"], g["P"], g["Lq"]
    mlp = M * L * P
    value = torch.randn(N, T2, S, M, D, generator=gen).to(_DT[c.dtype])
    proj = torch.cat((torch.randn(N, T1, Lq, 2 * mlp, generator=gen) * 2.0,
                      torch.randn(N, T1, Lq, mlp, generator=gen)), -1)
    ob, lb = torch.randn(2 * mlp, generator=gen), torch.randn(mlp, generator=gen)
    ref = torch.rand(N, T1, Lq, L, 2, generator=gen) * 1.2 - 0.1
    go = torch.randn(N, T1, Lq, M * D, generator=gen).to(_DT[c.dtype])
    mask = None
    if c.entry == "masked" or (c.entry in ("presummed", "planar", "deterministic") and c.seed % 2 == 0):
        if g["pixel_mask"]:
            mask = torch.rand(N, T2, S, generator=gen) < 0.2
        else:
            mask = torch.rand(N, T2, S, M * D, generator=gen) < 0.2
    return dict(value=value, shapes=shapes, lsi=level_start_index(shapes), proj=proj, ob=ob, lb=lb, ref=ref,
                grad_out=go, mask=mask)


# ------------------------------------------------------------------------------------------
# running a case: returns (launched kernels, forward output, [(name, got, want, kind)], extra failures)
# ------------------------------------------------------------------------------------------
def _launched(fn):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    names, device_events = set(), 0
    for e in prof.events():
        if e.device_type == DeviceType.CUDA:
            device_events += 1
        for name in [e.name] + [k.name for k in getattr(e, "kernels", [])]:
            n = dc.normalise(name)
            if dc.family(n) in dc.FAMILIES:
                names.add(n)
    assert device_events > 0, "the profiler recorded no device activity: the kernel check would pass vacuously"
    return names, result


def _run_percall(c):
    from snipper_b200 import capi, ops
    from oracle import c_oracle
    x = _percall_inputs(c)
    d = {k: v.to(DEV) for k, v in x.items()}
    v = d["value"]
    if c.geom["N"] > 1:             # value[:, t] of a frame-stacked tensor: batch stride != S*M*D
        big = torch.zeros(v.shape[0], 2, *v.shape[1:], dtype=v.dtype, device=DEV)
        big[:, 1] = v
        v = big[:, 1]
    args = (v, d["shapes"], d["lsi"], d["loc"], d["attn"])
    o64 = (x["value"].double(), x["shapes"], x["lsi"], x["loc"].double(), x["attn"].double())
    checks, extra = [], []
    if c.entry == "fwd":
        launched, out = _launched(lambda: torch.ops.snipper_b200.msda_forward(*args, 64))
        checks.append(("output", out, c_oracle.forward(*o64), "out"))
        return launched, out, checks, extra
    want = c_oracle.backward(*o64, x["grad_out"].double())
    if c.entry == "bwd":
        launched, got = _launched(lambda: torch.ops.snipper_b200.msda_backward(*args, d["grad_out"], 64, False))
    elif not (c.geom.get("offset_views") or c.geom.get("accumulate")):
        launched, got = _launched(lambda: torch.ops.snipper_b200.msda_backward(*args, d["grad_out"], 64, True))
        again = torch.ops.snipper_b200.msda_backward(*args, d["grad_out"], 64, True)
        if not all(torch.equal(a, b) for a, b in zip(got, again)):
            extra.append("deterministic backward differs between two runs")
    else:
        # through the C ABI: grad_output / grad_value 4 bytes past a 16-byte boundary, or accumulated into
        N, S, M, D, L, P, Lq = (c.geom[k] for k in ("N", "S", "M", "D", "L", "P", "Lq"))
        nv, ng = N * S * M * D, N * Lq * M * D
        flags = capi.MSDA_FLAG_DETERMINISTIC
        if c.geom.get("offset_views"):
            gv_buf = torch.zeros(nv + 4, device=DEV)
            gv = gv_buf[1:1 + nv]
            go_buf = torch.zeros(ng + 4, device=DEV)
            go_buf[1:1 + ng] = d["grad_out"].flatten()
            go = go_buf[1:1 + ng]
            assert gv.data_ptr() % 16 == 4 and go.data_ptr() % 16 == 4
            g0 = torch.zeros(nv, dtype=torch.float64)
        else:
            flags |= capi.MSDA_FLAG_ACCUMULATE_VALUE
            g0 = torch.randn(nv, generator=torch.Generator().manual_seed(c.seed), dtype=torch.float64)
            gv = g0.float().to(DEV)
            g0 = g0.float().double()
            go = d["grad_out"]
        gl, ga = torch.empty_like(d["loc"]), torch.empty_like(d["attn"])
        ws_bytes = capi.lib().msda_backward_workspace_bytes(N, S, M, D, L, Lq, P, capi.MSDA_DTYPE_F32, flags)
        ws, ws_ptr = ops._workspace(ws_bytes, torch.device(DEV))

        def call():
            st = capi.lib().msda_backward(
                v.data_ptr(), d["shapes"].data_ptr(), d["lsi"].data_ptr(), d["loc"].data_ptr(), d["attn"].data_ptr(),
                go.data_ptr(), gv.data_ptr(), gl.data_ptr(), ga.data_ptr(), N, S, M, D, L, Lq, P, v.stride(0), 64,
                capi.MSDA_DTYPE_F32, flags, ws_ptr, ws_bytes, torch.cuda.current_stream().cuda_stream)
            capi.check(st, "msda_backward")
            return gv.clone().view(N, S, M, D), gl, ga

        launched, got = _launched(call)
        want = (want[0] + g0.view(want[0].shape),) + tuple(want[1:])
    for name, a, b in zip(("grad_value", "grad_loc", "grad_attn"), got, want):
        checks.append((name, a, b, "value" if name == "grad_value" else "grad"))
    return launched, None, checks, extra


def _run_fused(c):
    from snipper_b200 import ops
    from snippet_oracle import snippet_attention_oracle
    x = _fused_inputs(c)
    g = c.geom
    N, T2, S, M, D = x["value"].shape
    mask = x["mask"]
    # the oracle: glue in fp32 in the kernel's order (same floor() cells), the gather and its gradients in float64
    leaves = [x["value"].double().requires_grad_(True)] + [t.clone().requires_grad_(True)
                                                          for t in (x["proj"], x["ob"], x["lb"], x["ref"])]
    vo = leaves[0]
    if mask is not None:
        m5 = mask[..., None, None] if mask.dim() == 3 else mask.view(N, T2, S, M, D)
        vo = vo.masked_fill(m5, 0.0)
    want_out = snippet_attention_oracle(vo, None, x["shapes"], x["lsi"], *leaves[1:], g["n_frame"])
    want_out.backward(x["grad_out"].double())
    want = [want_out.detach()] + [t.grad for t in leaves]

    d = {k: (v.to(DEV) if v is not None else None) for k, v in x.items()}

    def run():
        v = d["value"]
        if g["strided"]:            # value[:, :T2] of a longer clip: batch stride != T2*S*M*D
            big = torch.zeros(N, T2 + 1, S, M, D, dtype=v.dtype, device=DEV)
            big[:, :T2] = v
            v = big[:, :T2]
        lv = [v.detach().requires_grad_(True)] + [d[k].clone().requires_grad_(True) for k in ("proj", "ob", "lb", "ref")]
        ops.set_planar_slots(c.entry == "planar")
        ops.set_deterministic(c.entry == "deterministic")
        try:
            out = ops.snippet_attention(lv[0], d["mask"], d["shapes"], d["lsi"], lv[1], lv[2], lv[3], lv[4],
                                        g["n_frame"], presum=c.entry in ("presummed", "planar", "deterministic"))
            out.backward(d["grad_out"])
        finally:
            ops.set_planar_slots(False)
            ops.set_deterministic(False)
        return [out.detach()] + [t.grad for t in lv]

    launched, got = _launched(run)
    extra = []
    if c.entry == "deterministic":
        again = run()
        if not all(torch.equal(a, b) for a, b in zip(got, again)):
            extra.append("deterministic fused op differs between two runs")
    if mask is not None:
        gv = got[1].float().cpu()
        m5 = mask[..., None, None].expand(N, T2, S, M, D) if mask.dim() == 3 else mask.view(N, T2, S, M, D)
        if m5.any() and float(gv[m5].abs().max()) != 0.0:
            extra.append("grad_value is not zero on masked elements")
    names = ("output", "grad_value", "grad_proj", "grad_offsets_bias", "grad_logits_bias", "grad_reference_points")
    kinds = ("out", "value", "grad", "grad", "grad", "grad")
    checks = [(n, a, b, k) for n, a, b, k in zip(names, got, want, kinds)]
    return launched, got[0], checks, extra


def _run_misc(c):
    from snipper_b200 import ops
    gen = torch.Generator().manual_seed(3000 + c.seed)
    if c.entry == "masked_zero":
        data = torch.randn(c.geom["numel"], generator=gen).to(_DT[c.dtype])
        mask = torch.rand(c.geom["numel"], generator=gen) < 0.3
        dd, md = data.to(DEV), mask.to(DEV)
        launched, _ = _launched(lambda: ops.masked_zero_(dd, md))
        extra = [] if torch.equal(dd.cpu(), data.masked_fill(mask, 0)) else ["masked_zero_ result differs"]
        return launched, None, [], extra
    C, rows = c.geom["C"], c.geom["rows"]
    y, res, pos = (torch.randn(rows, C, generator=gen) for _ in range(3))
    bias, gamma, beta = (torch.randn(C, generator=gen) for _ in range(3))
    dv = [t.to(DEV) for t in (y, bias, res, gamma, beta, pos)]
    with torch.no_grad():
        launched, (out, out_pos) = _launched(lambda: ops.layer_tail(dv[0], dv[1], dv[2], dv[3], dv[4], dv[5], 1e-5))
    ref = torch.nn.functional.layer_norm((res + y + bias).double(), (C,), gamma.double(), beta.double(), 1e-5)
    return launched, out, [("output", out, ref, "grad"), ("output+pos", out_pos, ref + pos.double(), "grad")], []


def _tolerance_failures(c, checks):
    bf16 = c.dtype == "bf16"
    presum_bf16 = bf16 and c.entry == "presummed"
    fails = []
    for name, got, want, kind in checks:
        got = got.detach().double().cpu()
        want = want.detach().double().cpu()
        if got.shape != want.shape:
            got = got.reshape(want.shape)
        if presum_bf16:
            err, ok = rel_err(got, want), rel_err(got, want) < 1e-2
        elif bf16 and kind in ("out", "value"):
            bound = 2.0 ** -8 * want.abs() + 1e-5 * float(want.abs().max())
            err = float(((got - want).abs() - bound).max())
            ok = err <= 0.0
        else:
            tol = 1e-5 if kind == "out" else 1e-4
            err = rel_err(got, want)
            ok = err < tol
        if not ok:
            fails.append("%s: error %.3g" % (name, err))
    return fails


def run_case(c, knob_set="default"):
    """-> dict(id, ok, failures, launched, expected) and the forward output (CPU) or None"""
    if c.entry in ("fwd", "bwd", "bwd_det"):
        launched, out, checks, extra = _run_percall(c)
    elif c.entry in ("masked_zero", "layer_tail"):
        launched, out, checks, extra = _run_misc(c)
    else:
        launched, out, checks, extra = _run_fused(c)
    expected = set(c.expected(knob_set))
    fails = list(extra)
    if launched != expected:
        fails.append("launched %s, expected %s" % (sorted(launched), sorted(expected)))
    fails += _tolerance_failures(c, checks)
    res = dict(id=c.id, ok=not fails, failures=fails, launched=sorted(launched), expected=sorted(expected))
    return res, (out.detach().cpu() if out is not None else None)


# ------------------------------------------------------------------------------------------
# default knobs, in this process
# ------------------------------------------------------------------------------------------
_OBSERVED = {}          # knob set -> kernels seen launched
_DEFAULT_OUT = {}       # case id -> forward output under the default knobs
_RAN = {}


@pytest.fixture(scope="module", autouse=True)
def _no_knobs_here():
    for env in dc.KNOB_SETS["A"][0]:
        if env in os.environ:
            pytest.skip("%s is set in this process's environment: the default-knob cases would not be default" % env)


@pytest.mark.parametrize("case", dc.CASES, ids=lambda c: c.id)
def test_case_default_knobs(case):
    res, out = run_case(case)
    _OBSERVED.setdefault("default", set()).update(res["launched"])
    _RAN["default"] = _RAN.get("default", 0) + 1
    if out is not None:
        _DEFAULT_OUT[case.id] = out
    assert res["ok"], "\n".join(res["failures"])


# ------------------------------------------------------------------------------------------
# each knob set in a child process
# ------------------------------------------------------------------------------------------
def _child_main(knob_set, out_dir):
    cases = dc.knob_cases(knob_set)
    results, outs = [], {}
    for c in cases:
        try:
            res, out = run_case(c, knob_set)
        except Exception as e:                       # noqa: BLE001 -- reported to the parent, which fails
            res, out = dict(id=c.id, ok=False, failures=["%s: %s" % (type(e).__name__, e)], launched=[],
                            expected=sorted(c.expected(knob_set))), None
        results.append(res)
        if out is not None:
            outs[c.id] = out
    with open(os.path.join(out_dir, "results.json"), "w") as f:
        json.dump(results, f)
    torch.save(outs, os.path.join(out_dir, "forward_outputs.pt"))


def _same_family_but_pairs(a, b):
    """two forward kernel sets that differ only in the queries-per-tile template argument of one family"""
    def key(n):
        fam, args = n.split("<", 1) if "<" in n else (n, "")
        args = [s.strip() for s in args.rstrip(">").split(",")]
        pos = {"msda_fwd_fast_kernel": 2, "msda_snippet_fwd_kernel": 2, "msda_planar_fwd_kernel": 0}.get(fam)
        if pos is None:
            return n
        args[pos] = "*"
        return fam + "<" + ", ".join(args) + ">"
    fwd = lambda s: {n for n in s if "fwd" in dc.family(n)}   # noqa: E731
    return {key(n) for n in fwd(a)} == {key(n) for n in fwd(b)}


@pytest.mark.parametrize("knob_set", ["A", "B", "C"])
def test_knob_set_in_child_process(knob_set, tmp_path, capsys):
    env = dict(os.environ, **dc.KNOB_SETS[knob_set][0])
    proc = subprocess.run([sys.executable, os.path.abspath(__file__), knob_set, str(tmp_path)], env=env,
                          capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-4000:] + proc.stderr[-4000:]
    with open(tmp_path / "results.json") as f:
        results = json.load(f)
    outs = torch.load(tmp_path / "forward_outputs.pt")
    cases = {c.id: c for c in dc.knob_cases(knob_set)}
    assert [r["id"] for r in results] == list(cases)
    failures = ["%s: %s" % (r["id"], "; ".join(r["failures"])) for r in results if not r["ok"]]
    observed = set()
    for r in results:
        observed.update(r["launched"])
    _OBSERVED[knob_set] = observed
    _RAN[knob_set] = len(results)
    # "the knobs change speed, not results beyond rounding": the same family at another tile length sums every output
    # in the same order, so its forward is bit-identical; another family (split vs tile) agrees to the oracle tolerance
    for cid, out in outs.items():
        c = cases[cid]
        if cid not in _DEFAULT_OUT:
            _DEFAULT_OUT[cid] = run_case(c)[1]
        base = _DEFAULT_OUT[cid]
        if _same_family_but_pairs(c.expected("default"), c.expected(knob_set)):
            if not torch.equal(out, base):
                failures.append("%s: forward not bit-identical to the default knobs (%s vs %s)" % (
                    cid, sorted(c.expected(knob_set)), sorted(c.expected("default"))))
        else:
            # each side is within the oracle tolerance of the float64 result, so they are within twice that of each other
            tol = 2e-5 if c.dtype == "f32" else (2e-2 if c.entry == "presummed" else 2.0 ** -7)
            err = rel_err(out, base)
            if err >= tol:
                failures.append("%s: forward differs from the default knobs by %.3g" % (cid, err))
    with capsys.disabled():
        print("\n[dispatch coverage] knob set %s: %d cases in a child process, %d instantiations launched"
              % (knob_set, len(results), len(observed)))
    assert not failures, "\n".join(failures)


def test_observed_launches_equal_the_table(capsys):
    """Runs last: what the cases above saw launched, over all knob sets, is everything the table names."""
    if set(_OBSERVED) != {"default", "A", "B", "C"} or _RAN.get("default") != len(dc.CASES):
        pytest.skip("needs every case of this file in this session")
    seen = set().union(*_OBSERVED.values())
    inventory = dc.compiled_kernels()
    with capsys.disabled():
        print("\n[dispatch coverage] %d default-knob cases here, %s in children; %d instantiations observed launched, "
              "%d unreachable, %d compiled" % (_RAN["default"], {k: _RAN[k] for k in "ABC"}, len(seen),
                                               len(dc.UNREACHABLE), len(inventory) if inventory else -1))
    assert seen == dc.covered()
    if inventory is not None:
        assert seen | set(dc.UNREACHABLE) == inventory


if __name__ == "__main__":
    _child_main(sys.argv[1], sys.argv[2])

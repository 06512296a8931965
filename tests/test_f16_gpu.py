"""GPU tests of the float16 I/O mode (libmsda_b200_f16.so): value / output / grad_output and the pre-summed slots are
fp16; locations, weights, every gradient accumulation and all arithmetic are fp32; grad_value is rounded once.

Tolerances (rel_err = max |got - ref| / max |ref| per tensor, as in conftest.py), against float64 oracles evaluated on
the same fp16-rounded inputs:
  fp16 output and grad_value (fp32 sums rounded once to fp16):  |got - ref| <= 2^-10 |ref| + 1e-5 max|ref|;
  fp32 gradients 1e-4 (computed in fp32 from exactly representable inputs);
  the pre-summed path, whose neighbour-frame slot sums are themselves stored in fp16: 2e-3 for the output and every
  gradient.
"""
import copy
import dataclasses
import json
import os
import subprocess
import sys

import pytest
import torch

import dispatch_cases as dc
import test_dispatch_coverage_gpu as dcg
from conftest import level_start_index, make_case, rel_err
from oracle import c_oracle
from snippet_oracle import snippet_attention_oracle
from test_f16_library import bf16_kernels, to_f16
from test_msda_gpu import cuda_fwd_bwd

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32_TOL, PRESUM_TOL = 1e-4, 2e-3
LEVELS = [(19, 25), (10, 13), (5, 7)]


def f16_bound_excess(got, want):
    """max over elements of |got - want| - (2^-10 |want| + 1e-5 max|want|): <= 0 when every element is within"""
    got, want = got.detach().double().cpu().reshape(want.shape), want.detach().double().cpu()
    bound = 2.0 ** -10 * want.abs() + 1e-5 * float(want.abs().max())
    return float(((got - want).abs() - bound).max())


def within_one_ulp(got, want32):
    """every fp16 element of ``got`` within one fp16 ulp of the fp32 ``want32`` rounded once (ulp <= 2^-10 |x| for normal
    x, 2^-24 for subnormals)"""
    ref = want32.half().float()
    diff = (got.float() - ref).abs()
    return bool((diff <= 2.0 ** -10 * ref.abs() + 2.0 ** -24).all())


# ------------------------------------------------------------------------------------------
# per-call op against the float64 oracle
# ------------------------------------------------------------------------------------------
def _f16_case(N, M, D, P, Lq, regime, seed, levels=LEVELS):
    c = make_case(N, M, D, levels, P, Lq=Lq, regime=regime, seed=seed)
    c["value"] = c["value"].half()
    c["grad_out"] = c["grad_out"].half()
    return c


@pytest.mark.parametrize("D", [16, 32, 48, 64, 96, 128])
@pytest.mark.parametrize("regime", ["uniform", "local"])
def test_f16_percall_vs_oracle(D, regime):
    c = _f16_case(2, 8 if D == 48 else 3, D, 4, 157, regime, seed=D)
    out, (gv, gl, ga) = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], c["grad_out"])
    assert out.dtype == torch.float16 and gv.dtype == torch.float16
    assert gl.dtype == torch.float32 and ga.dtype == torch.float32
    args = (c["value"].double(), c["shapes"], c["lsi"], c["loc"].double(), c["attn"].double())
    ref_gv, ref_gl, ref_ga = c_oracle.backward(*args, c["grad_out"].double())
    assert f16_bound_excess(out, c_oracle.forward(*args)) <= 0
    assert f16_bound_excess(gv, ref_gv) <= 0
    assert rel_err(gl, ref_gl) < F32_TOL
    assert rel_err(ga, ref_ga) < F32_TOL


def test_f16_output_is_the_fp32_result_rounded_once():
    """Same inputs through the fp32 kernels: the fp16 output is that result rounded once, to within one fp16 ulp (the
    two kernels sum in fp32, in orders that may differ in the last bits)."""
    c = _f16_case(1, 8, 48, 4, None, "local", seed=5)
    out16, _ = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"])
    out32, _ = cuda_fwd_bwd(c["value"].float(), c["shapes"], c["lsi"], c["loc"], c["attn"])
    assert out16.dtype == torch.float16
    assert within_one_ulp(out16.cpu(), out32.cpu())


# ------------------------------------------------------------------------------------------
# fused op against the float64 oracle
# ------------------------------------------------------------------------------------------
def _fused_inputs(T2, T1, n_frame, Lq, seed, masked, levels=LEVELS, M=8, D=48, P=4, go_scale=None):
    gen = torch.Generator().manual_seed(seed)
    shapes = torch.as_tensor(levels, dtype=torch.long)
    S, L = int(shapes.prod(1).sum()), len(levels)
    Lq = Lq or S
    mlp = M * L * P
    value = torch.randn(1, T2, S, M, D, generator=gen).half()
    proj = torch.cat((torch.randn(1, T1, Lq, 2 * mlp, generator=gen) * 2.0, torch.randn(1, T1, Lq, mlp, generator=gen)), -1)
    ob, lb = torch.randn(2 * mlp, generator=gen), torch.randn(mlp, generator=gen)
    ref = torch.rand(1, T1, Lq, L, 2, generator=gen) * 1.2 - 0.1
    go = torch.randn(1, T1, Lq, M * D, generator=gen)
    if go_scale is not None:       # one sign, |go| in [go_scale / 2, go_scale] per channel
        go = (torch.rand(1, T1, Lq, M * D, generator=gen) * 0.5 + 0.5) * go_scale
    mask = (torch.rand(1, T2, S, generator=gen) < 0.2) if masked else None
    return dict(value=value, shapes=shapes, lsi=level_start_index(shapes), proj=proj, ob=ob, lb=lb, ref=ref,
                grad_out=go.half(), mask=mask, n_frame=n_frame)


def _run_fused_op(x, presum, dtype=None):
    """snippet_attention forward + backward on the GPU -> [out, grad_value, grad_proj, grad_ob, grad_lb, grad_ref]"""
    from snipper_b200 import ops
    v = x["value"] if dtype is None else x["value"].to(dtype)
    lv = [v.to(DEV).requires_grad_(True)] + [x[k].to(DEV).requires_grad_(True) for k in ("proj", "ob", "lb", "ref")]
    mask = x["mask"].to(DEV) if x["mask"] is not None else None
    out = ops.snippet_attention(lv[0], mask, x["shapes"].to(DEV), x["lsi"].to(DEV), *lv[1:], x["n_frame"],
                                presum=presum)
    out.backward(x["grad_out"].to(DEV).to(out.dtype))
    torch.cuda.synchronize()
    return [out.detach()] + [t.grad for t in lv]


def _oracle(x):
    leaves = [x["value"].double().requires_grad_(True)] + [x[k].clone().requires_grad_(True)
                                                           for k in ("proj", "ob", "lb", "ref")]
    vo = leaves[0]
    if x["mask"] is not None:
        vo = vo.masked_fill(x["mask"][..., None, None], 0.0)
    out = snippet_attention_oracle(vo, None, x["shapes"], x["lsi"], *leaves[1:], x["n_frame"])
    out.backward(x["grad_out"].double())
    return [out.detach()] + [t.grad for t in leaves]


@pytest.mark.parametrize("mode", ["direct", "masked", "presummed"])
@pytest.mark.parametrize("layer", ["encoder", "decoder"])
def test_f16_fused_vs_oracle(mode, layer):
    if layer == "encoder":       # Lq = S queries, the four observed frames
        x = _fused_inputs(4, 4, 4, None, seed=21, masked=mode != "direct")
    else:                        # 23 queries per frame, T1 = 6 query frames over 4 observed frames
        x = _fused_inputs(4, 6, 4, 23, seed=22, masked=mode != "direct")
    got = _run_fused_op(x, presum=mode == "presummed")
    want = _oracle(x)
    assert got[0].dtype == torch.float16 and got[1].dtype == torch.float16
    names = ("output", "grad_value", "grad_proj", "grad_offsets_bias", "grad_logits_bias", "grad_reference_points")
    for name, a, b in zip(names, got, want):
        if mode == "presummed":
            assert rel_err(a, b) < PRESUM_TOL, name
        elif name in ("output", "grad_value"):
            assert f16_bound_excess(a, b) <= 0, name
        else:
            assert rel_err(a, b) < F32_TOL, name
    if x["mask"] is not None:
        m5 = x["mask"][..., None, None].expand(got[1].shape)
        assert float(got[1].cpu()[m5].abs().max()) == 0.0


def test_f16_fused_output_is_the_fp32_result_rounded_once():
    x = _fused_inputs(4, 4, 4, None, seed=23, masked=False)
    out16 = _run_fused_op(x, presum=False)[0]
    out32 = _run_fused_op(x, presum=False, dtype=torch.float32)[0]
    assert within_one_ulp(out16.cpu(), out32.cpu())


# ------------------------------------------------------------------------------------------
# overflow of grad_value: +-inf exactly where .half() of the fp32 gradient overflows
# ------------------------------------------------------------------------------------------
def _check_overflow(g16, g32):
    ref = g32.half()
    inf = torch.isinf(ref)
    assert inf.any() and (~inf).any(), "the case must overflow in some entries and not in others"
    assert torch.equal(g16[inf], ref[inf])
    assert torch.isfinite(g16[~inf]).all()
    assert within_one_ulp(g16[~inf], g32[~inf])


def test_f16_percall_grad_value_overflows_like_half_of_fp32():
    c = make_case(1, 1, 16, [(4, 4), (2, 2)], 2, Lq=256, regime="uniform", seed=7)
    # channel c of grad_output in [1/2, 1] * 60000 * 2^-c, of one sign: 256 queries share 20 cells, so the cells' sums
    # overflow fp16 in the first channels only
    scale = 60000.0 * 2.0 ** -torch.arange(16, dtype=torch.float32)
    go = (torch.rand(c["grad_out"].shape, generator=torch.Generator().manual_seed(8)) * 0.5 + 0.5) * scale
    value = c["value"].half()
    _, (g16, _, _) = cuda_fwd_bwd(value, c["shapes"], c["lsi"], c["loc"], c["attn"], go.half())
    _, (g32, _, _) = cuda_fwd_bwd(value.float(), c["shapes"], c["lsi"], c["loc"], c["attn"], go.half().float())
    assert g16.dtype == torch.float16
    _check_overflow(g16.cpu(), g32.cpu())


def test_f16_presummed_grad_value_overflows_like_half_of_fp32():
    # 400 queries per frame over 54 cells, channel c of grad_output in [1/2, 1] * 60000 * 2^-c: a frame's gradient sums
    # the slots of up to three query frames, and overflows fp16 in the first channels only
    scale = 60000.0 * 2.0 ** -torch.arange(16, dtype=torch.float32).repeat(3)
    x = _fused_inputs(4, 4, 4, 400, seed=24, masked=False, levels=[(6, 7), (3, 4)], M=1, P=2, go_scale=scale)
    g16 = _run_fused_op(x, presum=True)[1]
    x32 = dict(x, grad_out=x["grad_out"].float())
    g32 = _run_fused_op(x32, presum=True, dtype=torch.float32)[1]
    assert g16.dtype == torch.float16
    _check_overflow(g16.cpu(), g32.cpu())


# ------------------------------------------------------------------------------------------
# dispatch: the bf16 cases of dispatch_cases.py with fp16 inputs launch exactly the fp16 twins
# ------------------------------------------------------------------------------------------
F16_CASES = [dataclasses.replace(c, dtype="f16") for c in dc.CASES
             if c.dtype == "bf16" and c.entry in ("fwd", "bwd", "direct", "masked", "presummed")]


def _f16_failures(c, checks):
    fails = []
    for name, got, want, kind in checks:
        want = want.detach().double().cpu()
        if c.entry == "presummed":
            err, ok = rel_err(got, want), rel_err(got, want) < PRESUM_TOL
        elif kind in ("out", "value"):
            err = f16_bound_excess(got, want)
            ok = err <= 0.0
        else:
            err = rel_err(got, want)
            ok = err < F32_TOL
        if not ok:
            fails.append("%s: error %.3g" % (name, err))
    return fails


def _child_main(out_dir):
    """Every case of F16_CASES under the profiler, in a process of its own whose profiler starts after
    libmsda_b200_f16.so is loaded (a process that profiled before loading it can miss the library's first kernels)."""
    from snipper_b200 import capi
    capi.f16_lib()
    dcg._DT["f16"] = torch.float16
    results = []
    for c in F16_CASES:
        try:
            launched, _, checks, extra = (dcg._run_percall if c.entry in ("fwd", "bwd") else dcg._run_fused)(c)
            results.append(dict(id=c.id, launched=sorted(launched), failures=list(extra) + _f16_failures(c, checks)))
        except Exception as e:                       # noqa: BLE001 -- reported to the parent, which fails
            results.append(dict(id=c.id, launched=[], failures=["%s: %s" % (type(e).__name__, e)]))
    with open(os.path.join(out_dir, "results.json"), "w") as f:
        json.dump(results, f)


@pytest.fixture(scope="module")
def dispatch_results(tmp_path_factory):
    out = tmp_path_factory.mktemp("f16_dispatch")
    proc = subprocess.run([sys.executable, os.path.abspath(__file__), str(out)], capture_output=True, text=True,
                          timeout=900)
    assert proc.returncode == 0, proc.stdout[-4000:] + proc.stderr[-4000:]
    with open(out / "results.json") as f:
        return {r["id"]: r for r in json.load(f)}


def _expected(case):
    return {to_f16(k) for k in dataclasses.replace(case, dtype="bf16").expected()}


@pytest.mark.parametrize("case", F16_CASES, ids=lambda c: c.id)
def test_dispatch_case_in_f16(case, dispatch_results):
    r = dispatch_results[case.id]
    assert not r["failures"], "\n".join(r["failures"])
    assert set(r["launched"]) == _expected(case)


def test_dispatch_cases_launch_every_reachable_f16_kernel(dispatch_results):
    """Together the cases launched every fp16 twin of a bf16 kernel the default knobs reach."""
    seen = set().union(*(set(r["launched"]) for r in dispatch_results.values()))
    reachable = set().union(*(_expected(c) for c in F16_CASES))
    assert seen == reachable
    assert reachable <= {to_f16(k) for k in bf16_kernels()}


# ------------------------------------------------------------------------------------------
# the module and the network under torch.autocast's default dtype (float16)
# ------------------------------------------------------------------------------------------
def test_module_under_default_autocast_runs_fp16_kernels(monkeypatch):
    from snipper_b200 import MSDeformAttn, ops
    torch.manual_seed(3)
    shapes = torch.as_tensor(LEVELS, dtype=torch.long, device=DEV)
    S = int(shapes.prod(1).sum())
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    mod = MSDeformAttn(384, 3, 8, 4, 4, "encoder").to(DEV)
    with torch.no_grad():
        mod.sampling_offsets[0].weight.normal_(0, 0.02)
        mod.attention_weights[0].weight.normal_(0, 0.05)
    q = torch.randn(1, 4, S, 384, device=DEV)
    src = torch.randn(1, 4, S, 384, device=DEV)
    refp = torch.rand(1, 4, S, 3, 2, device=DEV)
    want = mod(q, refp, src, shapes, lsi)
    assert torch.get_autocast_dtype("cuda") == torch.float16
    calls = []
    launch = ops._launch

    def spy(entry, tag, *args, f16=False, **kw):
        calls.append((tag, f16))
        return launch(entry, tag, *args, f16=f16, **kw)

    monkeypatch.setattr(ops, "_launch", spy)
    ops.STATS.reset()
    with torch.autocast("cuda"):
        got = mod(q, refp, src, shapes, lsi)
    # encoder-sized query set: the neighbour-frame sums and one gather, both in libmsda_b200_f16.so, nothing else
    assert ops.STATS.launches == 2
    assert calls == [("frame_sum", True), ("snippet_forward_presummed", True)]
    assert got.dtype == torch.float16
    assert rel_err(got.float(), want) < 1e-2


def _small_network(train=False):
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(5)
    net = build_snipper(snipper_b200.MSDeformAttn, num_frames=4, num_future_frames=0, enc_layers=2, dec_layers=2,
                        num_queries=7, **({"dropout": 0.0} if train else {}))
    with torch.no_grad():
        for n, p in net.named_parameters():
            if "sampling_offsets" in n and n.endswith("weight"):
                p.normal_(0, 0.02)
            if "attention_weights" in n:
                p.normal_(0, 0.2)
    net = net.to(DEV)
    return net.train() if train else net.eval()


_PRED = ("pred_logits", "pred_kpts2d", "pred_depth")


def _max_err(got, want):
    return max(rel_err(got[k].float(), want[k].float()) for k in want)


def test_network_under_default_autocast_eager_and_graph_replay():
    """The harness network under float16 autocast, eagerly and through GraphRunner: its predictions are at least as
    close to the fp32 network's as those under bfloat16 autocast, on the same seeded inputs."""
    import snipper_b200
    net = _small_network()

    def fn(x):
        out, _ = net(x)
        return {k: out[k] for k in _PRED}

    xs = [torch.rand(1, 12, 192, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(s)) for s in (1, 2)]
    with torch.no_grad():
        ref = [{k: v.clone() for k, v in fn(x).items()} for x in xs]
        with torch.autocast("cuda"):
            eager16 = [{k: v.clone() for k, v in fn(x).items()} for x in xs]
    r16 = snipper_b200.GraphRunner(fn, autocast_dtype=torch.float16)
    rbf = snipper_b200.GraphRunner(fn, autocast_dtype=torch.bfloat16)
    for x, want, e16 in zip(xs, ref, eager16):
        g16 = {k: v.clone() for k, v in r16(x).items()}
        gbf = {k: v.clone() for k, v in rbf(x).items()}
        assert all(torch.isfinite(v).all() for v in g16.values())
        assert _max_err(e16, want) <= _max_err(gbf, want)
        assert _max_err(g16, want) <= _max_err(gbf, want)


def _loss(out):
    loss = out["pred_kpts2d"].square().mean() + out["pred_depth"].square().mean() + out["pred_logits"].square().mean()
    for h in out["heatmaps"]:
        loss = loss + h.square().mean()
    return loss


def _grads(net):
    return {n: p.grad.detach().float().clone() for n, p in net.named_parameters() if p.grad is not None}


def _grad_err(g, g32):
    num = sum(float((g[n] - g32[n]).square().sum()) for n in g32)
    return (num / sum(float(v.square().sum()) for v in g32.values())) ** 0.5


def test_training_step_with_grad_scaler_under_default_autocast():
    """One GradScaler step under float16 autocast: finite loss, a finite gradient wherever fp32 has one, and unscaled
    gradients at least as close to fp32's as bfloat16 autocast's (relative L2 over all parameters)."""
    from snipper_b200 import ops
    base = _small_network(train=True)
    x = torch.rand(1, 12, 192, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    net32, netbf, net16 = base, copy.deepcopy(base), copy.deepcopy(base)
    _loss(net32(x)[0]).backward()
    g32 = _grads(net32)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        lbf = _loss(netbf(x)[0])
    lbf.backward()
    gbf = _grads(netbf)

    opt = torch.optim.AdamW([p for p in net16.parameters() if p.requires_grad], lr=1e-4)
    # a moderate initial scale: the default 2^16 may overflow on the first step, which GradScaler would then skip
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10)
    ops.STATS.reset()
    ops.STATS.timing = True
    try:
        with torch.autocast("cuda"):
            l16 = _loss(net16(x)[0])
        scaler.scale(l16).backward()
    finally:
        ops.STATS.timing = False
    tags = {tag for tag, _, _, _ in ops.STATS.events}
    assert {"frame_sum", "snippet_forward_presummed", "snippet_backward_presummed", "frame_unsum"} <= tags
    scaler.unscale_(opt)
    g16 = _grads(net16)
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 10          # no inf / NaN was found: the step was taken
    assert torch.isfinite(l16)
    assert g16.keys() == g32.keys() == gbf.keys()
    bad = [n for n, g in g16.items() if not torch.isfinite(g).all()]
    assert not bad, bad
    assert _grad_err(g16, g32) <= _grad_err(gbf, g32)


if __name__ == "__main__":
    _child_main(sys.argv[1])

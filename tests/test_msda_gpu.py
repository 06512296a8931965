"""GPU parity tests of the per-call op (through the C ABI via the torch custom op).

Tolerances are BASELINE.json's: forward <= 1e-5 relative (fp32), backward <= 1e-4 relative
(fp32), measured as max|a-b| / max|ref| per output tensor; fp64 runs are held to 1e-10.
The checker is the CPU oracle (oracle/), itself pinned to the reference by tests/golden/.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, make_case, rel_err
from oracle import c_oracle

pytestmark = pytest.mark.gpu

FWD_TOL, BWD_TOL, F64_TOL = 1e-5, 1e-4, 1e-10


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def cuda_fwd_bwd(value, shapes, lsi, loc, attn, grad_out=None, im2col_step=64):
    from snipper_b200 import MSDeformAttnFunction
    dev = "cuda:0"
    v = value.to(dev).requires_grad_(True)
    s = loc.to(dev).requires_grad_(True)
    a = attn.to(dev).requires_grad_(True)
    out = MSDeformAttnFunction.apply(v, shapes.to(dev), lsi.to(dev), s, a, im2col_step)
    if grad_out is None:
        return out.detach().cpu(), None
    out.backward(grad_out.to(dev))
    torch.cuda.synchronize()
    return out.detach().cpu(), (v.grad.cpu(), s.grad.cpu(), a.grad.cpu())


def check_against_oracle(c, fwd_tol, bwd_tol, ref_dtype=torch.float64):
    """CUDA (dtype of the case) vs C oracle evaluated in ref_dtype on the same inputs."""
    out, grads = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], c["grad_out"])
    args = (c["value"].to(ref_dtype), c["shapes"], c["lsi"], c["loc"].to(ref_dtype), c["attn"].to(ref_dtype))
    ref_out = c_oracle.forward(*args)
    ref_gv, ref_gl, ref_ga = c_oracle.backward(*args, c["grad_out"].to(ref_dtype))
    assert rel_err(out, ref_out) < fwd_tol
    assert rel_err(grads[0], ref_gv) < bwd_tol
    assert rel_err(grads[1], ref_gl) < bwd_tol
    assert rel_err(grads[2], ref_ga) < bwd_tol


# ---------------------------------------------------------------- reference test.py fixture
def test_testpy_forward_double_golden():
    g = load_golden("testpy_seed3")
    out, _ = cuda_fwd_bwd(T(g["dbl_value"]).double(), T(g["shapes"]), T(g["lsi"]),
                          T(g["dbl_loc"]).double(), T(g["dbl_attn"]).double(), im2col_step=2)
    assert torch.allclose(out, T(g["dbl_out"]))  # reference test.py:40
    assert rel_err(out, g["dbl_out"]) < F64_TOL


def test_testpy_forward_float_golden():
    g = load_golden("testpy_seed3")
    out, _ = cuda_fwd_bwd(T(g["flt_value"]), T(g["shapes"]), T(g["lsi"]), T(g["flt_loc"]),
                          T(g["flt_attn"]), im2col_step=2)
    assert torch.allclose(out, T(g["flt_out"]), rtol=1e-2, atol=1e-3)  # reference test.py:56
    assert rel_err(out, g["flt_out"]) < FWD_TOL


@pytest.mark.parametrize("D", [30, 32, 64, 71])
def test_testpy_gradients_golden(D):
    g = load_golden("testpy_seed3")
    k = "g%d_" % D
    out, grads = cuda_fwd_bwd(T(g[k + "value"]).double(), T(g["shapes"]), T(g["lsi"]),
                              T(g[k + "loc"]).double(), T(g[k + "attn"]).double(), T(g[k + "grad_out"]), 2)
    assert rel_err(out, g[k + "out"]) < F64_TOL
    assert rel_err(grads[0], g[k + "grad_value"]) < F64_TOL
    assert rel_err(grads[1], g[k + "grad_loc"]) < F64_TOL
    assert rel_err(grads[2], g[k + "grad_attn"]) < F64_TOL


@pytest.mark.parametrize("D", [1025, 2048, 3096])
def test_testpy_large_channels_vs_oracle(D):
    # the rest of reference test.py:85's channel list, checked against the oracle in fp64
    c = make_case(1, 2, D, [(6, 4), (3, 2)], 2, Lq=2, regime="uniform", seed=D, dtype=torch.float64)
    check_against_oracle(c, F64_TOL, F64_TOL)


def test_gradcheck_double():
    # reference test.py:63-78 runs torch.autograd.gradcheck on the Function in fp64
    from snipper_b200 import MSDeformAttnFunction
    c = make_case(1, 2, 6, [(6, 4), (3, 2)], 2, Lq=2, regime="uniform", seed=3, dtype=torch.float64)
    dev = "cuda:0"
    v = c["value"].to(dev).requires_grad_(True)
    s = c["loc"].to(dev).requires_grad_(True)
    a = c["attn"].to(dev).requires_grad_(True)
    assert torch.autograd.gradcheck(MSDeformAttnFunction.apply, (v, c["shapes"].to(dev), c["lsi"].to(dev), s, a, 2))


# ---------------------------------------------------------------- Snipper geometry goldens
@pytest.mark.parametrize("case", ["snipper_small", "frames_levels"])
def test_snipper_golden_fp32(case):
    g = load_golden(case)
    out, grads = cuda_fwd_bwd(T(g["value"]), T(g["shapes"]), T(g["lsi"]), T(g["loc"]), T(g["attn"]), T(g["grad_out"]))
    assert rel_err(out, g["out_f64"]) < FWD_TOL
    assert rel_err(grads[0], g["grad_value"]) < BWD_TOL
    assert rel_err(grads[1], g["grad_loc"]) < BWD_TOL
    assert rel_err(grads[2], g["grad_attn"]) < BWD_TOL


@pytest.mark.parametrize("case", ["snipper_small", "frames_levels"])
def test_snipper_golden_fp64(case):
    g = load_golden(case)
    out, grads = cuda_fwd_bwd(T(g["value"]).double(), T(g["shapes"]), T(g["lsi"]), T(g["loc"]).double(),
                              T(g["attn"]).double(), T(g["grad_out"]).double())
    assert rel_err(out, g["out_f64"]) < F64_TOL
    assert rel_err(grads[0], g["grad_value"]) < F64_TOL
    assert rel_err(grads[1], g["grad_loc"]) < F64_TOL
    assert rel_err(grads[2], g["grad_attn"]) < F64_TOL


# ---------------------------------------------------------------- seeded sweeps vs the oracle
SNIPPER_SMALL_LEVELS = [(19, 25), (10, 13), (5, 7)]


@pytest.mark.parametrize("D", [16, 32, 48, 64, 96, 128])
@pytest.mark.parametrize("regime", ["uniform", "local"])
def test_fast_path_channels(D, regime):
    c = make_case(2, 4, D, SNIPPER_SMALL_LEVELS, 4, Lq=77, regime=regime, seed=D)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


@pytest.mark.parametrize("D", [4, 12, 30, 40, 71, 144])
def test_generic_path_channels_fp32(D):
    c = make_case(2, 3, D, SNIPPER_SMALL_LEVELS, 3, Lq=41, regime="local", seed=D)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


@pytest.mark.parametrize("L,P", [(1, 1), (3, 8), (6, 4), (9, 4), (12, 4), (12, 8)])
def test_levels_points(L, P):
    # L*P up to 96 > the per-pass chunk of the fast kernels (multi-pass staging)
    shapes = [(7 + (i % 3), 9 - (i % 2)) for i in range(L)]
    c = make_case(1, 8, 48, shapes, P, Lq=50, regime="local", seed=L * 10 + P)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


@pytest.mark.parametrize("N", [1, 2, 5])
def test_batch_and_ragged_tail(N):
    # Lq*M*N not a multiple of the CTA's pair count -> exercises the tail masking
    c = make_case(N, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=61, regime="local", seed=N)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


def test_decoder_shape():
    c = make_case(2, 8, 48, [(75, 100), (38, 50), (19, 25)], 4, Lq=60, regime="uniform", seed=9)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


def test_batch_strided_value_no_copy():
    """value[:, t2] of a (N,T,S,M,D) tensor: accepted without a copy (batch stride only)."""
    from snipper_b200 import ms_deform_attn
    c = make_case(3, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=33, seed=4)
    dev = "cuda:0"
    big = torch.randn(3, 4, *c["value"].shape[1:], device=dev)
    big[:, 2] = c["value"].to(dev)
    view = big[:, 2]
    assert not view.is_contiguous()
    out = ms_deform_attn(view, c["shapes"].to(dev), c["lsi"].to(dev), c["loc"].to(dev), c["attn"].to(dev))
    ref = c_oracle.forward(c["value"].double(), c["shapes"], c["lsi"], c["loc"].double(), c["attn"].double())
    assert rel_err(out, ref) < FWD_TOL


# ---------------------------------------------------------------- edge cases
def test_all_samples_outside_give_zero():
    c = make_case(1, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=20, seed=1)
    c["loc"] = torch.full_like(c["loc"], 1.7)
    c["loc"][..., 0] = -0.9
    out, grads = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], c["grad_out"])
    assert out.abs().max() == 0
    assert all(g.abs().max() == 0 for g in grads)


def test_border_samples_partial_corners():
    """Samples within one pixel of the border: some corners invalid (zero padding)."""
    c = make_case(1, 8, 48, [(6, 8)], 4, Lq=64, regime="uniform", seed=2)
    H, W = 6, 8
    g = torch.Generator().manual_seed(5)
    edge = torch.rand(c["loc"].shape, generator=g)
    # x in (-1/W, 0.5/W) or (1-0.5/W, 1+1/W): straddles the image border
    c["loc"] = torch.where(edge < 0.5, edge * 3 / W - 1.0 / W, 1 - 0.5 / W + edge * 1.5 / W)
    check_against_oracle(c, FWD_TOL, BWD_TOL)


def test_exact_integer_coordinates():
    """Samples exactly on pixel centres / corners (the random-init regime, SURVEY section 7)."""
    c = make_case(1, 8, 48, [(8, 8)], 4, Lq=64, regime="uniform", seed=3)
    c["loc"] = (torch.randint(0, 17, c["loc"].shape).float() * 0.5) / 8.0  # multiples of half a pixel
    out, _ = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"])
    ref = c_oracle.forward(c["value"].double(), c["shapes"], c["lsi"], c["loc"].double(), c["attn"].double())
    assert rel_err(out, ref) < FWD_TOL


def test_empty_queries_and_empty_batch():
    from snipper_b200 import ms_deform_attn
    dev = "cuda:0"
    c = make_case(2, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=4, seed=1)
    out = ms_deform_attn(c["value"].to(dev), c["shapes"].to(dev), c["lsi"].to(dev),
                         c["loc"][:, :0].contiguous().to(dev), c["attn"][:, :0].contiguous().to(dev))
    assert out.shape == (2, 0, 8 * 48)
    out = ms_deform_attn(c["value"][:0].to(dev), c["shapes"].to(dev), c["lsi"].to(dev),
                         c["loc"][:0].to(dev), c["attn"][:0].to(dev))
    assert out.shape == (0, 4, 8 * 48)


def test_im2col_step_semantics():
    """batch % min(batch, im2col_step) must be 0 (reference ms_deform_attn_cuda.cu:50-52)."""
    from snipper_b200 import ms_deform_attn
    dev = "cuda:0"
    c = make_case(3, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=4, seed=1)
    args = [c[k].to(dev) for k in ("value", "shapes", "lsi", "loc", "attn")]
    with pytest.raises(RuntimeError, match=r"batch\(3\) must divide im2col_step\(2\)"):
        ms_deform_attn(*args, im2col_step=2)
    ref = ms_deform_attn(*args, im2col_step=64)
    for step in (1, 3, 64):  # results do not depend on the chunking
        assert torch.equal(ms_deform_attn(*args, im2col_step=step), ref)


def test_contiguity_and_device_errors():
    import snipper_b200
    shim = snipper_b200.install_extension_shim()
    dev = "cuda:0"
    c = make_case(1, 8, 48, SNIPPER_SMALL_LEVELS, 4, Lq=4, seed=1)
    args = [c[k].to(dev) for k in ("value", "shapes", "lsi", "loc", "attn")]
    bad = list(args)
    bad[3] = args[3].transpose(1, 2).contiguous().transpose(1, 2)
    with pytest.raises(RuntimeError, match="sampling_loc tensor has to be contiguous"):
        shim.ms_deform_attn_forward(*bad, 64)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        shim.ms_deform_attn_forward(*[c[k] for k in ("value", "shapes", "lsi", "loc", "attn")], 64)
    out = shim.ms_deform_attn_forward(*args, 64)
    gv, gl, ga = shim.ms_deform_attn_backward(*args, torch.ones_like(out), 64)
    assert gv.shape == args[0].shape and gl.shape == args[3].shape and ga.shape == args[4].shape


# ---------------------------------------------------------------- full BASELINE sizes
FULL = [(75, 100), (38, 50), (19, 25)]


@pytest.fixture(scope="module")
def full_case():
    return make_case(1, 8, 48, FULL, 4, regime="local", sigma_px=4.0, seed=0)


def test_full_size_vs_oracle(full_case):
    """Encoder call at BASELINE size (S = Lq = 9875, M=8, D=48, L=3, P=4), fwd + bwd."""
    check_against_oracle(full_case, FWD_TOL, BWD_TOL, ref_dtype=torch.float32)


def test_full_size_linearity_and_adjoint(full_case):
    """Size-independent properties: the op is linear in value, and backward is its adjoint:
    <grad_out, f(v)> == <grad_value, v>;  grad_attn contracts to the same number."""
    from snipper_b200 import ms_deform_attn
    dev = "cuda:0"
    c = {k: v.to(dev) for k, v in full_case.items()}
    v1, v2 = c["value"], torch.randn_like(c["value"])
    f = lambda v: ms_deform_attn(v, c["shapes"], c["lsi"], c["loc"], c["attn"])
    lhs = f(2.5 * v1 - v2)
    rhs = 2.5 * f(v1) - f(v2)
    assert rel_err(lhs, rhs) < 1e-5
    _, grads = cuda_fwd_bwd(full_case["value"], full_case["shapes"], full_case["lsi"], full_case["loc"],
                            full_case["attn"], full_case["grad_out"])
    out = f(v1).double().cpu()
    inner_out = (full_case["grad_out"].double() * out).sum()
    inner_val = (grads[0].double() * full_case["value"].double()).sum()
    inner_att = (grads[2].double() * full_case["attn"].double()).sum()
    assert abs(inner_out - inner_val) / abs(inner_out) < 1e-5
    assert abs(inner_out - inner_att) / abs(inner_out) < 1e-5


def test_full_size_constant_value_sums_weights():
    """value == 1 everywhere and all samples strictly inside -> out == sum of attention weights == 1."""
    from snipper_b200 import ms_deform_attn
    dev = "cuda:0"
    c = make_case(1, 8, 48, FULL, 4, regime="uniform", seed=1)
    loc = c["loc"] * 0.9 + 0.05
    out = ms_deform_attn(torch.ones_like(c["value"]).to(dev), c["shapes"].to(dev), c["lsi"].to(dev),
                         loc.to(dev), c["attn"].to(dev))
    assert (out - 1).abs().max() < 1e-5


# ---------------------------------------------------------------- vs the vendored CUDA op
def test_matches_vendored_cuda_op(full_case):
    """north_star: outputs must match the reference's vendored CUDA op (recompiled for sm_100a
    from the unmodified sources by oracle/build_ref.py) on identical inputs."""
    from oracle.build_ref import load_ref
    ref = load_ref()
    if ref is None:
        pytest.skip("the original's CUDA op is not built: build() compiles it into oracle/_ref when SNIPPER_REFERENCE "
                    "names the original Snipper source tree")
    dev = "cuda:0"
    c = {k: v.to(dev) for k, v in full_case.items()}
    out_ref = ref.ms_deform_attn_forward(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], 64)
    gv_ref, gl_ref, ga_ref = ref.ms_deform_attn_backward(c["value"], c["shapes"], c["lsi"], c["loc"],
                                                         c["attn"], c["grad_out"], 64)
    out, grads = cuda_fwd_bwd(full_case["value"], full_case["shapes"], full_case["lsi"], full_case["loc"],
                              full_case["attn"], full_case["grad_out"])
    assert rel_err(out, out_ref) < FWD_TOL
    assert rel_err(grads[0], gv_ref) < BWD_TOL
    assert rel_err(grads[1], gl_ref) < BWD_TOL
    assert rel_err(grads[2], ga_ref) < BWD_TOL


# ---------------------------------------------------------------- deterministic two-pass backward
@pytest.mark.parametrize("D,Lq", [(48, None), (30, 37)])
def test_deterministic_backward_is_bit_reproducible(D, Lq):
    """MSDA_FLAG_DETERMINISTIC: same bits run to run, still within the backward tolerance."""
    import snipper_b200
    c = make_case(2, 8 if D == 48 else 3, D, SNIPPER_SMALL_LEVELS, 4, Lq=Lq, regime="local", sigma_px=1.5, seed=21)
    dev = "cuda:0"
    args = [c[k].to(dev) for k in ("value", "shapes", "lsi", "loc", "attn", "grad_out")]
    runs = [torch.ops.snipper_b200.msda_backward(*args, 64, True) for _ in range(3)]
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    a64 = (c["value"].double(), c["shapes"], c["lsi"], c["loc"].double(), c["attn"].double())
    ref = c_oracle.backward(*a64, c["grad_out"].double())
    for got, want in zip(runs[0], ref):
        assert rel_err(got, want) < BWD_TOL
    # and through autograd with the process-wide switch
    snipper_b200.set_deterministic(True)
    try:
        _, g1 = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], c["grad_out"])
        _, g2 = cuda_fwd_bwd(c["value"], c["shapes"], c["lsi"], c["loc"], c["attn"], c["grad_out"])
    finally:
        snipper_b200.set_deterministic(False)
    assert all(torch.equal(x, y) for x, y in zip(g1, g2))
    assert torch.equal(g1[0], runs[0][0].cpu())


def test_deterministic_full_size(full_case):
    dev = "cuda:0"
    args = [full_case[k].to(dev) for k in ("value", "shapes", "lsi", "loc", "attn", "grad_out")]
    a = torch.ops.snipper_b200.msda_backward(*args, 64, True)
    b = torch.ops.snipper_b200.msda_backward(*args, 64, True)
    fast = torch.ops.snipper_b200.msda_backward(*args, 64, False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    for x, y in zip(a, fast):
        assert rel_err(x, y) < BWD_TOL


def test_pile_up_on_one_cell_long_list_path():
    """Every query samples the same location: one cell receives thousands of contributions
    (the in-kernel list spills past shared memory; exercises the long-list path)."""
    c = make_case(1, 2, 16, [(4, 4)], 2, Lq=300, regime="uniform", seed=2)
    c["loc"] = torch.full_like(c["loc"], 0.4)
    dev = "cuda:0"
    args = [c[k].to(dev) for k in ("value", "shapes", "lsi", "loc", "attn", "grad_out")]
    a = torch.ops.snipper_b200.msda_backward(*args, 64, True)
    b = torch.ops.snipper_b200.msda_backward(*args, 64, True)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    ref = c_oracle.backward(c["value"].double(), c["shapes"], c["lsi"], c["loc"].double(), c["attn"].double(),
                            c["grad_out"].double())
    for got, want in zip(a, ref):
        assert rel_err(got, want) < BWD_TOL


"""The layer tails under bf16 autocast (``layer_tail_amp``, libmsda_b200_amp.so) and the layers that opt into them with
``enable_fused_layer_tails(model, autocast=True)``.

A. The kernel against the fp32 ``layer_tail`` kernel: ``out`` has its bits on float(y), float(residual), and the bf16
   outputs are exactly torch's rounding of out and out + pos.  With the float64 validation of the fp32 kernel
   (test_layer_tails_oracle_gpu.py) that makes the amp kernel validated too.  Layouts, aliases and guard bands.
B. The bench harness' encoder / decoder layers at the bench shapes under bf16 autocast: the amp-tail stack and the
   stock autocast stack against the same layers in float64.
C. Which path runs: amp tails, fp32 tails or the stock forward, per case, and the dtypes that reach the tails.
D. CUDA-graph capture and replay under bf16 autocast with the amp tails.
E. The small network end to end against its fp32 predictions.

Errors are per row, as in test_layer_tails_oracle_gpu.py.
"""
import copy

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF16 = torch.bfloat16
T = 4
LEVELS = [(75, 100), (38, 50), (19, 25)]      # a 600x800 frame at strides 8 / 16 / 32
SMALL_LEVELS = [(12, 16), (6, 8), (3, 4)]
D_MODEL, FFN, HEADS, N_LEVELS, N_POINTS = 384, 1024, 8, 3, 4


@pytest.fixture(autouse=True)
def strict_fp32():
    """The fp32 references (GEMMs of the fp32 network, float64 comparisons) in full fp32, not TF32."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _bf16_autocast():
    return torch.autocast("cuda", dtype=BF16)


def _count(fn):
    """(fn(), {"layer_tail": n, "layer_tail_amp": n}) of the launches fn issued."""
    from snipper_b200 import ops
    ops.STATS.reset()
    ops.STATS.timing = True
    try:
        out = fn()
    finally:
        ops.STATS.timing = False
    tags = [e[0] for e in ops.STATS.events]
    return out, {t: tags.count(t) for t in ("layer_tail", "layer_tail_amp")}


def _row_abs_err(got, want):
    return (got.double() - want.double()).abs().flatten(0, -2).amax(1)


def _worst_row(err, allowed, want):
    ratio = err / allowed
    i = int(ratio.argmax())
    if ratio[i] <= 1:
        return ""
    scale = want.double().flatten(0, -2).abs().amax(1)[i].clamp_min(1e-300)
    return "row %d of %d: err %.3e (rel %.3e) > allowed %.3e; %d rows over" % (
        i, err.numel(), err[i], err[i] / scale, allowed[i], int((ratio > 1).sum()))


# ============================================================================================================
# A. the kernel against the fp32 kernel
# ============================================================================================================
ROWS = [1, 7, 8, 9, 240, 39500, 65541]
FAMILIES = ["normal", "offset_1e4", "offset_1e3", "constant", "outlier", "tiny", "gamma_zero_neg"]


def _tail_inputs(family, rows, C, gen):
    """bf16 y, fp32 residual, bias, pos, gamma, beta; the pre-norm rows residual + (y + bias) follow ``family`` (the
    row families of test_layer_tails_oracle_gpu.py)."""
    def n(*shape):
        return torch.randn(*shape, device=DEV, generator=gen)
    mean, std = {"offset_1e4": (1e4, 1.0), "offset_1e3": (1e3, 1e-2), "tiny": (0.0, 1e-20)}.get(family, (0.0, 1.0))
    s = std / 3 ** 0.5
    y, residual, bias = n(rows, C) * s, mean + n(rows, C) * s, n(C) * s
    if family == "constant":
        residual = (n(rows, 1) * 3).expand(rows, C).contiguous()
        y, bias = torch.zeros_like(y), torch.zeros_like(bias)
    if family == "outlier":
        residual[torch.arange(rows, device=DEV), torch.randint(0, C, (rows,), device=DEV, generator=gen)] = 1e4
    gamma, beta = n(C), n(C)
    if family in ("tiny", "gamma_zero_neg"):
        beta = torch.zeros(C, device=DEV)
    if family == "gamma_zero_neg":
        gamma = -gamma.abs()
        gamma[::3] = 0.0
        gamma[1::3] *= -1
    return y.to(BF16), residual, bias, n(rows, C), gamma, beta


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("C", [128 * k for k in range(1, 9)])
def test_amp_tail_matches_the_fp32_kernel_bit_for_bit(C, family):
    import snipper_b200  # noqa: F401
    lt, amp = torch.ops.snipper_b200.layer_tail, torch.ops.snipper_b200.layer_tail_amp
    gen = torch.Generator(device=DEV).manual_seed(2000 * C + FAMILIES.index(family))
    for rows in ROWS:
        y, res32, bias_full, pos_full, gamma, beta = _tail_inputs(family, rows, C, gen)
        for residual in (res32, res32.to(BF16)):
            for bias in (bias_full, None):
                for eps in (1e-5, 1e-6):
                    want = lt(y.float(), bias, residual.float(), gamma, beta, None, eps)[0]
                    for emit in (True, False):
                        for pos in (pos_full, None):
                            case = (rows, residual.dtype, bias is not None, eps, emit, pos is not None)
                            out, out16, out_pos16 = amp(y, bias, residual, gamma, beta, pos, eps, emit)
                            assert out.dtype == torch.float32 and out.shape == (rows, C), case
                            assert torch.equal(out, want), case
                            if emit:
                                assert out16.dtype == BF16 and torch.equal(out16, out.to(BF16)), case
                            else:
                                assert out16.numel() == 0, case
                            if pos is not None:
                                assert out_pos16.dtype == BF16 and torch.equal(out_pos16, (out + pos).to(BF16)), case
                            else:
                                assert out_pos16.numel() == 0, case


def test_amp_tail_layouts_aliases_and_refusals():
    """Views are taken as they are, operands may alias, 4-D activations are rows too, zero rows is empty, and what the
    kernel does not take is refused."""
    import snipper_b200  # noqa: F401
    amp = torch.ops.snipper_b200.layer_tail_amp
    gen = torch.Generator(device=DEV).manual_seed(17)
    rows, C = 1000, 384
    y_t = torch.randn(C, rows, device=DEV, generator=gen).to(BF16).t()          # transposed
    res_s = torch.randn(rows, 2 * C, device=DEV, generator=gen)[:, C:]         # column slice
    pos_s = torch.randn(2 * rows, C, device=DEV, generator=gen)[1::2]          # row stride 2
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    assert not (y_t.is_contiguous() or res_s.is_contiguous() or pos_s.is_contiguous())
    want = amp(y_t.contiguous(), bias, res_s.contiguous(), gamma, beta, pos_s.contiguous(), 1e-5, True)
    got = amp(y_t, bias, res_s, gamma, beta, pos_s, 1e-5, True)
    assert all(torch.equal(a, b) for a, b in zip(got, want))

    y = y_t.contiguous()
    want = amp(y, bias, y.clone(), gamma, beta, None, 1e-5, True)                 # bf16 residual
    got = amp(y, bias, y, gamma, beta, None, 1e-5, True)                         # residual is y
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    res = res_s.contiguous()
    want = amp(y, bias, res, gamma, beta, res.clone(), 1e-5, True)
    got = amp(y, bias, res, gamma, beta, res, 1e-5, True)                        # pos is residual
    assert all(torch.equal(a, b) for a, b in zip(got, want))

    y4 = torch.randn(2, 4, 60, C, device=DEV, generator=gen).to(BF16)
    r4 = torch.randn(2, 4, 60, C, device=DEV, generator=gen)
    got = amp(y4, bias, r4, gamma, beta, r4, 1e-5, True)
    want = amp(y4.reshape(-1, C), bias, r4.reshape(-1, C), gamma, beta, r4.reshape(-1, C), 1e-5, True)
    for g, w in zip(got, want):
        assert g.shape == y4.shape and torch.equal(g.reshape(-1, C), w)

    e16, e32 = torch.empty(0, C, device=DEV, dtype=BF16), torch.empty(0, C, device=DEV)
    out, out16, out_pos = amp(e16, bias, e32, gamma, beta, e32, 1e-5, True)
    assert out.shape == out16.shape == out_pos.shape == (0, C)

    strided = torch.randn(2 * C, device=DEV)[::2]
    for args in ((y, strided, res, gamma, beta), (y, bias, res, strided, beta), (y, bias, res, gamma, strided)):
        with pytest.raises(RuntimeError, match="contiguous"):
            amp(*args, None, 1e-5, False)
    for args in ((y.float(), bias, res, gamma, beta, None),                       # y must be bf16
                 (y, bias, res.double(), gamma, beta, None),                      # residual fp32 / bf16
                 (y, bias, res, gamma, beta, res.to(BF16)),                       # pos fp32
                 (y[:, :320], bias, res[:, :320], gamma, beta, None)):            # C = 128 * k
        with pytest.raises(RuntimeError, match="layer_tail_amp"):
            amp(*args, 1e-5, False)


@pytest.mark.parametrize("C", [128, 384, 1024])
@pytest.mark.parametrize("rows", [1, 9, 39500])
@pytest.mark.parametrize("res_dtype", [torch.float32, BF16])
def test_amp_tail_writes_exactly_its_rows(rows, C, res_dtype):
    """Through the C ABI, every output placed inside a NaN-filled buffer at a 16-byte aligned offset: the kernel writes
    rows x C elements of each, nothing before or after, and leaves its inputs as they were."""
    import snipper_b200  # noqa: F401
    from snipper_b200 import capi
    gen = torch.Generator(device=DEV).manual_seed(rows + C)
    y = torch.randn(rows, C, device=DEV, generator=gen).to(BF16)
    res = torch.randn(rows, C, device=DEV, generator=gen).to(res_dtype)
    pos = torch.randn(rows, C, device=DEV, generator=gen)
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    inputs = (y, bias, res, gamma, beta, pos)
    before = [t.clone() for t in inputs]
    n = rows * C
    bufs = [torch.full((pad + n + pad,), float("nan"), device=DEV, dtype=dt)
            for pad, dt in ((36, torch.float32), (72, BF16), (72, BF16))]   # 144 bytes: 16-byte aligned, not 128
    out, out16, out_pos16 = (b[pad:pad + n] for b, pad in zip(bufs, (36, 72, 72)))
    assert all(t.data_ptr() % 16 == 0 for t in (out, out16, out_pos16))
    status = capi.amp_lib().msda_amp_layer_tail(
        y.data_ptr(), bias.data_ptr(), res.data_ptr(), capi.MSDA_DTYPE_F32 if res_dtype == torch.float32 else
        capi.MSDA_DTYPE_BF16, gamma.data_ptr(), beta.data_ptr(), pos.data_ptr(), out.data_ptr(), out16.data_ptr(),
        out_pos16.data_ptr(), rows, C, 1e-5, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert status == capi.MSDA_OK
    want = torch.ops.snipper_b200.layer_tail_amp(y, bias, res, gamma, beta, pos, 1e-5, True)
    for got, w in zip((out, out16, out_pos16), want):
        assert torch.equal(got.view(rows, C), w)
    for b, pad in zip(bufs, (36, 72, 72)):
        assert b[:pad].isnan().all() and b[pad + n:].isnan().all()
    for t, b in zip(inputs, before):
        assert torch.equal(t, b)


# ============================================================================================================
# B. harness layers at the bench shapes under bf16 autocast, against their float64 copy
# ============================================================================================================
def _perturb(module, seed):
    """Random Linear weights, the MSDeformAttn init with perturbed sampling-offset / attention-weight weights, and
    non-trivial LayerNorm parameters and projection biases (as test_layer_tails_oracle_gpu.py does)."""
    import snipper_b200
    torch.manual_seed(seed)
    for m in module.modules():
        if isinstance(m, nn.Linear):
            m.reset_parameters()
    for m in module.modules():
        if isinstance(m, snipper_b200.MSDeformAttn):
            m._reset_parameters()
    with torch.no_grad():
        for name, p in module.named_parameters():
            if "sampling_offsets" in name and name.endswith("weight"):
                p.normal_(0, 0.02)
            elif "attention_weights" in name:
                p.normal_(0, 0.2)
            elif "norm" in name:
                p.copy_((1.0 if name.endswith("weight") else 0.0) + 0.2 * torch.randn_like(p))
            elif ("output_proj" in name or "value_proj" in name or "linear" in name) and name.endswith("bias"):
                p.normal_(0, 0.1)
    return module


def _level_inputs(N, padded, levels):
    """shapes, level_start_index, per-pixel padding mask (N,T,S,1) and valid ratios (N,L,2); ``padded``: the last
    batch element is padded on the right and at the bottom."""
    from snipper_b200.harness.snipper_net import Transformer
    masks = []
    for H, W in levels:
        m = torch.zeros(N, 1, T, H, W, dtype=torch.bool, device=DEV)
        if padded:
            m[-1, :, :, max(1, int(0.81 * H)):, :] = True
            m[-1, :, :, :, max(1, int(0.73 * W)):] = True
        masks.append(m)
    valid_ratios = torch.stack([Transformer.valid_ratio(m) for m in masks], 1)
    mask = torch.cat([m.flatten(3).permute(0, 2, 3, 1) for m in masks], 2)
    shapes = torch.as_tensor(levels, dtype=torch.long, device=DEV)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    return shapes, lsi, mask, valid_ratios


def _stack_checks(name, got, stock, want, failures):
    """The amp stack no less accurate than the stock autocast stack against float64: per row, amp error <= 2 x stock
    error + a floor.  The floor is the mean per-row stock error: the two stacks round to bf16 at the same places but
    from slightly different values, so on a row where stock happens to round well the amp stack must not fail; a
    wrong row or block is off by orders of magnitude more."""
    e_amp, e_stock = _row_abs_err(got, want), _row_abs_err(stock, want)
    bad = _worst_row(e_amp, 2 * e_stock + e_stock.mean(), want)
    if bad:
        failures.append("%s: %s" % (name, bad))


@pytest.mark.parametrize("N,padded,res_dtype", [(1, False, torch.float32), (2, True, torch.float32), (2, True, BF16)])
def test_encoder_layers_amp_vs_float64_at_bench_shapes(N, padded, res_dtype):
    """Three chained encoder layers under bf16 autocast.  Each layer hands the next its output in bf16 (value_proj's
    input) and out + pos in bf16 (the query), with the bits autocast's cast would give them.  A bf16 residual into
    the first layer is what the reference's encoder gets from its conv projection under autocast."""
    import snipper_b200
    from snipper_b200 import layers
    from snipper_b200.harness.snipper_net import Encoder, EncoderLayer
    from snipper_b200.modules import EncoderGrid
    enc = Encoder(EncoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 3)
    stock = _perturb(enc, 31 + N).to(DEV).eval()
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused, autocast=True) == 3
    shapes, lsi, mask, vr = _level_inputs(N, padded, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(N + 2 * padded)
    src = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen).to(res_dtype)
    pos = 0.5 * torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)

    def chain(layers_, x, p, ref):
        outs = []
        for layer in layers_:
            x = layer(x, p, ref, shapes, lsi, mask)
            outs.append(x)
        return outs

    with torch.no_grad():
        ref32 = Encoder.reference_points(LEVELS, vr, DEV).unsqueeze(1).expand(-1, T, -1, -1, -1)
        ref_d = Encoder.reference_points(LEVELS, vr.double(), DEV).unsqueeze(1).expand(-1, T, -1, -1, -1)
        want = chain(ref64.layers, src.double(), pos.double(), ref_d)
        with _bf16_autocast():
            base = chain(stock.layers, src, pos, ref32)
            got, n = _count(lambda: chain(fused.layers, src, pos, EncoderGrid(vr, LEVELS, T)))
    assert n == {"layer_tail": 0, "layer_tail_amp": 2 * 3}
    failures = []
    for i, (g, b, w) in enumerate(zip(got, base, want)):
        assert g.dtype == b.dtype == torch.float32
        _stack_checks("layer %d out" % i, g, b, w, failures)
        as16, plus_pos = getattr(g, layers._AS_BF16, None), getattr(g, layers._PLUS_POS, None)
        if i < 2:
            assert torch.equal(as16, g.to(BF16)), i
            assert plus_pos[0] is pos and torch.equal(plus_pos[1], (g + pos).to(BF16)), i
        else:                                       # the last layer hands nothing on
            assert as16 is None and plus_pos is None
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("N,padded", [(1, False), (2, True)])
@pytest.mark.parametrize("future", [0, 2])
def test_decoder_layers_amp_vs_float64_at_bench_shapes(future, N, padded):
    import snipper_b200
    from snipper_b200.harness.snipper_net import Decoder, DecoderLayer
    dec = Decoder(DecoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 2)
    stock = _perturb(dec, 41 + future).to(DEV).eval()
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused, autocast=True) == 2
    shapes, lsi, mask, vr = _level_inputs(N, padded, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    T1, NQ = T + future, 60
    gen = torch.Generator(device=DEV).manual_seed(200 + future + N)
    tgt = torch.randn(N, T1, NQ, D_MODEL, device=DEV, generator=gen)
    qpos = torch.randn(N, T1, NQ, D_MODEL, device=DEV, generator=gen)
    memory = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
    ref = (torch.rand(N, T1, NQ, 2, device=DEV, generator=gen) * 0.9 + 0.05)[:, :, :, None, :] * vr[:, None, None]

    def chain(layers_, x, qp, r, mem):
        outs = []
        for layer in layers_:
            x, _ = layer(x, qp, r, mem, shapes, lsi, mask)
            outs.append(x)
        return outs

    with torch.no_grad():
        want = chain(ref64.layers, tgt.double(), qpos.double(), ref.double(), memory.double())
        with _bf16_autocast():
            base = chain(stock.layers, tgt, qpos, ref, memory)
            got, n = _count(lambda: chain(fused.layers, tgt, qpos, ref, memory))
    assert n == {"layer_tail": 0, "layer_tail_amp": 3 * 2}
    failures = []
    for i, (g, b, w) in enumerate(zip(got, base, want)):
        assert g.dtype == b.dtype == torch.float32
        _stack_checks("layer %d out" % i, g, b, w, failures)
    assert not failures, "\n".join(failures)


# ============================================================================================================
# C. which path runs
# ============================================================================================================
class _Stack(nn.Module):
    def __init__(self, *layers_):
        super().__init__()
        self.layers = nn.ModuleList(layers_)


def _small_layer(kind, activation=None):
    import snipper_b200
    from snipper_b200.harness.snipper_net import DecoderLayer, EncoderLayer
    cls = EncoderLayer if kind == "encoder" else DecoderLayer
    layer = cls(snipper_b200.MSDeformAttn, 256, 512, 0.1, len(SMALL_LEVELS), 8, N_POINTS, T)
    if activation is not None:
        layer.activation = activation
    return _perturb(layer, 5).to(DEV).eval()


def _small_inputs(kind, seed=0):
    from snipper_b200.harness.snipper_net import Encoder
    shapes, lsi, mask, vr = _level_inputs(2, True, SMALL_LEVELS)
    S = sum(h * w for h, w in SMALL_LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    src = torch.randn(2, T, S, 256, device=DEV, generator=gen)
    if kind == "encoder":
        pos = torch.randn(2, T, S, 256, device=DEV, generator=gen)
        ref = Encoder.reference_points(SMALL_LEVELS, vr, DEV).unsqueeze(1).expand(-1, T, -1, -1, -1).contiguous()
        return [src, pos, ref, shapes, lsi, mask]
    tgt = torch.randn(2, T, 10, 256, device=DEV, generator=gen)
    qpos = torch.randn(2, T, 10, 256, device=DEV, generator=gen)
    ref = (torch.rand(2, T, 10, 2, device=DEV, generator=gen) * 0.9 + 0.05)[:, :, :, None, :] * vr[:, None, None]
    return [tgt, qpos, ref.contiguous(), src, shapes, lsi, mask]


def _out(res):
    return res[0] if isinstance(res, tuple) else res


def _run_as(layer, fn, **enable):
    """(fn(), the tail launches it made) with the layer's tails enabled with the keywords ``enable``."""
    import snipper_b200
    holder = _Stack(layer)
    assert snipper_b200.enable_fused_layer_tails(holder, **enable) == 1
    try:
        return _count(fn)
    finally:
        snipper_b200.disable_fused_layer_tails(holder)


NONE = {"layer_tail": 0, "layer_tail_amp": 0}


@pytest.mark.parametrize("kind", ["encoder", "decoder"])
def test_which_path_runs(kind):
    from snipper_b200 import layers
    layer = _small_layer(kind)
    args = _small_inputs(kind, seed=3)
    amp_tails = {"layer_tail": 0, "layer_tail_amp": 2 if kind == "encoder" else 3}
    fp32_tails = {"layer_tail": 2 if kind == "encoder" else 3, "layer_tail_amp": 0}

    def under(ctx):
        def fn():
            with torch.no_grad(), ctx():
                return _out(layer(*args)).clone()
        return fn

    stock_bf16, n = _count(under(_bf16_autocast))                              # the stock layer
    assert n == NONE
    got, n = _run_as(layer, under(_bf16_autocast), autocast=True)            # opt-in under bf16: amp tails only
    assert n == amp_tails and got.dtype == torch.float32
    assert rel_err(got, stock_bf16) < 5e-2
    got, n = _run_as(layer, under(_bf16_autocast))                           # default under bf16: stock
    assert n == NONE and torch.equal(got, stock_bf16)
    fp32_default, n = _run_as(layer, under(torch.no_grad))                    # no autocast: fp32 tails ...
    assert n == fp32_tails
    got, n = _run_as(layer, under(torch.no_grad), autocast=True)             # ... with or without the opt-in
    assert n == fp32_tails and torch.equal(got, fp32_default)

    # fp16 autocast: never the amp tails (the attention module does not take fp16, so the stock forward raises)
    import snipper_b200
    holder = _Stack(layer)
    snipper_b200.enable_fused_layer_tails(holder, autocast=True)
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            assert layers._eligible(layer, args[0], args[1], *args[2:]) is None
    finally:
        snipper_b200.disable_fused_layer_tails(holder)
    with torch.no_grad(), _bf16_autocast():
        assert layers._eligible(layer, args[0], args[1], *args[2:]) is None    # disabled: no flag left behind
    assert not hasattr(layer, "_amp_tails") and not hasattr(layer, "_stock_forward")


@pytest.mark.parametrize("kind", ["encoder", "decoder"])
def test_opt_in_keeps_the_stock_forward_where_the_tails_do_not_apply(kind):
    """Under bf16 autocast with the opt-in: an input that requires grad, active dropout or a non-ReLU activation runs
    the layer's own forward, bit for bit."""
    layer = _small_layer(kind)
    args = _small_inputs(kind, seed=9)

    def grad_input():
        a = list(args)
        a[1] = args[1].clone().requires_grad_(True)              # pos / query_pos from a trainable embedding
        with torch.autocast("cuda", dtype=BF16):
            return _out(layer(*a)).detach().clone()

    def seeded_train():
        torch.manual_seed(123)
        with torch.no_grad(), torch.autocast("cuda", dtype=BF16):
            return _out(layer(*args)).clone()

    layer.requires_grad_(False)
    want, n = _count(grad_input)
    got, n = _run_as(layer, grad_input, autocast=True)
    assert n == NONE and torch.equal(got, want)
    layer.train()
    want, _ = _count(seeded_train)
    got, n = _run_as(layer, seeded_train, autocast=True)
    assert n == NONE and torch.equal(got, want)
    layer.eval()
    layer.activation = F.gelu                       # what the reference's layers call; not ReLU: the layer's own forward
    want, _ = _count(seeded_train)
    got, n = _run_as(layer, seeded_train, autocast=True)
    assert n == NONE and torch.equal(got, want)


def test_enable_flag_updates_and_counts_only_new_layers():
    import snipper_b200
    holder = _Stack(_small_layer("encoder"), _small_layer("decoder"))
    assert snipper_b200.enable_fused_layer_tails(holder) == 2
    assert [l._amp_tails for l in holder.layers] == [False, False]
    assert snipper_b200.enable_fused_layer_tails(holder, autocast=True) == 0
    assert [l._amp_tails for l in holder.layers] == [True, True]
    assert snipper_b200.enable_fused_layer_tails(holder, autocast=False) == 0
    assert [l._amp_tails for l in holder.layers] == [False, False]
    assert snipper_b200.disable_fused_layer_tails(holder) == 2
    assert not any(hasattr(l, "_amp_tails") for l in holder.layers)


def _small_network():
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(5)
    net = build_snipper(snipper_b200.MSDeformAttn, num_frames=4, num_future_frames=0, enc_layers=2, dec_layers=2,
                        num_queries=7)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if "sampling_offsets" in n and n.endswith("weight"):
                p.normal_(0, 0.02)
            if "attention_weights" in n:
                p.normal_(0, 0.2)
    return net.to(DEV).eval()


def _predictions(out):
    res, _ = out
    return [res["pred_logits"], res["pred_kpts2d"], res["pred_depth"]] + list(res["heatmaps"])


def test_dtype_trace_of_the_small_network(monkeypatch):
    """The dtypes of y, the residual and pos that reach every tail of the small network under bf16 autocast: the GEMM
    outputs are bf16, the residual stream and the positional embeddings fp32."""
    import snipper_b200
    from snipper_b200 import layers
    net = _small_network()
    assert snipper_b200.enable_fused_layer_tails(net, autocast=True) == 4
    trace, tail = [], layers._tail

    def traced(y, bias, residual, norm, pos=None, amp=False, emit_bf16=False):
        trace.append((y.dtype, residual.dtype, None if pos is None else pos.dtype, amp, emit_bf16))
        return tail(y, bias, residual, norm, pos, amp, emit_bf16)

    monkeypatch.setattr(layers, "_tail", traced)
    x = torch.rand(1, 3 * T, 192, 256, device=DEV)
    with torch.no_grad(), _bf16_autocast():
        net(x)
    f32 = torch.float32
    enc = [(BF16, f32, None, True, True), (BF16, f32, f32, True, True)]          # layer 0 emits the next query
    enc_last = [(BF16, f32, None, True, True), (BF16, f32, None, True, False)]
    dec = [(BF16, f32, f32, True, False), (BF16, f32, None, True, True), (BF16, f32, None, True, False)]
    assert trace == enc + enc_last + dec + dec


# ============================================================================================================
# D. graph replay under bf16 autocast with the amp tails
# ============================================================================================================
def test_graph_replay_with_amp_tails():
    import snipper_b200
    from snipper_b200 import ops
    net = _small_network()
    assert snipper_b200.enable_fused_layer_tails(net, autocast=True) == 4

    def fn(x):
        out, _ = net(x)
        return {k: out[k] for k in ("pred_logits", "pred_kpts2d", "pred_depth")}

    xs = [torch.rand(1, 3 * T, 192, 256, device=DEV) for _ in range(2)]
    with torch.no_grad(), _bf16_autocast():
        eager = [{k: v.clone() for k, v in fn(x).items()} for x in xs]
        _, n = _count(lambda: fn(xs[0]))
        eager_launches = ops.STATS.launches
    assert n == {"layer_tail": 0, "layer_tail_amp": 2 * 2 + 3 * 2}
    runner = snipper_b200.GraphRunner(fn, autocast_dtype=BF16)
    for _ in range(2):
        for x, want in zip(xs, eager):
            got = runner(x)
            for k in want:
                assert torch.equal(got[k], want[k]), k
    assert runner.launches_per_replay(xs[0]) == eager_launches > 0


# ============================================================================================================
# E. the small network end to end
# ============================================================================================================
def test_small_network_amp_predictions_as_close_to_fp32_as_stock():
    """Under bf16 autocast, the opt-in network's predictions are no further from the fp32 network's than the stock
    autocast network's, within a factor 2 per prediction tensor (both round the same GEMM inputs to bf16; the
    amp tails add the biases in fp32)."""
    import snipper_b200
    net = _small_network()
    x = torch.rand(1, 3 * T, 192, 256, device=DEV)

    def run(ctx):
        with torch.no_grad(), ctx():
            return [t.float().clone() for t in _predictions(net(x))]

    fp32 = run(torch.no_grad)
    stock = run(_bf16_autocast)
    assert snipper_b200.enable_fused_layer_tails(net, autocast=True) == 4
    amp, n = _count(lambda: run(_bf16_autocast))
    assert n == {"layer_tail": 0, "layer_tail_amp": 10}
    report = []
    for i, (a, s, w) in enumerate(zip(amp, stock, fp32)):
        ea, es = rel_err(a, w), rel_err(s, w)
        report.append("pred %d: amp %.3e stock %.3e" % (i, ea, es))
        assert ea <= 2 * es + 1e-6, report

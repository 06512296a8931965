"""The fused layer tails against float64, and the rules that decide where they run (snipper_b200/layers.py).

A. ``layer_tail`` (csrc/msda_tail.cu) against a float64 LayerNorm, every instantiation C = 128*k, row counts on both
   sides of the kernel's 8 rows per block, rows that break a one-pass variance, layouts, aliases and guard bands.
B. The bench harness' encoder / decoder layers at the bench shapes: fused fp32 stack and stock fp32 stack against the
   same layers in float64 (whose MSDeformAttn runs the per-call float64 kernels, pinned to 1e-10 by test_module_gpu).
C. Eligibility: every case in which the fused forward would compute something else than the layer's own forward
   (autocast, inputs that require grad, a non-ReLU FFN, LayerNorm / Linear without parameters, unsupported widths,
   active dropout) runs the stock forward and gives its result.
D. CUDA-graph capture and replay under bf16 autocast with the tails enabled.

Errors are per row: max|got - want| over the row, against a bound of the same row, reported for the worst row.  A
whole-tensor maximum would hide a wrong partial last block or a single wrong row.
"""
import copy
import math

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24          # fp32 unit roundoff


@pytest.fixture(autouse=True)
def strict_fp32():
    """The float64 comparisons need the fp32 GEMMs of both stacks in full fp32, not TF32."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _row_abs_err(got, want):
    """max |got - want| of every row (last dim = channels), in float64."""
    return (got.double() - want.double()).abs().flatten(0, -2).amax(1)


def _worst_row(err, allowed, want):
    """'' when every row is within its bound, else a description of the worst row."""
    ratio = err / allowed
    i = int(ratio.argmax())
    if ratio[i] <= 1:
        return ""
    scale = want.double().flatten(0, -2).abs().amax(1)[i].clamp_min(1e-300)
    return "row %d of %d: err %.3e (rel %.3e) > allowed %.3e; %d rows over" % (
        i, err.numel(), err[i], err[i] / scale, allowed[i], int((ratio > 1).sum()))


def _ulp32(v):
    """fp32 ulp of the float64 magnitudes ``v`` (0 where v == 0)."""
    m, e = torch.frexp(v)
    return torch.where(v > 0, torch.ldexp(torch.ones_like(v), e - 24), torch.zeros_like(v))


def _count_tails(fn):
    """(fn(), number of layer_tail launches it issued)."""
    from snipper_b200 import ops
    ops.STATS.reset()
    ops.STATS.timing = True
    try:
        out = fn()
    finally:
        ops.STATS.timing = False
    return out, sum(e[0] == "layer_tail" for e in ops.STATS.events)


# ============================================================================================================
# A. the kernel against float64
# ============================================================================================================
ROWS = [1, 7, 8, 9, 240, 39500, 65541]        # 39500 = N*T*S of the bench encoder (not a multiple of 8), 240 = decoder
FAMILIES = ["normal", "offset_1e4", "offset_1e3", "constant", "outlier", "tiny", "gamma_zero_neg"]


def _tail_inputs(family, rows, C, gen):
    """y, residual, bias, pos, gamma, beta whose pre-norm rows residual + (y + bias) follow ``family``."""
    def n(*shape):
        return torch.randn(*shape, device=DEV, generator=gen)
    mean, std = {"offset_1e4": (1e4, 1.0), "offset_1e3": (1e3, 1e-2), "tiny": (0.0, 1e-20)}.get(family, (0.0, 1.0))
    s = std / math.sqrt(3)                                     # three addends of the row's spread
    y, residual, bias = n(rows, C) * s, mean + n(rows, C) * s, n(C) * s
    if family == "constant":                                   # y = bias = 0: the row is residual's constant
        residual = (n(rows, 1) * 3).expand(rows, C).contiguous()
        y, bias = torch.zeros_like(y), torch.zeros_like(bias)
    if family == "outlier":                                    # one channel per row carries nearly all the variance
        residual[torch.arange(rows, device=DEV), torch.randint(0, C, (rows,), device=DEV, generator=gen)] = 1e4
    gamma, beta = n(C), n(C)
    if family in ("tiny", "gamma_zero_neg"):                   # beta = 0 so that the normalised part is what is compared
        beta = torch.zeros(C, device=DEV)
    if family == "gamma_zero_neg":
        gamma = -gamma.abs()
        gamma[::3] = 0.0
        gamma[1::3] *= -1
    pos = n(rows, C)
    return y, residual, bias, pos, gamma, beta


def _tail_allowed(x32, want, gamma, eps32, torch_err):
    """Per-row error bound of the kernel: max of three terms.

    * 2 x the error of torch's own fp32 F.layer_norm on the same row: the kernel may not be less accurate than torch
      by more than a factor 2 on a row where torch's error is the largest term.
    * 8 fp32 ulps of the row's largest output.  The kernel rounds the subtraction, the product with rstd and the
      gamma/beta FMA once each, and rstd carries a few ulps of the squared-deviation sum; on the N(0,1) rows its worst
      row stays within 4 ulps, so 8 leaves a factor 2.
    * the rounding of the row mean, which every fp32 LayerNorm makes and which the normalisation amplifies by
      r = 1/sqrt(var + eps): |mean error| <= (VPL + 9) u mean|x| for a sum of depth VPL + 7 (VPL float4 per lane, the
      pair adds, 5 shuffle levels) plus the 1/C product, and it reaches every output as r |gamma| |mean error|.  This
      term is the bound on the offset rows (mean 1e4 / std 1, mean 1e3 / std 1e-2: mean|x| r is 1e4 and 1e5) and on
      the constant rows (variance 0, r = 1/sqrt(eps)): there the error of the kernel and of torch are both set by
      how the rounding of the mean falls on that row, so a per-row factor between the two is no bound.  A one-pass
      E[x^2] - E[x]^2 variance misses it by orders of magnitude on both offset families.
    """
    C = x32.shape[-1]
    x = x32.double()
    var = x.var(-1, unbiased=False)
    r = (var + eps32).rsqrt()
    mean_term = (C // 128 + 9) * U * r * x.abs().mean(-1) * gamma.double().abs().max()
    ulps = 8 * _ulp32(want.abs().amax(-1))
    return torch.maximum(torch.maximum(2 * torch_err, ulps), mean_term)


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("C", [128 * k for k in range(1, 9)])
def test_layer_tail_kernel_against_float64(C, family):
    import snipper_b200  # noqa: F401
    gen = torch.Generator(device=DEV).manual_seed(1000 * C + FAMILIES.index(family))
    failures = []
    for rows in ROWS:
        y, residual, bias_full, pos_full, gamma, beta = _tail_inputs(family, rows, C, gen)
        for eps in (1e-5, 1e-6):
            eps32 = float(torch.tensor(eps, dtype=torch.float32))         # the kernel takes eps as a float
            for with_bias in (True, False):
                bias = bias_full if with_bias else None
                # the oracle starts from the fp32 pre-norm row in the reference's order: residual + (y + bias)
                x32 = residual + (y + bias) if with_bias else residual + y
                want = F.layer_norm(x32.double(), (C,), gamma.double(), beta.double(), eps32)
                torch_err = _row_abs_err(F.layer_norm(x32, (C,), gamma, beta, eps32), want)
                allowed = _tail_allowed(x32, want, gamma, eps32, torch_err)
                for with_pos in (True, False):
                    pos = pos_full if with_pos else None
                    out, out_pos = torch.ops.snipper_b200.layer_tail(y, bias, residual, gamma, beta, pos, eps)
                    assert out.shape == (rows, C) and out.dtype == torch.float32
                    bad = _worst_row(_row_abs_err(out, want), allowed, want)
                    if bad:
                        failures.append("rows=%d eps=%g bias=%d pos=%d: %s" % (rows, eps, with_bias, with_pos, bad))
                    if with_pos:   # the kernel rounds out + pos once, as torch does
                        assert torch.equal(out_pos, out + pos), (rows, eps, with_bias)
                    else:
                        assert out_pos.numel() == 0
    assert not failures, "\n".join(failures)


def test_layer_tail_layouts_and_aliases():
    """Views are taken as they are, an operand may alias another, 4-D activations are rows too, zero rows is empty,
    and parameter vectors that are not contiguous are refused."""
    import snipper_b200  # noqa: F401
    lt = torch.ops.snipper_b200.layer_tail
    gen = torch.Generator(device=DEV).manual_seed(7)
    rows, C = 1000, 384
    y_t = torch.randn(C, rows, device=DEV, generator=gen).t()                 # transposed
    res_s = torch.randn(rows, 2 * C, device=DEV, generator=gen)[:, C:]         # column slice
    pos_s = torch.randn(2 * rows, C, device=DEV, generator=gen)[1::2]          # row stride 2
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    assert not (y_t.is_contiguous() or res_s.is_contiguous() or pos_s.is_contiguous())
    want = lt(y_t.contiguous(), bias, res_s.contiguous(), gamma, beta, pos_s.contiguous(), 1e-5)
    got = lt(y_t, bias, res_s, gamma, beta, pos_s, 1e-5)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])

    y = y_t.contiguous()
    want = lt(y, bias, y.clone(), gamma, beta, None, 1e-5)[0]
    assert torch.equal(lt(y, bias, y, gamma, beta, None, 1e-5)[0], want)                     # residual is y
    res = res_s.contiguous()
    want = lt(y, bias, res, gamma, beta, res.clone(), 1e-5)
    got = lt(y, bias, res, gamma, beta, res, 1e-5)                                          # pos is residual
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])

    y4 = torch.randn(2, 4, 60, C, device=DEV, generator=gen)
    r4 = torch.randn(2, 4, 60, C, device=DEV, generator=gen)
    got = lt(y4, bias, r4, gamma, beta, r4, 1e-5)
    want = lt(y4.reshape(-1, C), bias, r4.reshape(-1, C), gamma, beta, r4.reshape(-1, C), 1e-5)
    assert got[0].shape == y4.shape and torch.equal(got[0].reshape(-1, C), want[0])
    assert torch.equal(got[1].reshape(-1, C), want[1])

    e = torch.empty(0, C, device=DEV)
    out, out_pos = lt(e, bias, e, gamma, beta, e, 1e-5)
    assert out.shape == (0, C) and out_pos.shape == (0, C)
    out, out_pos = lt(e, None, e, gamma, beta, None, 1e-5)
    assert out.shape == (0, C) and out_pos.numel() == 0

    strided = torch.randn(2 * C, device=DEV)[::2]
    for args in ((y, strided, y, gamma, beta), (y, bias, y, strided, beta), (y, bias, y, gamma, strided)):
        with pytest.raises(RuntimeError, match="contiguous"):
            lt(*args, None, 1e-5)


@pytest.mark.parametrize("C", [128, 384, 1024])
@pytest.mark.parametrize("rows", [1, 9, 39500])
def test_layer_tail_writes_exactly_its_rows(rows, C):
    """Through the C ABI, outputs placed inside NaN-filled buffers at a 16-byte aligned offset: the kernel writes
    rows x C elements of each output, nothing before or after, and leaves its inputs as they were."""
    import snipper_b200  # noqa: F401
    from snipper_b200 import capi
    gen = torch.Generator(device=DEV).manual_seed(rows + C)
    y, res, pos = (torch.randn(rows, C, device=DEV, generator=gen) for _ in range(3))
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    inputs = (y, bias, res, gamma, beta, pos)
    before = [t.clone() for t in inputs]
    pad, n = 36, rows * C                                    # 36 floats = 144 bytes: 16-byte aligned, not 128
    bufs = [torch.full((pad + n + pad,), float("nan"), device=DEV) for _ in range(2)]
    out, out_pos = (b[pad:pad + n] for b in bufs)
    assert all(t.data_ptr() % 16 == 0 for t in (out, out_pos))
    status = capi.lib().msda_layer_tail(y.data_ptr(), bias.data_ptr(), res.data_ptr(), gamma.data_ptr(),
                                        beta.data_ptr(), pos.data_ptr(), out.data_ptr(), out_pos.data_ptr(), rows, C,
                                        1e-5, capi.MSDA_DTYPE_F32, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert status == capi.MSDA_OK
    want, want_pos = torch.ops.snipper_b200.layer_tail(y, bias, res, gamma, beta, pos, 1e-5)
    assert torch.equal(out.view(rows, C), want) and torch.equal(out_pos.view(rows, C), want_pos)
    for b in bufs:
        assert b[:pad].isnan().all() and b[pad + n:].isnan().all()
    for t, b in zip(inputs, before):
        assert torch.equal(t, b)


# ============================================================================================================
# B. harness layers at the bench shapes against their float64 copy
# ============================================================================================================
LEVELS = [(75, 100), (38, 50), (19, 25)]      # a 600x800 frame at strides 8 / 16 / 32
D_MODEL, FFN, HEADS, N_LEVELS, N_POINTS, T = 384, 1024, 8, 3, 4, 4


def _perturb(module, seed):
    """Random Linear weights per layer, then the MSDeformAttn init with the sampling-offset and attention-weight
    weights perturbed as the other GPU tests do (the init alone samples exactly on pixel centres); non-trivial
    LayerNorm parameters and projection biases so that every operand of the tails matters."""
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
            elif ("output_proj" in name or "value_proj" in name) and name.endswith("bias"):
                p.normal_(0, 0.1)
    return module


def _level_inputs(N, padded, levels):
    """shapes, level_start_index, per-pixel padding mask (N,T,S,1) and valid ratios (N,L,2) as the harness'
    Transformer derives them.  ``padded``: the last batch element is padded on the right and at the bottom."""
    from snipper_b200.harness.snipper_net import Transformer
    masks = []
    for H, W in levels:
        m = torch.zeros(N, 1, T, H, W, dtype=torch.bool, device=DEV)
        if padded:
            m[-1, :, :, max(1, int(0.81 * H)):, :] = True
            m[-1, :, :, :, max(1, int(0.73 * W)):] = True
        masks.append(m)
    valid_ratios = torch.stack([Transformer.valid_ratio(m) for m in masks], 1)
    if padded:
        assert (valid_ratios[-1] < 1).all()
    mask = torch.cat([m.flatten(3).permute(0, 2, 3, 1) for m in masks], 2)
    shapes = torch.as_tensor(levels, dtype=torch.long, device=DEV)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    return shapes, lsi, mask, valid_ratios


def _stack_checks(name, got, stock, want, failures):
    """Fused fp32 no less accurate than stock fp32 against float64: per row, fused error <= 2 x stock error + a floor,
    and the whole tensor within BASELINE.json's 1e-4.  The floor is the mean per-row stock error plus 16 fp32 ulps of
    the row's largest value: the two stacks round independently (the tails reorder the bias and residual adds, the
    FFN GEMMs run with other epilogues), and after a few layers a row on which stock happens to round well must not
    fail; a wrong row or block of the tails is off by orders of magnitude more."""
    e_fused, e_stock = _row_abs_err(got, want), _row_abs_err(stock, want)
    floor = e_stock.mean() + 16 * U * want.double().abs().flatten(0, -2).amax(1)
    bad = _worst_row(e_fused, 2 * e_stock + floor, want)
    if bad:
        failures.append("%s: %s" % (name, bad))
    if rel_err(got, want) >= 1e-4:
        failures.append("%s: rel_err %.3e >= 1e-4" % (name, rel_err(got, want)))


@pytest.mark.parametrize("N,padded", [(1, False), (1, True), (2, False), (2, True)])
def test_encoder_layers_fused_vs_float64_at_bench_shapes(N, padded):
    """Three chained encoder layers: the x + pos one tail hands the next layer and the reference points computed
    in-kernel from the valid ratios (EncoderGrid) are both on the path."""
    import snipper_b200
    from snipper_b200 import layers
    from snipper_b200.harness.snipper_net import Encoder, EncoderLayer
    from snipper_b200.modules import EncoderGrid
    enc = Encoder(EncoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 3)
    stock = _perturb(enc, 11 + N).to(DEV).eval()
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused) == 3
    shapes, lsi, mask, vr = _level_inputs(N, padded, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(N + 2 * padded)
    src = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
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
        base = chain(stock.layers, src, pos, ref32)
        got, n_tails = _count_tails(lambda: chain(fused.layers, src, pos, EncoderGrid(vr, LEVELS, T)))
    assert n_tails == 2 * 3
    failures = []
    for i, (g, b, w) in enumerate(zip(got, base, want)):
        _stack_checks("layer %d out" % i, g, b, w, failures)
        handoff = getattr(g, layers._PLUS_POS, None)
        if i < 2:                                   # layers 1 and 2 emit the next layer's query x + pos
            assert handoff is not None and handoff[0] is pos
            _stack_checks("layer %d x+pos" % i, handoff[1], b + pos, w + pos.double(), failures)
        else:
            assert handoff is None
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("N,padded", [(1, False), (2, True)])
@pytest.mark.parametrize("future", [0, 2])
def test_decoder_layers_fused_vs_float64_at_bench_shapes(future, N, padded):
    import snipper_b200
    from snipper_b200.harness.snipper_net import Decoder, DecoderLayer
    dec = Decoder(DecoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 2)
    stock = _perturb(dec, 21 + future).to(DEV).eval()
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused) == 2
    shapes, lsi, mask, vr = _level_inputs(N, padded, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    T1, NQ = T + future, 60
    gen = torch.Generator(device=DEV).manual_seed(100 + future + N)
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
        base = chain(stock.layers, tgt, qpos, ref, memory)
        got, n_tails = _count_tails(lambda: chain(fused.layers, tgt, qpos, ref, memory))
    assert n_tails == 3 * 2
    failures = []
    for i, (g, b, w) in enumerate(zip(got, base, want)):
        _stack_checks("layer %d out" % i, g, b, w, failures)
    assert not failures, "\n".join(failures)


# ============================================================================================================
# C. eligibility
# ============================================================================================================
SMALL_LEVELS = [(12, 16), (6, 8), (3, 4)]


class _Stack(nn.Module):
    """A parent with a ``layers`` list, which is where enable_fused_layer_tails looks for layers."""

    def __init__(self, *layers_):
        super().__init__()
        self.layers = nn.ModuleList(layers_)


class _ReferenceStyleEncoderLayer(nn.Module):
    """The reference's DeformableTransformerEncoderLayer (models/deformable_transformer.py:170-210): same attribute
    names, and the FFN activation is ``self.activation``."""

    def __init__(self, d_model, d_ffn, activation):
        super().__init__()
        import snipper_b200
        self.self_attn = snipper_b200.MSDeformAttn(d_model, len(SMALL_LEVELS), 8, N_POINTS, T, "encoder")
        self.dropout1, self.norm1 = nn.Dropout(0.1), nn.LayerNorm(d_model)
        self.linear1, self.activation, self.dropout2 = nn.Linear(d_model, d_ffn), activation, nn.Dropout(0.1)
        self.linear2, self.dropout3, self.norm2 = nn.Linear(d_ffn, d_model), nn.Dropout(0.1), nn.LayerNorm(d_model)

    def forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None):
        src2 = self.self_attn(src + pos, reference_points, src, spatial_shapes, level_start_index, padding_mask)
        src = self.norm1(src + self.dropout1(src2))
        src2 = self.linear2(self.dropout2(self.activation(self.linear1(src))))
        return self.norm2(src + self.dropout3(src2))


def _small_encoder_layer(d_model=256, heads=8):
    import snipper_b200
    from snipper_b200.harness.snipper_net import EncoderLayer
    return EncoderLayer(snipper_b200.MSDeformAttn, d_model, 512, 0.1, len(SMALL_LEVELS), heads, N_POINTS, T)


def _small_decoder_layer(d_model=256):
    import snipper_b200
    from snipper_b200.harness.snipper_net import DecoderLayer
    return DecoderLayer(snipper_b200.MSDeformAttn, d_model, 512, 0.1, len(SMALL_LEVELS), 8, N_POINTS, T)


def _small_inputs(kind, d_model, seed=0):
    """Keyword-free argument list of an encoder / decoder layer's forward at SMALL_LEVELS, N = 2, padded."""
    from snipper_b200.harness.snipper_net import Encoder
    shapes, lsi, mask, vr = _level_inputs(2, True, SMALL_LEVELS)
    S = sum(h * w for h, w in SMALL_LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    src = torch.randn(2, T, S, d_model, device=DEV, generator=gen)
    if kind == "encoder":
        pos = torch.randn(2, T, S, d_model, device=DEV, generator=gen)
        ref = Encoder.reference_points(SMALL_LEVELS, vr, DEV).unsqueeze(1).expand(-1, T, -1, -1, -1).contiguous()
        return [src, pos, ref, shapes, lsi, mask]
    tgt = torch.randn(2, T, 10, d_model, device=DEV, generator=gen)
    qpos = torch.randn(2, T, 10, d_model, device=DEV, generator=gen)
    ref = (torch.rand(2, T, 10, 2, device=DEV, generator=gen) * 0.9 + 0.05)[:, :, :, None, :] * vr[:, None, None]
    return [tgt, qpos, ref.contiguous(), src, shapes, lsi, mask]


def _out(res):
    return res[0] if isinstance(res, tuple) else res


def _fused_then_stock(layer, fn):
    """(result with the tails enabled, its layer_tail launches, result of the same layer with the tails disabled)"""
    import snipper_b200
    holder = _Stack(layer)
    assert snipper_b200.enable_fused_layer_tails(holder) == 1
    got, n = _count_tails(fn)
    assert snipper_b200.disable_fused_layer_tails(holder) == 1
    return got, n, fn()


def _per_row_close(got, want, tol):
    err = _row_abs_err(got, want)
    return _worst_row(err, tol * want.double().flatten(0, -2).abs().amax(1).clamp_min(1e-30), want)


def _small_layer(kind):
    return _perturb(_small_encoder_layer() if kind == "encoder" else _small_decoder_layer(), 5)


ENC_GRAD_ARGS = {"pos": 1, "reference_points": 2, "src": 0}
DEC_GRAD_ARGS = {"query_pos": 1, "reference_points": 2, "src": 3, "tgt": 0}


@pytest.mark.parametrize("kind,arg", [("encoder", a) for a in ENC_GRAD_ARGS] + [("decoder", a) for a in DEC_GRAD_ARGS])
def test_frozen_layer_with_an_input_that_requires_grad_runs_stock(kind, arg):
    """A frozen eval-mode layer fed a trainable input (e.g. pos from a trainable level_embed): the tail op has no
    autograd formula, so the stock forward must run and backward must give the stock gradients."""
    import snipper_b200
    layer = _small_layer(kind).to(DEV).eval().requires_grad_(False)
    args = _small_inputs(kind, 256, seed=4)
    i = (ENC_GRAD_ARGS if kind == "encoder" else DEC_GRAD_ARGS)[arg]
    go = torch.randn_like(_out(layer(*args)))

    def run():
        a = list(args)
        a[i] = args[i].clone().requires_grad_(True)
        out = _out(layer(*a))
        out.backward(go)
        return out.detach(), a[i].grad

    snipper_b200.set_deterministic(True)          # bit-reproducible backward: the two runs may be compared exactly
    (got, got_grad), n, (want, want_grad) = _fused_then_stock(layer, run)
    assert n == 0
    assert torch.equal(got, want)
    assert torch.equal(got_grad, want_grad)


def _gelu_layer():
    return _perturb(_ReferenceStyleEncoderLayer(256, 512, F.gelu), 5)


def _relu_layer():
    return _perturb(_ReferenceStyleEncoderLayer(256, 512, F.relu), 5)


def _norm_without_affine(kind):
    layer = _small_layer(kind)
    layer.norm2 = nn.LayerNorm(256, elementwise_affine=False)
    return layer


def _norm_without_bias(kind):
    layer = _small_layer(kind)
    setattr(layer, "norm1" if kind == "encoder" else "norm3", nn.LayerNorm(256, bias=False))
    return layer


def _linear_without_bias(kind, which):
    layer = _small_layer(kind)
    attn = layer.self_attn if kind == "encoder" else layer.cross_attn
    if which == "output_proj":
        attn.output_proj = nn.Linear(256, 256, bias=False)
    else:
        setattr(layer, which, nn.Linear(*getattr(layer, which).weight.shape[::-1], bias=False))
    return layer


# (case, layer factory, encoder or decoder, tails expected per call)
VARIANTS = [
    ("activation_gelu", _gelu_layer, "encoder", 0),
    ("activation_relu", _relu_layer, "encoder", 2),
    ("d_model_192", lambda: _perturb(_small_encoder_layer(192, 4), 5), "encoder", 0),
    ("d_model_256", lambda: _perturb(_small_encoder_layer(256, 8), 5), "encoder", 2),
]
for _k, _n in (("encoder", 2), ("decoder", 3)):
    VARIANTS += [
        ("%s_norm_no_affine" % _k, lambda k=_k: _norm_without_affine(k), _k, 0),
        ("%s_norm_no_bias" % _k, lambda k=_k: _norm_without_bias(k), _k, 0),
        ("%s_linear1_no_bias" % _k, lambda k=_k: _linear_without_bias(k, "linear1"), _k, 0),
        # the tail takes bias = None: a bias-less output_proj / linear2 keeps the fused path
        ("%s_output_proj_no_bias" % _k, lambda k=_k: _linear_without_bias(k, "output_proj"), _k, _n),
        ("%s_linear2_no_bias" % _k, lambda k=_k: _linear_without_bias(k, "linear2"), _k, _n),
    ]


@pytest.mark.parametrize("case,factory,kind,tails", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_layer_variants_take_the_path_that_computes_their_forward(case, factory, kind, tails):
    layer = factory().to(DEV).eval()      # the factories perturb before they swap a module for a bias-less one
    d_model = layer.linear2.weight.shape[0]
    args = _small_inputs(kind, d_model, seed=6)
    with torch.no_grad():
        got, n, want = _fused_then_stock(layer, lambda: _out(layer(*args)))
    assert n == tails
    if tails == 0:
        assert torch.equal(got, want)
    else:
        bad = _per_row_close(got, want, 1e-5)       # one layer, two op orders in fp32
        assert not bad, bad


def test_active_dropout_runs_stock_and_eval_mode_runs_fused():
    layer = _perturb(_small_encoder_layer(), 7).to(DEV)
    args = _small_inputs("encoder", 256, seed=8)

    def seeded():
        torch.manual_seed(123)                      # the same dropout masks in both runs
        return layer(*args)

    with torch.no_grad():
        layer.train()
        got, n, want = _fused_then_stock(layer, seeded)
        assert n == 0 and torch.equal(got, want)
        layer.eval()
        got, n, want = _fused_then_stock(layer, seeded)
    assert n == 2
    bad = _per_row_close(got, want, 1e-5)
    assert not bad, bad


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


def test_autocast_runs_the_stock_layers_bit_identically():
    """Under bf16 autocast the GEMMs feeding a tail return bf16: no tail may run, and the network with the tails
    enabled must give the bits of the network without them.  The encoder's in-kernel reference points (enabled with
    the tails) are computed in fp32 exactly as the reference-point tensor is; with bf16 values the kernels still
    take them in fp32, so they change no bit either."""
    import snipper_b200
    net = _small_network()
    x = torch.rand(1, 3 * T, 192, 256, device=DEV)
    assert snipper_b200.enable_fused_layer_tails(net) == 4

    def run():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            return [t.clone() for t in _predictions(net(x))]

    got, n = _count_tails(run)
    assert snipper_b200.disable_fused_layer_tails(net) == 4
    want = run()
    assert n == 0
    for a, b in zip(got, want):
        assert torch.equal(a, b)


# ============================================================================================================
# D. graph replay under autocast
# ============================================================================================================
def test_graph_replay_under_autocast_with_tails_enabled():
    import snipper_b200
    from snipper_b200 import ops
    net = _small_network()
    assert snipper_b200.enable_fused_layer_tails(net) == 4

    def fn(x):
        out, _ = net(x)
        return {k: out[k] for k in ("pred_logits", "pred_kpts2d", "pred_depth")}

    xs = [torch.rand(1, 3 * T, 192, 256, device=DEV) for _ in range(2)]
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        eager = [{k: v.clone() for k, v in fn(x).items()} for x in xs]
        _, n_tails = _count_tails(lambda: fn(xs[0]))
        eager_launches = ops.STATS.launches                     # _count_tails reset the counter
    assert n_tails == 0
    runner = snipper_b200.GraphRunner(fn, autocast_dtype=torch.bfloat16)
    for _ in range(2):
        for x, want in zip(xs, eager):
            got = runner(x)
            for k in want:
                assert torch.equal(got[k], want[k]), k
    assert runner.launches_per_replay(xs[0]) == eager_launches > 0

"""The training layer tails (libmsda_b200_train.so, ``layer_tail_train``, ``enable_fused_layer_tails(training=True)``).

1. Forward exactness: without a mask the kernel gives the bits of ``layer_tail``; with one, ``out`` has the bits of
   ``layer_tail`` on the pre-dropped input, h those of the fp32 residual add, and (mean, rstd) match float64.
2. Backward against float64 autograd of the same formula with the same mask, per row and per column, against the
   error of stock fp32 (dropout by mask + add + F.layer_norm).
3. Bit reproducibility of the backward, parameter gradients included.
4. NaN guard bands: the kernels write exactly their rows; views and misaligned inputs give the contiguous result.
5. The keep-masks: keep fraction, fresh per call, repeated under torch.manual_seed.
6. The bench harness' encoder / decoder layers at the bench shapes in train mode, output and every gradient against a
   float64 copy of the stock layers that applies the recorded masks.
7. Which forward runs (launches per STATS tag) in every case the opt-in does or does not cover.
8. One training step of the small network, and the peak memory of the encoder stack's training step.
"""
import copy
import math

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from conftest import rel_err
from test_layer_tails_oracle_gpu import (FAMILIES, LEVELS, _level_inputs, _perturb, _row_abs_err,
                                         _small_decoder_layer, _small_encoder_layer, _small_inputs, _Stack,
                                         _tail_inputs, _ulp32, _worst_row, _ReferenceStyleEncoderLayer)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
D_MODEL, FFN, HEADS, N_LEVELS, N_POINTS, T = 384, 1024, 8, 3, 4, 4


@pytest.fixture(autouse=True)
def strict_fp32():
    """The float64 comparisons need the fp32 GEMMs in full fp32, not TF32; every test starts deterministic-off."""
    import snipper_b200
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    snipper_b200.set_deterministic(False)


def _tt(*args):
    return torch.ops.snipper_b200.layer_tail_train(*args)


def _mask(shape, p, gen):
    return (torch.rand(shape, device=DEV, generator=gen) >= p).to(torch.uint8)


def _tags(fn):
    """(fn(), {tag: launches}) over the package's launches of fn."""
    from snipper_b200 import ops
    ops.STATS.reset()
    ops.STATS.timing = True
    try:
        out = fn()
        torch.cuda.synchronize()
    finally:
        ops.STATS.timing = False
    tags = {}
    for e in ops.STATS.events:
        tags[e[0]] = tags.get(e[0], 0) + 1
    return out, tags


# ============================================================================================================
# 1. forward exactness
# ============================================================================================================
ROWS = [1, 9, 240, 39500, 65541]


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("C", [128 * k for k in range(1, 9)])
def test_forward_is_layer_tail_on_the_pre_dropped_input(C, family):
    from snipper_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(3000 * C + FAMILIES.index(family))
    failures = []
    for rows in ROWS:
        y, residual, bias_full, pos_full, gamma, beta = _tail_inputs(family, rows, C, gen)
        for p in (0.0, 0.1, 0.5):
            mask = _mask((rows, C), p, gen) if p > 0 else None
            for with_bias, with_pos in ((True, True), (False, False), (True, False)):
                bias = bias_full if with_bias else None
                pos = pos_full if with_pos else None
                out, out_pos, h, mr = _tt(y, bias, residual, mask, p, gamma, beta, pos, 1e-5)
                yb = y + bias if with_bias else y
                if mask is None:
                    want = torch.ops.snipper_b200.layer_tail(y, bias, residual, gamma, beta, pos, 1e-5)
                    pre = yb
                else:
                    pre = (yb * ops.keep_scale(p)) * mask
                    want = torch.ops.snipper_b200.layer_tail(pre, None, residual, gamma, beta, pos, 1e-5)
                key = "rows=%d p=%g bias=%d pos=%d" % (rows, p, with_bias, with_pos)
                if not torch.equal(out, want[0]) or (with_pos and not torch.equal(out_pos, want[1])):
                    failures.append("%s: out differs from layer_tail" % key)
                if not with_pos:
                    assert out_pos.numel() == 0
                if not torch.equal(h, residual + pre):
                    failures.append("%s: h is not residual + d" % key)
                # (mean, rstd) against float64 of the fp32 row h
                h64 = h.double()
                mean64, var64 = h64.mean(-1), h64.var(-1, unbiased=False)
                eps32 = float(torch.tensor(1e-5, dtype=torch.float32))
                r64 = (var64 + eps32).rsqrt()
                delta = (C // 128 + 9) * U * h64.abs().mean(-1)          # the rounding of a row mean (oracle test)
                mean_ok = (mr[:, 0].double() - mean64).abs() <= delta + _ulp32(mean64.abs())
                rstd_rel = (mr[:, 1].double() - r64).abs() / r64
                rstd_ok = rstd_rel <= (C // 128 + 17) * U + 2 * r64 ** 2 * delta ** 2
                if not (mean_ok.all() and rstd_ok.all()):
                    failures.append("%s: mean_rstd off float64 on %d rows" % (key, int((~(mean_ok & rstd_ok)).sum())))
    assert not failures, "\n".join(failures)


# ============================================================================================================
# 2. backward against float64
# ============================================================================================================
def _formula(y, bias, residual, mask, scale, gamma, beta, pos, eps):
    """The tail in torch ops in the dtype of its inputs: dropout by ``mask``, add, F.layer_norm (+ pos)."""
    d = y + bias if bias is not None else y
    if mask is not None:
        d = (d * scale) * mask.to(d.dtype)
    out = F.layer_norm(residual + d, (y.shape[-1],), gamma, beta, eps)
    return out, (out + pos if pos is not None else None)


def _grads_of(args, go, gop, req):
    """Gradients of sum(out * go) + sum(out_pos * gop) with respect to the ``req`` entries of ``args``."""
    leaves = [a.detach().clone().requires_grad_(True) if (a is not None and i in req) else a for i, a in enumerate(args)]
    out, out_pos = _formula(*leaves)
    loss = (out * go).sum() + ((out_pos * gop).sum() if out_pos is not None else 0)
    gs = torch.autograd.grad(loss, [leaves[i] for i in req])
    return out.detach(), dict(zip(req, gs))


@pytest.mark.parametrize("C", [128, 384, 1024])
@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
def test_backward_against_float64(C, p):
    from snipper_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(C + int(100 * p))
    failures = []
    for rows in (9, 240, 39500):
        y, residual, bias, pos, gamma, beta = _tail_inputs("normal", rows, C, gen)
        mask = _mask((rows, C), p, gen) if p > 0 else None
        go = torch.randn(rows, C, device=DEV, generator=gen)
        gop = torch.randn(rows, C, device=DEV, generator=gen)
        for with_bias, with_pos in ((True, True), (False, False)):
            b = bias if with_bias else None
            ps = pos if with_pos else None
            # ours
            leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (y, b, residual)]
            g_, be_, ps_ = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True), \
                (ps.clone().requires_grad_(True) if ps is not None else None)
            out, out_pos, _, _ = _tt(leaves[0], leaves[1], leaves[2], mask, p, g_, be_, ps_, 1e-5)
            loss = (out * go).sum() + ((out_pos * gop).sum() if with_pos else 0)
            tensors = [leaves[0], leaves[2], g_, be_] + ([leaves[1]] if with_bias else []) + ([ps_] if with_pos else [])
            got = dict(zip(("y", "residual", "gamma", "beta", "bias", "pos")[:4] +
                           (("bias",) if with_bias else ()) + (("pos",) if with_pos else ()),
                           torch.autograd.grad(loss, tensors)))
            # float64 and stock fp32 of the same formula, same mask
            scale = ops.keep_scale(p)
            args = [y, b, residual, mask, scale, gamma, beta, ps, 1e-5]
            req = [0, 2, 5, 6] + ([1] if with_bias else []) + ([7] if with_pos else [])
            names = {0: "y", 1: "bias", 2: "residual", 5: "gamma", 6: "beta", 7: "pos"}
            a64 = [a.double() if torch.is_tensor(a) and a.is_floating_point() else a for a in args]
            _, w64 = _grads_of(a64, go.double(), gop.double(), req)
            _, s32 = _grads_of(args, go, gop, req)
            key = "rows=%d bias=%d pos=%d" % (rows, with_bias, with_pos)
            for i in req:
                n = names[i]
                want, stock, mine = w64[i], s32[i], got[n]
                if n in ("y", "residual"):
                    e_mine, e_stock = _row_abs_err(mine, want), _row_abs_err(stock, want)
                    allowed = torch.maximum(2 * e_stock, 8 * _ulp32(want.abs().flatten(0, -2).amax(1)))
                    bad = _worst_row(e_mine, allowed, want)
                else:
                    e_mine, e_stock = (mine.double() - want).abs(), (stock.double() - want).abs()
                    floor = 16 * U * math.sqrt(rows) * want.abs().max()
                    bad = "" if bool((e_mine <= 2 * e_stock + floor).all()) else \
                        "max err %.3e vs stock %.3e" % (e_mine.max(), e_stock.max())
                    if rel_err(mine, want) > 1e-4:
                        bad += " rel_err %.3e" % rel_err(mine, want)
                if bad:
                    failures.append("%s grad_%s: %s" % (key, n, bad))
    assert not failures, "\n".join(failures)


# ============================================================================================================
# 3. bit reproducibility
# ============================================================================================================
def test_backward_is_bit_reproducible():
    gen = torch.Generator(device=DEV).manual_seed(5)
    rows, C = 39500, 384
    y, residual, bias, pos, gamma, beta = _tail_inputs("normal", rows, C, gen)
    mask = _mask((rows, C), 0.1, gen)
    _, _, h, mr = _tt(y, bias, residual, mask, 0.1, gamma, beta, pos, 1e-5)
    go, gop = torch.randn(rows, C, device=DEV, generator=gen), torch.randn(rows, C, device=DEV, generator=gen)
    bwd = torch.ops.snipper_b200.layer_tail_train_backward
    first = bwd(go, gop, h, mr, mask, 0.1, gamma)
    for _ in range(2):
        again = bwd(go, gop, h, mr, mask, 0.1, gamma)
        for a, b in zip(first, again):
            assert torch.equal(a, b)


# ============================================================================================================
# 4. rows written, views, misaligned inputs
# ============================================================================================================
@pytest.mark.parametrize("C", [128, 384, 1024])
@pytest.mark.parametrize("rows", [1, 9, 39500])
def test_kernels_write_exactly_their_rows(rows, C):
    from snipper_b200 import capi, ops
    gen = torch.Generator(device=DEV).manual_seed(rows + C)
    y, res, pos, go, gop = (torch.randn(rows, C, device=DEV, generator=gen) for _ in range(5))
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    mask = _mask((rows, C), 0.1, gen)
    inputs = (y, bias, res, pos, gamma, beta, mask, go, gop)
    before = [t.clone() for t in inputs]
    pad = 36                                                   # 144 bytes: 16-byte aligned, not 128

    def banded(n):
        b = torch.full((pad + n + pad,), float("nan"), device=DEV)
        return b, b[pad:pad + n]

    (bo, out), (bop, out_pos), (bh, h), (bmr, mr) = (banded(rows * C), banded(rows * C), banded(rows * C),
                                                      banded(rows * 2))
    L = capi.train_lib()
    stream = torch.cuda.current_stream().cuda_stream
    s = ops.keep_scale(0.1)
    st = L.msda_train_layer_tail_forward(y.data_ptr(), bias.data_ptr(), res.data_ptr(), mask.data_ptr(), s,
                                         gamma.data_ptr(), beta.data_ptr(), pos.data_ptr(), out.data_ptr(),
                                         out_pos.data_ptr(), h.data_ptr(), mr.data_ptr(), rows, C, 1e-5, stream)
    assert st == capi.MSDA_OK
    ws_bytes = L.msda_train_layer_tail_workspace_bytes(rows, C)
    (bgr, gr), (bgy, gy), (bpg, pg), (bws, ws) = (banded(rows * C), banded(rows * C), banded(3 * C),
                                                  banded(ws_bytes // 4))
    st = L.msda_train_layer_tail_backward(go.data_ptr(), gop.data_ptr(), h.data_ptr(), mr.data_ptr(), mask.data_ptr(),
                                          s, gamma.data_ptr(), gr.data_ptr(), gy.data_ptr(), pg.data_ptr(),
                                          ws.data_ptr(), rows, C, stream)
    torch.cuda.synchronize()
    assert st == capi.MSDA_OK
    want = _tt(y, bias, res, mask, 0.1, gamma, beta, pos, 1e-5)
    for got, w in zip((out, out_pos, h, mr), want):
        assert torch.equal(got.view(w.shape), w)
    wb = torch.ops.snipper_b200.layer_tail_train_backward(go, gop, want[2], want[3], mask, 0.1, gamma)
    assert torch.equal(gr.view(rows, C), wb[0]) and torch.equal(gy.view(rows, C), wb[1])
    assert torch.equal(pg.view(3, C), wb[2])
    for b in (bo, bop, bh, bmr, bgr, bgy, bpg, bws):
        assert b[:pad].isnan().all() and b[-pad:].isnan().all()
    assert not ws.isnan().any()                                 # every partial row is written
    for t, b in zip(inputs, before):
        assert torch.equal(t, b)


def test_views_and_misaligned_inputs_give_the_contiguous_result():
    gen = torch.Generator(device=DEV).manual_seed(7)
    rows, C = 1000, 384
    y_t = torch.randn(C, rows, device=DEV, generator=gen).t()                   # transposed
    res_s = torch.randn(rows, 2 * C, device=DEV, generator=gen)[:, C:]          # column slice
    pos_m = torch.randn(rows * C + 1, device=DEV, generator=gen)[1:].view(rows, C)   # 4-byte offset: misaligned
    mask_m = _mask((rows * C + 3,), 0.1, gen)[3:].view(rows, C)                 # misaligned bytes
    bias, gamma, beta = (torch.randn(C, device=DEV, generator=gen) for _ in range(3))
    assert pos_m.data_ptr() % 16 and mask_m.data_ptr() % 16
    args = lambda yy, rr, mm, pp: (yy, bias, rr, mm, 0.1, gamma, beta, pp, 1e-5)   # noqa: E731
    want = _tt(*args(y_t.contiguous(), res_s.contiguous(), mask_m.clone(), pos_m.clone()))
    got = _tt(*args(y_t, res_s, mask_m, pos_m))
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    got_bool = _tt(*args(y_t, res_s, mask_m.bool(), pos_m))
    assert torch.equal(got_bool[0], want[0])
    go_m = torch.randn(rows * C + 1, device=DEV, generator=gen)[1:].view(rows, C)
    bwd = torch.ops.snipper_b200.layer_tail_train_backward
    wb = bwd(go_m.clone(), None, want[2], want[3], mask_m.clone(), 0.1, gamma)
    gb = bwd(go_m, None, want[2], want[3], mask_m, 0.1, gamma)
    for a, b in zip(gb, wb):
        assert torch.equal(a, b)

    # bias, gamma and beta that are contiguous but not 16-byte aligned (views into one flat parameter buffer): the op
    # copies them, and every copy must live until the kernel has read it.  Each call is repeated with the caching
    # allocator warm, which is when a copy freed too early is handed to the next one.
    flat = torch.randn(3 * C + 1, device=DEV, generator=gen)
    bias_m, gamma_m, beta_m = (flat[1 + i * C:1 + (i + 1) * C] for i in range(3))
    assert all(t.data_ptr() % 16 for t in (bias_m, gamma_m, beta_m))
    want = _tt(y_t, bias_m.clone(), res_s, mask_m, 0.1, gamma_m.clone(), beta_m.clone(), pos_m, 1e-5)
    wb = bwd(go_m, pos_m, want[2], want[3], mask_m, 0.1, gamma_m.clone())
    for _ in range(3):
        got = _tt(y_t, bias_m, res_s, mask_m, 0.1, gamma_m, beta_m, pos_m, 1e-5)
        for a, b in zip(got, want):
            assert torch.equal(a, b)
        gb = bwd(go_m, pos_m, want[2], want[3], mask_m, 0.1, gamma_m)
        for a, b in zip(gb, wb):
            assert torch.equal(a, b)
    with pytest.raises(RuntimeError, match="contiguous"):
        _tt(y_t, torch.randn(2 * C, device=DEV)[::2], res_s, None, 0.0, gamma, beta, None, 1e-5)
    with pytest.raises(RuntimeError, match=r"\[0, 1\)"):
        _tt(y_t, bias, res_s, mask_m, 1.0, gamma, beta, None, 1e-5)
    e = torch.empty(0, C, device=DEV)
    out, out_pos, h, mr = _tt(e, bias, e, None, 0.0, gamma, beta, e, 1e-5)
    assert out.shape == (0, C) and out_pos.shape == (0, C) and mr.shape == (0, 2)
    gr, gy, pg = bwd(e, None, h, mr, None, 0.0, gamma)
    assert gr.shape == (0, C) and torch.equal(pg, torch.zeros(3, C, device=DEV))


# ============================================================================================================
# 5. the keep-masks
# ============================================================================================================
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_keep_masks_are_torch_bernoulli(p):
    from snipper_b200 import layers
    n = 4 * 10 ** 6
    a = layers.draw_keep_mask((n,), p, DEV)
    b = layers.draw_keep_mask((n,), p, DEV)
    assert a.dtype == torch.uint8 and set(a.unique().tolist()) <= {0, 1}
    q = 1 - p
    sigma = math.sqrt(q * (1 - q) / n)
    for m in (a, b):
        assert abs(m.double().mean().item() - q) < 5 * sigma
    assert not torch.equal(a, b)
    torch.manual_seed(77)
    c = layers.draw_keep_mask((n,), p, DEV)
    torch.manual_seed(77)
    assert torch.equal(c, layers.draw_keep_mask((n,), p, DEV))


# ============================================================================================================
# 6. layers at the bench shapes, train mode, against a float64 copy applying the recorded masks
# ============================================================================================================
class _Recorder:
    """Stands in for layers.draw_keep_mask and keeps every mask it draws, in order."""

    def __init__(self, real):
        self.real, self.masks = real, []

    def __call__(self, shape, p, device):
        m = self.real(shape, p, device)
        self.masks.append((m, p))
        return m


class _MaskDropout(nn.Module):
    """A dropout that applies a given keep-mask: x * mask * scale."""

    def __init__(self, mask, scale):
        super().__init__()
        self.mask, self.scale = mask, scale

    def forward(self, x):
        return x * self.mask.to(x.dtype) * self.scale


def _replay(stack, masks, kind):
    """Replace every tail dropout of the layers of ``stack`` by the recorded mask it drew (in the tails' order)."""
    from snipper_b200 import layers, ops
    names = layers._TAIL_DROPOUTS[kind]
    it = iter(masks)
    for layer in stack.layers:
        for n in names:
            m, p = next(it)
            setattr(layer, n, _MaskDropout(m, ops.keep_scale(p)))
    assert next(it, None) is None


def _train_mode(stack):
    stack.train()
    for layer in stack.layers:
        (layer.dropout2 if hasattr(layer, "self_attn") and not hasattr(layer, "cross_attn") else layer.dropout3).p = 0.0
        if isinstance(getattr(layer, "self_attn", None), nn.MultiheadAttention):
            layer.self_attn.dropout = 0.0
    return stack


def _grad_checks(name, got, stock, want, failures):
    """Whole-tensor 2-norm: |fused - f64| <= 2 |stock - f64| + 1e-4 |f64|.  Not an elementwise maximum: the gradients
    upstream of the bilinear sampling are discontinuous in the sampling locations (a location that rounds into the
    next cell in fp32 switches its four corners), so single elements of either fp32 stack can be off by O(1) from
    float64, and the largest such element says which stack happened to round across a cell edge, not how accurate it
    is.  A wrong mask, a wrong gradient term or a wrong row is off by the whole size of the gradient."""
    e_f = (got.double() - want).norm()
    e_s = (stock.double() - want).norm()
    floor = 1e-4 * want.norm()
    if e_f > 2 * e_s + floor:
        failures.append("%s: err %.3e > 2 x stock %.3e + %.3e (2-norms)" % (name, e_f, e_s, floor))


def _compare_stacks(fused, stock, ref64, run, monkeypatch, kind):
    """run(stack, dtype) -> (outputs, leaves): forward the stack; compare outputs and every gradient."""
    from snipper_b200 import layers
    rec = _Recorder(layers.draw_keep_mask)
    monkeypatch.setattr(layers, "draw_keep_mask", rec)
    outs, leaves = run(fused, torch.float32, counting=True)
    n_layers = len(fused.layers)
    assert len(rec.masks) == n_layers * len(layers._TAIL_DROPOUTS[kind])
    _replay(stock, rec.masks, kind)
    _replay(ref64, rec.masks, kind)
    outs_s, leaves_s = run(stock, torch.float32)
    outs_w, leaves_w = run(ref64, torch.float64)
    failures = []
    for i, (g, s, w) in enumerate(zip(outs, outs_s, outs_w)):
        e_f, e_s = _row_abs_err(g, w), _row_abs_err(s, w)
        floor = e_s.mean() + 16 * U * w.double().abs().flatten(0, -2).amax(1)
        bad = _worst_row(e_f, 2 * e_s + floor, w)
        if bad:
            failures.append("output %d: %s" % (i, bad))
    gen = torch.Generator(device=DEV).manual_seed(99)
    gos = [torch.randn(o.shape, device=DEV, generator=gen) for o in outs]
    for model, os_, lv in ((fused, outs, leaves), (stock, outs_s, leaves_s), (ref64, outs_w, leaves_w)):
        torch.autograd.backward([o for o in os_], [g.to(o.dtype) for g, o in zip(gos, os_)])
    named = lambda m: dict(m.named_parameters())   # noqa: E731
    pf, ps, pw = named(fused), named(stock), named(ref64)
    for n in pf:
        if pf[n].grad is None:
            assert ps[n].grad is None, n
            continue
        _grad_checks(n, pf[n].grad, ps[n].grad, pw[n].grad.double(), failures)
    for n in leaves:
        _grad_checks("input " + n, leaves[n].grad, leaves_s[n].grad, leaves_w[n].grad.double(), failures)
    return failures


@pytest.mark.parametrize("padded", [False, True])
def test_encoder_layers_train_vs_float64_at_bench_shapes(padded, monkeypatch):
    import snipper_b200
    from snipper_b200.harness.snipper_net import Encoder, EncoderLayer
    enc = Encoder(EncoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 3)
    stock = _train_mode(_perturb(enc, 31 + padded).to(DEV))
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused, training=True) == 3
    N = 1
    shapes, lsi, mask, vr = _level_inputs(N, padded, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(7 + padded)
    src = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
    pos = 0.5 * torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
    sizes = [tuple(x) for x in LEVELS]

    def run(model, dtype, counting=False):
        leaves = {n: t.detach().clone().to(dtype).requires_grad_(True) for n, t in (("src", src), ("pos", pos))}

        def fwd():
            return [model(leaves["src"], sizes, shapes, lsi, vr.to(dtype), leaves["pos"], mask, T)]
        if counting:
            outs, tags = _tags(fwd)
            assert tags.get("layer_tail_train") == 2 * 3 and "layer_tail" not in tags, tags
            return outs, leaves
        return fwd(), leaves

    failures = _compare_stacks(fused, stock, ref64, run, monkeypatch, "encoder")
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("future", [0, 2])
def test_decoder_layers_train_vs_float64_at_bench_shapes(future, monkeypatch):
    import snipper_b200
    from snipper_b200.harness.snipper_net import Decoder, DecoderLayer
    dec = Decoder(DecoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 2)
    stock = _train_mode(_perturb(dec, 41 + future).to(DEV))
    fused = copy.deepcopy(stock)
    ref64 = copy.deepcopy(stock).double()
    assert snipper_b200.enable_fused_layer_tails(fused, training=True) == 2
    N = 1
    shapes, lsi, mask, vr = _level_inputs(N, True, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    T1, NQ = T + future, 60
    gen = torch.Generator(device=DEV).manual_seed(200 + future)
    tgt = torch.randn(N, T1, NQ, D_MODEL, device=DEV, generator=gen)
    qpos = torch.randn(N, T1, NQ, D_MODEL, device=DEV, generator=gen)
    memory = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
    ref = (torch.rand(N, T1, NQ, 2, device=DEV, generator=gen) * 0.9 + 0.05)

    def run(model, dtype, counting=False):
        leaves = {n: t.detach().clone().to(dtype).requires_grad_(True)
                  for n, t in (("tgt", tgt), ("qpos", qpos), ("memory", memory))}

        def fwd():
            outs = []
            x = leaves["tgt"]
            for layer in model.layers:
                r = ref.to(dtype)[:, :, :, None, :] * vr.to(dtype)[:, None, None]
                x, _ = layer(x, leaves["qpos"], r, leaves["memory"], shapes, lsi, mask)
                outs.append(x)
            return outs
        if counting:
            outs, tags = _tags(fwd)
            assert tags.get("layer_tail_train") == 3 * 2 and "layer_tail" not in tags, tags
            return outs, leaves
        return fwd(), leaves

    failures = _compare_stacks(fused, stock, ref64, run, monkeypatch, "decoder")
    assert not failures, "\n".join(failures)


# ============================================================================================================
# 7. which forward runs
# ============================================================================================================
def _run_layer(layer, args, grad):
    torch.manual_seed(123)                                   # the same stock dropout masks in every run
    with torch.set_grad_enabled(grad):
        res = layer(*args)
    out = res[0] if isinstance(res, tuple) else res
    if grad:
        out.sum().backward()
    return out.detach()


def _paths(layer, args, grad, **opt):
    """(out, tags) with the tails enabled with ``opt``, and the out of the same layer with them disabled."""
    import snipper_b200
    holder = _Stack(layer)
    assert snipper_b200.enable_fused_layer_tails(holder, **opt) == 1
    got, tags = _tags(lambda: _run_layer(layer, args, grad))
    assert snipper_b200.disable_fused_layer_tails(holder) == 1
    return got, tags, _run_layer(layer, args, grad)


TAIL_TAGS = ("layer_tail", "layer_tail_amp", "layer_tail_train", "layer_tail_train_backward")


def _tail_tags(tags):
    return {t: tags[t] for t in TAIL_TAGS if t in tags}


@pytest.mark.parametrize("kind", ["encoder", "decoder"])
def test_default_keeps_training_stock_and_opt_in_runs_the_train_tails(kind):
    layer = _perturb(_small_encoder_layer() if kind == "encoder" else _small_decoder_layer(), 5).to(DEV).train()
    args = _small_inputs(kind, 256, seed=4)
    n = 2 if kind == "encoder" else 3
    got, tags, want = _paths(layer, args, True)
    assert _tail_tags(tags) == {} and torch.equal(got, want)
    got, tags, _ = _paths(layer, args, True, training=True)
    assert _tail_tags(tags) == {"layer_tail_train": n, "layer_tail_train_backward": n}
    assert torch.isfinite(got).all()


def test_eval_no_grad_with_the_opt_in_runs_the_inference_tails_bit_identically():
    import snipper_b200
    layer = _perturb(_small_encoder_layer(), 5).to(DEV).eval()
    args = _small_inputs("encoder", 256, seed=4)
    holder = _Stack(layer)
    snipper_b200.enable_fused_layer_tails(holder)
    with torch.no_grad():
        want, tags_a = _tags(lambda: layer(*args))
        snipper_b200.enable_fused_layer_tails(holder, training=True)
        got, tags_b = _tags(lambda: layer(*args))
    assert _tail_tags(tags_a) == _tail_tags(tags_b) == {"layer_tail": 2}
    assert torch.equal(got, want)


def test_bf16_autocast_keeps_stock_in_training_and_amp_tails_under_no_grad():
    import snipper_b200
    layer = _perturb(_small_encoder_layer(), 5).to(DEV).train()
    args = _small_inputs("encoder", 256, seed=4)
    holder = _Stack(layer)
    snipper_b200.enable_fused_layer_tails(holder, autocast=True, training=True)

    def step(grad):
        torch.manual_seed(1)
        with torch.set_grad_enabled(grad), torch.autocast("cuda", dtype=torch.bfloat16):
            return layer(*args)
    _, tags = _tags(lambda: step(True))
    assert _tail_tags(tags) == {}
    layer.eval()
    _, tags = _tags(lambda: step(False))
    assert _tail_tags(tags) == {"layer_tail_amp": 2}


def _p_one(kind):
    layer = _perturb(_small_encoder_layer() if kind == "encoder" else _small_decoder_layer(), 5)
    layer.dropout1.p = 1.0
    return layer


def _non_affine(kind):
    layer = _perturb(_small_encoder_layer() if kind == "encoder" else _small_decoder_layer(), 5)
    layer.norm2 = nn.LayerNorm(256, elementwise_affine=False)
    return layer


STOCK_CASES = [("gelu", lambda: _perturb(_ReferenceStyleEncoderLayer(256, 512, F.gelu), 5), "encoder"),
               ("encoder_norm_no_affine", lambda: _non_affine("encoder"), "encoder"),
               ("decoder_norm_no_affine", lambda: _non_affine("decoder"), "decoder"),
               ("encoder_p1", lambda: _p_one("encoder"), "encoder"),
               ("decoder_p1", lambda: _p_one("decoder"), "decoder")]


@pytest.mark.parametrize("case,factory,kind", STOCK_CASES, ids=[c[0] for c in STOCK_CASES])
def test_uncovered_layers_train_stock(case, factory, kind):
    layer = factory().to(DEV).train()
    args = _small_inputs(kind, 256, seed=6)
    got, tags, want = _paths(layer, args, True, training=True)
    assert _tail_tags(tags) == {}
    assert torch.equal(got, want)


def test_reference_style_relu_layer_takes_the_train_tails():
    layer = _perturb(_ReferenceStyleEncoderLayer(256, 512, F.relu), 5).to(DEV).train()
    args = _small_inputs("encoder", 256, seed=6)
    _, tags, _ = _paths(layer, args, True, training=True)
    assert _tail_tags(tags) == {"layer_tail_train": 2, "layer_tail_train_backward": 2}


# ============================================================================================================
# 8. end to end
# ============================================================================================================
def _small_train_network():
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(5)
    net = build_snipper(snipper_b200.MSDeformAttn, num_frames=4, num_future_frames=0, enc_layers=2, dec_layers=2,
                        num_queries=7, dropout=0.0)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if "sampling_offsets" in n and n.endswith("weight"):
                p.normal_(0, 0.02)
            if "attention_weights" in n:
                p.normal_(0, 0.2)
    return net.to(DEV).train()


def _loss(out):
    loss = out["pred_kpts2d"].square().mean() + out["pred_depth"].square().mean() + out["pred_logits"].square().mean()
    for h in out["heatmaps"]:
        loss = loss + h.square().mean()
    return loss


def test_one_training_step_of_the_small_network_matches_stock():
    import snipper_b200
    stock = _small_train_network()
    fused = copy.deepcopy(stock)
    assert snipper_b200.enable_fused_layer_tails(fused, training=True) == 4
    x = torch.rand(1, 3 * T, 192, 256, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    results = []
    for net in (stock, fused):
        params = [p for p in net.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)
        out, tags = _tags(lambda: _loss(net(x)[0]))
        loss = out
        loss.backward()
        grads = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
        torch.nn.utils.clip_grad_norm_(params, 0.1)
        opt.step()
        results.append((float(loss.detach()), grads, {n: p.detach().clone() for n, p in net.named_parameters()},
                        _tail_tags(tags)))
    (l0, g0, p0, t0), (l1, g1, p1, t1) = results
    assert t0 == {} and t1 == {"layer_tail_train": 2 * 2 + 3 * 2}
    assert abs(l1 - l0) <= 1e-5 * abs(l0)
    assert g0.keys() == g1.keys()
    scale = max(float(g.abs().max()) for g in g0.values())
    bad = [n for n in g0 if float((g1[n] - g0[n]).abs().max()) > 1e-3 * float(g0[n].abs().max()) + 1e-6 * scale]
    assert not bad, bad
    # AdamW's first step moves an element by lr * g / (|g| + eps) (+ the decay): lr * sign(g) wherever |g| >> eps.
    # Only elements whose gradient is at the level of eps or of rounding noise can move differently, by <= 2 lr.
    lr = 1e-4
    for n in p0:
        d = (p1[n] - p0[n]).abs()
        assert float(d.max()) <= 2.001 * lr, n
        assert int((d > 0.1 * lr).sum()) <= max(1, d.numel() // 1000), n


def test_peak_memory_of_the_encoder_training_step_is_no_higher_than_stock():
    import snipper_b200
    from snipper_b200.harness.snipper_net import Encoder, EncoderLayer
    enc = Encoder(EncoderLayer(snipper_b200.MSDeformAttn, D_MODEL, FFN, 0.1, N_LEVELS, HEADS, N_POINTS, T), 6)
    stock = _perturb(enc, 3).to(DEV).train()
    fused = copy.deepcopy(stock)
    snipper_b200.enable_fused_layer_tails(fused, training=True)
    N = 2
    shapes, lsi, mask, vr = _level_inputs(N, True, LEVELS)
    S = sum(h * w for h, w in LEVELS)
    gen = torch.Generator(device=DEV).manual_seed(1)
    src = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)
    pos = torch.randn(N, T, S, D_MODEL, device=DEV, generator=gen)

    def peak(model):
        for _ in range(2):                                     # the second step is the one measured
            model.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            p = pos.clone().requires_grad_(True)
            out = model(src, LEVELS, shapes, lsi, vr, p, mask, T)
            out.square().mean().backward()
            torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    p_stock, p_fused = peak(stock), peak(fused)
    assert p_fused <= 1.01 * p_stock, (p_fused, p_stock)

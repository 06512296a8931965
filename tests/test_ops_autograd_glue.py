"""The autograd glue of the fused ops without a device: on ``meta`` tensors autograd runs the real setup-context and
backward formulas of snippet_attn / snippet_forward through the fake kernels, so the gradient each input receives
(its shape, or None) is checked here for every combination of the optional inputs."""
import itertools

import pytest
import torch

import snipper_b200  # noqa: F401  (registers the ops)

N, T2, T1, S, M, D, L, P, N_FRAME = 2, 4, 4, 50, 8, 48, 3, 4, 4


def _meta(*shape, grad=False, dtype=torch.float32):
    return torch.empty(*shape, device="meta", dtype=dtype).requires_grad_(grad)


def _check_grads(tensors, wanted):
    for name, t in tensors.items():
        if t is None:
            continue
        if name in wanted:
            assert t.grad is not None and t.grad.shape == t.shape, (name, t.grad)
        else:
            assert t.grad is None, name


@pytest.mark.parametrize("presum,planar", [(False, False), (True, False), (True, True)])
@pytest.mark.parametrize("biases", [False, True])
@pytest.mark.parametrize("refs", ["reference_points", "valid_ratios"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("wanted", [("value", "proj", "offsets_bias", "logits_bias", "reference_points"), ("value",),
                                    ("proj", "reference_points"), ("offsets_bias", "logits_bias")])
def test_snippet_attn_gradients(presum, planar, biases, refs, masked, wanted):
    Lq = S if refs == "valid_ratios" else 7
    t = dict(value=_meta(N, T2, S, M, D, grad="value" in wanted),
             proj=_meta(N, T1, Lq, 3 * M * L * P, grad="proj" in wanted),
             offsets_bias=_meta(2 * M * L * P, grad="offsets_bias" in wanted) if biases else None,
             logits_bias=_meta(M * L * P, grad="logits_bias" in wanted) if biases else None,
             reference_points=_meta(N, T1, Lq, L, 2, grad="reference_points" in wanted)
             if refs == "reference_points" else None)
    if not any(v is not None and v.requires_grad for v in t.values()):
        pytest.skip("no input of this combination requires grad")
    shapes = _meta(L, 2, dtype=torch.long)
    lsi = _meta(L, dtype=torch.long)
    vr = _meta(N, L, 2) if refs == "valid_ratios" else None
    mask = _meta(N, T2, S, M * D, dtype=torch.bool) if masked else None
    out, carry = torch.ops.snipper_b200.snippet_attn(t["value"], mask, shapes, lsi, t["proj"], t["offsets_bias"],
                                                     t["logits_bias"], t["reference_points"], vr, N_FRAME, presum,
                                                     planar)
    assert out.shape == (N, T1, Lq, M * D)
    out.backward(torch.empty_like(out))
    _check_grads(t, wanted)


@pytest.mark.parametrize("wanted", [c for n in range(1, 5) for c in itertools.combinations(
    ("value", "offsets", "logits", "reference_points"), n)])
def test_snippet_forward_gradients(wanted):
    Lq = 7
    t = dict(value=_meta(N, T2, S, M, D, grad="value" in wanted),
             offsets=_meta(N, T1, Lq, M, L, P, 2, grad="offsets" in wanted),
             logits=_meta(N, T1, Lq, M, L, P, grad="logits" in wanted),
             reference_points=_meta(N, T1, Lq, L, 2, grad="reference_points" in wanted))
    out = torch.ops.snipper_b200.snippet_forward(t["value"], _meta(L, 2, dtype=torch.long), _meta(L, dtype=torch.long),
                                                 t["offsets"], t["logits"], t["reference_points"], N_FRAME)
    assert out.shape == (N, T1, Lq, M * D)
    out.backward(torch.empty_like(out))
    _check_grads(t, wanted)

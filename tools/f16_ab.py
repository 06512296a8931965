"""float16 against bfloat16 storage, in one process: the fused encoder op through the C ABI, graph-replayed inference
of the bench network under autocast, and training steps under autocast.

    python tools/f16_ab.py --out DIR [--rounds 6] [--replays 20] [--train-steps 3]

Writes DIR/f16_ab.json with the GPU's name, power limit and max SM clock (read in the same run) and:
  * c_abi: the fused encoder forward (msda_frame_sum + presummed gather) and backward (presummed scatter +
    msda_frame_unsum) at N = 1, T = 4, S = 9875 (600x800 pyramid), M = 8, D = 48, L = 3, P = 4, in the "init" regime
    (pixel-centre reference points plus a fixed per-head direction, what a freshly initialised Snipper samples):
    CUDA events around 10 back-to-back launch pairs, median and min of 30 such samples, warm L2; fp16 and bf16 timed
    side by side (libmsda_b200_f16.so against libmsda_b200.so with MSDA_DTYPE_BF16);
  * inference: snippets/s of GraphRunner replay of the bench network (batch 1, 600x800, T = 4) under fp16 and bf16
    autocast, arms alternating round by round, and each arm's rel_err against the fp32 network;
  * training: ms per step of the tools/trainbench.py step (batch 2, AdamW, gradient clipping) under fp16 autocast with
    torch.amp.GradScaler and under bf16 autocast, arms alternating round by round.
Both arms run the stock layers (no fused layer tails exist for fp16).
"""
import argparse
import copy
import json
import math
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (seeded inputs and the packed result of bench.py)
from tools.amp_tails_ab import gpu_info  # noqa: E402
from tools.trainbench import synthetic_loss  # noqa: E402

LEVELS = [(75, 100), (38, 50), (19, 25)]


def encoder_calls(half, M=8, D=48, P=4, T=4, seed=0):
    """(forward, backward) closures of the fused encoder layer through the C ABI, ``half`` = torch.float16 or bfloat16"""
    from snipper_b200 import capi
    f16 = half == torch.float16
    L, F = capi.lib(), capi.f16_lib()
    g = torch.Generator().manual_seed(seed)
    shapes = torch.as_tensor(LEVELS, dtype=torch.long)
    Lv, S = len(LEVELS), int(shapes.prod(1).sum())
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    th = torch.arange(M, dtype=torch.float32) * (2.0 * math.pi / M)
    dd = torch.stack([th.cos(), th.sin()], -1)
    dd = dd / dd.abs().max(-1, keepdim=True)[0]
    offsets = (dd.view(1, 1, 1, M, 1, 1, 2) * torch.arange(1, P + 1, dtype=torch.float32).view(1, 1, 1, 1, 1, P, 1)
               ).expand(1, T, S, M, Lv, P, 2).contiguous().cuda()
    logits = torch.randn(1, T, S, M, Lv, P, generator=g).cuda()
    refs = []
    for H, W in LEVELS:
        ys, xs = torch.meshgrid(torch.arange(H) + 0.5, torch.arange(W) + 0.5, indexing="ij")
        refs.append(torch.stack([xs.reshape(-1) / W, ys.reshape(-1) / H], -1))
    ref = torch.cat(refs, 0)[None, None, :, None, :].expand(1, T, S, Lv, 2).contiguous().cuda()
    value = torch.randn(1, T, S, M, D, generator=g).to(half).cuda()
    go = torch.randn(1, T, S, M * D, generator=g).to(half).cuda()
    out = torch.empty_like(go)
    slots = L.msda_snippet_num_slots(T, T)
    vsum = torch.empty(1, slots, S, M, D, device="cuda", dtype=half)
    gsum = torch.empty(1, slots, S, M, D, device="cuda")
    gv, goff, glog = torch.empty_like(value), torch.empty_like(offsets), torch.empty_like(logits)
    shapes, lsi = shapes.cuda(), lsi.cuda()
    st = torch.cuda.current_stream().cuda_stream
    keep = (value, offsets, logits, ref, go, out, vsum, gsum, gv, goff, glog, shapes, lsi)
    PRE = capi.MSDA_FLAG_PRESUMMED
    dt = () if f16 else (capi.MSDA_DTYPE_BF16,)
    ws = () if f16 else (None, 0)
    lib = F if f16 else L
    pre = "msda_f16_" if f16 else "msda_"
    frame_sum, frame_unsum = getattr(lib, pre + "frame_sum"), getattr(lib, pre + "frame_unsum")
    snip_fwd, snip_bwd = getattr(lib, pre + "snippet_forward"), getattr(lib, pre + "snippet_backward")
    common = (shapes.data_ptr(), lsi.data_ptr(), offsets.data_ptr(), logits.data_ptr(), ref.data_ptr())
    dims = (1, T, T, T, S, M, D, Lv, S, P, 0, 0, 0, 0, 0, 0, None, None, None, None, 0, 0)

    def fwd():
        r = frame_sum(value.data_ptr(), None, vsum.data_ptr(), 1, T, T, T, S, M * D, 0, 0, 0, 0, *dt, st)
        assert r == 0, r
        r = snip_fwd(vsum.data_ptr(), *common, out.data_ptr(), *dims, *dt, PRE, st)
        assert r == 0, r

    def bwd():
        r = snip_bwd(vsum.data_ptr(), *common, go.data_ptr(), gsum.data_ptr(), goff.data_ptr(), glog.data_ptr(), *dims,
                     *dt, PRE, *ws, st)
        assert r == 0, r
        r = frame_unsum(gsum.data_ptr(), None, gv.data_ptr(), 1, T, T, T, S, M * D, 0, 0, *dt, st)
        assert r == 0, r

    return fwd, bwd, keep


def time_us(fn, samples=30, inner=10):
    """median and min over ``samples`` of the per-call device time of ``inner`` back-to-back calls (warm L2)"""
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(samples):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(inner):
            fn()
        e.record()
        e.synchronize()
        t.append(s.elapsed_time(e) * 1e3 / inner)
    return {"us_median": statistics.median(t), "us_min": min(t)}


def c_abi(rounds):
    calls = {name: encoder_calls(dt) for name, dt in (("f16", torch.float16), ("bf16", torch.bfloat16))}
    res = {name: {"forward": [], "backward": []} for name in calls}
    for r in range(rounds):                                      # arms alternate, order flipped every round
        for name in (("f16", "bf16") if r % 2 == 0 else ("bf16", "f16")):
            fwd, bwd, _ = calls[name]
            res[name]["forward"].append(time_us(fwd)["us_median"])
            res[name]["backward"].append(time_us(bwd)["us_median"])
    return {name: {k: {"us_median": statistics.median(v), "us_per_round": v} for k, v in r.items()}
            for name, r in res.items()}


def inference(rounds, replays):
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper
    dev = torch.device("cuda", 0)
    torch.manual_seed(42)                                        # bench.py's weights
    model = build_snipper(snipper_b200.MSDeformAttn).to(dev).eval()
    xs = [x.to(dev) for x in bench.synthetic_snippets(bench.N_INPUTS, seed=1000)]

    def forward_packed(x):
        out, _ = model(x)
        return bench.pack_result(out).float()

    with torch.no_grad():
        fp32 = [forward_packed(x).clone() for x in xs]
    arms = {name: dict(runner=snipper_b200.GraphRunner(forward_packed, warmup=2, autocast_dtype=dt), ms=[])
            for name, dt in (("f16", torch.float16), ("bf16", torch.bfloat16))}
    for a in arms.values():
        for i in range(3 * replays):
            a["runner"](xs[i % len(xs)])
    torch.cuda.synchronize()
    for r in range(rounds):
        for name in (("f16", "bf16") if r % 2 == 0 else ("bf16", "f16")):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(replays):
                arms[name]["runner"](xs[i % len(xs)])
            e.record()
            torch.cuda.synchronize()
            arms[name]["ms"].append(s.elapsed_time(e) / replays)
    out = {}
    for name, a in arms.items():
        errs = [float((a["runner"](x).double() - w.double()).abs().max() / w.double().abs().max())
                for x, w in zip(xs, fp32)]
        med = statistics.median(a["ms"])
        out[name] = {"ms_per_snippet_median": med, "snippets_per_s": 1e3 / med, "ms_per_round": a["ms"],
                     "rel_err_vs_fp32": errs}
    return out


def training(rounds, steps, batch=2):
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper
    dev = torch.device("cuda", 0)
    torch.manual_seed(42)
    base = build_snipper(snipper_b200.MSDeformAttn).to(dev).train()
    g = torch.Generator().manual_seed(1000)
    xs = [torch.rand(batch, 12, 600, 800, generator=g).to(dev) for _ in range(2)]
    arms = {}
    for name, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        model = copy.deepcopy(base)
        params = [p for p in model.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)
        scaler = torch.amp.GradScaler("cuda", enabled=dt == torch.float16)
        arms[name] = dict(model=model, params=params, opt=opt, scaler=scaler, dtype=dt, ms=[], losses=[])

    def step(a, i):
        with torch.autocast("cuda", dtype=a["dtype"]):
            out, _ = a["model"](xs[i % len(xs)])
            loss = synthetic_loss(out)
        a["opt"].zero_grad(set_to_none=True)
        a["scaler"].scale(loss).backward()
        a["scaler"].unscale_(a["opt"])
        torch.nn.utils.clip_grad_norm_(a["params"], 0.1)     # reference engine.py:75
        a["scaler"].step(a["opt"])
        a["scaler"].update()
        return loss

    for a in arms.values():
        for i in range(3):
            step(a, i)
    torch.cuda.synchronize()
    for r in range(rounds):
        for name in (("f16", "bf16") if r % 2 == 0 else ("bf16", "f16")):
            a = arms[name]
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(steps):
                loss = step(a, i)
            e.record()
            torch.cuda.synchronize()
            a["ms"].append(s.elapsed_time(e) / steps)
            a["losses"].append(float(loss.detach()))
    return {name: {"ms_per_step_median": statistics.median(a["ms"]), "ms_per_round": a["ms"],
                   "snippets_per_s": batch * 1e3 / statistics.median(a["ms"]), "final_losses": a["losses"],
                   "grad_scale": a["scaler"].get_scale() if a["dtype"] == torch.float16 else None}
            for name, a in arms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory for f16_ab.json")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--replays", type=int, default=20, help="graph replays per inference arm and round")
    ap.add_argument("--train-steps", type=int, default=3, help="training steps per arm and round")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "f16_ab.py needs a CUDA device"
    result = {"gpu": gpu_info(0), "torch": torch.__version__, "rounds": args.rounds,
              "c_abi": {"what": "fused encoder layer, N=1 T=4 S=9875 M=8 D=48 L=3 P=4, init regime, warm L2; "
                                "forward = frame_sum + presummed gather, backward = presummed scatter + frame_unsum; "
                                "CUDA events, median of 30 samples of 10 calls, per round",
                        **c_abi(args.rounds)},
              "inference": {"what": bench.WORKLOAD + ", GraphRunner replay under autocast, %d replays per arm and "
                                                     "round" % args.replays, **inference(args.rounds, args.replays)},
              "training": {"what": "tools/trainbench.py step at batch 2 under autocast (fp16 with GradScaler), "
                                   "%d steps per arm and round" % args.train_steps,
                           **training(args.rounds, args.train_steps)}}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "f16_ab.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    c = result["c_abi"]
    print(json.dumps({"c_abi_us": {k: {d: c[k][d]["us_median"] for d in ("forward", "backward")} for k in ("f16", "bf16")},
                      "inference_snippets_per_s": {k: result["inference"][k]["snippets_per_s"] for k in ("f16", "bf16")},
                      "train_ms_per_step": {k: result["training"][k]["ms_per_step_median"] for k in ("f16", "bf16")},
                      "gpu": result["gpu"], "json": path}))


if __name__ == "__main__":
    main()

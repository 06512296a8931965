"""A/B of the layer tails in training: the tools/trainbench.py step with the stock layers against
``enable_fused_layer_tails(model, training=True)`` (``layer_tail_train``), eager, one process.  With ``--bf16`` both
arms run under torch.autocast("cuda", dtype=torch.bfloat16) and the fused arm is
``enable_fused_layer_tails(model, amp_training=True)`` (``layer_tail_amp_train``).

    python tools/train_tails_ab.py --out DIR [--bf16] [--rounds 6] [--steps 5] [--warmup 3] [--profile-steps 2]

The step is trainbench.py's: forward, synthetic loss over every head, backward, clip_grad_norm_(0.1), AdamW; batch 2,
T = 4, 600x800, dropout 0.1, fp32.  Both arms are ONE model whose tails are switched on and off; they are timed
alternately (``--rounds`` blocks of ``--steps`` steps each, the arm order flipped every round).  Writes
DIR/train_tails_ab.json (DIR/train_tails_ab_bf16.json with ``--bf16``):

  * ms per step of each arm: median over the rounds, min, max, and the median / min / max of the per-round
    fused - stock differences;
  * peak memory of a step of each arm (torch.cuda.max_memory_allocated);
  * from a separate torch.profiler run of fused steps: us per training tail launch, forward and backward, and its
    bytes/s against the algorithmic bytes of that launch;
  * the GPU's name, power limit and max SM clock, read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from amp_tails_ab import gpu_info  # noqa: E402
from trainbench import synthetic_loss  # noqa: E402


def fwd_bytes(dims):
    """Forward launch: read y, residual (+ 1-byte mask) (+ pos), write out, h (+ out_pos), 8 bytes of (mean, rstd) per
    row, plus bias / gamma / beta."""
    rows, C, mask, pos = dims
    return rows * C * (4 + 4 + mask + 4 + 4 + 8 * pos) + 8 * rows + 3 * 4 * C


def bwd_bytes(dims):
    """Backward launch pair: read grad_out (+ grad_out_pos), h (+ mask), (mean, rstd); write grad_residual, grad_y.
    The CTA partials (under 4 MB) are left out."""
    rows, C, mask, pos = dims
    return rows * C * (4 + 4 * pos + 4 + mask + 4 + 4) + 8 * rows + 4 * C


def amp_fwd_bytes(dims):
    """bf16 forward launch: read y (bf16), residual (fp32 or bf16) (+ mask) (+ pos, fp32), write out, h, (mean, rstd)
    (+ the bf16 copy of out) (+ the bf16 out + pos), plus bias / gamma / beta."""
    rows, C, res_bytes, mask, emit, pos = dims
    return rows * C * (2 + res_bytes + mask + 4 + 4 + 2 * emit + 6 * pos) + 8 * rows + 3 * 4 * C


def amp_bwd_bytes(dims):
    """bf16 backward launch pair: read grad_out (+ the bf16 gradients of the copies), h (+ mask), (mean, rstd); write
    grad_residual (fp32 or bf16), grad_y (bf16).  The CTA partials are left out."""
    rows, C, res_bytes, mask, b16, pos = dims
    return rows * C * (4 + 2 * b16 + 2 * pos + 4 + mask + res_bytes + 2) + 8 * rows + 4 * C


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory for train_tails_ab.json")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=5, help="training steps per arm and round")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm before the first round")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--bf16", action="store_true", help="both arms under bf16 autocast, the fused arm amp_training=True")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "train_tails_ab.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    import snipper_b200
    from snipper_b200 import ops
    from snipper_b200.harness.snipper_net import build_snipper

    torch.manual_seed(42)                                        # trainbench.py's weights and inputs
    model = build_snipper(snipper_b200.MSDeformAttn).to(dev).train()
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)
    g = torch.Generator().manual_seed(1000)
    xs = [torch.rand(args.batch, 12, 600, 800, generator=g).to(dev) for _ in range(2)]

    def step(i):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=args.bf16):
            out, _ = model(xs[i % len(xs)])
            loss = synthetic_loss(out)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 0.1)
        opt.step()

    def set_arm(fused):
        if fused:
            return snipper_b200.enable_fused_layer_tails(model, **({"amp_training": True} if args.bf16 else
                                                                   {"training": True}))
        return snipper_b200.disable_fused_layer_tails(model)

    fused_arm = "amp_train_tails" if args.bf16 else "train_tails"
    fwd_tag = "layer_tail_amp_train" if args.bf16 else "layer_tail_train"
    arms = {"stock": dict(fused=False, ms=[]), fused_arm: dict(fused=True, ms=[])}
    order = list(arms)
    for name in order:                                           # warm-up, launch counts and peak memory per arm
        set_arm(arms[name]["fused"])
        for i in range(args.warmup):
            step(i)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ops.STATS.reset()
        ops.STATS.timing = True
        step(0)
        torch.cuda.synchronize()
        ops.STATS.timing = False
        arms[name]["peak_bytes"] = torch.cuda.max_memory_allocated()
        tags = {}
        for e in ops.STATS.events:
            tags[e[0]] = tags.get(e[0], 0) + 1
        arms[name]["launches_per_step"] = tags
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            set_arm(arms[name]["fused"])
            step(0)                                              # one untimed step after the switch
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(args.steps):
                step(i)
            e.record()
            torch.cuda.synchronize()
            arms[name]["ms"].append(s.elapsed_time(e) / args.steps)

    # separate profiler run: fused steps, kernel time of every training tail launch.  STATS records the dims of every
    # launch in launch order; everything runs on one stream, so the i-th forward (backward) kernel the profiler sees is
    # the i-th forward (backward) launch STATS recorded
    set_arm(True)
    from torch.profiler import ProfilerActivity, profile
    step(0)
    torch.cuda.synchronize()
    ops.STATS.reset()
    ops.STATS.timing = True
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(args.profile_steps):
            step(i)
        torch.cuda.synchronize()
    ops.STATS.timing = False
    fwd_dims = [e[1] for e in ops.STATS.events if e[0] == fwd_tag]
    bwd_dims = [e[1] for e in ops.STATS.events if e[0] == fwd_tag + "_backward"]
    evs = sorted((ev for ev in prof.events() if ev.device_type.name == "CUDA" and
                  (fwd_tag + "_fwd_kernel" in ev.name or fwd_tag + "_bwd_kernel" in ev.name or
                   "layer_tail_param_sum_kernel" in ev.name)), key=lambda ev: ev.time_range.start)
    fwd_us = [ev.time_range.elapsed_us() for ev in evs if "fwd_kernel" in ev.name]
    bwd_us = [ev.time_range.elapsed_us() for ev in evs if "bwd_kernel" in ev.name]
    sum_us = [ev.time_range.elapsed_us() for ev in evs if "param_sum_kernel" in ev.name]

    def by_dims(dims, us, nbytes, what):
        """one row per distinct launch dims: median / min kernel time and bytes/s of the algorithmic bytes"""
        if len(us) != len(dims):
            return []
        per = {}
        for d, t in zip(dims, us):
            per.setdefault(d, []).append(t)
        rows = []
        for d, ts in sorted(per.items()):
            med = statistics.median(ts)
            rows.append({**dict(zip(dim_names, d)), "launches": len(ts), "us_median": med, "us_min": min(ts),
                         "bytes": nbytes(d), "GB_per_s": nbytes(d) / med / 1e3, "kernel": what})
        return rows

    if args.bf16:
        dim_names = ("rows", "C", "residual_bytes", "mask", "bf16_copy", "pos")
        forward = by_dims(fwd_dims, fwd_us, amp_fwd_bytes, fwd_tag + "_fwd_kernel")
        dim_names = ("rows", "C", "grad_residual_bytes", "mask", "bf16_grad", "pos_grad")
        backward = by_dims(bwd_dims, bwd_us, amp_bwd_bytes, fwd_tag + "_bwd_kernel (without the parameter sum)")
    else:
        dim_names = ("rows", "C", "mask", "pos")
        forward = by_dims(fwd_dims, fwd_us, fwd_bytes, "layer_tail_train_fwd_kernel")
        backward = by_dims(bwd_dims, bwd_us, bwd_bytes, "layer_tail_train_bwd_kernel (without the parameter sum)")

    result = {"gpu": gpu_info(0), "torch": torch.__version__,
              "step": "tools/trainbench.py step: forward, synthetic loss, backward, clip_grad_norm_(0.1), AdamW; "
                      "batch %d, T = 4, 600x800, dropout 0.1, %s" % (
                          args.batch, "bf16 autocast" if args.bf16 else "fp32 (torch default TF32 settings)"),
              "rounds": args.rounds, "steps_per_round": args.steps, "warmup": args.warmup, "arms": {},
              "train_tail_profile": {"forward_launches_per_step": len(fwd_dims) // args.profile_steps,
                                     "backward_launches_per_step": len(bwd_dims) // args.profile_steps,
                                     "forward_kernels_seen": len(fwd_us), "backward_kernels_seen": len(bwd_us),
                                     "param_sum_kernels_seen": len(sum_us),
                                     "param_sum_us_median": statistics.median(sum_us) if sum_us else None,
                                     "forward": forward, "backward": backward,
                                     "us_per_step": (sum(fwd_us) + sum(bwd_us) + sum(sum_us)) / args.profile_steps}}
    for name in order:
        a = arms[name]
        result["arms"][name] = {"ms_per_step_median": statistics.median(a["ms"]), "ms_min": min(a["ms"]),
                                "ms_max": max(a["ms"]), "ms_per_round": a["ms"],
                                "snippets_per_s": args.batch * 1e3 / statistics.median(a["ms"]),
                                "peak_memory_bytes": a["peak_bytes"], "launches_per_step": a["launches_per_step"]}
    diffs = [b - a for a, b in zip(arms["stock"]["ms"], arms[fused_arm]["ms"])]
    result[fused_arm + "_minus_stock_ms"] = {"median": statistics.median(diffs), "min": min(diffs), "max": max(diffs)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "train_tails_ab_bf16.json" if args.bf16 else "train_tails_ab.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    summary = {k: result["arms"][k]["ms_per_step_median"] for k in order}
    print(json.dumps({"ms_per_step": summary, fused_arm + "_minus_stock_ms": result[fused_arm + "_minus_stock_ms"],
                      "peak_bytes": {k: result["arms"][k]["peak_memory_bytes"] for k in order},
                      "gpu": result["gpu"], "json": path}))


if __name__ == "__main__":
    main()

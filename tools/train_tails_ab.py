"""A/B of the layer tails in training: the tools/trainbench.py step with the stock layers against
``enable_fused_layer_tails(model, training=True)`` (``layer_tail_train``), eager, one process.

    python tools/train_tails_ab.py --out DIR [--rounds 6] [--steps 5] [--warmup 3] [--profile-steps 2]

The step is trainbench.py's: forward, synthetic loss over every head, backward, clip_grad_norm_(0.1), AdamW; batch 2,
T = 4, 600x800, dropout 0.1, fp32.  Both arms are ONE model whose tails are switched on and off; they are timed
alternately (``--rounds`` blocks of ``--steps`` steps each, the arm order flipped every round).  Writes
DIR/train_tails_ab.json:

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory for train_tails_ab.json")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=5, help="training steps per arm and round")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per arm before the first round")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--batch", type=int, default=2)
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
        out, _ = model(xs[i % len(xs)])
        loss = synthetic_loss(out)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 0.1)
        opt.step()

    def set_arm(fused):
        if fused:
            return snipper_b200.enable_fused_layer_tails(model, training=True)
        return snipper_b200.disable_fused_layer_tails(model)

    arms = {"stock": dict(fused=False, ms=[]), "train_tails": dict(fused=True, ms=[])}
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
    fwd_dims = [e[1] for e in ops.STATS.events if e[0] == "layer_tail_train"]
    bwd_dims = [e[1] for e in ops.STATS.events if e[0] == "layer_tail_train_backward"]
    evs = sorted((ev for ev in prof.events() if ev.device_type.name == "CUDA" and
                  ("layer_tail_train_fwd_kernel" in ev.name or "layer_tail_train_bwd_kernel" in ev.name or
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
            rows.append({"rows": d[0], "C": d[1], "mask": d[2], "pos": d[3], "launches": len(ts), "us_median": med,
                         "us_min": min(ts), "bytes": nbytes(d), "GB_per_s": nbytes(d) / med / 1e3, "kernel": what})
        return rows

    forward = by_dims(fwd_dims, fwd_us, fwd_bytes, "layer_tail_train_fwd_kernel")
    backward = by_dims(bwd_dims, bwd_us, bwd_bytes, "layer_tail_train_bwd_kernel (without the parameter sum)")

    result = {"gpu": gpu_info(0), "torch": torch.__version__,
              "step": "tools/trainbench.py step: forward, synthetic loss, backward, clip_grad_norm_(0.1), AdamW; "
                      "batch %d, T = 4, 600x800, dropout 0.1, fp32 (torch default TF32 settings)" % args.batch,
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
    diffs = [b - a for a, b in zip(arms["stock"]["ms"], arms["train_tails"]["ms"])]
    result["train_tails_minus_stock_ms"] = {"median": statistics.median(diffs), "min": min(diffs), "max": max(diffs)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "train_tails_ab.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    summary = {k: result["arms"][k]["ms_per_step_median"] for k in order}
    print(json.dumps({"ms_per_step": summary, "train_tails_minus_stock_ms": result["train_tails_minus_stock_ms"],
                      "peak_bytes": {k: result["arms"][k]["peak_memory_bytes"] for k in order},
                      "gpu": result["gpu"], "json": path}))


if __name__ == "__main__":
    main()

"""A/B of the layer tails under bf16 autocast: the bench network with the default tails (stock layers under autocast)
against the opt-in ``enable_fused_layer_tails(model, autocast=True)`` (``layer_tail_amp``), both graph-replayed.

    python tools/amp_tails_ab.py --out DIR [--rounds 10] [--steps 50] [--profile-steps 5]

Same network, weights and seeded inputs as ``bench.py --precision bf16`` (T = 4, 600x800, batch 1).  The two arms are
two CUDA graphs of ONE model, captured with the flag off and on, and timed alternately in one process (``--rounds``
blocks of ``--steps`` replays each, the arm order flipped every round).  Writes DIR/amp_tails_ab.json:

  * ms per snippet of each arm: median over the rounds, min, max, and the median of the per-round B - A differences;
  * package launches per replay of each arm and the tail launches of one eager step per tag;
  * from a separate torch.profiler run of eager opt-in steps: us per amp tail launch and its bytes/s against the
    algorithmic bytes of that launch (read y, residual (+ pos), write out (+ the bf16 copies));
  * rel_err (max |d| / max |ref|) of each arm's predictions against the fp32 network on the same inputs;
  * the GPU's name, power limit and max SM clock, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (seeded inputs and the packed result of bench.py)


def gpu_info(index):
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        line = "unavailable: %r" % (e,)
    return {"torch_name": torch.cuda.get_device_name(index), "nvidia_smi": dict(zip(q.split(","), line.split(", ")))}


def tail_bytes(dims):
    """Algorithmic bytes of one amp tail launch: y bf16 + residual (+ pos fp32) read, out fp32 (+ bf16 copies) written,
    plus bias / gamma / beta."""
    rows, C, res_bytes, emit, pos = dims
    per_elem = 2 + res_bytes + 4 + 2 * emit + (4 + 2) * pos
    return rows * C * per_elem + 3 * 4 * C


def tail_launches(fn):
    from snipper_b200 import ops
    ops.STATS.reset()
    ops.STATS.timing = True
    fn()
    torch.cuda.synchronize()
    ops.STATS.timing = False
    tags = [e[0] for e in ops.STATS.events]
    dims = [e[1] for e in ops.STATS.events if e[0] == "layer_tail_amp"]
    return {t: tags.count(t) for t in ("layer_tail", "layer_tail_amp")}, dims


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory for amp_tails_ab.json")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--steps", type=int, default=50, help="replays per arm and round")
    ap.add_argument("--warmup", type=int, default=120, help="untimed replays per arm before the first round")
    ap.add_argument("--profile-steps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "amp_tails_ab.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    import snipper_b200
    from snipper_b200.harness.snipper_net import build_snipper

    torch.manual_seed(42)                                        # bench.py's weights
    model = build_snipper(snipper_b200.MSDeformAttn).to(dev).eval()
    n_layers = snipper_b200.enable_fused_layer_tails(model)
    xs = [x.to(dev) for x in bench.synthetic_snippets(bench.N_INPUTS, seed=1000)]

    def forward_packed(x):
        out, _ = model(x)
        return bench.pack_result(out).float()

    def set_arm(amp):
        snipper_b200.enable_fused_layer_tails(model, autocast=amp)

    def eager(x, bf16):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            return forward_packed(x)

    # the fp32 network (fp32 tails) and the eager launch counts of each arm
    fp32 = [eager(x, False).clone() for x in xs]
    arms = {}
    for name, amp in (("stock", False), ("amp_tails", True)):
        set_arm(amp)
        tails, dims = tail_launches(lambda: eager(xs[0], True))
        runner = snipper_b200.GraphRunner(forward_packed, warmup=2, autocast_dtype=torch.bfloat16)
        arms[name] = dict(runner=runner, launches_per_replay=runner.launches_per_replay(xs[0]),
                          tail_launches_per_eager_step=tails, amp_dims=dims, ms=[])
    order = list(arms)

    for name in order:                                           # steady state before the first timed round
        for i in range(args.warmup):
            arms[name]["runner"](xs[i % len(xs)])
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            runner = arms[name]["runner"]
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(args.steps):
                runner(xs[i % len(xs)])
            e.record()
            torch.cuda.synchronize()
            arms[name]["ms"].append(s.elapsed_time(e) / args.steps)

    # accuracy: each arm's replayed predictions against the fp32 network, input by input
    for name in order:
        errs = []
        for x, want in zip(xs, fp32):
            got = arms[name]["runner"](x)
            errs.append(float((got.double() - want.double()).abs().max() / want.double().abs().max()))
        arms[name]["rel_err_vs_fp32"] = errs
    torch.cuda.synchronize()

    # separate profiler run: eager opt-in steps, kernel time of every amp tail launch
    set_arm(True)
    from torch.profiler import ProfilerActivity, profile
    eager(xs[0], True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(args.profile_steps):
            eager(xs[i % len(xs)], True)
        torch.cuda.synchronize()
    kern = sorted((ev for ev in prof.events() if "layer_tail_amp_kernel" in ev.name and ev.device_type.name == "CUDA"),
                  key=lambda ev: ev.time_range.start)
    dims = arms["amp_tails"]["amp_dims"]
    per_dims = {}
    if len(kern) == len(dims) * args.profile_steps:
        for i, ev in enumerate(kern):
            per_dims.setdefault(dims[i % len(dims)], []).append(ev.time_range.elapsed_us())
    profile_rows = []
    for d, us in sorted(per_dims.items()):
        med = statistics.median(us)
        profile_rows.append({"rows": d[0], "C": d[1], "residual_bytes": d[2], "emit_bf16": d[3], "pos": d[4],
                             "launches": len(us), "us_median": med, "us_min": min(us), "bytes": tail_bytes(d),
                             "GB_per_s": tail_bytes(d) / med / 1e3})
    us_step = sum(sum(v) for v in per_dims.values()) / max(args.profile_steps, 1)
    by_name = [{"kernel": e.key, "launches": e.count, "us_avg": e.device_time_total / e.count}
               for e in prof.key_averages() if "layer_tail_amp_kernel" in e.key]

    result = {"gpu": gpu_info(0), "torch": torch.__version__, "network": bench.WORKLOAD + " under bf16 autocast",
              "fused_layers": n_layers, "rounds": args.rounds, "steps_per_round": args.steps, "warmup": args.warmup,
              "arms": {}, "amp_tail_profile": {"kernels_seen": len(kern), "expected": len(dims) * args.profile_steps,
                                               "us_per_step": us_step, "launches": profile_rows,
                                               "by_kernel": by_name}}
    for name in order:
        a = arms[name]
        result["arms"][name] = {"ms_per_snippet_median": statistics.median(a["ms"]), "ms_min": min(a["ms"]),
                                "ms_max": max(a["ms"]), "ms_per_round": a["ms"],
                                "launches_per_replay": a["launches_per_replay"],
                                "tail_launches_per_eager_step": a["tail_launches_per_eager_step"],
                                "rel_err_vs_fp32": a["rel_err_vs_fp32"]}
    diffs = [b - a for a, b in zip(arms["stock"]["ms"], arms["amp_tails"]["ms"])]
    result["amp_minus_stock_ms"] = {"median": statistics.median(diffs), "min": min(diffs), "max": max(diffs)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "amp_tails_ab.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    summary = {k: result["arms"][k]["ms_per_snippet_median"] for k in order}
    print(json.dumps({"ms_per_snippet": summary, "amp_minus_stock_ms": result["amp_minus_stock_ms"],
                      "gpu": result["gpu"], "json": path}))


if __name__ == "__main__":
    main()

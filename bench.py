"""bench.py -- headline benchmark of the B200-native MSDeformAttn engine for Snipper.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], the config the metric is quoted on):
  Snipper T=4 snippet, 600x800, ResNet-50 -> 3 levels -> hidden 384, 8 heads, enc6/dec6, L=3,
  P=4, 60 queries x 15 keypoints, inference, batch 1 per GPU, random-init weights, synthetic
  frames.  A "step" is one snippet through the whole network; the hot path is the 12
  MSDeformAttn layers (fused snippet kernels, one launch per layer).  Backbone and Linear layers
  are stock cuDNN/cuBLAS (out of scope per north_star) in torch's default fp32 settings.

Output: ONE JSON line (rank 0).  `value` = snippets/s with inputs resident in HBM; `e2e` = same
through the public call (snipper_b200.GraphRunner) with pinned-host inputs (H2D + D2H inside the timed
region); `roofline` = the dominant kernel (fused encoder-layer forward gather) timed with CUDA events on
its stream, `roofline.kernels` = every kernel of the hot path the same way; `gpu_baseline` = the
UNMODIFIED reference network (baseline/_ref) running its own per-(t1,t2) loop and its own vendored CUDA op
recompiled for sm_100a (oracle/_ref) on the same GPU; `train` = BASELINE config 4 (forward + backward + clip
+ AdamW, batch 2 per GPU, DDP gradient all-reduce over NCCL when launched on N > 1 ranks); `cpu_baseline` =
the reference's PyTorch/grid_sample formulation (oracle port) on the host cores for a bounded sample.
--impl reference prints the CPU arm as its own line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "snippets_per_sec_T4_600x800"
UNIT = "snippets/s"
WORKLOAD = "snipper_T4_enc6_dec6_h384_M8_L3_P4_infer_b1_600x800"
H, W, T = 600, 800, 4
N_INPUTS = 4  # distinct synthetic snippets rotated through the steps


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_snippets(n, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(1, 3 * T, H, W, generator=g) for _ in range(n)]  # frames are /255 floats in [0,1]


HEADS = ("pred_logits", "pred_kpts2d", "pred_depth")


def pack_result(out):
    """The step's result a caller reads back: final-layer predictions."""
    return torch.cat([out[k].flatten() for k in HEADS])


def dump_outputs(out_dir, packed, head_shapes):
    """Write one step's packed predictions back out as DIR/<head>.npy (float32), one file per prediction head."""
    import numpy as np
    flat = packed.detach().cpu().float().numpy()
    sizes = [int(np.prod(s)) for s in head_shapes]
    assert flat.size == sum(sizes), (flat.size, head_shapes)
    os.makedirs(out_dir, exist_ok=True)
    for name, shape, part in zip(HEADS, head_shapes, np.split(flat, np.cumsum(sizes)[:-1])):
        np.save(os.path.join(out_dir, name + ".npy"), part.reshape(shape))


def fused_layer_gathered_bytes(dims, n_frame, e=4):
    """Bytes the fused layer kernel gathers through L1: 4 corners x D channels per sample and neighbour
    frame (reference ms_deform_attn.py:137-140: frames t1-1, t1, t1+1 clipped; all frames for future t1)."""
    N, T2, T1, S, M, D, L, Lq, P = dims
    pairs = sum(len([t for t in (t1 - 1, t1, t1 + 1) if 0 <= t < n_frame]) if t1 < n_frame else T2 for t1 in range(T1))
    return N * pairs * Lq * M * L * P * 4 * D * e


def measured_l1_gather_ceiling():
    """TB/s of 192-byte-slice gathers the L1 data pipe sustains on this GPU model (tools/micro/l1_tex_vs_ldg.cu,
    profiles/r01_run25_*): the on-chip ceiling of any one-load-per-corner formulation."""
    try:
        with open(os.path.join(ROOT, "profiles", "r01_run25_micro_l1_gather_ceiling_ldg_vs_tex.jsonl")) as f:
            return max(json.loads(line)["ldg_TBps"] for line in f if line.strip())
    except Exception:
        return None


def fused_layer_bytes(dims, e=4):
    """Algorithmic bytes of one fused layer launch (SURVEY.md 8d, fused-snippet accounting):
    value read once, offsets(2)+logits(1) once per sample, output once."""
    N, T2, T1, S, M, D, L, Lq, P = dims
    samples = N * T1 * Lq * M * L * P
    value = min(N * T2 * S * M * D, 4 * samples * D * 3)
    return e * (value + N * T1 * Lq * M * D) + 4 * 3 * samples  # offsets / logits are fp32 in every mode


# ------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, budget_s=150.0):
    """The reference's CPU path for this workload: the same network with the attention computed
    by the PyTorch grid_sample formulation (oracle/torch_ref.py restates
    ms_deform_attn_core_pytorch + the per-frame module loop).  One step = one full snippet."""
    from oracle import torch_ref
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(42)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = build_snipper(torch_ref.SnippetMSDeformAttnRef).eval()
    xs = synthetic_snippets(2, seed=1)
    times = []
    t_begin = time.perf_counter()
    with torch.no_grad():
        n_warm = min(warmup, 1)
        for i in range(n_warm + steps):
            t0 = time.perf_counter()
            out, _ = model(xs[i % len(xs)])
            pack_result(out)
            dt = time.perf_counter() - t0
            if i >= n_warm:
                times.append(dt)
            if times and (time.perf_counter() - t_begin) + dt > budget_s:
                break
    return times, cores


def run_reference_arm(args, rank):
    if rank != 0:
        return
    times, cores = cpu_reference_run(args.steps, args.warmup)
    ms = 1e3 * sum(times) / len(times)
    v = 1e3 / ms
    sample = "%d full snippet forward(s), batch 1, whole network, MSDA via grid_sample" % len(times)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": min(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "device": "cpu", "threads": cores},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------------
def kernel_table(per_kernel, steps, bf16):
    """tag -> launches / avg us / algorithmic bytes / GB/s for every kernel of the hot path (SURVEY.md 8d)."""
    e = 2 if bf16 else 4
    rows = []
    for (tag, dims), ms in sorted(per_kernel.items(), key=lambda kv: -sum(kv[1])):
        avg = sum(ms) / len(ms)
        nbytes = None
        if tag.startswith("snippet_forward"):
            nbytes = fused_layer_bytes(dims, e)
        elif tag.startswith("snippet_backward"):
            N, T2, T1, S, M, D, L, Lq, P = dims
            samples = N * T1 * Lq * M * L * P
            v = min(N * T2 * S * M * D, 4 * samples * D * 3)
            nbytes = e * (v + N * T1 * Lq * M * D) + 4 * (v + 6 * samples)
        elif tag in ("frame_sum_planar", "frame_unsum_planar"):   # T2 frames on one side, planar slots (4/3 the bytes) on the other
            N, T2, T1, S, C = dims
            nbytes = e * N * S * C * T2 + 4 * N * S * (C + C // 3) * (min(T1, T2) + (1 if T1 > T2 else 0))
        elif tag == "frame_sum":          # reads T2 frames, writes one slot per query frame
            N, T2, T1, S, C = dims
            nbytes = e * N * S * C * (T2 + min(T1, T2) + (1 if T1 > T2 else 0))
        elif tag == "frame_unsum":
            N, T2, T1, S, C = dims
            nbytes = N * S * C * (4 * (min(T1, T2) + (1 if T1 > T2 else 0)) + e * T2)
        elif tag == "layer_tail":          # reads y + residual (+ pos), writes out (+ out + pos); fp32
            n_rows, C, with_pos = dims
            nbytes = 4 * n_rows * C * (3 + 2 * with_pos)
        rows.append({"kernel": tag, "dims": "x".join(map(str, dims)), "launches_per_step": len(ms) / steps,
                     "avg_us": round(avg * 1e3, 2), "ms_per_step": round(sum(ms) / steps, 4),
                     "algorithmic_MB": None if nbytes is None else round(nbytes / 1e6, 2),
                     "GBps": None if nbytes is None else round(nbytes / (avg * 1e-3) / 1e9, 1)})
    return rows


def source_fingerprint():
    """Hash of the kernel sources: profiles/roofline_traffic.json is only quoted while it matches."""
    import hashlib
    h = hashlib.sha256()
    for f in ("msda_snippet.cu", "msda_snippet_common.cuh", "msda_planar.cu", "msda_fast.cuh", "msda_common.cuh", "msda_frames.cu"):
        with open(os.path.join(ROOT, "snipper_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


EXTRA_WARMUP = 120   # untimed replays before the timed regions, in addition to --warmup (see main)


def recorded_traffic(key):
    """dram__bytes of one launch of the dominant kernel from the committed ncu capture -- null (with the reason)
    when the kernel sources changed since the capture, instead of silently quoting a stale number."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            rec = json.load(f)
    except Exception:
        return None, "no profiles/roofline_traffic.json"
    if rec.get("source_fingerprint") != source_fingerprint():
        return None, "kernel sources changed since the ncu capture (%s)" % rec.get("captured_in", "?")
    return rec.get(key), rec.get("captured_in")


def gpu_baseline_run(dev, steps=8, warmup=10):   # warm-up long enough to reach the same steady state as the product arm
    """The reference's own GPU path on this box: the UNMODIFIED reference network (baseline/_ref, staged by
    baseline/stage_reference.py) with --use_pytorch_deform 0, i.e. its per-(t1,t2) Python loop
    (models/ops/modules/ms_deform_attn.py:130-225) calling its own vendored CUDA op, compiled in place for
    sm_100a (oracle/_ref).  Eager: the reference synchronises the stream in every attention call (:112), so it
    cannot be graph-captured.  None of this package's kernels run here."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "models", "ops", "modules")):
        return {"unavailable": "baseline/_ref not staged (run __graft_entry__.build() where /root/reference exists)"}
    from oracle.build_ref import load_ref
    vendored = load_ref()
    if vendored is None:
        return {"unavailable": "oracle/_ref/MultiScaleDeformableAttention.so not built"}
    import torchvision
    real_version = torchvision.__version__
    torchvision.__version__ = "0.9.0"            # reference util/misc.py:20-22 mis-parses "0.26"
    sys.path.insert(0, ref_dir)
    try:
        import models.backbone as bb
        bb.is_main_process = lambda: False       # random init, no download (models/backbone.py:105-107)
        import main as refmain
        import models.ops.functions.ms_deform_attn_func as ref_func
        ref_func.MSDA = vendored
        args = refmain.get_args_parser().parse_args([])
        args.device, args.hidden_dim, args.num_frames, args.num_future_frames = "cuda", 384, T, 0
        args.enc_layers = args.dec_layers = 6
        args.use_pytorch_deform = 0
        from models.model import build_model
        torch.manual_seed(42)
        model = build_model(args)[0].to(dev).eval()
        xs = [x.to(dev) for x in synthetic_snippets(2, seed=77)]
        with torch.no_grad():
            for i in range(warmup):
                model(xs[i % 2])
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(steps):
                out, _ = model(xs[i % 2])
                pack_result(out)
            e.record()
            torch.cuda.synchronize()
        ms = s.elapsed_time(e) / steps
        return {"value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "steps": steps,
                "what": "unmodified reference network (baseline/_ref), use_pytorch_deform=0: its own per-(t1,t2) loop + its "
                        "vendored CUDA op recompiled for sm_100a (oracle/_ref), eager, same GPU, same synthetic inputs shape"}
    except Exception as ex:  # a baseline must never take the product's line down
        return {"unavailable": "reference GPU path failed: %r" % (ex,)}
    finally:
        torchvision.__version__ = real_version
        if ref_dir in sys.path:
            sys.path.remove(ref_dir)
        for name in [n for n in sys.modules if n == "main" or n.split(".")[0] in ("models", "util", "datasets", "engine",
                                                                                 "eval_utils", "dataset_class")]:
            mod = sys.modules.get(name)
            if getattr(mod, "__file__", None) and ref_dir in str(mod.__file__):
                del sys.modules[name]


def synthetic_loss(out):
    """Dense loss over every prediction head (the Hungarian criterion is CPU scipy code outside the hot path)."""
    loss = out["pred_kpts2d"].square().mean() + out["pred_depth"].square().mean() + out["pred_logits"].square().mean()
    for h in out["heatmaps"]:
        loss = loss + h.square().mean()
    for aux in out.get("aux_outputs", []):
        loss = loss + aux["pred_kpts2d"].square().mean() + aux["pred_depth"].square().mean() + aux["pred_logits"].square().mean()
    return loss


def train_run(dev, rank, world, local_rank, steps=8, warmup=3, batch=2):
    """BASELINE config 4: Snipper T=4 training step, batch 2 per GPU, as the reference's train_one_epoch
    (engine.py:36-79: forward, loss, backward, clip_grad_norm_(0.1), AdamW.step); stock DDP when world > 1
    (main.py:184).  Returns the per-rank dict (rank 0 prints it)."""
    import torch.distributed as dist
    import snipper_b200
    from snipper_b200 import ops, sharding
    from snipper_b200.harness.snipper_net import build_snipper
    torch.manual_seed(42)
    model = build_snipper(snipper_b200.MSDeformAttn).to(dev).train()
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank]) if world > 1 else model
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)   # reference main.py:206-207
    g = torch.Generator().manual_seed(2000 + rank)
    xs = [torch.rand(batch, 3 * T, H, W, generator=g).to(dev) for _ in range(2)]

    def step(i, sync=True):
        import contextlib
        ctx = net.no_sync() if (world > 1 and not sync) else contextlib.nullcontext()
        with ctx:
            out, _ = net(xs[i % 2])
            loss = synthetic_loss(out)
            opt.zero_grad(set_to_none=True)
            loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 0.1)                # reference engine.py:75
        opt.step()
        return loss

    def timed(n, sync=True):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n):
            step(i, sync)
        e.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        return sharding.max_over_ranks(s.elapsed_time(e), dev) / n

    for i in range(warmup):
        step(i)
    ms = timed(steps)
    res = {"metric": "train_snippets_per_sec_T4_600x800", "value": world * batch / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms, "steps": steps, "batch_per_gpu": batch, "dtype": "f32",
           "parallelism": ("DDP x%d, NCCL gradient all-reduce" % world) if world > 1 else "single GPU",
           "loss": "synthetic dense loss over all heads; fwd + bwd + clip_grad_norm_(0.1) + AdamW"}
    if world > 1:
        # what the collective costs: the same step without gradient sync, and the all-reduce on its own
        ms_nosync = timed(max(steps // 2, 2), sync=False)
        n_grad = sum(p.numel() for p in params)
        buf = torch.empty(n_grad, device=dev)
        for _ in range(2):
            dist.all_reduce(buf)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(5):
            dist.all_reduce(buf)
        e.record()
        torch.cuda.synchronize()
        ar_ms = sharding.max_over_ranks(s.elapsed_time(e), dev) / 5
        res.update({"ms_per_step_without_gradient_sync": ms_nosync, "allreduce_exposed_ms": ms - ms_nosync,
                    "allreduce_alone_ms": ar_ms, "allreduce_MB": n_grad * 4 / 1e6,
                    "allreduce_busbw_GBps": 2 * (world - 1) / world * n_grad * 4 / (ar_ms * 1e-3) / 1e9})
    ops.STATS.reset()
    ops.STATS.timing = True
    for i in range(2):
        step(i)
    torch.cuda.synchronize()
    ops.STATS.timing = False
    per = ops.STATS.kernel_ms()
    msda_ms = sum(sum(v) for v in per.values()) / 2
    res.update({"msda_ms_per_step": msda_ms, "msda_share": msda_ms / ms, "msda_kernels": kernel_table(per, 2, False)})
    del net, model, opt
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline loops (resident and end to end) and of the per-kernel event loop; "
                         "the train and gpu_baseline entries always time 8 steps of their own")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-fused-tails", action="store_true", help="keep the stock layer tails (A/B of SURVEY 8f rank 3)")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32", "bf16"],
                    help="NOT the headline: 'tf32' lets cuBLAS use TF32 tensor cores for the stock Linear layers, "
                         "'bf16' runs the network under torch.autocast(bfloat16) (bf16 GEMMs, bf16 MSDA gathers). "
                         "The default and the headline number is fp32.")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the predictions of the last timed step as DIR/<head>.npy (float32; "
                         "rank 0); inputs and weights are seeded, so two builds can be compared output for output. "
                         "--impl ours only: the CPU reference arm runs other inputs, so its outputs are not comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import snipper_b200
    from snipper_b200 import ops, sharding
    from snipper_b200.harness.snipper_net import build_snipper

    args.warmup = max(args.warmup, 3)
    if args.precision == "tf32":
        torch.backends.cuda.matmul.allow_tf32 = True
    bf16 = args.precision == "bf16"
    import contextlib
    autocast = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if bf16 else contextlib.nullcontext
    torch.manual_seed(42)  # reference main.py:48
    model = build_snipper(snipper_b200.MSDeformAttn).to(dev).eval()
    # the package's opt-in layer tails (bias + residual + LayerNorm (+ pos) in one pass) and in-kernel encoder reference points
    fused_tails = 0 if args.no_fused_tails else snipper_b200.enable_fused_layer_tails(model)
    # snippet sharding: every rank takes its own contiguous slice of the job's snippets (no data-path collective)
    lo, hi = sharding.shard_range(N_INPUTS * world, rank, world)
    host = [x.pin_memory() for x in synthetic_snippets(hi - lo, seed=1000 + rank)]
    resident = [x.to(dev) for x in host]
    h2d_bytes = host[0].numel() * host[0].element_size()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the public call: a graphed runner over "snippet in -> packed predictions out" ----
    def forward_packed(x):
        out, _ = model(x)
        return pack_result(out).float()

    with torch.no_grad(), autocast():
        first, _ = model(resident[0])
        result = pack_result(first).float()
    head_shapes = [tuple(first[k].shape) for k in HEADS]
    del first
    d2h_bytes = result.numel() * result.element_size()
    host_out = torch.empty(result.shape, dtype=result.dtype).pin_memory()
    runner, launches_per_step = None, None
    if not args.no_graph:
        try:
            runner = snipper_b200.GraphRunner(forward_packed, warmup=2, autocast_dtype=torch.bfloat16 if bf16 else None)
            launches_per_step = runner.launches_per_replay(resident[0])
        except Exception as e:  # fall back to eager timing, say so in config
            print("[bench] CUDA graph capture failed (%r); timing eager launches" % (e,), file=sys.stderr)
            runner = None
            torch.cuda.synchronize()

    def call(x):
        if runner is not None:
            return runner(x)
        with torch.no_grad(), autocast():
            return forward_packed(x.to(dev, non_blocking=True))

    def step_resident(i):
        return call(resident[i % len(resident)])

    def step_e2e(i):
        out = call(host[i % len(host)])
        if runner is not None:   # the NEXT snippet's host-to-device copy rides a side stream under this step's compute
            runner.prefetch(host[(i + 1) % len(host)])
        host_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the result every step
        return host_out

    def timed(step_fn, steps, warmup):
        for i in range(warmup):
            step_fn(i)
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            step_fn(warmup + i)
        e.record()
        barrier()
        return sharding.max_over_ranks(s.elapsed_time(e), dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    # steady state: on a fresh box the first seconds of replays run ~2 % slower whatever the issue pattern
    # (profiles/r02_run22_replay_modes_probe.json, r02_run23_*), so the resident loop gets extra untimed replays on top
    # of --warmup: a fixed 120 (about 3 s), after which consecutive blocks of replays agree
    extra_warmup = EXTRA_WARMUP
    for i in range(extra_warmup):
        step_resident(i)
    ops.STATS.reset()
    ms_total = timed(step_resident, args.steps, args.warmup)
    eager_launches = ops.STATS.launches
    ms_e2e_total = timed(step_e2e, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # host_out holds the last timed step's result; both timed loops feed step warmup + steps - 1 the same input
        dump_outputs(args.dump_outputs, host_out, head_shapes)
    if launches_per_step is None:
        launches_per_step = eager_launches // (args.steps + args.warmup)

    # ---- roofline: events around every launch of the hot path, eager steps after the timed region ----
    ops.STATS.reset()
    ops.STATS.timing = True
    with torch.no_grad(), autocast():
        for i in range(args.steps):
            model(resident[i % len(resident)])
    torch.cuda.synchronize()
    ops.STATS.timing = False
    per_kernel = ops.STATS.kernel_ms()
    (dom_tag, dom_dims), dom_ms = max(((k, v) for k, v in per_kernel.items() if k[0].startswith("snippet_forward")),
                                      key=lambda kv: sum(kv[1]))
    dom_avg_ms = sum(dom_ms) / len(dom_ms)
    msda_ms_per_step = sum(sum(v) for v in per_kernel.values()) / args.steps
    peak, peak_src = measured_peak()
    e_bytes = 2 if bf16 else 4
    alg_bytes = fused_layer_bytes(dom_dims, e=e_bytes)
    achieved = alg_bytes / (dom_avg_ms * 1e-3) / 1e9
    planar = dom_tag.endswith("planar")
    presummed = dom_tag.endswith("presummed") or planar
    # bytes that cross the L1 data pipe: 4 corners x D channels per sample and GATHERED frame (one per query frame
    # when the neighbour frames are pre-summed, |nb(t1)| otherwise)
    N_, T2_, T1_, S_, M_, D_, L_, Lq_, P_ = dom_dims
    gathered = (N_ * T1_ * Lq_ * M_ * L_ * P_ * 4 * D_ * e_bytes) if presummed else \
        fused_layer_gathered_bytes(dom_dims, model.num_frames, e_bytes)
    ceiling = measured_l1_gather_ceiling()
    on_chip = {"what": "bytes gathered through L1 per launch / launch time, against the measured L1 gather ceiling for 192-byte "
                       "slices (tools/micro/l1_tex_vs_ldg.cu): the on-chip resource this gather runs against",
               "gathered_bytes_per_launch": gathered, "achieved_TBps": gathered / (dom_avg_ms * 1e-3) / 1e12,
               "measured_ceiling_TBps": ceiling,
               "frac": (gathered / (dom_avg_ms * 1e-3) / 1e12 / ceiling) if ceiling else None}
    traffic, traffic_src = recorded_traffic("snippet_forward_planar_encoder_dram_bytes_per_launch" if planar else
                                            "snippet_forward_presummed_encoder_dram_bytes_per_launch" if presummed
                                            else "snippet_forward_encoder_dram_bytes_per_launch")

    graphed = runner is not None
    train = None
    if not args.no_train and args.precision == "fp32":
        runner = None
        torch.cuda.empty_cache()
        train = train_run(dev, rank, world, local_rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = ms_total / args.steps
    value = world * args.steps / (ms_total * 1e-3)
    e2e_value = world * args.steps / (ms_e2e_total * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {"fp32": "f32", "tf32": "tf32-matmul (informational)", "bf16": "bf16-autocast (informational)"}[args.precision],
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "snippets_per_gpu_per_step": 1, "parallelism": "snippet-sharded x%d, no collective" % world,
                   "launch": "cuda_graph_replay (snipper_b200.GraphRunner; e2e: the next input's H2D copy is prefetched on a "
                             "side stream, every step still copies its own 23 MB in and its result out)" if graphed else "eager",
                   "l2": "working set per step (171 MB weights + >1 GB activations) exceeds the 126 MB L2; %d distinct inputs rotated" % len(resident),
                   "weights": "random init (seed 42): sampling offsets are the fixed per-head grid, best-case gather locality",
                   "precision_note": "fp32 = torch defaults: fp32 SIMT GEMMs for the Linear layers, cuDNN convolutions may use TF32 "
                                     "(torch.backends.cudnn.allow_tf32 default); the CPU arm is strict fp32",
                   "fused_layer_tails": "%d layers (snipper_b200.enable_fused_layer_tails)" % fused_tails,
                   "extra_untimed_warmup_steps": extra_warmup,
                   "msda_ms_per_step_eager_events": msda_ms_per_step},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_e2e_total / args.steps},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "%s (%s %s)" % (
                         "msda_planar_fwd_kernel<32>" if planar else
                         "msda_snippet_fwd_kernel<float,12,16,1536,%s>" % ("presummed" if presummed else "direct"),
                         dom_tag, "x".join(map(str, dom_dims))),
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "avg_launch_ms": dom_avg_ms, "launches_timed": len(dom_ms),
                     "how": "CUDA events on the launching stream around each launch, eager steps after the timed region",
                     "on_chip": on_chip, "kernels": kernel_table(per_kernel, args.steps, bf16)},
    }
    if train is not None:
        line["train"] = train
        # the backward's own roofline entry (BASELINE metric: "MSDeformAttn fwd/bwd HBM GB/s"): the fused encoder
        # backward as timed inside the training step (batch 2), same accounting as `roofline`
        bwd = next((k for k in train.get("msda_kernels", []) if k["kernel"].startswith("snippet_backward") and
                    k["algorithmic_MB"] and "x9875x4" in k["dims"] and k["dims"].split("x")[7] == "9875"), None)
        if bwd is not None:
            btraffic, bsrc = recorded_traffic("snippet_backward_presummed_encoder_dram_bytes_per_launch")
            n_batch = int(bwd["dims"].split("x")[0])
            line["roofline_backward"] = {
                "bound": "hbm", "kernel": "msda_snippet_bwd_kernel<float,12,16,1536,presummed> (%s %s)" % (bwd["kernel"], bwd["dims"]),
                "achieved": bwd["GBps"], "peak": peak, "unit": "GB/s", "frac": bwd["GBps"] / peak,
                "traffic": None if btraffic is None else btraffic * n_batch,
                "traffic_source": "%s, captured at batch 1 and scaled by the batch" % bsrc,
                "algorithmic_bytes_per_launch": int(bwd["algorithmic_MB"] * 1e6), "avg_launch_ms": bwd["avg_us"] / 1e3,
                "how": "CUDA events around each launch in two training steps after the timed region",
                "limiter": "SM->L2 request path (vector reductions), see DESIGN.md section 3"}
    if world == 1 and not args.no_gpu_baseline:
        line["gpu_baseline"] = gpu_baseline_run(dev)
    if world == 1 and not args.no_cpu_baseline:
        times, cores = cpu_reference_run(1, 0)
        v = len(times) / sum(times)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "%d full snippet forward, batch 1, whole network on host cores, MSDA via grid_sample (oracle port of the reference's PyTorch path)" % len(times)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

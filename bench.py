#!/usr/bin/env python
"""bench.py -- views/sec of the IGGT multi-view forward on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]

Workload (config C2 of BASELINE.json): one synthetic scene of 8 views at 518x518, random-init weights of the
reference architecture, fp16 trunk operands (fp32 accumulate / residual / LayerNorm), every output the
reference can produce at this (odd, 37x37) patch grid: pose_enc, depth(+conf), world_points(+conf).
`part_feat` needs an even patch grid in the reference (SURVEY F2) and is reported by `--size 532`.

N>1 (launched by torchrun, one rank per GPU): the views of every scene are sharded over the ranks (strong scaling)
with one all-gather of K|V per global block.  `--scenes B --views S` select the other BASELINE configs:
C3 = `--views 32` on 8 GPUs (4 views per GPU), C5 = `--scenes 4 --views 16 --dtype bf16` on 8 GPUs (each GPU holds
2 views of all 4 scenes), C4 = `--size 1036 --part`.

A step = one forward over the batch.  `value` is timed with inputs resident in HBM; `e2e` includes the
pinned-host -> device copy of the images and the device -> host copy of every prediction, each step.
`--impl reference` times the reference algorithm's CPU implementation (the oracle port, all host threads) on a
bounded sample of the same workload: `--ref-views` (default 1) of the views per step at the same resolution - its
`config` says so (`views_per_step`), its global attention spans that many views only.

`--dump-outputs DIR` writes the predictions of the last timed step as DIR/<name>.npy (see `dump_outputs`).  Weights
and images are seeded, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "views/sec (518^2, V=8)"
TENSOR_OPS = ("iggt_gemm_store16", "iggt_gemm_store32", "iggt_gemm_resid32", "iggt_gemm_qkv", "iggt_conv_nhwc",
              "iggt_attention_fwd")
DUMP_BYTES = 64 * 10 ** 6


# ------------------------------------------------------------------------------------------- helpers
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "gbs": d.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (sustained cuBLAS bf16 / stream copy)"}
    return {"tflops": 1400.0, "gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_outputs(out, path):
    """Writes the prediction dict `out` as `path`/<name>.npy in float32: every key a caller receives except `images`
    (the caller's own input handed back); `pose_enc`, one [B, S, 9] tensor per camera-head iteration, is stacked to
    [iters, B, S, 9].  If the arrays exceed DUMP_BYTES in all, each one is written as the same fraction of its
    elements: a 1-D array of the values at sorted flat positions drawn with a fixed seed, the same for every run."""
    arrays = {k: (torch.stack(v) if isinstance(v, list) else v).detach().float().cpu()
              for k, v in out.items() if k != "images"}
    total = sum(a.numel() * 4 for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in sorted(arrays.items()):
        if total > DUMP_BYTES:
            keep = a.numel() * DUMP_BYTES // total
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.numpy())
    print(f"[bench] {len(arrays)} outputs of the last timed step -> {path}"
          f"{f' (a sample of {total} bytes)' if total > DUMP_BYTES else ''}", file=sys.stderr)


def dist_setup(n_gpus):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


# ------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """CPU implementation of the reference algorithm (oracle port, fp32, all host threads)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_model, weights  # the one place bench.py executes oracle/: as the CPU baseline
    cores = cpu_threads()
    torch.set_num_threads(cores)
    S = args.ref_views
    sd = weights.make_state_dict(0, "default", prefixes=("aggregator.", "camera_head.", "depth_head.", "point_head."))
    g = torch.Generator().manual_seed(0)
    images = torch.rand(1, S, 3, args.size, args.size, generator=g)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        out = ref_model.forward(sd, images, model="vggt", skip_part=True, frames_chunk=2)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    ms = 1e3 * sum(times) / len(times)
    v = S / (ms / 1e3)
    sample = (f"{S} of {args.views} views at {args.size}x{args.size} per step, fp32, same heads "
              f"(global attention over {S} views), {cores} threads")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "views/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, 1), views_per_step=S, sample=sample,
                           parallelism=f"host CPU, {cores} threads"),
            "cpu_baseline": {"value": v, "unit": "views/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def config_name(args):
    key = (args.scenes, args.views, args.size)
    return {(1, 8, 518): "C2", (1, 32, 518): "C3", (1, 8, 1036): "C4", (4, 16, 518): "C5"}.get(key, "custom")


def workload_config(args, world):
    return {"workload": f"{config_name(args)}: {args.scenes} scene{'s' if args.scenes > 1 else ''} x {args.views} views, "
                        f"{args.size}x{args.size}, full forward "
                        f"(pose_enc, depth+conf, world_points+conf{', part_feat' if args.part else ''})",
            "scenes": args.scenes, "views": args.views, "image": [args.size, args.size],
            "weights": "random-init, reference architecture (1.30 B params)",
            "parallelism": f"view-shard x{world}" if world > 1 else "single GPU",
            "l2": "per-step working set (2.6 GB 16-bit weights + activations) >> 126 MB L2: no flush needed"}


# ------------------------------------------------------------------------------------------- our arm
def run_b200(args):
    import torch.distributed as dist
    rank, world, local = dist_setup(args.gpus)
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one process: run it with --gpus 1")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from iggt_official_b200 import ops
    from iggt_official_b200.models.vggt import IGGT, VGGT
    from iggt_official_b200.parallel import forward_sharded
    dt = {"fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    torch.manual_seed(0)
    model = (IGGT if args.part else VGGT)().eval().to(dev)
    model.compute_dtype = dt
    assert args.views % world == 0, "views must divide over the ranks"
    S_loc = args.views // world
    g = torch.Generator().manual_seed(0)
    images_host = torch.rand(args.scenes, args.views, 3, args.size, args.size, generator=g)[:, rank * S_loc:(rank + 1) * S_loc]
    images_host = images_host.contiguous().pin_memory()
    images_dev = images_host.to(dev)

    def eager_step(imgs):
        if world > 1:
            return forward_sharded(model, imgs, rank, world)
        return model(imgs)

    step = eager_step
    graphed = False
    if not args.no_graph and not args.quick:
        from iggt_official_b200.graphs import GraphedForward
        try:
            g_step = GraphedForward(eager_step, model=model)
            g_step(images_dev)                     # capture now; fall back to eager launches if it fails
            torch.cuda.synchronize()
            step, graphed = g_step, True
        except Exception as e:                     # pragma: no cover
            print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); running eager", file=sys.stderr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup if args.quick else max(args.warmup, 3)):
        out = step(images_dev)
    barrier()
    if args.quick:
        for _ in range(args.steps):
            out = step(images_dev)
        barrier()
        if args.dump_outputs:
            dump_outputs(out, args.dump_outputs)
        if rank == 0:
            print(json.dumps({"quick": True, "launches_per_step": ops.STATS["launches"] // (args.warmup + args.steps)}))
        _finish(world)
        return

    # ---- device-resident timing (value)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ops.STATS["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = step(images_dev)
    e1.record()
    barrier()
    if args.dump_outputs:                          # before later replays overwrite the graph's output buffers
        dump_outputs(out, args.dump_outputs)
    ms = e0.elapsed_time(e1) / args.steps
    launches = (ops.STATS["launches"] - launches0) // args.steps
    if graphed:                                    # replays bypass the Python counter: count one eager forward
        c0 = ops.STATS["launches"]
        eager_step(images_dev)
        torch.cuda.synchronize()
        launches = ops.STATS["launches"] - c0
    clocks = sampler.stop() if rank == 0 else None

    # ---- end-to-end through the public API: H2D of the images + D2H of every prediction, each step
    keys = [k for k in ("depth", "depth_conf", "world_points", "world_points_conf", "part_feat") if k in out]
    host_out = {k: torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory() for k in keys}
    host_pose = torch.empty((4,) + tuple(out["pose_enc"][0].shape), dtype=torch.float32).pin_memory()

    def e2e_step():
        imgs = images_host.to(dev, non_blocking=True)
        o = step(imgs)
        for k in keys:
            host_out[k].copy_(o[k], non_blocking=True)
        host_pose.copy_(torch.stack(o["pose_enc"]), non_blocking=True)

    for _ in range(2):
        e2e_step()
    barrier()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    h2d = images_host.numel() * 4 * world
    d2h = (sum(v.numel() * 4 for v in host_out.values()) + host_pose.numel() * 4) * world

    # ---- per-kernel trace (separate steps, CUDA events on the launching stream around every launch)
    ops.TRACE = []
    for _ in range(2):
        eager_step(images_dev)
    torch.cuda.synchronize()
    trace, ops.TRACE = ops.TRACE, None
    agg = {}
    for name, fl, nb, a, b, _dims in trace:
        d = agg.setdefault(name, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
        d["ms"] += a.elapsed_time(b); d["flops"] += fl; d["bytes"] += nb; d["n"] += 1
    total_ms = sum(d["ms"] for d in agg.values())
    peaks = measured_peaks()
    top = max(agg.items(), key=lambda kv: kv[1]["ms"])
    name, d = top
    if name in TENSOR_OPS:
        ach = d["flops"] / (d["ms"] * 1e-3) / 1e12
        roof = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": ach / peaks["tflops"], "traffic": None}
    else:
        ach = d["bytes"] / (d["ms"] * 1e-3) / 1e9
        roof = {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peaks["gbs"], "unit": "GB/s",
                "frac": ach / peaks["gbs"], "traffic": None}
    roof.update({"launches_per_step": d["n"] // 2, "avg_launch_ms": d["ms"] / d["n"], "share_of_step": d["ms"] / total_ms,
                 "peak_source": peaks["source"]})
    if name == "iggt_attention_fwd":
        # head_dim 64 attention is bounded by the exp unit (MUFU: 16 ex2/clk/SM measured, scripts/ubench/mufu.cu) before
        # the tensor pipe: 1 exp per 256 tensor FLOPs -> at most 0.5 of the tensor peak.  Report that roofline too.
        clk = (clocks or {}).get("sm_mhz") or 1965.0
        exps = d["flops"] / 256.0
        peak_exp = 16.0 * 148 * clk * 1e6
        roof["mufu_roofline"] = {"achieved_gexp_s": exps / (d["ms"] * 1e-3) / 1e9, "peak_gexp_s": peak_exp / 1e9,
                                 "frac": exps / (d["ms"] * 1e-3) / peak_exp,
                                 "note": "ncu (profiles/r02a_ncu_all_kernels.csv): sm__inst_executed_pipe_xu 75.7 % (global), 55.1 % (frame) of peak; the softmax warps are latency-bound, not MUFU-bound (profiles/r02b_attn_sweep.json)"}
        tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tp) and world == 1 and args.views == 8 and args.size == 518:
            t = json.load(open(tp))["iggt_attention_fwd"]
            # per launch, averaged over the 24 global + 48 frame launches of a step
            roof["traffic"] = (24 * t["global_c2_bytes_per_launch"] + 48 * t["frame_c2_bytes_per_launch"]) / 72
            roof["traffic_unit"] = "bytes per launch (dram read+write, ncu --set full)"
            roof["algorithmic_bytes_per_launch"] = d["bytes"] / d["n"]
    shares = {k: {"share": v["ms"] / total_ms, "ms_per_step": v["ms"] / 2, "n_per_step": v["n"] // 2,
                  "tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["flops"] else None,
                  "gbs": v["bytes"] / (v["ms"] * 1e-3) / 1e9}
              for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- max over ranks
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    if rank != 0:
        _finish(world)
        return
    n_views = args.scenes * args.views
    value = n_views / (ms * 1e-3)
    line = {"metric": METRIC if config_name(args) == "C2" else f"views/sec ({config_name(args)})", "value": value, "unit": "views/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": workload_config(args, world),
            "clocks": clocks, "gpu_launches": launches, "cuda_graph": graphed,
            "e2e": {"value": n_views / (ms_e2e * 1e-3), "unit": "views/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "roofline": roof, "kernel_shares": shares,
            "algorithmic_tflop_per_step": trunk_tflop(args)}
    line["model_flop_utilisation"] = {"achieved_tflops": line["algorithmic_tflop_per_step"] / (ms * 1e-3) / world,
                                      "peak_tflops": peaks["tflops"], "frac": line["algorithmic_tflop_per_step"] / (ms * 1e-3) / world / peaks["tflops"]}
    if world == 1 and not args.no_cpu_baseline:
        if not args.part:
            line["gpu_eager_baseline"] = gpu_eager_baseline(args, dt, images_dev)
        line["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(line))
    _finish(world)


def _finish(world):
    """Multi-rank teardown.  destroy_process_group() can hang while captured CUDA graphs still reference the
    NCCL communicator (observed on 2 GPUs: ranks idle until killed), so after a final barrier the ranks flush and
    leave with os._exit(0) -- everything measured has already been printed."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    try:
        torch.cuda.synchronize()
        dist.barrier()
    finally:
        os._exit(0)


def trunk_tflop(args):
    """BASELINE.md section 3: trunk 2.4896 + 0.3712 + 0.18558*S TFLOP/view at T=1374 (scaled by T), heads 0.2985 x2."""
    g = args.size // 14
    T = 5 + g * g
    S = args.views
    lin = T * 1.8119e-3
    frame = 48 * 4 * T * T * 1024 / 1e12
    glob = 24 * 4 * T * (S * T) * 1024 / 1e12
    heads = 2 * 0.2180e-3 * g * g
    return args.scenes * S * (lin + frame + glob + heads)


def cpu_threads():
    """PyTorch's CPU kernels stop scaling (and collapse from oversubscription: 246 s for the 2-view sample with
    128 threads on the 128-core bench host, 14 s with 8 threads on an 8-core box) well before 128 threads; the CPU
    legs use at most 32 and report that number as `cores`."""
    return max(1, min(os.cpu_count() or 1, 32))


def gpu_eager_baseline(args, dt, images_dev):
    """SURVEY 8(d)'s "real bar": the reference algorithm as PyTorch eager on THIS B200 - the oracle port with its
    Linear / SDPA calls issued natively in the autocast dtype (ref_model.NATIVE_16BIT: cuBLAS 16-bit GEMMs, the
    SDPA backend torch picks; heads fp32 with cuDNN TF32 convolutions, PyTorch's default), same inputs and config."""
    from oracle import ref_model, weights  # checker used as a baseline (never on the product path)
    sd = weights.make_state_dict(0, "default", prefixes=("aggregator.", "camera_head.", "depth_head.", "point_head."))
    sd = {k: v.to(images_dev.device) for k, v in sd.items()}
    ref_model.NATIVE_16BIT = True
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        for i in range(1 + reps):
            if i == 1:
                torch.cuda.synchronize()
                e0.record()
            ref_model.forward(sd, images_dev, model="vggt", amp=dt, skip_part=True, frames_chunk=8)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
    finally:
        ref_model.NATIVE_16BIT = False
        ref_model._W16.clear()
        torch.backends.cudnn.allow_tf32 = tf32
        del sd
        torch.cuda.empty_cache()
    n = args.scenes * args.views
    return {"value": n / (ms * 1e-3), "unit": "views/s", "ms_per_step": ms, "kind": "port",
            "what": f"oracle port as PyTorch {torch.__version__} eager on the same GPU: {args.dtype} Linear / SDPA "
                    "(cuBLAS + torch's SDPA backend), fp32 LayerNorm / residual, heads fp32 with cuDNN TF32 convolutions; "
                    f"{reps} forwards after 1 warm-up, CUDA events; device-resident inputs"}


def cpu_baseline(args):
    """Oracle port on the host cores, bounded sample: one timed forward of `--ref-views` views."""
    from oracle import ref_model, weights  # checker used as the CPU baseline (never on the product path)
    cores = cpu_threads()
    torch.set_num_threads(cores)
    S = args.ref_views
    sd = weights.make_state_dict(0, "default", prefixes=("aggregator.", "camera_head.", "depth_head.", "point_head."))
    g = torch.Generator().manual_seed(0)
    images = torch.rand(1, S, 3, args.size, args.size, generator=g)
    t0 = time.perf_counter()
    ref_model.forward(sd, images, model="vggt", skip_part=True, frames_chunk=2)
    dt = time.perf_counter() - t0
    return {"value": S / dt, "unit": "views/s", "cores": cores, "kind": "port",
            "sample": f"one fp32 forward of {S} of the {args.views} views at {args.size}x{args.size} ({dt:.1f} s), oracle port, "
                      f"{cores} threads"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--views", type=int, default=8, help="views per scene")
    ap.add_argument("--scenes", type=int, default=1, help="scenes per step (C5: 4)")
    ap.add_argument("--size", type=int, default=518)
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--part", action="store_true", help="IGGT with the part path (needs an even patch grid, e.g. --size 532)")
    ap.add_argument("--ref-views", type=int, default=1, help="views per step of the CPU legs (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--quick", action="store_true", help="profiling mode: warm-up + steps only (run this under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the B200 path)")
        run_b200(args)


if __name__ == "__main__":
    main()

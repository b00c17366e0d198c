#!/usr/bin/env python
"""Benchmark of the MERV fusion hot path (BASELINE.json metric: merv-full fusion videos/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one pass of the whole path (pool -> projector -> score/softmax -> mix) over one batch of 64 synthetic
videos PER GPU at merv-full shapes (frames [16,16,32,16] -> 16 temporal tokens each; BASELINE.json configs[1]).
Videos are independent, so ranks shard by batch with no collective on the data path ("scaling": "weak").
Rank 0 prints ONE JSON line.  `value` is device-resident throughput through the production call (one C call per step:
merv_fused_forward, three kernels chained by programmatic dependent launch); `e2e` is the same metric through the
host-buffer API (H2D of the inputs and D2H of the prefix inside the timed region).

Sub-records of the same line (each with its own clock record):
  sustained     the same step for >= 200 iterations (power-capped regime) next to the K-step burst `value`
  strong        N > 1: BASELINE.json configs[2] as written — 64 videos GLOBAL, 64 / N per rank — compute only
  gather        N > 1: the all-gather of the fused prefixes over NVLink for the strong and the weak shard size:
                compute-then-NCCL vs the GEMM whose epilogue stores every tile into all ranks' symmetric buffers
  configs       N = 1: configs[3] (SigLIP single encoder, B = 256) and configs[4] (generate: time-to-prefix, TTFT)
  kernels / roofline   per-kernel CUDA-event durations from an instrumented pass over the same K steps

--dump-outputs DIR writes what the last timed step returned (rank 0): DIR/weights.npy, the mixing weights [batch, 4], and
DIR/prefix_sample.npy, the prefix [batch, 1024, 4096] at DUMP_SAMPLE fixed, seeded flat positions (both float32).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.

--impl reference times the reference's own CPU implementation of the path (the unmodified merv/util/nn_utils.py modules
staged in oracle/_ref; oracle/torch_port.py where that file is absent) on the host cores, rank 0 only, without importing
merv_b200.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

DIMS = [1024, 1024, 768, 768]
PATCHES = [256, 256, 196, 196]
TOKENS_T = [16, 16, 16, 16]  # temporal tokens after the backbones for frames [16,16,32,16] (ViViT tubelet 2)
MUS = [0.0, 0.5, -0.5, 0.25]
LLM_DIM, OUT_TOKENS = 4096, 1024
Q_SCALE = 64.0  # non-degenerate mixing weights (SURVEY.md §7)
# SURVEY.md §8(d): algorithmic bytes / FLOPs per video (bf16)
BYTES_IN = sum(t * n * c * 2 for t, n, c in zip(TOKENS_T, PATCHES, DIMS))  # 26,411,008
BYTES_POOLED = sum(OUT_TOKENS * c * 2 for c in DIMS)  # 7,340,032
BYTES_Y = OUT_TOKENS * LLM_DIM * 2  # 8,388,608 per encoder
BYTES_OUT = OUT_TOKENS * LLM_DIM * 2
FLOPS_LINEAR = 2 * OUT_TOKENS * LLM_DIM * sum(DIMS)  # 30.065 GFLOP
FLOPS_GELU = FLOPS_LINEAR + 4 * 2 * OUT_TOKENS * LLM_DIM * LLM_DIM  # 167.5 GFLOP
GLOBAL_BATCH = 64  # BASELINE.json configs[2] / SURVEY.md §8d config 3
DUMP_SAMPLE, DUMP_SEED = 1 << 22, 0  # --dump-outputs: 16 MB of float32 out of the 1 GB (as float32) prefix of 64 videos


def ncu_traffic_bytes(*profile_txts: str):
    """dram read + write bytes per launch from the committed `ncu --set full` summary under profiles/ (first file present)."""
    for name in profile_txts:
        path = os.path.join(REPO, "profiles", name)
        if not os.path.isfile(path):
            continue
        for line in open(path):
            if line.strip().startswith("traffic (dram read + write)"):
                return float(line.split()[-2]) * 1e6
    return None


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")  # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.th.start()
            time.sleep(0.3)  # nvidia-smi start-up: make sure samples land inside the timed region
            self.lines.clear()
        except Exception:
            self.proc = None
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(power), "samples": len(sm), "reasons": sorted(reasons)}


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def make_cpu_inputs(batch: int, seed: int = 7):
    import torch

    g = torch.Generator().manual_seed(seed)
    return [torch.randn((batch, t, n, c), generator=g) + mu for t, n, c, mu in zip(TOKENS_T, PATCHES, DIMS, MUS)]


def cpu_reference_run(mlp_type: str, sample_videos: int, steps: int, warmup: int, dtype_name: str = "bf16"):
    """Times the reference's CPU implementation of the path on all host cores (oracle/reference_model.py: the unmodified reference
    modules when their file is reachable, the torch port otherwise).  No merv_b200 import, no CUDA.
    Returns (videos/s, ms/step, cores, kind, what)."""
    import torch

    from oracle import reference_model

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dtype = torch.bfloat16 if dtype_name == "bf16" else torch.float32
    fwd, kind, what = reference_model.build_cpu_arm(DIMS, LLM_DIM, TOKENS_T, 8, mlp_type, OUT_TOKENS, q_scale=Q_SCALE, dtype=dtype)
    feats = [f.to(dtype) for f in make_cpu_inputs(sample_videos)]
    for _ in range(warmup):
        fwd(feats)
    t0 = time.perf_counter()
    for _ in range(steps):
        fwd(feats)
    dt = time.perf_counter() - t0
    return sample_videos * steps / dt, dt / steps * 1e3, cores, kind, what


def dump_outputs(directory: str, out, w) -> None:
    """The arrays a caller of the timed path receives, as float32 .npy: the mixing weights whole, the prefix at DUMP_SAMPLE flat
    positions drawn from a generator seeded with DUMP_SEED (the same positions for every run of the same shape)."""
    import numpy as np
    import torch

    os.makedirs(directory, exist_ok=True)
    idx = torch.randint(0, out.numel(), (min(DUMP_SAMPLE, out.numel()),), generator=torch.Generator().manual_seed(DUMP_SEED))
    np.save(os.path.join(directory, "prefix_sample.npy"), out.reshape(-1)[idx.to(out.device)].float().cpu().numpy())
    np.save(os.path.join(directory, "weights.npy"), w.float().cpu().numpy())


def workload_config(args, world: int, note: str = ""):
    return {
        "workload": f"merv-full fusion bf16 batch {args.batch} per GPU on {world}xB200 (3d-avg pool + {args.projector} projector + cross-attn mix)",
        "encoders": ["languagebind", "dinov2", "vivit", "siglip"], "frames": [16, 16, 32, 16], "feature_shapes": [[16, 256, 1024], [16, 256, 1024], [16, 196, 768], [16, 196, 768]],
        "prefix_tokens": OUT_TOKENS, "llm_dim": LLM_DIM, "projector": args.projector, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
        "pipeline": args.mode, "parallelism": f"dp{world} (batch-sharded, no data-path collective)",
        "l2": f"inputs larger than L2: {args.input_sets} rotating input sets of {BYTES_IN * args.batch / 1e9:.2f} GB each", "note": note,
    }


def reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    sample = args.cpu_sample_videos
    value, ms, cores, kind, what = cpu_reference_run(args.projector, sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "merv-full fusion videos/sec", "value": value, "unit": "videos/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, world, note=f"reference arm: the same workload on the host CPU, each step a bounded sample of {sample} of its videos"),
        "cpu_baseline": {"value": value, "unit": "videos/s", "cores": cores, "cpu": cpu_model(), "kind": kind, "what": what,
                         "sample": f"{sample} merv-full videos per step, bf16, {args.steps} steps after {args.warmup} warm-up"},
        "e2e": {"value": value, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "fused_tokens_per_s": value * OUT_TOKENS, "gpu_launches": 0, "imports_merv_b200": "merv_b200" in sys.modules,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="videos per GPU per step (weak scaling, the default)")
    ap.add_argument("--global-batch", type=int, default=0, help="if > 0: make strong scaling the PRIMARY line, this many videos per step split over the ranks")
    ap.add_argument("--no-torch-eager", action="store_true", help="skip timing the reference's op sequence in torch eager on the same GPU")
    ap.add_argument("--projector", default="linear", choices=["linear", "gelu-mlp"])
    ap.add_argument("--mode", default="fused", choices=["fused", "unfused"])
    ap.add_argument("--input-sets", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--sustained-steps", type=int, default=300)
    ap.add_argument("--cpu-sample-videos", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="skip the all-gather sub-records (N > 1)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sub-record (N > 1)")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[3] / configs[4] sub-records (N = 1)")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--assist-ab", action="store_true",
                    help="N = 1: also A/B the opt-in pooling inside the GEMM launch (MERV_POOL_ASSIST=1) in the sustained regime; off by default so "
                         "that the default run only ever executes the production path")
    ap.add_argument("--gather-timeout", type=float, default=240.0, help="watchdog (s) around the multi-GPU gather sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/*.npy (float32; a fixed, seeded sample of the prefix)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    scaling = "weak"
    if args.global_batch > 0:
        assert args.global_batch % world == 0, "--global-batch must be a multiple of the number of ranks"
        args.batch, scaling = args.global_batch // world, "strong"
    if args.impl == "reference":
        return reference_arm(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist

    import merv_b200 as M
    from merv_b200 import ops
    from merv_b200.pipeline import HostPipeline

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: merv_b200 has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        try:  # one disjoint slice of the host cores per rank: the ranks' copy-issuing threads do not migrate onto each other
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, set(cores[local_rank * per:(local_rank + 1) * per]) or set(cores))
        except (AttributeError, OSError):
            pass

    peaks = load_peaks()
    B = args.batch

    def build_module(dims, frames, projector):
        m = M.MervFusion.build(dims, LLM_DIM, frames, 64, projector, seed=dims[0], fused=(args.mode == "fused"))
        with torch.no_grad():
            m.feature_fusion.Q.mul_(Q_SCALE)
        return m.to(device=dev, dtype=torch.bfloat16).eval().requires_grad_(False)

    module = build_module(DIMS, TOKENS_T, args.projector)

    def make_sets(batch, n_sets, seed0=7):
        sets = []
        for s in range(n_sets):
            g = torch.Generator(device=dev).manual_seed(seed0 + rank + 1000 * s)
            sets.append([(torch.randn((batch, t, n, c), generator=g, device=dev) + mu).to(torch.bfloat16)
                         for t, n, c, mu in zip(TOKENS_T, PATCHES, DIMS, MUS)])
        return sets

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(step_fn, steps: int, warmup: int = 0, clocks: bool = True):
        """`steps` calls of step_fn(i) between barrier + synchronize, CUDA events on the launching stream, max over ranks.
        Returns (ms per step, clock record of the timed region)."""
        for i in range(warmup):
            step_fn(i)
        barrier()
        sampler = ClockSampler(local_rank).start() if clocks else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            step_fn(i)
        e1.record()
        barrier()
        rec = sampler.stop() if sampler else None
        return max_over_ranks(e0.elapsed_time(e1)) / steps, rec

    sets = make_sets(B, args.input_sets)
    keep = {}

    def step(i):
        keep["out"], keep["w"] = module(sets[i % len(sets)])

    with torch.inference_mode():
        # ---- primary line: K steps of the production call -----------------------------------------------------------
        for i in range(args.warmup):
            step(i)
        with ops.KernelTimer(timing=False) as counter:  # counts the kernels launched inside the timed region (no events, no syncs)
            ms_step, clocks = timed(step, args.steps)
        launches = counter.launches
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, keep["out"], keep["w"])
        value = world * B * 1e3 / ms_step
        checksum = float(keep["out"].float().abs().mean().item())

        # ---- instrumented pass over the same K steps: per-kernel CUDA events (the roofline of the dominant kernel) ----
        with ops.KernelTimer(timing=True):
            for i in range(3):
                step(i)
        with ops.KernelTimer(timing=True) as kt:
            ms_instr, _ = timed(step, args.steps, clocks=False)
        durations = kt.durations_ms()

        # ---- strong scaling: BASELINE.json configs[2] — 64 videos global, 64 / N per rank (compute only) -----------------
        strong = None
        if world > 1 and not args.no_strong and scaling == "weak" and GLOBAL_BATCH % world == 0:
            Bs = GLOBAL_BATCH // world
            ssets = make_sets(Bs, 8, seed0=107)  # 8 rotating sets (> L2 together at every N)

            def sstep(i):
                keep["sout"], _ = module(ssets[i % len(ssets)])

            # the same number of videos as the primary line's timed region at N = 1 (K x 64): the same regime (burst clocks) on both
            # sides of the strong-scaling ratio; measured before the sustained run heats the part into its power cap
            n_steps = args.steps * world
            timed(sstep, 10, warmup=5, clocks=False)
            time.sleep(0.5)
            ms_s, clk_s = timed(sstep, n_steps)
            strong = {"scaling": "strong", "global_batch": GLOBAL_BATCH, "batch_per_gpu": Bs, "steps": n_steps, "ms_per_step": ms_s,
                      "value": GLOBAL_BATCH * 1e3 / ms_s, "unit": "videos/s", "clocks": clk_s,
                      "l2": f"8 rotating input sets of {BYTES_IN * Bs / 1e6:.0f} MB per rank",
                      "note": "compare with the N=1 line's value (64 videos on one GPU): strong-scaling speed-up = this value / that value"}
            del ssets

        # ---- sustained: the same step for hundreds of iterations (power-capped regime) ----------------------------------
        sustained = None
        if not args.no_sustained and args.sustained_steps > 0:
            ms_sus, clk_sus = timed(step, args.sustained_steps)
            sustained = {"steps": args.sustained_steps, "ms_per_step": ms_sus, "value": world * B * 1e3 / ms_sus, "unit": "videos/s", "clocks": clk_sus}
            # the opt-in pooling INSIDE the GEMM launch (MERV_POOL_ASSIST=1, DESIGN.md section 10), A/B in the regime the sustained run has just
            # established: alternating blocks of 100 steps, bit-identical outputs.  Only with --assist-ab (profiles/r2_bench_n1.json was taken with it).
            if args.assist_ab and world == 1 and args.mode == "fused" and args.projector == "linear":
                try:
                    ab = {"base_ms": [], "assist_ms": []}
                    for _ in range(3):
                        os.environ["MERV_POOL_ASSIST"] = "0"
                        ab["base_ms"].append(timed(step, 100, clocks=False)[0])
                        os.environ["MERV_POOL_ASSIST"] = "1"
                        ab["assist_ms"].append(timed(step, 100, clocks=False)[0])
                    ref_o, ref_w = keep["out"].clone(), keep["w"].clone()
                    os.environ["MERV_POOL_ASSIST"] = "0"
                    step(99)  # the same input set as the last assisted step (index 99 of its block)
                    ab["bit_identical"] = bool(torch.equal(ref_o, keep["out"]) and torch.equal(ref_w, keep["w"]))
                    ab["assist_over_base"] = sum(ab["assist_ms"]) / sum(ab["base_ms"])
                    ab["what"] = ("merv_fused_forward with the last 24 of 64 videos pooled, scored and soft-maxed by two spare warps of every GEMM CTA "
                                  "(release / acquire flags per video) vs the three-launch path; sustained regime, 3 x 100 steps each, alternating")
                    sustained["pool_assist_ab"] = ab
                except Exception as e:
                    sustained["pool_assist_ab"] = {"error": repr(e)[:300]}
                finally:
                    os.environ.pop("MERV_POOL_ASSIST", None)

        # ---- e2e: host buffers in, host buffers out, through the public host API ------------------------------------------
        e2e = None
        if not args.no_e2e:
            host_in = [torch.empty(f.shape, dtype=f.dtype).pin_memory() for f in sets[0]]  # pinned AFTER set_device: this rank's context
            for h, f in zip(host_in, sets[0]):
                h.copy_(f)
            host_out = torch.empty((B, OUT_TOKENS, LLM_DIM), dtype=torch.bfloat16).pin_memory()
            host_w = torch.empty((B, len(DIMS)), dtype=torch.bfloat16).pin_memory()
            pipe = HostPipeline(module, chunk_videos=8, device=dev)
            for _ in range(2):
                pipe(host_in, host_out, host_w)  # warm-up
            barrier()
            sampler = ClockSampler(local_rank).start()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                pipe(host_in, host_out, host_w)  # returns after the last D2H copy has landed (stream synchronize inside)
            torch.cuda.synchronize()
            dt = max_over_ranks(time.perf_counter() - t0)
            e2e = {"value": world * B * args.e2e_steps / dt, "unit": "videos/s", "h2d_bytes_per_step": BYTES_IN * B,
                   "d2h_bytes_per_step": BYTES_OUT * B + B * len(DIMS) * 2, "ms_per_step": dt / args.e2e_steps * 1e3,
                   "steps": args.e2e_steps, "clocks": sampler.stop(),
                   "api": "merv_b200.pipeline.HostPipeline (pinned host tensors, 8-video chunks with ramp-up/-down, copy/compute overlap)"}
            # what the bus alone allows for the same bytes with ALL ranks copying at once (not part of any reported throughput)
            dev_out = torch.empty((B, OUT_TOKENS, LLM_DIM), dtype=torch.bfloat16, device=dev)
            c0, c1, c2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            h2d, d2h = [], []
            for _ in range(3):
                barrier()
                c0.record()
                for h, f in zip(host_in, sets[0]):
                    f.copy_(h, non_blocking=True)
                c1.record()
                host_out.copy_(dev_out, non_blocking=True)
                c2.record()
                torch.cuda.synchronize()
                h2d.append(c0.elapsed_time(c1)); d2h.append(c1.elapsed_time(c2))
            e2e["h2d_only_ms"], e2e["d2h_only_ms"] = max_over_ranks(min(h2d)), max_over_ranks(min(d2h))
            # both directions at once on two streams, all ranks: the bound of a pipeline that overlaps copy-in and copy-out
            s_a, s_b = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            duplex = []
            for _ in range(3):
                barrier()
                d0, d1, d2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                d0.record()
                s_a.wait_event(d0); s_b.wait_event(d0)
                with torch.cuda.stream(s_a):
                    for h, f in zip(host_in, sets[0]):
                        f.copy_(h, non_blocking=True)
                    d1.record(s_a)
                with torch.cuda.stream(s_b):
                    host_out.copy_(dev_out, non_blocking=True)
                    d2.record(s_b)
                torch.cuda.synchronize()
                duplex.append(max(d0.elapsed_time(d1), d0.elapsed_time(d2)))
            e2e["h2d_and_d2h_concurrent_ms"] = max_over_ranks(min(duplex))
            e2e["frac_of_duplex_copy_limit"] = e2e["h2d_and_d2h_concurrent_ms"] / e2e["ms_per_step"]
            e2e["h2d_GBps_per_gpu_all_ranks_copying"] = BYTES_IN * B / e2e["h2d_only_ms"] / 1e6
            e2e["h2d_GBps_aggregate"] = world * e2e["h2d_GBps_per_gpu_all_ranks_copying"]
            e2e["frac_of_h2d_limit"] = e2e["h2d_only_ms"] / e2e["ms_per_step"]
            e2e["bound"] = ("host->device copy of the inputs with all ranks copying concurrently (PCIe / host memory, shared by the GPUs "
                            "of one root complex); frac_of_h2d_limit = that copy alone / e2e step")
            del host_in, host_out, dev_out, pipe

    def emit(gather):
        """Rank 0: derive the rooflines, run the N = 1 extras and print THE line."""
        # ---- rooflines (SURVEY.md §8d algorithmic bytes/FLOPs per video x videos per launch / measured duration) ----
        def avg(name):
            d = durations.get(name, [])
            return (sum(d) / len(d)) if d else None

        kernels = {}
        pool_calls = durations.get("merv_pool3d", [])
        pool_ms = (sum(pool_calls) / args.steps) if pool_calls else None  # per step (module-by-module mode pools each encoder separately)
        if pool_ms:
            gbs = (BYTES_IN + BYTES_POOLED) * B / (pool_ms * 1e-3) / 1e9
            kernels["merv_pool3d"] = {"bound": "hbm", "ms": pool_ms, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                                      "algorithmic_bytes": (BYTES_IN + BYTES_POOLED) * B,
                                      "traffic": ncu_traffic_bytes("r2_prof_pool3d_tma.txt", "r1g_prof_pool3d_tma.txt") if B == 64 else None}
        flops = FLOPS_LINEAR if args.projector == "linear" else FLOPS_GELU
        roofline = None
        if args.mode == "fused":
            gemm_name = "merv_fused_linear_mix"
            gemm_flops = (FLOPS_LINEAR if args.projector == "linear" else 4 * 2 * OUT_TOKENS * LLM_DIM * LLM_DIM) * B
            g_ms = avg(gemm_name)
            if g_ms:
                tf = gemm_flops / (g_ms * 1e-3) / 1e12
                # a 20-step timed region runs in the burst regime (boost clocks, no power cap yet): the burst cuBLAS figure is its peak;
                # the sustained fraction is stated next to it
                roofline = {"kernel": "gemm_bf16_tcgen05_kernel (merv_fused_linear_mix)", "bound": "tensor", "achieved": tf, "peak": peaks["tf_burst"],
                            "unit": "TFLOP/s", "frac": tf / peaks["tf_burst"], "frac_of_sustained_peak": tf / peaks["tf_sustained"],
                            "peak_source": peaks["source"] + " (burst cuBLAS bf16: the kernel is timed inside a short region)",
                            "ms_per_launch": g_ms, "timing": f"CUDA events around the launch in an instrumented pass over the same {args.steps} steps "
                                                             f"(step {ms_instr:.4f} ms with events vs {ms_step:.4f} ms in the timed region)",
                            "traffic": ncu_traffic_bytes("r2_prof_gemm_bf16_tcgen05.txt", "r1g_prof_gemm_bf16_tcgen05.txt") if (args.projector == "linear" and B == 64) else None,
                            "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum)",
                            "algorithmic_bytes": (BYTES_POOLED + BYTES_OUT) * B + sum(LLM_DIM * c * 2 for c in DIMS)}
                kernels[gemm_name] = roofline
        else:
            d = durations.get("merv_linear_bias_act", [])
            if d:
                per_step = sum(d) / args.steps
                tf = flops * B / (per_step * 1e-3) / 1e12
                roofline = {"kernel": "gemm_bf16_tcgen05_kernel (merv_linear_bias_act, all projector GEMMs of a step)", "bound": "tensor", "achieved": tf,
                            "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": tf / peaks["tf_burst"], "frac_of_sustained_peak": tf / peaks["tf_sustained"],
                            "peak_source": peaks["source"] + " (burst cuBLAS bf16)", "ms_per_step": per_step, "traffic": None}
            mix_ms = avg("merv_softmax_mix")
            if mix_ms:
                gbs = (4 * BYTES_Y + BYTES_OUT) * B / (mix_ms * 1e-3) / 1e9
                kernels["merv_softmax_mix"] = {"bound": "hbm", "ms": mix_ms, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"]}
        for name, d in durations.items():
            kernels.setdefault(name, {"ms": sum(d) / len(d)})
            kernels[name]["calls_per_step"] = len(d) / args.steps

        # ---- N = 1 extras: the other BASELINE.json configs, the torch-eager comparator, the CPU baseline ----
        configs = None
        if world == 1 and not args.no_configs:
            configs = {}
            with torch.no_grad():
                try:  # configs[3]: single-encoder SigLIP baseline (projector + spatial pool only, E = 1 mix is the identity), B = 256
                    B4 = 256
                    m4 = build_module([768], [16], "linear")
                    g = torch.Generator(device=dev).manual_seed(1)
                    x4 = [[torch.randn((B4, 16, 196, 768), generator=g, device=dev).to(torch.bfloat16)] for _ in range(2)]  # 2 x 1.23 GB > L2
                    r4 = {}

                    def step4(i):
                        r4["o"], r4["w"] = m4(x4[i % 2])

                    ms4, clk4 = timed(step4, 30, warmup=5)
                    fl4, by4 = 2 * OUT_TOKENS * LLM_DIM * 768 * B4, (16 * 196 * 768 * 2 + BYTES_OUT) * B4
                    configs["siglip_single_b256"] = {"workload": "single-encoder SigLIP (16 x 196 x 768) -> pool -> Linear(768, 4096), batch 256, bf16", "ms_per_step": ms4,
                                                     "value": B4 * 1e3 / ms4, "unit": "videos/s", "TFLOPs": fl4 / ms4 / 1e9, "frac_of_burst_tensor_peak": fl4 / ms4 / 1e9 / peaks["tf_burst"],
                                                     "compulsory_GBps": by4 / ms4 / 1e6, "weights_all_one": bool((r4["w"].float() == 1).all()), "steps": 30, "clocks": clk4}
                    del x4, r4, m4
                    torch.cuda.empty_cache()
                except Exception as e:
                    configs["siglip_single_b256"] = {"error": repr(e)[:300]}
                try:  # configs[4]: generate — fusion prefix feeding a random-init Llama-2-7B prefill (the LLM is a library consumer)
                    from transformers import LlamaConfig, LlamaForCausalLM

                    cfg = LlamaConfig()  # defaults = Llama-2-7B (4096 / 32 layers / 32 heads / 11008 / 32000)
                    cfg.vocab_size = 32064  # the reference pads the vocabulary to a multiple of 64 (llama2.py:74-76)
                    with torch.device("meta"):
                        llm = LlamaForCausalLM(cfg)
                    llm = llm.to_empty(device=dev).to(torch.bfloat16)
                    for p_ in llm.parameters():
                        p_.normal_(0, 0.02)
                    llm.eval()
                    g = torch.Generator(device=dev).manual_seed(2)
                    feats1 = [torch.randn((1, t, n, c), generator=g, device=dev).to(torch.bfloat16) for t, n, c in zip(TOKENS_T, PATCHES, DIMS)]
                    ids = torch.randint(0, 32000, (1, 33), device=dev)  # BOS + 32 text tokens (no tokenizer offline)

                    def prefix_only(i):
                        module(feats1)

                    def ttft(i):
                        emb = llm.get_input_embeddings()(ids)
                        buf, _ = module.forward_into_embeddings(feats1, emb, bos_token_length=1)  # [BOS | 1024 prefix | text], prefix written in place
                        llm(inputs_embeds=buf, use_cache=True).logits[:, -1].argmax(-1)

                    t_prefix, clk5 = timed(prefix_only, 200, warmup=10)
                    t_ttft, _ = timed(ttft, 5, warmup=2, clocks=False)
                    configs["generate_b1"] = {"workload": "merv-full generate, B = 1: fusion prefix -> random-init Llama-2-7B (bf16, HF transformers sdpa) prefill of 1 + 1024 + 32 tokens",
                                              "time_to_visual_prefix_ms": t_prefix, "ttft_ms": t_ttft, "prefill_tokens": 1 + OUT_TOKENS + 32, "clocks": clk5}
                    del llm, feats1
                    torch.cuda.empty_cache()
                except Exception as e:  # the LLM is only a timing sink
                    configs["generate_b1"] = {"error": repr(e)[:300]}

            try:  # the FSDP training step's share of the path (SURVEY.md §8 f-1): forward + hand-written backward + parameter-version bump
                tr = {}
                for Bt in (16, 64):  # 16 = the reference's per-device batch (conf/models.py:125)
                    gt = torch.Generator(device=dev).manual_seed(5)
                    ft = [torch.randn((Bt, t, n, c), generator=gt, device=dev).to(torch.bfloat16) for t, n, c in zip(TOKENS_T, PATCHES, DIMS)]
                    Gt = torch.randn((Bt, OUT_TOKENS, LLM_DIM), generator=gt, device=dev).to(torch.bfloat16)
                    mt = build_module(DIMS, TOKENS_T, "linear").train().requires_grad_(True)
                    mt.feature_fusion.fused_training = True
                    pt = list(mt.parameters())

                    def train_step(i):
                        o, _ = mt(ft)
                        o.backward(Gt)
                        mt.zero_grad(set_to_none=True)
                        with torch.no_grad():  # what an optimizer step does to the caches: every parameter gets a new version
                            torch._foreach_add_(pt, 0.0)

                    ms_t, clk_t = timed(train_step, 10, warmup=3)
                    tr[f"B{Bt}"] = {"ms_per_step": ms_t, "videos_per_s": Bt * 1e3 / ms_t, "steps": 10, "clocks": clk_t}
                    del mt, ft, Gt, pt
                    torch.cuda.empty_cache()
                tr["workload"] = ("merv-full fusion training step, bf16: fused forward + backward (weight gradients over per-video segments, "
                                  "merv_wgrad_video; no gradient into the frozen backbones' features) + parameter-version bump; same input every step")
                configs["train_step"] = tr
            except Exception as e:
                configs["train_step"] = {"error": repr(e)[:300]}

        # second comparator (SURVEY.md §8d "the real bar"): the reference's op sequence in PyTorch eager on this same B200
        torch_eager = None
        if world == 1 and not args.no_torch_eager:
            try:
                from oracle import torch_port

                pp = [{k: v for k, v in p.projector.state_dict().items()} for p in module.projectors]
                fp = dict(module.feature_fusion.state_dict())
                run = lambda i: torch_port.fusion_forward(sets[i % len(sets)], pp, fp, TOKENS_T, 8, args.projector, OUT_TOKENS)  # noqa: E731
                for i in range(3):
                    ref_out, _ = run(i)
                torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for i in range(5):
                    ref_out, _ = run(i)
                t1.record()
                torch.cuda.synchronize()
                ms_ref = t0.elapsed_time(t1) / 5
                with torch.inference_mode():
                    ours_out, _ = module(sets[4 % len(sets)])
                diff = float((ours_out.float() - ref_out.float()).abs().max() / ref_out.float().abs().max())
                torch_eager = {"value": B / (ms_ref * 1e-3), "unit": "videos/s", "ms_per_step": ms_ref, "speedup_of_this_repo": ms_ref / ms_step,
                               "max_rel_diff_vs_this_repo": diff,
                               "what": "oracle/torch_port.py (the reference's ATen op sequence: permute, adaptive_avg_pool3d, F.linear, stack, mean, MHA, bmm) in torch eager bf16 on the same GPU, same inputs"}
                del ref_out, ours_out
            except Exception as e:  # a comparator, never a dependency
                torch_eager = {"error": repr(e)[:200]}

        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            # bounded sample of the same workload: ~10-20 s of CPU work (a probe pass sizes the number of timed passes)
            _, probe_ms, _, _, _ = cpu_reference_run(args.projector, args.cpu_sample_videos, 1, 1)
            passes = max(3, min(40, int(12e3 / max(probe_ms, 1.0))))
            v, ms, cores, kind, what = cpu_reference_run(args.projector, args.cpu_sample_videos, passes, 1)
            cpu_baseline = {"value": v, "unit": "videos/s", "cores": cores, "cpu": cpu_model(), "kind": kind, "what": what, "ms_per_video": 1e3 / v,
                            "sample": f"{args.cpu_sample_videos} merv-full videos per pass (bf16), {passes} passes (~{passes * ms / 1e3:.0f} s) after 1 warm-up"}

        line = {
            "metric": "merv-full fusion videos/sec", "value": value, "unit": "videos/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, world),
            "fused_tokens_per_s": value * OUT_TOKENS,
            "path_effective_GBps_per_gpu": (BYTES_IN + BYTES_OUT) * B / (ms_step * 1e-3) / 1e9,
            "path_TFLOPs_per_gpu": flops * B / (ms_step * 1e-3) / 1e12,
            "path_frac_of_burst_tensor_peak": flops * B / (ms_step * 1e-3) / 1e12 / peaks["tf_burst"],
            "roofline": roofline, "kernels": kernels, "sustained": sustained, "strong": strong, "gather": gather, "configs": configs,
            "cpu_baseline": cpu_baseline, "torch_eager_same_gpu": torch_eager, "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_per_step": launches / args.steps, "clocks": clocks, "output_abs_mean": checksum,
            "call": "MervFusion.forward -> one C call per step (merv_fused_forward: pool3d_tma_kernel, scores_softmax_kernel, gemm_bf16_tcgen05_kernel chained by PDL)"
                    if args.mode == "fused" and args.projector == "linear" else "module-by-module",
            "peaks": peaks,
        }
        print(json.dumps(line), flush=True)

    gather = {}

    def finish(gather_rec, hard_exit: bool = False):
        if rank == 0:
            emit(gather_rec if gather_rec else None)
        if hard_exit:
            sys.stdout.flush()
            os._exit(0)

    with torch.inference_mode():
        # ---- all-gather of the fused prefixes (the only collective of the path; SURVEY.md §8e) ---------------------------
        # Runs LAST and under a watchdog: it is the only part of the bench in which the ranks depend on each other inside a
        # kernel (peer / multicast stores, symmetric-memory barriers).  If it does not finish in time every rank leaves and rank 0
        # still prints the line with everything measured so far.
        if world > 1 and not args.no_gather:
            gather.clear()
            watchdog = threading.Timer(args.gather_timeout, lambda: (finish({"error": f"watchdog: the gather sub-records did not finish within {args.gather_timeout} s",
                                                                             **gather}, hard_exit=True)))
            watchdog.daemon = True
            watchdog.start()
            from merv_b200.parallel import SymmetricPrefixBuffer, all_gather_prefix

            for name, Bg in (("strong_shards", GLOBAL_BATCH // world if GLOBAL_BATCH % world == 0 else 0), ("weak_shards", B)):
                if Bg <= 0:
                    continue
                rec = {"batch_per_gpu": Bg, "gathered_videos": Bg * world, "recv_bytes_per_gpu": (world - 1) * Bg * BYTES_OUT}
                try:
                    gsets = sets if Bg == B else make_sets(Bg, 4, seed0=207)
                    res = {}

                    def g_compute(i):
                        res["o"], _ = module(gsets[i % len(gsets)])

                    def g_nccl(i):
                        o, _ = module(gsets[i % len(gsets)])
                        res["g"] = all_gather_prefix(o, Bg * world)

                    def g_only(i):
                        res["g"] = all_gather_prefix(res["o"], Bg * world)

                    n_g = int(min(200, max(10, 100.0 / (0.03 * Bg * world))))
                    rec["steps"] = n_g
                    rec["compute_ms"], _ = timed(g_compute, n_g, warmup=3, clocks=False)
                    rec["nccl_allgather_only_ms"], _ = timed(g_only, n_g, warmup=3, clocks=False)
                    rec["compute_then_nccl_ms"], rec["clocks"] = timed(g_nccl, n_g, warmup=3)
                    buf = SymmetricPrefixBuffer(Bg, OUT_TOKENS, LLM_DIM, device=dev)

                    def g_fused(i):
                        res["f"], _ = module(gsets[i % len(gsets)], gather=buf)

                    g_nccl(0)
                    g_fused(0)
                    torch.cuda.synchronize()
                    same = torch.tensor([1 if torch.equal(res["f"], res["g"]) else 0], device=dev)
                    dist.all_reduce(same, op=dist.ReduceOp.MIN)
                    rec["fused_bit_identical_to_nccl_on_all_ranks"] = bool(same.item())
                    rec["fused_gemm_allgather_ms"], _ = timed(g_fused, n_g, warmup=3, clocks=False)
                    rec["fused_ingress_GBps_per_gpu"] = rec["recv_bytes_per_gpu"] / rec["fused_gemm_allgather_ms"] / 1e6
                    rec["fused_over_compute"] = rec["fused_gemm_allgather_ms"] / rec["compute_ms"]
                    # B200_PROFILING.md: the target of a fused compute + collective kernel is the slower of the compute and the bytes
                    # that must cross NVLink at the measured 770 GB/s per direction per GPU (every rank RECEIVES world - 1 blocks)
                    nvlink_ms = rec["recv_bytes_per_gpu"] / 770e9 * 1e3
                    rec["roofline"] = {"compute_ms": rec["compute_ms"], "nvlink_ingress_ms_at_770GBps": nvlink_ms, "floor_ms": max(rec["compute_ms"], nvlink_ms),
                                       "frac_of_floor": max(rec["compute_ms"], nvlink_ms) / rec["fused_gemm_allgather_ms"],
                                       "bound": "nvlink ingress" if nvlink_ms > rec["compute_ms"] else "tensor"}
                    rec["transport"] = getattr(buf, "transport", "unicast TMA stores to peer-mapped buffers")
                    del buf, res
                    if Bg != B:
                        del gsets
                except Exception as e:  # a sub-record never takes the primary line down
                    rec["error"] = repr(e)[:300]
                gather[name] = rec
            watchdog.cancel()


    if world > 1:
        barrier()
    finish(gather)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

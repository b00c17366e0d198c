"""Cost of the attentive pooler's attention backward (merv_cross_attention_backward_ex) and of whole `attntv` training steps.

    python scripts/gpu_attention_backward_cost.py [--out report.json] [--iters 20] [--steps 3]

Kernel: ops.cross_attention_backward on pre-built inputs, timed with CUDA events over `--iters` calls after a warm-up, at
  - the shipped shapes, 16 videos x 16 frames (256 frames), 64 queries, 8 heads: 256 keys with head_dim 128 (LanguageBind / DINOv2) and
    196 keys with head_dim 96 (ViViT / SigLIP), bf16, the tcgen05 kernel against the CUDA-core kernel forced with MERV_ATTN_IMPL=simt;
  - the CUDA-core kernel where it is the only one: 144 queries x 256 keys, 64 queries x 729 keys (bf16), and the shipped shapes in fp32.
Every time comes with the contraction FLOPs counted from the shapes, per frame and head: the five contractions of the backward (S = Q K^T
recomputed, dP = dO V^T, dV = P^T dO, dK = dS^T Q, dQ = dS K), 5 x 2 n_q n_kv hd, and separately the CUDA-core kernel's first sweep
over the keys, which recomputes S and dP for the softmax statistics and D, 2 x 2 n_q n_kv hd.

Training step: AttentivePooler(1024 -> 4096, 16 frames x 256 patches, 8 heads, linear projector) forward + backward at 16 videos, with
projector_token_length 64 and 144, in bf16 and in fp32, over `--steps` steps after one warm-up step.

Needs a B200; prints one JSON document and reads the card's name and power limit in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

import merv_b200 as M  # noqa: E402
from merv_b200 import ops  # noqa: E402

DEV = "cuda:0"
FRAMES, HEADS = 256, 8  # 16 videos x 16 frames


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def flops(frames, n_q, n_kv, hd):
    one = 2 * n_q * n_kv * hd * frames * HEADS
    return 5 * one, 2 * one


def kernel_case(name, dtype, n_q, n_kv, hd, impls, iters):
    g = torch.Generator(device=DEV).manual_seed(n_q + n_kv + hd)
    C_ = HEADS * hd
    q = torch.randn(n_q, C_, generator=g, device=DEV).to(dtype)
    kv = torch.randn(FRAMES * n_kv, 2 * C_, generator=g, device=DEV).to(dtype)
    dout = torch.randn(FRAMES, n_q, C_, generator=g, device=DEV).to(dtype)
    main, sweep = flops(FRAMES, n_q, n_kv, hd)
    rec = {"dtype": str(dtype).split(".")[-1], "frames": FRAMES, "heads": HEADS, "n_q": n_q, "n_kv": n_kv, "head_dim": hd,
           "contraction_GFLOP": main / 1e9, "simt_stats_sweep_GFLOP": sweep / 1e9}
    for impl in impls:
        if impl == "simt":
            os.environ["MERV_ATTN_IMPL"] = "simt"
        try:
            ms = timed(lambda: ops.cross_attention_backward(q, kv, dout, FRAMES, HEADS), iters)
        finally:
            os.environ.pop("MERV_ATTN_IMPL", None)
        done = main + (sweep if impl == "simt" else 0)
        rec[impl] = {"ms": round(ms, 4), "contraction_TFLOPs": round(main / ms / 1e9, 2), "all_computed_TFLOPs": round(done / ms / 1e9, 2)}
    print(name, rec, flush=True)
    return rec


def train_case(dtype, ptl, steps):
    torch.manual_seed(0)
    pool = M.AttentivePooler(1024, 4096, num_query_tokens=ptl, num_heads=HEADS, output_frames=16, mlp_type="linear").to(DEV, dtype).train()
    g = torch.Generator(device=DEV).manual_seed(ptl)
    x = torch.randn(16, 16, 256, 1024, generator=g, device=DEV).to(dtype)
    G = torch.randn(16, 16 * ptl, 4096, generator=g, device=DEV).to(dtype)

    def step():
        pool(x).backward(G)
        pool.zero_grad(set_to_none=True)

    ms = timed(step, steps, warmup=1)  # plain event timing: autograd's worker thread does not take part in a CUDA-graph capture
    with ops.KernelTimer(timing=True) as kt:
        step()
    per = {k: round(sum(v), 4) for k, v in kt.durations_ms().items()}
    main, sweep = flops(FRAMES, ptl, 256, 128)
    rec = {"dtype": str(dtype).split(".")[-1], "projector_token_length": ptl, "videos": 16, "step_ms": round(ms, 3),
           "device_ms_by_entry_point": dict(sorted(per.items(), key=lambda kv: -kv[1])),
           "attention_backward_contraction_GFLOP": main / 1e9, "attention_backward_simt_stats_sweep_GFLOP": sweep / 1e9}
    print("train", rec, flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rep = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "kernel": {}, "train_step": []}
    print(rep["device"], rep["nvidia_smi"], flush=True)
    bf, f32 = torch.bfloat16, torch.float32
    cases = [("shipped_256keys_hd128", bf, 64, 256, 128, ("tcgen05", "simt")), ("shipped_196keys_hd96", bf, 64, 196, 96, ("tcgen05", "simt")),
             ("q144_kv256_hd128", bf, 144, 256, 128, ("simt",)), ("q64_kv729_hd128", bf, 64, 729, 128, ("simt",)),
             ("fp32_256keys_hd128", f32, 64, 256, 128, ("simt",)), ("fp32_196keys_hd96", f32, 64, 196, 96, ("simt",))]
    for name, dt, n_q, n_kv, hd, impls in cases:
        rep["kernel"][name] = kernel_case(name, dt, n_q, n_kv, hd, impls, a.iters)
    for dt in (bf, f32):
        for ptl in (64, 144):
            rep["train_step"].append(train_case(dt, ptl, a.steps))
    text = json.dumps(rep, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

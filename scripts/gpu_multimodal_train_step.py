"""Cost of assembling the [BOS | prefix | text] embeddings in the training step at the merv-full shapes: E = 4 encoders, T = 1024 tokens,
K = 4096, bf16, 16 and 64 videos, text lengths 64 and 512.

    python scripts/gpu_multimodal_train_step.py [--out report.json] [--steps 5] [--reps 3]

For each shape, one training step (forward + backward of a loss on the embeddings and the mixing weights + a version bump of every parameter,
what an optimizer step does to the cached compute-dtype copies) is timed with CUDA events in two ways:
  - "multimodal": MervFusion.forward_multimodal — the mixer's autograd Function owns the buffer, the kernels write the prefix into its slot
    and read its gradient from the buffer's gradient in place;
  - "cat": MervFusion.forward followed by the reference's torch.cat assembly (merv.py:622-664) — the prefix is copied into the buffer and its
    gradient copied back out.
Both for the fused step (fused_training=True: _FusedLinearFn) and module by module (fused_training=False), alternated `--reps` times over
`--steps` steps each.  The parameter and input_embeddings gradients of the two ways are compared bit for bit on the first step.  Needs a B200;
prints one JSON document with the card's name and power limit.
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

DEV = "cuda:0"
T, K = 1024, 4096
DIMS, PATCHES = [1024, 1024, 768, 768], [256, 256, 196, 196]


def build(fused):
    m = M.MervFusion.from_config(DIMS, K, [16] * 4, arch_specifier="3davg+linear", feature_fusion="cross_attention_avg_lq",
                                 projector_token_length=64, visual_feature_length=T, fused_training=fused)
    return m.to(device=DEV, dtype=torch.bfloat16).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rep = {"gpu": smi.stdout.strip(), "shapes": []}
    models = {f: build(f) for f in (True, False)}
    for B in (16, 64):
        g = torch.Generator(device=DEV).manual_seed(B)
        feats = [torch.randn((B, 16, n, c), generator=g, device=DEV).to(torch.bfloat16) for n, c in zip(PATCHES, DIMS)]
        for L in (64, 512):
            emb = torch.randn((B, L, K), generator=g, device=DEV).to(torch.bfloat16)
            R = torch.randn((B, L + T, K), generator=g, device=DEV).to(torch.bfloat16)
            r = torch.randn((B, 4), generator=g, device=DEV)
            row = {"videos": B, "text": L}
            for fused, m in models.items():
                params = [p for p in m.parameters()]
                trained = [p for n, p in m.named_parameters() if "v_proj" not in n and "out_proj" not in n]  # dead in the reference too

                def step(way, m=m, params=params):
                    m.zero_grad(set_to_none=True)
                    e = emb.clone().requires_grad_(True)
                    if way == "multimodal":
                        buf, _, _, w = m.forward_multimodal(feats, e, bos_token_length=1)
                    else:
                        prefix, w = m(feats)
                        buf = torch.cat([e[:, :1], prefix, e[:, 1:]], 1)
                    ((buf * R).float().sum() + (w.float() * r).sum()).backward()
                    with torch.no_grad():
                        torch._foreach_add_(params, 0.0)
                    return e

                grads = {}
                for way in ("multimodal", "cat"):
                    e = step(way)
                    grads[way] = [p.grad.clone() for p in trained] + [e.grad.clone()]
                same = all(torch.equal(a, b) for a, b in zip(grads["multimodal"], grads["cat"]))
                del grads
                times = {"multimodal": [], "cat": []}
                for _ in range(args.reps):
                    for way in ("multimodal", "cat"):
                        step(way)
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(args.steps):
                            step(way)
                        e1.record()
                        torch.cuda.synchronize()
                        times[way].append(e0.elapsed_time(e1) / args.steps)
                row["fused" if fused else "module"] = {"ms_multimodal": times["multimodal"], "ms_cat": times["cat"], "grads_bit_identical": same}
            rep["shapes"].append(row)
            print(json.dumps(row), flush=True)
    out = json.dumps(rep, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out)


if __name__ == "__main__":
    main()

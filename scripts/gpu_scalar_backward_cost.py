"""Cost of training the scalar mixer (feature_fusion="scalar", ScalarAdapter) at the merv-full shapes: E = 4 encoders, T = 1024 tokens,
K = 4096, bf16, 16 and 64 videos.

    python scripts/gpu_scalar_backward_cost.py [--out report.json] [--iters 20] [--steps 10]

Kernel: merv_scalar_mix_backward called straight through the C ABI on pre-allocated buffers and timed with CUDA events over `--iters`
calls.  Its bandwidth counts the bytes the maths needs, (1 + 2E) B T K elements (dOut and every V_e read once, every dV_e written once);
"frac" is that over the HBM bandwidth measured in the same run with a 4 GiB device-to-device copy.  The working set (1.2 GB at 16 videos)
is far larger than the 126 MB L2.

Training step: MervFusion.from_config(arch_specifier="3davg+linear", feature_fusion="scalar") forward + backward + a version bump of every
parameter (what an optimizer step does to the cached compute-dtype copies), fused (fused_training=True: _FusedScalarLinearFn) and module
by module (fused_training=False: projector autograd + _ScalarMixFn), alternated three times over `--steps` steps each.  The gradients of
the two paths are compared on the first step.  Needs a B200; prints one JSON document and reads the card's name and power limit.
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
from merv_b200 import _lib  # noqa: E402

DEV = "cuda:0"
E, T, K = 4, 1024, 4096
DIMS, PATCHES = [1024, 1024, 768, 768], [256, 256, 196, 196]


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


def hbm_peak_gbs(iters):
    src = torch.empty(2 << 30, dtype=torch.bfloat16, device=DEV).fill_(1.0)  # 4 GiB
    dst = torch.empty_like(src)
    best = min(timed(lambda: dst.copy_(src), iters) for _ in range(3))
    nbytes = 2 * src.numel() * src.element_size()
    del src, dst
    return nbytes / best / 1e6


def kernel_cost(B, iters, hbm, rep):
    lib = _lib.load()
    g = torch.Generator(device=DEV).manual_seed(B)
    V = [(torch.randn(B, T, K, generator=g, device=DEV) + 0.25 * e).to(torch.bfloat16) for e in range(E)]
    dout = torch.randn(B, T, K, generator=g, device=DEV).to(torch.bfloat16)
    w = torch.softmax(torch.tensor([0.7, -0.4, 0.1, 0.3], device=DEV), 0)
    dw = torch.randn(E, generator=g, device=DEV)
    dV = [torch.empty_like(v) for v in V]
    dscalar = torch.empty(E, dtype=torch.float32, device=DEV)
    n = lib.merv_scalar_mix_backward_workspace(B, E, K)
    ws = torch.empty(n, dtype=torch.float32, device=DEV)
    args_ = (_lib.ptr_array([v.data_ptr() for v in V]), dout.data_ptr(), w.data_ptr(), dw.data_ptr(), _lib.ptr_array([d.data_ptr() for d in dV]),
             dscalar.data_ptr(), ws.data_ptr(), n, B, E, T, K, _lib.MERV_BF16, torch.cuda.current_stream().cuda_stream)
    call = lambda: _lib.check(lib.merv_scalar_mix_backward(*args_))  # noqa: E731
    ms = [timed(call, iters) for _ in range(3)]
    nbytes = (1 + 2 * E) * B * T * K * 2
    best = min(ms)
    gbs = nbytes / best / 1e6
    rep[f"B{B}_merv_scalar_mix_backward"] = {"ms_best": best, "ms_all": ms, "bytes": nbytes, "GBps": gbs, "frac_of_measured_hbm": gbs / hbm}
    print(f"B={B:3d} merv_scalar_mix_backward {best:8.3f} ms  {gbs:7.0f} GB/s  ({gbs / hbm:.2f} of measured HBM)", flush=True)
    del V, dout, dV, ws
    torch.cuda.empty_cache()


def step_cost(B, steps, rep):
    g = torch.Generator(device=DEV).manual_seed(5)
    feats = [torch.randn((B, 16, n, c), generator=g, device=DEV).to(torch.bfloat16) for n, c in zip(PATCHES, DIMS)]
    G = torch.randn((B, T, K), generator=g, device=DEV).to(torch.bfloat16)
    mods, fns, grads = {}, {}, {}
    for name, ft in (("fused", True), ("module_by_module", False)):
        m = M.MervFusion.from_config(DIMS, K, [16] * 4, arch_specifier="3davg+linear", feature_fusion="scalar", projector_token_length=64,
                                     visual_feature_length=T, seed=1024, fused_training=ft).to(device=DEV, dtype=torch.bfloat16).train()
        params = list(m.parameters())

        def step(m=m, params=params):
            out, w = m(feats)
            out.backward(G)
            m.zero_grad(set_to_none=True)
            with torch.no_grad():  # an optimizer step gives every parameter a new version: cached compute-dtype copies are rebuilt
                torch._foreach_add_(params, 0.0)

        out, _ = m(feats)
        fn_name = type(out.grad_fn).__name__
        out.backward(G)
        grads[name] = {k: p.grad.float().clone() for k, p in m.named_parameters()}
        m.zero_grad(set_to_none=True)
        mods[name], fns[name] = m, step
        rep[f"B{B}_step_{name}_autograd_fn"] = fn_name
    errs = {k: float((grads["fused"][k] - grads["module_by_module"][k]).abs().max() / grads["module_by_module"][k].abs().max().clamp_min(1e-30))
            for k in grads["fused"]}
    rep[f"B{B}_step_grad_rel_err_fused_vs_module_max"] = max(errs.values())
    del grads
    runs = {name: [] for name in fns}
    for _ in range(3):  # alternate the two paths so drift on a shared host hits both alike
        for name, fn in fns.items():
            runs[name].append(timed(fn, steps, warmup=2))
    for name, ms in runs.items():
        rep[f"B{B}_step_{name}"] = {"ms_best": min(ms), "ms_all": ms}
        print(f"B={B:3d} training step {name:18s} {min(ms):8.3f} ms", flush=True)
    rep[f"B{B}_step_fused_over_module"] = min(runs["fused"]) / min(runs["module_by_module"])
    del mods, fns, feats, G
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rep = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "shape": dict(E=E, T=T, K=K, dtype="bf16"),
           "bytes": "(1 + 2E) B T K elements: dOut and every V_e read once, every dV_e written once", "hbm_peak_GBps": hbm_peak_gbs(args.iters)}
    for B in (16, 64):
        kernel_cost(B, args.iters, rep["hbm_peak_GBps"], rep)
    for B in (16, 64):
        step_cost(B, args.steps, rep)
    print(json.dumps(rep, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(rep, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()

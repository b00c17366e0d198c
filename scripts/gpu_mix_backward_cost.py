"""Cost of the adapter backward per configuration: merv_mix_backward vs merv_mix_backward_ex at the merv-full shapes (E = 4 encoders,
T = 1024 tokens, K = 4096, bf16) for 16 and 64 videos.

    python scripts/gpu_mix_backward_cost.py [--out report.json] [--iters 20]

Cases: the shipped configuration through both entry points (alternated, same buffers), positional embedding (merv_mix_backward_ex with
pe), and one single-token encoder (encoder 3 with T_e = 1).  The entry points are called straight through the C ABI on pre-allocated
buffers and timed with CUDA events over `--iters` calls.  Bandwidth counts the bytes the maths needs: every T-token V_e and dOut read
once, every dV_e written once (the single-token encoder: one [B, K] row block each way); "frac" is that over the HBM bandwidth measured in
the same run with a 4 GiB device-to-device copy.  Needs a B200; prints one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from merv_b200 import _lib, ops  # noqa: E402

DEV = "cuda:0"
E, T, K, EMBED = 4, 1024, 4096, 3072


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    lib = _lib.load()
    dt, code, esz = torch.bfloat16, _lib.MERV_BF16, 2
    g = torch.Generator(device=DEV).manual_seed(0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rep = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "shape": dict(E=E, T=T, K=K, embed=EMBED, dtype="bf16"),
           "bytes": "T-token V_e and dOut read once, dV_e written once", "hbm_peak_GBps": hbm_peak_gbs(args.iters), "cases": {}}
    Q = (torch.randn(1, EMBED, generator=g, device=DEV) * 4).to(dt)
    Wq = (torch.randn(EMBED, EMBED, generator=g, device=DEV) / EMBED ** 0.5).to(dt)
    Wk = (torch.randn(EMBED, K, generator=g, device=DEV) / K ** 0.5).to(dt)
    bias = (torch.randn(3 * EMBED, generator=g, device=DEV) * 0.05).to(dt)
    pe = (torch.randn(E, K, generator=g, device=DEV) * 0.05).to(dt)
    u = ops.fusion_query_vec(Q, Wq, Wk, bias)
    for B in (16, 64):
        V = [(torch.randn(B, T, K, generator=g, device=DEV) + 0.25 * e).to(dt) for e in range(E)]
        dout = torch.randn(B, T, K, generator=g, device=DEV).to(dt)
        weights = torch.softmax(torch.randn(B, E, generator=g, device=DEV), -1)
        dV = [torch.empty_like(v) for v in V]
        dQ, dWq, dWk = torch.empty(1, EMBED, dtype=dt, device=DEV), torch.empty_like(Wq), torch.empty_like(Wk)
        dbias, dpe = torch.empty_like(bias), torch.empty_like(pe)
        n = lib.merv_mix_backward_ex_workspace(B, E, T, K, EMBED, 0)
        ws = torch.empty(n, dtype=torch.float32, device=DEV)
        stream = torch.cuda.current_stream().cuda_stream
        common_out = (dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr())

        def ex_call(Vs, dVs, pe_t):
            vp, dvp = _lib.ptr_array([v.data_ptr() for v in Vs]), _lib.ptr_array([d.data_ptr() for d in dVs])
            tok = _lib.i32_array([v.shape[1] for v in Vs])
            pe_p, dpe_p = (None, None) if pe_t is None else (pe_t.data_ptr(), dpe.data_ptr())
            args_ = (vp, tok, dout.data_ptr(), weights.data_ptr(), None, u.data_ptr(), 0, pe_p, K, Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(),
                     bias.data_ptr(), dvp, *common_out, dpe_p, ws.data_ptr(), n, B, E, T, K, EMBED, code, stream)
            return lambda: _lib.check(lib.merv_mix_backward_ex(*args_))

        vp, dvp = _lib.ptr_array([v.data_ptr() for v in V]), _lib.ptr_array([d.data_ptr() for d in dV])
        old_args = (vp, dout.data_ptr(), weights.data_ptr(), None, u.data_ptr(), Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(), bias.data_ptr(), dvp,
                    *common_out, ws.data_ptr(), n, B, E, T, K, EMBED, code, stream)
        old = lambda: _lib.check(lib.merv_mix_backward(*old_args))  # noqa: E731
        shipped_ex = ex_call(V, dV, None)
        pe_ex = ex_call(V, dV, pe)
        Vs1 = V[:3] + [V[3][:, :1].contiguous()]
        dVs1 = dV[:3] + [torch.empty_like(Vs1[3])]
        single_ex = ex_call(Vs1, dVs1, None)
        full_bytes = (2 * E + 1) * B * T * K * esz
        single_bytes = (2 * (E - 1) + 1) * B * T * K * esz + 2 * B * K * esz
        runs = {"shipped_mix_backward": [], "shipped_mix_backward_ex": [], "pe_mix_backward_ex": [], "single_token_mix_backward_ex": []}
        for _ in range(3):  # alternate the variants so drift on a shared host hits all of them alike
            runs["shipped_mix_backward"].append(timed(old, args.iters))
            runs["shipped_mix_backward_ex"].append(timed(shipped_ex, args.iters))
            runs["pe_mix_backward_ex"].append(timed(pe_ex, args.iters))
            runs["single_token_mix_backward_ex"].append(timed(single_ex, args.iters))
        for name, ms in runs.items():
            nbytes = single_bytes if name.startswith("single") else full_bytes
            best = min(ms)
            gbs = nbytes / best / 1e6
            rep["cases"][f"B{B}_{name}"] = {"ms_best": best, "ms_all": ms, "GBps": gbs, "frac_of_measured_hbm": gbs / rep["hbm_peak_GBps"],
                                            "bytes": nbytes}
            print(f"B={B:3d} {name:30s} {best:8.3f} ms  {gbs:7.0f} GB/s  ({gbs / rep['hbm_peak_GBps']:.2f} of measured HBM)", flush=True)
        del V, dout, dV, Vs1, dVs1, ws
        torch.cuda.empty_cache()
    print(json.dumps(rep, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(rep, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()

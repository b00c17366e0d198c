"""The FSDP drop-in (BASELINE.json north_star: "drops into ... the FSDP training step"): a stand-in MERV holding the reference's own
modules is wrapped by torch FSDP exactly as merv/training/strategies/fsdp.py:208-241 does, once unmodified and once after
``merv_b200.patch_merv``; both train for a few steps on two ranks and must agree (tests/fsdp_worker.py has the criteria).

* ``-m "not gpu"``: two gloo ranks on CPU with the kernels replaced by tests/kernel_emulation.py — the host logic under REAL FSDP
  (unit boundaries, flat-parameter views, resharding between forward and backward, cache invalidation, wrap-policy extension).
* ``-m gpu``: two nccl ranks, one B200 each, the real kernels (skipped on a box with fewer than 2 GPUs).
"""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_ranks(script: str, nproc: int, *args: str, timeout: int = 900):
    """torchrun-style launch of tests/<script> on `nproc` local ranks; returns the parsed '<TAG> {json}' lines of all ranks."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(REPO, "tests", script), *args]
    env = dict(os.environ, OMP_NUM_THREADS="2", PYTHONPATH=REPO + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=REPO, env=env)
    # the ranks share one stdout and their reports can land on the same line: scan for every "<TAG> {json}" occurrence
    lines, dec, pos = [], json.JSONDecoder(), 0
    while True:
        hits = [i for i in (r.stdout.find(tag, pos) for tag in ("FSDP_WORKER ", "GATHER_WORKER ")) if i >= 0]
        if not hits:
            break
        start = r.stdout.index("{", min(hits))
        obj, end = dec.raw_decode(r.stdout, start)
        lines.append(obj)
        pos = end
    assert r.returncode == 0, f"ranks failed (rc {r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    assert len(lines) == nproc, f"expected one report per rank, got {len(lines)}:\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}"
    return lines


@pytest.mark.parametrize("mode,mlp_type,resampler", [("per_unit", "linear", "3davg"), ("root_unit", "linear", "3davg"), ("per_unit", "gelu-mlp", "3davg"),
                                                     ("per_unit", "linear", "3dconv")])
def test_fsdp_two_ranks_host_logic_on_cpu(mode, mlp_type, resampler):
    reports = run_ranks("fsdp_worker.py", 2, "--backend", "gloo", "--mode", mode, "--mlp-type", mlp_type, "--resampler", resampler)
    for rep in reports:
        assert rep["ok"], rep
        if mode == "per_unit":  # the reference's own unit list: each resampler and its inner projector are FSDP units
            assert sum("projectors" in u for u in rep["units_ours"]) == 6
            assert rep["fused_fn"].startswith("_MixFn")
        else:  # projectors + adapter in the root unit -> the fused forward / backward
            assert not any("projectors" in u for u in rep["units_ours"])
            assert rep["fused_fn"].startswith("_FusedLinearFn")


@pytest.mark.gpu
@pytest.mark.parametrize("mode,mlp_type,resampler", [("per_unit", "linear", "3davg"), ("root_unit", "linear", "3davg"), ("per_unit", "gelu-mlp", "3davg"),
                                                     ("per_unit", "linear", "3dconv")])
def test_fsdp_two_gpus(mode, mlp_type, resampler):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    reports = run_ranks("fsdp_worker.py", 2, "--backend", "nccl", "--mode", mode, "--mlp-type", mlp_type, "--resampler", resampler)
    for rep in reports:
        assert rep["ok"], rep
        assert rep["native_lib"].endswith("libmerv_fusion.so")
        assert rep["fused_fn"].startswith("_FusedLinearFn" if mode == "root_unit" else "_MixFn")


def test_patch_merv_extends_the_models_fsdp_policy():
    """SURVEY.md §7.2: patch_merv makes vidlm.get_fsdp_wrapping_policy() (merv.py:465-497) cover the swapped-in classes."""
    import functools

    import torch.nn as nn
    from torch.distributed.fsdp.wrap import _module_wrap_policy, _or_policy

    import merv_b200 as M

    class Vid(nn.Module):
        def __init__(self):
            super().__init__()
            self.projectors = nn.ModuleList([M.AveragePooling3DProjector(16, 32, 2, 2, "linear"), M.AveragePooling3DProjector(24, 32, 2, 2, "linear")])
            self.feature_fusion = M.CrossAttentionAdapterLearnableQuery(24, 32, 8, averagetoken=True)

        def get_fsdp_wrapping_policy(self):
            return functools.partial(_or_policy, policies=[functools.partial(_module_wrap_policy, module_classes={nn.Embedding})])

    def wrapped(v):
        pol = v.get_fsdp_wrapping_policy()
        return [type(m).__name__ for m in v.modules() if pol(module=m, recurse=False, nonwrapped_numel=0)]

    v = M.patch_merv(Vid())
    assert wrapped(v).count("AveragePooling3DProjector") == 2 and wrapped(v).count("LinearProjector") == 2
    assert "CrossAttentionAdapterLearnableQuery" not in wrapped(v)  # folds into the root unit, as in the reference
    v = M.patch_merv(Vid(), fused_training=True)
    assert wrapped(v) == []  # projectors share the root unit with the adapter: the fused training step can see every weight
    pol = M.fsdp_wrap_policy()
    assert pol(module=M.MLPProjector(8, 8), recurse=False, nonwrapped_numel=0) and not pol(module=nn.Linear(2, 2), recurse=False, nonwrapped_numel=0)

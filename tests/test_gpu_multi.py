"""Multi-GPU parity (needs >= 2 B200s on the box): K1 all-reduce / reduce-scatter over peer memory, the sharded K2 with
its in-kernel parameter all-gather, cross-rank norm / inf exchange, loss mean and barrier -- against the CPU oracle with W
logical ranks.  Each case runs in its own torch.distributed.run job under a hard timeout."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(world, tmp_path, port, algo="ldg"):
    out = tmp_path / f"mgpu_{world}_{algo}.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_worker.py"), str(out)]
    # cross-rank K1 flavour: register-staged loads | bulk-async through smem | multimem (NVLS); tiny gradient buckets in the
    # Stoke-API section so that the per-bucket launches from autograd hooks are exercised on a small model
    env = dict(os.environ, STK_K1_ALGO=algo, STK_BUCKET_MB="0.0005", STK_OVERLAP="on", STK_SPIN_TIMEOUT_S="30")
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
    assert proc.returncode == 0, proc.stdout[-4000:] + proc.stderr[-4000:]
    with open(out) as f:
        res = json.load(f)
    keep = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(keep):   # evidence for profiles/: which memory mode / multicast binding each flavour really ran with
        with open(os.path.join(keep, f"mgpu_w{world}_{algo}.json"), "w") as f:
            json.dump(res, f, indent=1)
    return res


@pytest.mark.parametrize("algo", ["ldg", "bulk", "nvls"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_parity(world, algo, tmp_path):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    res = _run(world, tmp_path, 29500 + world + {"ldg": 0, "bulk": 10, "nvls": 20}[algo], algo)
    for name, r in res.items():
        if not isinstance(r, dict) or "rel_err" not in r:
            continue
        assert r["rel_err"] < r["tol"], (name, r)
        assert r["replicas_identical"], (name, r)
        assert r["model_is_rounded_master"], (name, r)
        if r["norm_rel_err"] is not None:
            assert r["norm_rel_err"] < max(1e-5, 0.1 * r["tol"]), (name, r)
    assert res["loss_sync"] == res["loss_sync_expected"]
    for key in ("kat_full_size", "kat_full_size_sharded"):
        kat = res[key]
        assert kat["exact"] and kat["bucket_zeroed"] and kat["norm_rel_err"] < 1e-6, (key, kat)
    for name, r in res["stoke_api"].items():
        assert r["replicas_identical"] and r["buffers_identical"] and r["loss_identical_across_ranks"], (name, r)
        assert r["resume_bit_identical"], (name, r)
        assert r["opt_steps"] == 6 and r["sharded"] and r["buckets"] > 1 and r["overlap"], (name, r)
    if algo == "nvls" and res["caps"]["multicast"]:
        # the multimem flavour really ran on multicast-bound buckets (otherwise the call silently fell back to bulk)
        assert res["kat_full_size"]["mc"] and res["ddp_adam_bf16_clipnorm"]["mc"], res["caps"]
    inf = res["inf_skip"]
    assert inf["unchanged"] and inf["scale"] == 128.0 and inf["skipped"] == 1 and inf["steps"] == 0

# -*- coding: utf-8 -*-
"""TEST INFRASTRUCTURE ONLY -- generates ``tests/golden/*`` by running the UNMODIFIED reference in this container.

    python oracle/make_golden.py            # needs /root/reference (build container only)

Fixtures written (all small, committed):

  tests/golden/sampler_golden.json   reference ``BucketedDistributedSampler`` (/root/reference/stoke/data.py:111-516) over a
                                     grid of (N, buckets, bs, W, drop_last, overlap, shuffle, seed, epoch): per case the
                                     per-replica length, rank-0 head, sha256 over all replicas' int64 lists; small cases
                                     also carry the full lists.  Includes SURVEY.md Appendix B's four cases.
  tests/golden/cfg1_*.npz            BASELINE.json configs[0]: BasicNN (128-256-256-1) + BCEWithLogitsLoss + Adam, CPU,
                                     fp32, grad_accum=2, 50 optimizer steps through the reference ``Stoke`` object
                                     (``DistributedNullCPU + NullFP16 + BaseOptimizer``): initial weights, final weights,
                                     per-micro-step losses, counter trace; variants without clip / clip-by-norm /
                                     clip-by-value.
  tests/golden/reference_traces.json reference runs that the CPU tests replay against the port, the facade and the
                                     sampler oracle: the configuration of each run, its per-micro-step losses / EMA /
                                     counters, a sha256 over its final fp32 weights, and for 25 random sampler
                                     configurations each checked replica's length and sha256 (or the exception raised).

The recipe for the data is in ``stoke_b200/synthetic.py`` so the GPU-side tests can rebuild the identical inputs.
"""
import hashlib
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402
sys.path.insert(0, os.path.dirname(HERE))
from stoke_b200 import synthetic as workloads  # noqa: E402

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")


def sampler_cases():
    cases = [
        # SURVEY.md Appendix B
        dict(n=1000, buckets=4, bs=8, w=2, drop_last=False, overlap=False, shuffle=True, seed=0, epoch=0),
        dict(n=1003, buckets=4, bs=8, w=2, drop_last=True, overlap=True, shuffle=True, seed=0, epoch=3),
        dict(n=1000, buckets=4, bs=8, w=2, drop_last=False, overlap=False, shuffle=False, seed=0, epoch=0),
        dict(n=5000, buckets=5, bs=16, w=8, drop_last=False, overlap=False, shuffle=True, seed=7, epoch=1),
    ]
    grid = [
        (1001, 3, 8, 4), (1237, 4, 5, 3), (2048, 2, 16, 8), (3001, 7, 4, 2), (997, 1, 16, 4), (4099, 8, 8, 1),
        (1500, 3, 7, 5), (10007, 10, 32, 8), (1024, 4, 16, 2), (1025, 4, 16, 2), (1279, 4, 16, 2),
    ]
    for (n, b, bs, w) in grid:
        for drop_last, overlap in ((False, False), (True, False), (True, True)):
            for shuffle in (True, False):
                cases.append(dict(n=n, buckets=b, bs=bs, w=w, drop_last=drop_last, overlap=overlap,
                                  shuffle=shuffle, seed=n % 11, epoch=n % 5))
    cases.append(dict(n=100003, buckets=16, bs=32, w=8, drop_last=False, overlap=False, shuffle=True, seed=0, epoch=0))
    cases.append(dict(n=100003, buckets=16, bs=32, w=8, drop_last=True, overlap=True, shuffle=True, seed=3, epoch=2))
    return cases


def run_reference_sampler(stoke, case):
    n = case["n"]
    sorted_idx = workloads.sampler_sorted_idx(n).tolist()
    ds = list(range(n))
    out = []
    for r in range(case["w"]):
        with redirect_stdout(io.StringIO()):
            s = stoke.BucketedDistributedSampler(
                ds, buckets=case["buckets"], batch_size=case["bs"], sorted_idx=sorted_idx,
                backend=stoke.DistributedOptions.ddp, allow_bucket_overlap=case["overlap"],
                num_replicas=case["w"], rank=r, shuffle=case["shuffle"], seed=case["seed"],
                drop_last=case["drop_last"], info_rank=-1,
            )
        s.set_epoch(case["epoch"])
        out.append([int(v) for v in iter(s)])
    return out


def make_sampler(stoke):
    rows = []
    for case in sampler_cases():
        row = dict(case)
        try:
            lists = run_reference_sampler(stoke, case)
        except (ValueError, AssertionError) as e:
            row["raises"] = type(e).__name__
            rows.append(row)
            continue
        h = hashlib.sha256()
        for lst in lists:
            h.update(np.asarray(lst, dtype="<i8").tobytes())
        row["len_per_replica"] = len(lists[0])
        row["rank0_head"] = lists[0][:16]
        row["sha256"] = h.hexdigest()
        if case["n"] <= 1300:
            row["lists"] = lists
        rows.append(row)
    with open(os.path.join(GOLD, "sampler_golden.json"), "w") as f:
        json.dump({"torch": torch.__version__, "numpy": np.__version__, "cases": rows}, f)
    print(f"sampler: {len(rows)} cases ({sum('raises' in r for r in rows)} raising)")


def make_cfg1(stoke):
    variants = {
        "noclip": None,
        "clipnorm": stoke.ClipGradNormConfig(max_norm=0.05, norm_type=2.0),
        "clipvalue": stoke.ClipGradConfig(clip_value=0.002),
    }
    for name, clip in variants.items():
        model = workloads.basic_nn()
        init = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy().copy()
        opt = stoke.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=workloads.CFG1_ADAM)
        with redirect_stdout(io.StringIO()):
            s = stoke.Stoke(model=model, optimizer=opt, loss=torch.nn.BCEWithLogitsLoss(),
                            batch_size_per_device=workloads.CFG1_BATCH, grad_accum_steps=workloads.CFG1_ACCUM,
                            grad_clip=clip, gpu=False, verbose=False)
        losses, trace = [], []
        for x, y in workloads.cfg1_batches(workloads.CFG1_OPT_STEPS * workloads.CFG1_ACCUM):
            out = s.model(x)
            l = s.loss(out, y)
            losses.append(s.step_loss)
            s.backward(l)
            s.step()
            trace.append((s._grad_accum_counter, s._backward_steps, s._optimizer_steps))
        final = torch.cat([p.detach().reshape(-1) for p in s.model_access.parameters()]).numpy()
        np.savez(os.path.join(GOLD, f"cfg1_{name}.npz"), init=init, final=final,
                 losses=np.asarray(losses, dtype=np.float64), trace=np.asarray(trace, dtype=np.int64))
        print(f"cfg1/{name}: final |w|={np.linalg.norm(final):.6f} last loss={losses[-1]:.6f} trace tail={trace[-1]}")


def weights_sha256(params) -> str:
    flat = torch.cat([p.detach().reshape(-1) for p in params]).numpy()
    return hashlib.sha256(np.ascontiguousarray(flat, dtype="<f4").tobytes()).hexdigest()


def _trace_losses(ref_stoke, rec):
    """Runs ``ref_stoke`` over ``rec``'s batches and records its host-side bookkeeping after every micro-step."""
    steps = []
    for x, y in workloads.cfg1_batches(rec["batches"], seed=rec["batch_seed"]):
        l = ref_stoke.loss(ref_stoke.model(x), y)
        ref_stoke.backward(l)
        ref_stoke.step()
        steps.append({"step_loss": ref_stoke.step_loss, "ema_loss": ref_stoke.ema_loss, "agg_loss": ref_stoke._agg_loss,
                      "counters": [ref_stoke._grad_accum_counter, ref_stoke._backward_steps, ref_stoke._optimizer_steps]})
    rec["steps"] = steps
    rec["final_sha256"] = weights_sha256(ref_stoke.model_access.parameters())
    return rec


def trace_losses():
    """The list of loss callables of the ``multiple_losses`` run (BCE on the logits + MSE against the labels)."""
    return [torch.nn.BCEWithLogitsLoss(), lambda out, y: ((out - y) ** 2).mean()]


def make_traces(stoke):
    out = {}
    # SGD-momentum + clip-by-norm + grad_accum=3: a configuration the cfg1 fixtures do not cover
    rec = {"model_seed": 3, "kwargs": {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4}, "accum": 3, "max_norm": 0.1,
           "batches": 31, "batch_seed": 5}
    with redirect_stdout(io.StringIO()):
        s = stoke.Stoke(model=workloads.basic_nn(rec["model_seed"]),
                        optimizer=stoke.StokeOptimizer(optimizer=torch.optim.SGD, optimizer_kwargs=rec["kwargs"]),
                        loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32, grad_accum_steps=rec["accum"],
                        grad_clip=stoke.ClipGradNormConfig(max_norm=rec["max_norm"], norm_type=2.0), gpu=False, verbose=False)
    out["sgd_clipnorm_accum3"] = _trace_losses(s, rec)
    # Adam, grad_accum=3, non-default EMA weight
    rec = {"model_seed": 2, "accum": 3, "ema_weight": 0.3, "batches": 20, "batch_seed": 9}
    with redirect_stdout(io.StringIO()):
        s = stoke.Stoke(model=workloads.basic_nn(rec["model_seed"]),
                        optimizer=stoke.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=workloads.CFG1_ADAM),
                        loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32, grad_accum_steps=rec["accum"],
                        gpu=False, verbose=False, ema_weight=rec["ema_weight"])
    out["adam_accum3_ema03"] = _trace_losses(s, rec)
    # a list of two loss callables: per-loss values, sums and EMAs, retain_graph backward over the list
    rec = {"model_seed": 8, "accum": 2, "batches": 9, "batch_seed": 4}
    with redirect_stdout(io.StringIO()):
        s = stoke.Stoke(model=workloads.basic_nn(rec["model_seed"]),
                        optimizer=stoke.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=workloads.CFG1_ADAM),
                        loss=trace_losses(), batch_size_per_device=32, grad_accum_steps=rec["accum"], gpu=False,
                        verbose=False)
    out["multiple_losses"] = _trace_losses(s, rec)
    # BucketedDistributedSampler over random configurations, first and last replica of each
    rng = np.random.default_rng(123)
    cases = []
    for _ in range(25):
        w = int(rng.integers(1, 9))
        bs = int(rng.integers(2, 33))
        buckets = int(rng.integers(1, 9))
        n = int(rng.integers(max(100, 2 * bs * w) * buckets + 1, 6 * max(100, 2 * bs * w) * buckets))
        drop_last = bool(rng.integers(0, 2))
        overlap = bool(rng.integers(0, 2))
        shuffle = bool(rng.integers(0, 2))
        seed, epoch = int(rng.integers(0, 100)), int(rng.integers(0, 10))
        for r in sorted({0, w - 1}):
            case = dict(n=n, buckets=buckets, bs=bs, w=w, rank=r, drop_last=drop_last, overlap=overlap, shuffle=shuffle,
                        seed=seed, epoch=epoch)
            try:
                with redirect_stdout(io.StringIO()):
                    smp = stoke.BucketedDistributedSampler(
                        list(range(n)), buckets=buckets, batch_size=bs, sorted_idx=workloads.sampler_sorted_idx(n).tolist(),
                        backend=stoke.DistributedOptions.ddp, allow_bucket_overlap=overlap, num_replicas=w, rank=r,
                        shuffle=shuffle, seed=seed, drop_last=drop_last, info_rank=-1)
                smp.set_epoch(epoch)
                lst = [int(v) for v in iter(smp)]
            except (ValueError, AssertionError) as e:
                case["raises"] = type(e).__name__
            else:
                case["len"] = len(lst)
                case["sha256"] = hashlib.sha256(np.asarray(lst, dtype="<i8").tobytes()).hexdigest()
            cases.append(case)
    out["sampler_random"] = cases
    with open(os.path.join(GOLD, "reference_traces.json"), "w") as f:
        json.dump({"torch": torch.__version__, "numpy": np.__version__, **out}, f)
    print(f"traces: {len(cases)} sampler replicas ({sum('raises' in c for c in cases)} raising)")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    ref = ref_shim.import_reference()
    make_sampler(ref)
    make_cfg1(ref)
    make_traces(ref)

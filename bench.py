# -*- coding: utf-8 -*-
"""bench.py -- the hot path's headline benchmark (BASELINE.json: samples/sec, ResNet-50 synthetic, DDP-mode, bf16 mixed
precision, grad_clip=1.0), measured through the ``Stoke`` API.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--oss]
                    [--workload resnet50|bert|allreduce_sweep] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One step = ``out = s.model(x); l = s.loss(out, y); s.backward(l); s.step()`` on one synthetic batch per GPU.
Prints ONE JSON line on rank 0:
  value      samples/sec over all N GPUs with the batch already resident in HBM (device-timed, max over ranks)
  e2e        the same loop with the batch copied from pinned host memory every step and the loss read back to the host
  roofline   the dominant kernel of the engine -- the one with the largest mean launch time in the timed region: the fused
             optimizer step K2 at N = 1, the cross-rank kernels at N > 1 -- algorithmic bytes / duration measured live
             (CUDA events recorded inside the library on the launch stream; cross-rank K1 also by the device timer between
             its barriers), against MEASURED_PEAKS.json (hbm_gbs) or NVLink 5 nominal; every engine kernel is listed
             under ``kernels``
  parity_check (N > 1) full-size known-answer reduce for every K1 flavour, replicas bit-identical, one sharded (OSS) step
             against the unsharded result -- run before the timed region; the run fails on a mismatch
  cpu_baseline  the reference's own CPU path on a bounded sample (rank 0, N = 1)
``--impl reference`` times the reference's CPU implementation alone: the UNMODIFIED reference package when
``oracle/_ref`` holds it (``oracle/build_ref.py``; ``kind: "reference"``), else the pinned port (``kind: "port"``).
``--workload bert`` is BASELINE configs[3] (BERT-base, length-bucketed sampler), ``--workload allreduce_sweep`` configs[4].
``--dump-outputs DIR`` writes, on rank 0, what the last step of the timed resident loop returned to its caller, so that two
builds can be compared output for output (the inputs depend only on the arguments): ``output.npy`` (the model's output,
float32), ``loss.npy`` (the loss, float64) and ``params.npy`` (the updated model parameters in registration order, float32;
a fixed sample of DUMP_PARAMS of them, drawn with seed 0, when there are more).  A dump run makes cuDNN use deterministic
algorithms instead of autotuning, so that repeating it reproduces the dump; take timings from runs without the flag.  On
one B200 two resnet50 dumps agreed bit for bit; two bert dumps did not (its attention backward is not deterministic):
with ``--steps 5 --warmup 3`` their outputs differed by 1.3e-2 and their parameters by 5e-4 in relative L2.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "samples/sec"
WORKLOAD = "resnet50_synthetic_3x224x224_ddp_bf16_adam_clipnorm1.0"
ADAM = {"lr": 1e-3}
CPU_SAMPLE_BATCH = 16
RESNET50_PARAMS = 25_557_032
DUMP_PARAMS = 1 << 22
DUMP_MAX_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (128 for resnet50, 32 for bert)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="resnet50", choices=["resnet50", "bert", "allreduce_sweep"])
    ap.add_argument("--oss", action="store_true", help="configs[2]: fairscale_oss=True (user-visible sharded optimizer)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the N > 1 parity check (profiling runs)")
    ap.add_argument("--ncu-step", action="store_true",
                    help="profiling helper: warm up, then run ONE step between cudaProfilerStart/Stop and exit "
                         "(use with ncu --profile-from-start off); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (resnet50 and bert workloads)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload == "allreduce_sweep"):
        ap.error("--dump-outputs needs --impl b200 and the resnet50 or bert workload")
    return args


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_arm(steps: int, warmup: int, batch: int = CPU_SAMPLE_BATCH):
    """The reference's CPU path on ResNet-50 fp32 (its only runnable configuration: gpu=False, stoke/status.py:215-222):
    samples/sec on the host cores.  Runs exactly ``warmup`` + ``steps`` steps and reports what it ran."""
    import torch

    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to the box's cores (physical, not hyper-threads)
    threads = max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(threads)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shim
    from stoke_b200 import synthetic

    model = synthetic.resnet50()
    kind = "port"
    if ref_shim.reference_available():
        import io
        from contextlib import redirect_stdout

        stoke = ref_shim.import_reference()   # the UNMODIFIED reference package (oracle/_ref or /root/reference)
        with redirect_stdout(io.StringIO()):
            s = stoke.Stoke(model=model, optimizer=stoke.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=ADAM),
                            loss=torch.nn.CrossEntropyLoss(), batch_size_per_device=batch, grad_accum_steps=1,
                            grad_clip=stoke.ClipGradNormConfig(max_norm=1.0, norm_type=2.0), gpu=False, verbose=False)
        kind = "reference"
    else:
        from stoke_port import StokePortCPU

        s = StokePortCPU(model, torch.optim.Adam, ADAM, torch.nn.CrossEntropyLoss(), grad_accum_steps=1,
                         clip=("norm", 1.0, 2.0))
    x, y = synthetic.resnet50_batch(batch)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = s.loss(s.model(x), y)
        s.backward(loss)
        s.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": batch * len(times) / total, "unit": METRIC, "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"resnet50 fp32 (the reference's CPU path), batch {batch}, {len(times)} timed steps after {warmup} "
                      f"warm-up, mean {total / len(times) * 1e3:.0f} / median {statistics.median(times) * 1e3:.0f} ms/step, "
                      f"{torch.get_num_threads()} threads of os.cpu_count()={os.cpu_count()}",
            "ms_per_step": total / len(times) * 1e3, "steps": len(times), "warmup": warmup}


class ClockSampler:
    """nvidia-smi sampled in the background during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
def parity_check(eng, rank, world):
    """Cross-rank correctness on THIS box before anything is timed (N > 1): exact expected values, no oracle needed.

      kat_<flavour>   ResNet-50-sized bf16 bucket, rank r holds (r+1) * pattern (small integers: every partial sum is exact
                      in bf16 and fp32): the all-reduced fp32 main grads must EQUAL pattern * (W+1)/2 on every rank, the
                      local bucket must be zero afterwards and the fused L2 norm must match the closed form; for every K1
                      flavour this box supports (register-staged, bulk-async, multimem/NVLS)
      sharded_kat     the same through the reduce-scatter route (what DDP mode runs): this rank's shards of every bucket
      oss_vs_unsharded  three Adam steps with clip-by-norm from per-rank seeded gradients: sharded route (reduce-scatter +
                      sharded fused step + in-kernel parameter all-gather) against the all-reduce route -- bit-identical
                      master weights and model copies; replicas bit-identical across ranks
    """
    import torch
    import torch.distributed as dist

    from stoke_b200 import _lib
    from stoke_b200.engine import ClipSpec
    from stoke_b200.optim import B200FusedOptimizer

    dev = torch.device("cuda", eng.device)
    res, ok = {}, True

    class Big(torch.nn.Module):
        def __init__(self, n, pieces=7):
            super().__init__()
            sizes = [n // pieces] * (pieces - 1)
            sizes.append(n - sum(sizes))
            self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.zeros(k)) for k in sizes])

    def all_true(flag: bool) -> bool:
        t = torch.tensor([1.0 if flag else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() == 1.0)

    def same_on_all_ranks(x: torch.Tensor) -> bool:
        ref = x.clone()
        dist.broadcast(ref, src=0)
        return all_true(bool(torch.equal(ref, x)))

    clip = ClipSpec(_lib.CLIP_NORM, max_norm=1.0, norm_type=2.0)
    flavours = ["ldg", "bulk"]
    for route in ("allreduce", "sharded"):
        net = Big(RESNET50_PARAMS).to(dev)
        opt = B200FusedOptimizer(net, torch.optim.SGD, {"lr": 0.0}, engine=eng, clip=clip, lp_dtype=torch.bfloat16,
                                 route=route, bucket_mb=8.0)
        path = opt.path
        if route == "allreduce" and path.G.mc_ptr and path.MAIN.mc_ptr:
            flavours.append("nvls")
        base = ((torch.arange(path.n, device=dev) % 7) - 3).float()
        expect = base * (world + 1) / 2.0
        exp_norm = float(expect.double().pow(2).sum().sqrt())
        for fl in (flavours if route == "allreduce" else ["bulk"]):
            eng.set_k1_algo(fl)
            path.g_flat.copy_((base * (rank + 1)).to(torch.bfloat16))
            path.after_backward(sync=True, unscale=False)
            if route == "allreduce":
                exact = bool(torch.equal(path.main_flat, expect))
            else:
                exact = all(bool(torch.equal(path.main_flat[l0: l0 + (g1 - g0)], expect[g0:g1])) for g0, g1, l0, _ in path.segs)
            norm = eng.scaler_get(path.state_id).grad_norm
            zeroed = float(path.g_flat.float().abs().max()) == 0.0
            eng.step_epilogue()
            row = {"exact": all_true(exact), "bucket_zeroed": all_true(zeroed), "norm_rel_err": abs(norm - exp_norm) / exp_norm,
                   "buckets": len(path.buckets)}
            good = row["exact"] and row["bucket_zeroed"] and row["norm_rel_err"] < 1e-6
            if fl == "nvls" and not good:
                # the multimem flavour is opt-in (never on this benchmark's training path): report, do not fail the run
                row["optional_flavour_failed"] = True
            else:
                ok &= good
            res[("kat_" + fl) if route == "allreduce" else "sharded_kat"] = row
        eng.set_k1_algo("bulk")
        opt.close()
        del opt, path, net
    # sharded vs unsharded optimizer steps
    outs = {}
    for route in ("allreduce", "sharded"):
        torch.manual_seed(4321)
        net = Big(2_000_003 * 2).to(dev)
        with torch.no_grad():
            for p in net.parameters():
                p.copy_(torch.randn_like(p) * 0.05)
        opt = B200FusedOptimizer(net, torch.optim.Adam, {"lr": 1e-3}, engine=eng, clip=clip, lp_dtype=torch.bfloat16,
                                 route=route, bucket_mb=2.0)
        path = opt.path
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        for _ in range(3):
            path.g_flat.copy_((torch.randn(path.n, device=dev, generator=gen) * 1e-2).to(torch.bfloat16))
            path.after_backward(sync=True, unscale=False)
            opt.step()
        outs[route] = (path.gather_master().clone(), path.p_flat.clone(), len(path.buckets))
        res.setdefault("replicas_identical", True)
        res["replicas_identical"] &= same_on_all_ranks(path.p_flat.float())
        opt.close()
        del opt, path, net
    same = bool(torch.equal(outs["allreduce"][0], outs["sharded"][0])) and bool(torch.equal(outs["allreduce"][1], outs["sharded"][1]))
    res["oss_vs_unsharded"] = {"bit_identical": all_true(same), "buckets": outs["sharded"][2]}
    ok &= res["oss_vs_unsharded"]["bit_identical"] and res["replicas_identical"]
    eng.comm_check()
    res["ok"] = bool(ok)
    res["flavours"] = flavours
    return res


# ---------------------------------------------------------------------------------------------------------------------
def dump_outputs(directory, s, last_step):
    """Writes the model output and loss of the last resident step and the model parameters after it (see --dump-outputs)."""
    import numpy as np
    import torch

    params = torch.cat([p.detach().reshape(-1).float() for p in s.model_access.parameters()])
    if params.numel() > DUMP_PARAMS:
        pick = np.sort(np.random.default_rng(0).choice(params.numel(), DUMP_PARAMS, replace=False))
        params = params[torch.from_numpy(pick).to(params.device)]
    arrays = {"output": last_step["output"].detach().float().cpu().numpy(),
              "loss": last_step["loss"].detach().double().reshape(1).cpu().numpy(),
              "params": params.cpu().numpy()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES} byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def build_workload(args, sb, torch, local_rank, world, rank):
    """(stoke object, resident step fn, e2e step fn, per-GPU batch, h2d bytes per step, workload name, extras, last_step).
    ``last_step`` holds the model output and loss of the most recent resident step (references only: no copy, no sync)."""
    from stoke_b200 import synthetic
    from stoke_b200.data import DevicePrefetcher

    dev = torch.device("cuda", local_rank)
    configs = [sb.DDPConfig(local_rank=local_rank)] if world > 1 else None
    common = dict(gpu=True, fp16="bf16", distributed="ddp" if world > 1 else None,
                  fairscale_oss=bool(args.oss and world > 1), configs=configs, verbose=False,
                  grad_clip=sb.ClipGradNormConfig(max_norm=1.0, norm_type=2.0))
    if args.workload == "resnet50":
        batch = args.batch or 128
        model = synthetic.resnet50().to(memory_format=torch.channels_last)
        s = sb.Stoke(model=model, optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=ADAM),
                     loss=torch.nn.CrossEntropyLoss(), batch_size_per_device=batch, **common)
        x_host, y_host = synthetic.resnet50_batch(batch, rank)
        x_host = x_host.contiguous(memory_format=torch.channels_last).pin_memory()
        y_host = y_host.pin_memory()
        x_dev, y_dev = x_host.to(dev), y_host.to(dev)
        last_step = {}

        def step_resident():
            last_step["output"] = s.model(x_dev)
            last_step["loss"] = s.loss(last_step["output"], y_dev)
            s.backward(last_step["loss"])
            s.step()

        def host_batches():
            while True:
                yield x_host, y_host   # the same pinned batch every step: the H2D copy is real, the data is synthetic

        feed = iter(DevicePrefetcher(host_batches()))  # what StokeDataLoader uses: batch i+1 is copied while i computes

        def step_e2e():
            # every step's synced loss is read back on the host exactly once, one step behind (the value landed in pinned
            # memory during the previous step; reading it here does not drain the queue of the step being launched)
            last = s.step_loss
            x, y = next(feed)                   # 77 MB host -> device copy per step, inside the timed region
            s.backward(s.loss(s.model(x), y))
            s.step()
            return last

        h2d = x_host.numel() * x_host.element_size() + y_host.numel() * y_host.element_size()
        return s, step_resident, step_e2e, batch, h2d, WORKLOAD + ("_oss" if common["fairscale_oss"] else ""), {}, last_step

    # ---- configs[3]: BERT-base, length-bucketed batches from BucketedDistributedSampler ----
    import numpy as np
    from transformers import BertConfig, BertForSequenceClassification

    batch = args.batch or 32
    torch.manual_seed(0)
    model = BertForSequenceClassification(BertConfig())
    s = sb.Stoke(model=model, optimizer=sb.StokeOptimizer(optimizer=torch.optim.AdamW, optimizer_kwargs={"lr": 1e-4}),
                 loss=torch.nn.CrossEntropyLoss(), batch_size_per_device=batch, **common)
    n_items = 200_003
    lens = synthetic.sampler_lengths(n_items, 16, 513)
    t0 = time.perf_counter()
    sorted_idx = sb.argsort_lengths(lens)
    smp = sb.BucketedDistributedSampler(range(n_items), buckets=16, batch_size=batch, sorted_idx=sorted_idx,
                                        num_replicas=world, rank=rank if world > 1 else 0, shuffle=True, seed=0, info_rank=-1)
    idx = smp.indices_tensor().cpu().numpy()
    torch.cuda.synchronize()
    sampler_ms = (time.perf_counter() - t0) * 1e3
    rng = np.random.default_rng(1234 + rank)
    # a fixed pool of pre-built pinned host batches (built OFF the timed path): the timed loop only copies and computes
    pool = []
    for b in range(min(len(idx) // batch, 24)):
        ii = idx[b * batch:(b + 1) * batch]
        ll = lens[ii]
        L = int((ll.max() + 63) // 64 * 64)
        ids = torch.from_numpy(rng.integers(0, 30522, size=(batch, L))).pin_memory()
        mask = torch.from_numpy((np.arange(L)[None, :] < ll[:, None]).astype(np.int64)).pin_memory()
        y = torch.from_numpy(rng.integers(0, 2, size=(batch,))).pin_memory()
        pool.append((ids, mask, y))
    pool.sort(key=lambda b: b[0].shape[1])
    # one batch per distinct padded length first, so that a short warm-up visits every shape
    firsts, rest, seen = [], [], set()
    for b in pool:
        (firsts if b[0].shape[1] not in seen else rest).append(b)
        seen.add(b[0].shape[1])
    pool = firsts + rest
    resident = [tuple(t.to(dev) for t in b) for b in pool]
    counter = {"i": 0}
    last_step = {}

    def step_resident():
        ids, mask, y = resident[counter["i"] % len(resident)]
        counter["i"] += 1
        last_step["output"] = s.model(input_ids=ids, attention_mask=mask).logits
        last_step["loss"] = s.loss(last_step["output"], y)
        s.backward(last_step["loss"])
        s.step()

    def host_batches():
        i = 0
        while True:
            yield pool[i % len(pool)]
            i += 1

    feed = iter(DevicePrefetcher(host_batches()))

    def step_e2e():
        last = s.step_loss                      # the previous step's synced loss (see the resnet50 workload)
        ids, mask, y = next(feed)
        s.backward(s.loss(s.model(input_ids=ids, attention_mask=mask).logits, y))
        s.step()
        return last

    h2d = int(sum(sum(t.numel() * t.element_size() for t in b) for b in pool) / len(pool))
    extras = {"_distinct_shapes": len(seen), "sampler_setup_ms": sampler_ms, "dataset_items": n_items, "buckets": 16,
              "mean_padded_len": float(sum(b[0].shape[1] for b in pool) / len(pool))}
    return s, step_resident, step_e2e, batch, h2d, "bert_base_synthetic_bucketed_sampler_ddp_bf16_adamw_clipnorm1.0", extras, \
        last_step


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        base = cpu_reference_arm(max(1, args.steps), max(0, args.warmup))
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": METRIC, "n_gpus": args.gpus,
                "steps": base["steps"], "warmup": base["warmup"], "ms_per_step": base["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "note": "the reference's own CPU call path (gpu=False: the only configuration "
                           "the reference can run without CUDA), fp32, bounded per-step sample", "per_step_batch": CPU_SAMPLE_BATCH},
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if args.workload == "allreduce_sweep":
        if world < 2:
            if rank == 0:
                print(json.dumps({"metric": "fused grad all-reduce bus bandwidth", "unavailable":
                                  "configs[4] needs at least 2 GPUs: launch with torch.distributed.run --nproc-per-node N"}))
            return
        import bench_allreduce

        bench_allreduce.main(["--json-line"])
        return

    import torch

    import stoke_b200 as sb

    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local_rank)
    torch.backends.cudnn.benchmark = True
    if args.dump_outputs:
        # the autotuner's choice and cuDNN's non-deterministic algorithms change the last bits from run to run, and Adam
        # on the repeated batch amplifies them into different weights: a dump run uses fixed, deterministic algorithms
        torch.backends.cudnn.benchmark = False
        torch.backends.cudnn.deterministic = True
    dev = torch.device("cuda", local_rank)

    s, step_resident, step_e2e, batch, h2d_bytes, workload, extras, last_step = build_workload(args, sb, torch, local_rank,
                                                                                               world, rank)
    eng = s.engine
    path = s.optimizer.path

    parity = None
    if world > 1 and not args.no_parity and not args.ncu_step:
        parity = parity_check(eng, rank, world)
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"error": "parity_check failed", "parity_check": parity}))
            raise SystemExit(3)

    def fence():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        fence()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        fence()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    warm = max(3, args.warmup)
    if args.workload == "bert":
        warm = max(warm, extras.pop("_distinct_shapes", 0) + 2)   # every padded length once: cuBLASLt / SDPA plans are per shape
    for _ in range(warm):
        step_resident()
    if args.ncu_step:
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return

    # ---- timed region 1: inputs resident; kernel events recorded live for the roofline ----
    eng.profile(True)  # CUDA events recorded inside the library, immediately around each K1 / K2 / norm launch
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = eng.launches
    ms_total = timed(step_resident, args.steps)
    launches = eng.launches - launches0
    clock_info = clocks.stop() if rank == 0 else None
    ev = {}
    for key, kind in (("k1", 0), ("k2", 1), ("acc", 2), ("norm", 3)):
        tot, cnt = eng.profile_read(kind)
        ev[key] = (tot, cnt)
    k1_dev_ms, k1_dev_n, k1_zero_ms = eng.profile_read_k1_device()
    k2_dev_ms, k2_dev_n = eng.profile_read_k2_device()
    eng.profile(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, s, last_step)

    # ---- timed region 2: end to end (H2D of the batch + D2H of the loss inside the timed region) ----
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    if rank != 0:
        return
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    n, n_local = path.n, path.n_local
    steps = args.steps
    per_step = lambda key: ev[key][0] / steps  # noqa: E731 -- total launch time of this kernel kind per step
    per_launch = lambda key: ev[key][0] / max(ev[key][1], 1)  # noqa: E731
    traffic_tab = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_r02.json")) as f:
            traffic_tab = json.load(f)
    except (OSError, ValueError):
        pass

    def traffic_of(kernel_key):
        row = traffic_tab.get(kernel_key)
        return row.get("dram_bytes_per_launch") if row and row.get("n_elements") == n else None

    kernels = {}
    nv = lambda w: (w - 1) / w  # noqa: E731
    if world == 1:
        # K2, raw-bucket route: g read 2 + p,m,v read 12 + p,m,v write 12 + bf16 param write 2 + bucket zeroing 2 = 30 B/elem
        kernels["k2"] = {"kernel": "k_optim_step (fused Adam + clip + bf16 param write, reads and zeroes the raw bucket)",
                         "bound": "hbm", "bytes_per_launch": n * 30, "ms_per_launch": per_launch("k2"), "peak": hbm_peak,
                         "traffic": traffic_of("k_optim_step_raw")}
        if ev["norm"][1]:
            kernels["k1"] = {"kernel": "k_grad_norm (norm + inf pass over the raw bf16 bucket: the W=1 form of K1)",
                             "bound": "hbm", "bytes_per_launch": n * 2, "ms_per_launch": per_launch("norm"), "peak": hbm_peak,
                             "traffic": traffic_of("k_grad_norm")}
    else:
        wire_in = 2 if path.model_dtype != torch.float32 else 4
        if path.sharded:
            k1_bytes = nv(world) * n * wire_in                # reduce-scatter: peers' shards in
            k2_bytes = nv(world) * n * wire_in                # parameter all-gather: updated shard out
            k2_name = "k_optim_step (sharded fused step + in-kernel parameter all-gather, 32-byte peer stores)"
            k2_bound, k2_peak = "nvlink", 900.0
        else:
            k1_bytes = nv(world) * n * (wire_in + 4)
            k2_bytes, k2_name, k2_bound, k2_peak = n * 30, "k_optim_step (local fused step on fp32 main grads)", "hbm", hbm_peak
        nb = max(len(path.buckets), 1)
        k1_launches = max(k1_dev_n, 1)
        kernels["k1"] = {"kernel": f"k_grad_reduce ({'reduce-scatter' if path.sharded else 'all-reduce'}, {nb} bucket(s) per step, "
                                   "launched from autograd hooks)", "bound": "nvlink",
                         "bytes_per_launch": k1_bytes / nb, "ms_per_launch": k1_dev_ms / k1_launches,
                         "ms_per_launch_events": per_launch("k1"), "ms_zero_tail": k1_zero_ms / k1_launches, "peak": 900.0,
                         "timer": "device timer between K1's start and end barriers (the NVLink phase); events also listed",
                         "traffic": None}
        kernels["k2"] = {"kernel": k2_name, "bound": k2_bound, "bytes_per_launch": k2_bytes,
                         "ms_per_launch": (k2_dev_ms / k2_dev_n) if (path.sharded and k2_dev_n) else per_launch("k2"),
                         "ms_per_launch_events": per_launch("k2"), "peak": k2_peak, "traffic": None}
        if path.sharded:
            kernels["k2"]["timer"] = "device timer between the sharded step's barriers (local update + parameter all-gather); " \
                                     "events (which include the wait for the slowest rank to arrive) also listed"
    for k in kernels.values():
        k["achieved"] = k["bytes_per_launch"] / (k["ms_per_launch"] * 1e-3) / 1e9 if k["ms_per_launch"] else None
        k["unit"] = "GB/s"
        k["frac"] = k["achieved"] / k["peak"] if k["achieved"] else None
        k["peak_source"] = hbm_src if k["bound"] == "hbm" else "NVLink 5 nominal per direction (measured peer copy 770 GB/s)"
    step_ms = {"k1": (k1_dev_ms / steps) if world > 1 else per_step("norm"),
               "k2": (k2_dev_ms / steps) if (world > 1 and path.sharded and k2_dev_n) else per_step("k2")}
    dominant = max(kernels, key=lambda k: step_ms.get(k, 0.0))
    roofline = dict(kernels[dominant])
    roofline["dominant_by"] = "largest share of the step among the engine's kernels (ms per step: " + \
        ", ".join(f"{k} {step_ms[k]:.4f}" for k in kernels) + ")"
    roofline["kernels"] = kernels
    # the whole engine against HBM at N = 1: algorithmic bytes of all its kernels / their summed time
    if world == 1:
        tot_b = sum(k["bytes_per_launch"] for k in kernels.values())
        tot_ms = sum(k["ms_per_launch"] for k in kernels.values())
        roofline["engine"] = {"bytes_per_step": tot_b, "ms_per_step": tot_ms, "achieved": tot_b / (tot_ms * 1e-3) / 1e9,
                              "frac": tot_b / (tot_ms * 1e-3) / 1e9 / hbm_peak,
                              "note": "norm pass + fused step = 32 B/element per optimizer step (round 1: 8 + 30)"}
    samples = batch * world * args.steps
    line = {"metric": METRIC, "value": samples / (ms_total * 1e-3), "unit": METRIC, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict({"workload": workload, "per_gpu_batch": batch,
                            "global_batch": batch * world, "parallelism": f"dp{world}", "params": n, "route": path.route,
                            "grad_buckets": len(path.buckets), "mem_mode": "vmm" if eng.mem_mode == 1 else "ipc",
                            "multicast_bound": bool(path.G.mc_ptr),
                            "l2": "per-step working set (activations, 0.9 GB of optimizer state) exceeds the 126 MB L2; no flush"},
                           **extras),
            "e2e": {"value": samples / (ms_e2e * 1e-3), "unit": METRIC, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 8, "ms_per_step": ms_e2e / args.steps,
                    "note": "batch copied from pinned host memory by the prefetcher every step; the synced loss of step i is written "
                            "to pinned host memory by the loss kernel and read by the host while step i+1 is being launched"},
            "gpu_launches": launches, "clocks": clock_info, "roofline": roofline}
    if parity is not None:
        line["parity_check"] = parity
    if world == 1 and not args.no_cpu_baseline:
        base = cpu_reference_arm(12, 3)
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line))


if __name__ == "__main__":
    main()

# -*- coding: utf-8 -*-
"""BASELINE.json configs[4]: gradient all-reduce bandwidth sweep, 64 KB - 1 GB bf16 buckets, at W = 2/4/8.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W --master-addr 127.0.0.1 --master-port P \
        bench_allreduce.py [--max-mb 1024] [--out gpurun_out/allreduce_W.json]

Per size, device-timed (CUDA events on the launch stream, 10 warm-up + 50 timed back-to-back launches, max over ranks):

  ours_*      default flavour of K1 (bulk-async staging); ours_ldg_*: the register-staged flavour, for comparison
  ours_bf16   K1 fused all-reduce, bf16 in -> bf16 out  (+ fused 1/W scale, inf test, sum-of-squares, cross-rank norm
              exchange): same wire bytes as NCCL, busbw = 2 (W-1)/W S / t
  ours_fp32   K1 as the training path uses it: bf16 in -> fp32 main grads out (b_out = 4): busbw = (W-1)/W n (2+4) / t
  nccl        torch.distributed.all_reduce on the same bf16 buffer (the incumbent the reference's DDP path calls)
  nccl_ddp    all_reduce + cast to fp32 + _amp_foreach_non_finite_check_and_unscale_ + _foreach_norm (what the reference runs per bucket:
              stoke/extensions.py:207-215, stoke/fp16.py:180-183, 233)
  symm_*      torch symmetric-memory two_shot / multimem all-reduce where the build exposes them

Roofline: NVLink 5, 900 GB/s nominal per direction per GPU; measured peer copy on this pool 770 GB/s
(/opt/skills/guides/B200_PROFILING.md).
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def time_op(fn, warmup=10, iters=50):
    for _ in range(warmup):
        fn()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def study(args, eng, rank, world, G, O16, O32, have_nvls):
    """Grid-size studies on this box (each cell: 10 warm-up + 50 timed launches, CUDA events, max over ranks)."""
    from stoke_b200 import _lib

    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.current_stream().cuda_stream
    gp, o16, o32 = _lib.ptr_array(G.peer_ptrs()), _lib.ptr_array(O16.peer_ptrs()), _lib.ptr_array(O32.peer_ptrs())
    out = {"world": world, "nvls_grid": [], "reduce_scatter": [], "allreduce_grid": []}

    def launch(mode, n, outp, odt):
        rc = lib.stk_grad_reduce(ctx, mode, gp, _lib.BF16, None, outp, odt, n, 1.0 / world, _lib.NORM_L2, 2.0, _lib.RF_FINAL, stream)
        if rc != 0:
            _lib.check(rc, ctx)

    # (a) multimem all-reduce (bf16 -> bf16) vs grid
    if have_nvls:
        eng.set_k1_algo("nvls")
        for S in (1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20):
            if S > args.max_mb << 20:
                continue
            for cap in (8, 16, 32, 64, 96, 148):
                eng.option_set(_lib.OPT_NVLS_MAX_BLOCKS, cap)
                t = time_op(lambda: launch(_lib.REDUCE_ALL, S // 2, o16, _lib.BF16))
                out["nvls_grid"].append({"bytes": S, "blocks": cap, "us": t * 1e3, "busbw": 2 * (world - 1) / world * S / (t * 1e-3) / 1e9})
                if rank == 0:
                    print(json.dumps(out["nvls_grid"][-1]), flush=True)
        eng.option_set(_lib.OPT_NVLS_MAX_BLOCKS, 0)
    # (b) reduce-scatter of a ResNet-50-sized bf16 bucket (the in-step K1 of the sharded route) vs flavour and grid
    n = 25_557_040
    for algo in ("bulk", "ldg") + (("nvls",) if have_nvls else ()):
        eng.set_k1_algo(algo)
        for cap in (148, 128, 96, 64, 32):
            eng.option_set(_lib.OPT_K1_MAX_BLOCKS, cap if cap < 148 else 0)
            t = time_op(lambda: launch(_lib.REDUCE_SCATTER, n, o32, _lib.F32))
            row = {"algo": algo, "blocks": cap, "us": t * 1e3, "wire_gbs": (world - 1) / world * n * 2 / (t * 1e-3) / 1e9}
            out["reduce_scatter"].append(row)
            if rank == 0:
                print(json.dumps(row), flush=True)
    # (c) bulk all-reduce (bf16 -> bf16) at 64 MiB vs grid
    eng.set_k1_algo("bulk")
    for cap in (148, 96, 64):
        eng.option_set(_lib.OPT_K1_MAX_BLOCKS, cap if cap < 148 else 0)
        S = 64 << 20
        t = time_op(lambda: launch(_lib.REDUCE_ALL, S // 2, o16, _lib.BF16))
        out["allreduce_grid"].append({"bytes": S, "blocks": cap, "us": t * 1e3, "busbw": 2 * (world - 1) / world * S / (t * 1e-3) / 1e9})
    eng.option_set(_lib.OPT_K1_MAX_BLOCKS, 0)
    eng.comm_check()
    if rank == 0 and args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-mb", type=int, default=1024)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-baselines", action="store_true", help="skip NCCL / symmetric-memory rows")
    ap.add_argument("--study", action="store_true",
                    help="tuning study instead of the sweep: multimem flavour vs grid size, reduce-scatter of a ResNet-50-sized "
                         "bucket vs flavour and grid size (device-timed); writes --out")
    ap.add_argument("--json-line", action="store_true", help="print ONE bench.py-shaped JSON line (bench.py --workload allreduce_sweep)")
    args = ap.parse_args(argv)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from stoke_b200 import _lib
    from stoke_b200.engine import get_engine

    eng = get_engine(local, rank, world)
    sizes = [s for s in (64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20, 1 << 30)
             if s <= args.max_mb << 20]
    n_max = max(sizes) // 2
    G = eng.alloc(n_max * 2, multicast=True)
    O16 = eng.alloc(n_max * 2, multicast=True)
    O32 = eng.alloc(n_max * 4, multicast=True)
    have_nvls = bool(G.mc_ptr and O16.mc_ptr and O32.mc_ptr)
    g = G.tensor(torch.bfloat16, n_max)
    torch.manual_seed(2000 + rank)
    g.copy_(torch.randn(n_max, device="cuda") * 1e-3)

    symm = None
    try:
        import torch.distributed._symmetric_memory as sm

        t_sym = sm.empty(n_max, dtype=torch.bfloat16, device="cuda")
        sm.rendezvous(t_sym, dist.group.WORLD.group_name)
        t_sym.zero_()
        symm = (sm, t_sym, dist.group.WORLD.group_name)
    except Exception as e:  # noqa: BLE001
        if rank == 0:
            print(f"symm_mem unavailable: {type(e).__name__}: {e}", file=sys.stderr)

    if args.study:
        study(args, eng, rank, world, G, O16, O32, have_nvls)
        dist.barrier()
        dist.destroy_process_group()
        return

    rows = []
    for S in sizes:
        n = S // 2
        row = {"bytes": S, "world": world}

        # the C ABI called the way a C host would: pointer tables built once, no per-launch Python marshalling (at the small
        # sizes the launch rate is host-bound otherwise)
        gp = _lib.ptr_array(G.peer_ptrs())
        outs = {torch.bfloat16: _lib.ptr_array(O16.peer_ptrs()), torch.float32: _lib.ptr_array(O32.peer_ptrs())}
        dts = {torch.bfloat16: _lib.BF16, torch.float32: _lib.F32}
        stream = torch.cuda.current_stream().cuda_stream
        lib, ctx = eng.lib, eng.ctx

        def ours(out_buf, out_dtype):
            rc = lib.stk_grad_reduce(ctx, _lib.REDUCE_ALL, gp, _lib.BF16, None, outs[out_dtype], dts[out_dtype], n, 1.0 / world,
                                     _lib.NORM_L2, 2.0, _lib.RF_FINAL, stream)
            if rc != 0:
                _lib.check(rc, ctx)
            eng.launches += 1

        t = time_op(lambda: ours(O16, torch.bfloat16))
        row["ours_bf16_us"] = t * 1e3
        row["ours_bf16_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
        t = time_op(lambda: ours(O32, torch.float32))
        row["ours_fp32_us"] = t * 1e3
        row["ours_fp32_busbw"] = (world - 1) / world * n * 6 / (t * 1e-3) / 1e9

        eng.set_k1_algo("ldg")
        t = time_op(lambda: ours(O16, torch.bfloat16))
        row["ours_ldg_bf16_us"] = t * 1e3
        row["ours_ldg_bf16_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
        t = time_op(lambda: ours(O32, torch.float32))
        row["ours_ldg_fp32_us"] = t * 1e3
        row["ours_ldg_fp32_busbw"] = (world - 1) / world * n * 6 / (t * 1e-3) / 1e9
        eng.set_k1_algo("bulk")
        if have_nvls:
            # multimem flavour: the NVSwitch reduces (multimem.ld_reduce) and replicates (multimem.st)
            eng.set_k1_algo("nvls")
            t = time_op(lambda: ours(O16, torch.bfloat16))
            row["ours_nvls_bf16_us"] = t * 1e3
            row["ours_nvls_bf16_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
            t = time_op(lambda: ours(O32, torch.float32))
            row["ours_nvls_fp32_us"] = t * 1e3
            row["ours_nvls_fp32_busbw"] = (world - 1) / world * n * 6 / (t * 1e-3) / 1e9
            eng.set_k1_algo("bulk")
        if args.no_baselines:
            rows.append(row)
            if rank == 0:
                print(json.dumps(row), flush=True)
            continue
        buf = torch.zeros(n, dtype=torch.bfloat16, device="cuda")
        t = time_op(lambda: dist.all_reduce(buf))
        row["nccl_us"] = t * 1e3
        row["nccl_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
        found_inf = torch.zeros(1, device="cuda")
        inv = torch.ones(1, device="cuda")

        def ddp_like():
            dist.all_reduce(buf)
            f32 = buf.float()  # bf16 grads -> fp32 (the unscale kernel has no bf16 build; the reference's grads are fp32)
            torch._amp_foreach_non_finite_check_and_unscale_([f32], found_inf, inv)
            torch._foreach_norm([f32], 2.0)

        t = time_op(ddp_like)
        row["nccl_ddp_us"] = t * 1e3
        row["nccl_ddp_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
        if symm is not None:
            sm, t_sym, gname = symm
            view = t_sym[:n]
            for name, op in (("symm_two_shot", "two_shot_all_reduce_"), ("symm_multimem", "multimem_all_reduce_"),
                             ("symm_one_shot", "one_shot_all_reduce")):
                if name == "symm_one_shot" and S > (4 << 20):
                    continue
                try:
                    fn = getattr(torch.ops.symm_mem, op)
                    t = time_op(lambda: fn(view, "sum", gname))
                    row[name + "_us"] = t * 1e3
                    row[name + "_busbw"] = 2 * (world - 1) / world * S / (t * 1e-3) / 1e9
                except Exception as e:  # noqa: BLE001
                    row[name + "_error"] = f"{type(e).__name__}: {str(e)[:120]}"
        del buf
        eng.comm_check()
        rows.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
    # correctness spot check of the fused kernel on the last size: all ranks hold the same reduced values
    n = sizes[-1] // 2
    eng.grad_reduce(_lib.REDUCE_ALL, G.peer_ptrs(), torch.bfloat16, None, O32.peer_ptrs(), torch.float32, n, 1.0 / world,
                    _lib.NORM_L2, 2.0, _lib.RF_FINAL)
    mine = O32.tensor(torch.float32, n)[: 1 << 20].clone()
    ref = g[: 1 << 20].float().clone()
    dist.all_reduce(ref)
    ref /= world
    ok = bool(torch.allclose(mine, ref, rtol=1e-6, atol=1e-9))
    nvls_ok = None
    if have_nvls:
        # the multimem flavour on the same data: equal to the exact flavours up to the bf16 rounding of the switch's sum
        eng.set_k1_algo("nvls")
        eng.grad_reduce(_lib.REDUCE_ALL, G.peer_ptrs(), torch.bfloat16, None, O32.peer_ptrs(), torch.float32, n, 1.0 / world,
                        _lib.NORM_L2, 2.0, _lib.RF_FINAL)
        eng.set_k1_algo("bulk")
        mm = O32.tensor(torch.float32, n)[: 1 << 20].clone()
        nvls_ok = bool(torch.allclose(mm, ref, rtol=2.0**-7, atol=1e-9))
    if rank == 0:
        summary = {"world": world, "rows": rows, "spot_check_ok": ok, "nvls_spot_check_ok": nvls_ok, "nvls": have_nvls,
                   "nvlink_nominal_gbs": 900, "nvlink_measured_peer_copy_gbs": 770}
        if args.out:
            with open(args.out, "w") as f:
                json.dump(summary, f, indent=1)
        if args.json_line:
            big = rows[-1]
            best = max((big.get(k, 0.0), k) for k in ("ours_bf16_busbw", "ours_ldg_bf16_busbw", "ours_nvls_bf16_busbw"))
            print(json.dumps({"metric": "fused grad all-reduce bus bandwidth (NCCL convention 2(W-1)/W*S/t), largest bucket",
                              "value": best[0], "unit": "GB/s", "n_gpus": world, "steps": 50, "warmup": 10,
                              "ms_per_step": big[best[1].replace("_busbw", "_us")] * 1e-3, "higher_is_better": True,
                              "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                              "config": {"workload": "grad_allreduce_sweep_64KB_1GB", "flavour": best[1], "l2": "buckets >= 256 MB exceed L2"},
                              "roofline": {"bound": "nvlink", "achieved": best[0], "peak": 900.0, "unit": "GB/s",
                                           "frac": best[0] / 900.0, "traffic": None}, "rows": rows,
                              "spot_check_ok": ok, "nvls_spot_check_ok": nvls_ok}))
        else:
            print("spot check", ok, "nvls", nvls_ok)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

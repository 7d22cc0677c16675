"""CPU tests: the C-ABI library loads and exports every symbol include/stoke_b200.h declares (no compute calls without a
GPU), and the host-side functions of the library (mt19937 randperm, sampler planning, padding tables, shard ranges) agree
with torch / the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from stoke_b200 import _lib, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from stoke_b200.csrc.build import build

    build()
    return _lib.load()


def test_header_symbols_exported(lib):
    header = open(os.path.join(ROOT, "include", "stoke_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(stk_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.stk_version() >= 100


def test_option_and_optimizer_constants_match_header():
    """Every STK_OPT_<NAME> of the header (option keys are #defines, optimizer kinds an enum) is _lib.OPT_<NAME> with the
    same value, and _lib has no OPT_ constant the header lacks."""
    header = open(os.path.join(ROOT, "include", "stoke_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    pairs = re.findall(r"#define\s+STK_OPT_([A-Z0-9_]+)\s+(\d+)\b", header)
    pairs += re.findall(r"\bSTK_OPT_([A-Z0-9_]+)\s*=\s*(\d+)\b", header)
    declared = {name: int(v) for name, v in pairs}
    assert len(declared) == len(pairs) and {"K1_ALGO", "ADAM"} <= set(declared)
    mine = {k[len("OPT_"):]: v for k, v in vars(_lib).items() if k.startswith("OPT_")}
    assert mine == declared, set(mine.items()) ^ set(declared.items())


def test_struct_layouts_match_header():
    # sizes the C side static-asserts implicitly through use; guards against ctypes drift
    assert C.sizeof(_lib.ScalerState) == 48
    assert C.sizeof(_lib.SamplerPlan) == 8 * 5 + 4 * 3 + 4 + 8 * 10 + 8  # with alignment padding
    assert C.sizeof(_lib.OptimHyper) == 8 + 8 * 7 + 4 * 3 + 4 + 16


def test_no_gpu_fails_loudly(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    ctx = C.c_void_p()
    assert lib.stk_ctx_create(0, 1, 0, 0, C.byref(ctx)) == _lib.ERR_CUDA
    from stoke_b200.engine import Engine

    with pytest.raises(_lib.StokeB200Error):
        Engine(0)
    import stoke_b200 as sb

    with pytest.raises(ValueError):
        sb.Stoke(torch.nn.Linear(2, 2), sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs={}),
                 torch.nn.MSELoss(), 4, gpu=True)
    with pytest.raises(ValueError):  # no CPU path at all
        sb.Stoke(torch.nn.Linear(2, 2), sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs={}),
                 torch.nn.MSELoss(), 4, gpu=False)


def test_randperm_bit_exact_with_torch(lib):
    for seed, lens in ((0, [1000]), (7, [1000, 17, 0, 1, 2, 625, 62501]), (2**40 + 5, [50, 50]), (123456789, [300000])):
        arr = (C.c_int64 * len(lens))(*lens)
        out = np.zeros(sum(lens), dtype=np.int32)
        _lib.check(lib.stk_randperm(seed, arr, len(lens), out.ctypes.data))
        g = torch.Generator()
        g.manual_seed(seed)
        off = 0
        for n in lens:
            ref = torch.randperm(n, generator=g).numpy()
            assert np.array_equal(out[off: off + n], ref), (seed, n)
            off += n


def _plan(lib, n, buckets, bs, w, rank=0, drop_last=False, overlap=False, shuffle=True):
    p = _lib.SamplerPlan()
    p.n, p.buckets, p.batch_size, p.world, p.rank = n, buckets, bs, w, rank
    p.drop_last, p.allow_bucket_overlap, p.shuffle = int(drop_last), int(overlap), int(shuffle)
    return p, lib.stk_sampler_plan(C.byref(p))


def test_sampler_plan_matches_oracle(lib):
    from sampler_oracle import SamplerPlan

    rng = np.random.default_rng(0)
    ok = bad = 0
    for _ in range(400):
        n = int(rng.integers(50, 6000)); buckets = int(rng.integers(1, 12)); bs = int(rng.integers(1, 40))
        w = int(rng.integers(1, 9)); dl = bool(rng.integers(0, 2)); ov = bool(rng.integers(0, 2))
        p, code = _plan(lib, n, buckets, bs, w, 0, dl, ov)
        try:
            ref = SamplerPlan(n, buckets, bs, w, dl, ov)
        except ValueError:
            assert code == _lib.ERR_INVALID
            assert lib.stk_last_error(None).decode().startswith("Stoke -- ")
            bad += 1
            continue
        assert code == 0
        assert (p.slice_size, p.per_bucket, p.slices_per_bucket, p.rounded_per_bucket, p.rounded_per_replica) == (
            ref.slice_size, ref.per_bucket, ref.slices_per_bucket, ref.rounded_per_bucket, ref.rounded_per_replica)
        sizes = [len(a) for a in np.array_split(np.arange(n), buckets)]
        assert sizes == [p.bucket_base + (1 if b < p.bucket_rem else 0) for b in range(buckets)]
        ok += 1
    assert ok > 50 and bad > 10


def test_last_slice_table_matches_oracle_padding(lib):
    from sampler_oracle import SamplerPlan, _pad_bucket

    rng = np.random.default_rng(1)
    checked = 0
    for _ in range(300):
        buckets = int(rng.integers(1, 6)); bs = int(rng.integers(1, 20)); w = int(rng.integers(1, 9))
        n = int(rng.integers(200, 6000))
        p, code = _plan(lib, n, buckets, bs, w)
        if code != 0:
            continue
        ref = SamplerPlan(n, buckets, bs, w)
        for ln in {p.bucket_base + 1 if p.bucket_rem else p.bucket_base, p.bucket_base}:
            if p.rounded_per_bucket <= ln:
                continue
            tab = np.zeros(p.slice_size, dtype=np.int32)
            _lib.check(lib.stk_sampler_last_slice(C.byref(p), ln, tab.ctypes.data))
            bucket = np.arange(ln, dtype=np.int64)  # identity "permuted bucket": values are positions
            padded = _pad_bucket(bucket, ref)
            assert np.array_equal(padded[-p.slice_size:], tab)
            checked += 1
    assert checked > 100


def test_shard_ranges_partition(lib):
    for n in (8, 64, 99_080, 25_557_040, 109_483_784):
        for w in (1, 2, 3, 4, 8):
            prev = 0
            for r in range(w):
                b, e = C.c_size_t(), C.c_size_t()
                assert lib.stk_shard_range(n, w, r, C.byref(b), C.byref(e)) == 0
                assert b.value == prev and e.value >= b.value and b.value % 8 == 0
                prev = e.value
            assert prev == n


def test_replicas_are_disjoint_and_cover(lib):
    """N>1 host-side property on the oracle side of the sampler (the device kernel is checked on the GPU box)."""
    from sampler_oracle import oracle_indices

    n, buckets, bs, w = 4099, 4, 8, 4
    sorted_idx = synthetic.sampler_sorted_idx(n)
    lists = [oracle_indices(sorted_idx, buckets, bs, w, r, True, 3, 1) for r in range(w)]
    assert len({len(l) for l in lists}) == 1
    counts = np.bincount(np.concatenate(lists), minlength=n)
    assert counts.min() >= 1


def test_descriptor_passing_between_processes(tmp_path):
    """The VMM back end hands cuMemExportToShareableHandle descriptors to the peer ranks over an abstract unix socket
    (stoke_b200/csrc/fdpass.h, SCM_RIGHTS).  Pure POSIX: compiled with g++ and run between two processes here."""
    import shutil
    import subprocess

    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "test_fdpass"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-pthread", os.path.join(root, "tools", "test_fdpass.cpp"), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "fdpass ok" in out.stdout, out.stdout + out.stderr

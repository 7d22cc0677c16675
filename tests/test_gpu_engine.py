"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C ABI vs the CPU oracle on identical inputs.

Float bar (BASELINE.json north_star): fp32 master weights within 1e-5 relative of the oracle after N steps of
gradient-injection (both sides consume the same, bf16- or fp32-representable, gradients).  Integer work is bit-exact.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-5  # relative L2 error on the fp32 master weights (north_star)


class OddNet(torch.nn.Module):
    """Parameters with awkward sizes (not multiples of 8), a matrix, a 4-D weight and a scalar."""

    def __init__(self, scale=1):
        super().__init__()
        g = torch.Generator().manual_seed(11)
        shapes = [(257 * scale, 129), (129,), (3, 5, 7, 11), (1,), (1000 * scale + 3,), (64, 64)]
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(*s, generator=g) * 0.1) for s in shapes])

    def forward(self, x):
        return sum(p.sum() for p in self.ps) * x


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _oracle_flat(path, oracle_weights):
    flat = torch.zeros(path.n)
    for dst, w in zip(path.unflatten(flat), oracle_weights):
        dst.copy_(w)
    return flat


def _make(optim_cls, kwargs, lp, clip=None, accum=1, scale=1, route=None, stock=False):
    from stoke_b200 import _lib
    from stoke_b200.engine import ClipSpec, get_engine
    from stoke_b200.optim import B200FusedOptimizer

    torch.cuda.set_device(0)
    net = OddNet(scale).cuda()
    init = [p.detach().cpu().clone() for p in net.parameters()]
    spec = None
    if clip is not None:
        spec = ClipSpec(_lib.CLIP_NORM, max_norm=clip[1], norm_type=clip[2]) if clip[0] == "norm" else \
            ClipSpec(_lib.CLIP_VALUE, clip_value=clip[1])
    if stock:
        from stoke_b200.optim import B200StockOptimizer

        opt = B200StockOptimizer(net, optim_cls, kwargs, engine=get_engine(0), grad_accum=accum, clip=spec, lp_dtype=lp)
    else:
        opt = B200FusedOptimizer(net, optim_cls, kwargs, engine=get_engine(0), grad_accum=accum, clip=spec, lp_dtype=lp,
                                 route=route)
    return net, init, opt


def _inject(path, step, rank, dtype, scale=1.0):
    """Writes a seeded gradient into the flat bucket through the param.grad views; returns per-param fp32 copies."""
    from stoke_b200 import synthetic

    out = []
    for i, gv in enumerate(path.grad_views):
        g = synthetic.injected_grad(gv.numel(), rank, step * 100 + i, dtype=dtype, scale=scale).view(gv.shape)
        gv.copy_(g.cuda())
        out.append(g.float())
    return out


CASES = [
    (torch.optim.Adam, {"lr": 1e-3, "betas": (0.9, 0.98), "eps": 1e-9}, torch.bfloat16, ("norm", 1.0, 2.0), 1),
    (torch.optim.Adam, {"lr": 1e-3, "weight_decay": 0.01}, torch.bfloat16, None, 1),
    (torch.optim.Adam, {"lr": 2e-3}, None, ("norm", 0.5, 2.0), 1),
    (torch.optim.Adam, {"lr": 1e-3}, torch.bfloat16, ("value", 0.3), 2),
    (torch.optim.AdamW, {"lr": 1e-3, "weight_decay": 0.05}, torch.bfloat16, ("norm", 2.0, float("inf")), 1),
    (torch.optim.AdamW, {"lr": 1e-3}, None, ("norm", 1.0, 3.0), 3),
    (torch.optim.SGD, {"lr": 0.05, "momentum": 0.9, "weight_decay": 1e-4}, torch.bfloat16, ("norm", 1.0, 2.0), 1),
    (torch.optim.SGD, {"lr": 0.05, "momentum": 0.9, "nesterov": True}, None, None, 2),
    (torch.optim.SGD, {"lr": 0.1}, torch.bfloat16, None, 1),
]


@pytest.mark.parametrize("route", ["local", "main"])
@pytest.mark.parametrize("optim_cls,kwargs,lp,clip,accum", CASES)
def test_gradient_injection_parity_w1(optim_cls, kwargs, lp, clip, accum, route):
    """route="local": k_grad_norm + the fused step reading the raw bucket (the training path at world 1);
    route="main": K1's W == 1 form materialising fp32 main grads + the fused step reading those."""
    from engine_oracle import OracleEngine

    net, init, opt = _make(optim_cls, kwargs, lp, clip, accum, route=route)
    path = opt.path
    assert path.route == route
    oracle = OracleEngine(init, 1, optim_cls, kwargs, grad_accum=accum, clip=clip)
    gdtype = lp or torch.float32
    n_steps = 12
    for step in range(n_steps):
        for micro in range(accum):
            grads = _inject(path, step * accum + micro, 0, gdtype)
            oracle.micro_step([grads])
            path.after_backward(sync=(micro == accum - 1), unscale=False)
        opt.step()
        oracle.step()
        assert float(path.g_flat.float().abs().max()) == 0.0  # bucket zeroed after consumption
    ref = _oracle_flat(path, oracle.weights())
    got = path.gather_master().cpu()
    assert _rel(got, ref) < TOL
    if clip is not None and clip[0] == "norm":
        assert abs(path.engine.scaler_get(path.state_id).grad_norm - float(oracle.last_total_norm)) / float(oracle.last_total_norm) < 1e-5
    if lp is not None:  # the model copy is the rounded master
        assert torch.equal(path.p_flat.cpu(), got.to(lp))
    # optimizer state in torch's layout
    sd = opt.state_dict()
    if optim_cls is not torch.optim.SGD:
        for i, p in enumerate(oracle.params):
            st = oracle.optimizer.state[p]
            assert _rel(sd["state"][i]["exp_avg"].cpu(), st["exp_avg"]) < 1e-5
            assert _rel(sd["state"][i]["exp_avg_sq"].cpu(), st["exp_avg_sq"]) < 1e-5
            assert float(sd["state"][i]["step"]) == float(st["step"])


def test_large_flat_parity_and_full_size_properties():
    """ResNet-50-sized flat buffer (25.6 M elements): one step equals the oracle on a strided sample; linearity of the
    reduce (size-independent property): reduce(a) + reduce(b) == reduce(a + b) for exactly representable inputs."""
    from engine_oracle import OracleEngine

    class Big(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(25_557_032))

    from stoke_b200 import _lib
    from stoke_b200.engine import ClipSpec, get_engine
    from stoke_b200.optim import B200FusedOptimizer

    torch.cuda.set_device(0)
    net = Big().cuda()
    torch.manual_seed(0)
    with torch.no_grad():
        net.w.copy_(torch.randn_like(net.w) * 0.05)
    init = [net.w.detach().cpu().clone()]
    kw = {"lr": 1e-3}
    opt = B200FusedOptimizer(net, torch.optim.Adam, kw, engine=get_engine(0),
                             clip=ClipSpec(_lib.CLIP_NORM, max_norm=1.0, norm_type=2.0), lp_dtype=torch.bfloat16, route="main")
    path = opt.path
    oracle = OracleEngine(init, 1, torch.optim.Adam, kw, clip=("norm", 1.0, 2.0))
    for step in range(3):
        g = (torch.randn(path.n, device="cuda") * 1e-3).to(torch.bfloat16)
        path.g_flat.copy_(g)
        oracle.micro_step([[g[: net.w.numel()].float().cpu()]])
        path.after_backward(sync=True, unscale=False)
        opt.step()
        oracle.step()
    got = path.gather_master().cpu()[: net.w.numel()]
    assert _rel(got, oracle.flat_weights()) < TOL
    # linearity on small integers (exact in bf16 and fp32)
    a = torch.randint(-8, 9, (path.n,), device="cuda").to(torch.bfloat16)
    b = torch.randint(-8, 9, (path.n,), device="cuda").to(torch.bfloat16)
    outs = []
    for v in (a, b, a + b):
        path.g_flat.copy_(v)
        path.after_backward(sync=True, unscale=False)
        outs.append(path.main_flat.clone())
        path.engine.step_epilogue()
    assert torch.equal(outs[0] + outs[1], outs[2])
    norm = math.sqrt(float(((a + b).double() ** 2).sum()))
    # grad_norm was reset by the epilogue's reduce of a+b? it is written by the FINAL reduce and kept until the next one
    assert abs(path.engine.scaler_get(path.state_id).grad_norm - norm) / norm < 1e-5


def test_full_size_local_route_matches_main_route():
    """ResNet-50-sized bucket: the world-1 training route (norm pass + raw-bucket step) and the main-grad route agree on
    master weights, norms and zeroed buckets from the same gradients (size-independent property).  Not bit-identical: the
    two norm reductions use different (each fixed) summation trees, so the clip coefficient may differ in its last bit."""
    from stoke_b200 import _lib
    from stoke_b200.engine import ClipSpec, get_engine
    from stoke_b200.optim import B200FusedOptimizer

    class Big(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(25_557_032))

    torch.cuda.set_device(0)
    outs = {}
    for route in ("local", "main"):
        net = Big().cuda()
        torch.manual_seed(0)
        with torch.no_grad():
            net.w.copy_(torch.randn_like(net.w) * 0.05)
        opt = B200FusedOptimizer(net, torch.optim.AdamW, {"lr": 1e-3, "weight_decay": 0.01}, engine=get_engine(0),
                                 clip=ClipSpec(_lib.CLIP_NORM, max_norm=1.0, norm_type=2.0), lp_dtype=torch.bfloat16,
                                 route=route)
        path = opt.path
        gen = torch.Generator(device="cuda").manual_seed(5)
        norms = []
        for _ in range(3):
            path.g_flat.copy_((torch.randn(path.n, device="cuda", generator=gen) * 1e-3).to(torch.bfloat16))
            path.after_backward(sync=True, unscale=False)
            opt.step()
            norms.append(path.engine.scaler_get(path.state_id).grad_norm)
            assert float(path.g_flat.float().abs().max()) == 0.0
        outs[route] = (path.gather_master().clone(), path.p_flat.clone(), norms)
        opt.close()
    assert _rel(outs["local"][0], outs["main"][0]) < 1e-6
    assert (outs["local"][1] != outs["main"][1]).float().mean() < 1e-3   # bf16 copies: at most a rounding flip here and there
    for a, b in zip(outs["local"][2], outs["main"][2]):
        assert abs(a - b) / b < 1e-6   # different (fixed) summation trees


def test_amp_scaler_skip_backoff_growth():
    """inf/nan in the gradients: no update at all, scale backs off, tracker resets; growth after the interval
    (GradScaler semantics as the reference uses them, stoke/fp16.py:805-806)."""
    from engine_oracle import OracleEngine
    from stoke_b200.fp16 import DeviceGradScaler

    kw = {"lr": 1e-2}
    net, init, opt = _make(torch.optim.Adam, kw, None, ("norm", 1.0, 2.0), 1)
    path = opt.path
    scaler = DeviceGradScaler(path.engine, init_scale=2.0**10, growth_interval=3, state_id=path.state_id)
    oracle = OracleEngine(init, 1, torch.optim.Adam, kw, clip=("norm", 1.0, 2.0),
                          amp=dict(init_scale=2.0**10, growth_interval=3))
    plan = [False, True, False, False, False, True, False]
    for step, bad in enumerate(plan):
        s = scaler.get_scale()
        assert s == oracle.loss_scale
        grads = _inject(path, step, 0, torch.float32, scale=s)
        if bad:
            path.grad_views[2].view(-1)[5] = float("inf") if step == 1 else float("nan")
            grads[2].view(-1)[5] = float("inf") if step == 1 else float("nan")
        oracle.micro_step([grads])
        before = path.gather_master().clone()
        path.after_backward(sync=True, unscale=True)
        opt.step()
        stepped = oracle.step()
        assert stepped == (not bad)
        if bad:
            assert torch.equal(before, path.gather_master())
    st = path.engine.scaler_get(path.state_id)
    assert st.opt_steps == 5 and st.skipped_steps == 2
    assert scaler.get_scale() == oracle.loss_scale
    assert scaler.state_dict()["_growth_tracker"] == oracle.scaler.state_dict()["_growth_tracker"]
    assert _rel(path.gather_master().cpu(), _oracle_flat(path, oracle.weights())) < TOL


@pytest.mark.parametrize("name", ["noclip", "clipnorm", "clipvalue"])
def test_cfg1_through_stoke_api_vs_reference_fixture(golden_dir, name):
    """BASELINE configs[0] end to end through ``Stoke`` on the GPU (fp32) against the fixture produced by the unmodified
    reference on CPU.  Forward/backward run in cuBLAS instead of CPU BLAS, so this is not gradient-injection: the bar is
    the loss trajectory and the counters; weights are compared with a looser bound and reported."""
    import stoke_b200 as sb
    from stoke_b200 import synthetic

    gold = np.load(os.path.join(golden_dir, f"cfg1_{name}.npz"))
    clip = {"noclip": None, "clipnorm": sb.ClipGradNormConfig(max_norm=0.05, norm_type=2.0),
            "clipvalue": sb.ClipGradConfig(clip_value=0.002)}[name]
    torch.backends.cuda.matmul.allow_tf32 = False
    model = synthetic.basic_nn()
    s = sb.Stoke(model=model, optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=synthetic.CFG1_ADAM),
                 loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=synthetic.CFG1_BATCH,
                 grad_accum_steps=synthetic.CFG1_ACCUM, grad_clip=clip, gpu=True, verbose=False)
    losses, trace = [], []
    for x, y in synthetic.cfg1_batches(synthetic.CFG1_OPT_STEPS * synthetic.CFG1_ACCUM):
        l = s.loss(s.model(x.cuda()), y.cuda())
        losses.append(s.step_loss)
        s.backward(l)
        s.step()
        trace.append((s._grad_accum_counter, s._backward_steps, s._optimizer_steps))
    assert np.array_equal(np.asarray(trace), gold["trace"])
    assert np.allclose(np.asarray(losses), gold["losses"], rtol=2e-3, atol=1e-6)
    final = torch.cat([p.detach().reshape(-1) for p in s.model_access.parameters()]).cpu().numpy()
    rel = np.linalg.norm(final - gold["final"]) / np.linalg.norm(gold["final"])
    print(f"cfg1/{name}: end-to-end weight rel err vs reference CPU run = {rel:.3e}")
    assert rel < 3e-2  # chaotic amplification through Adam (eps 1e-9); the 1e-5 bar is the gradient-injection tests'


def test_loss_sync_and_barrier_world1():
    from stoke_b200.engine import get_engine

    eng = get_engine(0)
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        t = torch.tensor(1.375, device="cuda", dtype=dt)
        assert eng.loss_sync(t) == 1.375
    eng.barrier()
    eng.comm_check()


def test_removed_option_keys_are_rejected():
    """Keys 4 (non-cooperative launch), 6 (multimem.st publish) and 7 (one-shot all-reduce) no longer exist."""
    from stoke_b200 import _lib
    from stoke_b200.engine import get_engine

    eng = get_engine(0)
    for key in (4, 6, 7):
        with pytest.raises(_lib.StokeB200Error) as e:
            eng.option_set(key, 0)
        assert e.value.code == _lib.ERR_INVALID
        with pytest.raises(_lib.StokeB200Error) as e:
            eng.option_get(key)
        assert e.value.code == _lib.ERR_INVALID
    for key in (_lib.OPT_K1_ALGO, _lib.OPT_MEM_MODE, _lib.OPT_K1_MAX_BLOCKS, _lib.OPT_NVLS_MAX_BLOCKS):
        eng.option_get(key)


def test_save_load_roundtrip(tmp_path):
    import stoke_b200 as sb
    from stoke_b200 import synthetic

    def make():
        return sb.Stoke(model=synthetic.basic_nn(), optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam,
                        optimizer_kwargs=synthetic.CFG1_ADAM), loss=torch.nn.BCEWithLogitsLoss(),
                        batch_size_per_device=32, grad_clip=sb.ClipGradNormConfig(1.0, 2.0), gpu=True, fp16="bf16",
                        verbose=False)

    def run(s, batches):
        for x, y in batches:
            s.backward(s.loss(s.model(x.cuda()), y.cuda()))
            s.step()

    batches = list(synthetic.cfg1_batches(10))
    a = make()
    run(a, batches[:5])
    path, tag = a.save(str(tmp_path), name="ck", extras={"foo": "bar"})
    run(a, batches[5:])
    wa = a.optimizer.path.gather_master().clone()
    b = make()
    extras = b.load(path, tag)
    assert extras == {"foo": "bar"} and b._optimizer_steps == 5
    run(b, batches[5:])
    assert torch.equal(wa, b.optimizer.path.gather_master())
    sd = torch.load(f"{path}/{tag}", weights_only=False)
    assert set(sd) == {"backward_step", "grad_accum_step", "optimizer_step", "stoke_status", "model_state_dict",
                       "optimizer_state_dict", "scaler_state_dict", "extras"}


def test_amp_fp16_through_stoke_api_matches_torch_amp():
    """``fp16="amp"`` end to end: fp16 autocast + device-resident loss scaler, against the same loop written with torch's
    own ``torch.amp.GradScaler`` + ``clip_grad_norm_`` + ``torch.optim.Adam`` on the GPU (the calls the reference's
    NativeAmpFP16 makes, stoke/fp16.py:733-806).  Same forward/backward kernels on both sides, so the weights agree to fp32
    round-off; an overflow forced through a huge init_scale must be skipped identically."""
    import stoke_b200 as sb
    from stoke_b200 import synthetic

    kw = {"lr": 1e-3}
    init_scale = 2.0**24  # overflows fp16 on the first steps -> skipped steps and back-off on both sides
    m_new, m_ref = synthetic.basic_nn(5), synthetic.basic_nn(5).cuda()
    s = sb.Stoke(model=m_new, optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=kw),
                 loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32,
                 grad_clip=sb.ClipGradNormConfig(max_norm=0.1, norm_type=2.0), gpu=True, fp16="amp",
                 configs=[sb.AMPConfig(init_scale=init_scale, growth_interval=4)], verbose=False)
    opt = torch.optim.Adam(m_ref.parameters(), **kw)
    scaler = torch.amp.GradScaler("cuda", init_scale=init_scale, growth_interval=4)
    lossf = torch.nn.BCEWithLogitsLoss()
    for x, y in synthetic.cfg1_batches(24, seed=3):
        x, y = x.cuda() * 30.0, y.cuda()
        s.backward(s.loss(s.model(x), y))
        s.step()
        with torch.autocast("cuda", dtype=torch.float16):
            l = lossf(m_ref(x), y)
        scaler.scale(l).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(m_ref.parameters(), 0.1, 2.0)
        scaler.step(opt)
        scaler.update()
        opt.zero_grad(set_to_none=True)
        assert s.scaler.get_scale() == scaler.get_scale()
    st = s.engine.scaler_get(s.optimizer.path.state_id)
    assert st.skipped_steps >= 1 and st.opt_steps + st.skipped_steps == 24
    ref = torch.cat([p.detach().reshape(-1) for p in m_ref.parameters()]).cpu()
    got = torch.cat([p.detach().reshape(-1) for p in s.model_access.parameters()]).cpu()
    # different Adam / clip kernels on the two sides (torch's foreach path vs K2) + fp16 forward: loose bound here, the 1e-5
    # bar is the gradient-injection tests'; the scaler trajectory above is exact
    assert _rel(got, ref) < 1e-3
    assert s.scaler.state_dict()["_growth_tracker"] == scaler.state_dict()["_growth_tracker"]


def test_device_prefetcher_order_and_values():
    from stoke_b200.data import DevicePrefetcher

    batches = [(torch.full((4, 3), float(i)).pin_memory(), {"y": torch.tensor([i])}) for i in range(7)]
    out = list(DevicePrefetcher(iter(batches)))
    assert len(out) == 7
    for i, (x, d) in enumerate(out):
        assert x.is_cuda and float(x.sum()) == 12.0 * i and int(d["y"]) == i


# ---- parameter groups, unused parameters, the stock-optimizer route, reference-format checkpoints ---------------------
@pytest.mark.parametrize("lp", [torch.bfloat16, None])
def test_parameter_groups_parity(lp):
    """Two torch-style parameter groups (the usual no-weight-decay split + a different lr), alternating through the flat
    layout: per-group hyper-parameters are selected inside the fused kernel by element range."""
    from engine_oracle import OracleEngine
    from stoke_b200.engine import get_engine
    from stoke_b200.optim import B200FusedOptimizer

    torch.cuda.set_device(0)
    net = OddNet().cuda()
    params = list(net.parameters())
    init = [p.detach().cpu().clone() for p in params]
    idx_a, idx_b = [0, 2, 4], [1, 3, 5]
    kw = {"lr": 1e-3, "weight_decay": 0.05}
    groups_dev = [{"params": [params[i] for i in idx_a]},
                  {"params": [params[i] for i in idx_b], "weight_decay": 0.0, "lr": 3e-3, "betas": (0.8, 0.95)}]
    opt = B200FusedOptimizer(net, torch.optim.AdamW, dict(kw, params=groups_dev), engine=get_engine(0), lp_dtype=lp)
    path = opt.path
    oracle = OracleEngine(init, 1, torch.optim.AdamW, kw,
                          groups=[(idx_a, {}), (idx_b, {"weight_decay": 0.0, "lr": 3e-3, "betas": (0.8, 0.95)})])
    for step in range(10):
        grads = _inject(path, step, 0, lp or torch.float32)
        oracle.micro_step([grads])
        path.after_backward(sync=True, unscale=False)
        if step == 5:
            opt.param_groups[1]["lr"] = 1e-3           # a scheduler edit reaches the kernel
            oracle.optimizer.param_groups[1]["lr"] = 1e-3
        opt.step()
        oracle.step()
    assert _rel(path.gather_master().cpu(), _oracle_flat(path, oracle.weights())) < TOL
    sd = opt.state_dict()
    ref_sd = oracle.optimizer.state_dict()
    assert [g["params"] for g in sd["param_groups"]] == [g["params"] for g in ref_sd["param_groups"]]
    for j, st in ref_sd["state"].items():
        assert _rel(sd["state"][j]["exp_avg"].cpu(), st["exp_avg"]) < 1e-5
    opt.close()


def test_unused_parameters_are_skipped_like_torch():
    """A parameter that receives no gradient in a step keeps its value AND its optimizer state (torch skips p.grad is None
    after zero_grad(set_to_none=True), stoke/utils.py:103-106) -- no moment decay, no weight decay -- and from then on step
    counts are kept per parameter, like torch's state[p]["step"], so the sometimes-unused head gets its own Adam bias
    corrections: every parameter follows the oracle to 1e-5."""
    from engine_oracle import OracleEngine
    import stoke_b200 as sb

    class TwoHeads(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(3)
            self.body = torch.nn.Linear(16, 24)
            self.a = torch.nn.Linear(24, 1)
            self.b = torch.nn.Linear(24, 1)
            self.use_b = True

        def forward(self, x):
            h = torch.tanh(self.body(x))
            return self.a(h) + (self.b(h) if self.use_b else 0.0)

    torch.cuda.set_device(0)
    kw = {"lr": 1e-2, "weight_decay": 0.1}
    model = TwoHeads()
    init = [p.detach().clone() for p in model.parameters()]
    s = sb.Stoke(model=model, optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=kw),
                 loss=torch.nn.MSELoss(), batch_size_per_device=8, gpu=True, verbose=False)
    oracle = OracleEngine(init, 1, torch.optim.Adam, kw)
    path = s.optimizer.path
    g = torch.Generator().manual_seed(0)
    for step in range(9):
        model.use_b = step % 3 != 1            # head b unused on steps 1, 4, 7
        x, y = torch.randn(8, 16, generator=g).cuda(), torch.randn(8, 1, generator=g).cuda()
        loss = s.loss(s.model(x), y)
        b_before = (model.b.weight.detach().clone(), s.optimizer.state_dict()["state"][4]["exp_avg"].clone())
        # gradient injection: the oracle consumes the gradients autograd produced on the device
        path.begin_backward(sync=True, unscale=False)
        loss.backward()
        grads = [gv.detach().float().cpu().clone() if path._touched[i] else None for i, gv in enumerate(path.grad_views)]
        assert (grads[4] is None) == (not model.use_b)
        oracle.micro_step([grads])
        s._grad_accum_counter += 1
        path.after_backward(sync=True, unscale=False)
        s._backward_steps += 1
        s.step()
        oracle.step()
        same = torch.equal(b_before[0], model.b.weight.detach()) and \
            torch.equal(b_before[1], s.optimizer.state_dict()["state"][4]["exp_avg"])
        assert same == (not model.use_b)
    got = [p.detach().float().cpu() for p in model.parameters()]
    for a, b in zip(got, oracle.weights()):
        assert _rel(a.reshape(-1), b.reshape(-1)) < TOL
    sd = s.optimizer.state_dict()
    for j, p in enumerate(oracle.params):   # per-parameter step counts: 9 for the always-used parameters, 6 for head b
        assert float(sd["state"][j]["step"]) == float(oracle.optimizer.state[p]["step"])
    assert [float(sd["state"][j]["step"]) for j in range(6)] == [9.0, 9.0, 9.0, 9.0, 6.0, 6.0]
    # round trip: a second Stoke loads the per-parameter counts and continues identically
    model2 = TwoHeads()
    s2 = sb.Stoke(model=model2, optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=kw),
                  loss=torch.nn.MSELoss(), batch_size_per_device=8, gpu=True, verbose=False)
    model2.load_state_dict(model.state_dict())
    s2.optimizer.load_state_dict(sd)
    assert s2.optimizer.path.param_steps() == [9, 9, 9, 9, 6, 6]
    for st, mdl in ((s, model), (s2, model2)):
        mdl.use_b = True
        x, y = torch.ones(8, 16).cuda(), torch.ones(8, 1).cuda()
        st.backward(st.loss(st.model(x), y))
        st.step()
    for a, b in zip(model.parameters(), model2.parameters()):
        assert torch.equal(a.detach(), b.detach())


@pytest.mark.parametrize("optim_cls,kwargs,lp,clip", [
    (torch.optim.RMSprop, {"lr": 1e-3, "momentum": 0.5}, torch.bfloat16, ("norm", 1.0, 2.0)),
    (torch.optim.Adam, {"lr": 1e-3, "amsgrad": True}, None, ("value", 0.3)),
    (torch.optim.Adagrad, {"lr": 1e-2}, torch.bfloat16, None),
])
def test_stock_optimizer_route_parity(optim_cls, kwargs, lp, clip):
    """Any torch.optim class (the reference instantiates whatever the user passes, stoke/extensions.py:53-78): the engine's
    gradient path (K1 + k_grad_scale) feeding the stock optimizer on fp32 master views."""
    from engine_oracle import OracleEngine

    net, init, opt = _make(optim_cls, kwargs, lp, clip, accum=2, stock=True)
    path = opt.path
    oracle = OracleEngine(init, 1, optim_cls, kwargs, grad_accum=2, clip=clip)
    for step in range(8):
        for micro in range(2):
            grads = _inject(path, step * 2 + micro, 0, lp or torch.float32)
            oracle.micro_step([grads])
            path.after_backward(sync=(micro == 1), unscale=False)
        opt.step()
        oracle.step()
    assert _rel(path.gather_master().cpu(), _oracle_flat(path, oracle.weights())) < TOL
    if lp is not None:
        assert torch.equal(path.p_flat.cpu(), path.gather_master().cpu().to(lp))
    opt.close()


def test_stock_route_through_stoke_api():
    import stoke_b200 as sb
    from stoke_b200 import synthetic
    from stoke_b200.optim import B200StockOptimizer

    s = sb.Stoke(model=synthetic.basic_nn(), optimizer=sb.StokeOptimizer(optimizer=torch.optim.RMSprop, optimizer_kwargs={"lr": 1e-3}),
                 loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32, grad_clip=sb.ClipGradNormConfig(1.0, 2.0),
                 gpu=True, fp16="bf16", verbose=False)
    assert isinstance(s.optimizer, B200StockOptimizer)
    first = None
    for x, y in synthetic.cfg1_batches(30):
        s.backward(s.loss(s.model(x.cuda()), y.cuda()))
        s.step()
        first = s.step_loss if first is None else first
    assert s.step_loss < first and s._optimizer_steps == 30


def test_load_checkpoint_written_by_the_reference_format(tmp_path):
    """A checkpoint in the reference's layout (stoke/io_ops.py:224-236: plain torch optimizer state dict, no engine keys)
    written from a stock torch run: load it into a bf16 Stoke and continue -- the fp32 master weights must be rebuilt from
    the loaded model weights (they used to keep their old values and overwrite the loaded model at the next step)."""
    from engine_oracle import OracleEngine
    import stoke_b200 as sb
    from stoke_b200 import synthetic

    torch.cuda.set_device(0)
    kw = dict(synthetic.CFG1_ADAM)
    ref_model = synthetic.basic_nn(7)
    with torch.no_grad():
        for p in ref_model.parameters():
            p.copy_(p.to(torch.bfloat16).float())     # weights exactly representable in the model dtype
    ref_opt = torch.optim.Adam(ref_model.parameters(), **kw)
    lossf = torch.nn.BCEWithLogitsLoss()
    batches = list(synthetic.cfg1_batches(4, seed=9))
    for x, y in batches[:2]:
        lossf(ref_model(x), y).backward()
        ref_opt.step()
        ref_opt.zero_grad(set_to_none=True)
    with torch.no_grad():
        for p in ref_model.parameters():
            p.copy_(p.to(torch.bfloat16).float())
    tag = "stoke-ref-backward-step-2.pt"
    torch.save({"backward_step": 2, "grad_accum_step": 0, "optimizer_step": 2, "stoke_status": {},
                "model_state_dict": ref_model.state_dict(), "optimizer_state_dict": ref_opt.state_dict(),
                "scaler_state_dict": None, "extras": {"who": "reference"}}, str(tmp_path / tag))
    s = sb.Stoke(model=synthetic.basic_nn(0), optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs=kw),
                 loss=lossf, batch_size_per_device=32, gpu=True, fp16="bf16", verbose=False)
    extras = s.load(str(tmp_path), tag)
    assert extras == {"who": "reference"} and s._optimizer_steps == 2
    path = s.optimizer.path
    loaded = torch.cat([p.detach().reshape(-1) for p in ref_model.parameters()])
    got = torch.cat([m.reshape(-1) for m in path.unflatten(path.gather_master())]).cpu()
    assert torch.equal(got, loaded)                     # master == the loaded weights, not the constructor's
    assert path.engine.scaler_get(path.state_id).opt_steps == 2
    # continue one step with an injected gradient against the oracle continuing from the same state
    oracle = OracleEngine([p.detach() for p in ref_model.parameters()], 1, torch.optim.Adam, kw)
    oracle.optimizer.load_state_dict(ref_opt.state_dict())
    grads = _inject(path, 0, 0, torch.bfloat16)
    oracle.micro_step([grads])
    path.after_backward(sync=True, unscale=False)
    s.optimizer.step()
    oracle.step()
    got = torch.cat([m.reshape(-1) for m in path.unflatten(path.gather_master())]).cpu()
    assert _rel(got, oracle.flat_weights()) < TOL


def test_two_optimizers_in_one_process_do_not_share_state():
    """GAN-style: two Stoke objects alive at once, one with AMP loss scaling, one without -- step counters, found_inf, the
    loss scale and the clip norm are per optimizer (they used to live in the per-process engine)."""
    from engine_oracle import OracleEngine
    from stoke_b200.fp16 import DeviceGradScaler

    kw = {"lr": 1e-2}
    net_a, init_a, opt_a = _make(torch.optim.Adam, kw, None, ("norm", 1.0, 2.0))
    net_b, init_b, opt_b = _make(torch.optim.SGD, {"lr": 0.1, "momentum": 0.9}, torch.bfloat16, ("norm", 0.5, 2.0))
    pa, pb = opt_a.path, opt_b.path
    assert pa.state_id != pb.state_id
    scaler = DeviceGradScaler(pa.engine, init_scale=2.0**8, growth_interval=1000, state_id=pa.state_id)
    ora = OracleEngine(init_a, 1, torch.optim.Adam, kw, clip=("norm", 1.0, 2.0), amp=dict(init_scale=2.0**8, growth_interval=1000))
    orb = OracleEngine(init_b, 1, torch.optim.SGD, {"lr": 0.1, "momentum": 0.9}, clip=("norm", 0.5, 2.0))
    for step in range(6):
        ga = _inject(pa, step, 0, torch.float32, scale=scaler.get_scale())
        if step == 2:
            pa.grad_views[0].view(-1)[3] = float("inf")
            ga[0].view(-1)[3] = float("inf")
        ora.micro_step([ga])
        pa.after_backward(sync=True, unscale=True)
        gb = _inject(pb, step, 1, torch.bfloat16)
        orb.micro_step([gb])
        pb.after_backward(sync=True, unscale=False)   # interleaved: B's reduce runs between A's reduce and A's step
        opt_b.step()
        opt_a.step()
        ora.step()
        orb.step()
    sa, sb_ = pa.engine.scaler_get(pa.state_id), pb.engine.scaler_get(pb.state_id)
    assert (sa.opt_steps, sa.skipped_steps) == (5, 1) and (sb_.opt_steps, sb_.skipped_steps) == (6, 0)
    assert sa.scale == 2.0**7 and sb_.scale == 1.0 and sb_.enabled == 0
    assert _rel(pa.gather_master().cpu(), _oracle_flat(pa, ora.weights())) < TOL
    assert _rel(pb.gather_master().cpu(), _oracle_flat(pb, orb.weights())) < TOL
    opt_a.close()
    opt_b.close()


def test_fp16_loss_is_scaled_in_fp32():
    """scaler.scale(loss) with an fp16 loss tensor: 65536 is not representable in fp16, the product must be fp32."""
    from stoke_b200.engine import get_engine
    from stoke_b200.fp16 import DeviceGradScaler

    eng = get_engine(0)
    sid = eng.state_create()
    scaler = DeviceGradScaler(eng, init_scale=2.0**16, state_id=sid)
    out = scaler.scale(torch.tensor(0.5, device="cuda", dtype=torch.float16))
    assert out.dtype == torch.float32 and float(out) == 32768.0
    eng.state_destroy(sid)


def test_lazy_loss_values_and_order():
    """Stoke.loss launches the loss mean without synchronising; step_loss / ema_loss fold the queued values in order and
    equal the eagerly synchronised ones."""
    import stoke_b200 as sb
    from stoke_b200 import synthetic

    def make():
        return sb.Stoke(model=synthetic.basic_nn(), optimizer=sb.StokeOptimizer(optimizer=torch.optim.Adam,
                        optimizer_kwargs=synthetic.CFG1_ADAM), loss=torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32,
                        grad_accum_steps=2, gpu=True, verbose=False)

    a, b = make(), make()
    eager, lazy_last = [], None
    for x, y in synthetic.cfg1_batches(300):
        la = a.loss(a.model(x.cuda()), y.cuda())
        eager.append((a.step_loss, a.ema_loss))           # read every micro-step
        a.backward(la)
        a.step()
        lb = b.loss(b.model(x.cuda()), y.cuda())          # never read inside the loop (queue folds itself at 128)
        b.backward(lb)
        b.step()
    assert len(b._loss_queue) > 0
    assert (b.step_loss, b.ema_loss) == eager[-1]
    assert b._agg_loss == a._agg_loss


def test_close_releases_device_memory():
    from stoke_b200.engine import get_engine
    from stoke_b200.optim import B200FusedOptimizer

    class Big(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.ones(20_000_000))

    torch.cuda.set_device(0)
    eng = get_engine(0)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(3):
        net = Big().cuda()
        opt = B200FusedOptimizer(net, torch.optim.Adam, {"lr": 1e-3}, engine=eng, lp_dtype=torch.bfloat16)
        opt.close()
        assert net.w.dtype == torch.bfloat16 and float(net.w.float().sum()) == 20_000_000.0  # parameters survive close()
        del net, opt
    torch.cuda.empty_cache()
    assert free0 - torch.cuda.mem_get_info()[0] < 64 << 20

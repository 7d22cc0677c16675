"""CPU tests of the facade's own bookkeeping (accumulation cadence, loss tracking, EMA, wrap order) with a recording test
double in place of the runner -- the engine itself needs a GPU.  The expected values are the unmodified reference's
(tests/golden/cfg1_*.npz: counter trace; tests/golden/reference_traces.json: per-micro-step loss bookkeeping)."""
import hashlib
import json
import os
from contextlib import nullcontext

import numpy as np
import pytest
import torch

import stoke_b200 as sb
from stoke_b200 import status as status_mod
from stoke_b200 import stoke as facade
from stoke_b200 import synthetic


class FakeRunner:
    """Plays the runner's method set on CPU with plain torch (test double only)."""

    def __init__(self, optimizer_cls, kwargs, params, clip):
        self.calls = []
        self.opt = optimizer_cls(params, **kwargs)
        self.clip = clip
        self.scaler = None
        self.rank, self.world_size, self.engine = "gpu", 1, None
        self.model_context = nullcontext()
        self.loss_context = nullcontext()

    def setup_distributed(self): self.calls.append("setup")
    def wrap_distributed(self, model, grad_accum, optimizer=None): self.calls.append("wrap_dist"); return model, optimizer
    def wrap_fp16(self, model, optimizer=None): self.calls.append("wrap_fp16"); return model, optimizer
    def build_optimizer(self, optimizer, optimizer_kwargs, model): self.calls.append("build_opt"); return self.opt
    def detach_and_sync_loss(self, loss, device=None): return loss.item()
    def grad_accum_context(self, model): self.calls.append("no_sync"); return nullcontext()
    def step_context(self, optimizer): return nullcontext()
    def backward_call(self, loss, model, optimizer):
        self.calls.append("backward")
        if isinstance(loss, (list, tuple)):
            for idx, val in enumerate(loss):
                val.backward(retain_graph=(idx == 0))
        else:
            loss.backward()
    def clip_grad(self, grad_clip, model, optimizer, **kw):
        self.calls.append("clip")
        torch.nn.utils.clip_grad_norm_(model.parameters(), grad_clip.max_norm, grad_clip.norm_type)
    def step_call(self, model, optimizer): self.calls.append("step"); optimizer.step()
    def print_device(self, msg, rank=0, single_line=False): pass
    def barrier(self): pass


@pytest.fixture
def fake_stoke(monkeypatch):
    def make(model, accum, clip=None, optimizer=torch.optim.Adam, kwargs=None, loss=None):
        kwargs = synthetic.CFG1_ADAM if kwargs is None else kwargs
        holder = {}

        def fake_build(status, verbose, info_rank, loss, configs):
            holder["r"] = FakeRunner(optimizer, kwargs, list(model.parameters()), clip)
            return holder["r"], ["fake"]

        monkeypatch.setattr(facade, "build_runner", fake_build)
        monkeypatch.setattr(status_mod, "_cuda_available", lambda: True)
        monkeypatch.setattr(torch.nn.Module, "cuda", lambda self, device=None: self)
        s = sb.Stoke(model=model, optimizer=sb.StokeOptimizer(optimizer=optimizer, optimizer_kwargs=kwargs),
                     loss=loss if loss is not None else torch.nn.BCEWithLogitsLoss(), batch_size_per_device=32,
                     grad_accum_steps=accum,
                     grad_clip=clip, gpu=True, verbose=False)
        return s, holder["r"]
    return make


def test_counter_trace_and_weights_match_reference_fixture(fake_stoke, golden_dir):
    gold = np.load(os.path.join(golden_dir, "cfg1_clipnorm.npz"))
    model = synthetic.basic_nn()
    s, runner = fake_stoke(model, synthetic.CFG1_ACCUM, sb.ClipGradNormConfig(max_norm=0.05, norm_type=2.0))
    assert runner.calls[:4] == ["setup", "wrap_dist", "wrap_fp16", "build_opt"]  # model-then-optimizer order
    losses, trace = [], []
    for x, y in synthetic.cfg1_batches(synthetic.CFG1_OPT_STEPS * synthetic.CFG1_ACCUM):
        l = s.loss(s.model(x), y)
        losses.append(s.step_loss)
        s.backward(l)
        s.step()
        trace.append((s._grad_accum_counter, s._backward_steps, s._optimizer_steps))
    assert np.array_equal(np.asarray(trace), gold["trace"])
    assert np.array_equal(np.asarray(losses), gold["losses"])
    final = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    assert np.array_equal(final, gold["final"])
    per_step = [c for c in runner.calls[4:]]
    # every second backward runs under the no-sync context, clip precedes step
    assert per_step[:6] == ["no_sync", "backward", "backward", "clip", "step", "no_sync"]


def _reference_trace(golden_dir, name):
    with open(os.path.join(golden_dir, "reference_traces.json")) as f:
        return json.load(f)[name]


def test_loss_tracking_matches_live_reference(fake_stoke, golden_dir):
    rec = _reference_trace(golden_dir, "adam_accum3_ema03")
    m_new = synthetic.basic_nn(rec["model_seed"])
    s_new, _ = fake_stoke(m_new, rec["accum"])
    s_new._ema_weight = rec["ema_weight"]
    batches = list(synthetic.cfg1_batches(rec["batches"], seed=rec["batch_seed"]))
    assert len(batches) == len(rec["steps"])
    for (x, y), ref in zip(batches, rec["steps"]):
        l = s_new.loss(s_new.model(x), y)
        s_new.backward(l)
        s_new.step()
        assert ref["step_loss"] == s_new.step_loss
        assert ref["ema_loss"] == s_new.ema_loss
        assert ref["agg_loss"] == s_new._agg_loss
        assert ref["counters"] == [s_new._grad_accum_counter, s_new._backward_steps, s_new._optimizer_steps]
    m_new.eval()
    x, y = next(iter(synthetic.cfg1_batches(1)))
    assert torch.equal(s_new.loss(s_new.model(x), y), torch.nn.BCEWithLogitsLoss()(m_new(x), y))  # no /accum in eval


def test_constructor_errors(monkeypatch):
    monkeypatch.setattr(status_mod, "_cuda_available", lambda: True)
    opt = sb.StokeOptimizer(optimizer=torch.optim.Adam, optimizer_kwargs={})
    lin, mse = torch.nn.Linear(2, 2), torch.nn.MSELoss()
    with pytest.raises(TypeError):
        sb.Stoke("not a module", opt, mse, 4, gpu=True)
    with pytest.raises(TypeError):
        sb.Stoke(lin, opt, mse, 4, gpu=True, grad_clip=1.0)
    with pytest.raises(ValueError):
        sb.Stoke(lin, opt, mse, 4, gpu=True, distributed="horovod")
    with pytest.raises(ValueError):
        sb.Stoke(lin, opt, mse, 4, gpu=True, fp16="apex_O1")
    with pytest.raises(ValueError):  # SDDP requires OSS (reference status.py:239-243)
        sb.Stoke(lin, opt, mse, 4, gpu=True, distributed="ddp", fairscale_sddp=True)
    with pytest.raises(ValueError):  # OSS + clip-by-value (reference status.py:259-266)
        sb.Stoke(lin, opt, mse, 4, gpu=True, distributed="ddp", fairscale_oss=True,
                 grad_clip=sb.ClipGradConfig(clip_value=1.0))
    with pytest.raises(ValueError):  # fairscale needs ddp
        sb.Stoke(lin, opt, mse, 4, gpu=True, fairscale_oss=True)


def test_exports_cover_reference_names():
    expected = {"Stoke", "ParamNormalize", "FP16Options", "DistributedOptions", "StokeOptimizer", "ClipGradNormConfig",
                "ClipGradConfig", "FairscaleOSSConfig", "FairscaleSDDPConfig", "FairscaleFSDPConfig", "HorovodConfig",
                "ApexConfig", "DeepspeedConfig", "DDPConfig", "AMPConfig", "DeepspeedAIOConfig",
                "DeepspeedActivationCheckpointingConfig", "DeepspeedFlopsConfig", "DeepspeedFP16Config",
                "DeepspeedPLDConfig", "DeepspeedOffloadOptimizerConfig", "DeepspeedOffloadParamConfig",
                "DeepspeedTensorboardConfig", "DeepspeedZeROConfig", "BucketedDistributedSampler"}
    assert expected <= set(sb.__all__)
    for name in expected:
        assert hasattr(sb, name)


def test_multiple_losses_bookkeeping_matches_live_reference(fake_stoke, golden_dir):
    """List / tuple of loss callables (stoke/stoke.py:889-901): per-loss synced values, aggregated sums, EMA, the division by
    grad_accum, and the retain_graph backward over the list -- against the unmodified reference's run on CPU."""
    rec = _reference_trace(golden_dir, "multiple_losses")

    def losses():
        return [torch.nn.BCEWithLogitsLoss(), lambda out, y: ((out - y) ** 2).mean()]

    m_new = synthetic.basic_nn(rec["model_seed"])
    s_new, _ = fake_stoke(m_new, rec["accum"], loss=losses())
    batches = list(synthetic.cfg1_batches(rec["batches"], seed=rec["batch_seed"]))
    assert len(batches) == len(rec["steps"])
    for (x, y), ref in zip(batches, rec["steps"]):
        l = s_new.loss(s_new.model(x), y)
        assert isinstance(l, list) and len(l) == 2
        s_new.backward(l)
        s_new.step()
        assert ref["step_loss"] == s_new.step_loss
        assert ref["agg_loss"] == s_new._agg_loss
        assert ref["ema_loss"] == s_new.ema_loss
    b = torch.cat([p.detach().reshape(-1) for p in m_new.parameters()]).numpy()
    assert hashlib.sha256(np.ascontiguousarray(b, dtype="<f4").tobytes()).hexdigest() == rec["final_sha256"]


def test_lazy_loss_queue_folds_in_order(fake_stoke):
    """With a runner that offers ``sync_loss_begin`` / ``sync_loss_wait`` (the engine's pinned ring) ``Stoke.loss`` only queues
    tickets; ``step_loss`` / ``ema_loss`` / the accumulated loss fold them in order -- including the accumulated-loss resets
    that ``step()`` interleaves -- and equal the eager bookkeeping."""
    def run(lazy):
        model = synthetic.basic_nn()
        s, runner = fake_stoke(model, 3)
        waits = []
        if lazy:
            store = {}
            runner.sync_loss_begin = lambda loss: store.setdefault(len(store), loss.item()) and len(store) - 1 or len(store) - 1
            runner.sync_loss_wait = lambda t: (waits.append(t), store[t])[1]
        seen = []
        for i, (x, y) in enumerate(synthetic.cfg1_batches(200)):
            l = s.loss(s.model(x), y)
            s.backward(l)
            s.step()
            if not lazy or i % 50 == 49:
                seen.append((i, s.step_loss, s.ema_loss, s._agg_loss))
        return s, seen, waits

    s_eager, eager, _ = run(False)
    s_lazy, lazy, waits = run(True)
    assert waits == sorted(waits) and len(waits) == 200            # every ticket waited once, in order
    by_step = {i: rest for i, *rest in eager}
    for i, *rest in lazy:
        assert rest == by_step[i]
    assert s_lazy._rolling_loss_steps == s_eager._rolling_loss_steps == 200

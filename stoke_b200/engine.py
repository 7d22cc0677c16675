# -*- coding: utf-8 -*-
"""Host side of the B200 gradient-path engine: one ``Engine`` per process (one process per GPU) owning the C-ABI
context, the peer-visible flat buffers and the launch bookkeeping, and one ``GradPath`` per model that lays the model's
parameters / gradients / optimizer state out in those flat buffers and drives K1 (reduce) and K2 (optimizer step).

torch is used here for what it is good at -- tensors as typed views of device memory, streams, autograd, and
``torch.distributed`` for process-group bring-up (rank/world discovery, the one-time exchange of memory handles and the
initial parameter broadcast).  Every byte of the per-step gradient path moves through the hand-written kernels in
``csrc/``; if the library is missing or a call fails this module raises -- there is no torch fallback.

Routes of one optimizer step (``GradPath.route``):

  ``local``    world == 1.  ``k_grad_norm`` (only when a norm / inf verdict is needed) reads the raw bucket once; the fused
               step reads it again -- from L2 when it fits -- scales, updates and zeroes it.  No fp32 main-grad copy.
  ``sharded``  world > 1 (default under DDP, and what ``fairscale_oss`` asks for).  Per gradient bucket, launched from
               autograd hooks while backward is still running: K1 reduce-scatter over peer memory (owner sums its shard
               of the bucket from all W ranks, fused 1/W, unscale, inf test, norm partial, bucket zeroing).  After backward:
               ONE sharded K2 over the concatenation of this rank's shards, which pushes the updated low-precision
               parameters to every rank (parameter all-gather inside the kernel).  4 bytes per element on the wire.
  ``allreduce`` world > 1, replicated optimizer state (``STK_DDP_SHARD=0``, or the stock-optimizer route): K1 all-reduce
               per bucket into fp32 main grads on every rank, then a local K2.  6 bytes per element on the wire.
  ``main``     world == 1 with materialised fp32 main grads (K1's W == 1 form + K2): what the stock-optimizer route and a
               few tests use.
"""
import ctypes as C
import os
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, layout
from ._lib import StokeB200Error, check

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
_ESZ = {torch.float32: 4, torch.bfloat16: 2, torch.float16: 2}
ALIGN_ELEMS = layout.ALIGN_ELEMS  # every parameter starts on a 16-element boundary (32 B of bf16 / 64 B of fp32)
DEFAULT_BUCKET_MB = 25.0  # DDPConfig.bucket_cap_mb of the reference (stoke/configs.py:178-188)


class DeviceBuffer:
    """A device allocation owned by the library, mapped into every peer (VMM / CUDA IPC) when world > 1."""

    def __init__(self, engine: "Engine", ptr: int, nbytes: int, peers: List[int], mc_ptr: Optional[int] = None):
        self.engine, self.ptr, self.nbytes, self.peers, self.mc_ptr = engine, ptr, nbytes, peers, mc_ptr
        self.__cuda_array_interface__ = {
            "shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None,
        }

    def tensor(self, dtype: torch.dtype, numel: Optional[int] = None, offset_elems: int = 0) -> torch.Tensor:
        raw = torch.as_tensor(self, device=torch.device("cuda", self.engine.device))
        t = raw.view(dtype)
        if numel is None:
            numel = t.numel() - offset_elems
        return t[offset_elems: offset_elems + numel]

    def peer_ptrs(self, offset_bytes: int = 0) -> List[int]:
        return [p + offset_bytes for p in self.peers]


class Engine:
    """Process-wide handle on libstoke_b200 (context + signal pads)."""

    def __init__(self, device: int, rank: int = 0, world: int = 1, group=None):
        if not torch.cuda.is_available():
            raise StokeB200Error(_lib.ERR_CUDA, "no CUDA device: stoke_b200 has no CPU path")
        self.lib = _lib.load()
        self.device, self.rank, self.world, self.group = int(device), int(rank), int(world), group
        self._buffers: List[DeviceBuffer] = []
        self.launches = 0  # kernels launched through this engine (bench.py reports it as gpu_launches)
        self._cur_state = 0
        ctx = C.c_void_p()
        check(self.lib.stk_ctx_create(self.rank, self.world, self.device, 0, C.byref(ctx)))
        self.ctx = ctx
        handle = C.create_string_buffer(_lib.STK_IPC_HANDLE_BYTES)
        self._check(self.lib.stk_comm_local(self.ctx, handle))
        handles = self._exchange(handle.raw)
        self._check(self.lib.stk_comm_connect(self.ctx, handles))
        if self.world > 1:
            torch.distributed.barrier(group=self.group)  # every pad is zeroed and mapped before the first kernel
        caps = _lib.Caps()
        self._check(self.lib.stk_caps(self.ctx, C.byref(caps)))
        self.sm_count = caps.sm_count
        self.multicast = bool(caps.multicast)
        self.mem_mode = self.option_get(_lib.OPT_MEM_MODE)
        if self.world > 1 and self.mem_mode == 1:
            self._probe_vmm()

    # -- plumbing ---------------------------------------------------------------------------------------------------
    def _check(self, code):
        check(code, self.ctx)

    def _stream(self, stream=None) -> int:
        return (stream or torch.cuda.current_stream(self.device)).cuda_stream

    def _exchange(self, blob: bytes) -> bytes:
        if self.world == 1:
            return blob
        out = [None] * self.world
        torch.distributed.all_gather_object(out, blob, group=self.group)
        return b"".join(out)

    def _all_ok(self, ok: bool) -> bool:
        """True iff ``ok`` on every rank (bring-up only)."""
        if self.world == 1:
            return ok
        flags = [None] * self.world
        torch.distributed.all_gather_object(flags, bool(ok), group=self.group)
        return all(flags)

    def option_get(self, key: int) -> int:
        v = C.c_int()
        self._check(self.lib.stk_option_get(self.ctx, key, C.byref(v)))
        return v.value

    def option_set(self, key: int, value: int):
        self._check(self.lib.stk_option_set(self.ctx, key, int(value)))

    def _probe_vmm(self):
        """One trial allocation through the VMM back end (cuMemCreate + descriptor passing between the rank processes).
        If ANY rank cannot do it (sandboxed sockets, driver quirks) every rank falls back to cudaMalloc + CUDA IPC --
        peer memory keeps working, only the NVLS multicast flavour is lost."""
        ok, why = True, ""
        try:
            buf = self._alloc_raw(1 << 20)
        except StokeB200Error as e:
            ok, why, buf = False, str(e), None
        all_ok = self._all_ok(ok)
        if buf is not None and ok:
            try:
                self.free(buf)
            except StokeB200Error:
                pass
        if not all_ok:
            if self.rank == 0:
                print(f"stoke_b200: VMM peer memory unavailable ({why or 'a peer failed'}); using CUDA IPC (no NVLS)")
            self.option_set(_lib.OPT_MEM_MODE, 0)
            self.mem_mode, self.multicast = 0, False

    def _alloc_raw(self, nbytes: int) -> DeviceBuffer:
        """alloc + exchange + open.  A local failure still takes part in the exchange (no rank is left hanging)."""
        nbytes = max(int(nbytes), 256)
        ptr = C.c_void_p()
        handle = C.create_string_buffer(_lib.STK_IPC_HANDLE_BYTES)
        err = None
        code = self.lib.stk_mem_alloc_shared(self.ctx, nbytes, C.byref(ptr), handle)
        if code != 0:
            err = StokeB200Error(code, (self.lib.stk_last_error(self.ctx) or b"alloc failed").decode())
        handles = self._exchange(handle.raw)
        if not self._all_ok(err is None):
            if err is None:
                self.lib.stk_mem_free_shared(self.ctx, ptr)
                err = StokeB200Error(_lib.ERR_CUDA, "a peer rank failed to allocate peer-visible memory")
            raise err
        peers = (C.c_void_p * _lib.STK_MAX_WORLD)()
        code = self.lib.stk_mem_open_peers(self.ctx, ptr, handles, peers)
        if code != 0:
            err = StokeB200Error(code, (self.lib.stk_last_error(self.ctx) or b"open failed").decode())
        if not self._all_ok(err is None):
            self.lib.stk_mem_free_shared(self.ctx, ptr)
            raise err or StokeB200Error(_lib.ERR_CUDA, "a peer rank failed to map peer-visible memory")
        return DeviceBuffer(self, ptr.value, nbytes, [peers[r] for r in range(self.world)])

    def alloc(self, nbytes: int, multicast: bool = False) -> DeviceBuffer:
        """Peer-visible buffer.  ``multicast=True`` additionally tries to bind it to an NVSwitch multicast object
        (``buf.mc_ptr``; None when the device / driver / memory mode has no NVLS -- the buffer works either way)."""
        buf = self._alloc_raw(nbytes)
        if multicast and self.world > 1 and self.multicast:
            torch.distributed.barrier(group=self.group)  # every rank has added its device to the multicast object
            mc = C.c_void_p()
            code = self.lib.stk_multicast_try_bind(self.ctx, buf.ptr, C.byref(mc))
            if self._all_ok(code == 0):
                buf.mc_ptr = mc.value
            elif code == 0:
                self.lib.stk_multicast_release(self.ctx, buf.ptr)
            torch.distributed.barrier(group=self.group)
        self._buffers.append(buf)
        return buf

    def free(self, buf: DeviceBuffer):
        if buf is None or buf.ptr is None or self.ctx is None:
            return
        self._check(self.lib.stk_mem_free_shared(self.ctx, buf.ptr))
        if buf in self._buffers:
            self._buffers.remove(buf)
        buf.ptr = None

    def shard_range(self, n: int, rank: Optional[int] = None) -> Tuple[int, int]:
        b, e = C.c_size_t(), C.c_size_t()
        check(self.lib.stk_shard_range(n, self.world, self.rank if rank is None else rank, C.byref(b), C.byref(e)))
        return b.value, e.value

    def close(self):
        if getattr(self, "ctx", None):
            torch.cuda.synchronize(self.device)
            self.lib.stk_ctx_destroy(self.ctx)
            self.ctx = None

    # -- per-optimizer state ----------------------------------------------------------------------------------------
    def state_create(self) -> int:
        sid = C.c_int()
        self._check(self.lib.stk_state_create(self.ctx, C.byref(sid)))
        return sid.value

    def state_select(self, sid: int):
        if sid != self._cur_state:
            self._check(self.lib.stk_state_select(self.ctx, sid))
            self._cur_state = sid

    def state_destroy(self, sid: int):
        if self.ctx is not None and sid > 0:
            self.lib.stk_state_destroy(self.ctx, sid)
            if self._cur_state == sid:
                self._cur_state = 0

    # -- scaler / step state (of the selected state) -------------------------------------------------------------------
    def scaler_get(self, state: Optional[int] = None) -> _lib.ScalerState:
        if state is not None:
            self.state_select(state)
        st = _lib.ScalerState()
        self._check(self.lib.stk_scaler_get(self.ctx, C.byref(st), self._stream()))
        return st

    def scaler_set(self, state: Optional[int] = None, **fields):
        st = self.scaler_get(state)
        for k, v in fields.items():
            setattr(st, k, v)
        self._check(self.lib.stk_scaler_set(self.ctx, C.byref(st), self._stream()))

    def scale_tensor(self, state: Optional[int] = None) -> torch.Tensor:
        """0-dim float32 view of the live loss scale on the device (``scaler.scale(loss)`` multiplies by it)."""
        if state is not None:
            self.state_select(state)
        ptr = self.lib.stk_scaler_scale_ptr(self.ctx)

        class _V:
            pass

        v = _V()
        v.__cuda_array_interface__ = {"shape": (1,), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}
        v._keep = self
        return torch.as_tensor(v, device=torch.device("cuda", self.device))[0]

    # -- kernels ----------------------------------------------------------------------------------------------------
    def grad_accumulate(self, grad_ptr: int, dtype: torch.dtype, acc_ptr: int, n: int, first: bool, zero_grad: bool):
        self._check(self.lib.stk_grad_accumulate(self.ctx, grad_ptr, _DT[dtype], acc_ptr, n, int(first), int(zero_grad),
                                                 self._stream()))
        self.launches += 1

    def grad_reduce(self, mode: int, grad_ptrs: Sequence[int], grad_dtype: torch.dtype,
                    acc_ptrs: Optional[Sequence[int]], out_ptrs: Sequence[int], out_dtype: torch.dtype, n: int,
                    mul: float, norm_kind: int, norm_p: float, flags: int, stream=None):
        acc = _lib.ptr_array(acc_ptrs) if acc_ptrs is not None else None
        self._check(self.lib.stk_grad_reduce(self.ctx, mode, _lib.ptr_array(grad_ptrs), _DT[grad_dtype], acc,
                                             _lib.ptr_array(out_ptrs), _DT[out_dtype], n, mul, norm_kind, norm_p, flags,
                                             self._stream(stream)))
        self.launches += 1

    def grad_norm(self, grad_ptr: int, dtype: torch.dtype, acc_ptr: Optional[int], n: int, mul: float, norm_kind: int,
                  norm_p: float, flags: int):
        self._check(self.lib.stk_grad_norm(self.ctx, grad_ptr, _DT[dtype], acc_ptr, n, mul, norm_kind, norm_p, flags,
                                           self._stream()))
        self.launches += 1

    def grad_scale(self, grad_ptr: int, n: int, clip_kind: int, max_norm: float, clip_value: float):
        self._check(self.lib.stk_grad_scale(self.ctx, grad_ptr, n, clip_kind, max_norm, clip_value, self._stream()))
        self.launches += 1

    def optim_step_ex(self, args: _lib.OptimArgs):
        self._check(self.lib.stk_optim_step_ex(self.ctx, C.byref(args), self._stream()))
        self.launches += 1

    def step_epilogue(self):
        self._check(self.lib.stk_step_epilogue(self.ctx, self._stream()))
        self.launches += 1

    def loss_sync(self, loss: torch.Tensor) -> float:
        """Mean over ranks of a scalar device tensor, as a python float (one stream synchronise)."""
        if loss.dtype not in _DT:
            loss = loss.float()
        out = C.c_double()
        self._check(self.lib.stk_loss_sync(self.ctx, loss.data_ptr(), _DT[loss.dtype], C.byref(out), self._stream()))
        self.launches += 1
        return out.value

    def loss_sync_begin(self, loss: torch.Tensor) -> int:
        """Launches the loss mean and returns a ticket; no host synchronisation (``loss_sync_wait`` reads the value)."""
        if loss.dtype not in _DT:
            loss = loss.float()
        ticket = C.c_int64()
        self._check(self.lib.stk_loss_sync_begin(self.ctx, loss.data_ptr(), _DT[loss.dtype], C.byref(ticket), self._stream()))
        self.launches += 1
        return ticket.value

    def loss_sync_wait(self, ticket: int) -> float:
        out = C.c_double()
        self._check(self.lib.stk_loss_sync_wait(self.ctx, ticket, C.byref(out)))
        return out.value

    def barrier(self):
        self._check(self.lib.stk_barrier(self.ctx, self._stream()))
        self.launches += 1 if self.world > 1 else 0

    def bcast(self, buf: DeviceBuffer, nbytes: int, root: int = 0, offset_bytes: int = 0):
        if self.world == 1:
            return
        self._check(self.lib.stk_bcast(self.ctx, _lib.ptr_array(buf.peer_ptrs(offset_bytes)), nbytes, root, self._stream()))
        self.launches += 1

    def set_k1_algo(self, algo: str):
        """Cross-rank K1 flavour: "ldg" (register-staged 16-byte loads), "bulk" (bulk-async copies through shared
        memory) or "nvls" (multimem over NVSwitch multicast; needs multicast-bound buffers, else falls back to bulk)."""
        self.option_set(_lib.OPT_K1_ALGO, {"ldg": 0, "bulk": 1, "nvls": 2}[algo])

    def profile(self, on: bool):
        """Brackets K1 / K2 / accumulate / norm launches with CUDA events inside the library (for bench.py's roofline)."""
        self._check(self.lib.stk_profile_enable(self.ctx, int(on)))

    def profile_read(self, kind: int):
        """(total ms, launches) since the last read for kind 0 = K1, 1 = K2, 2 = accumulate, 3 = norm pass."""
        ms, n = C.c_double(), C.c_int()
        self._check(self.lib.stk_profile_read(self.ctx, kind, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def profile_read_k1_device(self):
        """(ms of K1's barrier-to-barrier NVLink phase, launches, ms of the bucket-zeroing tail) from the device timer."""
        ms, n, z = C.c_double(), C.c_int(), C.c_double()
        self._check(self.lib.stk_profile_read_k1_device(self.ctx, C.byref(ms), C.byref(n), C.byref(z), self._stream()))
        return ms.value, n.value, z.value

    def profile_read_k2_device(self):
        """(ms between the sharded step's start and end barriers, launches) from the device timer."""
        ms, n = C.c_double(), C.c_int()
        self._check(self.lib.stk_profile_read_k2_device(self.ctx, C.byref(ms), C.byref(n), self._stream()))
        return ms.value, n.value

    def comm_check(self):
        self._check(self.lib.stk_comm_check(self.ctx, self._stream()))

    def comm_poll(self):
        """Non-blocking: raises STK_ERR_PEER if a kernel of this rank gave up waiting for a peer."""
        self._check(self.lib.stk_comm_poll(self.ctx))


_ENGINES: Dict[int, Engine] = {}


def get_engine(device: Optional[int] = None, rank: Optional[int] = None, world: Optional[int] = None, group=None) -> Engine:
    """One engine per (process, device).  Without an explicit rank / world the existing engine of the device is returned
    (a sampler or a kernel benchmark inside a DDP process shares the DDP engine); a new world-1 engine is only created
    when there is none."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    eng = _ENGINES.get(device)
    if eng is not None and eng.ctx is not None and (rank is None or (eng.rank == rank and eng.world == (world or 1))):
        return eng
    if eng is not None and eng.ctx is not None:
        eng.close()  # a different (rank, world) for this device: the old context is replaced, not leaked
    eng = Engine(device, rank or 0, world or 1, group)
    _ENGINES[device] = eng
    return eng


# ======================================================================================================================
class ClipSpec:
    """Gradient clipping folded into K1 (norm reduction) and K2 (scaling) -- ClipGradNormConfig / ClipGradConfig."""

    def __init__(self, kind: int = _lib.CLIP_NONE, max_norm: float = 0.0, norm_type: float = 2.0, clip_value: float = 0.0):
        self.kind, self.max_norm, self.norm_type, self.clip_value = kind, float(max_norm), float(norm_type), float(clip_value)

    @property
    def norm_kind(self) -> int:
        if self.kind != _lib.CLIP_NORM:
            return _lib.NORM_NONE
        if self.norm_type == 2.0:
            return _lib.NORM_L2
        if self.norm_type == float("inf"):
            return _lib.NORM_INF
        if self.norm_type <= 0:
            raise ValueError(f"Stoke -- unsupported norm_type {self.norm_type}")
        return _lib.NORM_P


class GradPath:
    """Flat-buffer layout of one model + the per-step launches.

    Layout (all flat, identical element offsets, every parameter 16-element aligned, ``n`` = padded total):

      P      model parameters, model dtype (bf16 | fp32)      peer-visible   what forward/backward read
      G      gradients, model dtype                            peer-visible   ``param.grad`` are views of this
      ACC    fp32 local accumulator (grad_accum > 1 only)      peer-visible
      MAIN   fp32 reduced / unscaled gradients                 peer-visible   owned shards (sharded) | all n (allreduce, main)
                                                                              | absent (local route)
      MASTER fp32 master weights                               local          aliases P when the model is fp32 and unsharded
      M, V   fp32 optimizer state                              local          owned shards (sharded) | all n

    Gradient buckets: contiguous element ranges cut at parameter boundaries, ``bucket_mb`` of gradient bytes each, in
    reverse registration order (what DDP does, torch/nn/parallel/distributed.py) -- bucket 0 holds the LAST parameters,
    whose gradients arrive first.  Every bucket is partitioned over the W ranks by ``stk_shard_range``; a rank's local state
    is the concatenation (by ascending element offset) of its shard of every bucket (``self.segs``).
    """

    def __init__(self, engine: Engine, params: Sequence[torch.nn.Parameter], grad_accum: int = 1,
                 clip: Optional[ClipSpec] = None, sharded: bool = False, lp_dtype: Optional[torch.dtype] = None,
                 module: Optional[torch.nn.Module] = None, sync_init: bool = True, needs_second_moment: bool = True,
                 needs_first_moment: bool = True, bucket_mb: Optional[float] = None, state_id: Optional[int] = None,
                 route: Optional[str] = None, group_of: Optional[Sequence[int]] = None, overlap: bool = True):
        self.engine = engine
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("Stoke -- model has no trainable parameters")
        dev = torch.device("cuda", engine.device)
        for p in self.params:
            if p.device != dev:
                raise ValueError(f"Stoke -- parameter on {p.device}, engine on {dev}")
            if p.dtype != torch.float32:
                raise TypeError("Stoke -- hand the engine an fp32 model; low precision is selected with fp16=...")
        self.grad_accum = max(1, int(grad_accum))
        self.clip = clip or ClipSpec()
        W = engine.world
        self.model_dtype = lp_dtype or torch.float32
        self.low_precision = self.model_dtype != torch.float32
        if route is None:
            if W == 1:
                route = "local"
            else:
                # DDP runs sharded internally unless told otherwise: 4 instead of 6 bytes per element on the wire, and the
                # update itself is 1/W of the work.  Replicated semantics are kept by state_dict() (all-gathers).
                route = "sharded" if (sharded or os.environ.get("STK_DDP_SHARD", "1") != "0") else "allreduce"
        if W == 1 and route in ("sharded", "allreduce"):
            route = "local"
        if route not in ("local", "main", "sharded", "allreduce"):
            raise ValueError(f"Stoke -- unknown engine route {route}")
        if W > 1 and route in ("local", "main"):
            raise ValueError("Stoke -- the local routes need world == 1")
        self.route = route
        self.sharded = route == "sharded"
        self.user_sharded = bool(sharded) and W > 1   # the user asked for OSS (reporting only)
        self.state_id = engine.state_create() if state_id is None else state_id
        self._own_state = state_id is None

        # ---- layout (planned by the pure-Python module layout.py, unit-tested on CPU) ----
        self.offsets, self.padded, self.n = layout.param_offsets([p.numel() for p in self.params])
        esz = _ESZ[self.model_dtype]

        # ---- buckets (launch order: reverse registration order) ----
        if bucket_mb is None:
            bucket_mb = float(os.environ.get("STK_BUCKET_MB", DEFAULT_BUCKET_MB))
        cap = max(int(bucket_mb * (1 << 20) / esz), ALIGN_ELEMS) if W > 1 else self.n
        # Overlap policy (STK_OVERLAP=auto|on|off).  A reduce launched from an autograd hook shares the GPU with the backward
        # kernels still running; measured on ResNet-50 (2 buckets of 25 MiB, profiles/scaling_r02.md) that costs more than the
        # ~30 us it hides, while one launch over the whole buffer after backward is also the most efficient shape for the
        # wire.  "auto" therefore buckets (and overlaps) only when there are at least 4 buckets' worth of gradients.
        mode = os.environ.get("STK_OVERLAP", "auto")
        nominal = (self.n + cap - 1) // cap
        if W > 1 and (not overlap or mode == "off" or (mode == "auto" and nominal < 4)):
            cap = self.n
        self.buckets: List[Tuple[int, int]] = layout.plan_buckets(self.offsets, self.n, cap)
        self.param_bucket = [0] * len(self.params)
        for k, (b0, b1) in enumerate(self.buckets):
            for i, o in enumerate(self.offsets):
                if b0 <= o < b1:
                    self.param_bucket[i] = k
        self.bucket_nparams = [self.param_bucket.count(k) for k in range(len(self.buckets))]

        # ---- segments: rank r's shard of every bucket, by ascending element offset ----
        self.segs_by_rank, self.n_local_by_rank = layout.plan_segments(
            self.buckets, W, self.sharded, shard_fn=lambda n_, w_, r_: engine.shard_range(n_, r_))
        self.segs = self.segs_by_rank[engine.rank]
        self.n_local = self.n_local_by_rank[engine.rank]
        self.n_local_max = max(self.n_local_by_rank)
        self.shard = (self.segs[0][0], self.segs[-1][1]) if self.segs else (0, 0)  # informational (single-bucket case)

        # ---- fp32 source values (rank 0's after the init sync: DDP's _sync_module_states) ----
        full32 = torch.zeros(self.n, dtype=torch.float32, device=dev)
        for p, o in zip(self.params, self.offsets):
            self._strided(full32, p, o).copy_(p.detach())
        if W > 1 and sync_init:
            torch.distributed.broadcast(full32, src=0, group=engine.group)  # bring-up only (NCCL)

        # ---- buffers ----
        nl = max(self.n_local, ALIGN_ELEMS)
        self._bufs: List[DeviceBuffer] = []

        def alloc(nbytes, multicast=False):
            b = engine.alloc(nbytes, multicast=multicast)
            self._bufs.append(b)
            return b

        self.P = alloc(self.n * esz, multicast=W > 1)
        self.G = alloc(self.n * esz, multicast=W > 1)
        self.ACC = alloc(self.n * 4) if self.grad_accum > 1 else None
        self.MAIN = alloc(nl * 4, multicast=(route == "allreduce")) if route != "local" else None
        separate_master = self.low_precision or self.sharded
        self.MASTER = alloc(nl * 4) if separate_master else None
        self.M = alloc(nl * 4) if needs_first_moment else None
        self.V = alloc(nl * 4) if needs_second_moment else None

        self.p_flat = self.P.tensor(self.model_dtype, self.n)
        self.g_flat = self.G.tensor(self.model_dtype, self.n)
        self.main_flat = self.MAIN.tensor(torch.float32, self.n_local) if self.MAIN else None
        self.m_flat = self.M.tensor(torch.float32, self.n_local) if self.M else None
        self.v_flat = self.V.tensor(torch.float32, self.n_local) if self.V else None
        self.p_flat.copy_(full32)  # round-to-nearest-even, same as the kernel's cast
        if separate_master:
            self.master_flat = self.MASTER.tensor(torch.float32, self.n_local)
            self.scatter_local(full32, self.master_flat)
            self.master_ptr = self.MASTER.ptr
        else:
            self.master_flat = self.p_flat
            self.master_ptr = self.P.ptr
        del full32

        # ---- parameter groups / unused parameters: the range table of the fused step ----
        self.group_of = list(group_of) if group_of is not None else [0] * len(self.params)
        ends = np.cumsum(np.asarray(self.padded, dtype=np.int64)) // 8
        self._range_end = torch.from_numpy(ends.astype(np.uint32).view(np.int32)).to(dev)
        self._range_group = torch.tensor(self.group_of, dtype=torch.uint8).to(dev)
        self._range_skip_live = False   # the device table currently carries skip bits
        self._range_steps = None        # int32 per parameter once per-parameter step counts are on (enable_per_param_steps)
        self._range_bc = None
        self._touched = np.ones(len(self.params), dtype=bool)
        self._track_touched = False

        # ---- re-point the module at the flat buffers ----
        if self.low_precision and module is not None:
            module.to(self.model_dtype)  # buffers (and any frozen parameter) follow the model dtype
        self.grad_views = []
        for p, o in zip(self.params, self.offsets):
            p.data = self._strided(self.p_flat, p, o)
            gv = self._strided(self.g_flat, p, o)
            p.grad = gv
            self.grad_views.append(gv)
        self._micro = 0
        self._raw_has_acc = False
        self._bucket_tabs = {}
        # ---- autograd hooks: per-bucket launches while backward runs, and unused-parameter detection ----
        self.overlap = bool(overlap) and W > 1 and len(self.buckets) > 1
        self._comm_stream = torch.cuda.Stream(engine.device) if self.overlap else None
        self._hooks = []
        self._armed = False          # hooks launch K1 for this backward
        self._arm_unscale = False
        self._pending = None
        self._next_bucket = 0
        self._seen = None
        ref = weakref.ref(self)
        for idx, p in enumerate(self.params):
            self._hooks.append(p.register_post_accumulate_grad_hook(self._make_hook(ref, idx)))
        self._closed = False
        torch.cuda.synchronize(engine.device)
        if W > 1:
            torch.distributed.barrier(group=engine.group)

    # -- layout helpers -----------------------------------------------------------------------------------------------
    @staticmethod
    def _strided(flat: torch.Tensor, like: torch.Tensor, offset: int) -> torch.Tensor:
        if like.is_contiguous():
            return flat[offset: offset + like.numel()].view(like.shape)
        return torch.as_strided(flat, like.shape, like.stride(), storage_offset=flat.storage_offset() + offset)

    def scatter_local(self, full: torch.Tensor, local: torch.Tensor):
        """local <- this rank's segments of a full-length vector."""
        for g0, g1, l0, _ in self.segs:
            local[l0: l0 + (g1 - g0)].copy_(full[g0:g1])

    @staticmethod
    def _make_hook(ref, idx):
        def hook(_param):
            self = ref()
            if self is not None:
                self._on_grad(idx)
        return hook

    # -- per-step API -------------------------------------------------------------------------------------------------
    def ensure_grad_views(self):
        """``zero_grad(set_to_none=True)`` from user code would detach the views; re-attach before backward."""
        for p, gv in zip(self.params, self.grad_views):
            if p.grad is not gv:
                p.grad = gv

    def begin_backward(self, sync: bool, unscale: bool, last: bool = True):
        """Arms the hooks for one ``loss.backward()``: they record which parameters receive a gradient and, on the
        synchronising micro-step of the cross-rank routes, launch K1 for each bucket as soon as it is complete
        (``last=False``: more backward calls follow in this micro-step -- several losses -- so nothing is launched yet)."""
        self.ensure_grad_views()
        if not self._track_touched:
            self._touched[:] = False
            self._track_touched = True
        self._armed = bool(sync) and bool(last) and self.overlap
        self._arm_unscale = bool(unscale)
        if self._armed:
            self._pending = list(self.bucket_nparams)
            self._seen = np.zeros(len(self.params), dtype=bool)
            self._next_bucket = 0

    def _on_grad(self, idx: int):
        self._touched[idx] = True
        if not self._armed or self._seen[idx]:
            return
        self._seen[idx] = True
        k = self.param_bucket[idx]
        self._pending[k] -= 1
        # in-order launches: the same sequence on every rank, whatever order autograd finishes the parameters in
        while self._next_bucket < len(self.buckets) - 1 and self._pending[self._next_bucket] == 0:
            self._launch_bucket(self._next_bucket, final=False, unscale=self._arm_unscale, side_stream=True)
            self._next_bucket += 1

    def _launch_bucket(self, k: int, final: bool, unscale: bool, side_stream: bool):
        e = self.engine
        b0, b1 = self.buckets[k]
        esz = _ESZ[self.model_dtype]
        has_acc = self.ACC is not None and self._micro > 0
        flags = _lib.RF_ZERO_INPUT | (_lib.RF_UNSCALE if unscale else 0) | (_lib.RF_FINAL if final else 0)
        if self.sharded:
            mine = [s for s in self.segs if s[3] == k]
            if mine:
                g0, _, l0, _ = mine[0]
                base = self.MAIN.ptr + (l0 - (g0 - b0)) * 4   # element v of the bucket lands at local l0 + (v - shard begin)
            else:
                base = self.MAIN.ptr                            # empty shard: nothing is written
            out_ptrs, mode = [base] * e.world, _lib.REDUCE_SCATTER
        else:
            out_ptrs, mode = self.MAIN.peer_ptrs(b0 * 4), _lib.REDUCE_ALL
        stream = None
        if side_stream and self._comm_stream is not None:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(e.device))
            self._comm_stream.wait_event(ev)
            stream = self._comm_stream
        e.state_select(self.state_id)
        # pointer tables per bucket are built once (the hooks run on the autograd thread: keep them short)
        key = (k, has_acc)
        tabs = self._bucket_tabs.get(key)
        if tabs is None:
            tabs = (_lib.ptr_array(self.G.peer_ptrs(b0 * esz)),
                    _lib.ptr_array(self.ACC.peer_ptrs(b0 * 4)) if has_acc else None, _lib.ptr_array(out_ptrs))
            self._bucket_tabs[key] = tabs
        e._check(e.lib.stk_grad_reduce(e.ctx, mode, tabs[0], _DT[self.model_dtype], tabs[1], tabs[2], _lib.F32, b1 - b0,
                                       1.0 / e.world, self.clip.norm_kind, self.clip.norm_type, flags, e._stream(stream)))
        e.launches += 1

    def after_backward(self, sync: bool, unscale: bool):
        """Called once per backward.  ``sync=False``: local accumulation (no_sync); ``sync=True``: the reduce of the
        route (buckets the hooks have not launched yet, in order; the last one finishes norm / found_inf)."""
        e, n = self.engine, self.n
        e.state_select(self.state_id)
        if not sync:
            if self.ACC is None:
                raise StokeB200Error(_lib.ERR_STATE, "backward without sync but the path was built with grad_accum == 1")
            e.grad_accumulate(self.G.ptr, self.model_dtype, self.ACC.ptr, n, first=(self._micro == 0), zero_grad=True)
            self._micro += 1
            self._armed = False
            return
        has_acc = self.ACC is not None and self._micro > 0
        if self.route == "local":
            # norm / inf verdict only when something consumes it; the fused step reads the raw bucket itself
            if self.clip.norm_kind != _lib.NORM_NONE or unscale:
                flags = _lib.RF_FINAL | (_lib.RF_UNSCALE if unscale else 0)
                e.grad_norm(self.G.ptr, self.model_dtype, self.ACC.ptr if has_acc else None, n, 1.0, self.clip.norm_kind,
                            self.clip.norm_type, flags)
            self._raw_has_acc = has_acc
        elif self.route == "main":
            flags = _lib.RF_FINAL | _lib.RF_ZERO_INPUT | (_lib.RF_UNSCALE if unscale else 0)
            e.grad_reduce(_lib.REDUCE_ALL, self.G.peer_ptrs(), self.model_dtype, self.ACC.peer_ptrs() if has_acc else None,
                          self.MAIN.peer_ptrs(), torch.float32, n, 1.0, self.clip.norm_kind, self.clip.norm_type, flags)
        else:
            start = self._next_bucket if self._armed else 0
            last = len(self.buckets) - 1
            for k in range(start, last + 1):
                self._launch_bucket(k, final=(k == last), unscale=unscale, side_stream=self._armed)
            if self._armed and self._comm_stream is not None:
                torch.cuda.current_stream(e.device).wait_stream(self._comm_stream)
        self._armed = False
        self._micro = 0

    # -- the fused step ---------------------------------------------------------------------------------------------------
    def _ranges_for_step(self):
        """(n_ranges, end_ptr, group_ptr) for K2: the table is only consulted when there are several parameter groups or
        some parameter received no gradient in this accumulation window (torch skips ``p.grad is None``)."""
        skip = self._track_touched and not bool(self._touched.all())
        multi = max(self.group_of) > 0
        if skip and self._range_steps is None:
            # From the first skipped parameter on, step counts are kept per parameter (torch: state[p]["step"]); until then
            # every parameter has taken exactly the optimizer-wide number of steps.
            self.enable_per_param_steps()
        if not skip and not multi and self._range_steps is None:
            return 0, None, None
        if skip or self._range_skip_live:
            tab = np.asarray(self.group_of, dtype=np.uint8) | np.where(self._touched | (not skip), 0, 0x80).astype(np.uint8)
            # pageable source: the runtime stages the bytes before returning, so the table may be rewritten next step
            self._range_group.copy_(torch.from_numpy(tab))
            self._range_skip_live = skip
        return len(self.params), self._range_end.data_ptr(), self._range_group.data_ptr()

    def enable_per_param_steps(self, steps: Optional[Sequence[int]] = None):
        """Switches the fused step to per-parameter step counts (one synchronisation to read the optimizer-wide count)."""
        dev = self._range_end.device
        if steps is None:
            done = int(self.engine.scaler_get(self.state_id).opt_steps)
            steps = [done] * len(self.params)
        self._range_steps = torch.tensor(list(steps), dtype=torch.int32, device=dev)
        self._range_bc = torch.zeros(len(self.params), 4, dtype=torch.float32, device=dev)

    def param_steps(self) -> List[int]:
        """Steps taken by every parameter (what torch reports as ``state[p]["step"]``)."""
        if self._range_steps is None:
            return [int(self.engine.scaler_get(self.state_id).opt_steps)] * len(self.params)
        return [int(v) for v in self._range_steps.cpu().tolist()]

    def optimizer_step(self, hypers):
        """One fused K2 launch (+ the one-thread epilogue).  ``hypers``: one ``OptimHyper`` or a list (one per group)."""
        e = self.engine
        e.state_select(self.state_id)
        if isinstance(hypers, _lib.OptimHyper):
            hypers = [hypers]
        ng = len(hypers)
        if ng > _lib.MAX_GROUPS:
            raise NotImplementedError(f"Stoke -- the fused step handles up to {_lib.MAX_GROUPS} parameter groups")
        harr = (_lib.OptimHyper * ng)(*hypers)
        harr[0].clip_kind = self.clip.kind
        harr[0].clip_max_norm = self.clip.max_norm
        harr[0].clip_value = self.clip.clip_value
        a = _lib.OptimArgs()
        a.hyper, a.n_groups = harr, ng
        a.master = self.master_ptr
        a.exp_avg = self.M.ptr if self.M else None
        a.exp_avg_sq = self.V.ptr if self.V else None
        a.n_local = self.n_local
        a.grid_n = self.n_local_max
        keep = [harr]
        if self.route == "local":
            a.grad, a.grad_dtype, a.grad_raw, a.grad_mul = self.G.ptr, _DT[self.model_dtype], 1, 1.0
            a.acc = self.ACC.ptr if self._raw_has_acc else None
        else:
            a.grad, a.grad_dtype, a.grad_raw = self.MAIN.ptr, _lib.F32, 0
        if self.sharded:
            lp = _lib.ptr_array(self.P.peer_ptrs())
            a.lp_ptrs, a.lp_world, a.lp_dtype = lp, e.world, _DT[self.model_dtype]
            ns = len(self.segs)
            sl = (C.c_size_t * (ns + 1))(*([s[2] for s in self.segs] + [self.n_local]))
            sg = (C.c_size_t * max(ns, 1))(*[s[0] for s in self.segs]) if ns else (C.c_size_t * 1)(0)
            a.n_seg, a.seg_local, a.seg_global = ns, sl, sg
            keep += [lp, sl, sg]
            if ns == 0:
                a.n_seg = 0
        elif self.low_precision:
            lp = _lib.ptr_array([self.P.ptr])
            a.lp_ptrs, a.lp_world, a.lp_dtype = lp, 1, _DT[self.model_dtype]
            keep.append(lp)
        else:
            a.lp_ptrs, a.lp_world, a.lp_dtype = None, 0, _lib.F32
        nr, rend, rgrp = self._ranges_for_step()
        a.n_ranges, a.range_end_vec, a.range_group = nr, rend, rgrp
        if nr and self._range_steps is not None:
            e._check(e.lib.stk_optim_range_prologue(e.ctx, harr, ng, nr, rgrp, self._range_steps.data_ptr(),
                                                    self._range_bc.data_ptr(), e._stream()))
            e.launches += 1
            a.range_bc = self._range_bc.data_ptr()
        e.optim_step_ex(a)
        e.step_epilogue()
        self._track_touched = False
        self._raw_has_acc = False
        e.comm_poll()  # a peer that went missing during this step surfaces here (no synchronisation)

    # -- inspection (tests, checkpoints) ----------------------------------------------------------------------------------
    def gather_master(self) -> torch.Tensor:
        """Full fp32 master vector (all-gathered across shards when sharded)."""
        if not self.sharded:
            return self.master_flat.float().clone() if self.master_flat.dtype != torch.float32 else self.master_flat.clone()
        return self._gather_shards(self.master_flat)

    def _gather_shards(self, local: torch.Tensor) -> torch.Tensor:
        """Full-length vector from every rank's local state (bring-up / checkpoint path: NCCL all-gather)."""
        e = self.engine
        pad = torch.zeros(max(self.n_local_max, 1), dtype=local.dtype, device=local.device)
        pad[: local.numel()] = local
        out = [torch.empty_like(pad) for _ in range(e.world)]
        torch.distributed.all_gather(out, pad, group=e.group)
        full = torch.zeros(self.n, dtype=local.dtype, device=local.device)
        for r in range(e.world):
            for g0, g1, l0, _ in self.segs_by_rank[r]:
                full[g0:g1] = out[r][l0: l0 + (g1 - g0)]
        return full

    def unflatten(self, flat: torch.Tensor) -> List[torch.Tensor]:
        return [self._strided(flat, p, o) for p, o in zip(self.params, self.offsets)]

    # -- teardown -----------------------------------------------------------------------------------------------------------
    def close(self):
        """Gives the model its parameters back in ordinary torch storage and frees the flat buffers (peer mappings,
        multicast bindings, the per-optimizer device state).  Collective in spirit: every rank should close its path at
        the same point of the program (peers must not be inside a kernel that reads this rank's buffers)."""
        if self._closed:
            return
        self._closed = True
        for h in self._hooks:
            h.remove()
        self._hooks = []
        e = self.engine
        if e.ctx is None:
            return
        torch.cuda.synchronize(e.device)
        with torch.no_grad():
            for p in self.params:
                p.data = p.data.clone()
                p.grad = None
        self.grad_views = []
        self.p_flat = self.g_flat = self.main_flat = self.m_flat = self.v_flat = self.master_flat = None
        for b in self._bufs:
            try:
                e.free(b)
            except StokeB200Error:
                pass
        self._bufs = []
        if self._own_state:
            e.state_destroy(self.state_id)

    def __del__(self):
        try:
            if not self._closed and self.engine.world == 1:
                self.close()  # single process: safe at any time; multi-rank paths are closed explicitly (Stoke.close)
        except Exception:  # noqa: BLE001 -- interpreter shutdown
            pass

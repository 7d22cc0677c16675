// k2_optim.cu -- K2: single-pass fused optimizer step (Adam / AdamW / SGD-momentum), plus the step epilogue.
//
// One sweep over (grad, master, exp_avg, exp_avg_sq) does what the reference spreads over clip_grad_norm_'s scaling pass /
// clip_grad_value_, GradScaler.step's inf gate, the ~7 foreach kernels of torch.optim.Adam and (mixed precision) the
// fp32 -> bf16 parameter cast; in sharded (OSS / ZeRO-1) mode the updated low-precision shard is stored straight into
// every rank's parameter buffer, which is the parameter all-gather (K3).  HBM bytes per element: read g,p,m,v (16) +
// write p,m,v (12) [+ 2 for the bf16 copy] = 28 / 30.  The clip coefficient, the skip decision and the bias corrections
// come from device memory, so there is no host synchronisation anywhere on the step.
//
// Gradient sources:  MAIN  -- fp32 reduced / unscaled gradients written by K1 (cross-rank routes), indexed like the state;
//                    RAW   -- the local model-dtype bucket itself (+ optional fp32 accumulator), scaled by mul and 1/scale
//                             here and zeroed after the read: the world == 1 route (k_grad_norm supplies norm / inf), which
//                             drops the 6 B/element fp32 main-grad round trip.
// Layout extras: segments (the local state is the concatenation of this rank's shard of every gradient bucket) and a range
// table over the flat index space selecting the parameter group (per-group lr / betas / eps / weight decay ...) or skipping
// parameters that received no gradient this step (torch skips `p.grad is None`, torch/optim/optimizer.py).
//
// Arithmetic follows torch/optim/adam.py (_single_tensor_adam, the path torch takes on CPU -- the oracle) and
// torch/optim/sgd.py (_single_tensor_sgd); the clip follows torch/nn/utils/clip_grad.py:165-174 (coef = max_norm /
// (total_norm + 1e-6), clamped to 1) and :291-292 (clamp).
#include "k1_common.cuh"

namespace stk {

struct GroupHyperD {   // host-side doubles, converted exactly like torch converts python scalars
  double lr, beta1, beta2, eps, weight_decay, momentum, dampening;
  int nesterov, maximize;
};
struct GroupHyperS {   // what the inner loop reads (shared memory, one entry per parameter group)
  float step_size, bc2_sqrt, b2, eps, wd, one_m_b1, one_m_b2, lr, one_m_damp, decay_mul, mom;
  int nesterov, maximize;
};

struct OptimParams {
  float* master;
  float* m;
  float* v;
  const void* grad;     // MAIN: float*, local indexing.  RAW: model-dtype bucket, global indexing
  const float* acc;     // RAW only
  size_t nvec;          // 8-float vector count of the local state
  PtrTable lp;          // low-precision / remote parameter destinations (bases; indexed globally)
  unsigned long long* prof_ns;  // optional {ns between the barriers, launches} (block 0), nullptr when off
  int lp_world;         // 0: none
  int lp_rank_skip;     // lp dtype == f32 and destination == master's own buffer: skip that rank (aliased)
  const stk_scaler_state_t* scaler;
  PeerPads pads;
  int rank, world;
  uint32_t epoch;
  int cross_rank;       // 1: start/end block barriers around the peer stores
  int kind, clip_kind;
  float clip_max_norm, clip_value;
  float grad_mul;       // RAW
  int unscale;          // RAW: multiply by 1/loss_scale
  int any_mom;          // SGD: some group has momentum != 0 (the buffer is written)
  int n_groups;
  GroupHyperD g[STK_MAX_GROUPS];
  int n_seg;                                 // >= 1
  uint32_t seg_local[STK_MAX_SEGMENTS + 1];  // vector units
  uint32_t seg_global[STK_MAX_SEGMENTS];     // vector units
  int n_ranges;                              // 0: group 0 everywhere
  const uint32_t* range_end;                 // device, ascending, vector units (global)
  const uint8_t* range_group;                // device; bit 7: skip
  const float4* range_bc;                    // device, optional: per-range {step_size, bc2_sqrt, first_step, 0}
};

// local vector index -> global vector index
__device__ __forceinline__ size_t to_global(const OptimParams& p, size_t i) {
  if (p.n_seg == 1) return p.seg_global[0] + (i - p.seg_local[0]);
  int lo = 0, hi = p.n_seg - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (p.seg_local[mid] <= i) lo = mid;
    else hi = mid - 1;
  }
  return p.seg_global[lo] + (i - p.seg_local[lo]);
}
// global vector index -> range index (first j with range_end[j] > gv)
__device__ __forceinline__ int range_of(const OptimParams& p, size_t gv) {
  int lo = 0, hi = p.n_ranges - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(&p.range_end[mid]) > gv) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}

template <int LP_DT, int VPT>  // -1: none, STK_BF16, STK_F32;  VPT vectors (8 elements each), adjacent in memory
__device__ __forceinline__ void store_lp(const OptimParams& p, size_t gv, const float (&x)[VPT][8], int nv) {
  if constexpr (LP_DT == STK_BF16) {
    uint4 u[VPT];
#pragma unroll
    for (int k = 0; k < VPT; ++k)
      u[k] = make_uint4(pack_bf16(x[k][0], x[k][1]), pack_bf16(x[k][2], x[k][3]), pack_bf16(x[k][4], x[k][5]),
                        pack_bf16(x[k][6], x[k][7]));
#pragma unroll 1
    for (int d = 0; d < p.lp_world; ++d) {
      const int dst = p.lp_world == 1 ? 0 : (p.rank + d) % p.lp_world;
      uint4* q = reinterpret_cast<uint4*>(p.lp.p[dst]) + gv;
      if (VPT == 2 && nv == 2) {
        // one 32-byte store: a full sector per posted peer write (two 16-byte halves run at half the NVLink rate)
        asm volatile("st.global.L1::no_allocate.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(q), "r"(u[0].x), "r"(u[0].y),
                     "r"(u[0].z), "r"(u[0].w), "r"(u[VPT - 1].x), "r"(u[VPT - 1].y), "r"(u[VPT - 1].z), "r"(u[VPT - 1].w)
                     : "memory");
      } else {
        st_stream16(q, u[0]);
      }
    }
  } else if constexpr (LP_DT == STK_F32) {
#pragma unroll 1
    for (int d = 0; d < p.lp_world; ++d) {
      const int dst = p.lp_world == 1 ? 0 : (p.rank + d) % p.lp_world;
      if (dst == p.lp_rank_skip) continue;
#pragma unroll
      for (int k = 0; k < VPT; ++k)
        if (k < nv) st_stream_f8(reinterpret_cast<float*>(p.lp.p[dst]) + (gv + k) * 8, x[k]);
    }
  }
}

// GRAD: STK_F32 with RAW = false -> MAIN.  RAW = true -> the raw bucket of dtype GRAD.
// PERSIST = false: one-shot launch, VPT vectors per thread (local step; measured ~14% faster than a persistent
// grid-stride loop on B200, tools/membench.cu).  PERSIST = true: co-resident grid-stride loop, required when the kernel
// pushes its shard to peers and therefore carries the cross-rank block barriers (sharded / OSS step).
template <int KIND, int LP_DT, bool PERSIST, int VPT, int GRAD, bool RAW>
__global__ void __launch_bounds__(256) k_optim_step(const OptimParams p) {
  __shared__ GroupHyperS s_g[STK_MAX_GROUPS];
  __shared__ int s_skip, s_first;
  __shared__ float s_inv_scale;
  if (PERSIST && p.cross_rank && !block_barrier_all_ranks(p.pads, p.rank, p.world, 0, p.epoch)) return;
  unsigned long long t_begin = 0;
  if (PERSIST && p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) t_begin = globaltimer_ns();

  const bool use_m = (KIND != STK_OPT_SGD) || p.m != nullptr;
  const size_t stride = PERSIST ? size_t(gridDim.x) * blockDim.x * VPT : 0;
  size_t i = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * VPT;

  float g[VPT][8], w[VPT][8], m[VPT][8], v[VPT][8];
  size_t gv = 0;
  int nv = 0;
  auto load = [&]() {
    // issue this thread's loads before the (serial, double-precision) bias-correction prologue so that the pow()
    // latency hides behind the memory latency: 32-byte loads (LDG.E.256), all in flight together
    nv = (i + VPT <= p.nvec) ? VPT : (i < p.nvec ? 1 : 0);
    if (nv == 0) return;
    gv = to_global(p, i);
#pragma unroll
    for (int k = 0; k < VPT; ++k)
      if (k < nv) {
        if constexpr (RAW) InVec<GRAD>::load(p.grad, gv + k, g[k]);
        else InVec<STK_F32>::load(p.grad, i + k, g[k]);
        InVec<STK_F32>::load(p.master, i + k, w[k]);
        if (use_m) InVec<STK_F32>::load(p.m, i + k, m[k]);
        if (KIND != STK_OPT_SGD) InVec<STK_F32>::load(p.v, i + k, v[k]);
      }
    if constexpr (RAW) {
      if (p.acc != nullptr) {
#pragma unroll
        for (int k = 0; k < VPT; ++k)
          if (k < nv) {
            float a[8];
            InVec<STK_F32>::load(p.acc, gv + k, a);
#pragma unroll
            for (int e = 0; e < 8; ++e) g[k][e] += a[e];
          }
      }
    }
  };
  load();

  if (threadIdx.x == 0) {
    s_skip = p.scaler->found_inf != 0;  // GradScaler.step: no optimizer.step() at all when any grad is inf/nan
    s_first = (p.scaler->opt_steps == 0) ? 1 : 0;  // SGD: first step seeds the momentum buffer with the gradient
    s_inv_scale = (RAW && p.unscale) ? (float)(1.0 / (double)p.scaler->scale) : 1.f;
  }
  if (threadIdx.x < (unsigned)p.n_groups) {
    const GroupHyperD& h = p.g[threadIdx.x];
    GroupHyperS o;
    // bias corrections in double, exactly as the python scalars in torch/optim/adam.py:531-547
    const double t = (double)(p.scaler->opt_steps + 1);
    o.step_size = 0.f;
    o.bc2_sqrt = 1.f;
    if (KIND != STK_OPT_SGD) {
      const double bc1 = 1.0 - pow(h.beta1, t);
      const double bc2 = 1.0 - pow(h.beta2, t);
      o.step_size = (float)(h.lr / bc1);
      o.bc2_sqrt = (float)sqrt(bc2);
    }
    o.b2 = (float)h.beta2;
    o.eps = (float)h.eps;
    o.wd = (float)h.weight_decay;
    o.one_m_b1 = (float)(1.0 - h.beta1);
    o.one_m_b2 = (float)(1.0 - h.beta2);
    o.lr = (float)h.lr;
    o.one_m_damp = (float)(1.0 - h.dampening);
    o.decay_mul = (float)(1.0 - h.lr * h.weight_decay);  // AdamW: param.mul_(1 - lr * wd)
    o.mom = (float)h.momentum;
    o.nesterov = h.nesterov;
    o.maximize = h.maximize;
    s_g[threadIdx.x] = o;
  }
  __syncthreads();
  const bool skip_all = s_skip != 0;
  const bool first_step = s_first != 0;
  float coef = 1.f;
  if (p.clip_kind == STK_CLIP_NORM) coef = fminf(p.clip_max_norm / (p.scaler->grad_norm + 1e-6f), 1.0f);
  const float cv = p.clip_value;
  const float inv_scale = s_inv_scale;

  while (nv > 0) {
    unsigned rb = 0;
    float4 bc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.n_ranges > 0) {  // the VPT vectors of a thread never straddle a parameter (16-element alignment)
      const int rj = range_of(p, gv);
      rb = __ldg(&p.range_group[rj]);
      if (p.range_bc != nullptr) bc = __ldg(&p.range_bc[rj]);
    }
    GroupHyperS h = s_g[rb & 0x7f];
    bool first_here = first_step;
    if (p.range_bc != nullptr) {  // per-parameter step counts (torch's `state[p]["step"]`)
      h.step_size = bc.x;
      h.bc2_sqrt = bc.y;
      first_here = bc.z != 0.f;
    }
    const bool skip = skip_all || (rb & 0x80u);
    if (!skip) {
#pragma unroll
      for (int k = 0; k < VPT; ++k) {
        if (k >= nv) continue;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float gg = g[k][e];
          if constexpr (RAW) {
            gg *= p.grad_mul;
            gg *= inv_scale;
          }
          if (p.clip_kind == STK_CLIP_NORM) gg *= coef;
          else if (p.clip_kind == STK_CLIP_VALUE) gg = fminf(fmaxf(gg, -cv), cv);
          if (h.maximize) gg = -gg;
          float ww = w[k][e];
          if (KIND == STK_OPT_ADAM || KIND == STK_OPT_ADAMW) {
            if (KIND == STK_OPT_ADAMW) ww *= h.decay_mul;
            else if (h.wd != 0.f) gg = fmaf(ww, h.wd, gg);          // grad.add(param, alpha=wd)
            float mm = m[k][e];
            mm = fmaf(h.one_m_b1, gg - mm, mm);                      // exp_avg.lerp_(grad, 1 - beta1)
            float vv = v[k][e] * h.b2;
            vv = fmaf(h.one_m_b2 * gg, gg, vv);                      // mul_(beta2).addcmul_(grad, grad, value=1-beta2)
            const float denom = sqrtf(vv) / h.bc2_sqrt + h.eps;
            ww = ww - h.step_size * (mm / denom);                    // addcdiv_(exp_avg, denom, value=-step_size)
            m[k][e] = mm;
            v[k][e] = vv;
          } else {  // SGD
            if (h.wd != 0.f) gg = fmaf(ww, h.wd, gg);
            if (h.mom != 0.f) {
              const float bb = first_here ? gg : fmaf(m[k][e], h.mom, h.one_m_damp * gg);
              m[k][e] = bb;
              gg = h.nesterov ? fmaf(bb, h.mom, gg) : bb;
            }
            ww = fmaf(-h.lr, gg, ww);
          }
          w[k][e] = ww;
        }
      }
#pragma unroll
      for (int k = 0; k < VPT; ++k)
        if (k < nv) {
          st_stream_f8(p.master + (i + k) * 8, w[k]);
          if (use_m && (KIND != STK_OPT_SGD || p.any_mom)) st_stream_f8(p.m + (i + k) * 8, m[k]);
          if (KIND != STK_OPT_SGD) st_stream_f8(p.v + (i + k) * 8, v[k]);
        }
      store_lp<LP_DT, VPT>(p, gv, w, nv);
    }
    if constexpr (RAW) {
      // the bucket is consumed (also on a skipped step): zero it for the next backward's in-place accumulation
#pragma unroll
      for (int k = 0; k < VPT; ++k)
        if (k < nv) InVec<GRAD>::zero(const_cast<void*>(p.grad), gv + k);
    }
    if (!PERSIST) break;
    i += stride;
    load();
  }
  if (PERSIST && p.cross_rank) block_barrier_all_ranks(p.pads, p.rank, p.world, 1, p.epoch);
  if (PERSIST && p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&p.prof_ns[0], globaltimer_ns() - t_begin);
    atomicAdd(&p.prof_ns[1], 1ull);
  }
}

struct RangePrologueParams {
  GroupHyperD g[STK_MAX_GROUPS];
  int n_ranges, kind;
  const uint8_t* range_group;
  int32_t* range_steps;
  float4* range_bc;
  const stk_scaler_state_t* scaler;
};

// one thread per range: bias corrections of that range's NEXT step (double, like the python scalars of torch/optim/adam.py)
// and the step count itself (torch increments state[p]["step"] only for parameters that are stepped)
__global__ void k_range_prologue(const RangePrologueParams p) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.n_ranges) return;
  const unsigned b = p.range_group[j];
  const GroupHyperD& h = p.g[b & 0x7f];
  const int32_t done = p.range_steps[j];
  const double t = (double)(done + 1);
  float4 o = make_float4(0.f, 1.f, done == 0 ? 1.f : 0.f, 0.f);
  if (p.kind != STK_OPT_SGD) {
    o.x = (float)(h.lr / (1.0 - pow(h.beta1, t)));
    o.y = (float)sqrt(1.0 - pow(h.beta2, t));
  }
  p.range_bc[j] = o;
  if (!(b & 0x80u) && p.scaler->found_inf == 0) p.range_steps[j] = done + 1;
}

// scaler.update() (torch/amp/grad_scaler.py:549-556 -> _amp_update_scale_), step counters, per-step accumulator reset
__global__ void k_step_epilogue(stk_scaler_state_t* st, StepAccum* acc) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const bool inf = st->found_inf != 0;
  if (inf) st->skipped_steps += 1;
  else st->opt_steps += 1;
  if (st->enabled) {
    if (inf) {
      st->scale = st->scale * st->backoff_factor;
      st->growth_tracker = 0;
    } else {
      int t = st->growth_tracker + 1;
      if (t == st->growth_interval) {
        float ns = st->scale * st->growth_factor;
        if (finitef(ns)) st->scale = ns;   // _amp_update_scale_: do not grow past the largest finite fp32
        t = 0;
      }
      st->growth_tracker = t;
    }
  }
  st->found_inf = 0;
  acc->norm_partial = 0.f;
  acc->found_inf = 0u;
}

}  // namespace stk

using namespace stk;

static size_t g_grid_nvec = 0;  // set under the context lock by stk_optim_step_ex (cross-rank launches only)

template <typename K>
static cudaError_t launch_one(stk_ctx* c, K kernel, const OptimParams& p, bool persist, int vpt, cudaStream_t s) {
  const size_t per_block = size_t(256) * vpt;
  const size_t nvec = (persist && g_grid_nvec) ? g_grid_nvec : p.nvec;  // same grid on every rank
  size_t grid = (nvec + per_block - 1) / per_block;  // one-shot: VPT vectors per thread
  if (grid < 1) grid = 1;
  if (persist) {  // co-resident grid-stride loop: at most two blocks per SM
    size_t res = (size_t)std::min(blocks_per_sm(c, kernel, 256), 2) * c->sm_count;
    if (res > (size_t)kMaxBlocks) res = kMaxBlocks;
    if (grid > res) grid = res;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(256);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (persist) coop_attr(cfg, attr);
  ProfScope prof(c, 1, s);
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

template <int KIND>
static cudaError_t launch_optim(stk_ctx* c, const OptimParams& p, int lp_dtype, int grad_dtype, bool raw, bool pair,
                                cudaStream_t s) {
  if (raw) {
    // raw route: local step only (world == 1)
    if (grad_dtype == STK_BF16 && p.lp_world == 1 && lp_dtype == STK_BF16)
      return launch_one(c, k_optim_step<KIND, STK_BF16, false, 1, STK_BF16, true>, p, false, 1, s);
    if (grad_dtype == STK_F32 && p.lp_world == 0)
      return launch_one(c, k_optim_step<KIND, -1, false, 1, STK_F32, true>, p, false, 1, s);
    return cudaErrorNotSupported;
  }
  if (p.cross_rank) {
    if (lp_dtype == STK_BF16) {
      if (pair) return launch_one(c, k_optim_step<KIND, STK_BF16, true, 2, STK_F32, false>, p, true, 2, s);
      return launch_one(c, k_optim_step<KIND, STK_BF16, true, 1, STK_F32, false>, p, true, 1, s);
    }
    return launch_one(c, k_optim_step<KIND, STK_F32, true, 1, STK_F32, false>, p, true, 1, s);
  }
  if (p.lp_world == 0) return launch_one(c, k_optim_step<KIND, -1, false, 1, STK_F32, false>, p, false, 1, s);
  if (lp_dtype == STK_BF16) return launch_one(c, k_optim_step<KIND, STK_BF16, false, 1, STK_F32, false>, p, false, 1, s);
  return launch_one(c, k_optim_step<KIND, STK_F32, false, 1, STK_F32, false>, p, false, 1, s);
}

extern "C" {

int stk_optim_step_ex(stk_ctx* c, const stk_optim_args_t* a, void* stream) {
  STK_REQUIRE(c, c && a && a->hyper && a->master && a->grad, "stk_optim_step_ex: NULL argument");
  STK_REQUIRE(c, a->n_groups >= 1 && a->n_groups <= STK_MAX_GROUPS, "stk_optim_step_ex: n_groups must be in [1, 8]");
  STK_REQUIRE(c, a->n_local % 8 == 0, "stk_optim_step_ex: n_local must be a multiple of 8");
  const stk_optim_hyper_t* h = a->hyper;
  STK_REQUIRE(c, h->kind >= STK_OPT_ADAM && h->kind <= STK_OPT_SGD, "stk_optim_step_ex: bad optimizer kind");
  STK_REQUIRE(c, h->kind == STK_OPT_SGD || (a->exp_avg && a->exp_avg_sq), "stk_optim_step_ex: Adam needs exp_avg and exp_avg_sq");
  bool any_mom = false;
  for (int gi = 0; gi < a->n_groups; ++gi) {
    STK_REQUIRE(c, h[gi].kind == h->kind, "stk_optim_step_ex: all groups must use the same optimizer kind");
    any_mom |= h[gi].momentum != 0.0;
  }
  STK_REQUIRE(c, !(h->kind == STK_OPT_SGD && any_mom && !a->exp_avg), "stk_optim_step_ex: SGD momentum needs a buffer");
  STK_REQUIRE(c, a->lp_ptrs == nullptr || a->lp_world == 1 || a->lp_world == c->world, "stk_optim_step_ex: lp_world must be 1 or world");
  STK_REQUIRE(c, a->lp_ptrs == nullptr || a->lp_dtype == STK_BF16 || a->lp_dtype == STK_F32, "stk_optim_step_ex: lp dtype");
  STK_REQUIRE(c, a->n_seg >= 0 && a->n_seg <= STK_MAX_SEGMENTS, "stk_optim_step_ex: too many segments");
  STK_REQUIRE(c, a->n_seg == 0 || (a->seg_local && a->seg_global), "stk_optim_step_ex: segment arrays are NULL");
  STK_REQUIRE(c, a->n_ranges == 0 || (a->range_end_vec && a->range_group), "stk_optim_step_ex: range arrays are NULL");
  STK_REQUIRE(c, !a->grad_raw || c->world == 1 || a->lp_world <= 1, "stk_optim_step_ex: the raw gradient route is local (no peer stores)");
  STK_REQUIRE(c, a->grad_raw || a->grad_dtype == STK_F32, "stk_optim_step_ex: reduced main gradients are fp32");
  if (a->n_local == 0 && !(a->lp_ptrs && a->lp_world > 1)) return STK_OK;
  const bool cross = a->lp_ptrs != nullptr && a->lp_world > 1;
  if (cross) {
    if (!c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_optim_step (sharded) before stk_comm_connect");
    STK_POLL(c);
  }
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);

  OptimParams p{};
  p.master = a->master;
  p.m = a->exp_avg;
  p.v = a->exp_avg_sq;
  p.grad = a->grad;
  p.acc = a->grad_raw ? a->acc : nullptr;
  p.nvec = a->n_local / 8;
  p.lp_world = a->lp_ptrs ? a->lp_world : 0;
  p.lp_rank_skip = -1;
  // segments (vector units); the plain call is one segment at lp_offset
  bool pair_ok = true;
  if (a->n_seg == 0) {
    STK_REQUIRE(c, a->lp_offset % 8 == 0, "stk_optim_step_ex: lp_offset must be a multiple of 8");
    p.n_seg = 1;
    p.seg_local[0] = 0;
    p.seg_local[1] = (uint32_t)p.nvec;
    p.seg_global[0] = (uint32_t)(a->lp_offset / 8);
    pair_ok = (p.seg_global[0] % 2) == 0;
  } else {
    p.n_seg = a->n_seg;
    for (int k = 0; k <= a->n_seg; ++k) {
      STK_REQUIRE(c, a->seg_local[k] % 8 == 0, "stk_optim_step_ex: segment bounds must be multiples of 8");
      p.seg_local[k] = (uint32_t)(a->seg_local[k] / 8);
      if (k < a->n_seg) {
        STK_REQUIRE(c, a->seg_global[k] % 8 == 0, "stk_optim_step_ex: segment offsets must be multiples of 8");
        p.seg_global[k] = (uint32_t)(a->seg_global[k] / 8);
        pair_ok &= (p.seg_local[k] % 2) == 0 && (p.seg_global[k] % 2) == 0;
      }
    }
    STK_REQUIRE(c, p.seg_local[0] == 0 && p.seg_local[a->n_seg] == p.nvec, "stk_optim_step_ex: segments must tile [0, n_local)");
  }
  for (int r = 0; r < p.lp_world; ++r) {
    STK_REQUIRE(c, a->lp_ptrs[r] != nullptr, "stk_optim_step_ex: NULL lp pointer");
    p.lp.p[r] = a->lp_ptrs[r];
    if (a->lp_dtype == STK_F32 && p.n_seg == 1 &&
        static_cast<char*>(a->lp_ptrs[r]) + size_t(p.seg_global[0]) * 32 == reinterpret_cast<char*>(a->master))
      p.lp_rank_skip = r;
  }
  p.prof_ns = (cross && c->profiling) ? c->prof_ns_dev + 4 : nullptr;
  p.scaler = c->scaler_dev;
  p.pads = c->pads;
  p.rank = c->rank;
  p.world = c->world;
  p.cross_rank = cross ? 1 : 0;
  p.epoch = p.cross_rank ? ++c->blk_epoch : 0;
  p.kind = h->kind;
  p.clip_kind = h->clip_kind;
  p.clip_max_norm = (float)h->clip_max_norm;
  p.clip_value = (float)h->clip_value;
  p.grad_mul = (float)a->grad_mul;
  p.unscale = 0;
  p.n_groups = a->n_groups;
  for (int gi = 0; gi < a->n_groups; ++gi) {
    GroupHyperD& o = p.g[gi];
    o.lr = h[gi].lr; o.beta1 = h[gi].beta1; o.beta2 = h[gi].beta2; o.eps = h[gi].eps; o.weight_decay = h[gi].weight_decay;
    o.momentum = h[gi].momentum; o.dampening = h[gi].dampening; o.nesterov = h[gi].nesterov; o.maximize = h[gi].maximize;
  }
  p.any_mom = any_mom ? 1 : 0;
  p.n_ranges = a->n_ranges;
  p.range_end = a->range_end_vec;
  p.range_group = a->range_group;
  p.range_bc = a->n_ranges > 0 ? reinterpret_cast<const float4*>(a->range_bc) : nullptr;
  if (a->grad_raw) {
    // 1/loss_scale is applied when the scaler is live; the device flag decides (enabled), so no host read
    p.unscale = 1;
  }

  cudaError_t err;
  const bool raw = a->grad_raw != 0;
  g_grid_nvec = cross ? (a->grid_n ? (a->grid_n + 7) / 8 : p.nvec) : 0;
  switch (h->kind) {
    case STK_OPT_ADAM: err = launch_optim<STK_OPT_ADAM>(c, p, a->lp_dtype, a->grad_dtype, raw, pair_ok, s); break;
    case STK_OPT_ADAMW: err = launch_optim<STK_OPT_ADAMW>(c, p, a->lp_dtype, a->grad_dtype, raw, pair_ok, s); break;
    default: err = launch_optim<STK_OPT_SGD>(c, p, a->lp_dtype, a->grad_dtype, raw, pair_ok, s); break;
  }
  if (err == cudaErrorNotSupported)
    return stk_fail(c, STK_ERR_UNSUPPORTED, "stk_optim_step_ex: this gradient dtype / parameter dtype pair has no raw route");
  if (err != cudaSuccess) return stk_fail(c, STK_ERR_CUDA, std::string("k_optim_step launch: ") + cudaGetErrorString(err));
  return STK_OK;
}

int stk_optim_step(stk_ctx* c, const stk_optim_hyper_t* h, float* master, float* exp_avg, float* exp_avg_sq,
                   const float* grad, size_t n_local, void* const* lp_ptrs, int lp_world, int lp_dtype, size_t lp_offset,
                   void* stream) {
  STK_REQUIRE(c, c && h && master && grad, "stk_optim_step: NULL argument");
  stk_optim_args_t a{};
  a.hyper = h;
  a.n_groups = 1;
  a.master = master;
  a.exp_avg = exp_avg;
  a.exp_avg_sq = exp_avg_sq;
  a.grad = grad;
  a.grad_dtype = STK_F32;
  a.n_local = n_local;
  a.lp_ptrs = lp_ptrs;
  a.lp_world = lp_world;
  a.lp_dtype = lp_dtype;
  a.lp_offset = lp_offset;
  return stk_optim_step_ex(c, &a, stream);
}

int stk_optim_range_prologue(stk_ctx* c, const stk_optim_hyper_t* h, int n_groups, int n_ranges, const uint8_t* range_group,
                             int32_t* range_steps, float* range_bc, void* stream) {
  STK_REQUIRE(c, c && h && range_group && range_steps && range_bc, "stk_optim_range_prologue: NULL argument");
  STK_REQUIRE(c, n_groups >= 1 && n_groups <= STK_MAX_GROUPS, "stk_optim_range_prologue: n_groups must be in [1, 8]");
  STK_REQUIRE(c, n_ranges >= 1, "stk_optim_range_prologue: no ranges");
  STK_REQUIRE(c, (reinterpret_cast<uintptr_t>(range_bc) & 15) == 0, "stk_optim_range_prologue: range_bc must be 16-byte aligned");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  RangePrologueParams p{};
  for (int gi = 0; gi < n_groups; ++gi) {
    GroupHyperD& o = p.g[gi];
    o.lr = h[gi].lr; o.beta1 = h[gi].beta1; o.beta2 = h[gi].beta2; o.eps = h[gi].eps; o.weight_decay = h[gi].weight_decay;
    o.momentum = h[gi].momentum; o.dampening = h[gi].dampening; o.nesterov = h[gi].nesterov; o.maximize = h[gi].maximize;
  }
  p.n_ranges = n_ranges;
  p.kind = h->kind;
  p.range_group = range_group;
  p.range_steps = range_steps;
  p.range_bc = reinterpret_cast<float4*>(range_bc);
  p.scaler = c->scaler_dev;
  k_range_prologue<<<(n_ranges + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

int stk_step_epilogue(stk_ctx* c, void* stream) {
  STK_REQUIRE(c, c != nullptr, "stk_step_epilogue: NULL ctx");
  STK_POLL(c);
  DeviceGuard g(c->device);
  k_step_epilogue<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(c->scaler_dev, c->accum_dev);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

}  // extern "C"

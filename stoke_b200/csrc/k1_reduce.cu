// k1_reduce.cu -- K1: the gradient path between backward and the optimizer step.
//
//   k_grad_accumulate : acc (+)= float(grad)                      (local micro-steps under no_sync; HBM-bound)
//   k_grad_reduce     : main = (sum over ranks of grad [+ acc]) * mul * inv_scale   for the shard this rank owns,
//                       pushed to every rank (all-reduce) or kept (reduce-scatter); fused inf/nan test and
//                       norm partial (sum g^2 | max |g| | sum |g|^p); last block finishes them across ranks.
//
// Replaces, in one pass: DDP bucket copy-in (/W), NCCL all-reduce, bucket copy-out, GradScaler.unscale_, and the two
// reduction passes of clip_grad_norm_ (see include/stoke_b200.h for reference file:line).
//
// Cross-rank protocol (world > 1): block b of every rank (1) start barrier: "my gradients are complete" (the kernel is
// stream-ordered after backward), (2) reads its vectors of the owned shard from all W peers over NVLink (16-byte loads,
// >= 8 in flight per thread), reduces in rank order in fp32 registers, and stores the result straight into every
// rank's main-grad buffer (posted 16-byte peer stores), (3) end barrier: all my reads of peer gradients and all my
// writes to peer buffers are done.  No staging buffer, no second pass: bus bytes per GPU and direction =
// (W-1)/W * n * (b_in + b_out).  All blocks are co-resident (cooperative launch) because they spin on peers.
#include "k1_common.cuh"

namespace stk {

// ---------------------------------------------------------------------------------------------------------------------
template <int IN_DT>
__global__ void __launch_bounds__(256) k_grad_accumulate(void* __restrict__ grad, float* __restrict__ acc, size_t nvec,
                                                         int first, int zero_grad) {
  // one vector per thread, one block per chunk: measured 10-15% faster than a persistent grid-stride loop on B200
  // (tools/membench.cu; profiles/membench_r01.md)
  const size_t v = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v < nvec) {
    float g[8];
    InVec<IN_DT>::load(grad, v, g);
    if (!first) {
      float a[8];
      InVec<STK_F32>::load(acc, v, a);
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] += a[i];
    }
    store_out<STK_F32>(acc, v, g);
    if (zero_grad) InVec<IN_DT>::zero(grad, v);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
template <int W>
struct Unroll {
  static constexpr int value = W == 1 ? 2 : (W == 2 ? 2 : 1);
};

// W_T: compile-time world size (1, 2, 4, 8) or 0 = runtime p.world
template <int IN_DT, int OUT_DT, int W_T>
__global__ void __launch_bounds__(W_T == 1 ? 256 : 512, W_T == 1 ? 6 : 1) k_grad_reduce(const ReduceParams p) {
  const int W = W_T ? W_T : p.world;
  constexpr int U = Unroll<W_T>::value;
  constexpr int WMAX = W_T ? W_T : kMaxWorld;
  const bool has_acc = p.acc.p[0] != nullptr;
  const bool zero_in = (p.flags & STK_RF_ZERO_INPUT) && W == 1;

  if (W > 1 && !block_barrier_all_ranks(p.pads, p.rank, W, 0, p.epoch)) return;  // peer missing: error word set
  // device-side timing of the data phase (after the start barrier = after the slowest rank has arrived, up to the end
  // barrier): the NVLink time of this launch without the cross-rank launch skew that host-side events include
  unsigned long long t_begin = 0;
  if (p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) t_begin = globaltimer_ns();

  float inv_scale = 1.f;
  if (p.flags & STK_RF_UNSCALE) inv_scale = (float)(1.0 / (double)p.scaler->scale);
  const float mul = p.mul;

  float part = 0.f;   // norm partial of this thread
  bool bad = false;   // saw inf/nan

  // W == 1 (local, HBM-bound): one-shot launch, each block owns U * blockDim contiguous vectors (no grid-stride loop:
  // 10-15% faster on B200, tools/membench.cu).  W > 1 (NVLink-bound, blocks spin on peers): persistent grid-stride.
  const size_t stride = (W_T == 1) ? size_t(blockDim.x) : size_t(gridDim.x) * blockDim.x;
  const size_t first = (W_T == 1) ? p.vec_begin + size_t(blockIdx.x) * blockDim.x * U + threadIdx.x
                                  : p.vec_begin + size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t step = (W_T == 1) ? ~size_t(0) / 2 : stride * U;
  for (size_t v0 = first; v0 < p.vec_end; v0 += step) {
    float g[U][WMAX][8];
    float a[U][8];
    // issue every load before the first use (latency over NVLink is ~2 us)
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t v = v0 + u * stride;
      if (v < p.vec_end) {
#pragma unroll
        for (int r = 0; r < WMAX; ++r)
          if (r < W) InVec<IN_DT>::load(p.grad.p[r], v, g[u][r]);
      }
    }
    if (has_acc) {
      // accumulators are summed per rank before the cross-rank sum: (g_r + acc_r) is what rank r's param.grad held
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const size_t v = v0 + u * stride;
        if (v < p.vec_end) {
#pragma unroll
          for (int r = 0; r < WMAX; ++r)
            if (r < W) {
              InVec<STK_F32>::load(p.acc.p[r], v, a[u]);
#pragma unroll
              for (int i = 0; i < 8; ++i) g[u][r][i] += a[u][i];
            }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t v = v0 + u * stride;
      if (v < p.vec_end) {
        float s[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float x = g[u][0][i];
#pragma unroll
          for (int r = 1; r < WMAX; ++r)
            if (r < W) x += g[u][r][i];
          x *= mul;
          bad |= !finitef(x);
          x *= inv_scale;
          s[i] = x;
          if (p.norm_kind == STK_NORM_L2) part = fmaf(x, x, part);
          else if (p.norm_kind == STK_NORM_INF) part = fmaxf(part, fabsf(x));
          else if (p.norm_kind == STK_NORM_P) part += __powf(fabsf(x), p.norm_p);
        }
        if (OUT_DT == STK_BF16 && p.norm_kind != STK_NORM_NONE) { /* norm is of the fp32 value, before rounding */ }
#pragma unroll
        for (int d = 0; d < WMAX; ++d)
          if (d < p.n_dst) {
            // rotate destinations so the W owners do not all hit the same peer at the same time
            int dst = p.n_dst == 1 ? p.rank : (p.rank + d) % W;
            store_out<OUT_DT>(p.out.p[dst], v, s);
          }
        if (zero_in) InVec<IN_DT>::zero(p.grad.p[0], v);
      }
    }
  }

  reduce_tail<IN_DT, W_T>(p, part, bad, t_begin);
}

template <int IN_DT, int OUT_DT>
static cudaError_t launch_reduce(stk_ctx* c, const ReduceParams& p, int grid, bool coop, cudaStream_t s) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(p.world == 1 ? 256 : 512);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (coop) coop_attr(cfg, attr);
  ProfScope prof(c, 0, s);
  switch (p.world) {
    case 1: return cudaLaunchKernelEx(&cfg, k_grad_reduce<IN_DT, OUT_DT, 1>, p);
    case 2: return cudaLaunchKernelEx(&cfg, k_grad_reduce<IN_DT, OUT_DT, 2>, p);
    case 4: return cudaLaunchKernelEx(&cfg, k_grad_reduce<IN_DT, OUT_DT, 4>, p);
    case 8: return cudaLaunchKernelEx(&cfg, k_grad_reduce<IN_DT, OUT_DT, 8>, p);
    default: return cudaLaunchKernelEx(&cfg, k_grad_reduce<IN_DT, OUT_DT, 0>, p);
  }
}

}  // namespace stk

using namespace stk;

extern "C" {

int stk_grad_accumulate(stk_ctx* c, void* grad, int grad_dtype, float* acc, size_t n, int first, int zero_grad,
                        void* stream) {
  STK_REQUIRE(c, c && grad && acc, "stk_grad_accumulate: NULL argument");
  STK_REQUIRE(c, n % 8 == 0, "stk_grad_accumulate: n must be a multiple of 8");
  if (n == 0) return STK_OK;
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t nvec = n / 8;
  const unsigned grid = (unsigned)((nvec + 255) / 256);
  ProfScope prof(c, 2, s);
  switch (grad_dtype) {
    case STK_F32: k_grad_accumulate<STK_F32><<<grid, 256, 0, s>>>(grad, acc, nvec, first, zero_grad); break;
    case STK_BF16: k_grad_accumulate<STK_BF16><<<grid, 256, 0, s>>>(grad, acc, nvec, first, zero_grad); break;
    case STK_F16: k_grad_accumulate<STK_F16><<<grid, 256, 0, s>>>(grad, acc, nvec, first, zero_grad); break;
    default: return stk_fail(c, STK_ERR_INVALID, "stk_grad_accumulate: bad dtype");
  }
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

int stk_grad_reduce(stk_ctx* c, int mode, void* const* grad_ptrs, int grad_dtype, float* const* acc_ptrs,
                    void* const* out_ptrs, int out_dtype, size_t n, double mul, int norm_kind, double norm_p,
                    unsigned flags, void* stream) {
  STK_REQUIRE(c, c && grad_ptrs && out_ptrs, "stk_grad_reduce: NULL argument");
  STK_REQUIRE(c, n % 8 == 0, "stk_grad_reduce: n must be a multiple of 8");
  STK_REQUIRE(c, mode == STK_REDUCE_ALL || mode == STK_REDUCE_SCATTER, "stk_grad_reduce: bad mode");
  STK_REQUIRE(c, out_dtype == STK_F32 || out_dtype == STK_BF16, "stk_grad_reduce: out dtype must be f32 or bf16");
  STK_REQUIRE(c, norm_kind >= STK_NORM_NONE && norm_kind <= STK_NORM_P, "stk_grad_reduce: bad norm kind");
  if (c->world > 1 && !c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_grad_reduce before stk_comm_connect");
  STK_POLL(c);
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int W = c->world;

  ReduceParams p{};
  for (int r = 0; r < W; ++r) {
    STK_REQUIRE(c, grad_ptrs[r] && out_ptrs[r], "stk_grad_reduce: NULL peer pointer");
    p.grad.p[r] = grad_ptrs[r];
    p.out.p[r] = out_ptrs[r];
    p.acc.p[r] = acc_ptrs ? acc_ptrs[r] : nullptr;
  }
  p.pads = c->pads;
  p.scaler = c->scaler_dev;
  p.accum = c->accum_dev;
  p.blk_partial = c->blk_partial_dev;
  p.grp_partial = c->grp_partial_dev;
  p.grp_count = c->grp_count_dev;
  p.prof_ns = c->profiling ? c->prof_ns_dev : nullptr;
  size_t b = 0, e = 0;
  stk_shard_range(n, W, c->rank, &b, &e);
  p.vec_begin = b / 8;
  p.vec_end = (e + 7) / 8;
  p.vec_total = (n + 7) / 8;
  p.vec_per_shard = ((n + 7) / 8 + W - 1) / W;
  p.vec_per_shard += p.vec_per_shard & 1;  // same partition as stk_shard_range
  p.mul = (float)mul;
  p.norm_p = (float)norm_p;
  p.rank = c->rank;
  p.world = W;
  p.n_dst = (mode == STK_REDUCE_ALL) ? W : 1;
  p.norm_kind = norm_kind;
  p.flags = flags;
  p.epoch = ++c->blk_epoch;
  p.aux_epoch = (flags & STK_RF_FINAL) ? ++c->aux_epoch[0] : c->aux_epoch[0];

  // grid: identical on every rank (depends on n and W only).  Cross-rank kernels spin on peers, so every block must be
  // resident: one 512-thread block per SM, cooperative launch.
  const size_t nvec_shard = p.vec_per_shard;
  const int U = W == 1 ? 2 : (W == 2 ? 2 : 1);
  const size_t threads = W == 1 ? 256 : 512;
  size_t want = (nvec_shard + threads * U - 1) / (threads * U);
  int grid;
  const size_t cap = c->k1_max_blocks > 0 ? (size_t)std::min(c->k1_max_blocks, c->sm_count) : (size_t)c->sm_count;
  if (W > 1) grid = (int)std::max<size_t>(1, std::min<size_t>(want, cap));
  else grid = (int)std::max<size_t>(1, want);  // one-shot: every block does one chunk
  {
    int rc = stk_grow_partials(c, (size_t)grid, s);
    if (rc != STK_OK) return rc;
    p.blk_partial = c->blk_partial_dev;
    p.grp_partial = c->grp_partial_dev;
    p.grp_count = c->grp_count_dev;
  }
  const bool coop = W > 1;
  if (coop && grid > kMaxReduceBlocks) grid = kMaxReduceBlocks;

  cudaError_t err = cudaErrorNotSupported;
  if (coop && c->k1_algo == 2 && acc_ptrs == nullptr) {
    // multimem flavour: needs the multicast mappings of the gradient bucket and (all-reduce) of the output bucket
    p.grad_mc = stk_mc_lookup(c, grad_ptrs[c->rank]);
    p.out_mc = (mode == STK_REDUCE_ALL) ? stk_mc_lookup(c, out_ptrs[c->rank]) : nullptr;
    if (p.grad_mc && (mode == STK_REDUCE_SCATTER || p.out_mc)) {
      // The switch-side reduction saturates with few requesters: measured at W = 8 (profiles/study_w8_r02.json) 8 blocks beat
      // 148 at every size from 1 MiB to 256 MiB (16 MiB: 501 vs 392 GB/s busbw, 64 MiB: 706 vs 593, 256 MiB: 800 vs 764).
      const size_t bytes = n * (grad_dtype == STK_F32 ? 4 : 2);
      const int nvls_default = bytes < (size_t(128) << 20) ? 8 : 16;
      const int ngrid = std::min(grid, c->nvls_max_blocks > 0 ? c->nvls_max_blocks : nvls_default);
      err = launch_reduce_nvls(c, p, grad_dtype, out_dtype, ngrid, s);
      if (err != cudaSuccess && err != cudaErrorNotSupported)
        return stk_fail(c, STK_ERR_CUDA, std::string("k_grad_reduce_nvls launch: ") + cudaGetErrorString(err));
    }
  }
  if (err == cudaSuccess) return STK_OK;
  if (coop && c->k1_algo >= 1) {
    err = launch_reduce_bulk(c, p, grad_dtype, out_dtype, grid, s);
    if (err != cudaSuccess && err != cudaErrorNotSupported)
      return stk_fail(c, STK_ERR_CUDA, std::string("k_grad_reduce_bulk launch: ") + cudaGetErrorString(err));
  }
  if (err == cudaSuccess) return STK_OK;
#define STK_DISPATCH(IN, OUT) err = launch_reduce<IN, OUT>(c, p, grid, coop, s)
  if (grad_dtype == STK_BF16 && out_dtype == STK_F32) STK_DISPATCH(STK_BF16, STK_F32);
  else if (grad_dtype == STK_BF16 && out_dtype == STK_BF16) STK_DISPATCH(STK_BF16, STK_BF16);
  else if (grad_dtype == STK_F32 && out_dtype == STK_F32) STK_DISPATCH(STK_F32, STK_F32);
  else if (grad_dtype == STK_F32 && out_dtype == STK_BF16) STK_DISPATCH(STK_F32, STK_BF16);
  else if (grad_dtype == STK_F16 && out_dtype == STK_F32) STK_DISPATCH(STK_F16, STK_F32);
  else return stk_fail(c, STK_ERR_INVALID, "stk_grad_reduce: unsupported dtype combination");
#undef STK_DISPATCH
  if (err != cudaSuccess) return stk_fail(c, STK_ERR_CUDA, std::string("k_grad_reduce launch: ") + cudaGetErrorString(err));

  return STK_OK;
}

}  // extern "C"

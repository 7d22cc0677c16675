// k1_bulk.cu -- K1 (cross-rank, 16-bit gradients) with the peer reads staged through shared memory by bulk-async copies.
//
// Same protocol and results as k_grad_reduce (k1_reduce.cu); only the way the W peer gradients reach the SM differs:
// instead of W 16-byte register loads per thread per round (64 KB in flight per SM at W = 8, one round = one NVLink
// round trip), one thread per CTA issues `cp.async.bulk.shared::cluster.global` copies (TMA engine, SASS UBLKCP) of a
// whole 8 KB tile from each peer into a ring of shared-memory stages, completion signalled on an mbarrier.  The ring keeps
// up to 192 KB per SM in flight regardless of the register file, which is what the latency-bound middle of the size range
// (tens of MB per bucket, 5-6 rounds per launch) needs.  Consumers read their 16 bytes per peer from shared memory, reduce
// in rank order in fp32, and store exactly like the register-staged flavour (32-byte posted peer stores).
#include "k1_common.cuh"

namespace stk {

constexpr int kBulkThreads = 512;                       // one 8-element vector per thread per tile
constexpr int kBulkTileBytes = kBulkThreads * 16;       // 8 KB per peer per stage
constexpr int kBulkSmemBudget = 192 * 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <int IN_DT, int OUT_DT, int W_T>
__global__ void __launch_bounds__(kBulkThreads, 1) k_grad_reduce_bulk(const ReduceParams p, const int nstage) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full_bar[8];
  static_assert(IN_DT == STK_BF16 || IN_DT == STK_F16, "bulk flavour stages 16-bit gradients");
  const int W = W_T ? W_T : p.world;
  constexpr int WMAX = W_T ? W_T : kMaxWorld;
  const int tid = threadIdx.x;

  if (tid == 0) {
    for (int s = 0; s < nstage; ++s) mbar_init(&full_bar[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // peers' gradients are complete (and barriers are initialised); a missing peer: give up, the error word is set
  if (!block_barrier_all_ranks(p.pads, p.rank, W, 0, p.epoch)) return;
  unsigned long long t_begin = 0;
  if (p.prof_ns && blockIdx.x == 0 && tid == 0) t_begin = globaltimer_ns();

  float inv_scale = 1.f;
  if (p.flags & STK_RF_UNSCALE) inv_scale = (float)(1.0 / (double)p.scaler->scale);
  const float mul = p.mul;
  float part = 0.f;
  bool bad = false;

  // tiles of kBulkThreads vectors inside the owned shard, dealt round-robin to the blocks
  const size_t shard_vecs = p.vec_end - p.vec_begin;
  const size_t ntiles = (shard_vecs + kBulkThreads - 1) / kBulkThreads;
  const size_t my_tiles = ntiles > blockIdx.x ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const size_t stage_bytes = size_t(W) * kBulkTileBytes;

  auto issue = [&](size_t k) {  // thread 0: start the W copies of this block's k-th tile into stage k % nstage
    const int s = (int)(k % nstage);
    const size_t tile = blockIdx.x + k * gridDim.x;
    const size_t v0 = p.vec_begin + tile * kBulkThreads;
    const size_t nv = (p.vec_end - v0) < (size_t)kBulkThreads ? (p.vec_end - v0) : (size_t)kBulkThreads;
    const uint32_t bytes = (uint32_t)(nv * 16);
    mbar_expect_tx(&full_bar[s], bytes * W);
    for (int r = 0; r < W; ++r)
      bulk_g2s(smem + s * stage_bytes + size_t(r) * kBulkTileBytes, reinterpret_cast<const uint4*>(p.grad.p[r]) + v0, bytes,
               &full_bar[s]);
  };

  if (tid == 0) {
    // the start barrier's acquire was made by generic-proxy loads; order the async-proxy reads after it
    asm volatile("fence.proxy.async;" ::: "memory");
    for (size_t k = 0; k < my_tiles && k < (size_t)nstage; ++k) issue(k);
  }

  for (size_t k = 0; k < my_tiles; ++k) {
    const int s = (int)(k % nstage);
    const uint32_t parity = (uint32_t)((k / nstage) & 1);
    while (!mbar_try_wait(&full_bar[s], parity)) {
    }
    const size_t tile = blockIdx.x + k * gridDim.x;
    const size_t v = p.vec_begin + tile * kBulkThreads + tid;
    const bool active = v < p.vec_end;
    uint4 raw[WMAX];
    if (active) {
#pragma unroll
      for (int r = 0; r < WMAX; ++r)
        if (r < W) raw[r] = *reinterpret_cast<const uint4*>(smem + s * stage_bytes + size_t(r) * kBulkTileBytes + tid * 16);
    }
    __syncthreads();  // every thread has taken its bytes out of the stage: it can be refilled
    if (tid == 0 && k + nstage < my_tiles) issue(k + nstage);
    if (active) {
      float x[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = 0.f;
#pragma unroll
      for (int r = 0; r < WMAX; ++r)
        if (r < W) {  // rank order, fp32
          const uint32_t w4[4] = {raw[r].x, raw[r].y, raw[r].z, raw[r].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (IN_DT == STK_BF16) {
              x[2 * j] += bf16lo(w4[j]);
              x[2 * j + 1] += bf16hi(w4[j]);
            } else {
              x[2 * j] += f16lo(w4[j]);
              x[2 * j + 1] += f16hi(w4[j]);
            }
          }
        }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float y = x[i] * mul;
        bad |= !finitef(y);
        y *= inv_scale;
        x[i] = y;
        if (p.norm_kind == STK_NORM_L2) part = fmaf(y, y, part);
        else if (p.norm_kind == STK_NORM_INF) part = fmaxf(part, fabsf(y));
        else if (p.norm_kind == STK_NORM_P) part += __powf(fabsf(y), p.norm_p);
      }
#pragma unroll
      for (int d = 0; d < WMAX; ++d)
        if (d < p.n_dst) {
          const int dst = p.n_dst == 1 ? p.rank : (p.rank + d) % W;
          store_out<OUT_DT>(p.out.p[dst], v, x);
        }
    }
  }
  reduce_tail<IN_DT, W_T>(p, part, bad, t_begin);
}

template <int IN_DT, int OUT_DT>
static cudaError_t launch_bulk_t(stk_ctx* c, const ReduceParams& p, int grid, cudaStream_t s) {
  int nstage = kBulkSmemBudget / (p.world * kBulkTileBytes);
  if (nstage > 8) nstage = 8;
  if (nstage < 2) nstage = 2;
  const size_t smem = size_t(nstage) * p.world * kBulkTileBytes;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kBulkThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  coop_attr(cfg, attr);
  ProfScope prof(c, 0, s);
#define STK_BULK(WT)                                                                                              \
  {                                                                                                               \
    auto k = k_grad_reduce_bulk<IN_DT, OUT_DT, WT>;                                                               \
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);              \
    if (e != cudaSuccess) return e;                                                                               \
    return cudaLaunchKernelEx(&cfg, k, p, nstage);                                                                \
  }
  switch (p.world) {
    case 2: STK_BULK(2)
    case 4: STK_BULK(4)
    case 8: STK_BULK(8)
    default: STK_BULK(0)
  }
#undef STK_BULK
}

// returns cudaErrorNotSupported when this flavour does not cover the combination (caller falls back to k_grad_reduce)
cudaError_t launch_reduce_bulk(stk_ctx* c, const ReduceParams& p, int grad_dtype, int out_dtype, int grid, cudaStream_t s) {
  if (p.world < 2 || p.acc.p[0] != nullptr) return cudaErrorNotSupported;
  if (grad_dtype == STK_BF16 && out_dtype == STK_F32) return launch_bulk_t<STK_BF16, STK_F32>(c, p, grid, s);
  if (grad_dtype == STK_BF16 && out_dtype == STK_BF16) return launch_bulk_t<STK_BF16, STK_BF16>(c, p, grid, s);
  if (grad_dtype == STK_F16 && out_dtype == STK_F32) return launch_bulk_t<STK_F16, STK_F32>(c, p, grid, s);
  return cudaErrorNotSupported;
}

}  // namespace stk

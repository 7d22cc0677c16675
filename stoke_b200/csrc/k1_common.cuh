// k1_common.cuh -- pieces shared by the two flavours of K1 (k1_reduce.cu: register-staged loads; k1_bulk.cu: bulk-async
// copies staged through shared memory): launch parameters, typed 8-element vector access, and the common tail (block
// partial -> end barrier carrying the partials -> in-kernel bucket zeroing -> ticket -> norm / inf finalisation).
#pragma once
#include "ctx.cuh"

namespace stk {

struct ReduceParams {
  PtrTable grad;      // W peer pointers to the gradient bucket
  PtrTable acc;       // W peer pointers to the fp32 local accumulators (p[0] == nullptr: none)
  PtrTable out;       // W peer pointers to the main-grad bucket
  const void* grad_mc;  // multicast mapping of the gradient bucket (multimem flavour only)
  void* out_mc;         // multicast mapping of the output bucket (multimem flavour, all-reduce mode)
  PeerPads pads;
  stk_scaler_state_t* scaler;
  StepAccum* accum;
  float* blk_partial;   // [grid] per-block norm partials
  float* grp_partial;   // [grid / 64 + 1] per-group partials
  uint32_t* grp_count;  // [grid / 64 + 1] group tickets
  unsigned long long* prof_ns;  // optional {barrier-to-barrier ns, launches, zeroing-tail ns} (block 0), nullptr when off
  size_t vec_begin, vec_end;  // owned shard in units of 8 elements
  size_t vec_total, vec_per_shard;  // whole bucket / shard stride (for zeroing the local bucket after the end barrier)
  float mul;
  float norm_p;
  int rank, world, n_dst;
  int norm_kind;
  uint32_t flags;
  uint32_t epoch, aux_epoch;
};

template <int DT>
struct InVec;  // 8 input elements -> 8 floats
template <>
struct InVec<STK_F32> {
  static constexpr int kBytes = 32;
  __device__ static void load(const void* base, size_t v, float (&f)[8]) {
    f8 a = ld_stream_f8(reinterpret_cast<const float*>(base) + v * 8);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = a.v[i];
  }
  __device__ static void zero(void* base, size_t v) {
    const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    st_stream_f8(reinterpret_cast<float*>(base) + v * 8, z);
  }
};
template <>
struct InVec<STK_BF16> {
  static constexpr int kBytes = 16;
  __device__ static void load(const void* base, size_t v, float (&f)[8]) {
    uint4 u = ld_stream16(reinterpret_cast<const uint4*>(base) + v);
    f[0] = bf16lo(u.x); f[1] = bf16hi(u.x); f[2] = bf16lo(u.y); f[3] = bf16hi(u.y);
    f[4] = bf16lo(u.z); f[5] = bf16hi(u.z); f[6] = bf16lo(u.w); f[7] = bf16hi(u.w);
  }
  __device__ static void zero(void* base, size_t v) {
    st_stream16(reinterpret_cast<uint4*>(base) + v, make_uint4(0, 0, 0, 0));
  }
};
template <>
struct InVec<STK_F16> {
  static constexpr int kBytes = 16;
  __device__ static void load(const void* base, size_t v, float (&f)[8]) {
    uint4 u = ld_stream16(reinterpret_cast<const uint4*>(base) + v);
    f[0] = f16lo(u.x); f[1] = f16hi(u.x); f[2] = f16lo(u.y); f[3] = f16hi(u.y);
    f[4] = f16lo(u.z); f[5] = f16hi(u.z); f[6] = f16lo(u.w); f[7] = f16hi(u.w);
  }
  __device__ static void zero(void* base, size_t v) {
    st_stream16(reinterpret_cast<uint4*>(base) + v, make_uint4(0, 0, 0, 0));
  }
};

template <int DT>
__device__ __forceinline__ void store_out(void* base, size_t v, const float (&f)[8]) {
  if constexpr (DT == STK_F32) {
    st_stream_f8(reinterpret_cast<float*>(base) + v * 8, f);  // one 32-byte store: full sectors over NVLink
  } else {
    st_stream16(reinterpret_cast<uint4*>(base) + v,
                make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7])));
  }
}


// Everything after a block's data phase.  `part` / `bad`: this thread's norm partial and inf/nan flag; t_begin: device
// timestamp taken after the start barrier (block 0 / thread 0, profiling only).  Must be called by all threads of the block.
template <int IN_DT, int W_T>
__device__ __forceinline__ void reduce_tail(const ReduceParams& p, float part, bool bad, unsigned long long t_begin) {
  __shared__ float s_red[32];
  __shared__ unsigned s_bad[32];
  const int W = W_T ? W_T : p.world;
  // ---- per-block partials (fixed tree: run-to-run deterministic); ONE block-wide barrier, then only warp 0 continues ----
  {
    const bool mx = p.norm_kind == STK_NORM_INF;
    const float wsum = mx ? warp_reduce<true>(part) : warp_reduce<false>(part);
    const unsigned wbad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0) {
      s_red[threadIdx.x >> 5] = wsum;
      s_bad[threadIdx.x >> 5] = wbad;
    }
  }
  __syncthreads();

  // block partial (warp 0): needed before the end barrier at W > 1, where it rides to the peers with the barrier flag
  float blk = 0.f;
  unsigned any_bad = 0;
  if (threadIdx.x < 32) {
    const unsigned nwarp = (blockDim.x + 31) >> 5;
    blk = threadIdx.x < nwarp ? s_red[threadIdx.x] : 0.f;
    blk = (p.norm_kind == STK_NORM_INF) ? warp_reduce<true>(blk) : warp_reduce<false>(blk);
    any_bad = __any_sync(0xffffffffu, threadIdx.x < nwarp && s_bad[threadIdx.x] != 0);
  }

  if (W > 1) {
    // Publish this block's (norm partial, inf flag) to every rank BEFORE signalling the end barrier: the same thread then
    // does fence.sys + st.release of the flag, so whoever sees the flag sees the partial.  Every rank later sums all
    // W x grid partials in the same (rank, block) order -> bit-identical totals everywhere, with no third cross-GPU
    // round trip after the data phase.
    if (threadIdx.x < (unsigned)W) {
      RankScalars* slot = &p.pads.p[threadIdx.x]->blk_scal[p.rank][blockIdx.x];
      st_relaxed_sys_f32(&slot->norm_partial, blk);
      st_relaxed_sys_u32(&slot->found_inf, any_bad);
    }
    // a peer that never arrives: give up (error word is set, the host raises STK_ERR_PEER at its next call); nothing is
    // zeroed or finalised on top of an incomplete exchange
    if (!block_barrier_all_ranks(p.pads, p.rank, W, 1, p.epoch)) return;
  }
  // end of the NVLink data phase (all peer reads and peer writes of this block are complete on every rank)
  unsigned long long t_data_end = 0;
  if (p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) t_data_end = globaltimer_ns();
  if (W > 1 && (p.flags & STK_RF_ZERO_INPUT)) {
    // Zero the LOCAL gradient bucket inside the kernel (no separate memset between backward and step).  Block b may only
    // clear what the peers' blocks b have finished reading -- exactly this block's own index pattern, replicated in every
    // shard: shard q of my bucket is read by rank q's block b at the same offsets, and that block has passed the end barrier.
    for (int q = 0; q < W; ++q) {
      const size_t qb = p.vec_per_shard * q;
      size_t qe = qb + p.vec_per_shard;
      if (qe > p.vec_total) qe = p.vec_total;
      for (size_t v = qb + size_t(blockIdx.x) * blockDim.x + threadIdx.x; v < qe; v += size_t(gridDim.x) * blockDim.x)
        InVec<IN_DT>::zero(p.grad.p[p.rank], v);
    }
  }
  if (p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&p.prof_ns[0], t_data_end - t_begin);         // barrier-to-barrier: the NVLink phase
    atomicAdd(&p.prof_ns[1], 1ull);
    atomicAdd(&p.prof_ns[2], globaltimer_ns() - t_data_end);  // local (HBM) bucket-zeroing tail of block 0
  }

  // Only warp 0 stays for the bookkeeping: the other warps retire now, so a block never sits idle on the ticket's
  // fence + atomic round trip.
  if (threadIdx.x >= 32) return;
  const unsigned lane = threadIdx.x;
  const bool mx = p.norm_kind == STK_NORM_INF;

  if (W > 1) {
    // ---- cross-rank flavour: plain ticket over the (<= SM count) co-resident blocks ----
    unsigned last = 0;
    if (lane == 0) {
      __threadfence();
      last = (atomicAdd(&p.accum->blocks_done, 1u) == gridDim.x - 1);
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    // every local block has passed its end barrier, so every peer block's partial has landed in this rank's pad
    float total = 0.f;
    unsigned inf = 0;
    for (int r = 0; r < W; ++r) {
      float x = 0.f;
      for (unsigned b = lane; b < gridDim.x; b += 32) {
        const RankScalars* slot = &p.pads.p[p.rank]->blk_scal[r][b];
        const float y = ld_relaxed_sys_f32(&slot->norm_partial);
        x = mx ? fmaxf(x, y) : x + y;
        inf |= ld_relaxed_sys_u32(&slot->found_inf);
      }
      x = mx ? warp_reduce<true>(x) : warp_reduce<false>(x);
      total = mx ? fmaxf(total, x) : total + x;
    }
    inf = __any_sync(0xffffffffu, inf != 0);
    if (lane == 0) {
      float run = p.accum->norm_partial;   // running over the buckets of this optimizer step (global values)
      run = mx ? fmaxf(run, total) : run + total;
      unsigned run_inf = p.accum->found_inf | (inf ? 1u : 0u);
      p.accum->blocks_done = 0;
      if (p.flags & STK_RF_FINAL) {
        float norm = run;
        if (p.norm_kind == STK_NORM_L2) norm = sqrtf(run);
        else if (p.norm_kind == STK_NORM_P) norm = powf(run, 1.f / p.norm_p);
        p.scaler->grad_norm = norm;
        // the inf gate belongs to the loss scaler (GradScaler.step); without one the reference steps regardless
        p.scaler->found_inf = (run_inf && (p.flags & STK_RF_UNSCALE)) ? 1 : 0;
        run = 0.f;
        run_inf = 0;
      }
      p.accum->norm_partial = run;
      p.accum->found_inf = run_inf;
    }
    return;
  }

  // ---- local flavour (W == 1) ----
  // Two-level ticket (groups of 64 blocks): the last block of a group folds the group's partials, the last group folds
  // the group partials -- fixed order at both levels (deterministic), and the serial tail stays short even with the tens
  // of thousands of one-shot blocks of a W == 1 launch.
  const unsigned grp = blockIdx.x >> 6, ngroups = (gridDim.x + 63) >> 6;
  const unsigned gsize = min(64u, gridDim.x - (grp << 6));
  unsigned last = 0;
  if (lane == 0) {
    if (p.norm_kind != STK_NORM_NONE) p.blk_partial[blockIdx.x] = blk;
    if (any_bad) atomicOr(&p.accum->found_inf, 1u);
    __threadfence();
    last = (atomicAdd(&p.grp_count[grp], 1u) == gsize - 1);
  }
  last = __shfl_sync(0xffffffffu, last, 0);
  if (!last) return;
  __threadfence();
  {
    float x = 0.f;
    if (p.norm_kind != STK_NORM_NONE) {
      const float a = lane < gsize ? __ldcg(&p.blk_partial[(grp << 6) + lane]) : 0.f;
      const float b = lane + 32 < gsize ? __ldcg(&p.blk_partial[(grp << 6) + 32 + lane]) : 0.f;
      x = mx ? warp_reduce<true>(fmaxf(a, b)) : warp_reduce<false>(a + b);
    }
    last = 0;
    if (lane == 0) {
      p.grp_partial[grp] = x;
      p.grp_count[grp] = 0;
      __threadfence();
      last = (atomicAdd(&p.accum->blocks_done, 1u) == ngroups - 1);
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
  }

  // ---- last group of this rank: fold the bucket into the step accumulators; on FINAL exchange across ranks ----
  __threadfence();
  float tot = 0.f;
  if (p.norm_kind != STK_NORM_NONE) {
    float x = 0.f;
    for (unsigned i = lane; i < ngroups; i += 32) {  // fixed lane/iteration order -> deterministic
      const float y = __ldcg(&p.grp_partial[i]);
      x = mx ? fmaxf(x, y) : x + y;
    }
    tot = mx ? warp_reduce<true>(x) : warp_reduce<false>(x);
  }
  if (lane == 0) {
    float run = p.accum->norm_partial;
    run = (p.norm_kind == STK_NORM_INF) ? fmaxf(run, tot) : run + tot;
    p.accum->norm_partial = run;
    p.accum->blocks_done = 0;
    __threadfence();
  }
  if (!(p.flags & STK_RF_FINAL)) return;
  if (lane == 0) {
    const float total = p.accum->norm_partial;
    const uint32_t inf = atomicOr(&p.accum->found_inf, 0u);
    float norm = total;
    if (p.norm_kind == STK_NORM_L2) norm = sqrtf(total);
    else if (p.norm_kind == STK_NORM_P) norm = powf(total, 1.f / p.norm_p);
    p.scaler->grad_norm = norm;
    // the inf gate belongs to the loss scaler (GradScaler.step); without one the reference steps regardless
    p.scaler->found_inf = (inf && (p.flags & STK_RF_UNSCALE)) ? 1 : 0;
    p.accum->norm_partial = 0.f;
    p.accum->found_inf = 0u;
  }
}

// k1_bulk.cu: shared-memory / bulk-async flavour for cross-rank 16-bit buckets; cudaErrorNotSupported -> use k_grad_reduce
cudaError_t launch_reduce_bulk(stk_ctx* c, const ReduceParams& p, int grad_dtype, int out_dtype, int grid, cudaStream_t s);
// k1_nvls.cu: multimem (NVSwitch in-network reduction) flavour; cudaErrorNotSupported -> next flavour
cudaError_t launch_reduce_nvls(stk_ctx* c, const ReduceParams& p, int grad_dtype, int out_dtype, int grid, cudaStream_t s);

}  // namespace stk

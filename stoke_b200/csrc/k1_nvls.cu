// k1_nvls.cu -- K1 over NVSwitch multicast (NVLS): the switch does the cross-rank sum.
//
// Same protocol, tail and fused work as k_grad_reduce (k1_reduce.cu) -- start barrier, owned shard, 1/W scale, inf/nan test,
// unscale, norm partial, end barrier carrying the partials, in-kernel zeroing of the local bucket -- but the W-way sum is one
// `multimem.ld_reduce` on the bucket's multicast address (SASS LDGMC.E.ADD.*: the switch pulls the vector from every rank,
// adds in fp32 and returns ONE vector), and the all-reduce publish is one `multimem.st` (the switch replicates the store
// into every rank's output bucket).  Per GPU and direction the bus carries n*b_in/W + n*b_out bytes inbound and
// n*b_in + n*b_out/W outbound instead of (W-1)/W*n*(b_in+b_out) each way: at W = 8 with 2-byte elements 2.25 n vs 3.5 n.
//
// Numerics: for 16-bit inputs the switch returns the sum rounded to the input type (fp32 accumulation inside the switch,
// `.acc::f32`) -- what NCCL's NVLS all-reduce gives the reference's DDP path -- so this flavour differs from the
// register-staged / bulk flavours (exact fp32 sums of the 16-bit inputs) in the last bit of a 16-bit value; fp32 inputs are
// summed in fp32 in switch order.  One owner reduces each element and every rank receives that owner's value, so replicas
// stay bit-identical.  The training path selects it only on request (STK_K1_ALGO=nvls); the bandwidth sweep reports it.
#include "k1_common.cuh"

namespace stk {

constexpr int kNvlsThreads = 512;

template <int IN_DT, int OUT_DT, int U>
__global__ void __launch_bounds__(kNvlsThreads, 1) k_grad_reduce_nvls(const ReduceParams p) {
  const int W = p.world;
  if (!block_barrier_all_ranks(p.pads, p.rank, W, 0, p.epoch)) return;
  unsigned long long t_begin = 0;
  if (p.prof_ns && blockIdx.x == 0 && threadIdx.x == 0) t_begin = globaltimer_ns();

  float inv_scale = 1.f;
  if (p.flags & STK_RF_UNSCALE) inv_scale = (float)(1.0 / (double)p.scaler->scale);
  const float mul = p.mul;
  float part = 0.f;
  bool bad = false;
  constexpr int kInBytes = InVec<IN_DT>::kBytes;  // bytes of one 8-element input vector
  const char* gmc = reinterpret_cast<const char*>(p.grad_mc);
  const bool all = p.n_dst > 1;

  const size_t stride = size_t(gridDim.x) * blockDim.x;
  const unsigned lane = threadIdx.x & 31;
  // the loop variable is warp-uniform (all lanes of a warp iterate together: the fp32 publish below shuffles between lanes);
  // a lane past the end of the shard is merely inactive
  for (size_t w0 = p.vec_begin + size_t(blockIdx.x) * blockDim.x + (threadIdx.x - lane); w0 < p.vec_end; w0 += stride * U) {
    const size_t v0 = w0 + lane;
    float x[U][8];
    // every multimem load of this round is issued before the first use (one switch round trip per round)
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t v = v0 + u * stride;
      if (v < p.vec_end) {
        if constexpr (IN_DT == STK_F32) {
          const float4 a = mm_ld_reduce_f32x4(gmc + v * kInBytes);
          const float4 b = mm_ld_reduce_f32x4(gmc + v * kInBytes + 16);
          x[u][0] = a.x; x[u][1] = a.y; x[u][2] = a.z; x[u][3] = a.w;
          x[u][4] = b.x; x[u][5] = b.y; x[u][6] = b.z; x[u][7] = b.w;
        } else {
          const uint4 r = (IN_DT == STK_BF16) ? mm_ld_reduce_bf16x8(gmc + v * kInBytes) : mm_ld_reduce_f16x8(gmc + v * kInBytes);
          const uint32_t w4[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            x[u][2 * j] = (IN_DT == STK_BF16) ? bf16lo(w4[j]) : f16lo(w4[j]);
            x[u][2 * j + 1] = (IN_DT == STK_BF16) ? bf16hi(w4[j]) : f16hi(w4[j]);
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[u][i] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t v = v0 + u * stride;
      const bool active = v < p.vec_end;
      if (active) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float y = x[u][i] * mul;
          bad |= !finitef(y);
          y *= inv_scale;
          x[u][i] = y;
          if (p.norm_kind == STK_NORM_L2) part = fmaf(y, y, part);
          else if (p.norm_kind == STK_NORM_INF) part = fmaxf(part, fabsf(y));
          else if (p.norm_kind == STK_NORM_P) part += __powf(fabsf(y), p.norm_p);
        }
      }
      if (all) {  // uniform
        if constexpr (OUT_DT == STK_F32) {
          // multimem.st moves at most 16 bytes per thread; two 16-byte stores per thread at a 32-byte thread stride would
          // write half sectors (measured with plain peer stores: half the NVLink rate).  Lane pairs swap halves instead, so
          // that each store instruction covers whole 32-byte sectors: the even lane's vector, then the odd lane's.
          // (shards start on even vector indices -- stk_shard_range -- so lane parity == vector parity)
          const bool odd = lane & 1;
          float take[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) take[i] = __shfl_xor_sync(0xffffffffu, odd ? x[u][i] : x[u][4 + i], 1);
          const bool pair_ok = active && ((v ^ 1) < p.vec_end);
          if (pair_ok) {
            // ONE store instruction per sector row for both lanes of the pair (select data and address, do not branch)
            char* even_vec = reinterpret_cast<char*>(p.out_mc) + (v & ~size_t(1)) * 32 + (odd ? 16 : 0);
            float d1[4], d2[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              d1[i] = odd ? take[i] : x[u][i];        // row of the even vector: [even lane: its 0..3 | odd lane: even's 4..7]
              d2[i] = odd ? x[u][4 + i] : take[i];    // row of the odd vector:  [even lane: odd's 0..3 | odd lane: its 4..7]
            }
            mm_st16(even_vec, make_uint4(__float_as_uint(d1[0]), __float_as_uint(d1[1]), __float_as_uint(d1[2]), __float_as_uint(d1[3])));
            mm_st16(even_vec + 32, make_uint4(__float_as_uint(d2[0]), __float_as_uint(d2[1]), __float_as_uint(d2[2]), __float_as_uint(d2[3])));
          } else if (active) {
            char* mine = reinterpret_cast<char*>(p.out_mc) + v * 32;
            mm_st16(mine, make_uint4(__float_as_uint(x[u][0]), __float_as_uint(x[u][1]), __float_as_uint(x[u][2]),
                                     __float_as_uint(x[u][3])));
            mm_st16(mine + 16, make_uint4(__float_as_uint(x[u][4]), __float_as_uint(x[u][5]), __float_as_uint(x[u][6]),
                                          __float_as_uint(x[u][7])));
          }
        } else if (active) {
          mm_st16(reinterpret_cast<char*>(p.out_mc) + v * 16,
                  make_uint4(pack_bf16(x[u][0], x[u][1]), pack_bf16(x[u][2], x[u][3]), pack_bf16(x[u][4], x[u][5]),
                             pack_bf16(x[u][6], x[u][7])));
        }
      } else if (active) {
        store_out<OUT_DT>(p.out.p[p.rank], v, x[u]);
      }
    }
  }
  reduce_tail<IN_DT, 0>(p, part, bad, t_begin);
}

template <int IN_DT, int OUT_DT>
static cudaError_t launch_nvls_t(stk_ctx* c, const ReduceParams& p, int grid, cudaStream_t s) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kNvlsThreads);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  coop_attr(cfg, attr);
  ProfScope prof(c, 0, s);
  // small shards: one round per thread is enough; large shards: 4 independent switch requests in flight per thread
  const size_t shard_vecs = p.vec_end - p.vec_begin;
  if (shard_vecs <= size_t(grid) * kNvlsThreads) return cudaLaunchKernelEx(&cfg, k_grad_reduce_nvls<IN_DT, OUT_DT, 1>, p);
  return cudaLaunchKernelEx(&cfg, k_grad_reduce_nvls<IN_DT, OUT_DT, 4>, p);
}

cudaError_t launch_reduce_nvls(stk_ctx* c, const ReduceParams& p, int grad_dtype, int out_dtype, int grid, cudaStream_t s) {
  if (p.world < 2 || p.acc.p[0] != nullptr || p.grad_mc == nullptr) return cudaErrorNotSupported;
  if (grad_dtype == STK_BF16 && out_dtype == STK_F32) return launch_nvls_t<STK_BF16, STK_F32>(c, p, grid, s);
  if (grad_dtype == STK_BF16 && out_dtype == STK_BF16) return launch_nvls_t<STK_BF16, STK_BF16>(c, p, grid, s);
  if (grad_dtype == STK_F32 && out_dtype == STK_F32) return launch_nvls_t<STK_F32, STK_F32>(c, p, grid, s);
  if (grad_dtype == STK_F16 && out_dtype == STK_F32) return launch_nvls_t<STK_F16, STK_F32>(c, p, grid, s);
  return cudaErrorNotSupported;
}

}  // namespace stk

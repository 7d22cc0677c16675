// k1_norm.cu -- the norm / inf pass when there is no cross-rank reduce to fuse it into (world == 1), and the in-place clip of
// reduced gradients for the stock-optimizer route.
//
//   k_grad_norm  : reads the raw gradient bucket ONCE (2 B/element for bf16), accumulates sum g^2 | max |g| | sum |g|^p and the
//                  inf/nan flag of x = (g [+ acc]) * mul / scale, finishes them into the state (grad_norm, found_inf).  Writes
//                  nothing: the fused optimizer step (k_optim_step, raw route) reads the bucket a second time -- from L2 when
//                  the bucket fits (loads here carry an L2 evict_last policy; ResNet-50's 51 MB bucket sits in the 126 MB L2) --
//                  and zeroes it.  Replaces the W == 1 form of k_grad_reduce on the training path: 2 + 30 B/element through
//                  HBM instead of 8 + 30 (no fp32 main-grad round trip).
//   k_grad_scale : grad *= clip coefficient, or clamp (clip_grad_norm_'s scaling pass / clip_grad_value_,
//                  torch/nn/utils/clip_grad.py) for optimizers the fused step does not cover.
#include "k1_common.cuh"

namespace stk {

__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
// Bypass L1, keep in L2: the fused step's second read of a bucket that fits L2 then hits (measured -4 us on K2 at
// ResNet-50 size, profiles/kernels_r02.md).
__device__ __forceinline__ uint4 ld16_keep(const void* p, uint64_t pol) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(pol));
  return v;
}

struct NormParams {
  const void* grad;
  const float* acc;
  size_t nvec;       // 8-element vectors
  float mul, norm_p;
  int norm_kind;
  uint32_t flags;
  stk_scaler_state_t* scaler;
  StepAccum* accum;
  float* blk_partial;
};

template <int IN_DT>
struct RawVec;  // the raw words of one 8-element vector (kept packed until use: 4 registers per 16-bit vector in flight)
template <>
struct RawVec<STK_F32> {
  uint4 a, b;
  __device__ void load(const void* base, size_t v, uint64_t pol) {
    const uint4* q = reinterpret_cast<const uint4*>(base) + 2 * v;
    a = ld16_keep(q, pol);
    b = ld16_keep(q + 1, pol);
  }
  __device__ void unpack(float (&f)[8]) const {
    f[0] = __uint_as_float(a.x); f[1] = __uint_as_float(a.y); f[2] = __uint_as_float(a.z); f[3] = __uint_as_float(a.w);
    f[4] = __uint_as_float(b.x); f[5] = __uint_as_float(b.y); f[6] = __uint_as_float(b.z); f[7] = __uint_as_float(b.w);
  }
};
template <int DT16>
struct RawVec16 {
  uint4 u;
  __device__ void load(const void* base, size_t v, uint64_t pol) {
    u = ld16_keep(reinterpret_cast<const uint4*>(base) + v, pol);
  }
  __device__ void unpack(float (&f)[8]) const {
    const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      f[2 * j] = (DT16 == STK_BF16) ? bf16lo(w4[j]) : f16lo(w4[j]);
      f[2 * j + 1] = (DT16 == STK_BF16) ? bf16hi(w4[j]) : f16hi(w4[j]);
    }
  }
};
template <>
struct RawVec<STK_BF16> : RawVec16<STK_BF16> {};
template <>
struct RawVec<STK_F16> : RawVec16<STK_F16> {};

constexpr int kNormThreads = 256;
constexpr int kNormUnroll = 8;  // 8 independent 16-byte loads per thread: 32 KB in flight per block

// One-shot blocks (one tile of kNormThreads * kNormUnroll vectors each, the shape that streams best on this part,
// tools/membench.cu): load, reduce, write ONE partial, retire -- no ticket, no fence, no block waits on an atomic.  The
// partials are folded by k_grad_norm_finish, a single block launched right behind on the same stream (stream order is the
// only synchronisation), in a fixed order -> run-to-run deterministic.
template <int IN_DT, bool HAS_ACC>
__global__ void __launch_bounds__(kNormThreads) k_grad_norm(const NormParams p) {
  __shared__ float s_red[32];
  const uint64_t pol = policy_evict_last();
  float inv_scale = 1.f;
  if (p.flags & STK_RF_UNSCALE) inv_scale = (float)(1.0 / (double)p.scaler->scale);
  const float mul = p.mul;
  float part = 0.f;
  bool bad = false;
  const size_t t0 = size_t(blockIdx.x) * kNormThreads * kNormUnroll;
  RawVec<IN_DT> raw[kNormUnroll];
#pragma unroll
  for (int u = 0; u < kNormUnroll; ++u) {
    const size_t v = t0 + size_t(u) * kNormThreads + threadIdx.x;
    if (v < p.nvec) raw[u].load(p.grad, v, pol);
  }
#pragma unroll
  for (int u = 0; u < kNormUnroll; ++u) {
    const size_t v = t0 + size_t(u) * kNormThreads + threadIdx.x;
    if (v < p.nvec) {
      float g[8];
      raw[u].unpack(g);
      if (HAS_ACC) {
        float a[8];
        InVec<STK_F32>::load(p.acc, v, a);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] += a[i];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float x = g[i] * mul;
        bad |= !finitef(x);
        x *= inv_scale;
        if (p.norm_kind == STK_NORM_L2) part = fmaf(x, x, part);
        else if (p.norm_kind == STK_NORM_INF) part = fmaxf(part, fabsf(x));
        else if (p.norm_kind == STK_NORM_P) part += __powf(fabsf(x), p.norm_p);
      }
    }
  }
  const bool mx = p.norm_kind == STK_NORM_INF;
  const float blk = mx ? block_reduce<true>(part, s_red) : block_reduce<false>(part, s_red);
  const int any_bad = __syncthreads_or(bad ? 1 : 0);
  if (threadIdx.x == 0) {
    // sign bit of the partial carries the block's inf/nan verdict (partials are >= 0 for every norm kind)
    p.blk_partial[blockIdx.x] = any_bad ? -1.f - fminf(blk, 3.0e38f) : blk;
  }
}

__global__ void __launch_bounds__(1024) k_grad_norm_finish(const NormParams p, unsigned nblocks) {
  __shared__ float s_red[32];
  const bool mx = p.norm_kind == STK_NORM_INF;
  float x = 0.f;
  bool bad = false;
  for (unsigned b = threadIdx.x; b < nblocks; b += blockDim.x) {
    float y = __ldcg(&p.blk_partial[b]);
    if (y < 0.f) {
      bad = true;
      y = -1.f - y;
    }
    x = mx ? fmaxf(x, y) : x + y;
  }
  const float tot = mx ? block_reduce<true>(x, s_red) : block_reduce<false>(x, s_red);
  const int any_bad = __syncthreads_or(bad ? 1 : 0);
  if (threadIdx.x == 0) {
    float run = p.accum->norm_partial;
    run = mx ? fmaxf(run, tot) : run + tot;
    uint32_t inf = p.accum->found_inf | (any_bad ? 1u : 0u);
    if (p.flags & STK_RF_FINAL) {
      float norm = run;
      if (p.norm_kind == STK_NORM_L2) norm = sqrtf(run);
      else if (p.norm_kind == STK_NORM_P) norm = powf(run, 1.f / p.norm_p);
      if (inf) norm = __int_as_float(0x7f800000);  // an inf/nan gradient: torch's total_norm is inf (or nan) too
      p.scaler->grad_norm = norm;
      // the inf gate belongs to the loss scaler (GradScaler.step); without one the reference steps regardless
      p.scaler->found_inf = (inf && (p.flags & STK_RF_UNSCALE)) ? 1 : 0;
      run = 0.f;
      inf = 0;
    }
    p.accum->norm_partial = run;
    p.accum->found_inf = inf;
  }
}

__global__ void __launch_bounds__(256) k_grad_scale(float* __restrict__ grad, size_t nvec, int clip_kind, float max_norm,
                                                     float clip_value, const stk_scaler_state_t* scaler) {
  const size_t v = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (v >= nvec) return;
  float coef = 1.f;
  if (clip_kind == STK_CLIP_NORM) coef = fminf(max_norm / (scaler->grad_norm + 1e-6f), 1.0f);
  f8 g = ld_stream_f8(grad + v * 8);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (clip_kind == STK_CLIP_NORM) g.v[i] *= coef;
    else g.v[i] = fminf(fmaxf(g.v[i], -clip_value), clip_value);
  }
  st_stream_f8(grad + v * 8, g.v);
}

}  // namespace stk

using namespace stk;

extern "C" {

int stk_grad_norm(stk_ctx* c, const void* grad, int grad_dtype, const float* acc, size_t n, double mul, int norm_kind,
                  double norm_p, unsigned flags, void* stream) {
  STK_REQUIRE(c, c && grad, "stk_grad_norm: NULL argument");
  STK_REQUIRE(c, n % 8 == 0, "stk_grad_norm: n must be a multiple of 8");
  STK_REQUIRE(c, norm_kind >= STK_NORM_NONE && norm_kind <= STK_NORM_P, "stk_grad_norm: bad norm kind");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  NormParams p{};
  p.grad = grad;
  p.acc = acc;
  p.nvec = n / 8;
  p.mul = (float)mul;
  p.norm_p = (float)norm_p;
  p.norm_kind = norm_kind;
  p.flags = flags;
  p.scaler = c->scaler_dev;
  p.accum = c->accum_dev;
  const size_t tile = size_t(kNormThreads) * kNormUnroll;
  size_t want = (p.nvec + tile - 1) / tile;
  if (want < 1) want = 1;
  void (*kern)(NormParams) = nullptr;
#define STK_PICK(DT) kern = acc ? k_grad_norm<DT, true> : k_grad_norm<DT, false>;
  switch (grad_dtype) {
    case STK_F32: STK_PICK(STK_F32) break;
    case STK_BF16: STK_PICK(STK_BF16) break;
    case STK_F16: STK_PICK(STK_F16) break;
    default: return stk_fail(c, STK_ERR_INVALID, "stk_grad_norm: bad dtype");
  }
#undef STK_PICK
  const unsigned grid = (unsigned)want;
  int rc = stk_grow_partials(c, grid, s);
  if (rc != STK_OK) return rc;
  p.blk_partial = c->blk_partial_dev;
  ProfScope prof(c, 3, s);
  kern<<<grid, kNormThreads, 0, s>>>(p);
  k_grad_norm_finish<<<1, 1024, 0, s>>>(p, grid);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

int stk_grad_scale(stk_ctx* c, float* grad, size_t n, int clip_kind, double clip_max_norm, double clip_value, void* stream) {
  STK_REQUIRE(c, c && grad, "stk_grad_scale: NULL argument");
  STK_REQUIRE(c, n % 8 == 0, "stk_grad_scale: n must be a multiple of 8");
  STK_REQUIRE(c, clip_kind == STK_CLIP_NORM || clip_kind == STK_CLIP_VALUE, "stk_grad_scale: clip kind must be norm or value");
  if (n == 0) return STK_OK;
  DeviceGuard g(c->device);
  const size_t nvec = n / 8;
  k_grad_scale<<<(unsigned)((nvec + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      grad, nvec, clip_kind, (float)clip_max_norm, (float)clip_value, c->scaler_dev);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

}  // extern "C"

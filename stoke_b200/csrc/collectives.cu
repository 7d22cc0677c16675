// collectives.cu -- the small cross-rank operations that ride on the signal pads: loss mean, barrier, broadcast.
//
//   stk_loss_sync : replaces loss.item() + barrier() + all_reduce(1 elem) + item()/W   (stoke/distributed.py:619-646)
//                   with one 1-block kernel that pushes the scalar to every peer's slot, waits for the peers' slots, sums
//                   in rank order and writes the mean to pinned host memory; one stream synchronise total.
//   stk_barrier   : torch.distributed.barrier()                                         (stoke/distributed.py:673)
//   stk_bcast     : rank `root` -> all: DDP's init parameter sync and the per-forward BatchNorm buffer broadcast
//                   (broadcast_buffers=True, stoke/configs.py:182) as a peer pull.
#include "ctx.cuh"

namespace stk {

template <int DT>
__device__ __forceinline__ float load_scalar(const void* p) {
  if constexpr (DT == STK_F32) return *reinterpret_cast<const float*>(p);
  else if constexpr (DT == STK_BF16) return __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(p));
  else return __half2float(*reinterpret_cast<const __half*>(p));
}

template <int DT>
__global__ void k_loss_sync(const void* loss, double* out_host, PeerPads pads, int rank, int world, uint32_t epoch) {
  __shared__ float s_val[kMaxWorld];
  const float mine = load_scalar<DT>(loss);
  if (world == 1) {
    if (threadIdx.x == 0) {
      *out_host = (double)mine;
      __threadfence_system();
    }
    return;
  }
  const int par = epoch & 1;
  if (threadIdx.x < (unsigned)world) {
    const int peer = threadIdx.x;
    st_relaxed_sys_f32(&pads.p[peer]->loss_slot[par][rank], mine);
    __threadfence_system();
    st_release_sys(&pads.p[peer]->aux_flag[1][rank], epoch);
    wait_flag(&pads.p[rank]->aux_flag[1][peer], epoch, pads.p[rank]);
    s_val[peer] = ld_relaxed_sys_f32(&pads.p[rank]->loss_slot[par][peer]);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // the reference all-reduces in the loss dtype and divides the python float by W (distributed.py:640-646)
    float sum = 0.f;
    for (int r = 0; r < world; ++r) sum += s_val[r];
    *out_host = (double)sum / (double)world;
    __threadfence_system();
  }
}

__global__ void k_barrier(PeerPads pads, int rank, int world, uint32_t epoch) {
  if (threadIdx.x < (unsigned)world) {
    const int peer = threadIdx.x;
    __threadfence_system();
    st_release_sys(&pads.p[peer]->aux_flag[2][rank], epoch);
    wait_flag(&pads.p[rank]->aux_flag[2][peer], epoch, pads.p[rank]);
  }
}

// peers pull `nvec16` 16-byte vectors from src (root's buffer, peer-mapped) into dst (local)
__global__ void __launch_bounds__(512) k_bcast_pull(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t nvec16,
                                                     size_t tail_bytes, PeerPads pads, int rank, int world, int is_root,
                                                     uint32_t epoch) {
  // root's data is complete (stream order on the root); a missing peer: give up (error word set)
  if (!block_barrier_all_ranks(pads, rank, world, 0, epoch)) return;
  if (!is_root) {
    const size_t stride = size_t(gridDim.x) * blockDim.x;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec16; i += stride) dst[i] = ld_stream16(src + i);
    if (blockIdx.x == 0 && threadIdx.x < tail_bytes) {
      const unsigned char* s8 = reinterpret_cast<const unsigned char*>(src + nvec16);
      unsigned char* d8 = reinterpret_cast<unsigned char*>(dst + nvec16);
      d8[threadIdx.x] = s8[threadIdx.x];
    }
  }
  block_barrier_all_ranks(pads, rank, world, 1, epoch);  // root may overwrite its buffer after this
}

}  // namespace stk

using namespace stk;

extern "C" {

static int launch_loss_sync(stk_ctx* c, const void* loss_dev, int dtype, double* dst, cudaStream_t s) {
  uint32_t epoch = ++c->aux_epoch[1];
  switch (dtype) {
    case STK_F32: k_loss_sync<STK_F32><<<1, 32, 0, s>>>(loss_dev, dst, c->pads, c->rank, c->world, epoch); break;
    case STK_BF16: k_loss_sync<STK_BF16><<<1, 32, 0, s>>>(loss_dev, dst, c->pads, c->rank, c->world, epoch); break;
    case STK_F16: k_loss_sync<STK_F16><<<1, 32, 0, s>>>(loss_dev, dst, c->pads, c->rank, c->world, epoch); break;
    default: --c->aux_epoch[1]; return stk_fail(c, STK_ERR_INVALID, "stk_loss_sync: bad dtype");
  }
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

int stk_loss_sync(stk_ctx* c, const void* loss_dev, int dtype, double* out_host, void* stream) {
  STK_REQUIRE(c, c && loss_dev && out_host, "stk_loss_sync: NULL argument");
  if (c->world > 1 && !c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_loss_sync before stk_comm_connect");
  STK_POLL(c);
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int rc = launch_loss_sync(c, loss_dev, dtype, c->host_scratch_dev /* slot 0 of the pinned, mapped scratch */, s);
  if (rc != STK_OK) return rc;
  STK_CUDA(c, cudaStreamSynchronize(s));
  STK_POLL(c);  // this call synchronised: a peer that never arrived is reported here, not one step later
  *out_host = c->host_scratch[0];
  return STK_OK;
}

int stk_loss_sync_begin(stk_ctx* c, const void* loss_dev, int dtype, int64_t* ticket_out, void* stream) {
  STK_REQUIRE(c, c && loss_dev && ticket_out, "stk_loss_sync_begin: NULL argument");
  if (c->world > 1 && !c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_loss_sync_begin before stk_comm_connect");
  STK_POLL(c);
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t ticket = c->loss_ticket;
  const int slot = (int)(ticket % STK_LOSS_RING);
  if (!c->loss_events[slot]) STK_CUDA(c, cudaEventCreateWithFlags(&c->loss_events[slot], cudaEventDisableTiming));
  int rc = launch_loss_sync(c, loss_dev, dtype, c->loss_ring_dev + slot, s);
  if (rc != STK_OK) return rc;
  STK_CUDA(c, cudaEventRecord(c->loss_events[slot], s));
  c->loss_ticket = ticket + 1;
  *ticket_out = ticket;
  return STK_OK;
}

int stk_loss_sync_wait(stk_ctx* c, int64_t ticket, double* out_host) {
  STK_REQUIRE(c, c && out_host, "stk_loss_sync_wait: NULL argument");
  cudaEvent_t ev;
  {
    std::lock_guard<std::mutex> lk(c->mu);
    STK_REQUIRE(c, ticket >= 0 && ticket < c->loss_ticket, "stk_loss_sync_wait: no such ticket");
    if (c->loss_ticket - ticket > STK_LOSS_RING)
      return stk_fail(c, STK_ERR_STATE, "stk_loss_sync_wait: the ticket's slot has been overwritten (more than STK_LOSS_RING outstanding)");
    ev = c->loss_events[ticket % STK_LOSS_RING];
  }
  DeviceGuard g(c->device);
  STK_CUDA(c, cudaEventSynchronize(ev));
  STK_POLL(c);
  *out_host = c->loss_ring[ticket % STK_LOSS_RING];
  return STK_OK;
}

int stk_barrier(stk_ctx* c, void* stream) {
  STK_REQUIRE(c, c != nullptr, "stk_barrier: NULL ctx");
  if (c->world == 1) return STK_OK;
  if (!c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_barrier before stk_comm_connect");
  STK_POLL(c);
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  k_barrier<<<1, 32, 0, s>>>(c->pads, c->rank, c->world, ++c->aux_epoch[2]);
  STK_CUDA(c, cudaGetLastError());
  STK_CUDA(c, cudaStreamSynchronize(s));
  STK_POLL(c);
  return STK_OK;
}

int stk_bcast(stk_ctx* c, void* const* ptrs, size_t bytes, int root, void* stream) {
  STK_REQUIRE(c, c && ptrs, "stk_bcast: NULL argument");
  STK_REQUIRE(c, root >= 0 && root < c->world, "stk_bcast: bad root");
  if (c->world == 1 || bytes == 0) return STK_OK;
  if (!c->comm_ready) return stk_fail(c, STK_ERR_STATE, "stk_bcast before stk_comm_connect");
  STK_POLL(c);
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t nvec = bytes / 16, tail = bytes % 16;
  int grid = (int)std::max<size_t>(1, std::min<size_t>((nvec + 511) / 512, (size_t)c->sm_count));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(512);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  coop_attr(cfg, attr);
  const uint4* src = reinterpret_cast<const uint4*>(ptrs[root]);
  uint4* dst = reinterpret_cast<uint4*>(ptrs[c->rank]);
  uint32_t epoch = ++c->blk_epoch;
  cudaError_t err = cudaLaunchKernelEx(&cfg, k_bcast_pull, src, dst, nvec, tail, c->pads, c->rank, c->world,
                                       (int)(root == c->rank), epoch);
  if (err != cudaSuccess) return stk_fail(c, STK_ERR_CUDA, std::string("k_bcast_pull launch: ") + cudaGetErrorString(err));
  return STK_OK;
}

}  // extern "C"

// ctx.cuh -- host-side context shared by the translation units of libstoke_b200.so
#pragma once
#include <atomic>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

struct StepAccum {          // per-optimizer-step accumulators on the device (local shard)
  float norm_partial;       // running sum / max over the buckets reduced so far
  uint32_t found_inf;
  uint32_t blocks_done;     // last-block detection counter (self-resetting)
  uint32_t pad_;
};

struct StepState {          // one per optimizer (stk_state_*): loss scaler + step counters + norm accumulators
  stk_scaler_state_t* scaler_dev = nullptr;
  StepAccum* accum_dev = nullptr;
};

struct FdServer;            // vmm.cu: serves exported POSIX file descriptors to the peer processes (SCM_RIGHTS)

struct stk_ctx {
  int rank = 0, world = 1, device = 0;
  int sm_count = 148;
  std::mutex mu;
  std::string err;
  // peer-visible allocations made through stk_mem_alloc_shared: local ptr -> peer mappings
  struct Shared {
    size_t bytes = 0;            // mapped size (rounded)
    void* peers[STK_MAX_WORLD] = {};
    bool opened = false;
    bool vmm = false;
    // vmm back end (driver handles kept as integers so this header needs no cuda.h)
    unsigned long long mem_handle = 0;               // CUmemGenericAllocationHandle of the local memory
    unsigned long long peer_handles[STK_MAX_WORLD] = {};
    int mem_fd = -1;                                 // exported descriptor (served to peers until the buffer is freed)
    unsigned long long mc_handle = 0;                // multicast object (0: none)
    int mc_fd = -1;                                  // rank 0: exported descriptor of the multicast object
    bool mc_added = false, mc_bound = false;
    void* mc_ptr = nullptr;                          // multicast mapping (nullptr: not bound)
  };
  std::map<void*, Shared> shared;
  int mem_mode = 0;             // 0: cudaMalloc + cudaIpc, 1: VMM + POSIX fd
  bool multicast_ok = false;    // device + driver support multicast objects
  FdServer* fd_server = nullptr;
  int serial = 0;               // process-unique context number (names the fd server's socket)
  // signal pads
  stk::SignalPad* pad_local = nullptr;
  stk::PeerPads pads{};
  bool comm_ready = false;
  uint32_t blk_epoch = 0;       // block-barrier epoch (identical sequence on every rank)
  uint32_t aux_epoch[4] = {0, 0, 0, 0};
  int k1_algo = 1;              // cross-rank K1 flavour: 0 = register-staged loads, 1 = bulk-async (default), 2 = multimem (NVLS)
  int k1_max_blocks = 0;        // 0: one block per SM
  int nvls_max_blocks = 0;      // grid bound of the multimem flavour (0: like the other flavours)
  // device state
  std::vector<StepState> states;      // [0] is created with the context
  int cur_state = 0;
  stk_scaler_state_t* scaler_dev = nullptr;   // == states[cur_state]
  StepAccum* accum_dev = nullptr;
  float* blk_partial_dev = nullptr;   // [blk_partial_cap] per-block norm partials of K1
  float* grp_partial_dev = nullptr;   // [blk_partial_cap / 64 + 1] per-group partials (two-level ticket)
  uint32_t* grp_count_dev = nullptr;  // [blk_partial_cap / 64 + 1] group tickets (self-resetting)
  size_t blk_partial_cap = 0;
  // optional launch timing (stk_profile_*): CUDA-event pairs recorded around the kernel launch, on the launch stream
  bool profiling = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof[4];  // 0: K1 reduce, 1: K2 optimizer step, 2: accumulate, 3: norm pass
  unsigned long long* prof_ns_dev = nullptr;                   // {ns, launches} written by K1's block 0 (device timer)
  std::map<const void*, int> occupancy;                       // kernel -> resident blocks per SM (cached query)
  // pinned, mapped host scratch: [0..3] doubles (loss sync), [4..11] scaler staging, word at [12] = error mirror
  double* host_scratch = nullptr;     // [16]
  double* host_scratch_dev = nullptr; // device alias of host_scratch
  // async loss ring
  double* loss_ring = nullptr;        // [STK_LOSS_RING] pinned, mapped
  double* loss_ring_dev = nullptr;
  cudaEvent_t loss_events[STK_LOSS_RING] = {};
  int64_t loss_ticket = 0;

  volatile uint32_t* host_err() const { return reinterpret_cast<volatile uint32_t*>(host_scratch + 12); }
};

extern thread_local std::string g_tls_err;
int stk_fail(stk_ctx* ctx, int code, const std::string& msg);

#define STK_CUDA(ctx, call)                                                                              \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess)                                                                              \
      return stk_fail(ctx, STK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));           \
  } while (0)

#define STK_REQUIRE(ctx, cond, msg)                                   \
  do {                                                                \
    if (!(cond)) return stk_fail(ctx, STK_ERR_INVALID, (msg));        \
  } while (0)

// every cross-rank entry point: a kernel on this rank gave up on a peer earlier -> fail instead of launching on garbage
#define STK_POLL(ctx)                                                                                                 \
  do {                                                                                                                \
    if ((ctx)->host_scratch && *(ctx)->host_err() != 0)                                                               \
      return stk_fail(ctx, STK_ERR_PEER, "a peer rank did not arrive within the spin bound (dead or out-of-order rank)"); \
  } while (0)

int stk_grow_partials(stk_ctx* c, size_t blocks, cudaStream_t s);

// vmm.cu
bool stk_vmm_available(int device, bool* multicast);
int stk_vmm_alloc(stk_ctx* c, size_t bytes, void** local_ptr, unsigned char* handle_out);
int stk_vmm_open(stk_ctx* c, stk_ctx::Shared& sh, const unsigned char* handles);
int stk_vmm_free(stk_ctx* c, void* local_ptr, stk_ctx::Shared& sh);
int stk_vmm_mc_bind(stk_ctx* c, stk_ctx::Shared& sh);
int stk_vmm_mc_release(stk_ctx* c, stk_ctx::Shared& sh);
void stk_vmm_ctx_shutdown(stk_ctx* c);
// multicast address corresponding to a local address inside a bound shared buffer (nullptr: not bound)
void* stk_mc_lookup(stk_ctx* c, const void* local);

struct ProfScope {  // records an event pair around a launch when profiling is on
  stk_ctx* c;
  int kind;
  cudaStream_t s;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  ProfScope(stk_ctx* ctx, int k, cudaStream_t st) : c(ctx), kind(k), s(st) {
    if (c->profiling && cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess) cudaEventRecord(e0, s);
  }
  ~ProfScope() {
    if (e0 && e1) {
      cudaEventRecord(e1, s);
      c->prof[kind].emplace_back(e0, e1);
    }
  }
};

template <typename K>
static inline int blocks_per_sm(stk_ctx* c, K kernel, int threads, size_t smem = 0) {
  const void* key = reinterpret_cast<const void*>(kernel);
  auto it = c->occupancy.find(key);
  if (it != c->occupancy.end()) return it->second;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  c->occupancy[key] = per_sm;
  return per_sm;
}

// Every cross-rank kernel spins on its peers' blocks, so all of its blocks must be co-resident: the cooperative attribute
// makes the launch fail instead of deadlocking when the grid does not fit.  `attr` must outlive the launch call.
inline void coop_attr(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr) {
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

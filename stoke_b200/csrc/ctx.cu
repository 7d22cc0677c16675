// ctx.cu -- context, peer-visible memory (CUDA IPC), signal pads, scaler state.  Host code + two tiny kernels.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "ctx.cuh"

thread_local std::string g_tls_err;

int stk_fail(stk_ctx* ctx, int code, const std::string& msg) {
  g_tls_err = msg;
  if (ctx) ctx->err = msg;
  return code;
}

int stk_grow_partials(stk_ctx* c, size_t blocks, cudaStream_t s) {
  if (blocks <= c->blk_partial_cap) return STK_OK;
  const size_t groups = blocks / 64 + 1;
  float *bp = nullptr, *gp = nullptr;
  uint32_t* gc = nullptr;
  STK_CUDA(c, cudaMalloc(&bp, sizeof(float) * blocks));
  STK_CUDA(c, cudaMalloc(&gp, sizeof(float) * groups));
  STK_CUDA(c, cudaMalloc(&gc, sizeof(uint32_t) * groups));
  STK_CUDA(c, cudaMemset(gc, 0, sizeof(uint32_t) * groups));
  if (c->blk_partial_dev) {
    STK_CUDA(c, cudaStreamSynchronize(s));  // a previous launch may still use the old arrays
    cudaFree(c->blk_partial_dev);
    cudaFree(c->grp_partial_dev);
    cudaFree(c->grp_count_dev);
  }
  c->blk_partial_dev = bp;
  c->grp_partial_dev = gp;
  c->grp_count_dev = gc;
  c->blk_partial_cap = blocks;
  return STK_OK;
}

extern "C" {

int stk_version(void) { return 201; }

const char* stk_last_error(stk_ctx* ctx) {
  if (ctx && !ctx->err.empty()) return ctx->err.c_str();
  return g_tls_err.c_str();
}

int stk_ctx_create(int rank, int world, int device, unsigned flags, stk_ctx** out) {
  (void)flags;
  STK_REQUIRE(nullptr, out != nullptr, "stk_ctx_create: out is NULL");
  STK_REQUIRE(nullptr, world >= 1 && world <= STK_MAX_WORLD, "stk_ctx_create: world must be in [1, 8]");
  STK_REQUIRE(nullptr, rank >= 0 && rank < world, "stk_ctx_create: rank out of range");
  int ndev = 0;
  STK_CUDA(nullptr, cudaGetDeviceCount(&ndev));
  STK_REQUIRE(nullptr, device >= 0 && device < ndev, "stk_ctx_create: no such CUDA device");
  DeviceGuard g(device);
  cudaDeviceProp prop;
  STK_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return stk_fail(nullptr, STK_ERR_UNSUPPORTED, "stoke_b200 needs an sm_100 (Blackwell) device");
  stk_ctx* c = new stk_ctx();
  c->rank = rank;
  c->world = world;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (const char* algo = std::getenv("STK_K1_ALGO"))
    c->k1_algo = (std::strcmp(algo, "nvls") == 0) ? 2 : (std::strcmp(algo, "bulk") == 0) ? 1 : 0;
  // memory back end: VMM (needed for NVLS multicast) when there are peers and the driver supports it
  bool mc = false;
  const bool vmm = stk_vmm_available(device, &mc);
  c->multicast_ok = vmm && mc && world > 1;
  c->mem_mode = (vmm && world > 1) ? 1 : 0;
  if (const char* m = std::getenv("STK_MEM")) {
    if (std::strcmp(m, "ipc") == 0) c->mem_mode = 0;
    else if (std::strcmp(m, "vmm") == 0 && vmm) c->mem_mode = 1;
  }
  if (const char* m = std::getenv("STK_MULTICAST"))
    if (std::atoi(m) == 0) c->multicast_ok = false;   // keep VMM memory but never create / bind multicast objects
  if (c->mem_mode == 0) c->multicast_ok = false;
  cudaError_t e;
  if ((e = cudaMalloc(&c->prof_ns_dev, 8 * sizeof(unsigned long long))) != cudaSuccess ||
      (e = cudaMemset(c->prof_ns_dev, 0, 8 * sizeof(unsigned long long))) != cudaSuccess ||
      (e = cudaHostAlloc(&c->host_scratch, sizeof(double) * 16, cudaHostAllocMapped)) != cudaSuccess ||
      (e = cudaHostGetDevicePointer(&c->host_scratch_dev, c->host_scratch, 0)) != cudaSuccess ||
      (e = cudaHostAlloc(&c->loss_ring, sizeof(double) * STK_LOSS_RING, cudaHostAllocMapped)) != cudaSuccess ||
      (e = cudaHostGetDevicePointer(&c->loss_ring_dev, c->loss_ring, 0)) != cudaSuccess) {
    delete c;
    return stk_fail(nullptr, STK_ERR_CUDA, std::string("stk_ctx_create: ") + cudaGetErrorString(e));
  }
  std::memset(c->host_scratch, 0, sizeof(double) * 16);
  std::memset(c->loss_ring, 0, sizeof(double) * STK_LOSS_RING);
  {
    int id = -1;
    if (stk_state_create(c, &id) != STK_OK || id != 0) {
      delete c;
      return STK_ERR_CUDA;
    }
    stk_state_select(c, 0);
  }
  if (stk_grow_partials(c, stk::kMaxBlocks, nullptr) != STK_OK) {
    delete c;
    return STK_ERR_CUDA;
  }
  for (int i = 0; i < STK_MAX_WORLD; ++i) c->pads.p[i] = nullptr;
  *out = c;
  return STK_OK;
}

int stk_ctx_destroy(stk_ctx* c) {
  if (!c) return STK_OK;
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();
  for (auto& kv : c->shared) {
    if (kv.second.vmm) {
      stk_vmm_free(c, kv.first, kv.second);
      continue;
    }
    if (kv.second.opened)
      for (int r = 0; r < c->world; ++r)
        if (r != c->rank && kv.second.peers[r]) cudaIpcCloseMemHandle(kv.second.peers[r]);
    cudaFree(kv.first);
  }
  c->shared.clear();
  stk_vmm_ctx_shutdown(c);
  if (c->comm_ready)
    for (int r = 0; r < c->world; ++r)
      if (r != c->rank && c->pads.p[r]) cudaIpcCloseMemHandle(c->pads.p[r]);
  if (c->pad_local) cudaFree(c->pad_local);
  for (auto& st : c->states) {
    if (st.scaler_dev) cudaFree(st.scaler_dev);
    if (st.accum_dev) cudaFree(st.accum_dev);
  }
  for (auto& ev : c->loss_events)
    if (ev) cudaEventDestroy(ev);
  if (c->loss_ring) cudaFreeHost(c->loss_ring);
  cudaFree(c->blk_partial_dev);
  cudaFree(c->grp_partial_dev);
  cudaFree(c->grp_count_dev);
  cudaFree(c->prof_ns_dev);
  cudaFreeHost(c->host_scratch);
  delete c;
  return STK_OK;
}

int stk_caps(stk_ctx* c, stk_caps_t* out) {
  STK_REQUIRE(c, c && out, "stk_caps: NULL argument");
  DeviceGuard g(c->device);
  cudaDeviceProp prop;
  STK_CUDA(c, cudaGetDeviceProperties(&prop, c->device));
  out->sm_major = prop.major;
  out->sm_minor = prop.minor;
  out->sm_count = prop.multiProcessorCount;
  out->rank = c->rank;
  out->world = c->world;
  out->device = c->device;
  out->peer_access = (c->world == 1) || c->comm_ready;
  out->multicast = c->multicast_ok ? 1 : 0;
  out->hbm_bytes = prop.totalGlobalMem;
  return STK_OK;
}

// ---- peer-visible memory ---------------------------------------------------------------------------------------------
int stk_mem_alloc_shared(stk_ctx* c, size_t bytes, void** local_ptr, unsigned char handle_out[STK_IPC_HANDLE_BYTES]) {
  STK_REQUIRE(c, c && local_ptr && handle_out, "stk_mem_alloc_shared: NULL argument");
  STK_REQUIRE(c, bytes > 0, "stk_mem_alloc_shared: zero bytes");
  static_assert(sizeof(cudaIpcMemHandle_t) == STK_IPC_HANDLE_BYTES, "IPC handle size");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  if (c->mem_mode == 1 && c->world > 1) return stk_vmm_alloc(c, bytes, local_ptr, handle_out);
  void* p = nullptr;
  size_t rounded = (bytes + 255) & ~size_t(255);
  STK_CUDA(c, cudaMalloc(&p, rounded));
  STK_CUDA(c, cudaMemset(p, 0, rounded));
  std::memset(handle_out, 0, STK_IPC_HANDLE_BYTES);
  if (c->world > 1) {
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
      cudaFree(p);
      return stk_fail(c, STK_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    }
    std::memcpy(handle_out, &h, sizeof(h));
  }
  stk_ctx::Shared s{};
  s.bytes = rounded;
  s.peers[c->rank] = p;
  c->shared[p] = s;
  *local_ptr = p;
  return STK_OK;
}

int stk_mem_open_peers(stk_ctx* c, void* local_ptr, const unsigned char* handles, void** peer_ptrs_out) {
  STK_REQUIRE(c, c && local_ptr && peer_ptrs_out, "stk_mem_open_peers: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  auto it = c->shared.find(local_ptr);
  STK_REQUIRE(c, it != c->shared.end(), "stk_mem_open_peers: pointer was not allocated by stk_mem_alloc_shared");
  DeviceGuard g(c->device);
  if (!it->second.opened && c->world > 1 && it->second.vmm) {
    STK_REQUIRE(c, handles != nullptr, "stk_mem_open_peers: handles is NULL");
    int rc = stk_vmm_open(c, it->second, handles);
    if (rc != STK_OK) return rc;
  } else if (!it->second.opened && c->world > 1) {
    STK_REQUIRE(c, handles != nullptr, "stk_mem_open_peers: handles is NULL");
    for (int r = 0; r < c->world; ++r) {
      if (r == c->rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles + size_t(r) * STK_IPC_HANDLE_BYTES, sizeof(h));
      void* p = nullptr;
      STK_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      it->second.peers[r] = p;
    }
  }
  it->second.opened = true;
  for (int r = 0; r < c->world; ++r) peer_ptrs_out[r] = it->second.peers[r];
  return STK_OK;
}

int stk_mem_free_shared(stk_ctx* c, void* local_ptr) {
  STK_REQUIRE(c, c != nullptr, "stk_mem_free_shared: NULL ctx");
  if (!local_ptr) return STK_OK;
  std::lock_guard<std::mutex> lk(c->mu);
  auto it = c->shared.find(local_ptr);
  STK_REQUIRE(c, it != c->shared.end(), "stk_mem_free_shared: unknown pointer");
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();  // no kernel of this process may still be using the mapping
  if (it->second.vmm) {
    stk_vmm_free(c, local_ptr, it->second);
  } else {
    if (it->second.opened)
      for (int r = 0; r < c->world; ++r)
        if (r != c->rank && it->second.peers[r]) cudaIpcCloseMemHandle(it->second.peers[r]);
    cudaFree(local_ptr);
  }
  c->shared.erase(it);
  return STK_OK;
}

int stk_multicast_try_bind(stk_ctx* c, void* local_ptr, void** mc_ptr_out) {
  STK_REQUIRE(c, c && local_ptr && mc_ptr_out, "stk_multicast_try_bind: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  auto it = c->shared.find(local_ptr);
  STK_REQUIRE(c, it != c->shared.end(), "stk_multicast_try_bind: pointer was not allocated by stk_mem_alloc_shared");
  *mc_ptr_out = nullptr;
  if (!c->multicast_ok || !it->second.vmm || !it->second.opened)
    return stk_fail(c, STK_ERR_UNSUPPORTED, "multicast is not available for this buffer (no NVLS support, ipc memory mode, or peers not opened)");
  DeviceGuard g(c->device);
  int rc = stk_vmm_mc_bind(c, it->second);
  if (rc != STK_OK) return rc;
  *mc_ptr_out = it->second.mc_ptr;
  return STK_OK;
}

int stk_multicast_release(stk_ctx* c, void* local_ptr) {
  STK_REQUIRE(c, c && local_ptr, "stk_multicast_release: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  auto it = c->shared.find(local_ptr);
  STK_REQUIRE(c, it != c->shared.end(), "stk_multicast_release: unknown pointer");
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();
  if (it->second.vmm) stk_vmm_mc_release(c, it->second);
  return STK_OK;
}

// ---- signal pads -----------------------------------------------------------------------------------------------------
int stk_comm_local(stk_ctx* c, unsigned char handle_out[STK_IPC_HANDLE_BYTES]) {
  STK_REQUIRE(c, c && handle_out, "stk_comm_local: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  if (!c->pad_local) {
    STK_CUDA(c, cudaMalloc(&c->pad_local, sizeof(stk::SignalPad)));
    STK_CUDA(c, cudaMemset(c->pad_local, 0, sizeof(stk::SignalPad)));
    // local-only fields: the spin bound and the error word's mirror in mapped host memory
    uint64_t timeout = stk::kDefaultSpinTimeoutNs;
    if (const char* t = std::getenv("STK_SPIN_TIMEOUT_S")) {
      double sec = std::atof(t);
      if (sec > 0) timeout = (uint64_t)(sec * 1e9);
    }
    uint32_t* herr = reinterpret_cast<uint32_t*>(c->host_scratch_dev + 12);
    STK_CUDA(c, cudaMemcpy(&c->pad_local->timeout_ns, &timeout, sizeof(timeout), cudaMemcpyHostToDevice));
    STK_CUDA(c, cudaMemcpy(&c->pad_local->host_err, &herr, sizeof(herr), cudaMemcpyHostToDevice));
    STK_CUDA(c, cudaDeviceSynchronize());
  }
  std::memset(handle_out, 0, STK_IPC_HANDLE_BYTES);
  if (c->world > 1) {
    cudaIpcMemHandle_t h;
    STK_CUDA(c, cudaIpcGetMemHandle(&h, c->pad_local));
    std::memcpy(handle_out, &h, sizeof(h));
  }
  return STK_OK;
}

int stk_comm_connect(stk_ctx* c, const unsigned char* handles) {
  STK_REQUIRE(c, c != nullptr, "stk_comm_connect: NULL ctx");
  std::lock_guard<std::mutex> lk(c->mu);
  if (!c->pad_local) return stk_fail(c, STK_ERR_STATE, "stk_comm_connect before stk_comm_local");
  if (c->comm_ready) return STK_OK;
  DeviceGuard g(c->device);
  c->pads.p[c->rank] = c->pad_local;
  if (c->world > 1) {
    STK_REQUIRE(c, handles != nullptr, "stk_comm_connect: handles is NULL");
    for (int r = 0; r < c->world; ++r) {
      if (r == c->rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles + size_t(r) * STK_IPC_HANDLE_BYTES, sizeof(h));
      void* p = nullptr;
      STK_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      c->pads.p[r] = reinterpret_cast<stk::SignalPad*>(p);
    }
  }
  c->comm_ready = true;
  return STK_OK;
}

int stk_comm_check(stk_ctx* c, void* stream) {
  STK_REQUIRE(c, c != nullptr, "stk_comm_check: NULL ctx");
  if (!c->pad_local) return STK_OK;
  DeviceGuard g(c->device);
  uint32_t err = 0;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  STK_CUDA(c, cudaMemcpyAsync(&err, &c->pad_local->error, sizeof(err), cudaMemcpyDeviceToHost, s));
  STK_CUDA(c, cudaStreamSynchronize(s));
  if (err || *c->host_err() != 0)
    return stk_fail(c, STK_ERR_PEER, "a peer rank did not arrive within the spin bound (dead or out-of-order rank)");
  return STK_OK;
}

int stk_comm_poll(stk_ctx* c) {
  STK_REQUIRE(c, c != nullptr, "stk_comm_poll: NULL ctx");
  STK_POLL(c);
  return STK_OK;
}

// ---- per-optimizer state ---------------------------------------------------------------------------------------------
int stk_state_create(stk_ctx* c, int* id_out) {
  STK_REQUIRE(c, c && id_out, "stk_state_create: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  StepState st;
  STK_CUDA(c, cudaMalloc(&st.scaler_dev, sizeof(stk_scaler_state_t)));
  STK_CUDA(c, cudaMalloc(&st.accum_dev, sizeof(StepAccum)));
  stk_scaler_state_t init{};
  init.scale = 1.f;
  init.growth_factor = 2.f;
  init.backoff_factor = 0.5f;
  init.growth_interval = 2000;
  STK_CUDA(c, cudaMemcpy(st.scaler_dev, &init, sizeof(init), cudaMemcpyHostToDevice));
  STK_CUDA(c, cudaMemset(st.accum_dev, 0, sizeof(StepAccum)));
  int id = -1;
  for (size_t i = 0; i < c->states.size(); ++i)
    if (!c->states[i].scaler_dev) {
      id = (int)i;
      break;
    }
  if (id < 0) {
    id = (int)c->states.size();
    c->states.emplace_back();
  }
  c->states[id] = st;
  *id_out = id;
  return STK_OK;
}

int stk_state_select(stk_ctx* c, int id) {
  STK_REQUIRE(c, c != nullptr, "stk_state_select: NULL ctx");
  std::lock_guard<std::mutex> lk(c->mu);
  STK_REQUIRE(c, id >= 0 && id < (int)c->states.size() && c->states[id].scaler_dev, "stk_state_select: no such state");
  c->cur_state = id;
  c->scaler_dev = c->states[id].scaler_dev;
  c->accum_dev = c->states[id].accum_dev;
  return STK_OK;
}

int stk_state_destroy(stk_ctx* c, int id) {
  STK_REQUIRE(c, c != nullptr, "stk_state_destroy: NULL ctx");
  std::lock_guard<std::mutex> lk(c->mu);
  STK_REQUIRE(c, id > 0 && id < (int)c->states.size() && c->states[id].scaler_dev, "stk_state_destroy: no such state (state 0 lives with the context)");
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();
  cudaFree(c->states[id].scaler_dev);
  cudaFree(c->states[id].accum_dev);
  c->states[id] = StepState{};
  if (c->cur_state == id) {
    c->cur_state = 0;
    c->scaler_dev = c->states[0].scaler_dev;
    c->accum_dev = c->states[0].accum_dev;
  }
  return STK_OK;
}

// ---- scaler state ----------------------------------------------------------------------------------------------------
int stk_scaler_set(stk_ctx* c, const stk_scaler_state_t* st, void* stream) {
  STK_REQUIRE(c, c && st, "stk_scaler_set: NULL argument");
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // staged through the pinned scratch so the async copy reads stable memory
  std::lock_guard<std::mutex> lk(c->mu);
  STK_CUDA(c, cudaStreamSynchronize(s));
  std::memcpy(c->host_scratch + 4, st, sizeof(*st));
  STK_CUDA(c, cudaMemcpyAsync(c->scaler_dev, c->host_scratch + 4, sizeof(*st), cudaMemcpyHostToDevice, s));
  STK_CUDA(c, cudaStreamSynchronize(s));
  return STK_OK;
}

int stk_scaler_get(stk_ctx* c, stk_scaler_state_t* st, void* stream) {
  STK_REQUIRE(c, c && st, "stk_scaler_get: NULL argument");
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  STK_CUDA(c, cudaMemcpyAsync(st, c->scaler_dev, sizeof(*st), cudaMemcpyDeviceToHost, s));
  STK_CUDA(c, cudaStreamSynchronize(s));
  return STK_OK;
}

void* stk_scaler_scale_ptr(stk_ctx* c) { return c ? static_cast<void*>(&c->scaler_dev->scale) : nullptr; }

int stk_option_set(stk_ctx* c, int key, int value) {
  STK_REQUIRE(c, c != nullptr, "stk_option_set: NULL ctx");
  std::lock_guard<std::mutex> lk(c->mu);
  switch (key) {
    case STK_OPT_K1_ALGO:
      STK_REQUIRE(c, value >= 0 && value <= 2, "stk_option_set: K1 algo must be 0 (ldg), 1 (bulk) or 2 (nvls)");
      c->k1_algo = value;
      return STK_OK;
    case STK_OPT_MEM_MODE:
      STK_REQUIRE(c, value == 0 || value == 1, "stk_option_set: memory mode must be 0 (ipc) or 1 (vmm)");
      if (value == 1 && !stk_vmm_available(c->device, nullptr))
        return stk_fail(c, STK_ERR_UNSUPPORTED, "stk_option_set: the driver / device has no VMM + POSIX descriptor support");
      c->mem_mode = value;
      if (value == 0) c->multicast_ok = false;
      return STK_OK;
    case STK_OPT_K1_MAX_BLOCKS:
      STK_REQUIRE(c, value >= 0 && value <= stk::kMaxReduceBlocks, "stk_option_set: K1 max blocks out of range");
      c->k1_max_blocks = value;
      return STK_OK;
    case STK_OPT_NVLS_MAX_BLOCKS:
      STK_REQUIRE(c, value >= 0 && value <= stk::kMaxReduceBlocks, "stk_option_set: NVLS max blocks out of range");
      c->nvls_max_blocks = value;
      return STK_OK;
    default:
      return stk_fail(c, STK_ERR_INVALID, "stk_option_set: unknown key");
  }
}

int stk_option_get(stk_ctx* c, int key, int* value) {
  STK_REQUIRE(c, c && value, "stk_option_get: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  switch (key) {
    case STK_OPT_K1_ALGO: *value = c->k1_algo; return STK_OK;
    case STK_OPT_MEM_MODE: *value = c->mem_mode; return STK_OK;
    case STK_OPT_K1_MAX_BLOCKS: *value = c->k1_max_blocks; return STK_OK;
    case STK_OPT_NVLS_MAX_BLOCKS: *value = c->nvls_max_blocks; return STK_OK;
    default: return stk_fail(c, STK_ERR_INVALID, "stk_option_get: unknown key");
  }
}

int stk_profile_enable(stk_ctx* c, int on) {
  STK_REQUIRE(c, c != nullptr, "stk_profile_enable: NULL ctx");
  std::lock_guard<std::mutex> lk(c->mu);
  c->profiling = on != 0;
  return STK_OK;
}

int stk_profile_read(stk_ctx* c, int kind, double* ms_total, int* launches) {
  STK_REQUIRE(c, c && ms_total && launches && kind >= 0 && kind < 4, "stk_profile_read: bad argument");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  double tot = 0.0;
  int n = 0;
  for (auto& pr : c->prof[kind]) {
    float ms = 0.f;
    if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
      tot += ms;
      ++n;
    }
    cudaEventDestroy(pr.first);
    cudaEventDestroy(pr.second);
  }
  c->prof[kind].clear();
  *ms_total = tot;
  *launches = n;
  return STK_OK;
}

int stk_profile_read_k1_device(stk_ctx* c, double* ms_total, int* launches, double* ms_zero_tail, void* stream) {
  STK_REQUIRE(c, c && ms_total && launches, "stk_profile_read_k1_device: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  unsigned long long v[4] = {0, 0, 0, 0};
  STK_CUDA(c, cudaMemcpyAsync(v, c->prof_ns_dev, sizeof(v), cudaMemcpyDeviceToHost, s));
  STK_CUDA(c, cudaMemsetAsync(c->prof_ns_dev, 0, sizeof(v), s));
  STK_CUDA(c, cudaStreamSynchronize(s));
  *ms_total = (double)v[0] * 1e-6;
  *launches = (int)v[1];
  if (ms_zero_tail) *ms_zero_tail = (double)v[2] * 1e-6;
  return STK_OK;
}

int stk_profile_read_k2_device(stk_ctx* c, double* ms_total, int* launches, void* stream) {
  STK_REQUIRE(c, c && ms_total && launches, "stk_profile_read_k2_device: NULL argument");
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard g(c->device);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  unsigned long long v[2] = {0, 0};
  STK_CUDA(c, cudaMemcpyAsync(v, c->prof_ns_dev + 4, sizeof(v), cudaMemcpyDeviceToHost, s));
  STK_CUDA(c, cudaMemsetAsync(c->prof_ns_dev + 4, 0, sizeof(v), s));
  STK_CUDA(c, cudaStreamSynchronize(s));
  *ms_total = (double)v[0] * 1e-6;
  *launches = (int)v[1];
  return STK_OK;
}

int stk_shard_range(size_t n, int world, int rank, size_t* begin, size_t* end) {
  if (!begin || !end || world < 1 || rank < 0 || rank >= world) return stk_fail(nullptr, STK_ERR_INVALID, "stk_shard_range: bad argument");
  // shards are multiples of 16 elements (32 B of bf16: the sharded optimizer step pushes 32-byte sectors to its peers)
  size_t vecs = (n + 7) / 8;
  size_t per = (vecs + world - 1) / world;
  per += per & 1;
  size_t b = per * rank * 8, e = per * (rank + 1) * 8;
  if (b > n) b = n;
  if (e > n) e = n;
  *begin = b;
  *end = e;
  return STK_OK;
}

}  // extern "C"

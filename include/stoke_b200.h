/*
 * stoke_b200.h -- C ABI of libstoke_b200.so (hand-written sm_100a kernels for the post-backward gradient path of
 * fidelity/stoke).  Plain C: opaque context, raw device pointers, sizes, and a cudaStream_t passed as void*.  No torch
 * types.  Every function returns 0 on success or a negative stk_status; the message is available through
 * stk_last_error().  No function synchronises the device unless its comment says so.  A context may be used from any
 * host thread (internally locked); all launches go to the stream the caller passes.
 *
 * What each entry point replaces in the reference (paths relative to /root/reference):
 *
 *   stk_ctx_create / stk_comm_*     process-group bring-up            stoke/distributed.py:491-538 (DistributedDDP)
 *   stk_mem_*                        DDP bucket storage (torch Reducer buckets, NCCL buffers)  stoke/extensions.py:207-215
 *   stk_grad_accumulate              local accumulation under no_sync  stoke/distributed.py:648-669, stoke/stoke.py:978-984
 *   stk_grad_reduce                  DDP bucket copy-in + all-reduce + copy-out (stoke/extensions.py:207-215), fused with
 *                                    GradScaler.unscale_ (stoke/fp16.py:180-183,222-225) and the norm / inf reductions of
 *                                    clip_grad_norm_ (stoke/fp16.py:233); reduce-scatter flavour = fairscale SDDP/OSS
 *                                    reduce-to-owner (stoke/extensions.py:277-285)
 *   stk_optim_step                   clip_grad_norm_/clip_grad_value_ scaling (stoke/fp16.py:184,233), scaler.step gate +
 *                                    optimizer.step() (stoke/fp16.py:298,805), OSS shard step + parameter broadcast
 *                                    (stoke/extensions.py:136-141 -> fairscale OSS.step)
 *   stk_step_epilogue                scaler.update() (stoke/fp16.py:806) + zero_grad bookkeeping (stoke/utils.py:83-106)
 *   stk_loss_sync                    detach_and_sync_loss: item + barrier + all_reduce + item  stoke/distributed.py:619-646
 *   stk_barrier                      torch.distributed.barrier()      stoke/distributed.py:673
 *   stk_bcast                        DDP init param sync / per-forward buffer broadcast (broadcast_buffers=True,
 *                                    stoke/configs.py:182)
 *   stk_randperm / stk_argsort_u32 / stk_sampler_*    BucketedDistributedSampler  stoke/data.py:156-266, 380-498
 *   stk_state_*                      one scaler / step-counter / norm state per optimizer (the reference keeps them per
 *                                    GradScaler / per optimizer object: stoke/fp16.py:733-806, stoke/extensions.py:53-78)
 *   stk_multicast_try_bind           NCCL's NVLS transport under DDP (stoke/extensions.py:207-215): an NVSwitch multicast
 *                                    mapping of a peer-visible buffer, used by the multimem flavour of stk_grad_reduce
 *   stk_grad_norm                    the two reduction passes of clip_grad_norm_ + GradScaler.unscale_'s inf test
 *                                    (stoke/fp16.py:180-183, 233) when there is no cross-rank reduce to fuse them into
 *   stk_grad_scale                   clip_grad_norm_'s scaling pass / clip_grad_value_ (stoke/fp16.py:184, 233) for the
 *                                    stock-optimizer route (any torch.optim class, stoke/extensions.py:53-78)
 *   stk_loss_sync_begin/_wait        detach_and_sync_loss without the per-micro-step host synchronisation
 *   stk_optim_range_prologue         torch's per-parameter `state[p]["step"]` (torch/optim/adam.py: a parameter whose grad is None
 *                                    is not stepped and keeps its own count) for models with sometimes-unused parameters
 */
#ifndef STOKE_B200_H
#define STOKE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STK_MAX_WORLD 8
#define STK_IPC_HANDLE_BYTES 64

typedef struct stk_ctx stk_ctx;

typedef enum {
  STK_OK = 0,
  STK_ERR_INVALID = -1,   /* bad argument */
  STK_ERR_CUDA = -2,      /* a CUDA runtime call failed (no device, OOM, launch failure, ...) */
  STK_ERR_STATE = -3,     /* call order violated (e.g. reduce before comm connect) */
  STK_ERR_PEER = -4,      /* a peer did not arrive within the spin bound (dead or out-of-order rank) */
  STK_ERR_UNSUPPORTED = -5
} stk_status;

typedef enum { STK_F32 = 0, STK_BF16 = 1, STK_F16 = 2 } stk_dtype;

typedef enum {
  STK_REDUCE_ALL = 0,     /* all-reduce: owner reduces its shard and pushes the result to every rank */
  STK_REDUCE_SCATTER = 1  /* reduce-scatter: owner keeps its shard (ZeRO-1 / OSS) */
} stk_reduce_mode;

typedef enum { STK_NORM_NONE = 0, STK_NORM_L2 = 1, STK_NORM_INF = 2, STK_NORM_P = 3 } stk_norm_kind;
typedef enum { STK_CLIP_NONE = 0, STK_CLIP_NORM = 1, STK_CLIP_VALUE = 2 } stk_clip_kind;
typedef enum { STK_OPT_ADAM = 0, STK_OPT_ADAMW = 1, STK_OPT_SGD = 2 } stk_optim_kind;

/* flags of stk_grad_reduce */
#define STK_RF_FINAL 1u        /* last bucket of this optimizer step: finish norm / found_inf (cross-rank exchange) */
#define STK_RF_ZERO_INPUT 2u   /* zero the local gradient bucket (and accumulator) after it has been consumed */
#define STK_RF_UNSCALE 4u      /* multiply by 1/loss_scale (device scaler state) and test for inf/nan */

typedef struct {
  int sm_major, sm_minor, sm_count;
  int rank, world, device;
  int peer_access;        /* 1 if every peer's memory is mapped */
  int multicast;          /* 1 if the device reports CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED and the driver's VMM / multicast
                             entry points resolved (whether a given buffer is bound: stk_multicast_try_bind) */
  size_t hbm_bytes;
} stk_caps_t;

/* device-resident loss-scaler / step state (one per context); mirrors torch.amp.GradScaler's state_dict */
typedef struct {
  float scale;            /* current loss scale */
  float growth_factor, backoff_factor;
  int32_t growth_interval;
  int32_t growth_tracker;
  int32_t enabled;        /* 0: scale is fixed at 1 and never updated */
  int32_t found_inf;      /* result of the last finished reduce (all ranks agree) */
  float grad_norm;        /* total gradient norm of the last finished reduce (before clipping) */
  int64_t opt_steps;      /* optimizer steps actually applied (not skipped) */
  int64_t skipped_steps;
} stk_scaler_state_t;

typedef struct {
  int kind;               /* stk_optim_kind */
  double lr, beta1, beta2, eps, weight_decay;   /* Adam / AdamW */
  double momentum, dampening;                   /* SGD */
  int nesterov;
  int maximize;
  int clip_kind;          /* stk_clip_kind */
  double clip_max_norm;   /* STK_CLIP_NORM: max_norm (norm kind / p were given to stk_grad_reduce) */
  double clip_value;      /* STK_CLIP_VALUE */
} stk_optim_hyper_t;

/* ---- library / context -------------------------------------------------------------------------------------------- */
int stk_version(void);
const char* stk_last_error(stk_ctx* ctx); /* ctx may be NULL: last error of the calling thread */

int stk_ctx_create(int rank, int world, int device, unsigned flags, stk_ctx** out);
int stk_ctx_destroy(stk_ctx* ctx);
int stk_caps(stk_ctx* ctx, stk_caps_t* out);

/* ---- peer-visible device memory; the 64-byte handles are exchanged by the caller ------------------------------------
 * Two back ends behind the same calls (STK_OPT_MEM_MODE / env STK_MEM=ipc|vmm, default vmm when world > 1 and the driver
 * supports it): "vmm" = cuMemCreate + POSIX file-descriptor export (the descriptor travels over a unix socket served by the
 * owning context) -- required for NVLS multicast; "ipc" = cudaMalloc + cudaIpc*.  All ranks must use the same mode. */
int stk_mem_alloc_shared(stk_ctx* ctx, size_t bytes, void** local_ptr, unsigned char handle_out[STK_IPC_HANDLE_BYTES]);
/* handles: world * 64 bytes in rank order; peer_ptrs_out[rank] == local_ptr.  In vmm mode this also imports the multicast
 * object rank 0 created for the buffer (if any) and adds this rank's device to it. */
int stk_mem_open_peers(stk_ctx* ctx, void* local_ptr, const unsigned char* handles, void** peer_ptrs_out);
int stk_mem_free_shared(stk_ctx* ctx, void* local_ptr);
/* Binds the buffer's memory to its multicast object and maps it: *mc_ptr_out is an address whose loads/stores address the
 * same offset of EVERY rank's buffer (multimem.* instructions).  Collective: call on every rank after every rank has returned
 * from stk_mem_open_peers (caller barrier), and barrier again before the first use.  Returns STK_ERR_UNSUPPORTED (and leaves
 * the buffer fully usable through its peer pointers) when the device, driver or buffer has no multicast support.
 * stk_multicast_release undoes a bind (used when some other rank failed to bind). */
int stk_multicast_try_bind(stk_ctx* ctx, void* local_ptr, void** mc_ptr_out);
int stk_multicast_release(stk_ctx* ctx, void* local_ptr);

/* signal pads (flags + scalar slots) used by every cross-rank kernel: two-phase like the buffers above */
int stk_comm_local(stk_ctx* ctx, unsigned char handle_out[STK_IPC_HANDLE_BYTES]);
int stk_comm_connect(stk_ctx* ctx, const unsigned char* handles);
/* copies the device error word to the host (synchronises `stream`); returns STK_ERR_PEER if a spin bound was hit */
int stk_comm_check(stk_ctx* ctx, void* stream);
/* same verdict without synchronising: reads the error word's mirror in mapped host memory (a kernel that gave up on a peer
 * writes it).  Every cross-rank entry point calls this first, so after a peer failure the next call returns STK_ERR_PEER. */
int stk_comm_poll(stk_ctx* ctx);

/* tuning knobs.  STK_OPT_K1_ALGO: how the cross-rank K1 brings the peers' 16-bit gradients into the SM -- 0 = 16-byte
 * register loads, 1 = bulk-async copies (TMA engine) staged through shared memory (default; +10..20 % bus bandwidth).  Same
 * results either way; fp32 gradients and launches with a local accumulator always take flavour 0.
 * Also settable at context creation through the environment variable STK_K1_ALGO=ldg|bulk. */
#define STK_OPT_K1_ALGO 1
/* 2 = multimem (NVLS): multimem.ld_reduce of the owned shard + multimem.st of the result; taken when the gradient and
 *     output buffers are multicast-bound and there is no local accumulator, otherwise the call falls back to 1 / 0.
 *     16-bit sums are rounded to the input type by the switch (fp32 accumulation inside it) -- NCCL's NVLS numerics.
 * STK_OPT_MEM_MODE: 0 = ipc, 1 = vmm (see stk_mem_alloc_shared).  STK_OPT_K1_MAX_BLOCKS: grid bound of the cross-rank
 * K1 (0, the default: one block per SM).  STK_OPT_NVLS_MAX_BLOCKS: grid bound of the multimem flavour alone (0, the
 * default: 8 blocks below 128 MiB of input, 16 above).  The two grid bounds exist for bandwidth studies.
 * Cross-rank kernels always use cooperative launches: their blocks spin on the peers' blocks and must be co-resident. */
#define STK_OPT_MEM_MODE 2
#define STK_OPT_K1_MAX_BLOCKS 3
#define STK_OPT_NVLS_MAX_BLOCKS 5
int stk_option_set(stk_ctx* ctx, int key, int value);
int stk_option_get(stk_ctx* ctx, int key, int* value);

/* launch timing for bench.py's roofline: when enabled, K1 (kind 0), K2 (kind 1) and the accumulate kernel (kind 2) are
 * bracketed by CUDA events on the launch stream; stk_profile_read synchronises those events, returns the summed
 * duration and the launch count since the last read, and clears the list. */
int stk_profile_enable(stk_ctx* ctx, int on);
int stk_profile_read(stk_ctx* ctx, int kind, double* ms_total, int* launches);
/* K1 only: time between its start and end barriers (the NVLink data phase) taken with the device timer by block 0 --
 * excludes the wait for the slowest rank to arrive, which host-side events include; ms_zero_tail (may be NULL) receives
 * the time block 0 then spent zeroing its part of the local bucket (HBM work).  Synchronises `stream`. */
int stk_profile_read_k1_device(stk_ctx* ctx, double* ms_total, int* launches, double* ms_zero_tail, void* stream);
/* the same for the sharded optimizer step (cross-rank K2): time between its start and end barriers = local update + the
 * parameter all-gather, without the wait for the slowest rank to arrive.  Synchronises `stream`. */
int stk_profile_read_k2_device(stk_ctx* ctx, double* ms_total, int* launches, void* stream);

/* ---- scaler / step state ------------------------------------------------------------------------------------------- */
/* One device-resident state (loss scaler, found_inf, grad_norm, step counters, per-step norm accumulators) per optimizer.
 * State 0 exists from stk_ctx_create.  stk_state_select makes `id` the state that stk_scaler_*, stk_grad_reduce,
 * stk_grad_norm, stk_grad_scale, stk_optim_step* and stk_step_epilogue read and write until the next select. */
int stk_state_create(stk_ctx* ctx, int* id_out);
int stk_state_select(stk_ctx* ctx, int id);
int stk_state_destroy(stk_ctx* ctx, int id);
int stk_scaler_set(stk_ctx* ctx, const stk_scaler_state_t* st, void* stream);
int stk_scaler_get(stk_ctx* ctx, stk_scaler_state_t* st, void* stream); /* synchronises `stream` */
void* stk_scaler_scale_ptr(stk_ctx* ctx); /* device float*: the live loss scale (for scaler.scale(loss)) */

/* ---- K1: gradient path --------------------------------------------------------------------------------------------- */
/* acc[i] (+)= float(grad[i]); optionally zero grad.  Local, HBM-bound.  first != 0 overwrites acc. */
int stk_grad_accumulate(stk_ctx* ctx, void* grad, int grad_dtype, float* acc, size_t n, int first, int zero_grad,
                        void* stream);

/* main[i] = (sum_r (grad_r[i] [+ acc_r[i]])) * mul * (1/scale)   for i in the shard this rank owns (all i if world==1),
 * written to every rank (STK_REDUCE_ALL) or kept locally (STK_REDUCE_SCATTER); accumulates the norm partial and the
 * inf/nan flag; with STK_RF_FINAL finishes them across ranks into the scaler state.
 *   grad_ptrs / acc_ptrs / out_ptrs: `world` device pointers in rank order (peer mappings); acc_ptrs may be NULL.
 *   n: elements in the bucket (multiple of 8);  mul: e.g. 1/world;  norm_kind / norm_p: which norm to accumulate. */
int stk_grad_reduce(stk_ctx* ctx, int mode, void* const* grad_ptrs, int grad_dtype, float* const* acc_ptrs,
                    void* const* out_ptrs, int out_dtype, size_t n, double mul, int norm_kind, double norm_p,
                    unsigned flags, void* stream);

/* Norm / inf pass without a reduce (world == 1, or gradients that were reduced elsewhere): accumulates the norm partial and
 * the inf/nan flag of x[i] = (float(grad[i]) [+ acc[i]]) * mul * (1/scale) over [0, n) into the selected state and, with
 * STK_RF_FINAL, finishes them (grad_norm, found_inf).  Reads grad once, writes nothing: stk_optim_step_ex then consumes the
 * raw bucket directly (no fp32 main-grad round trip through HBM).  Loads keep the bucket L2-resident for that second read. */
int stk_grad_norm(stk_ctx* ctx, const void* grad, int grad_dtype, const float* acc, size_t n, double mul, int norm_kind,
                  double norm_p, unsigned flags, void* stream);

/* In-place clip of already reduced fp32 gradients for the stock-optimizer route: grad[i] *= min(max_norm/(norm+1e-6), 1)
 * (STK_CLIP_NORM, norm from the selected state) or clamp (STK_CLIP_VALUE). */
int stk_grad_scale(stk_ctx* ctx, float* grad, size_t n, int clip_kind, double clip_max_norm, double clip_value, void* stream);

/* element range [begin, end) of the shard `rank` owns in a bucket of n elements (same partition the kernels use) */
int stk_shard_range(size_t n, int world, int rank, size_t* begin, size_t* end);

/* ---- K2: fused optimizer step (+ K3 parameter all-gather when sharded) ---------------------------------------------- */
/* Updates master/exp_avg/exp_avg_sq over [0, n_local) from grad (fp32, already reduced & unscaled); applies the clip
 * coefficient from the scaler state; skips everything if found_inf.  If lp_ptrs != NULL the updated parameters are also
 * written as lp_dtype to lp_ptrs[r] + lp_offset for r in [0, lp_world) (lp_world == 1: local low-precision copy;
 * lp_world == world: sharded step pushing its shard to every rank = parameter all-gather). */
int stk_optim_step(stk_ctx* ctx, const stk_optim_hyper_t* hyper, float* master, float* exp_avg, float* exp_avg_sq,
                   const float* grad, size_t n_local, void* const* lp_ptrs, int lp_world, int lp_dtype, size_t lp_offset,
                   void* stream);

/* Extended form.  Everything stk_optim_step does, plus:
 *  - raw gradient source (grad_raw = 1): `grad` is the local model-dtype bucket (+ optional fp32 accumulator), scaled by
 *    grad_mul and 1/loss_scale inside the kernel and ZEROED after it has been read (also on a skipped step); pairs with
 *    stk_grad_norm -- the world == 1 route: 2 + 30 B/element instead of 8 + 30.
 *  - segments: the local state [0, n_local) is the concatenation of n_seg pieces; piece k covers local elements
 *    [seg_local[k], seg_local[k+1]) and global (flat-buffer) elements starting at seg_global[k].  lp_ptrs / raw grads /
 *    the range table are indexed globally.  n_seg = 0: one piece, global offset lp_offset (the plain call).
 *  - parameter groups and unused parameters: n_ranges > 0 gives a table over the GLOBAL flat index space; range j ends at
 *    element range_end[j] (ascending, device memory, multiples of 8) and uses hyper[range_group[j] & 0x7f]; bit 7 set = skip
 *    the range this step (parameter received no gradient: torch skips it, torch/optim/optimizer.py).  n_ranges = 0: hyper[0]
 *    everywhere.  With 32-byte peer stores (bf16 parameters, segments on 16-element boundaries) a thread handles two adjacent
 *    vectors and looks the range up once: ranges must then end on 16-element boundaries. */
#define STK_MAX_GROUPS 8
#define STK_MAX_SEGMENTS 64
typedef struct {
  const stk_optim_hyper_t* hyper;   /* n_groups entries (clip fields taken from hyper[0]) */
  int n_groups;
  float* master; float* exp_avg; float* exp_avg_sq;
  const void* grad; int grad_dtype;  /* STK_F32 reduced main grads (local indexing) | raw bucket (global indexing) */
  int grad_raw;
  const float* acc;                  /* raw route only: fp32 accumulator added to grad (global indexing), may be NULL */
  double grad_mul;                   /* raw route only */
  size_t n_local;
  void* const* lp_ptrs; int lp_world; int lp_dtype; size_t lp_offset;
  int n_seg; const size_t* seg_local; const size_t* seg_global;   /* host arrays: n_seg + 1 and n_seg entries */
  int n_ranges; const uint32_t* range_end_vec; const uint8_t* range_group;  /* DEVICE arrays; ends in units of 8 elements */
  size_t grid_n;   /* cross-rank (lp_world > 1) launches: the LARGEST n_local over the ranks, identical on every rank, so that
                      every rank launches the same grid (the block barriers pair block b with block b); 0: n_local */
  const float* range_bc;  /* DEVICE, 4 floats per range {step_size, bias_correction2_sqrt, first_step, 0} written by
                             stk_optim_range_prologue: per-PARAMETER step counts (torch keeps `step` per parameter, so a
                             parameter that skipped some steps has its own bias corrections); NULL: the optimizer-wide
                             counter of the selected state is used for every range */
} stk_optim_args_t;
int stk_optim_step_ex(stk_ctx* ctx, const stk_optim_args_t* args, void* stream);
/* Per-range step bookkeeping for stk_optim_step_ex (call it right before, same stream): for every range j computes the
 * bias corrections of step range_steps[j] + 1 with its group's hyper-parameters into range_bc[4j..4j+3] and, unless the range
 * is skipped this step (bit 7 of range_group[j]) or the selected state says found_inf, increments range_steps[j].
 * All three arrays live in device memory. */
int stk_optim_range_prologue(stk_ctx* ctx, const stk_optim_hyper_t* hyper, int n_groups, int n_ranges,
                             const uint8_t* range_group, int32_t* range_steps, float* range_bc, void* stream);

/* scaler.update(), opt_steps/skipped_steps bookkeeping, reset of the per-step accumulators */
int stk_step_epilogue(stk_ctx* ctx, void* stream);

/* ---- small collectives on the signal pads -------------------------------------------------------------------------- */
/* mean over ranks of *loss_dev (float32/bf16/f16 scalar) -> *out_host (pinned, mapped) ; synchronises `stream` */
int stk_loss_sync(stk_ctx* ctx, const void* loss_dev, int dtype, double* out_host, void* stream);
/* The same mean without the host synchronisation: _begin launches the kernel, which writes the mean to a slot of a pinned
 * ring and returns a ticket; _wait blocks until that launch has finished (no-op if it already has) and returns the value.
 * At most STK_LOSS_RING tickets may be outstanding (older slots are overwritten). */
#define STK_LOSS_RING 256
int stk_loss_sync_begin(stk_ctx* ctx, const void* loss_dev, int dtype, int64_t* ticket_out, void* stream);
int stk_loss_sync_wait(stk_ctx* ctx, int64_t ticket, double* out_host);
int stk_barrier(stk_ctx* ctx, void* stream);
/* every rank copies bytes from ptrs[root] to ptrs[rank] (peer pull) with start/end barriers */
int stk_bcast(stk_ctx* ctx, void* const* ptrs, size_t bytes, int root, void* stream);

/* ---- sampler (stoke/data.py) ---------------------------------------------------------------------------------------- */
/* torch.randperm(n, generator=g) for each n in lens[0..k) drawn from ONE mt19937 seeded with `seed` (host, bit-exact
 * with torch's CPU generator); out receives the k permutations back to back as int32. */
int stk_randperm(uint64_t seed, const int64_t* lens, int k, int32_t* out_host);

typedef struct {
  int64_t n, buckets, batch_size, world, rank;
  int32_t drop_last, allow_bucket_overlap, shuffle;
  /* derived (filled by stk_sampler_plan) */
  int64_t slice_size, per_bucket, slices_per_bucket, rounded_per_bucket, rounded_per_replica;
  int64_t bucket_base, bucket_rem;   /* np.array_split: first bucket_rem buckets have bucket_base + 1 elements */
  int64_t n_bucket_batches, n_overlap_batches, n_batches;
  int32_t needs_padding;
} stk_sampler_plan_t;

/* Fills the derived fields; returns STK_ERR_INVALID with the reference's message for its three ValueError guards. */
int stk_sampler_plan(stk_sampler_plan_t* plan);
/* Positions (into the permuted bucket) of the padded last slice for a bucket of length `bucket_len`:
 * out[j], j in [0, slice_size), is the position that lands at offset j of the last slice (stoke/data.py:450-498). */
int stk_sampler_last_slice(const stk_sampler_plan_t* plan, int64_t bucket_len, int32_t* out_host);

/* stable argsort of u32 keys on the device (LSD radix, 8-bit digits): idx_out[i] = index of the i-th smallest key.
 * tmp must hold stk_argsort_tmp_bytes(n) bytes. */
size_t stk_argsort_tmp_bytes(size_t n);
int stk_argsort_u32(stk_ctx* ctx, const uint32_t* keys, size_t n, int64_t* idx_out, void* tmp, void* stream);

/* out[j] for j in [0, rounded_per_replica): this replica's epoch indices.
 *   sorted_idx: int64[n] (device); bucket_perm: int32[n] per-bucket permutations back to back (NULL if !shuffle);
 *   batch_perm: int32[n_batches] (NULL if !shuffle); last_slice: int32[2][slice_size] tables for bucket lengths
 *   bucket_base + 1 and bucket_base (NULL if !needs_padding). */
int stk_sampler_indices(stk_ctx* ctx, const stk_sampler_plan_t* plan, const int64_t* sorted_idx,
                        const int32_t* bucket_perm, const int32_t* batch_perm, const int32_t* last_slice,
                        int64_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STOKE_B200_H */

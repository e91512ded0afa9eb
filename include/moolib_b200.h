/*
 * moolib_b200.h -- the thin C-ABI between the C++/pybind11 host layer (moolib_b200/csrc/host, which mirrors
 * moolib's Python API) and the hand-written sm_100a kernels (the .cu files under moolib_b200/csrc -> libmoolib_b200.so).
 *
 * Nothing here exists in the reference: the reference has no device code at all (SURVEY.md correction 3).  Each
 * entry point names the reference code whose arithmetic/byte movement it replaces ("replaces: file:line", paths
 * relative to the reference tree).  INTEGRATION.md shows the call a reference maintainer would add at each site.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / pybind types.
 *   - every function returns 0 on success or a negative MB_E* code; mb_last_error() returns a thread-local message.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Nothing synchronises the stream
 *     unless stated; nothing allocates on the hot path (contexts own their scratch).
 *   - pointers are device pointers on the current device unless stated; "host-mapped" means pinned host memory
 *     that the device can address (cudaHostAlloc / cudaHostRegister'd shm slab).
 *   - functions are thread-safe per context; copy functions are stateless.
 */
#ifndef MOOLIB_B200_H_
#define MOOLIB_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MB_VERSION 1

#if defined(__GNUC__)
#define MB_API __attribute__((visibility("default")))
#else
#define MB_API
#endif

/* error codes */
#define MB_OK 0
#define MB_EINVAL (-1)   /* bad argument */
#define MB_ECUDA (-2)    /* CUDA runtime error (see mb_last_error) */
#define MB_ETIMEOUT (-3) /* a peer did not arrive at the allreduce barrier in time */
#define MB_ESTATE (-4)   /* call made in the wrong state (e.g. peer not imported) */
#define MB_ENOMEM (-5)
/* positive status of a gated allreduce round (mb_ar_reduce_gated / mb_ar_result): the summed batch size of all peers
 * is below the requested minimum, nothing was reduced (replaces: src/accumulator.cc:1051 `size < virtualBatchSize`) */
#define MB_AR_SHORT 1

typedef void* mb_stream_t; /* cudaStream_t */

MB_API int mb_version(void);
MB_API const char* mb_last_error(void);
/* number of SMs of `device` (grid sizing is derived from it); negative on error */
MB_API int mb_sm_count(int device);

/* =====================================================================================================
 * HP-B  batch gather / stack / cat  (bit-exact byte movement)
 * ===================================================================================================== */

/* One pitched 2-D byte copy: `rows` rows of `row_bytes` bytes; row r is read at src + r*src_pitch and written
 * at dst + r*dst_pitch.  Everything HP-B does reduces to a table of these:
 *   stack slot k along dim d   : rows = prod(shape[:d]), row_bytes = inner, src_pitch = inner, dst_pitch = size*inner,
 *                                dst += k*inner                      (replaces: src/moolib.cc:676,751 select().copy_)
 *   cat/narrow along dim d     : rows = prod(shape[:d]), row_bytes = n*inner, src_pitch = n_src*inner,
 *                                dst_pitch = n_dst*inner             (replaces: src/moolib.cc:665-668,745-748)
 *   env slab row fill          : rows = 1                            (replaces: src/env.h:248-263 fillBatch memcpy)
 *   torch::stack of N leaves   : N jobs, one per input               (replaces: src/batch_utils.cc:295)
 * src may be device memory or host-mapped memory; dst is device memory (or host-mapped). */
typedef struct mb_copy_job {
  const void* src;
  void* dst;
  uint64_t row_bytes;
  uint64_t rows;
  int64_t src_pitch; /* bytes */
  int64_t dst_pitch; /* bytes */
} mb_copy_job;

/* Max jobs carried inline in the kernel parameters of one launch (<= 64: the classic 4 KiB parameter block; <= 512: the
 * 32 KiB parameter space of CUDA 12.1+); larger tables are split into several launches by mb_copy2d_batch, or uploaded
 * once and read from device memory by mb_copy2d_table. */
#define MB_COPY_MAX_INLINE_JOBS 512

/* Execute `njobs` pitched copies in as few launches as possible (one per 512 jobs).  `jobs` is a HOST array, read
 * before the call returns.  Overlapping src/dst between jobs is undefined.  Returns the number of kernel launches
 * (>= 0) or a negative error. */
MB_API int mb_copy2d_batch(const mb_copy_job* jobs, int njobs, mb_stream_t stream);

/* Where the sources of a table live.  DEVICE / HOST_MAPPED is the caller's promise for EVERY job of the call (the host
 * layer knows: tensor.is_cuda() vs a pinned slab) and saves one driver query per bulk job; UNKNOWN asks the driver. */
#define MB_SRC_UNKNOWN 0
#define MB_SRC_DEVICE 1
#define MB_SRC_HOST_MAPPED 2 /* PCIe-bound: the launch is limited to a few dozen CTAs so the SMs stay free */
MB_API int mb_copy2d_batch_ex(const mb_copy_job* jobs, int njobs, int src_kind, mb_stream_t stream);

/* Tables of ANY length in ONE launch: the normalised table is written into pinned staging owned by the context,
 * uploaded with one async copy and read by the kernels from device memory (tables of <= MB_COPY_MAX_INLINE_JOBS jobs
 * still travel in the kernel parameters, no upload).  This is what lets a whole unroll -- T time steps x leaves x
 * learner batches, ~1200 pitched copies -- be gathered straight into its final layout by one kernel instead of T stack
 * launches followed by a re-tiling pass.  max_jobs bounds one launch; longer tables are split.
 * (replaces: src/moolib.cc:813-845 stack x T followed by :767-811 cat, i.e. two passes over every observation byte) */
typedef struct mb_copy_ctx mb_copy_ctx;
MB_API int mb_copy_ctx_create(int device, uint32_t max_jobs, mb_copy_ctx** out);
MB_API int mb_copy_ctx_destroy(mb_copy_ctx* ctx);
MB_API int mb_copy2d_table(mb_copy_ctx* ctx, const mb_copy_job* jobs, int njobs, int src_kind, mb_stream_t stream);

/* K-B1/K-B4: gather `nrows` rows of `row_bytes` from the pointers in the DEVICE array `src_rows_dev` into
 * dst + i*dst_pitch.  (replaces: src/env.h:258 per-env memcpy + experiment.py:492 H2D; src/batch_utils.cc:295) */
MB_API int mb_gather_rows(void* dst, uint64_t dst_pitch, const void* const* src_rows_dev, uint64_t row_bytes,
                   uint64_t nrows, mb_stream_t stream);

/* K-B2: write one item into slot `slot` of a [outer, size, inner_bytes] batch.
 * (replaces: src/moolib.cc:676 and :751  tensor.select(dim, k).copy_(src)) */
MB_API int mb_stack_slot(void* dst_base, uint64_t outer, uint64_t size, uint64_t slot, uint64_t inner_bytes,
                  const void* src, mb_stream_t stream);

/* K-B3: dst[:, dst_off:dst_off+n, :] = src[:, src_off:src_off+n, :] for dst [outer, dst_dim, inner_bytes] and
 * src [outer, src_dim, inner_bytes].  (replaces: src/moolib.cc:665-668, 745-748  narrow().copy_(narrow())) */
MB_API int mb_cat_narrow(void* dst, const void* src, uint64_t outer, uint64_t dst_dim, uint64_t dst_off, uint64_t src_dim,
                  uint64_t src_off, uint64_t n, uint64_t inner_bytes, mb_stream_t stream);

/* B3 (action scatter): for i < n: counters[i*counter_stride_u32] += 1 + (uint32_t)actions[i]; counters is a
 * host-mapped array of 32-bit words (the EnvPool's per-env action mailboxes), actions a device int64 array.
 * Stores are made visible at system scope before the kernel ends.
 * (replaces: src/env.cc:310-319 pinned copy + stream sync and :340-345 the `prev + 1 + a` store loop) */
MB_API int mb_scatter_actions(uint32_t* counters_hostmapped, uint64_t counter_stride_u32, const int64_t* actions,
                       uint64_t n, mb_stream_t stream);

/* =====================================================================================================
 * HP-A  gradient allreduce over NVLink peer memory (fp32 sums of fp32 / bf16 / fp16 gradients, fixed rank order,
 *       fused 1/numGradients scale)
 * ===================================================================================================== */

typedef struct mb_ar_ctx mb_ar_ctx;

/* The three counters moolib reduces next to the gradients, plus whether this peer contributes gradients at all
 * (a peer that only called skip_gradients() contributes an EMPTY list).
 * (replaces: src/group.h:195-212 AccumulatorReductionType {numGradients,numSkipped,batchSize} and add()) */
typedef struct mb_ar_hdr {
  uint64_t num_gradients;
  uint64_t num_skipped;
  uint64_t batch_size;
  uint64_t has_grads; /* 0/1 on input; on output = number of peers that had gradients */
} mb_ar_hdr;

/* Opaque, fixed-size, memcpy-able description of one rank's symmetric buffers, to be carried to the other ranks
 * by whatever control plane the host has (Group/Rpc, torch.distributed, a pipe).  Holds two cudaIpcMemHandle_t
 * plus pid/device/pointers so that peers living in the SAME process map the memory with cudaDeviceEnablePeerAccess
 * instead of CUDA IPC. */
#define MB_AR_HANDLE_BYTES 192
typedef struct mb_ar_handle {
  unsigned char bytes[MB_AR_HANDLE_BYTES];
} mb_ar_handle;

#define MB_AR_MAX_WORLD 8
#define MB_AR_MAX_SLOTS 4 /* staging slots = moolib's set_parallel_gradients ring (src/accumulator.cc:889-903) */
/* Every slot owns a ring of 3 staging buffers.  Round k of a slot is reduced out of ring position k mod 3; a rank may
 * write position (k+1) mod 3 while slow peers are still reading position k, and position (k+2) mod 3 = (k-1) mod 3 is
 * free because every peer has finished round k-1 before it can take part in round k.  The third buffer is what lets
 * gradients be PRODUCED in the staging memory (no stage kernel): see mb_ar_buffer. */
#define MB_AR_BUFS_PER_SLOT 3

/* algorithm selector for mb_ar_allreduce */
#define MB_AR_ALGO_AUTO 0
#define MB_AR_ALGO_ONESHOT 1 /* every rank pulls all peers' buffers (P2P loads), lowest latency */
#define MB_AR_ALGO_TWOSHOT 2 /* reduce-scatter by P2P loads + all-gather by P2P stores, 2(N-1)/N traffic */

/* Allocate rank `rank`'s symmetric staging (nslots x 3 x max_bytes + one publish region, cudaMalloc so it is IPC-exportable), barrier
 * flags and the pinned result block on `device`.  world <= MB_AR_MAX_WORLD, 1 <= nslots <= MB_AR_MAX_SLOTS.
 * (replaces: src/accumulator.cc:847-874 allocateGradients -- pinned CPU staging) */
MB_API int mb_ar_ctx_create(int rank, int world, int device, uint64_t max_bytes, int nslots, mb_ar_ctx** out);
MB_API int mb_ar_ctx_destroy(mb_ar_ctx* ctx);
MB_API int mb_ar_ctx_export(mb_ar_ctx* ctx, mb_ar_handle* out);
/* Map peer `peer_rank`'s buffers.  Must be called for every peer != rank before the first collective, and again
 * for all peers after mb_ar_ctx_reset (membership / sync_id change). */
MB_API int mb_ar_ctx_import(mb_ar_ctx* ctx, int peer_rank, const mb_ar_handle* handle);
/* Drop all peer mappings and restart the barrier epoch (group resync: src/group.h:453-461, accumulator.cc:555-575).
 * All ranks must reset together; synchronises the device. */
MB_API int mb_ar_ctx_reset(mb_ar_ctx* ctx, int new_rank, int new_world);
/* Device pointer of the CURRENT staging buffer of `slot` (flat fp32, max_bytes): what the next allreduce on the slot
 * reduces.  == mb_ar_buffer(ctx, slot, 0). */
MB_API void* mb_ar_staging(mb_ar_ctx* ctx, int slot);
/* Ring buffer `ahead` positions after the slot's current staging buffer (0 <= ahead < MB_AR_BUFS_PER_SLOT).
 * ahead = 1 is the buffer that becomes current after the next successful round: a host that points its gradient
 * tensors at it (flat layout of mb_ar_stage, zero-filled) has its next contribution staged by construction -- backward()
 * writes where the peers will read, K-A1 never runs.
 * (replaces: src/accumulator.cc:847-874 allocateGradients + :941-980 the D2H staging copies) */
MB_API void* mb_ar_buffer(mb_ar_ctx* ctx, int slot, int ahead);
/* Move the slot's ring to the next buffer.  mb_ar_allreduce does this itself after every launch; after
 * mb_ar_reduce_gated the HOST calls it once it has seen the round end with status MB_OK (a round that ended MB_AR_SHORT
 * reduced nothing and keeps accumulating into the same staging buffer).  All ranks advance together. */
MB_API int mb_ar_slot_advance(mb_ar_ctx* ctx, int slot);
/* What MB_AR_ALGO_AUTO resolves to for a message of `bytes` at this context's world size.  A host that wants the
 * result IN PLACE -- flat_dst == mb_ar_buffer(ctx, slot, 0), possible with the two-shot algorithm only, whose all-gather
 * leaves the reduced values in every rank's staging buffer: the kernel then skips its final local copy -- asks first. */
MB_API int mb_ar_algo_for(mb_ar_ctx* ctx, uint64_t bytes);
MB_API int mb_ar_world(mb_ar_ctx* ctx);
MB_API int mb_ar_rank(mb_ar_ctx* ctx);

/* K-A1  stage: staging[slot] (=|+=) concat(grads[i]) and optionally zero grads[i], one launch for all tensors.
 * Tensor i occupies floats [offset_i, offset_i+numel_i) of the flat staging, offset_i = sum of numel_j (j<i), each
 * rounded up to 4 floats (16 B) so every tensor starts vector-aligned.  `grads`/`numel` are HOST arrays.
 * (replaces: src/accumulator.cc:941-980 -- 36x copy_ / to(cpu)+add_ -- and :410-418 detach_/zero_) */
MB_API int mb_ar_stage(mb_ar_ctx* ctx, int slot, const float* const* grads, const uint64_t* numel, int ntensors,
                int accumulate, int zero_src, mb_stream_t stream);

/* K-A2  allreduce: barrier with all peers, then for every element
 *          sum = (((g_r0 + g_r1) + g_r2) + ...)        over the ranks with has_grads, in ascending rank order
 *          out = sum * (1.0f / (float)sum(num_gradients))   (fp32 multiply by reciprocal, as the reference)
 *        written to dst[i] (the .grad tensors, same flat layout as mb_ar_stage) -- or, if dst == NULL, to the flat
 *        buffer `flat_dst`.  If scale_by_num_gradients == 0 the plain sum is written (group.all_reduce).  The
 *        summed header is written to the context's pinned result block (mb_ar_result).
 *        If no rank has gradients the destinations are zeroed (src/accumulator.cc:426-428).
 * All ranks must call with the same slot, layout, algo and epoch order.  total_numel = padded flat length.
 * (replaces: src/group.h:570-654,687-787 tree reduce + share over RPC; src/accumulator.cc:433-452 copy_ + mul_) */
MB_API int mb_ar_allreduce(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, float* const* dst, const uint64_t* numel,
                    int ntensors, float* flat_dst, uint64_t flat_numel, int scale_by_num_gradients, int algo,
                    uint32_t timeout_ms, mb_stream_t stream);

/* K-A0 + K-A2  gated allreduce: the virtual-batch gate of moolib's Accumulator evaluated ON THE DEVICE.
 *   launch 1 (K-A0, one warp): push my_hdr into every peer's sync block, wait for theirs (bounded by timeout_ms / mb_ar_abort),
 *            sum them; gate open  <=>  sum(batch_size) >= min_batch_size.
 *   launch 2 (K-A2): gate open -> reduce exactly as mb_ar_allreduce but without its start barrier (a peer's header only
 *            arrives after its staging is complete); gate closed -> returns immediately.
 * Result (mb_ar_result, once the stream has passed both launches): status MB_OK + summed header when reduced,
 * MB_AR_SHORT + summed header when the gate was closed, MB_ETIMEOUT when a peer did not show up.  Every rank reaches the
 * same verdict (same headers, same min_batch_size).  The slot's ring does NOT advance: call mb_ar_slot_advance after MB_OK.
 * With world == 1 the gate is evaluated on the host and only K-A2 is launched (or nothing, when short).
 * The context brackets the two launches with its own CUDA events: see mb_ar_round_times.
 * Returns the number of kernel launches.
 * (replaces: src/accumulator.cc:1035-1078 startCount -- an 8-byte allreduce over the RPC tree and one extra update() tick
 *  per step -- and :1005-1033 startReduce) */
MB_API int mb_ar_reduce_gated(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, uint64_t min_batch_size,
                       float* const* dst, const uint64_t* numel, int ntensors, float* flat_dst, uint64_t flat_numel,
                       int scale_by_num_gradients, int algo, uint32_t timeout_ms, mb_stream_t stream);

/* Device times of the most recent gated round on `slot`, once the stream has passed it: gate_us = K-A0 (includes the
 * wait for the slowest peer), reduce_us = K-A2 (the data movement).  MB_ESTATE if the round launched no kernel. */
MB_API int mb_ar_round_times(mb_ar_ctx* ctx, int slot, float* gate_us, float* reduce_us);

/* One-way bulk transfer of a tensor list between two members over NVLink (late-joiner model / buffer sync): the sender
 * packs its tensors (flat layout of mb_ar_stage) into its PUBLISH region -- part of the symmetric block every peer has
 * mapped --, tells the receiver over the host's control plane once its stream has passed the pack, and the receiver
 * pulls the region into its own tensors with P2P loads.  No serialisation, no host staging, no socket payload.
 * The host keeps the publisher from overwriting the region while a fetch is outstanding.
 * (replaces: src/accumulator.cc:719-759, 810-836 -- parameters and buffers copied to the CPU, serialised and sent over the
 *  RPC transport to every requesting peer) */
MB_API int mb_ar_xfer_pack(mb_ar_ctx* ctx, const float* const* tensors, const uint64_t* numel, int ntensors,
                           mb_stream_t stream);
MB_API int mb_ar_xfer_unpack(mb_ar_ctx* ctx, int src_rank, float* const* tensors, const uint64_t* numel, int ntensors,
                             mb_stream_t stream);

/* Result of the most recent allreduce on `slot`: summed header and status (0 ok, MB_ETIMEOUT ...).  Reads pinned
 * host memory written by the kernel; only meaningful once the stream has reached the end of that allreduce
 * (query an event / synchronise first).  `status_out` may be NULL. */
MB_API int mb_ar_result(mb_ar_ctx* ctx, int slot, mb_ar_hdr* sum_out, int* status_out);

/* Padded flat length (in floats) of a tensor list under the layout rule above. */
MB_API uint64_t mb_ar_flat_numel(const uint64_t* numel, int ntensors);

/* ---- low-precision gradients (bf16 / fp16), alone or mixed with fp32 in one list ----------------------------------
 * Element dtypes of the _ex entry points.  For bf16 and fp16 every element is reduced as
 *     widen each rank's value to fp32;  sum in fp32 in ascending rank order over the ranks with has_grads;
 *     multiply by the fp32 reciprocal 1.0f/sum(num_gradients) (when scaling);  round ONCE (nearest-even) to the dtype.
 * All ranks hold identical bits, one-shot and two-shot give identical bits, and a single contributor's result equals
 * the reference's copy_ + mul_ in the dtype.  The reference instead rounds to the dtype after every tree add
 * (src/group.h:597-603) and again in mul_ (src/accumulator.cc:442), so it differs in the last bits (DESIGN.md §2). */
#define MB_DT_F32 0
#define MB_DT_BF16 1
#define MB_DT_F16 2

/* One dtype run of the flat layout: bytes [begin, end) hold only tensors of `dtype`. */
typedef struct mb_ar_segment {
  uint64_t begin;
  uint64_t end;
  int32_t dtype;
  int32_t reserved;
} mb_ar_segment;

/* The flat layout of a mixed tensor list, the one rule every _ex call, K-A1 and K-A2 use.  Tensors are grouped by dtype
 * (fp32, then bf16, then fp16; list order within a group), so each dtype is one contiguous run of 16 B vectors, and every
 * tensor starts 16 B aligned (padded to 4 fp32 or 8 half-width elements; padding is zero).  For an all-fp32 list the
 * offsets are exactly those of mb_ar_stage (offset_bytes[i] = 4 * float offset).  Writes offset_bytes[ntensors] (may be
 * NULL), *total_bytes (may be NULL) and up to 3 non-empty segments (may be NULL).  Returns the number of segments. */
MB_API int mb_ar_layout(const uint64_t* numel, const int32_t* dtype, int ntensors, uint64_t* offset_bytes,
                        uint64_t* total_bytes, mb_ar_segment* segments);

/* K-A1 for a mixed list: staging (=|+=) the list in the layout of mb_ar_layout, optionally zeroing the sources.
 * `+=` rounds in the tensor's dtype, like the reference's add_.  An all-fp32 list runs mb_ar_stage.
 * (replaces: src/accumulator.cc:941-980 copy_ / add_ for bf16 and fp16 gradients, and :410-418 zero_) */
MB_API int mb_ar_stage_ex(mb_ar_ctx* ctx, int slot, const void* const* grads, const uint64_t* numel,
                          const int32_t* dtype, int ntensors, int accumulate, int zero_src, mb_stream_t stream);

/* K-A2 for a mixed list.  `numel`, `dtype`, `ntensors` describe the layout (mb_ar_layout) and are always required;
 * the result goes to the tensors `dst` (HOST array of device pointers), or, if dst == NULL, to the 16 B-aligned flat
 * buffer `flat_dst` of exactly flat_bytes == total_bytes in the same layout.  fp32 segments are reduced exactly as
 * mb_ar_allreduce, bf16 / fp16 segments as stated above; an all-fp32 list runs mb_ar_allreduce itself.
 * (replaces: src/group.h:570-654,687-787 tree reduce + share of bf16 / fp16 tensors; src/accumulator.cc:433-452) */
MB_API int mb_ar_allreduce_ex(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, void* const* dst,
                              const uint64_t* numel, const int32_t* dtype, int ntensors, void* flat_dst,
                              uint64_t flat_bytes, int scale_by_num_gradients, int algo, uint32_t timeout_ms,
                              mb_stream_t stream);
/* K-A0 + K-A2 for a mixed list: mb_ar_reduce_gated with the arguments of mb_ar_allreduce_ex.
 * (replaces: src/accumulator.cc:1005-1078 startCount + startReduce for bf16 / fp16 models) */
MB_API int mb_ar_reduce_gated_ex(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, uint64_t min_batch_size,
                                 void* const* dst, const uint64_t* numel, const int32_t* dtype, int ntensors,
                                 void* flat_dst, uint64_t flat_bytes, int scale_by_num_gradients, int algo,
                                 uint32_t timeout_ms, mb_stream_t stream);

/* Host-side abort: makes every in-flight and future barrier wait on this context fail with MB_ETIMEOUT promptly
 * (peer death / regroup, SURVEY.md section 5 "Hook for HP-A").  Cleared by mb_ar_ctx_reset. */
MB_API int mb_ar_abort(mb_ar_ctx* ctx);

/* =====================================================================================================
 * Learner-side steps next to the hot paths (launch-bound chains of tiny ops in the reference's example)
 * ===================================================================================================== */

/* K-L1  V-trace from log importance weights, [T, B] fp32 contiguous inputs, bootstrap_value [B]:
 *   rho = exp(log_rho); c = min(rho, 1); delta = min(rho, clip_rho) * (r + d * V_{t+1} - V_t)
 *   acc_t = delta_t + d_t * c_t * acc_{t+1};  vs_t = acc_t + V_t
 *   pg_adv_t = min(rho, clip_pg_rho) * (r_t + d_t * vs_{t+1} - V_t)
 * in the reference's operation order, every fp32 rounding kept.  has_clip_* == 0 disables that clamp (None).
 * (replaces: examples/common/vtrace.py:207-242 from_importance_weights -- ~100 kernel launches for T = 20) */
MB_API int mb_vtrace_f32(const float* log_rhos, const float* discounts, const float* rewards, const float* values,
                         const float* bootstrap_value, int has_clip_rho, float clip_rho, int has_clip_pg_rho,
                         float clip_pg_rho, uint64_t T, uint64_t B, float* vs_out, float* pg_advantages_out,
                         mb_stream_t stream);

/* K-L2  dst[i] = (float)src[i] * scale  (scale = 1.0f/255.0f: the observation normalisation; ATen evaluates
 * `x.float() / 255.0` as a multiplication by the fp32 reciprocal, so the results are bit-identical).
 * (replaces: examples/atari/models.py:94 -- two elementwise passes) */
MB_API int mb_u8_to_f32(const uint8_t* src, float* dst, uint64_t n, float scale, mb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MOOLIB_B200_H_ */

/*
 * mafed_distill.h -- C ABI of the B200-native MAFED feature-distillation hot path.
 *
 * The reference (MalvinaNikandrou/mafed) is pure Python: it has no FFI / operator boundary of its
 * own.  Its plug-in boundary is the Python class registry mafed/methods/__init__.py:6-11
 * (CLMethod["featdistill"] -> FeatureDistillation), mirrored by mafed_b200/methods/.  This header
 * is the boundary UNDERNEATH that mirror: plain pointers and sizes, no torch types, one entry
 * point per stage of the path.  Each function cites the reference code it replaces.
 *
 * Conventions
 *   - every `*_ptrs` argument is a HOST array of n_layers DEVICE pointers, one per selected layer;
 *     hidden states are separately allocated, contiguous [B, T, D] tensors (vl_pythia.py:320-326).
 *   - `attn_mask` is the DEVICE int64 [B, T - n_vis] left-padded text attention mask
 *     (data/vl_pythia_vqa_dataset.py:141-142).  Positions t <  n_vis are visual tokens with
 *     weight 1 (distillation.py:140-144); t >= n_vis are text tokens weighted by
 *     attn_mask[b, t - n_vis] (distillation.py:135-139).
 *   - `stream` is a cudaStream_t passed as void*.
 *   - return value: 0 = ok; < 0 = argument error (MAFED_E_*); > 0 = a cudaError_t.
 *   - no allocation and no host synchronisation inside any call: every call only enqueues kernels
 *     on `stream` and is CUDA-graph capturable.
 *
 * Two ways to run a step (both produce the reference's loss and gradients):
 *   one-pass : mafed_distill_step -- ONE kernel launch: modality masks, gradient scale, loss sums AND gradients from
 *              a single read of student and teacher, losses (3*D*e bytes of HBM traffic per token*layer) -- and, in
 *              the backward of the autograd graph, mafed_distill_bwd(skip_if_equals): a 1-CTA gate that returns at
 *              once when the upstream gradient is the one assumed and otherwise starts the exact backward itself.
 *   two-pass : mafed_distill_fwd_step (forward + losses + scale table, one launch) ... mafed_distill_bwd
 *              (5*D*e bytes per token*layer).
 * Across batch shards (one process per GPU) both forms take a peer-memory communicator (mafed_comm_*) and stay one
 * launch; without one the stages are available separately for an NCCL sequence:
 * mafed_distill_fwd | mafed_distill_fused -> mafed_distill_scalar_stage(REDUCE|COUNTS) -> allreduce(sums) ->
 * mafed_distill_scalar_stage(LOSSES|SCALE).
 * The library has no process-global knobs: the few overrides travel with the call (mafed_shape_t::tuning).  What it
 * remembers between calls is bookkeeping only (per-device attribute caches, the round-robin index of its arrival
 * counters, and which streams a gate was last sent to -- see mafed_distill_bwd).
 */
#ifndef MAFED_DISTILL_H_
#define MAFED_DISTILL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAFED_ABI_VERSION 4
#define MAFED_MAX_LAYERS 64

enum { MAFED_F32 = 0, MAFED_BF16 = 1, MAFED_F16 = 2 };
enum { MAFED_LOSS_MSE = 0, MAFED_LOSS_COSINE = 1 };
/* modality weighting (distillation_loss_weights.py:71-79):
 *   EQUAL: w_text = n_text/(n_text+n_vis) from the mask counts (:148-155);
 *   TABLE: w_text = lang_weight[l], w_vis = 1 - w_text (balanced :165-166 -> 0.5; adaptive :168-174);
 *   CLS  : only row 0 of each sample, mean over B (distillation.py:251-257);
 *   TEXT_ONLY: layer loss = masked text loss alone -- one call of _compute_*_distillation_loss
 *          with an arbitrary [B, T] mask (distillation.py:226-249; use n_vis = 0). */
enum { MAFED_MODW_EQUAL = 0, MAFED_MODW_TABLE = 1, MAFED_MODW_CLS = 2, MAFED_MODW_TEXT_ONLY = 3 };

enum {
  MAFED_E_ARG = -1,      /* null pointer / non-positive size / too many layers */
  MAFED_E_DTYPE = -2,    /* unknown dtype or loss kind */
  MAFED_E_ALIGN = -3,    /* a pointer is not aligned to its element size */
  MAFED_E_NODEVICE = -4  /* no CUDA device */
};

/* flags of mafed_distill_scalar_stage */
enum { MAFED_STAGE_REDUCE = 1, MAFED_STAGE_COUNTS = 2, MAFED_STAGE_LOSSES = 4, MAFED_STAGE_SCALE = 8 };

/* Overrides of ONE call, for tests and benchmarks that compare a default launch with another form of it.  All zero =
 * the library's defaults, which is also what a NULL mafed_shape_t::tuning means.  Three indices of v are read; every
 * other index is ignored (the layout is kept for callers built against earlier versions of this header):
 *   v[MAFED_TUNE_NO_TAIL]     1: the losses come from a separate scalar-stage launch instead of the last CTA
 *   v[MAFED_TUNE_VARIANT_ALL] kernel family of every pass: 1 register-staged (LDG), 2 TMA ring (0: default)
 *   v[MAFED_TUNE_NO_GATE]     1: the backward fix-up is a full grid whose CTAs return at once instead of a gate */
enum { MAFED_TUNE_NO_TAIL = 17, MAFED_TUNE_VARIANT_ALL = 18, MAFED_TUNE_NO_GATE = 19 };
typedef struct mafed_tuning {
  int32_t v[24];
} mafed_tuning_t;

/* Geometry of one step.  rows of a layer: N = B*T (or B in CLS mode). */
typedef struct mafed_shape {
  int32_t n_layers;   /* selected layers in this call, 1..MAFED_MAX_LAYERS */
  int32_t B;          /* samples in this rank's shard */
  int32_t T;          /* n_vis + text positions */
  int32_t n_vis;      /* 256 in the reference (distillation.py:73) */
  int32_t D;          /* hidden size */
  int32_t dtype;      /* MAFED_F32 | MAFED_BF16 | MAFED_F16 (student, teacher and gradient) */
  int32_t loss_kind;  /* MAFED_LOSS_MSE (distillation.py:237-249) | MAFED_LOSS_COSINE (:226-235) */
  int32_t cls;        /* 1: CLS distillation (distillation.py:126-132,251-257) */
  const mafed_tuning_t* tuning;   /* NULL: defaults */
} mafed_shape_t;

/* Host-side weight tables (distillation.py:110-113,163; distillation_loss_weights.py:49-60). */
typedef struct mafed_weights {
  int32_t modality_kind;                   /* MAFED_MODW_* */
  float distill_coeff;                     /* self.distillation_coeff */
  float layer_coeff[MAFED_MAX_LAYERS];     /* get_layer_loss_weight(layer) for each selected layer */
  float lang_weight[MAFED_MAX_LAYERS];     /* TABLE only */
} mafed_weights_t;

int mafed_distill_abi_version(void);
const char* mafed_distill_error_string(int code);

/* Bytes of device workspace mafed_distill_fwd / _fused need (per-CTA partial sums). */
size_t mafed_distill_ws_bytes(int n_layers);
/* Length (in doubles) of the `sums` vector: 2*n_layers partial sums + [n_text, n_vis]. */
int mafed_distill_sums_len(int n_layers);
/* Length (in floats) of the `out` vector: total, n_layers layer losses, 2*n_layers modality losses. */
int mafed_distill_out_len(int n_layers);

/* ---- peer-memory communicator: the batch-sharded step without NCCL on the critical path -----------------
 * One process per GPU of one NVLink/NVSwitch box.  Each rank creates a small mailbox (cudaMalloc + CUDA IPC
 * handle), the handles are exchanged out of band (torch.distributed all_gather in mafed_b200/comm.py) and every
 * rank maps its peers' mailboxes.  Exchanges are one-shot SUM-allreduces of <= 2L+2 doubles performed INSIDE the
 * path's kernels with NVLink peer stores of self-validating words (value halves tagged with the epoch; no fence,
 * no flag); results are bit-identical on all ranks; the epochs live on the device (CUDA-graph replayable); spins
 * are bounded (mafed_comm_set_timeout; a timeout sets the status and yields NaN). */
typedef struct mafed_comm mafed_comm_t;
enum { MAFED_COMM_SUMS = 1, MAFED_COMM_COUNTS = 2 };
int mafed_comm_handle_bytes(void);
int mafed_comm_create(int world, int rank, void* ipc_handle_out, mafed_comm_t** out);
/* all_handles == NULL: diagnostic loop-back (all peers map to the own mailbox; every exchange times out). */
int mafed_comm_connect(mafed_comm_t* comm, const void* all_handles /* world x handle_bytes, rank order */);
/* Spin bound of one in-kernel wait (default 60 s, or MAFED_B200_COMM_TIMEOUT_S at creation).  A wait that runs
 * into it sets the status and yields NaN: the step's loss and gradients come out NaN instead of silently wrong. */
int mafed_comm_set_timeout(mafed_comm_t* comm, double seconds);
/* The status word lives in mapped pinned host memory (the kernels store into it on a timeout): this is a plain
 * host read that never synchronises.  It reflects every exchange of the kernels that have finished. */
int mafed_comm_status(mafed_comm_t* comm, int* status_out /* 0 ok, 1 a peer timed out */);
/* SM-cycle totals since creation (synchronises the device): [0] in-kernel counts exchange as seen by CTA 0,
 * [1] own peer stores of a sums exchange, [2] waiting for the peers' vectors, [3] sums exchanges. */
int mafed_comm_trace(mafed_comm_t* comm, unsigned long long* out4);
/* The same four totals as a stream-ordered snapshot: an asynchronous copy into `out4` (pinned host or device memory)
 * behind the work already queued on `stream`; no synchronisation.  Two snapshots bracket the steps between them. */
int mafed_comm_trace_async(mafed_comm_t* comm, unsigned long long* out4, void* stream);
int mafed_comm_destroy(mafed_comm_t* comm);

/* Token counts ahead of the step.  The counts depend only on the attention mask, which is known when the memory
 * batch is drawn -- before the student forward (distillation.py:85-91).  This 1-CTA launch sums the mask, writes
 * {n_text, n_vis rows} of this rank into every peer's mailbox (fire and forget, no wait) and leaves a ticket
 * (int64[4]: exchange epoch, then this rank's two counts as doubles) in `ticket`.  A later mafed_distill_step given the same ticket reads
 * finished global counts from its own mailbox instead of exchanging them at its start.  Up to 3 prefetched
 * batches may be outstanding.  comm == NULL (single rank): only the local counts are left in the ticket. */
int mafed_distill_prefetch_counts(const mafed_shape_t* shape, const int64_t* attn_mask, mafed_comm_t* comm,
                                  int64_t* ticket, void* stream);

/* ---- the whole step as ONE call (what mafed_b200 uses) ----------------------------------------------------
 * mafed_distill_step = all of FeatureDistillation.distill (distillation.py:105-166) plus the backward of its
 * autograd graph: modality masks, counts -> gradient scale, loss sums + gradients from a single read of student and
 * teacher, losses.  The gradient scale depends only on the token counts and the host weight tables (not on the
 * loss), so it is known before the pass; the upstream gradient is assumed to be `assumed_grad_out` (1/accumulate_
 * grad_batches under Lightning, vqa_cont_learner.py:213-236) and checked later by mafed_distill_bwd(skip_if_equals).
 * For shapes the TMA-ring kernel takes (rows <= 32 KB, 16-byte aligned) and masks of <= 16 Ki entries it is ONE
 * kernel launch: every CTA derives the gradient scale itself, all CTAs together write the two modality masks, and
 * the CTA that finishes LAST reduces the per-CTA partial sums in fixed order (bit-reproducible) and forms the
 * losses.  With a communicator the counts are exchanged inside the kernel behind its first tiles -- or, with a
 * `counts_ticket` from mafed_distill_prefetch_counts, simply read from the own mailbox, where they landed long ago
 * -- and the last CTA exchanges the 2L sums with the peers.  Other shapes run the same step as separate launches.
 * out[1+3L] = {total, layer losses, (text, vision) losses}; bwd_scale[2L] is written for the later gate; sums
 * (optional single-rank, required with comm) receives the global [2L+2] vector; lang_mask / image_mask (both or
 * neither, int64 [B, T]) are optional; a NULL entry in grad_ptrs still contributes to the sums. */
int mafed_distill_step(const mafed_shape_t* shape, const void* const* student_ptrs,
                       const void* const* teacher_ptrs, void* const* grad_ptrs, const int64_t* attn_mask,
                       const mafed_weights_t* weights, float assumed_grad_out, void* ws, float* out,
                       float* bwd_scale, double* sums, int64_t* lang_mask, int64_t* image_mask,
                       mafed_comm_t* comm, const int64_t* counts_ticket, void* stream);
/* The two-pass form's first half: fused forward + REDUCE|COUNTS|LOSSES|SCALE in one launch (sharded: sums and
 * counts exchanged in the tail). */
int mafed_distill_fwd_step(const mafed_shape_t* shape, const void* const* student_ptrs,
                           const void* const* teacher_ptrs, const int64_t* attn_mask,
                           const mafed_weights_t* weights, void* ws, float* out, float* bwd_scale, double* sums,
                           mafed_comm_t* comm, void* stream);

/* Fused backward: grad[l][row] = g * bwd_scale[l][m(row)] * w(row) * d f(h,p)/dh with g = *grad_out *
 * grad_out_scale, zero for padded text rows; one pass, 2 reads + 1 write (replaces autograd's per-layer,
 * per-modality chains of distillation.py:226-249).  `grad_out` is a DEVICE float scalar (NULL = 1.0),
 * `grad_out_scale` a host factor (e.g. world_size to undo DDP's gradient averaging).  A NULL entry in grad_ptrs
 * skips that layer.  If `skip_if_equals` is not NULL (a HOST float) the call is the one-pass step's gate: a 1-CTA
 * launch compares g with *skip_if_equals on the device and returns at once when they match (the gradients of
 * mafed_distill_step are already right); otherwise it starts the backward itself, stream-ordered behind it
 * (device-side tail launch).  `grad_out_seen` (optional, device-accessible, e.g. pinned host memory) receives g,
 * so that a caller can learn the upstream gradient its steps really get without synchronising.  The kernel this
 * library sends to `stream` right after a gate is launched without the programmatic-dependent-launch attribute, so
 * that it cannot occupy the SMs before a backward the gate started. */
int mafed_distill_bwd(const mafed_shape_t* shape, const void* const* student_ptrs,
                      const void* const* teacher_ptrs, void* const* grad_ptrs, const int64_t* attn_mask,
                      const float* bwd_scale, const float* grad_out, float grad_out_scale,
                      const float* skip_if_equals, float* grad_out_seen, void* stream);

/* ---- the stages separately (NCCL sequence, tests) -------------------------------------------------------------
 * Fused forward over all selected layers: one pass over student and teacher (replaces the 2 x
 * _compute_{mse,cosine}_distillation_loss passes per layer, distillation.py:152-162,226-249).  Writes per-CTA
 * partial [layer][text|vision] sums to `ws`. */
int mafed_distill_fwd(const mafed_shape_t* shape, const void* const* student_ptrs,
                      const void* const* teacher_ptrs, const int64_t* attn_mask, void* ws, void* stream);

/* The streaming kernel of the one-pass step alone: gradients + per-CTA partial sums (no losses).  `weights` != NULL:
 * the call also produces `bwd_scale` from the mask counts (with `comm`, from the counts exchanged inside the
 * kernel); `weights` == NULL: `bwd_scale` is an input (SCALE stage run on allreduced counts). */
int mafed_distill_fused(const mafed_shape_t* shape, const void* const* student_ptrs,
                        const void* const* teacher_ptrs, void* const* grad_ptrs, const int64_t* attn_mask,
                        const mafed_weights_t* weights, float* bwd_scale, float assumed_grad_out, void* ws,
                        mafed_comm_t* comm, void* stream);

/* The single-CTA scalar stage; `flags` selects its parts (MAFED_STAGE_*):
 *   REDUCE : deterministic fp64 reduction of `ws` (fixed order) -> sums[0 .. 2L)
 *   COUNTS : n_text = sum(attn_mask), n_vis = B*n_vis           -> sums[2L], sums[2L+1]
 *   LOSSES : sums -> out[1+3L] = {total, layer losses, (text, vision) losses}
 *            (distillation.py:110-120,163; distillation_loss_weights.py:148-174)
 *   SCALE  : counts -> bwd_scale[2L] = c_l * coeff * w_m * k / n_m  (k = 2/D for mse, 1 for cosine)
 * Parts that are not selected read their inputs from `sums`; parts that are write them there (when `sums` is not
 * NULL).  With `comm` the selected part of the sums vector (`comm_what`: MAFED_COMM_SUMS = [0, 2L),
 * MAFED_COMM_COUNTS = [2L, 2L+2)) is allreduced over the peer mailboxes after REDUCE/COUNTS and before
 * LOSSES/SCALE (`sums` must then not be NULL).  The usual combinations: REDUCE|COUNTS (rank-local vector before an
 * allreduce), LOSSES|SCALE (after it), COUNTS|SCALE (before mafed_distill_fused with weights == NULL). */
int mafed_distill_scalar_stage(const mafed_shape_t* shape, const mafed_weights_t* weights, int flags,
                               const int64_t* attn_mask, const void* ws, double* sums, float* out,
                               float* bwd_scale, mafed_comm_t* comm, int comm_what, void* stream);

/* Gradient-norm modality importances (distillation_loss_weights.py:122-137): for every tensor of the
 * table (one per selected layer, [B, T, D]) the per-token L2 norm over D (`torch.linalg.norm(grad,
 * dim=-1)`, :131) summed per modality with the mask weights (:133-137), all layers in one pass.
 * Writes per-CTA partials to `ws`; follow with mafed_distill_reduce to obtain
 * sums[2l] = sum_text w*|g|, sums[2l+1] = sum_vision |g|, sums[2L], sums[2L+1] = token counts.
 * shape->loss_kind is ignored. */
int mafed_distill_token_norm_sums(const mafed_shape_t* shape, const void* const* tensor_ptrs,
                                  const int64_t* attn_mask, void* ws, void* stream);

/* The two [B, T] int64 masks the reference stores into the batch dict (distillation.py:134-144):
 * lang_mask[:, n_vis:] = attn_mask, image_mask[:, :n_vis] = 1, zeros elsewhere -- one launch, on the
 * device (the reference builds them on the CPU and copies them over, per layer). */
int mafed_distill_modality_masks(const mafed_shape_t* shape, const int64_t* attn_mask, int64_t* lang_mask,
                                 int64_t* image_mask, void* stream);

/* ---- host-buffer step: the whole path for callers whose hidden states live in HOST memory ----------
 * create: allocates the device staging pool (mafed_host_step_device_bytes), three streams and events.
 * run   : per layer H2D(student, teacher) -> one-pass fused kernel -> D2H(gradient), pipelined over the
 *         three streams; returns when gradients (h_grad[l], student dtype) and h_out[1+3L] = {total, layer
 *         losses, (text, vision) losses} are in host memory.  `grad_out` is the upstream gradient (host
 *         value).  Host buffers should be pinned (mafed_host_register) for full PCIe bandwidth.
 *         With `comm` the step is batch-sharded: the counts are sent ahead once (mafed_distill_prefetch_counts,
 *         right after the mask copy) and every layer's launch exchanges its sums with the peers.
 * Same results as mafed_distill_step on device-resident tensors. */
typedef struct mafed_host_step mafed_host_step_t;
size_t mafed_host_step_device_bytes(const mafed_shape_t* shape);
int mafed_host_step_create(const mafed_shape_t* shape, mafed_host_step_t** out);
int mafed_host_step_run(mafed_host_step_t* step, const mafed_weights_t* weights, const void* const* h_student,
                        const void* const* h_teacher, void* const* h_grad, const int64_t* h_mask, float grad_out,
                        float* h_out, mafed_comm_t* comm /* NULL: single rank */);
int mafed_host_step_destroy(mafed_host_step_t* step);
int mafed_host_register(void* ptr, size_t bytes);
int mafed_host_unregister(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* MAFED_DISTILL_H_ */

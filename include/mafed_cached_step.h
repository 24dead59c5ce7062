/* mafed_cached_step.h -- C ABI of libmafed_cached_step.so: the one-pass distillation step of a replay batch whose
 * teacher hidden states come from the per-task teacher cache (FeatureDistillation(teacher_cache=True)), read by the
 * step's kernels straight from the cache -- no gathered [B, T, D] copy is made.
 *
 * The cache holds, per distilled layer, one contiguous [M, T_c, D] tensor (mafed_teacher_gather.h).  Sample b of the
 * step is memory sample idx[b]; its teacher row t is
 *
 *   cache[l][idx[b], t, :]                 t <  n_vis   (visual prefix)
 *   cache[l][idx[b], t + (T_c - T), :]     t >= n_vis   (right-aligned text block)
 *
 * which is exactly what mafed_teacher_gather would write into out[l][b, t, :].  The loss, gradients, modality masks and
 * scale table are bit-identical to mafed_teacher_gather followed by mafed_distill_step / mafed_distill_bwd on the
 * gathered tensors: the same kernels (TMA ring) run the same arithmetic on the same rows.
 *
 * Conventions as mafed_distill.h (host pointer tables, device tensors, int64 attention mask [B, T - n_vis], cudaStream_t
 * passed as void*, 0 = ok, MAFED_E_* < 0, a cudaError_t > 0).  No allocation and no host synchronisation.  Every kernel
 * of this library is launched without the programmatic-dependent-launch attribute, so that none of them can occupy the
 * SMs ahead of a backward that a gate of libmafed_distill.so started from the device. */
#ifndef MAFED_CACHED_STEP_H_
#define MAFED_CACHED_STEP_H_

#include <stdint.h>

#include "mafed_distill.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MAFED_CACHED_ABI_VERSION 1
#define MAFED_CACHED_MAX_SAMPLES 2048 /* samples of one call: the index table travels in the kernel parameters */

int mafed_cached_step_abi_version(void);
const char* mafed_cached_step_error_string(int code);

/* 1 if mafed_cached_step takes this step, 0 if not (the caller then gathers and runs mafed_distill_step).  Decided
 * from the shape, the tuning and the pointers alone, without a device:
 *   - shape valid for mafed_distill_step, not CLS, B <= MAFED_CACHED_MAX_SAMPLES, 1 <= M <= 2^31 - 1,
 *     0 <= n_vis <= T <= T_c, B * T <= 2^31 - 1;
 *   - a dtype the TMA-ring kernels read: one of f32 / bf16 / f16 on both sides, or an f32 student with a bf16 / f16
 *     teacher (the cache's type), with D % 8 == 0 for such a pair;
 *   - student rows of whole 16-byte chunks and at most 32 KB, every student pointer and every cache pointer 16-byte
 *     aligned (the step on gathered tensors would take the TMA ring; the cache's rows are whole chunks too);
 *   - no tuning that sends the step elsewhere (MAFED_TUNE_VARIANT_ALL = LDG, MAFED_TUNE_NO_TAIL). */
int mafed_cached_step_supported(const mafed_shape_t* shape, const void* const* student_ptrs,
                                const void* const* cache_ptrs, int64_t M, int32_t T_c);

/* mafed_distill_step for a single rank, with the teacher read from the cache:
 *   cache_ptrs[l] : device pointer of layer l's [M, T_c, D] cache (the teacher type of shape->dtype)
 *   idx           : host array of shape->B memory indices, each in [0, M) (read during the call)
 * Every other argument as mafed_distill_step (sums optional).  Shapes that mafed_cached_step_supported refuses are
 * MAFED_E_ARG, as are an index outside [0, M), T > T_c, T < n_vis and more than MAFED_CACHED_MAX_SAMPLES samples. */
int mafed_cached_step(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* cache_ptrs,
                      int64_t M, int32_t T_c, const int64_t* idx, void* const* grad_ptrs, const int64_t* attn_mask,
                      const mafed_weights_t* weights, float assumed_grad_out, void* ws, float* out, float* bwd_scale,
                      double* sums, int64_t* lang_mask, int64_t* image_mask, void* stream);

/* The backward of mafed_cached_step, as mafed_distill_bwd with the teacher read from the cache.  With skip_if_equals
 * (a HOST float) it is the step's fix-up: a full grid whose CTAs return at once when g = *grad_out * grad_out_scale
 * equals *skip_if_equals (the gradients of mafed_cached_step are already right) and otherwise recompute them exactly.
 * grad_out_seen (optional, device-accessible, e.g. pinned host memory) receives g in either case. */
int mafed_cached_step_bwd(const mafed_shape_t* shape, const void* const* student_ptrs, const void* const* cache_ptrs,
                          int64_t M, int32_t T_c, const int64_t* idx, void* const* grad_ptrs, const int64_t* attn_mask,
                          const float* bwd_scale, const float* grad_out, float grad_out_scale,
                          const float* skip_if_equals, float* grad_out_seen, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* MAFED_CACHED_STEP_H_ */

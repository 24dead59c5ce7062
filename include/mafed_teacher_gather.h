/* mafed_teacher_gather.h -- C ABI of libmafed_teacher_gather.so: the replay step's teacher hidden states gathered from a
 * per-task cache of the episodic memory (FeatureDistillation(teacher_cache=True)).
 *
 * The cache holds, per distilled layer, one contiguous [M, T_c, D] tensor: the teacher's hidden states of every memory
 * sample, computed once at T_c = n_vis + (longest text of the memory set) with the text left-padded.  A batch of B
 * samples (memory indices idx[b]) at length T <= T_c is gathered into one [B, T, D] tensor per layer:
 *
 *   out[l][b, t, :] = cache[l][idx[b], t, :]                 t <  n_vis   (visual prefix)
 *   out[l][b, t, :] = cache[l][idx[b], t + (T_c - T), :]     t >= n_vis   (right-aligned text block)
 *
 * so each (layer, sample) is two contiguous runs of rows.  A sample whose index is >= M (or negative) reads nothing and
 * gets NaN rows (the project's marker of a poisoned step).  No torch types: pointers, sizes and a cudaStream_t. */
#ifndef MAFED_TEACHER_GATHER_H
#define MAFED_TEACHER_GATHER_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAFED_GATHER_ABI_VERSION 1

/* element types (as mafed_distill.h) */
#define MAFED_GATHER_F32 0
#define MAFED_GATHER_BF16 1
#define MAFED_GATHER_F16 2

/* return codes */
#define MAFED_GATHER_OK 0
#define MAFED_GATHER_EINVAL 1      /* an argument is out of range (see mafed_teacher_gather) */
#define MAFED_GATHER_ECUDA 2       /* a CUDA call failed (device query or launch) */

int mafed_teacher_gather_abi_version(void);
const char* mafed_teacher_gather_error_string(int code);

/* Gather n_layers layers for B samples, stream-ordered on `stream` (a cudaStream_t; NULL: the legacy stream).
 *   out[l]   : device pointer of layer l's [B, T, D] output (contiguous)
 *   cache[l] : device pointer of layer l's [M, T_c, D] cache (contiguous)
 *   idx      : host array of B memory indices (read during the call; any value, see above)
 *   dtype    : MAFED_GATHER_F32 / _BF16 / _F16 (the element type of every out[l] and cache[l])
 * Requires n_layers >= 1, B >= 1, M >= 1, 0 <= n_vis <= T <= T_c, D >= 1 and non-NULL tables and entries.  Any number
 * of layers and samples: the call launches once per 64 layers and 2048 samples (one launch at the sizes of a step). */
int mafed_teacher_gather(void* const* out, const void* const* cache, const int64_t* idx, int n_layers, int B, int64_t M,
                         int T, int T_c, int n_vis, int D, int dtype, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* MAFED_TEACHER_GATHER_H */

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

#define MAFED_GATHER_ABI_VERSION 2

/* element types (as mafed_distill.h) */
#define MAFED_GATHER_F32 0
#define MAFED_GATHER_BF16 1
#define MAFED_GATHER_F16 2

/* return codes */
#define MAFED_GATHER_OK 0
#define MAFED_GATHER_EINVAL 1      /* an argument is out of range (see mafed_teacher_gather) */
#define MAFED_GATHER_ECUDA 2       /* a CUDA call failed (device query or launch) */
#define MAFED_GATHER_ESHARD 3      /* a shard could not be allocated, exported or mapped (mafed_teacher_shard_*) */

#define MAFED_GATHER_MAX_RANKS 16  /* ranks of one sharded cache (one NVLink box) */

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

/* ---- a cache sharded across the ranks of one box (FeatureDistillation(shard_teacher_cache=True))
 *
 * Each rank holds one device buffer (its shard) for all cached layers: layer l starts at the same byte offset
 * layer_off[l] in every rank's shard, and slot s of layer l is the [T_c, D] block at layer_off[l] + s * T_c * D * e.
 * Every rank allocates the same capacity.  The buffers are exchanged as CUDA-IPC handles (the caller carries the
 * handle bytes between processes, e.g. with torch.distributed) and mapped into every peer, whose gather then reads
 * the rows with plain loads over NVLink. */
typedef struct mafed_teacher_shard mafed_teacher_shard_t;

int mafed_teacher_shard_handle_bytes(void); /* size of one rank's handle (a cudaIpcMemHandle_t) */

/* Allocate this rank's shard of `bytes` bytes (cudaMalloc: 256-byte aligned) on the current device and write its IPC
 * handle to ipc_handle_out (mafed_teacher_shard_handle_bytes() bytes).  1 <= world <= MAFED_GATHER_MAX_RANKS. */
int mafed_teacher_shard_create(int world, int rank, int64_t bytes, void* ipc_handle_out, mafed_teacher_shard_t** out);

/* Map every peer's shard: all_handles holds the world ranks' handles, in rank order (this rank's own is skipped). */
int mafed_teacher_shard_connect(mafed_teacher_shard_t* shard, const void* all_handles);

/* Device address of rank `rank`'s shard as this process sees it (its own buffer, or the mapping of a peer's). */
int mafed_teacher_shard_base(const mafed_teacher_shard_t* shard, int rank, void** base_out);

/* Close the peers' mappings, then free this rank's buffer.  Not a synchronisation: every rank's reads of this shard
 * must have finished (e.g. a device synchronise and a barrier on every rank first). */
int mafed_teacher_shard_destroy(mafed_teacher_shard_t* shard);

/* Gather from a sharded cache: as mafed_teacher_gather, with sample b read from slot slot[b] of rank src_rank[b]:
 *   out[l][b, t, :] = rows of (bases[src_rank[b]] + layer_off[l] + slot[b] * T_c * D * e), mapped as above
 *   bases     : n_ranks device addresses of the shards (mafed_teacher_shard_base), 1 <= n_ranks <= 16
 *   layer_off : n_layers byte offsets (>= 0) of the layers in every shard
 *   src_rank, slot : host arrays of B entries; a slot outside [0, slots) or a rank outside [0, n_ranks) gives NaN rows
 * Every base + offset and every out[l] must be aligned to the element size.  One launch per 64 layers and 2048
 * samples, one kernel for local and peer rows. */
int mafed_teacher_gather_sharded(void* const* out, const void* const* bases, int n_ranks, const int64_t* layer_off,
                                 const int32_t* src_rank, const int64_t* slot, int n_layers, int B, int64_t slots,
                                 int T, int T_c, int n_vis, int D, int dtype, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* MAFED_TEACHER_GATHER_H */

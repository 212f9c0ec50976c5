/*
 * spt_b200.h — C ABI of libspt_b200.so, the B200 (sm_100a) implementation of the SPT hot path:
 * PQ sparse multi-head attention (cdist -> lookup -> sddmm -> softmax -> spmm, fwd + bwd, CSR->CSC)
 * and the routed-FFN grouped GEMM.
 *
 * This is the drop-in boundary: it replaces the 7 pybind entry points of the reference's torch
 * extension `naive_gpt.ext` (reference extension/entry.cpp:43-56) and adds the fused / FFN entry
 * points listed in SURVEY.md section 8(b).  Plain pointers and sizes only — no torch types.
 * The Python binding that mirrors the reference's `naive_gpt.ext` on top of this ABI is
 * spt_proto_b200/ext.py; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - tensors are dense, row-major, contiguous (the reference's CHECK_DIM requires contiguity,
 *     extension/common.h:13-18);
 *   - `dtype` selects the element type of q/k/v-like operands: SPT_F32 or SPT_BF16 (SPT_F16 where
 *     stated, see spt_dtype).  Indices are
 *     int32, CSR values / probabilities / distances are always fp32, accumulation is fp32;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Every kernel is
 *     launched on it; nothing synchronises the device;
 *   - the return value is an spt_status; spt_last_error() returns a thread-local message;
 *   - the callee never allocates device memory: outputs and workspaces are caller-provided
 *     (ownership rule of SURVEY.md section 8(b): the torch caching allocator owns everything).
 */
#ifndef SPT_B200_H
#define SPT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *spt_stream_t; /* cudaStream_t */

typedef enum {
    SPT_OK = 0,
    SPT_ERR_INVALID_ARGUMENT = 1, /* bad shape / null pointer; maps to TORCH_CHECK -> RuntimeError */
    SPT_ERR_UNSUPPORTED = 2,      /* legal in principle, no kernel instantiated                    */
    SPT_ERR_CUDA = 3              /* launch or runtime error (cudaGetLastError)                    */
} spt_status;

/* SPT_F16 is accepted by spt_pq_encode, spt_pq_encode_pair, spt_pq_train_fwd / _bwd, the fused attention
 * (spt_sparse_attn_fwd / _bwd, their _ex and _varlen variants) and the routed FFN: spt_grouped_gemm,
 * spt_gather_rows_bf16 (a 16-bit row copy), spt_ffn_combine, spt_group_colsum, spt_scale_add_fwd / _bwd,
 * spt_lora_glu_fwd_ex / _bwd_ex and spt_silu_mul_fwd_ex / _bwd_ex.  Every other entry point takes SPT_F32 /
 * SPT_BF16 only.  bf16 and fp16 never mix in one call. */
typedef enum { SPT_F32 = 0, SPT_BF16 = 1, SPT_F16 = 2 } spt_dtype;

#define SPT_ABI_VERSION 1

int spt_abi_version(void);
const char *spt_last_error(void);
/* Number of kernel launches issued through this library by the calling process (all threads).
 * bench.py uses the difference across the timed region for its `gpu_launches` claim. */
uint64_t spt_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * (1) cdist — replaces cdist_forward_cuda / cdist_backward_cuda (extension/cdist.cu:185-333).
 * query [m, n, dc] (dtype), table [m, c, dc] fp32.
 * distance [m, n, c] fp32 (may be NULL: codes only), indices [m, n] int32.
 * L1 distance summed over i ascending in fp32, strict-< running minimum: lowest index wins ties.
 * Lifted restrictions vs the reference: any n, any c >= 1, dc in [1, 64].
 * ------------------------------------------------------------------------------------------ */
int spt_cdist_fwd(const void *query, const float *table, float *distance, int32_t *indices,
                  int m, int64_t n, int c, int dc, int dtype, spt_stream_t stream);

/* grad_distance [m, n, c] -> grad_query [m, n, dc], grad_table [m, c, dc] (all fp32).
 * sgn(q - t) = +1 if q - t > 0 else -1 (cdist.cu:117,168).  grad_table is accumulated with a
 * deterministic two-stage reduction; `workspace` must hold spt_cdist_bwd_workspace_bytes(). */
size_t spt_cdist_bwd_workspace_bytes(int m, int64_t n, int c, int dc);
int spt_cdist_bwd(const float *query, const float *table, const float *grad_distance,
                  float *grad_query, float *grad_table, void *workspace,
                  int m, int64_t n, int c, int dc, spt_stream_t stream);

/* Fused PQBase.forward(mode='encode') (naive_gpt/layers/basic/quantizer.py:26-77): z [rows, m*dc]
 * (dtype) in its natural head-major layout -> codes [rows, m] int32.  No transposed copy, no
 * distance tensor. */
int spt_pq_encode(const void *z, const float *table, int32_t *codes,
                  int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream);
/* The same for two tensors of identical shape that share the codebook — the q and k of one attention
 * call (naive_gpt/layers/sparse/attention.py:105-106) — in a single launch. */
int spt_pq_encode_pair(const void *z0, const void *z1, const float *table, int32_t *codes0, int32_t *codes1,
                       int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream);

/* Fused PQBase.forward(mode='train') (quantizer.py:81-111): z [rows, m*dc] (dtype), table [m, c, dc] fp32.
 *   fwd: zq_out [rows, m*dc] fp32 (hard centroids, may be NULL); partial [spt_pq_train_blocks(rows, m)] fp32 with
 *        sum(partial) / (rows*m*dc) = mean((zw - zq)^2) + mean((z - zq)^2), zw = soft centroid (see cdist.cu).
 *   bwd: grad_loss [1] fp32 (device), grad_zq [rows, m*dc] fp32 or NULL -> grad_z [rows, m*dc] (dtype) and
 *        grad_table_partial [spt_pq_train_blocks(rows, m)][m][c][dc] fp32 (sum over the first axis = grad_table).
 * Covers c = 16, dc = 8 (the reference's configuration, utils/adapter.py:94-97), m <= 64. */
int spt_pq_train_blocks(int64_t rows, int m);
int spt_pq_train_fwd(const void *z, const float *table, float *zq_out, float *partial,
                     int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream);
int spt_pq_train_bwd(const void *z, const float *table, const float *grad_zq, const float *grad_loss,
                     void *grad_z, float *grad_table_partial,
                     int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (2) lookup — replaces lookup_forward_cuda (extension/lookup.cu:87-174).
 * query_codes, key_codes [B, S, m] int32 -> output [B, S, nnz] int32, nnz = S / sparse_coeff.
 * Bit-exact with the reference kernel's semantics (bucketed causal candidate selection, zero
 * padding; see oracle/spt_oracle.py::lookup_spec).  Codes are compared modulo 2^16 like the
 * reference's uint16 shared-memory caches.  Every output element is written (no pre-zeroing).
 * Requirements: m >= 4, nnz % 4 == 0, nnz >= 8, S <= 65536.  The (m, nnz) whitelist of the
 * reference (lookup.cu:113-169) is lifted.
 * `workspace` must hold spt_lookup_workspace_bytes(); it may be NULL when that returns 0.
 * ------------------------------------------------------------------------------------------ */
size_t spt_lookup_workspace_bytes(int B, int S, int m, int nnz);
int spt_lookup_fwd(const int32_t *query_codes, const int32_t *key_codes, int32_t *output,
                   void *workspace, int B, int S, int m, int nnz, spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (3) sddmm — replaces sddmm_forward_cuda (extension/sddmm.cpp:3-73) for op(A)=N, op(B)=T:
 * values[b, e] = <query[b, row(e), :], key[b, indices[b, e], :]>.
 * indptr [S+1] int32 is shared by the whole batch (stride-0 batch, sddmm.cpp:49);
 * indices [B, nnz] int32; query, key [B, S, d] (dtype); values [B, nnz] fp32.
 * `scale`/`clamp`: values = clamp(scale * dot, -clamp, +clamp) when clamp > 0 (fuses
 * attention.py:125-127); pass scale = 1, clamp = 0 for the plain reference semantics.
 * ------------------------------------------------------------------------------------------ */
int spt_sddmm_fwd(const int32_t *indptr, const int32_t *indices, const void *query, const void *key,
                  float *values, int B, int S, int d, int64_t nnz, float scale, float clamp,
                  int dtype, spt_stream_t stream);

/* Backward of the fused scale + clamp of spt_sddmm_fwd (the reference does them as two eager passes whose autograd
 * backward is a masked multiply, layers/sparse/attention.py:125-127): out = scale * grad where |clamped| < clamp, else 0.
 * n (multiple of 4) fp32 elements, 16-byte aligned; clamp <= 0 means no clamp. */
int spt_clamp_scale_bwd(const float *grad, const float *clamped, float *out, int64_t n, float scale, float clamp,
                        spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5) spmm — replaces spmm_forward_cuda (extension/spmm.cpp:3-72).
 * trans = 0: y[b, r, :]  = sum_{e in row r} values[b, e] * x[b, indices[b, e], :]
 * trans = 1: y[b, c, :]  = sum_{e : indices[b,e] = c} values[b, e] * x[b, row(e), :]
 *            (the reference's CUSPARSE_OPERATION_TRANSPOSE path used for dK / dV).
 * x, y [B, S, d]; x is (dtype), y is (out_dtype).  trans = 1 needs the CSC built by
 * spt_csr2csc (col_ptr, row_idx, perm).  Summation order: fp32 x (and every shape the dense-tile
 * kernel does not take): row ascending, CSR order inside a row => bit-reproducible run to run,
 * unlike the atomics-based cuSPARSE path.  bf16 x with d 64 / 128: 64-row chunks ascending,
 * tensor-core order inside a chunk, fp32 weights kept as bf16 hi + lo (~16 bits); deterministic
 * except for the order in which DUPLICATE entries of one (row, column) cell add up.  Lists that
 * are not in ascending row order are accepted (slower gathered loop for the blocks concerned).
 * ------------------------------------------------------------------------------------------ */
int spt_spmm_fwd(const int32_t *indptr, const int32_t *indices, const float *values, const void *x,
                 void *y, int B, int S, int d, int64_t nnz, int dtype, int out_dtype,
                 spt_stream_t stream);
int spt_spmm_t_fwd(const int32_t *col_ptr, const int32_t *row_idx, const int32_t *perm,
                   const float *values, const void *x, void *y, int B, int S, int d, int64_t nnz,
                   int dtype, int out_dtype, spt_stream_t stream);

/* (5b) tile index of the pattern + the transposed product on it — the form the backward passes
 * (reference kernels/spmm.py:42-47, kernels/sddmm.py:44-49: cuSPARSE TRANSPOSE) use for bf16 x with
 * head dim 64 / 128.  Instead of a full CSR -> CSC transposition the index only buckets the entries
 * by (64-column tile, 64-row chunk):
 *   tile_ptr [B, n*n + 1] int32, n = ceil(S / 64): bucket (ct, rc) of head b = entries
 *            tile_ptr[b][ct*n + rc] .. tile_ptr[b][ct*n + rc + 1] of tile_ent[b]
 *   tile_ent [B, nnz] uint32: c_local | r_local << 6 | e << 12, e = position in the head's CSR
 * (so a head holds at most 2^20 entries and S <= 8192: spt_csr_tiles_supported).  The SET of entries
 * of a bucket is deterministic, their order inside it is not (shared-memory atomics).
 * spt_spmm_t_tiles_fwd: y[b, c, :] = sum_{e : indices[b,e] = c} values[b, e] * x[b, row(e), :],
 * x bf16 [B, S, d], d 64 / 128, y bf16 or fp32; fp32 weights enter the tensor cores as bf16 hi + lo
 * (~16 bits), accumulation fp32; duplicates of one (row, column) cell add up in an unspecified order. */
int spt_csr_tiles_supported(int S, int64_t nnz);
int64_t spt_csr_tiles_ptr_len(int S);
int spt_csr_tiles(const int32_t *indptr, const int32_t *indices, int32_t *tile_ptr, uint32_t *tile_ent,
                  int B, int S, int64_t nnz, spt_stream_t stream);
int spt_spmm_t_tiles_fwd(const int32_t *tile_ptr, const uint32_t *tile_ent, const float *values,
                         const void *x, void *y, int B, int S, int d, int64_t nnz, int dtype,
                         int out_dtype, spt_stream_t stream);
/* values[b, e] = clamp(scale * <query[b, row(e)], key[b, col(e)]>) on the same index (the spt_sddmm_fwd
 * product, bf16 operands, head dim 64 / 128): dense 64 x 64 score tiles on the tensor cores, every
 * entry picks its cell. */
int spt_sddmm_tiles_fwd(const int32_t *tile_ptr, const uint32_t *tile_ent, const void *query,
                        const void *key, float *values, int B, int S, int d, int64_t nnz, float scale,
                        float clamp, int dtype, spt_stream_t stream);
/* both directions on the same index: trans = 0 is y[b, r, :] = sum_{e in row r} values[b, e] *
 * x[b, indices[b, e], :] (the spt_spmm_fwd product), trans = 1 the one above */
int spt_spmm_tiles_fwd(const int32_t *tile_ptr, const uint32_t *tile_ent, const float *values,
                       const void *x, void *y, int B, int S, int d, int64_t nnz, int dtype,
                       int out_dtype, int trans, spt_stream_t stream);

/* (a-7) CSR -> CSC (implicit in the reference's transposed cuSPARSE calls, explicit in
 * legacy/csr2csc.cpp:3-54).  indptr [S+1] shared, indices [B, nnz] ->
 * col_ptr [B, S+1], row_idx [B, nnz], perm [B, nnz] (values_csc = values[perm]).
 * Stable: rows ascending inside a column, duplicates keep CSR order. */
size_t spt_csr2csc_workspace_bytes(int B, int S, int64_t nnz);
int spt_csr2csc(const int32_t *indptr, const int32_t *indices, int32_t *col_ptr, int32_t *row_idx,
                int32_t *perm, void *workspace, int B, int S, int64_t nnz, spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (4) softmax — replaces softmax_forward_cuda / softmax_backward_cuda (extension/softmax.cu:84-148).
 * Row softmax over the stored entries with the causal predicate (indices[e] <= row) as a 0/1
 * factor, no max subtraction, denominator clamped to >= 1e-9 (softmax.cu:16-46).
 * Backward is the TRUE gradient y * (dy - sum(y*dy)) — the reference kernel's clamp of the sum to
 * >= 1e-9 (softmax.cu:69) is a bug and is not reproduced by default (DESIGN.md section 3).
 * spt_softmax_bwd_ex(reference_clamp = 1) reproduces the shipped kernel for A/B training-parity
 * runs (Python: ext.REFERENCE_SOFTMAX_CLAMP / env SPT_REFERENCE_SOFTMAX_CLAMP=1).
 * ------------------------------------------------------------------------------------------ */
int spt_softmax_fwd(const int32_t *indptr, const int32_t *indices, const float *values, float *output,
                    int B, int S, int64_t nnz, spt_stream_t stream);
int spt_softmax_bwd(const int32_t *indptr, const int32_t *indices, const float *output,
                    const float *grad_output, float *grad_values, int B, int S, int64_t nnz,
                    spt_stream_t stream);
int spt_softmax_bwd_ex(const int32_t *indptr, const int32_t *indices, const float *output,
                       const float *grad_output, float *grad_values, int B, int S, int64_t nnz,
                       int reference_clamp, spt_stream_t stream);
/* softmax backward through v = clamp(scale * raw, -clamp, clamp) (the layer's eager `clamp_(scaling * values, -10, 10)`,
 * naive_gpt/layers/sparse/attention.py:125-127, in front of the softmax): grad_raw = scale * dv where |clamped| < clamp,
 * else 0, with dv as above — spt_softmax_bwd_ex followed by spt_clamp_scale_bwd in one pass, bit-identical. */
int spt_softmax_clamp_bwd(const int32_t *indptr, const int32_t *indices, const float *output,
                          const float *grad_output, const float *clamped, float *grad_raw, int B, int S,
                          int64_t nnz, float scale, float clamp, int reference_clamp, spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Fused sparse attention (fast path of SparseVanillaAttentionV2 / SparseRotaryAttentionV2,
 * naive_gpt/layers/sparse/attention.py:105-141) as masked dense tiles on the tensor cores.
 *
 * spt_lookup_mask_fwd: same selection as spt_lookup_fwd, emitted as a per-row bitmask
 *   mask [B, S, S/32] uint32, lane-major: bit i of word 4 g + t <=> key 128 g + 4 i + t selected, and
 *   extra0 [B, S] int32 = number of zero-padding slots of the row (multiplicity of key 0 beyond its
 *   own bit).  `output` (the int32 index tensor) may be NULL on this path.  Needs S % 128 == 0.
 *   S <= 65536.  Mask-only calls (output NULL) at m = 8, 10 or 16 take no more shared memory than a
 *   fixed amount at any S (DESIGN.md section 4.1).  Codes >= 16 are handled by a fallback kernel,
 *   decided on the device; its row images (32 nnz 2 + S 4 + 32 m 2 bytes) must fit 200 KB, i.e.
 *   S up to about 16 k at sparse_coeff 8.  Beyond that spt_lookup_mask_fwd fails.
 * spt_lookup_mask_fwd_ex: the same, with the caller's promise that every code is < n_codewords.
 *   Where the fallback fits, it launches exactly what spt_lookup_mask_fwd launches.  Where it does
 *   not: n_codewords > 16 returns SPT_ERR_UNSUPPORTED before any CUDA call; n_codewords <= 16 runs
 *   without the fallback (mask-only calls at m 8, 10, 16 only), and a code >= 16 that arrives all
 *   the same matches no key: the result stays deterministic and nothing is written outside mask and
 *   extra0.
 *
 * spt_sparse_attn_fwd: q, k, v [B, S, d] bf16 or fp16 (dtype SPT_BF16 / SPT_F16) ->
 *   y [B, S, d] (same type) = sum_j p_rj v_j,  p = w * exp(clamp(scale * q.k, -clamp, clamp)) / Z,
 *   zsum [B, S] fp32 = Z (row sums, >= 1e-9) saved for the backward.  d = 64, 80 or 128 (others
 *   return SPT_ERR_UNSUPPORTED), S % 128 == 0.  d = 80 (OPT-2.7B) is padded to 128 in shared
 *   memory and tensor memory only: every global read and write is exactly d columns wide.
 *   fp16 keeps every packed probability in range with a power-of-two scale per row that cancels in
 *   y and in the gradients (DESIGN.md section 4.1); it needs clamp <= 10 (SPT_ERR_UNSUPPORTED beyond).
 * spt_sparse_attn_bwd: grad_y -> grad_q, grad_k, grad_v [B, S, d] (dtype).  Recomputes p from q, k
 *   (nothing of size S x k is read or written); deterministic (no atomics).
 *   workspace: spt_sparse_attn_bwd_workspace_bytes(B, S) = B*S*4 + B*S*128*2 bytes (delta' fp32 and
 *   dO', sized for d = 128).
 * Layout: H = 1 means head-major [B, S, *] operands (the reference's layout after its transposes);
 * H > 1 means the layer's native [N, S, H, *] layout with B = N*H heads interleaved (codes
 * [N, S, H, m]; q/k/v/y and their gradients [N, S, H, d]) — the kernels stride over it directly, so
 * the reference's transpose(1,2).contiguous() copies (attention.py:92-95,138-142) disappear.
 * mask / extra0 / zsum are always head-major [B, S, ...].
 * _ex variants take `flags`: SPT_ATTN_Y_TRANSPOSED = y (forward output, and y / grad_y of the
 * backward) live in the SHIPPED reference layer's output layout — _apply_attn un-transposes the
 * [N*H, S, E] result with transpose(1, 2).contiguous().view(v_size) (attention.py:139-142), i.e.
 * y^T [B, d, S] memory re-interpreted as [N, S, H, E].  The kernels write / read that memory
 * directly (forward epilogue, backward row prologue): the drop-in default costs no extra pass.
 * ------------------------------------------------------------------------------------------ */
#define SPT_ATTN_Y_TRANSPOSED 1
int spt_lookup_mask_fwd(const int32_t *query_codes, const int32_t *key_codes, int32_t *output,
                        uint32_t *mask, int32_t *extra0, void *workspace, int B, int S, int m, int nnz,
                        int H, spt_stream_t stream);
int spt_lookup_mask_fwd_ex(const int32_t *query_codes, const int32_t *key_codes, int32_t *output,
                           uint32_t *mask, int32_t *extra0, void *workspace, int B, int S, int m, int nnz,
                           int H, int n_codewords, spt_stream_t stream);
int spt_sparse_attn_fwd(const void *q, const void *k, const void *v, const uint32_t *mask,
                        const int32_t *extra0, void *y, float *zsum, int B, int S, int d, int H,
                        float scale, float clamp, int dtype, spt_stream_t stream);
int spt_sparse_attn_fwd_ex(const void *q, const void *k, const void *v, const uint32_t *mask,
                           const int32_t *extra0, void *y, float *zsum, int B, int S, int d, int H,
                           float scale, float clamp, int dtype, int flags, spt_stream_t stream);
size_t spt_sparse_attn_bwd_workspace_bytes(int B, int S);
int spt_sparse_attn_bwd(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                        const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q,
                        void *grad_k, void *grad_v, void *workspace, int B, int S, int d, int H,
                        float scale, float clamp, int dtype, spt_stream_t stream);
/* ------------------------------------------------------------------------------------------
 * Packed variable-length sequences (DESIGN.md section 4.5).  n_seq sequences of lengths S_i are
 * concatenated along the token axis, T = sum S_i; cu_seqlens int32 [n_seq + 1] (device) holds the
 * offsets, cu[0] = 0, cu[n_seq] = T.  Sequence i (rows cu[i] .. cu[i+1]) gets exactly what the
 * fixed-length calls give for it alone as a batch of one: keys are relative to its first token
 * (key 0 = that token, which zero padding aliases), attention is causal from there.  Needs
 * S_i % 32 == 0, S_i % (4 sparse_coeff) == 0, S_i >= 8 sparse_coeff, S_i <= max_seqlen; S_i and
 * cu[i] need not be multiples of 128.  Nothing synchronises with the host (graph-capturable).
 *
 * spt_varlen_worklist: cu_seqlens -> work list `work` (spt_varlen_worklist_bytes(n_seq, T), 16-byte
 *   aligned): one item per (sequence, 128-row tile), heaviest tiles first.  Built once and passed
 *   to the lookup, the forward and the backward.  Every sequence is clamped to [0, T] and to
 *   max_seqlen on the device, so a bad device-side cu_seqlens cannot send a kernel outside its
 *   tensors (validate host-side offsets before the copy).
 * spt_lookup_mask_varlen_fwd: codes [T, H, m] (m = 8, 10 or 16) -> mask [H, T, Wm] uint32,
 *   Wm = 4 ceil(max_seqlen / 128), lane-major words relative to the sequence start (words past a
 *   row's sequence are zero), extra0 [H, T]; nnz_i = S_i / sparse_coeff.  workspace:
 *   spt_lookup_mask_varlen_workspace_bytes.  spt_lookup_mask_varlen_max_seqlen(m) is the longest
 *   max_seqlen the mask-only kernels take at m: 65536 at m 8, 10 and 16, 0 otherwise.  The codes
 *   >= 16 fallback needs its row images (32 nnz_max 2 + 32 Wm 4 + 32 m 2 bytes, nnz_max =
 *   max_seqlen / sparse_coeff) within 200 KB; beyond that spt_lookup_mask_varlen_fwd fails.
 * spt_lookup_mask_varlen_fwd_ex: as spt_lookup_mask_fwd_ex for the packed call (codes < n_codewords).
 * spt_sparse_attn_varlen_fwd / _bwd: as the _ex calls on q, k, v [T, H, d]; zsum [H, T].
 *   SPT_ATTN_Y_TRANSPOSED: sequence i's y (and grad_y) memory is its own y_i^T [H, d, S_i] at
 *   token offset cu[i] — the reference layer's layout for that sequence alone.
 * ------------------------------------------------------------------------------------------ */
size_t spt_varlen_worklist_bytes(int n_seq, int T);
int spt_varlen_worklist(const int32_t *cu_seqlens, int n_seq, int T, int max_seqlen, void *work,
                        spt_stream_t stream);
size_t spt_lookup_mask_varlen_workspace_bytes(int n_seq, int T, int H, int m);
int spt_lookup_mask_varlen_max_seqlen(int m);
int spt_lookup_mask_varlen_fwd(const int32_t *query_codes, const int32_t *key_codes, const void *work,
                               uint32_t *mask, int32_t *extra0, void *workspace, int n_seq, int T,
                               int max_seqlen, int H, int m, int sparse_coeff, spt_stream_t stream);
int spt_lookup_mask_varlen_fwd_ex(const int32_t *query_codes, const int32_t *key_codes, const void *work,
                                  uint32_t *mask, int32_t *extra0, void *workspace, int n_seq, int T,
                                  int max_seqlen, int H, int m, int sparse_coeff, int n_codewords,
                                  spt_stream_t stream);
int spt_sparse_attn_varlen_fwd(const void *q, const void *k, const void *v, const uint32_t *mask,
                               const int32_t *extra0, void *y, float *zsum, const void *work, int n_seq,
                               int T, int max_seqlen, int d, int H, float scale, float clamp, int dtype,
                               int flags, spt_stream_t stream);
size_t spt_sparse_attn_varlen_bwd_workspace_bytes(int T, int H);
int spt_sparse_attn_varlen_bwd(const void *q, const void *k, const void *v, const void *y,
                               const void *grad_y, const uint32_t *mask, const int32_t *extra0,
                               const float *zsum, void *grad_q, void *grad_k, void *grad_v,
                               void *workspace, const void *work, int n_seq, int T, int max_seqlen,
                               int d, int H, float scale, float clamp, int dtype, int flags,
                               spt_stream_t stream);
/* diagnostics: in-kernel phase timers of the attention kernels, 3 kernels x 16 slots of summed clock64() deltas
 * (zeros and return value 0 unless the library was built with -DSPT_ATTN_PROF); reset != 0 clears them */
int spt_debug_attn_prof(unsigned long long *out48, int reset);
int spt_sparse_attn_bwd_ex(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                           const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q,
                           void *grad_k, void *grad_v, void *workspace, int B, int S, int d, int H,
                           float scale, float clamp, int dtype, int flags, spt_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (6) routed FFN — the grouped GEMM the reference only sketches (legacy/routed.cpp:10-68,
 * legacy/test_routed.py:9-26) and ships as a Python loop (layers/sparse/feedforward.py:47-85).
 *
 * spt_route_bucket: prob [T, nb] fp32 (router output) -> top-`k_active` blocks per token (ties:
 * lowest block index; only set membership matters, feedforward.py:67-70) bucketed by block, every
 * bucket padded to a multiple of 128 rows:
 *   bucket_ptr [nb+1], bucket_rows [nb] (real row counts), tile_group [R/128] (block of each 128-row
 *   tile, -1 past the end), row_token [R] (token of each bucket row, ascending per bucket, -1 =
 *   padding), row_prob [R] (prob[token, block], 0 = padding), token_rows [T, k_active] (bucket rows
 *   of the token's active blocks, blocks ascending — the accumulation order of feedforward.py:66-81).
 * R: caller's upper bound, multiple of 128, >= T*k_active + 127*nb.  nb <= 64.
 * ------------------------------------------------------------------------------------------ */
size_t spt_route_bucket_workspace_bytes(int64_t T, int nb);
int spt_route_bucket(const float *prob, int32_t *bucket_ptr, int32_t *bucket_rows, int32_t *tile_group,
                     int32_t *row_token, float *row_prob, int32_t *token_rows, void *workspace,
                     int64_t T, int nb, int k_active, int64_t R, spt_stream_t stream);
/* Router gradient of the LoRA-routed FFN (naive_gpt/layers/tuning/lora_ffn.py:92,206: the block outputs are scaled by
 * 2 * prob[token, block]): grad_prob [T, nb] fp32 (cleared here) receives 2 * grad_coeff[r] at (row_token[r], block of
 * row r) for every real bucket row — the backward of coeff = 2 * row_prob without torch's sort-based index_put. */
int spt_row_coeff_bwd(const float *grad_coeff, const int32_t *row_token, const int32_t *tile_group,
                      float *grad_prob, int64_t R, int64_t T, int nb, spt_stream_t stream);

/* dst[r, :] = src[row_token[r], :] for r < R, zeros where row_token[r] < 0 (any 16-bit elements, bf16 or fp16:
 * the copy does not look at the values; C % 8 == 0). */
int spt_gather_rows_bf16(const void *src, const int32_t *row_token, void *dst, int64_t R, int C,
                         spt_stream_t stream);

/* Deterministic combine: y[t, :] = bias + sum_j partial[token_rows[t, j], :], j ascending (= block
 * order); fp32 accumulation; bias may be NULL.  (partial, y) dtypes: fp32 with fp32, bf16 or fp16; a
 * 16-bit type with itself or fp32.  Any other pair is SPT_ERR_INVALID_ARGUMENT. */
int spt_ffn_combine(const void *partial, const int32_t *token_rows, const float *bias, void *y, int64_t T,
                    int C, int k_active, int partial_dtype, int y_dtype, spt_stream_t stream);

/* out[g, c] = sum of x[row, c] over the (padded) rows of bucket g — bias gradients; x [R, C] of `dtype`
 * (SPT_BF16 or SPT_F16), out fp32.  spt_group_colsum_bf16 is spt_group_colsum with dtype = SPT_BF16. */
size_t spt_group_colsum_workspace_bytes(int n_groups, int C);
int spt_group_colsum(const void *x, const int32_t *bucket_ptr, float *out, void *workspace,
                     int n_groups, int C, int dtype, spt_stream_t stream);
int spt_group_colsum_bf16(const void *x, const int32_t *bucket_ptr, float *out, void *workspace,
                          int n_groups, int C, spt_stream_t stream);

/* Grouped GEMM on the tcgen05 tensor cores (bf16 or fp16 operands, fp32 accumulation in TMEM, TMA-fed).
 * Operands are described as STORED: a row-major matrix [rows, cols] with leading dimension ld.
 *   K-major operand  (x_mn_major = 0): stored [MN, K]  (reduction dim contiguous)
 *   MN-major operand (x_mn_major = 1): stored [K, MN]  (consumed in place through an MN-major UMMA
 *                                      descriptor, no transposed copy)
 * mode 0 (M-grouped; fc1, fc2, dH, dX): C[i, 0:N] = epi(A[i, :] . op(B_g)), i over 128-row tiles,
 *   g = tile_group[i / 128] (-1: skip).  B_g is addressed by the per-group coordinate offsets
 *   b_k_off (along K) and b_mn_off (along N), both multiplied by g.  A must be K-major.
 *   epi: + bias[g * bias_stride + n], activation (0 none, 1 relu, 2 silu), * row_scale[i]; then, if `gate`
 *   (operand type [rows of C, N], leading dimension ldg) is given, the result is zeroed wherever gate <= 0 —
 *   the ReLU backward mask applied to dH in the epilogue of the GEMM that produces it.
 * mode 1 (K-grouped; weight gradients): for every group g, C_g[0:M, 0:N] = A_g . B_g^T reduced over
 *   rows group_ptr[g] .. group_ptr[g+1] (multiples of 64); C_g origin = (g*c_row_off, g*c_col_off).
 * ab_dtype: the type of A, B and gate, SPT_BF16 or SPT_F16.  C is fp32 or of type ab_dtype, with leading
 * dimension ldc; bias and row_scale are fp32.  A 16-bit C takes one round-to-nearest of the fp32 result, with no
 * saturation: an fp16 C holds inf where |result| rounds above 65504, as torch's fp16 matmul does.  Any other
 * ab_dtype or c_dtype is rejected before any CUDA call.  spt_grouped_gemm_bf16 is spt_grouped_gemm with
 * ab_dtype = SPT_BF16. */
int spt_grouped_gemm(int mode, const void *A, long long a_rows, long long a_cols, long long lda,
                     int a_mn_major, const void *B, long long b_rows, long long b_cols, long long ldb,
                     int b_mn_major, const int32_t *tile_group, int n_m_tiles, const int32_t *group_ptr,
                     int n_groups, int M, int N, int K, int a_k_off, int a_mn_off, int b_k_off, int b_mn_off,
                     long long c_row_off, long long c_col_off, void *C, long long ldc, int c_dtype,
                     const float *bias, int bias_stride, const float *row_scale, int act, const void *gate,
                     long long ldg, int ab_dtype, spt_stream_t stream);
int spt_grouped_gemm_bf16(int mode, const void *A, long long a_rows, long long a_cols, long long lda,
                          int a_mn_major, const void *B, long long b_rows, long long b_cols,
                          long long ldb, int b_mn_major, const int32_t *tile_group, int n_m_tiles,
                          const int32_t *group_ptr, int n_groups, int M, int N, int K, int a_k_off,
                          int a_mn_off, int b_k_off, int b_mn_off, long long c_row_off,
                          long long c_col_off, void *C, long long ldc, int c_dtype, const float *bias,
                          int bias_stride, const float *row_scale, int act, const void *gate, long long ldg,
                          spt_stream_t stream);

/* LlamaRMSNorm (naive_gpt/layers/basic/utils.py:22-38) and RotaryEmbedding (basic/position.py:5-48) of the block
 * around the SPT operators, one kernel per direction, bf16 with the torch expression's intermediate roundings.
 *   rmsnorm: x, out [R, C] bf16, w [C] bf16, inv_rms [R] fp32 (saved for backward); C % 8 == 0, C <= 8192.
 *            backward writes dx [R, C] bf16 and dw_partial [spt_rmsnorm_bwd_blocks(R), C] fp32 (sum over dim 0 = dw).
 *   rope   : x, out [N, S, H, E] bf16 (rows = N*S*H), cos / sin [S, E] bf16 gathered by position; E % 16 == 0;
 *            transpose != 0 applies the transposed rotation (the backward). */
int spt_rmsnorm_bwd_blocks(int64_t R);
int spt_rmsnorm_fwd_bf16(const void *x, const void *w, void *out, float *inv_rms, int64_t R, int C, float eps,
                         spt_stream_t stream);
int spt_rmsnorm_bwd_bf16(const void *g, const void *x, const void *w, const float *inv_rms, void *dx,
                         float *dw_partial, int64_t R, int C, spt_stream_t stream);
int spt_rope_bf16(const void *x, const void *cos, const void *sin, void *out, int64_t rows, int S, int H, int E,
                  int transpose, spt_stream_t stream);

/* Layout copies of the stage path: the reference layer's `transpose(1, 2).contiguous()` of q / k / v and of the
 * product (naive_gpt/layers/sparse/attention.py:92-95, 138-142) as 16-byte-word row moves.
 *   swap_dims12    : out[a, c, b, :] = in[a, b, c, :]; rows of row_bytes (multiple of 16), both 16-byte aligned.
 *   transpose_last2: out[b, c, r] = in[b, r, c], elements of 2 or 4 bytes (the shipped layer's output layout). */
int spt_swap_dims12(const void *in, void *out, int64_t A, int64_t B, int64_t C, int64_t row_bytes, spt_stream_t stream);
int spt_transpose_last2(const void *in, void *out, int64_t batch, int R, int C, int elem_bytes, spt_stream_t stream);

/* Host-side replay of the CTA-pair grouped GEMM's mode-0 schedule (no GPU needed; used by the CPU tests).
 * tile_group is a HOST array [n_m_tiles] (n_m_tiles <= 1024).  One record of 6 ints per (unit, CTA rank):
 *   unit, rank, group, m_tile, n_tile, role | mma << 4     (role: 0 idle, 1 active, 2 zero-fill).
 * Returns the number of records (at most `cap` are written), or a negative spt_status. */
int spt_grouped_gemm_plan(const int32_t *tile_group, int n_m_tiles, int tiles_n, int32_t *out, int cap);

/* Gated unit of the plain RoutedLLaMaFFN: h = silu(gate) * side (layers/sparse/feedforward.py:172-176 with the LLaMA
 * activation), 16-bit in / out with fp32 math, and its backward (both gradients in one pass).  n elements, multiple of 8,
 * 16-byte aligned.  _ex: every operand is of `dtype` (SPT_BF16 or SPT_F16); the plain names are bf16. */
int spt_silu_mul_fwd(const void *gate, const void *side, void *h, int64_t n, spt_stream_t stream);
int spt_silu_mul_bwd(const void *gate, const void *side, const void *grad_h, void *grad_gate, void *grad_side, int64_t n,
                     spt_stream_t stream);
int spt_silu_mul_fwd_ex(const void *gate, const void *side, void *h, int64_t n, int dtype, spt_stream_t stream);
int spt_silu_mul_bwd_ex(const void *gate, const void *side, const void *grad_h, void *grad_gate, void *grad_side,
                        int64_t n, int dtype, spt_stream_t stream);

/* Fused elementwise stages of the LoRA-routed FFN (naive_gpt/layers/tuning/lora_ffn.py:87-115,201-222).
 * coeff [R] fp32 = 2 * router probability of the bucket row.  C % 4 == 0.
 *   scale_add: out = coeff[r] * a + b;   bwd: da = coeff[r] * dout (a's dtype), dcoeff[r] = sum_c dout * a.
 *              a, b, out (and dout) are each SPT_F32 or one 16-bit type, SPT_BF16 or SPT_F16.
 *   lora_glu : h = silu(coeff*bg + lg) * (coeff*bs + ls), all inputs fp32 [R, C];
 *              bwd: gradients of the four inputs (fp32) and dcoeff[r].  h and grad_h are bf16 in the plain
 *              names; the _ex names take their type (h_dtype / dh_dtype: SPT_BF16 or SPT_F16). */
int spt_scale_add_fwd(const float *coeff, const void *a, int a_dtype, const void *b, int b_dtype, void *out,
                      int o_dtype, int64_t R, int C, spt_stream_t stream);
int spt_scale_add_bwd(const float *coeff, const void *a, int a_dtype, const void *dout, int g_dtype, void *da,
                      float *dcoeff, int64_t R, int C, spt_stream_t stream);
int spt_lora_glu_fwd(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                     void *h, int64_t R, int C, spt_stream_t stream);
int spt_lora_glu_bwd(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                     const void *dh, float *d_bg, float *d_lg, float *d_bs, float *d_ls, float *dcoeff,
                     int64_t R, int C, spt_stream_t stream);
int spt_lora_glu_fwd_ex(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                        void *h, int64_t R, int C, int h_dtype, spt_stream_t stream);
int spt_lora_glu_bwd_ex(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                        const void *dh, float *d_bg, float *d_lg, float *d_bs, float *d_ls, float *dcoeff,
                        int64_t R, int C, int dh_dtype, spt_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPT_B200_H */

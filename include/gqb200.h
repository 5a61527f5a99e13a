/*
 * gqb200.h -- C ABI of libgqb200.so, the B200 (sm_100a) implementation of the
 * gradient-compression hot path of xinyandai/gradient-quantization.
 *
 * Boundary rules
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every pointer marked "device" is a CUDA device pointer on the current
 *     device; "host" pointers are ordinary (preferably pinned) host memory.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*)
 *     unless it says otherwise; no call allocates device memory: the caller
 *     supplies outputs and the workspace (size from gq_*_workspace_bytes).
 *   - return value: 0 = GQ_OK, otherwise a GQ_ERR_* code; gq_last_error()
 *     returns a thread-local, human-readable message for the last failure.
 *   - there is no CPU fallback: without a usable sm_100 device the calls fail
 *     with GQ_ERR_CUDA.
 *
 * Each entry point cites the reference interface it replaces (file:line,
 * relative to the reference checkout).  The Python classes of the same names as
 * the reference's (gradient-quantization_b200/compressors, quantizers) are thin
 * ctypes callers of these functions; INTEGRATION.md shows the binding.
 *
 * Data layout ("packed record", one per simulated user / rank)
 *   chunk matrix : fp32 [n_chunks, d] row-major = the gradient tensors of one
 *                  codec group laid end to end (every tensor a multiple of d).
 *   seg_start    : int64 [n_seg + 1], chunk index where tensor s starts;
 *                  seg_start[n_seg] == n_chunks.  Per-tensor quantities
 *                  (lb/ub of the norm quantizer) are indexed by s.
 *   codes        : uint8 [n_chunks] (K <= 256) or int32 [n_chunks]
 *   l            : uint8 [n_chunks] (wire) or int32 [n_chunks] (reference dtype)
 *   lbub         : fp32 [2 * n_seg] = (lb_0, ub_0, lb_1, ub_1, ...)
 */
#ifndef GQB200_H
#define GQB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GQ_OK 0
#define GQ_ERR_INVALID 1     /* bad argument (message says which)            */
#define GQ_ERR_CUDA 2        /* CUDA runtime/driver error, or no sm_100 GPU   */
#define GQ_ERR_UNSUPPORTED 3 /* valid request this build has no kernel for    */
#define GQ_ERR_WORKSPACE 4   /* workspace too small                           */

/* HSQ search algorithm selector */
#define GQ_ALGO_AUTO 0   /* tcgen05 path when (d, K) allow it, else exact CUDA-core */
#define GQ_ALGO_EXACT 1  /* fp32 CUDA-core search (any d <= 128, any K)             */
#define GQ_ALGO_TC 2     /* tcgen05 TF32 search + fp32 rescoring (d == 16, K == 256) */

typedef void *gq_stream_t; /* cudaStream_t */

const char *gq_last_error(void);
int gq_abi_version(void);
/* device facts used by the host code to size grids/workspaces; synchronous. */
int gq_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);

/* ------------------------------------------------------------------------- */
/* HSQ encode: nearest-codeword search + n-bit norm quantization.
 * Replaces NearestNeighborCompressor.compress
 *   (compressors/nearest_neighbor_compressor.py:63-78) and the
 *   ProbabilisticScalarCompressor.compress it calls
 *   (compressors/probabilistic_scalar_compressor.py:12-27), for a whole group
 *   of tensors in one call (the per-parameter loop of
 *   quantizers/ps_quantizer.py:33-44).
 *
 * grad      device fp32 [n_chunks*d]   chunk matrix (16-byte aligned)
 * codebook  device fp32 [K*d]          unit-norm rows, row-major
 * seg_start device int64 [n_seg+1]
 * n_bit     norm bits; 32 = keep fp32 norms (u_out is then the result, l/lbub untouched)
 * random    0: truncate, 1: stochastic rounding (l += (frac > r))
 * uniforms  device fp32 [n_chunks] of U[0,1) draws indexed by chunk, or NULL to
 *           use the built-in Philox4x32-10 stream (philox_seed, philox_offset + chunk)
 * codes     device out, code_bytes in {1, 4}  (1 requires K <= 256)
 * l         device out, l_bytes in {1, 4}     (values 0..2^n_bit; 1 requires n_bit <= 7)
 * lbub      device out fp32 [2*n_seg]
 * u_out     device out fp32 [n_chunks]: signed projection of every chunk
 * bit-exactness: codes, u, lb/ub and (given the same uniforms) l equal the
 * reference's CPU result bit for bit (sequential ascending-j fp32 FMA chain,
 * first index wins ties).
 */
size_t gq_hsq_encode_workspace_bytes(int64_t n_chunks, int d, int K, int n_seg);
int gq_hsq_encode(const float *grad, int64_t n_chunks, int d,
                  const float *codebook, int K,
                  const int64_t *seg_start, int n_seg,
                  int n_bit, int random, const float *uniforms,
                  uint64_t philox_seed, uint64_t philox_offset,
                  void *codes, int code_bytes, void *l, int l_bytes,
                  float *lbub, float *u_out,
                  void *workspace, size_t workspace_bytes, int algo, gq_stream_t stream);

/* The two halves of gq_hsq_encode, exposed because the reference exposes them
 * as separate classes (ResidualCompressor / PVC reuse the norm quantizer). */
int gq_hsq_search(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                  void *codes, int code_bytes, float *u_out,
                  const int64_t *seg_start, int n_seg, uint32_t *minmax_keys /* [2*n_seg] or NULL */,
                  void *workspace, size_t workspace_bytes, int algo, gq_stream_t stream);

/* ProbabilisticScalarCompressor.compress (probabilistic_scalar_compressor.py:12-27)
 * over every segment of u: per-segment lb/ub, then l.  minmax_keys is scratch
 * [2*n_seg] uint32 (filled here when precomputed == 0). */
int gq_norm_quantize(const float *u, int64_t n, const int64_t *seg_start, int n_seg,
                     int n_bit, int random, const float *uniforms,
                     uint64_t philox_seed, uint64_t philox_offset,
                     void *l, int l_bytes, float *lbub,
                     uint32_t *minmax_keys, int precomputed, gq_stream_t stream);

/* ProbabilisticScalarCompressor.decompress (probabilistic_scalar_compressor.py:29-33):
 * out[i] = l[i] * (ub - lb) / 2^n_bit + lb. */
int gq_norm_dequantize(const void *l, int l_bytes, int64_t n, const int64_t *seg_start, int n_seg,
                       int n_bit, const float *lbub, float *out, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* HSQ decode-and-reduce over users.
 * Replaces NearestNeighborCompressor.decompress
 *   (compressors/nearest_neighbor_compressor.py:80-90) +
 *   ProbabilisticScalarCompressor.decompress (probabilistic_scalar_compressor.py:29-33)
 *   for U users and the stack(...).mean(0) of PSQuantizer.apply
 *   (quantizers/ps_quantizer.py:48), or the `grad += previous` of
 *   RingQuantizer.record (quantizers/ring_quantizer.py:31-32).
 *
 * User u's arrays live at codes + u*user_stride_bytes, l + u*user_stride_bytes,
 * (char*)lbub + u*user_stride_bytes (the all-gathered packed records); when
 * n_bit == 32, `l` is unused and norms_f32 (+ u*user_stride_bytes) holds fp32 norms.
 *   r[i]   = sum_{u=0..U-1} codebook[code_u[c], j] * norm_u[c]   (user order)
 *   mean   : r /= U                 (true division)
 *   out[i] = r[i] (accumulate 0), out[i] + r[i] (1), out[i] - r[i] (2: error feedback,
 *            error = grad - decompress(compress(grad)), ps_quantizer.py:39)
 */
int gq_hsq_decode_reduce(const void *codes, int code_bytes, const void *l, int l_bytes,
                         const float *lbub, const float *norms_f32,
                         int64_t user_stride_bytes, int n_users,
                         int64_t n_chunks, int d, const float *codebook, int K,
                         const int64_t *seg_start, int n_seg, int n_bit,
                         int mean, int accumulate, float *out, gq_stream_t stream);

/* Same reduction, but user u's arrays are found at (pointer of user 0) + user_byte_offsets[u]
 * (host array, n_users <= 8, offsets may be any 64-bit distance): the packed records need not be
 * equally spaced -- with peer-to-peer exchange each user's record lives in another GPU's memory
 * (mapped with gq_ipc_open) and is read over NVLink by the decode kernel itself.
 * Chunk dims 4, 8, 16 with a codebook of at most 64 KB; quantized norms only. */
/* One user's encode and decode with the norm quantization moved from the encode into the decode
 * (HSQ d = 16, K = 256, uint8 codes and levels, n_bit 1..7, n_seg <= 1024; tcgen05 search).  The
 * quantization needs every tensor's final min/max, i.e. a grid-wide point after the search; the
 * boundary between the two kernels provides it without a barrier inside the encode.
 * gq_hsq_encode_search: gq_hsq_encode without the norm quantization -- writes codes and u_out and
 *   leaves the per-tensor min/max keys in the workspace (its first 2*n_seg uint32 words); l and lbub
 *   are not written.  Carries a pending gq_attach_f32_reduce like gq_hsq_encode.
 * gq_hsq_decode_quantize: the rest of that encode fused into gq_hsq_decode_reduce with n_users = 1:
 *   reads u and the keys (minmax_keys = that workspace), writes l and lbub into the record -- the same
 *   bytes gq_hsq_encode writes for the same Philox range or uniforms -- and decodes the record into
 *   out (accumulate 0, 1, 2 as in gq_hsq_decode_reduce).  Pointers 16-byte aligned.
 * A record that must be complete without being decoded: gq_norm_quantize(u_out, ..., minmax_keys =
 * the workspace, precomputed = 1) gives the same l and lbub. */
int gq_hsq_encode_search(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                         const int64_t *seg_start, int n_seg, void *codes, int code_bytes, float *u_out,
                         void *workspace, size_t workspace_bytes, gq_stream_t stream);
int gq_hsq_decode_quantize(const void *codes, void *l, float *lbub, const float *u, const uint32_t *minmax_keys,
                           int64_t n_chunks, int d, const float *codebook, int K, const int64_t *seg_start,
                           int n_seg, int n_bit, int random, const float *uniforms, uint64_t philox_seed,
                           uint64_t philox_offset, int accumulate, float *out, gq_stream_t stream);

int gq_hsq_decode_reduce_scattered(const void *codes, int code_bytes, const void *l, int l_bytes,
                                   const float *lbub, const int64_t *user_byte_offsets, int n_users,
                                   int64_t n_chunks, int d, const float *codebook, int K,
                                   const int64_t *seg_start, int n_seg, int n_bit, int mean, int accumulate,
                                   float *out, gq_stream_t stream);
int gq_f32_reduce_users_scattered(const float *in, const int64_t *user_byte_offsets, int n_users, int64_t n,
                                  int mean, int accumulate, float *out, gq_stream_t stream);

/* Attach a small gq_f32_reduce_users[_scattered] job (the identity tensors of a model: n_users = 1
 * copy at encode time, sum / mean over users at decode time) to the NEXT gq_hsq_encode,
 * gq_hsq_decode_reduce, gq_hsq_decode_reduce_scattered, gq_qsgd_encode, gq_qsgd_decode_reduce,
 * gq_sign_encode[_t5], gq_sign_decode_reduce[_t5], gq_topk_select or gq_topk_scatter_reduce call made by
 * this host thread: it runs
 * inside that call's first kernel (or, if that code path cannot carry it, in a launch of its own
 * issued by that call) instead of costing a separate ~3 us launch.  Same arguments and results as
 * gq_f32_reduce_users (user_byte_offsets == NULL: user u at in + u * user_stride_bytes) /
 * gq_f32_reduce_users_scattered.  n_users <= 8.  The job is dropped if no such call follows. */
int gq_attach_f32_reduce(const float *in, int64_t user_stride_bytes, const int64_t *user_byte_offsets,
                         int n_users, int64_t n, int mean, int accumulate, float *out);

/* out[i] = (sum_u in[u*user_stride_bytes + 4*i]) / U (mean) -- identity tensors
 * (compressors/identical_compressor.py:5-11 under ps_quantizer.py:48). */
int gq_f32_reduce_users(const float *in, int64_t user_stride_bytes, int n_users, int64_t n,
                        int mean, int accumulate, float *out, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* QSGD / TernGrad.  Replaces QSGDCompressor.compress / decompress
 *   (compressors/qsgd_compressor.py:42-64, 66-71).
 * grad fp32 [n_chunks*dim]; norm out fp32 [n_chunks] (L-inf per chunk).
 * unpacked outputs (reference dtypes): signs uint8 [n] (0/1), l int32 [n]
 *   (an all-zero chunk yields INT32_MIN like the reference's NaN cast).
 * packed output (wire): bits_per_elem in {4, 8, 16}: (sign << (bits-1)) | l.
 * Either `packed` or both `signs` and `l` may be NULL.
 * uniforms: device fp32 [n] or NULL for Philox. */
int gq_qsgd_wire_bits(int n_bit);
/* n = total elements.  Chunks are either uniform (chunk_start == NULL,
 * n == n_chunks*dim) or variable (chunk_start int64 [n_chunks+1] on the device,
 * e.g. one chunk per tensor for TernGrad's c_dim == 0; dim ignored). */
int gq_qsgd_encode(const float *grad, int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim,
                   int n_bit, int random, const float *uniforms, uint64_t philox_seed,
                   uint64_t philox_offset, float *norm, uint8_t *signs, int32_t *l, void *packed,
                   gq_stream_t stream);
/* decode-and-reduce over users from the packed wire format
 * (qsgd_compressor.py:66-71 + ps_quantizer.py:48 / ring_quantizer.py:31-32);
 * user u's norm / packed arrays are at + u*user_stride_bytes. */
int gq_qsgd_decode_reduce(const float *norm, const void *packed, int64_t user_stride_bytes, int n_users,
                          int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit,
                          int mean, int accumulate, float *out, gq_stream_t stream);
/* decode one user from the unpacked (reference-dtype) signature */
int gq_qsgd_decode_unpacked(const float *norm, const uint8_t *signs, const int32_t *l, int64_t n,
                            const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit, float *out,
                            gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* SignSGD.  Replaces SignSGDCompressor.compress (compressors/signsgd_compressor.py:8-9).
 * out_f32 (reference dtype, {-1,0,+1}) and/or packed (2 bits/elem, 4 per byte:
 * 0 -> 0, 1 -> +1, 2 -> -1; n rounded up to a multiple of 4). */
int gq_sign_encode(const float *grad, int64_t n, float *out_f32, uint8_t *packed, gq_stream_t stream);
int gq_sign_decode_reduce(const uint8_t *packed, int64_t user_stride_bytes, int n_users, int64_t n,
                          int mean, int accumulate, float *out, gq_stream_t stream);

/* The same codec on the denser base-3 wire (SURVEY 8f-4 "ternary sign 5-per-byte"): five elements per
 * byte, byte = t0 + 3 t1 + 9 t2 + 27 t3 + 81 t4 with the digit code of the 2-bit form (0 -> 0, 1 -> +1,
 * 2 -> -1); 20 elements per little-endian 32-bit word, gq_sign_t5_bytes(n) = 4 * ceil(n / 20) bytes per
 * section (elements past n encode as 0).  Decoded values are those of gq_sign_decode_reduce, bit for bit
 * (compressors/signsgd_compressor.py:8-12 fixes only the values, not the container). */
int64_t gq_sign_t5_bytes(int64_t n);
int gq_sign_encode_t5(const float *grad, int64_t n, void *packed, gq_stream_t stream);
int gq_sign_decode_reduce_t5(const void *packed, int64_t user_stride_bytes, int n_users, int64_t n,
                             int mean, int accumulate, float *out, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Top-k sparsification.  Replaces TopKSparsificationCompressor.compress
 *   (compressors/topk_sparsification_compressor.py:18-23): per tensor
 *   (segment) keep the k_s largest |v| (ties at the cut: lowest index first),
 *   zero the rest.
 * seg_start int64 [n_seg+1] in ELEMENTS; k int64 [n_seg] (both device).
 * out_dense (reference form, vec*mask incl. signed zeros) may be NULL;
 * out_idx int32 [sum k] / out_val fp32 [sum k] (wire form, ascending index
 * inside each segment, segment s at offset k_prefix[s]) may be NULL. */
size_t gq_topk_workspace_bytes(int64_t n, int n_seg);
int gq_topk_select(const float *grad, int64_t n, const int64_t *seg_start, const int64_t *k,
                   const int64_t *k_prefix, int n_seg, float *out_dense, int32_t *out_idx,
                   float *out_val, void *workspace, size_t workspace_bytes, gq_stream_t stream);
/* out = [accumulate? out : 0] + sum over users (user order) of the sparse entries, / U if mean.
 * idx are GLOBAL element indices (seg_start[s] + local index). */
int gq_topk_scatter_reduce(const int32_t *idx, const float *val, int64_t user_stride_bytes,
                           int n_users, int64_t k_total, int64_t n, int mean, int accumulate,
                           float *out, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Probabilistic vector compressor search (INTENDED semantics of
 *   compressors/probabilistic_vector_compressor.py:42-65; the shipped class does
 *   not run -- DESIGN.md "PVC").  dagger = pinv(C^T) fp32 [K*d] row-major.
 *   code = first k with cumsum(|p|/l1)_k >= r - 1e-5 ; u = sign(p_code) * l1.
 * uniforms: device fp32 [n_chunks] or NULL for Philox. */
int gq_pvc_search(const float *grad, int64_t n_chunks, int d, const float *dagger, int K,
                  const float *uniforms, uint64_t philox_seed, uint64_t philox_offset,
                  void *codes, int code_bytes, float *u_out, gq_stream_t stream);

/* Diagnostic hook for the tcgen05 path (d == 16, K == 256): runs the search and
 * also dumps the raw TF32 tensor-core scores of the first dbg_tiles 128-chunk
 * tiles (fp32 [dbg_tiles*128, 256], device) so tests can measure the
 * approximation error that the fp32 rescoring margin has to cover. */
int gq_hsq_tc_debug(const float *grad, int64_t n_chunks, const float *codebook, void *codes,
                    float *u_out, const int64_t *seg_start, int n_seg, float *dbg_scores,
                    int dbg_tiles, gq_stream_t stream);

/* Multi-tensor gather: copy n_tensors fp32 tensors (src_ptrs: HOST array of device pointers,
 * sizes in elements) to dst + dst_offsets[t] (elements) -- how the per-parameter gradients of
 * main.py:229-230 (param.grad after loss.backward()) reach the codec arena that
 * PSQuantizer.record / RingQuantizer.record (quantizers/ps_quantizer.py:33-44) encode from.
 * One launch per 128 tensors; the pointer table travels as a kernel parameter.
 * feedback = 1: dst holds the user's error state e and becomes src + scale * e
 *   (`grad += scale * error`, ps_quantizer.py:35 / ring_quantizer.py:34, same two roundings);
 * feedback = 2: that sum is also written back to the source tensors (the reference mutates
 *   param.grad in place).  The decode entry points' accumulate = 2 (out = out - decoded) then turn
 *   the same buffer into the new error (ps_quantizer.py:39) without another sweep. */
int gq_gather_f32(const void *const *src_ptrs, const int64_t *dst_offsets, const int64_t *sizes,
                  int n_tensors, float *dst, int feedback, float scale, gq_stream_t stream);

/* Diagnostic hook for the second-generation tcgen05 kernel: search only (l == NULL) or the whole
 * one-launch encode (6-bit norms, Philox), and CTA 0 time-stamps the pipeline events of its first 128
 * tiles into trace (device int64 [16 * 128], clock64 values; event list in hsq_tc2.cu), followed by
 * four wall-clock stamps (ns) per CTA: start, main loop done, grid barrier passed, tail done
 * (trace needs 16 * 128 + 4 * SM-count entries).  How tests/tc2_trace.py measures where the time goes. */
int gq_hsq_tc2_trace(const float *grad, int64_t n_chunks, const float *codebook, void *codes,
                     float *u_out, const int64_t *seg_start, int n_seg, void *l, float *lbub,
                     void *workspace, int64_t *trace, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Peer-to-peer exchange of packed records (one user per GPU on one NVLink/NVSwitch node).
 * Replaces the exchange step of PSQuantizer (quantizers/ps_quantizer.py:44-48, a Python list
 * append in the reference; an NCCL all-gather in the plain distributed path).
 * gq_ipc_alloc: cudaMalloc + zero a buffer and return its 64-byte CUDA IPC handle (ship it to the
 *   other ranks, e.g. torch.distributed.all_gather_object).  gq_ipc_open maps a peer's buffer.
 * gq_peer_barrier: on `stream`, announce `epoch` in every rank's flag array (system-scope release
 *   store) and wait until every rank announced it here.  flag_ptrs is a HOST array of n_ranks
 *   device addresses (uint32[8] each; flag_ptrs[rank] is the local array), epochs increase by 1.
 *   Traps (sticky CUDA error) instead of hanging if a peer never arrives. */
int gq_ipc_alloc(size_t bytes, void **dev_ptr, void *handle_out_64);
int gq_ipc_free(void *dev_ptr);
int gq_ipc_open(const void *handle_64, void **peer_ptr);
int gq_ipc_close(void *peer_ptr);
int gq_peer_barrier(void *const *flag_ptrs, int rank, int n_ranks, uint32_t epoch, gq_stream_t stream);
/* After the barrier: pull n_ranks records of `bytes` each (multiple of 16) from src_ptrs[r] (HOST
 * array of device addresses, peer-mapped or local) into dst + r*dst_stride with wide loads. */
int gq_peer_gather(void *dst, void *const *src_ptrs, size_t bytes, size_t dst_stride, int n_ranks,
                   gq_stream_t stream);

/* Push variant of the same exchange: before gq_peer_barrier, copy the local record (`bytes`, a
 * multiple of 16) into each of the n_dst (<= 8) peer-mapped addresses of the HOST array dst_ptrs.
 * Remote stores are posted, so this is cheaper than pulling; the barrier that follows on the same
 * stream publishes the data (system-scope release).  Replaces the NCCL all-gather of
 * quantizers/ps_quantizer.py's exchange, like gq_peer_gather. */
int gq_peer_push(const void *src, void *const *dst_ptrs, size_t bytes, int n_dst, gq_stream_t stream);

/* The same push through an NVSwitch multicast (NVLS) mapping of the ranks' symmetric buffers:
 * mc_dst = multicast address of the destination row (identical offset in every rank's buffer).
 * One multimem.st per 16 bytes is replicated by the switch to every rank (the sender included). */
int gq_peer_push_multicast(const void *src, void *mc_dst, size_t bytes, gq_stream_t stream);

/* Exchange fused into the codec kernels (default for HSQ d=16 K=256 on one NVSwitch node).
 * Sending side: the next gq_hsq_encode on this host thread also stores every finished section of
 * the record at (local address + delta[i]), i < n_remote -- the same record row in the peers'
 * receive blocks -- or once through an NVLS multicast mapping (multicast = 1, n_remote = 1),
 * mirrors the identity section [ident, ident + ident_bytes), and when the whole record is out stores
 * `epoch` (system-scope release) into flag_ptrs[0..n_flags): this rank's word in every rank's flag
 * array.  Receiving side: the next HSQ decode first waits until n_ranks words of local_flags have
 * reached `epoch`.  Together they replace gq_peer_push* + gq_peer_barrier (two launches per step)
 * of the exchange step of PSQuantizer (quantizers/ps_quantizer.py:44-48). */
int gq_attach_remote_record(int n_remote, int multicast, const int64_t *delta, const void *ident,
                            int64_t ident_bytes, void *const *flag_ptrs, int n_flags, uint32_t epoch);
int gq_attach_peer_wait(const void *local_flags, int n_ranks, uint32_t epoch);

/* ------------------------------------------------------------------------- */
/* Elementwise helpers the quantizers need around the codecs.
 * out = a + alpha*b  (ps_quantizer.py:35 error feedback; ring_quantizer.py:32)
 * out = a - b        (ps_quantizer.py:39; residual_compressor.py:21) */
int gq_axpy(const float *a, const float *b, float alpha, int64_t n, float *out, gq_stream_t stream);
int gq_sub(const float *a, const float *b, int64_t n, float *out, gq_stream_t stream);

/* ------------------------------------------------------------------------- */
/* Host-buffer convenience entry (the end-to-end form: host fp32 gradient in,
 * host fp32 decoded gradient out; H2D/D2H inside).  Encodes one user's chunk
 * matrix with HSQ and decodes it again (ps_quantizer.py:36-43 for one user).
 * Synchronous.  dev_scratch is a device buffer of gq_hsq_host_scratch_bytes(). */
size_t gq_hsq_host_scratch_bytes(int64_t n_chunks, int d, int K, int n_seg);
int gq_hsq_roundtrip_host(const float *host_grad, float *host_out, int64_t n_chunks, int d,
                          const float *dev_codebook, int K, const int64_t *dev_seg_start, int n_seg,
                          int n_bit, int random, uint64_t philox_seed, uint64_t philox_offset,
                          void *dev_scratch, size_t scratch_bytes, int algo, gq_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GQB200_H */

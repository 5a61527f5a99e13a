// gq_internal.cuh -- declarations shared between the translation units of libgqb200.
#pragma once
#include "gq_common.cuh"

namespace gq {

// hsq_exact.cu
int launch_minmax_init(uint32_t *keys, int n_seg, cudaStream_t st, uint32_t *barrier = nullptr);

// A small fp32 user-reduction (the identity tensors of a model: copy at encode time, sum / mean
// over users at decode time) that rides inside the first kernel of the next HSQ encode or decode
// call instead of paying a launch of its own (gq_attach_f32_reduce).  n == 0: none.
struct Rider {
    const float *in;
    int64_t off[8];      // byte offset of user u's data from `in`
    int n_users;
    int64_t n;
    int mean, accumulate;
    float *out;
};
// thread-local pending rider of the calling host thread (n == 0 when none); take_rider() clears it
Rider take_rider();
void set_rider(const Rider &r);
int launch_rider(const Rider &r, cudaStream_t st);   // stand-alone launch (no carrier available)
__device__ __forceinline__ void rider_run(const Rider &r, int64_t tid, int64_t nthreads)
{
    for (int64_t i = tid; i < r.n; i += nthreads) {
        float acc = 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (u < r.n_users) {
                const float x = *reinterpret_cast<const float *>(reinterpret_cast<const char *>(r.in) + r.off[u] + 4 * i);
                acc = (u == 0) ? x : __fadd_rn(acc, x);
            }
        }
        if (r.mean) acc = __fdiv_rn(acc, (float)r.n_users);
        if (r.accumulate) acc = (r.accumulate == 2) ? __fsub_rn(r.out[i], acc) : __fadd_rn(r.out[i], acc);
        r.out[i] = acc;
    }
}
int launch_minmax_init_rider(uint32_t *keys, int n_seg, cudaStream_t st, uint32_t *barrier, const Rider &rider);
int hsq_search_exact(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                     void *codes, int code_bytes, float *u_out, const int64_t *seg_start, int n_seg,
                     uint32_t *minmax_keys, cudaStream_t st);

// hsq_tc.cu (tcgen05 path; d == 16, K == 256)
bool hsq_tc_supported(int d, int K, int code_bytes);
size_t hsq_tc_workspace_bytes(int64_t n_chunks);
int hsq_search_tc(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                  void *codes, int code_bytes, float *u_out, const int64_t *seg_start, int n_seg,
                  uint32_t *minmax_keys, void *workspace, size_t workspace_bytes, cudaStream_t st);

// same, and the kernel itself resets the min/max keys (flag: 8-byte scratch word in the workspace)
// and runs `rider`: an encode without a separate init launch
int hsq_search_tc_prepared(const float *grad, int64_t n_chunks, const float *codebook, void *codes, float *u_out,
                           const int64_t *seg_start, int n_seg, uint32_t *minmax_keys, uint64_t *flag,
                           const Rider &rider, cudaStream_t st);

// hsq_tc.cu: search + grid barrier + n-bit norm quantization in ONE persistent kernel
// (keys must have been initialised and *barrier zeroed by launch_minmax_init before)
int hsq_encode_tc_fused(const float *grad, int64_t n_chunks, const float *codebook, void *codes, float *u_out,
                        const int64_t *seg_start, int n_seg, uint32_t *minmax_keys, uint32_t *barrier,
                        int n_bit, int random, const float *uniforms, uint64_t seed, uint64_t offset,
                        uint8_t *l, float *lbub, cudaStream_t st);

// hsq_tck.cu: tcgen05 search for large codebooks (d == 16, K = 512..4096, int32 codes)
bool hsq_tck_supported(int d, int K, int code_bytes);
size_t hsq_tck_workspace_bytes(int d, int K);
int hsq_search_tck(const float *grad, int64_t n_chunks, const float *codebook, int K, void *codes, float *u_out,
                   const int64_t *seg_start, int n_seg, uint32_t *minmax_keys, void *workspace, size_t workspace_bytes,
                   cudaStream_t st);

int tc_generation();   // abi.cu: 1 = hsq_tc.cu + separate quantize launch, 2 (default) = hsq_tc2.cu

// hsq_tc2.cu: second-generation tcgen05 encode (d in {8, 16, 32}, K == 256, uint8 codes).  One launch does the
// key reset, the identity rider, the search and -- when `tail` is given -- the norm quantization
// behind a grid barrier; with `remote` it also stores every finished record section into the
// peers' receive blocks (or once through an NVLS multicast mapping) and announces the step epoch.
struct Tc2Tail {
    uint8_t *l;
    float *lbub;
    const float *uniforms;
    uint64_t seed, offset;
    int n_bit, random;
};
struct Tc2Remote {
    int n;                  // remote destinations (0 = none); with multicast: 1
    int multicast;
    int64_t delta[7];       // remote address = local record address + delta[i]
    const uint8_t *ident;   // identity section inside the local record (mirrored too), may be null
    int64_t ident_bytes;
    uint32_t *flag[8];      // words that receive `epoch` (st.release.sys) when the record is delivered
    int n_flag;
    uint32_t epoch;
};
bool hsq_tc2_tail_supported(int n_seg, int n_bit, int l_bytes, const void *u_out, const void *uniforms, const void *l,
                            const void *codes);
bool hsq_tc2_supported(int d, int K, int code_bytes);   // d in {8, 16, 32}, K == 256, uint8 codes
int hsq_encode_tc2(const float *grad, int64_t n_chunks, int d, const float *codebook, void *codes, float *u_out,
                   const int64_t *seg_start, int n_seg, uint32_t *keys, uint64_t *flag, uint32_t *barrier,
                   const Rider &rider, const Tc2Tail *tail, const Tc2Remote *remote, cudaStream_t st);
int hsq_tc2_trace(const float *grad, int64_t n_chunks, const float *codebook, void *codes, float *u_out,
                  const int64_t *seg_start, int n_seg, uint32_t *keys, uint64_t *flag, uint32_t *barrier,
                  const Tc2Tail *tail, long long *trace, cudaStream_t st);
// thread-local pending remote delivery of the calling host thread, consumed by the next gq_hsq_encode
Tc2Remote take_remote();
void set_remote(const Tc2Remote &r);

// Wait (inside the next decode kernel, or a one-warp kernel of its own) until every rank has
// announced `epoch` in this rank's flag array: the receiving side of the fused peer-to-peer push.
struct PeerWait {
    const uint32_t *flags;   // local flag array, flags[r] = last epoch rank r has delivered
    int n;                   // ranks (0: nothing to wait for)
    uint32_t epoch;
    unsigned long long timeout_ns;
};
void set_wait(const PeerWait &w);
PeerWait take_wait();
int flush_wait(cudaStream_t st);
// bounded by wall clock (not by a poll count): rank skew of seconds is normal in training (evaluation
// or a checkpoint on one rank), minutes are not; on timeout the kernel traps (sticky error on this rank)
__device__ __forceinline__ void peer_wait_flag(const uint32_t *flag, uint32_t epoch, unsigned long long timeout_ns)
{
    unsigned long long t0 = 0ull;
    for (;;) {
        uint32_t seen;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(flag) : "memory");
        if ((int32_t)(seen - epoch) >= 0) return;
        __nanosleep(64);
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0ull) t0 = now;
        else if (now - t0 > timeout_ns) __trap();
    }
}
unsigned long long peer_timeout_ns();   // p2p.cu
#define GQ_CUDA_INT(expr) do { int _e2 = (expr); if (_e2) return _e2; } while (0)

// hsq_tail.cu
int launch_seg_minmax(const float *u, int64_t n, const int64_t *seg_start, int n_seg, uint32_t *keys,
                      cudaStream_t st);
int launch_norm_quantize(const float *u, int64_t n, const int64_t *seg_start, int n_seg, int n_bit,
                         int random, const float *uniforms, uint64_t seed, uint64_t offset, void *l,
                         int l_bytes, float *lbub, const uint32_t *keys, cudaStream_t st);
int launch_norm_dequantize(const void *l, int l_bytes, int64_t n, const int64_t *seg_start, int n_seg,
                           int n_bit, const float *lbub, float *out, cudaStream_t st);
// byte offsets of each user's arrays relative to user 0's pointers (packed records need not be
// equally spaced: with peer-to-peer exchange every user's record lives in a different GPU's memory)
struct UserOffsets {
    int64_t off[8];
};
int hsq_decode_reduce(const void *codes, int code_bytes, const void *l, int l_bytes, const float *lbub,
                      const float *norms_f32, int64_t user_stride, const int64_t *user_offsets, int n_users,
                      int64_t n_chunks, int d,
                      const float *codebook, int K, const int64_t *seg_start, int n_seg, int n_bit,
                      int mean, int accumulate, float *out, cudaStream_t st);
// one user's record whose levels the decode computes itself (d = 16, K = 256, uint8 codes and levels):
// the norm quantization of the search that left u and the min/max keys behind, then the decode
int hsq_decode_quantize(const void *codes, void *l, float *lbub, const float *u, const uint32_t *keys,
                        int64_t n_chunks, const float *codebook, const int64_t *seg_start, int n_seg, int n_bit,
                        int random, const float *uniforms, uint64_t seed, uint64_t offset, int accumulate,
                        float *out, cudaStream_t st);
int launch_f32_reduce_users(const float *in, int64_t user_stride, const int64_t *user_offsets, int n_users,
                            int64_t n, int mean, int accumulate, float *out, cudaStream_t st);
int launch_axpy(const float *a, const float *b, float alpha, int64_t n, float *out, int sub,
                cudaStream_t st);

// Per-chunk epilogue shared by all search kernels: store code and u, fold u into
// the per-tensor min/max keys (lb/ub of the norm quantizer).
template <typename CodeT>
__device__ __forceinline__ void search_epilogue(bool valid, int64_t c, int best_k, float best_u,
                                                CodeT *__restrict__ codes, float *__restrict__ u_out,
                                                const int64_t *__restrict__ seg_start, int n_seg,
                                                uint32_t *__restrict__ minmax_keys, SegCache &segc)
{
    if (valid) {
        codes[c] = (CodeT)best_k;
        u_out[c] = best_u;
    }
    if (minmax_keys == nullptr) return;
    int seg = valid ? cached_segment(segc, seg_start, n_seg, c) : -1;
    // warp-uniform fast path: every valid lane in the same tensor
    int seg0 = __shfl_sync(0xffffffffu, seg, 0);
    bool uniform = __all_sync(0xffffffffu, (seg == seg0) || !valid) && (seg0 >= 0);
    if (valid && best_u != best_u) atomicMax(minmax_keys + 2 * seg + 1, GQ_KEY_NAN);   // NaN propagates (see minmax_add_warp)
    if (uniform) {
        float mn = warp_min(valid ? best_u : INFINITY);
        float mx = warp_max(valid ? best_u : -INFINITY);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(minmax_keys + 2 * seg0, float_to_key(mn));
            atomicMax(minmax_keys + 2 * seg0 + 1, float_to_key(mx));
        }
    } else if (valid) {
        atomicMin(minmax_keys + 2 * seg, float_to_key(best_u));
        atomicMax(minmax_keys + 2 * seg + 1, float_to_key(best_u));
    }
}


// n-bit norm quantization of u[i_begin, i_end) by `nthreads` cooperating threads (thread `tid`):
// four consecutive chunks per thread and iteration (float4 of u, one Philox block, one packed
// store).  i_begin must be a multiple of 4.  keys hold the per-tensor min/max (ordered-uint form).
// Shared by norm_quantize_kernel and the fused tail of the tcgen05 search kernel.
template <typename LT, bool VOLATILE_KEYS>
__device__ __forceinline__ void quantize_range(const float *__restrict__ u, int64_t i_begin, int64_t i_end,
                                               int64_t n, int tid, int nthreads,
                                               const int64_t *__restrict__ seg_start, int n_seg, float s,
                                               int random, const float *__restrict__ uniforms, uint64_t seed,
                                               uint64_t offset, LT *__restrict__ l, const uint32_t *keys)
{
    SegCache segc;
    float lb = 0.0f, ub = 0.0f;
    int cur = -1;
    const bool aligned = ((reinterpret_cast<uintptr_t>(u) & 15) == 0) &&
                         (uniforms == nullptr || (reinterpret_cast<uintptr_t>(uniforms) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(l) & (4 * sizeof(LT) - 1)) == 0);
    for (int64_t i0 = i_begin + 4 * (int64_t)tid; i0 < i_end; i0 += 4 * (int64_t)nthreads) {
        const int64_t q = i0 >> 2;
        const bool full = aligned && (i0 + 3 < n);
        float x[4], r[4] = {0.f, 0.f, 0.f, 0.f};
        if (full) {
            const float4 t = VOLATILE_KEYS ? __ldcg(reinterpret_cast<const float4 *>(u) + q)
                                           : __ldg(reinterpret_cast<const float4 *>(u) + q);
            x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) x[t] = (i0 + t < n) ? u[i0 + t] : 0.0f;
        }
        if (random) {
            if (uniforms) {
                if (full) {
                    const float4 t = __ldg(reinterpret_cast<const float4 *>(uniforms) + q);
                    r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
                } else {
#pragma unroll
                    for (int t = 0; t < 4; ++t) r[t] = (i0 + t < n) ? uniforms[i0 + t] : 0.0f;
                }
            } else if (((offset + (uint64_t)i0) & 3u) == 0) {
                const uint4 w = philox4x32_10(seed, (offset + (uint64_t)i0) >> 2);
                r[0] = u01(w.x); r[1] = u01(w.y); r[2] = u01(w.z); r[3] = u01(w.w);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) r[t] = philox_uniform(seed, offset, (uint64_t)(i0 + t));
            }
        }
        int lv[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int64_t i = i0 + t;
            if (i < n) {
                const int seg = cached_segment(segc, seg_start, n_seg, i);
                if (seg != cur) {
                    cur = seg;
                    if (VOLATILE_KEYS) {
                        lb = key_to_float(__ldcg(keys + 2 * seg));
                        ub = key_to_float(__ldcg(keys + 2 * seg + 1));
                    } else {
                        lb = key_to_float(__ldg(keys + 2 * seg));
                        ub = key_to_float(__ldg(keys + 2 * seg + 1));
                    }
                }
                lv[t] = psc_level(x[t], lb, ub, s, random, r[t]);
            } else {
                lv[t] = 0;
            }
        }
        if (full) {
            if (sizeof(LT) == 1) {
                reinterpret_cast<uint32_t *>(l)[q] =
                    (uint32_t)lv[0] | ((uint32_t)lv[1] << 8) | ((uint32_t)lv[2] << 16) | ((uint32_t)lv[3] << 24);
            } else {
                reinterpret_cast<int4 *>(l)[q] = make_int4(lv[0], lv[1], lv[2], lv[3]);
            }
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (i0 + t < n) l[i0 + t] = (LT)lv[t];
        }
    }
}

// Running per-tensor min/max of u kept in registers while a warp walks CONSECUTIVE chunks
// (the tcgen05 kernel gives every CTA a contiguous range of tiles): one atomic pair per warp
// per tensor instead of one per tile.  Both functions are warp-collective.
struct MinMaxAcc {
    int seg = -1;
    float mn = INFINITY, mx = -INFINITY;
};
__device__ __forceinline__ void minmax_flush_warp(MinMaxAcc &a, uint32_t *__restrict__ keys)
{
    const uint32_t have = __ballot_sync(0xffffffffu, a.seg >= 0);
    if (have != 0u) {
        const int seg0 = __shfl_sync(0xffffffffu, a.seg, __ffs(have) - 1);
        const bool uniform = __all_sync(0xffffffffu, a.seg == seg0 || a.seg < 0);
        if (uniform) {
            const float mn = warp_min(a.mn), mx = warp_max(a.mx);
            if ((threadIdx.x & 31) == 0) {
                atomicMin(keys + 2 * seg0, float_to_key(mn));
                atomicMax(keys + 2 * seg0 + 1, float_to_key(mx));
            }
        } else if (a.seg >= 0) {
            atomicMin(keys + 2 * a.seg, float_to_key(a.mn));
            atomicMax(keys + 2 * a.seg + 1, float_to_key(a.mx));
        }
    }
    a.seg = -1;
    a.mn = INFINITY;
    a.mx = -INFINITY;
}
__device__ __forceinline__ void minmax_add_warp(MinMaxAcc &a, bool valid, int seg, float u,
                                                uint32_t *__restrict__ keys)
{
    if (__any_sync(0xffffffffu, valid && a.seg >= 0 && seg != a.seg)) minmax_flush_warp(a, keys);
    // fminf / fmaxf drop NaN; the reference's torch.min / torch.max propagate it (the whole tensor then
    // decodes to NaN): a NaN score goes straight into the max key, which orders above +inf
    if (valid && u != u) atomicMax(keys + 2 * seg + 1, GQ_KEY_NAN);
    if (valid) {
        a.seg = seg;
        a.mn = fminf(a.mn, u);
        a.mx = fmaxf(a.mx, u);
    }
}

}  // namespace gq

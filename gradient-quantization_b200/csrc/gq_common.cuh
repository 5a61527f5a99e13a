// gq_common.cuh -- shared device/host helpers for libgqb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gqb200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libgqb200 is written for sm_100a (B200) only"
#endif

namespace gq {

// ---------------------------------------------------------------- errors ---
void set_error(const char *fmt, ...);
int check_cuda(cudaError_t e, const char *what);
int sm_count();

#define GQ_REQUIRE(cond, ...)                \
    do {                                     \
        if (!(cond)) {                       \
            gq::set_error(__VA_ARGS__);      \
            return GQ_ERR_INVALID;           \
        }                                    \
    } while (0)

#define GQ_CUDA(expr)                                        \
    do {                                                     \
        int _e = gq::check_cuda((expr), #expr);              \
        if (_e) return _e;                                   \
    } while (0)

#define GQ_LAUNCH_CHECK(name) GQ_CUDA((cudaError_t)cudaPeekAtLastError())

static inline cudaStream_t as_stream(gq_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// ------------------------------------------- programmatic dependent launch ---
// The kernels of one encode/decode step are short (2-80 us) and strictly chained, so launch
// latency and prologues (codebook staging, TMEM allocation) are a visible fraction of the step.
// Every kernel of the chain calls pdl_launch_dependents() first (the next kernel's grid may be
// scheduled as soon as SMs free up) and pdl_wait() before it touches anything a predecessor
// wrote; launches go through launch_pdl().  GQ_PDL=0 in the environment turns the attribute off.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// ---------------------------------------------------- ordered float keys ---
// Monotone map fp32 -> uint32 so that unsigned atomicMin/atomicMax implement
// float min/max (used for the per-tensor lb/ub of the norm quantizer).
__host__ __device__ __forceinline__ uint32_t float_to_key(float f)
{
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t b = c.u;
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float key_to_float(uint32_t k)
{
    uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    union { float f; uint32_t u; } c; c.u = b; return c.f;
#endif
}
#define GQ_KEY_MIN_INIT 0xffffffffu
#define GQ_KEY_MAX_INIT 0x00000000u
#define GQ_KEY_NAN 0xffc00000u      // key of +NaN: above +inf, so a NaN input reaches ub (and the decoded tensor)

// ---------------------------------------------------------------- philox ---
// Philox4x32-10, counter = (idx_lo, idx_hi, 0, 0), key = seed.  One call gives
// four 32-bit words; uniform = 24 high bits * 2^-24 (in [0,1), like torch.rand).
__device__ __forceinline__ uint4 philox4x32_10(uint64_t seed, uint64_t idx)
{
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32), c2 = 0u, c3 = 0u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
// one uniform per logical index (4 indices share one Philox block)
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t offset, uint64_t i)
{
    uint64_t g = offset + i;
    uint4 w = philox4x32_10(seed, g >> 2);
    uint32_t s = (uint32_t)(g & 3u);
    uint32_t x = (s == 0) ? w.x : (s == 1) ? w.y : (s == 2) ? w.z : w.w;
    return u01(x);
}
// the uniforms of logical indices i .. i + 3 (== philox_uniform of each): one Philox block when
// offset + i is a multiple of 4, else the two blocks the four words straddle
__device__ __forceinline__ void philox_uniform4(uint64_t seed, uint64_t offset, uint64_t i, float (&r)[4])
{
    const uint64_t g = offset + i;
    const uint4 a = philox4x32_10(seed, g >> 2);
    const uint32_t sh = (uint32_t)(g & 3u);
    if (sh == 0) {
        r[0] = u01(a.x); r[1] = u01(a.y); r[2] = u01(a.z); r[3] = u01(a.w);
        return;
    }
    const uint4 b = philox4x32_10(seed, (g >> 2) + 1);
    r[0] = u01(sh == 1 ? a.y : sh == 2 ? a.z : a.w);
    r[1] = u01(sh == 1 ? a.z : sh == 2 ? a.w : b.x);
    r[2] = u01(sh == 1 ? a.w : sh == 2 ? b.x : b.y);
    r[3] = u01(sh == 1 ? b.x : sh == 2 ? b.y : b.z);
}

// --------------------------------------------------------- segment lookup ---
// seg_start is sorted, seg_start[0] == 0, seg_start[n_seg] == n.  Returns s with
// seg_start[s] <= i < seg_start[s+1].
__device__ __forceinline__ int find_segment(const int64_t *__restrict__ seg_start, int n_seg, int64_t i)
{
    int lo = 0, hi = n_seg;  // invariant: seg_start[lo] <= i < seg_start[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(seg_start + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// Per-thread cache of the last segment looked up.  Grid-stride loops visit increasing
// indices, so almost every lookup is two compares instead of a binary search of
// dependent loads (tensors hold 64 .. 147 456 chunks).
struct SegCache {
    int seg = 0;
    int64_t lo = 0, hi = 0;   // cached segment covers [lo, hi); empty at start
};
__device__ __forceinline__ int cached_segment(SegCache &sc, const int64_t *__restrict__ seg_start, int n_seg,
                                              int64_t i)
{
    if (i < sc.lo || i >= sc.hi) {
        sc.seg = find_segment(seg_start, n_seg, i);
        sc.lo = __ldg(seg_start + sc.seg);
        sc.hi = __ldg(seg_start + sc.seg + 1);
    }
    return sc.seg;
}

// The same two functions over a copy of the table in SHARED memory (plain loads): a binary search is
// seven ~30-cycle steps instead of seven dependent L2 round trips -- kernels whose CTAs jump between
// distant tiles (the decode kernels) pay that search at every jump.
__device__ __forceinline__ int find_segment_smem(const int64_t *s_seg, int n_seg, int64_t i)
{
    int lo = 0, hi = n_seg;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (s_seg[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ int cached_segment_smem(SegCache &sc, const int64_t *s_seg, int n_seg, int64_t i)
{
    if (i < sc.lo || i >= sc.hi) {
        sc.seg = find_segment_smem(s_seg, n_seg, i);
        sc.lo = s_seg[sc.seg];
        sc.hi = s_seg[sc.seg + 1];
    }
    return sc.seg;
}

// ------------------------------------------------ reference scalar codecs ---
// ProbabilisticScalarCompressor.compress, element-wise part
// (compressors/probabilistic_scalar_compressor.py:17-26), exact op order.
__device__ __forceinline__ int psc_level(float v, float lb, float ub, float s, int random, float r)
{
    if (lb - ub == 0.0f) return 0;
    float scaled = fabsf(__fdiv_rn(__fsub_rn(v, lb), __fsub_rn(ub, lb))) * s;
    float c = fminf(fmaxf(scaled, 0.0f), s - 1.0f);
    int li = (int)c;  // truncation toward zero
    if (random) {
        float prob = __fsub_rn(scaled, (float)li);
        li += (prob > r) ? 1 : 0;
    }
    return li;
}
// psc_level() for lb != ub, with den = ub - lb computed by the caller (same operations)
__device__ __forceinline__ int psc_level_nz(float v, float lb, float den, float s, int random, float r)
{
    const float scaled = fabsf(__fdiv_rn(__fsub_rn(v, lb), den)) * s;
    const float c = fminf(fmaxf(scaled, 0.0f), s - 1.0f);
    int li = (int)c;
    if (random) li += (__fsub_rn(scaled, (float)li) > r) ? 1 : 0;
    return li;
}
// Levels of the four consecutive chunks i0 .. i0 + 3 (i0 < n) from a tensor-boundary table and the
// (lb, ub) pairs in shared memory.  `seg` is a tensor at or before i0's and is advanced to it.  When all
// four chunks lie in one tensor (almost always) lb, ub and ub - lb are fetched once.  Every kernel that
// quantizes norms in groups of four (the tcgen05 encode's tail, the stand-alone quantizer, the fused
// quantize-and-decode) computes its levels here, so their records agree bit for bit.
template <typename SegT, typename IdxT>
__device__ __forceinline__ void psc_levels4(const float (&x)[4], const float (&r)[4], IdxT i0, IdxT n,
                                            const SegT *s_seg, const float2 *s_lbub, int &seg, float s, int random,
                                            int (&lv)[4])
{
    while (i0 >= s_seg[seg + 1]) ++seg;
    if (i0 + 3 < s_seg[seg + 1]) {
        const float2 b = s_lbub[seg];
        if (b.x - b.y == 0.0f) {
            lv[0] = lv[1] = lv[2] = lv[3] = 0;
        } else {
            const float den = __fsub_rn(b.y, b.x);
#pragma unroll
            for (int t = 0; t < 4; ++t) lv[t] = psc_level_nz(x[t], b.x, den, s, random, r[t]);
        }
    } else {
        int sg = seg;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const IdxT i = i0 + t;
            if (i < n) {
                while (i >= s_seg[sg + 1]) ++sg;
                const float2 b = s_lbub[sg];
                lv[t] = psc_level(x[t], b.x, b.y, s, random, r[t]);
            } else {
                lv[t] = 0;
            }
        }
    }
}
// ProbabilisticScalarCompressor.decompress (probabilistic_scalar_compressor.py:31-32)
// s = 2^n is a power of two, so "/ s" is done as an exact multiplication by inv_s = 1/s
// (identical result for every input, including subnormals).
__device__ __forceinline__ float psc_value(int l, float lb, float ub, float inv_s)
{
    return __fadd_rn(__fmul_rn(__fmul_rn((float)l, __fsub_rn(ub, lb)), inv_s), lb);
}

__device__ __forceinline__ float warp_min(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// streaming 128-bit load that does not allocate in L1
__device__ __forceinline__ float4 ld_stream_f4(const float4 *p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

}  // namespace gq

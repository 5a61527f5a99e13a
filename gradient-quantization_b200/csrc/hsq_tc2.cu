// hsq_tc2.cu -- second-generation tcgen05 HSQ encode for d in {8, 16, 32}, K == 256 (uint8 codes):
// ONE launch = min/max key reset + identity rider + TF32 search with exact fp32 rescoring +
// (after a grid-wide barrier) the n-bit norm quantization of every CTA's own chunk range, and
// optionally the delivery of the finished record sections into the peers' receive blocks.
//
// Same pipeline as hsq_tc.cu (TMA -> smem ring -> 2 x tcgen05.mma kind::tf32 M128 N256 K8 ->
// two TMEM buffers -> one epilogue thread per row), same exactness argument (every codeword of
// every group whose approximate maximum lies within 2*eps of the row maximum is rescored with
// the ascending-j fmaf chain, first index wins).  What changed is the instruction budget of the
// epilogue, which is what bounds the kernel (ALU pipe / issue slots, not HBM or the tensor pipe):
//   PAIR   the B operand holds c_{2i} + c_{2i+1} and c_{2i} - c_{2i+1} instead of the codewords:
//          max(|s_a|, |s_b|) = (|s_a + s_b| + |s_a - s_b|) / 2, so the first reduction level of
//          the group maxima is one FADD with |.| operand modifiers on the FMA pipe instead of an
//          FMNMX on the (half as wide, busier) ALU pipe; everything downstream works on doubled
//          values.  The error bound scales with (||b_p|| + ||b_m||) / 2 <= sqrt(2) max||c||.
//   FMASK  the 64-group candidate mask is built on the FMA pipe: b_g = sat((gm_g - thr') * S) is
//          exactly 0 or 1 (S = 2^(24 - exponent(thr)), thr' = the float below thr), accumulated as
//          m = 2 m + b_g in four fp32 chains whose mantissas are the mask -- no FADD + funnel shift.
//   F2     rescoring with packed FFMA2 (fma.rn.f32x2): two codewords per instruction, bit-identical
//          lanes; the codebook planes are pair-interleaved.
//   waits  mbarrier.try_wait with a suspend-time hint instead of hot polling loops.
//   tail   norm quantization fused behind a grid barrier (all CTAs are co-resident: grid <= SMs,
//          one CTA per SM), every thread's loads issued before any is consumed.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <atomic>
#include <mutex>

#include "gq_internal.cuh"
#include "tc_ptx.cuh"

namespace gq {
namespace tc2 {

using namespace tcptx;

constexpr int kK = 256;
constexpr int kTileM = 128;
constexpr int kGroup = 4;
constexpr int kNumGroups = kK / kGroup;           // 64
// Per chunk dimension D: a tile row is one swizzle atom row of the TMA / UMMA layouts (32, 64 or
// 128 bytes -> SWIZZLE_32B / 64B / 128B), D / 8 tcgen05.mma K-steps per tile.
template <int D>
struct Dim {
    static_assert(D == 8 || D == 16 || D == 32, "chunk dimension");
    static constexpr uint32_t kRowBytes = D * 4;
    static constexpr uint32_t kTileBytes = kTileM * kRowBytes;   // 4 / 8 / 16 KB
    static constexpr uint32_t kCbBytes = kK * kRowBytes;         // TF32 B operand
    static constexpr int kUnits = D / 4;                         // 16-byte units per row
    static constexpr uint32_t kPlanesBytes = (D == 8) ? 65536 : 131072;   // rescoring planes (replicated codebook)
    static constexpr uint64_t kSwizzleCode = (D == 8) ? 6 : (D == 16 ? 4 : 2);   // UMMA layout type
    // 16-byte unit u of row r is stored at unit u ^ sw(r) (Swizzle<1|2|3, 4, 3>)
    __device__ static __forceinline__ uint32_t sw(int r)
    {
        return D == 8 ? (uint32_t)((r >> 2) & 1) : (D == 16 ? (uint32_t)((r >> 1) & 3) : (uint32_t)(r & 7));
    }
};
constexpr int kTailMaxSeg = 1024;                 // segment tables of the fused tail live in the stage ring
// 2 * eps / (||v|| * norm scale), see hsq_tc.cu (kMargin) for the derivation; the PAIR variant adds
// the fp32 rounding of c_a +- c_b (2^-24) and of |p| + |m| (2^-24), covered by the larger slack
constexpr float kMargin = 2.0f * (1.5f / 1024.0f + 4.0e-6f);
constexpr float kMarginPair = 2.0f * (1.5f / 1024.0f + 8.0e-6f);
constexpr float kMarginExtra32 = 2.0f * 4.0e-6f;   // D == 32: twice as many fp32 accumulation steps
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((kK >> 3) << 17) | ((kTileM >> 4) << 24);

template <int G, int D = 16>
struct Layout {
    // D == 32: four 16 KB stages (64 KB in flight per SM) leave room for four 32 KB rescoring planes
    static constexpr int kStages = (D == 32) ? 4 : ((G == 4) ? 8 : 6);
    static constexpr uint32_t kOffA = 0;
    static constexpr uint32_t kOffCb = kStages * Dim<D>::kTileBytes;
    static constexpr uint32_t kOffPlanes = kOffCb + Dim<D>::kCbBytes;
    static constexpr uint32_t kOffBar = kOffPlanes + Dim<D>::kPlanesBytes;
    static constexpr uint32_t kSmemBytes = kOffBar + 1024 + 1024;   // barriers + code staging, + alignment slack
    static_assert(kSmemBytes <= 232448, "shared memory budget");
    static_assert(kStages * Dim<D>::kTileBytes >= 4 * (kTailMaxSeg + 2) + 8 * kTailMaxSeg, "tail tables live in the stage ring");
};

// Where else the finished record sections go (multi-GPU ps exchange fused into the encode):
// every address the tail writes inside the local record is also written at address + delta[i].
struct Remote {
    int n;                  // number of remote destinations (0: none)
    int multicast;          // 1: delta[0] leads into an NVLS multicast mapping (multimem.st)
    int64_t delta[7];
    const uint8_t *ident;   // identity section of the local record (written by the rider), mirrored too
    int64_t ident_bytes;    // multiple of 16
    uint32_t *done;         // local arrival counter (zeroed together with the grid barrier word)
    uint32_t *flag[8];      // where to announce `epoch` once every CTA has delivered (n_flag entries)
    int n_flag;
    uint32_t epoch;
};

struct Enc2 {
    const float *codebook;
    int n_chunks;
    uint8_t *codes;
    float *u_out;
    const int64_t *seg_start;
    int n_seg;
    uint32_t *keys;              // [2 * n_seg] min/max keys, nullptr: no min/max wanted
    unsigned long long *flag;    // in-kernel key reset handshake (nullptr: keys are ready)
    unsigned long long id;
    Rider rider;
    uint8_t *l;                  // fused tail when != nullptr
    float *lbub;
    uint32_t *barrier;
    const float *uniforms;
    uint64_t seed, offset;
    float s;
    int random;
    Remote remote;
    long long *trace;            // TRACE builds only
};

__device__ __forceinline__ float4 lds_f4(uint32_t a)
{
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(a));
    return r;
}
__device__ __forceinline__ void lds_2x64(uint32_t a, unsigned long long &lo, unsigned long long &hi)
{
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "r"(a));
}
__device__ __forceinline__ unsigned long long pack2(float a, float b)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &a, float &b)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long fmul2(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float fma_sat(float a, float b, float c)
{
    float r;
    asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }
// doubled maximum of |score| over a group of four codewords from its accumulators (p_a, m_a, p_b, m_b):
// max(|p_a| + |m_a|, |p_b| + |m_b|).  (With the B rows ordered p_a, p_b, m_a, m_b one packed FADD2 with |.|
// modifiers serves both pairs -- 64 fewer instructions per row, and measured 2.5 - 4 us SLOWER per launch:
// the first pass is bound by the TMEM read-back, not by issue slots, and FADD2 is no cheaper than two FADDs.)
__device__ __forceinline__ float pair_group_max(uint32_t pa, uint32_t ma, uint32_t pb, uint32_t mb)
{
    return fmaxf(__fadd_rn(fabsf(__uint_as_float(pa)), fabsf(__uint_as_float(ma))),
                 __fadd_rn(fabsf(__uint_as_float(pb)), fabsf(__uint_as_float(mb))));
}

// store 4 bytes / 16 bytes at a local record address and at every remote copy of it
__device__ __forceinline__ void remote_st32(const Remote &R, void *local, uint32_t v)
{
    if (R.multicast) {
        asm volatile("multimem.st.weak.global.u32 [%0], %1;" ::"l"((char *)local + R.delta[0]), "r"(v) : "memory");
    } else {
#pragma unroll
        for (int i = 0; i < 7; ++i)
            if (i < R.n) *reinterpret_cast<uint32_t *>((char *)local + R.delta[i]) = v;
    }
}
__device__ __forceinline__ void remote_st128(const Remote &R, void *local, uint4 v)
{
    if (R.multicast) {
        asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};"
                     ::"l"((char *)local + R.delta[0]), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)),
                       "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w)) : "memory");
    } else {
#pragma unroll
        for (int i = 0; i < 7; ++i)
            if (i < R.n) *reinterpret_cast<uint4 *>((char *)local + R.delta[i]) = v;
    }
}

// K-major operand descriptor: rows of one swizzle atom (32 / 64 / 128 B), 8-row groups 8 * row bytes apart
template <int D>
__device__ __forceinline__ uint64_t make_desc_d(uint32_t saddr)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;                                   // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)((8 * Dim<D>::kRowBytes) >> 4) << 32;      // stride byte offset
    d |= (uint64_t)1 << 46;                                   // descriptor version (Blackwell)
    d |= Dim<D>::kSwizzleCode << 61;
    return d;
}

// the D / 8 K-steps of one 128 x 256 x D tile product, then the commit that arrives on `bar`
template <int D>
__device__ __forceinline__ void issue_tile_mma(uint32_t a_addr, uint32_t b_addr, uint32_t taddr, uint32_t bar)
{
    const uint64_t adesc = make_desc_d<D>(a_addr), bdesc = make_desc_d<D>(b_addr);
#pragma unroll
    for (int ks = 0; ks < D / 8; ++ks)   // k = 8 ks .. 8 ks + 7: bytes 32 ks .. of each row, +32 B = +2 units
        mma_tf32(taddr, adesc + 2 * ks, bdesc + 2 * ks, ks ? 1u : 0u, kIdesc);
    mma_commit(bar);
}

// TRACE builds: CTA 0 time-stamps pipeline events of its first 128 tiles, trace[event * 128 + it] =
// clock64(): 0 TMA issued, 1 MMA issued, 2 accumulators seen by the epilogue warp, 3 TMEM released
// (first pass done), 4 smem stage released, 5 candidate mask done, 6 rescoring done, 7 tile done,
// 8 rescoring iterations of the warp (count, not a time); taken by quadrant 0 / lane 0 of each group;
// 9..11 TMEM released by quadrants 1..3, 12 / 13 MMA warp past its TMEM-empty / smem-full wait,
// 14 MMA commit seen by a polling observer thread (spare warp 3).
template <int G, bool PAIR, bool FMASK, bool F2, bool R2 = false, bool TRACE = false, int D = 16>
__global__ void __launch_bounds__(128 + 128 * G, 1)
hsq_encode_tc2_kernel(const __grid_constant__ CUtensorMap map_grad, const __grid_constant__ Enc2 P)
{
    static_assert(D != 8 || F2, "d = 8 uses the packed rescoring layout");
    static_assert(D != 32 || !F2, "d = 32 rescoring is scalar (register budget)");
    constexpr int kD = D;
    constexpr uint32_t kTileBytes = Dim<D>::kTileBytes;
    constexpr uint32_t kRowBytes = Dim<D>::kRowBytes;
    constexpr int kUnits = Dim<D>::kUnits;
#define GQ_TRACE(ev, it_) do { if (TRACE && blockIdx.x == 0 && (it_) < 128) P.trace[(ev) * 128 + (it_)] = clock64(); } while (0)
    using L = Layout<G, D>;
    constexpr int kThreads = 128 + 128 * G;
    constexpr int kStages = L::kStages;
    pdl_launch_dependents();
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *s_a = smem + L::kOffA;
    uint8_t *s_cb = smem + L::kOffCb;
    uint8_t *s_planes = smem + L::kOffPlanes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + L::kOffBar);
    const uint32_t bar_full = smem_u32(bars);
    const uint32_t bar_empty = bar_full + 8 * kStages;
    const uint32_t bar_tfull = bar_empty + 8 * kStages;
    const uint32_t bar_tempty = bar_tfull + 8 * kStages;
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(smem + L::kOffBar + 8 * (4 * kStages));
    float *s_cn = reinterpret_cast<float *>(smem + L::kOffBar + 8 * (4 * kStages) + 8);   // [8] per-warp norm maxima
    int *s_misc = reinterpret_cast<int *>(smem + L::kOffBar + 8 * (4 * kStages) + 8 + 32);
    static_assert(8 * (4 * kStages) + 8 + 32 + 16 <= 512, "barrier region");
    uint8_t *s_codes = smem + L::kOffBar + 512;   // [4 * G warps][32] codes of a warp-tile, staged for 16-byte stores
    static_assert(4 * G * 32 <= 512, "code staging");

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n_chunks = P.n_chunks;
    const int n_tiles = (n_chunks + kTileM - 1) / kTileM;
    const int tq = n_tiles / (int)gridDim.x, trem = n_tiles % (int)gridDim.x;
    const int tile0 = (int)blockIdx.x * tq + min((int)blockIdx.x, trem);
    const int my_tiles = tq + (((int)blockIdx.x < trem) ? 1 : 0);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 4);
            mbar_init(bar_tfull + 8 * s, 1);
            mbar_init(bar_tempty + 8 * s, 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    const float *codebook = P.codebook;
    // ---- rescoring planes (exact fp32 codewords, replicated so that lane-divergent LDS.128 never conflict)
    if constexpr (F2 && D == 8) {
        // 4 planes (rotation r) x 128 codeword pairs x 128 bytes; the pair's four 16-byte units
        // (c_2p[2t], c_2p+1[2t], c_2p[2t+1], c_2p+1[2t+1]) twice (half h) at bank group 4h + ((t + r) & 3)
        for (int i = threadIdx.x; i < 4 * 128 * 2 * 4; i += kThreads) {
            const int t = i & 3, h = (i >> 2) & 1, p = (i >> 3) & 127, r = i >> 10;
            const float2 a = __ldg(reinterpret_cast<const float2 *>(codebook + (2 * p) * kD) + t);
            const float2 b = __ldg(reinterpret_cast<const float2 *>(codebook + (2 * p + 1) * kD) + t);
            *reinterpret_cast<float4 *>(s_planes + r * 16384 + p * 128 + 16 * (4 * h + ((t + r) & 3))) =
                make_float4(a.x, b.x, a.y, b.y);
        }
    } else if constexpr (F2) {
        // 8 planes (one per lane class c = lane & 7) x 128 codeword pairs x 128 bytes; 16-byte unit t of
        // pair p = (c_2p[2t], c_2p+1[2t], c_2p[2t+1], c_2p+1[2t+1]) stored at bank group (t + c) & 7
        for (int i = threadIdx.x; i < 8 * 128 * 8; i += kThreads) {
            const int t = i & 7, p = (i >> 3) & 127, c = i >> 10;
            const float2 a = __ldg(reinterpret_cast<const float2 *>(codebook + (2 * p) * kD) + t);
            const float2 b = __ldg(reinterpret_cast<const float2 *>(codebook + (2 * p + 1) * kD) + t);
            *reinterpret_cast<float4 *>(s_planes + c * 16384 + p * 128 + 16 * ((t + c) & 7)) =
                make_float4(a.x, b.x, a.y, b.y);
        }
    } else if constexpr (D == 32) {
        // 4 planes (rotation r = lane & 3) x 256 codewords x 128 bytes: unit u at bank group (u + r) & 7
        // (lanes c and c + 4 of a quarter-warp share a plane: at most two wavefronts per LDS.128)
        for (int i = threadIdx.x; i < 4 * kK * 8; i += kThreads) {
            const int u = i & 7, k = (i >> 3) & (kK - 1), r = i >> 11;
            const float4 val = __ldg(reinterpret_cast<const float4 *>(codebook) + k * 8 + u);
            *reinterpret_cast<float4 *>(s_planes + r * 32768 + k * 128 + 16 * ((u + r) & 7)) = val;
        }
    } else {
        // 4 planes (rotation r) x 256 codewords x 128 bytes: unit u twice (half h) at bank group 4h + ((u + r) & 3)
        for (int i = threadIdx.x; i < 4 * kK * 8; i += kThreads) {
            const int u = i & 3, h = (i >> 2) & 1, k = (i >> 3) & (kK - 1), r = i >> 11;
            const float4 val = __ldg(reinterpret_cast<const float4 *>(codebook) + k * 4 + u);
            *reinterpret_cast<float4 *>(s_planes + r * 32768 + k * 128 + 16 * (4 * h + ((u + r) & 3))) = val;
        }
    }
    // ---- MMA B operand, K-major swizzled (row k = one atom row, unit u at u ^ sw(k)), rounded
    //      to nearest TF32; PAIR: row 2i = c_2i + c_2i+1, row 2i+1 = c_2i - c_2i+1
    for (int i = threadIdx.x; i < kK * kUnits; i += kThreads) {
        const int u = i % kUnits, k = i / kUnits;
        float4 val;
        if (PAIR) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(codebook) + (k & ~1) * kUnits + u);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(codebook) + (k | 1) * kUnits + u);
            val = (k & 1) ? make_float4(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z), __fsub_rn(a.w, b.w))
                          : make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
        } else {
            val = __ldg(reinterpret_cast<const float4 *>(codebook) + k * kUnits + u);
        }
        uint4 t;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t.x) : "f"(val.x));
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t.y) : "f"(val.y));
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t.z) : "f"(val.z));
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t.w) : "f"(val.w));
        *reinterpret_cast<uint4 *>(s_cb + k * kRowBytes + ((u ^ Dim<D>::sw(k)) << 4)) = t;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    // ---- norm scale of the error bound: max ||c_k||, or (PAIR) max over pairs of ||c_a + c_b|| + ||c_a - c_b||
    if (threadIdx.x < kK) {
        float val;
        if (PAIR) {
            const int p = threadIdx.x >> 1;   // both threads of a pair compute the same value
            float sp = 0.0f, sm = 0.0f;
#pragma unroll
            for (int j = 0; j < kD; ++j) {
                const float a = __ldg(codebook + (2 * p) * kD + j), b = __ldg(codebook + (2 * p + 1) * kD + j);
                const float ps = __fadd_rn(a, b), ms = __fsub_rn(a, b);
                sp = fmaf(ps, ps, sp);
                sm = fmaf(ms, ms, sm);
            }
            val = __fadd_rn(sqrtf(sp), sqrtf(sm));
        } else {
            float c2 = 0.0f;
#pragma unroll
            for (int j = 0; j < kD; ++j) {
                const float a = __ldg(codebook + threadIdx.x * kD + j);
                c2 = fmaf(a, a, c2);
            }
            val = sqrtf(c2);
        }
        if (!(val < 3.0e38f)) val = __int_as_float(0x7f800000);   // NaN -> +inf so that the max keeps it
        val = warp_max(val);
        if (lane == 0) s_cn[warp] = val;
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    float cn = s_cn[0];
#pragma unroll
    for (int w = 1; w < kK / 32; ++w) cn = fmaxf(cn, s_cn[w]);
    // (a non-finite codebook gives margin = +inf: threshold -inf / NaN, every group is rescored)
    const float margin = ((PAIR ? kMarginPair : kMargin) + (D == 32 ? kMarginExtra32 : 0.0f)) * (1.0f + 1.0e-5f) * cn;
    pdl_wait();
    // TRACE: per-CTA wall-clock stamps (ns) after the trace table: start, main loop done, grid barrier passed, tail done
#define GQ_STAMP(k) do { if (TRACE && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); \
        P.trace[16 * 128 + 4 * blockIdx.x + (k)] = (long long)t_; } } while (0)
    GQ_STAMP(0);

    if (warp == 0) {
        // ------------------------------------------------------ TMA producer ---
        if (lane == 0) {
            for (int it = 0; it < my_tiles; ++it) {
                const int s = it % kStages;
                mbar_wait_sleep(bar_empty + 8 * s, ((it / kStages) & 1) ^ 1);
                mbar_expect_tx(bar_full + 8 * s, kTileBytes);
                tma_load_2d(smem_u32(s_a + s * kTileBytes), &map_grad, bar_full + 8 * s, 0, (tile0 + it) * kTileM);
                GQ_TRACE(0, it);
            }
        }
    } else if (warp == 1) {
        // -------------------------------------------------------- MMA issuer ---
        // (Issuing the MMA of tile it + 2 from the last epilogue warp to leave the TMEM buffer instead of
        //  from this warp removes ~900 cycles between release and issue -- and was measured SLOWER, 64 vs
        //  56 us: the buffer turnaround is set by the slowest of the group's four warps in the first pass,
        //  ~1500 cycles under contention with the other groups' rescoring, and an MMA running against the
        //  other group's TMEM loads costs them more than the early issue gains; tests/tc2_trace.py.)
        if (lane == 0) {
            const uint64_t bdesc = make_desc_d<D>(smem_u32(s_cb));
            for (int it = 0; it < my_tiles; ++it) {
                const int s = it % kStages;
                const int b = it & 1;
                // the operand tile landed long ago (the producer runs kStages ahead): take that wait first,
                // so that nothing but the issue itself follows the release of the TMEM buffer
                mbar_wait_sleep(bar_full + 8 * s, (it / kStages) & 1);
                GQ_TRACE(12, it);
                // everything the issue needs is in registers BEFORE the wait for the TMEM buffer (the empty
                // asm pins it there): this single thread competes with three busy warps for its scheduler,
                // and every instruction between the release and the MMA is on the kernel's critical chain
                uint64_t adesc = make_desc_d<D>(smem_u32(s_a + s * kTileBytes));
                uint64_t bd = bdesc;
                uint32_t taddr = tmem_base + (uint32_t)(b * kK);
                uint32_t tfull = bar_tfull + 8 * s;
                asm volatile("" : "+l"(adesc), "+l"(bd), "+r"(taddr), "+r"(tfull));
                // (plain try_wait; the suspend-hint form and a test_wait spin measured the same, GQ_TC2_WAIT A/B)
                if (it >= 2) mbar_wait_hw(bar_tempty + 8 * ((it - 2) % kStages), ((it - 2) / kStages) & 1);
                GQ_TRACE(13, it);
                tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < D / 8; ++ks)
                    mma_tf32(taddr, adesc + 2 * ks, bd + 2 * ks, ks ? 1u : 0u, kIdesc);
                mma_commit(tfull);
                GQ_TRACE(1, it);
            }
        }
    } else if (warp < 4) {
        // ------------------------------------- spare warps 2, 3: preparation ---
        if (P.flag != nullptr && blockIdx.x == 0 && warp == 3) {
            for (int i = lane; i < 2 * P.n_seg; i += 32) P.keys[i] = (i & 1) ? GQ_KEY_MAX_INIT : GQ_KEY_MIN_INIT;
            if (lane == 0 && P.barrier != nullptr) {
                P.barrier[0] = 0u;
                if (P.remote.done != nullptr) P.remote.done[0] = 0u;
            }
            __threadfence();
            __syncwarp();
            if (lane == 0)
                asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(P.flag), "l"(P.id) : "memory");
        }
        rider_run(P.rider, (int64_t)blockIdx.x * 64 + (threadIdx.x - 64), (int64_t)gridDim.x * 64);
        if (TRACE && blockIdx.x == 0 && warp == 3 && lane == 0) {
            // observer: polls (no sleep) for the completion of each tile's MMA commit -> event 14
            for (int it = 0; it < my_tiles && it < 128; ++it) {
                const int s = it % kStages;
                while (!mbar_test_wait(bar_tfull + 8 * s, (it / kStages) & 1)) { }
                GQ_TRACE(14, it);
            }
        }
    } else {
        // ----------------------------------------------------------- epilogue ---
        bool keys_ready = P.flag == nullptr;
        const int egroup = (warp - 4) >> 2;
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        uint32_t pbase;
        uint32_t uo[F2 ? kD / 2 : kUnits];
        if constexpr (F2 && D == 8) {
            const int rot = (lane & 7) >> 1, hlf = lane & 1;
            pbase = smem_u32(s_planes) + rot * 16384 + 64 * hlf;
#pragma unroll
            for (int t = 0; t < 4; ++t) uo[t] = 16u * ((t + rot) & 3);
        } else if constexpr (F2) {
            const int cls = lane & 7;
            pbase = smem_u32(s_planes) + cls * 16384;
#pragma unroll
            for (int t = 0; t < 8; ++t) uo[t] = 16u * ((t + cls) & 7);
        } else if constexpr (D == 32) {
            const int rot = lane & 3;
            pbase = smem_u32(s_planes) + rot * 32768;
#pragma unroll
            for (int u = 0; u < 8; ++u) uo[u] = 16u * ((u + rot) & 7);
        } else {
            const int rot = (lane & 7) >> 1, hlf = lane & 1;
            pbase = smem_u32(s_planes) + rot * 32768 + 64 * hlf;
#pragma unroll
            for (int u = 0; u < 4; ++u) uo[u] = 16u * ((u + rot) & 3);
        }
        SegCache segc;
        MinMaxAcc mm;
        const bool codes16 = (reinterpret_cast<uintptr_t>(P.codes) & 15) == 0;
        for (int it = egroup; it < my_tiles; it += G) {
            const int s = it % kStages;
            const uint32_t ph = (it / kStages) & 1;
            const int b = it & 1;
            const int c = (tile0 + it) * kTileM + row;
            const bool valid = c < n_chunks;
            // (TMEM address in a register before the waits: nothing but the loads follows the commit)
            uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(b * kK);
            asm volatile("" : "+r"(taddr));
            mbar_wait_hw(bar_tfull + 8 * s, ph);   // accumulators complete
            __syncwarp();
            tc_fence_after();
            const bool tracer = TRACE && quad == 0 && lane == 0;
            if (tracer) GQ_TRACE(2, it);

            // ---- pass over the 256 approximate scores of this row: maximum per group of 4 codewords
            //      (PAIR: doubled values, |p| + |m| per codeword pair)
            float gm[kNumGroups];
            {
                uint32_t sa[16], sb[16];
                tmem_ld16(taddr, sa);
                tmem_ld_wait16(sa);
#pragma unroll
                for (int h = 0; h < kK / 32; ++h) {
                    tmem_ld16(taddr + h * 32 + 16, sb);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        if (PAIR) {
                            gm[h * 8 + g] = pair_group_max(sa[4 * g], sa[4 * g + 1], sa[4 * g + 2], sa[4 * g + 3]);
                        } else {
                            const float m = fmaxf(fabsf(__uint_as_float(sa[4 * g])), fabsf(__uint_as_float(sa[4 * g + 1])));
                            gm[h * 8 + g] = max3(m, fabsf(__uint_as_float(sa[4 * g + 2])), fabsf(__uint_as_float(sa[4 * g + 3])));
                        }
                    }
                    tmem_ld_wait16(sb);
                    if (h + 1 < kK / 32) tmem_ld16(taddr + h * 32 + 32, sa);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        if (PAIR) {
                            gm[h * 8 + 4 + g] = pair_group_max(sb[4 * g], sb[4 * g + 1], sb[4 * g + 2], sb[4 * g + 3]);
                        } else {
                            const float m = fmaxf(fabsf(__uint_as_float(sb[4 * g])), fabsf(__uint_as_float(sb[4 * g + 1])));
                            gm[h * 8 + 4 + g] = max3(m, fabsf(__uint_as_float(sb[4 * g + 2])), fabsf(__uint_as_float(sb[4 * g + 3])));
                        }
                    }
                    if (h + 1 < kK / 32) tmem_ld_wait16(sa);
                }
            }
            // TMEM buffer b may be overwritten by the MMA of local tile it + 2
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + 8 * s);
            if (tracer) GQ_TRACE(3, it);
            if (TRACE && quad != 0 && lane == 0) GQ_TRACE(8 + quad, it);   // 9..11: the other quadrants' releases

            // ---- this row's chunk, from the (swizzled) smem tile.  The tile landed before its MMA was even
            //      issued; this thread still has to observe the TMA barrier itself before it reads the data,
            //      and does so here, off the TMEM turnaround chain (the wait returns at once)
            mbar_wait_hw(bar_full + 8 * s, ph);
            float v[kD];
            {
                const uint32_t arow = smem_u32(s_a) + s * kTileBytes + row * kRowBytes;
                const uint32_t sw = Dim<D>::sw(row);
#pragma unroll
                for (int u = 0; u < kUnits; ++u) {
                    const float4 t = lds_f4(arow + ((u ^ sw) << 4));
                    v[4 * u] = t.x; v[4 * u + 1] = t.y; v[4 * u + 2] = t.z; v[4 * u + 3] = t.w;
                }
            }
            float n2 = 0.0f;
#pragma unroll
            for (int j = 0; j < kD; ++j) n2 = fmaf(v[j], v[j], n2);
            // release the smem stage only after EVERY lane's loads of v have returned (see hsq_tc.cu)
            const uint32_t all_loaded = __ballot_sync(0xffffffffu, !(n2 < 0.0f));   // always all ones
            if (lane == 0) mbar_arrive(bar_empty + 8 * s + ((all_loaded == 0u) ? 8u : 0u));
            if (tracer) GQ_TRACE(4, it);

            // ---- row maximum (four chains of FMNMX3) and threshold
            float am[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                am[q] = max3(gm[16 * q], gm[16 * q + 1], gm[16 * q + 2]);
#pragma unroll
                for (int g = 3; g < 15; g += 2) am[q] = max3(am[q], gm[16 * q + g], gm[16 * q + g + 1]);
                am[q] = fmaxf(am[q], gm[16 * q + 15]);
            }
            const float amax = fmaxf(fmaxf(am[0], am[1]), fmaxf(am[2], am[3]));
            // (sqrt.approx: 1 MUFU instead of the IEEE sequence; its relative error of 2^-22 is inside the
            //  1e-5 slack of `margin`, and any superset of the candidate set gives the same exact result)
            float nrm;
            asm("sqrt.approx.f32 %0, %1;" : "=f"(nrm) : "f"(n2));
            const float thr = amax - margin * nrm;
            // ---- candidate groups: gm[g] >= thr
            uint32_t clo, chi;
            bool special;
            if (FMASK) {
                // thr in [1e-30, 3e38): S = 2^(24 - e(thr)) is a normal float, (gm - thr') * S is >= 1 for
                // every gm > thr' (thr' = the float below thr, i.e. gm >= thr) and <= 0 otherwise, so the
                // saturating FMA yields exactly 1.0 or 0.0; m = 2 m + b accumulates 16 of them exactly.
                special = !(n2 < 3.0e38f) || !(amax < 3.0e38f) || (n2 < 1.0e-30f) || !(thr >= 1.0e-30f);
                const uint32_t tb = __float_as_uint(thr);
                const float thrm = __uint_as_float(tb - 1u);
                const float S = __uint_as_float(0x8B000000u - (tb & 0x7F800000u));
                const float T = -__fmul_rn(thrm, S);
                // (the shift-accumulate step runs two chains per instruction: packed fma.rn.f32x2)
                const unsigned long long two2 = pack2(2.0f, 2.0f);
                unsigned long long mk01 = pack2(1.0f, 1.0f), mk23 = mk01;
#pragma unroll
                for (int g = 15; g >= 0; --g) {
                    mk01 = ffma2(mk01, two2, pack2(fma_sat(gm[g], S, T), fma_sat(gm[16 + g], S, T)));
                    mk23 = ffma2(mk23, two2, pack2(fma_sat(gm[32 + g], S, T), fma_sat(gm[48 + g], S, T)));
                }
                float mk[4];
                unpack2(mk01, mk[0], mk[1]);
                unpack2(mk23, mk[2], mk[3]);
                clo = ((__float_as_uint(mk[0]) >> 7) & 0xffffu) | ((__float_as_uint(mk[1]) << 9) & 0xffff0000u);
                chi = ((__float_as_uint(mk[2]) >> 7) & 0xffffu) | ((__float_as_uint(mk[3]) << 9) & 0xffff0000u);
            } else {
                special = !(n2 < 3.0e38f) || !(amax < 3.0e38f) || (n2 < 1.0e-30f);
                uint32_t bl[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int g = 15; g >= 0; --g) {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        bl[q] = __funnelshift_l(__float_as_uint(gm[16 * q + g] - thr), bl[q], 1);
                }
                clo = ~((bl[0] & 0xffffu) | (bl[1] << 16));
                chi = ~((bl[2] & 0xffffu) | (bl[3] << 16));
            }
            if (special || (clo | chi) == 0u) {
                // non-finite or vanishing norm, NaN scores, threshold out of range, empty set: rescore
                // everything; an all-zero row scores +-0 against every codeword: codeword 0 wins
                uint32_t any = 0u;
#pragma unroll
                for (int j = 0; j < kD; ++j) any |= __float_as_uint(v[j]);
                const bool zero = (any << 1) == 0u;
                clo = zero ? 1u : 0xffffffffu;
                chi = zero ? 0u : 0xffffffffu;
            }

            if (TRACE) {
                __syncwarp();
                if (tracer) GQ_TRACE(5, it);
            }
            // ---- exact rescoring of the candidate groups
            int n_iter = 0;
            int best_bits = -1, best_k = 0;
            float best_u = 0.0f;
            unsigned long long vv[F2 ? kD : 1];
            if constexpr (F2) {
#pragma unroll
                for (int j = 0; j < kD; ++j) vv[j] = pack2(v[j], v[j]);
            }
            // exact scores of the four codewords of group g (ascending-j chain, as hsq_exact.cu)
            auto score_group = [&](int g, float (&p)[kGroup]) {
                if constexpr (F2) {
                    const uint32_t slot = pbase + (uint32_t)g * 256u;   // pair 2g at slot, pair 2g + 1 at slot + 128
                    unsigned long long a01, a23;
#pragma unroll
                    for (int t = 0; t < kD / 2; ++t) {
                        unsigned long long c0, c1, e0, e1;
                        lds_2x64(slot + uo[t], c0, c1);
                        lds_2x64(slot + 128u + uo[t], e0, e1);
                        if (t == 0) {
                            a01 = fmul2(c0, vv[0]);
                            a23 = fmul2(e0, vv[0]);
                        } else {
                            a01 = ffma2(c0, vv[2 * t], a01);
                            a23 = ffma2(e0, vv[2 * t], a23);
                        }
                        a01 = ffma2(c1, vv[2 * t + 1], a01);
                        a23 = ffma2(e1, vv[2 * t + 1], a23);
                    }
                    unpack2(a01, p[0], p[1]);
                    unpack2(a23, p[2], p[3]);
                } else {
                    // unit by unit over the four codewords: four independent ascending-j chains
                    const uint32_t rowa = pbase + (uint32_t)(g * kGroup) * 128u;
#pragma unroll
                    for (int u = 0; u < kUnits; ++u) {
#pragma unroll
                        for (int i = 0; i < kGroup; ++i) {
                            const float4 c = lds_f4(rowa + 128u * i + uo[u]);
                            p[i] = (u == 0) ? __fmul_rn(c.x, v[0]) : __fmaf_rn(c.x, v[4 * u], p[i]);
                            p[i] = __fmaf_rn(c.y, v[4 * u + 1], p[i]);
                            p[i] = __fmaf_rn(c.z, v[4 * u + 2], p[i]);
                            p[i] = __fmaf_rn(c.w, v[4 * u + 3], p[i]);
                        }
                    }
                }
            };
            // group maximum first (3 FMNMX), one compare against the running best, and only a winning
            // group pays for locating its first maximal codeword (first index wins ties: groups ascend)
            auto take_group = [&](int g, const float (&p)[kGroup]) {
                const float gmax = fmaxf(fmaxf(fabsf(p[0]), fabsf(p[1])), fmaxf(fabsf(p[2]), fabsf(p[3])));
                const int gb = __float_as_int(gmax);
                const float psum = (p[0] + p[1]) + (p[2] + p[3]);   // NaN (or inf - inf) takes the slow path
                if (gb > best_bits || psum != psum) {
#pragma unroll
                    for (int i = 0; i < kGroup; ++i) {
                        const int ab = __float_as_int(p[i]) & 0x7fffffff;
                        if (ab > best_bits) { best_bits = ab; best_k = g * kGroup + i; best_u = p[i]; }
                    }
                }
            };
            uint32_t cur = clo, nxt = chi;
            int gbase = 0;
            if (cur == 0u) { cur = nxt; nxt = 0u; gbase = 32; }
            while (cur != 0u) {
                const int g0 = gbase + __ffs((int)cur) - 1;
                cur &= cur - 1u;
                if (cur == 0u) { cur = nxt; nxt = 0u; gbase = 32; }
                if constexpr (R2) {
                    // two candidate groups per pass: their FMA chains interleave (twice the ILP of a
                    // latency-bound loop).  About a fifth of the rows have a second candidate, so nearly
                    // every warp ran a second pass anyway; a row without one rescoring its group twice is
                    // harmless (the repeat never beats the running best).
                    int g1 = g0;
                    if (cur != 0u) {
                        g1 = gbase + __ffs((int)cur) - 1;
                        cur &= cur - 1u;
                        if (cur == 0u) { cur = nxt; nxt = 0u; gbase = 32; }
                    }
                    float p0[kGroup], p1[kGroup];
                    score_group(g0, p0);
                    score_group(g1, p1);
                    take_group(g0, p0);
                    take_group(g1, p1);
                } else {
                    float p0[kGroup];
                    score_group(g0, p0);
                    take_group(g0, p0);
                }
                if (TRACE) ++n_iter;
            }
            __syncwarp();
            if (TRACE) {
                n_iter = (int)__reduce_max_sync(0xffffffffu, (unsigned)n_iter);
                if (tracer) {
                    GQ_TRACE(6, it);
                    if (blockIdx.x == 0 && it < 128) P.trace[8 * 128 + it] = n_iter;
                }
            }
            if (valid) P.u_out[c] = best_u;
            if (codes16) {
                // the warp's 32 codes leave as two 16-byte stores (and, multi-GPU, go to the peers' receive
                // blocks from here: that half of the record crosses NVLink while the search is still running)
                uint8_t *slot = s_codes + (warp - 4) * 32;
                slot[lane] = valid ? (uint8_t)best_k : (uint8_t)0;
                __syncwarp();
                if ((lane & 15) == 0) {
                    const uint4 w = *reinterpret_cast<const uint4 *>(slot + lane);
                    if (c + 15 < n_chunks) {
                        *reinterpret_cast<uint4 *>(P.codes + c) = w;
                    } else {
                        for (int t = 0; t < 16; ++t)
                            if (c + t < n_chunks) P.codes[c + t] = slot[lane + t];
                    }
                    if (P.remote.n > 0 && c < n_chunks) remote_st128(P.remote, P.codes + c, w);
                }
                __syncwarp();
            } else if (valid) {
                P.codes[c] = (uint8_t)best_k;
            }
            if (P.keys != nullptr) {
                if (!keys_ready) {   // CTA 0 has reset the keys; bounded wait, then trap
                    unsigned long long seen;
                    uint32_t spins = 0;
#pragma unroll 1
                    do {
                        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(P.flag) : "memory");
                        if (seen == P.id) break;
                        __nanosleep(64);
                    } while (++spins < (1u << 22));
                    if (seen != P.id) __trap();
                    keys_ready = true;
                }
                const int seg = valid ? cached_segment(segc, P.seg_start, P.n_seg, (int64_t)c) : -1;
                minmax_add_warp(mm, valid, seg, best_u, P.keys);
            }
            if (tracer) GQ_TRACE(7, it);
        }
        if (P.keys != nullptr) minmax_flush_warp(mm, P.keys);
    }

    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    }
    GQ_STAMP(1);
    if (P.l == nullptr) return;

    // =============================================== fused tail: n-bit norm quantization ===
    // Grid barrier: every CTA's min/max atomics are performed before anyone reads lb/ub.  A CTA arrives,
    // then does everything that does not depend on lb/ub WHILE it waits for the slower CTAs: the
    // segment table, the loads of its own u values (and codes / uniforms) and the Philox draws.
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(P.barrier, 1u);
    }
    const int n_seg = P.n_seg;
    int *s_seg = reinterpret_cast<int *>(smem + L::kOffA);                                   // [n_seg + 1]
    float2 *s_lbub = reinterpret_cast<float2 *>(smem + L::kOffA + 4 * ((n_seg + 2) & ~1));   // [n_seg]
    for (int i = threadIdx.x; i <= n_seg; i += kThreads) s_seg[i] = (int)P.seg_start[i];
    const Remote &R = P.remote;
    const int c_begin = tile0 * kTileM;
    const int c_end = min((tile0 + my_tiles) * kTileM, n_chunks);
    const int qb = c_begin >> 2, qe = (c_end + 3) >> 2;
    const float s = P.s;
    const int random = P.random;
    const bool ext = random && P.uniforms != nullptr;
    const bool philox = random && P.uniforms == nullptr;
    const bool philox_aligned = (P.offset & 3u) == 0;
    constexpr int J = 5;   // float4 groups per thread and pass: 512 threads x 5 x 4 = 10240 chunks >= 78 tiles
    // u (and codes / uniforms / Philox draws) of up to J groups of four chunks, q0, q0 + kThreads, ...
    auto load_pass = [&](int q0, float4 (&xv)[J], float4 (&rv)[J]) {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const int q = q0 + j * kThreads;
            xv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            rv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q < qe) {
                if (q * 4 + 3 < n_chunks) {
                    xv[j] = __ldcg(reinterpret_cast<const float4 *>(P.u_out) + q);
                    if (ext) rv[j] = __ldg(reinterpret_cast<const float4 *>(P.uniforms) + q);
                } else {
                    float x[4] = {0.f, 0.f, 0.f, 0.f}, r[4] = {0.f, 0.f, 0.f, 0.f};
                    for (int t = 0; t < 4; ++t) {
                        if (q * 4 + t < n_chunks) {
                            x[t] = __ldcg(P.u_out + q * 4 + t);
                            if (ext) r[t] = __ldg(P.uniforms + q * 4 + t);
                        }
                    }
                    xv[j] = make_float4(x[0], x[1], x[2], x[3]);
                    rv[j] = make_float4(r[0], r[1], r[2], r[3]);
                }
            }
        }
        if (philox) {
#pragma unroll
            for (int j = 0; j < J; ++j) {
                const int q = q0 + j * kThreads;
                if (q >= qe) continue;
                const int i0 = q * 4;
                if (philox_aligned) {
                    const uint4 w = philox4x32_10(P.seed, (P.offset + (uint64_t)i0) >> 2);
                    rv[j] = make_float4(u01(w.x), u01(w.y), u01(w.z), u01(w.w));
                } else {
                    rv[j] = make_float4(philox_uniform(P.seed, P.offset, (uint64_t)i0), philox_uniform(P.seed, P.offset, (uint64_t)(i0 + 1)),
                                        philox_uniform(P.seed, P.offset, (uint64_t)(i0 + 2)), philox_uniform(P.seed, P.offset, (uint64_t)(i0 + 3)));
                }
            }
        }
    };
    // levels of those groups (needs lb/ub: after the barrier), stored locally and -- four lanes' words
    // gathered into one 16-byte store -- at the remote copies (the codes went out from the main loop)
    auto finish_pass = [&](int q0, const float4 (&xv)[J], const float4 (&rv)[J], int &seg) {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const int q = q0 + j * kThreads;
            const bool act = q < qe;
            uint32_t packed = 0u;
            if (act) {
            const int i0 = q * 4;
            const float x[4] = {xv[j].x, xv[j].y, xv[j].z, xv[j].w};
            const float r[4] = {rv[j].x, rv[j].y, rv[j].z, rv[j].w};
            int lv[4];
            psc_levels4(x, r, i0, n_chunks, s_seg, s_lbub, seg, s, random, lv);
            packed = (uint32_t)lv[0] | ((uint32_t)lv[1] << 8) | ((uint32_t)lv[2] << 16) | ((uint32_t)lv[3] << 24);
            if (i0 + 3 < n_chunks) {
                reinterpret_cast<uint32_t *>(P.l)[q] = packed;
            } else {
                for (int t = 0; t < 4; ++t)
                    if (i0 + t < n_chunks) P.l[i0 + t] = (uint8_t)lv[t];
            }
            }
            if (R.n > 0) {   // the record sections are padded to 256 bytes: whole 16-byte words may be written remotely
                const uint32_t p1 = __shfl_down_sync(0xffffffffu, packed, 1), p2 = __shfl_down_sync(0xffffffffu, packed, 2);
                const uint32_t p3 = __shfl_down_sync(0xffffffffu, packed, 3);
                if (act && (threadIdx.x & 3) == 0)
                    remote_st128(R, reinterpret_cast<uint32_t *>(P.l) + q, make_uint4(packed, p1, p2, p3));
            }
        }
    };
    float4 xv[J], rv[J];
    int q0 = qb + (int)threadIdx.x;
    load_pass(q0, xv, rv);
    if (threadIdx.x == 0) {
        uint32_t seen, spins = 0;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(P.barrier) : "memory");
            if (seen >= gridDim.x) break;
            __nanosleep(32);
        } while (++spins < (1u << 24));
        if (seen < gridDim.x) __trap();
    }
    __syncthreads();
    GQ_STAMP(2);
    for (int i = threadIdx.x; i < n_seg; i += kThreads) {
        const float lb = key_to_float(__ldcg(P.keys + 2 * i)), ub = key_to_float(__ldcg(P.keys + 2 * i + 1));
        s_lbub[i] = make_float2(lb, ub);
        if (blockIdx.x == 0) {   // the reference returns lb/ub (probabilistic_scalar_compressor.py:27)
            P.lbub[2 * i] = lb;
            P.lbub[2 * i + 1] = ub;
            if (R.n > 0) {
                remote_st32(R, P.lbub + 2 * i, __float_as_uint(lb));
                remote_st32(R, P.lbub + 2 * i + 1, __float_as_uint(ub));
            }
        }
    }
    __syncthreads();
    {
        int seg = 0;
        {   // segment of this CTA's first chunk (binary search in shared memory)
            int lo = 0, hi = n_seg;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_seg[mid] <= c_begin) lo = mid; else hi = mid;
            }
            seg = lo;
        }
        finish_pass(q0, xv, rv, seg);
        for (q0 += J * kThreads; q0 - (int)threadIdx.x < qe; q0 += J * kThreads) {   // (only when a CTA owns more than 80 tiles)
            load_pass(q0, xv, rv);
            finish_pass(q0, xv, rv, seg);
        }
    }
    if (TRACE) __syncthreads();
    GQ_STAMP(3);
    if (R.n > 0) {
        // identity section (written by the riders of all CTAs before the grid barrier), then the
        // delivery handshake: the last CTA to finish announces the epoch to every rank
        const int64_t n16 = R.ident_bytes >> 4;
        for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n16; i += (int64_t)gridDim.x * kThreads) {
            const uint4 w = __ldcg(reinterpret_cast<const uint4 *>(R.ident) + i);
            remote_st128(R, const_cast<uint8_t *>(R.ident) + 16 * i, w);
        }
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t prev = atomicAdd(R.done, 1u);
            s_misc[0] = (prev == gridDim.x - 1) ? 1 : 0;
            __threadfence_system();
        }
        __syncthreads();
        if (s_misc[0] && (int)threadIdx.x < R.n_flag)
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(R.flag[threadIdx.x]), "r"(R.epoch) : "memory");
    }
}

// ------------------------------------------------------------------ host side ---
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

static int make_map(CUtensorMap *map, const float *base, int64_t rows, int kD = 16)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return GQ_ERR_CUDA;
    }
    cuuint64_t dims[2] = {(cuuint64_t)kD, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)kD * 4};
    cuuint32_t box[2] = {(cuuint32_t)kD, (cuuint32_t)kTileM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE,
                    kD == 8 ? CU_TENSOR_MAP_SWIZZLE_32B : (kD == 16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (base %p, rows %lld)", (int)r, (const void *)base,
                  (long long)rows);
        return GQ_ERR_CUDA;
    }
    return GQ_OK;
}

struct Variant {
    int groups;
    bool pair, fmask, f2, r2;
};

// GQ_TC2 = comma-separated switches, read at every launch (A/B runs): g3 | g4, pair | nopair,
// fmask | nofmask, f2 | nof2, r2 | r1.  Only the combinations instantiated below exist.
static Variant pick_variant()
{
    Variant v = {3, true, true, true, false};   // measured best: 3 groups, pair sums, FMA-pipe mask, FFMA2, one group per pass
    if (const char *e = getenv("GQ_TC2")) {
        if (strstr(e, "g4")) v.groups = 4;
        if (strstr(e, "g3")) v.groups = 3;
        if (strstr(e, "nopair")) v.pair = false; else if (strstr(e, "pair")) v.pair = true;
        if (strstr(e, "nofmask")) v.fmask = false; else if (strstr(e, "fmask")) v.fmask = true;
        if (strstr(e, "nof2")) v.f2 = false; else if (strstr(e, "f2")) v.f2 = true;
        if (strstr(e, "r1")) v.r2 = false; else if (strstr(e, "r2")) v.r2 = true;
    }
    return v;
}

template <int G, bool PAIR, bool FMASK, bool F2, bool R2, int D = 16>
static int launch_one(const CUtensorMap &mg, const Enc2 &P, int grid, cudaStream_t st)
{
    auto kern = hsq_encode_tc2_kernel<G, PAIR, FMASK, F2, R2, false, D>;
    static bool attr_set = false;   // per instantiation
    if (!attr_set) {
        GQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Layout<G, D>::kSmemBytes));
        attr_set = true;
    }
    GQ_CUDA(launch_pdl(kern, dim3(grid), dim3(128 + 128 * G), (size_t)Layout<G, D>::kSmemBytes, st, mg, P));
    return GQ_OK;
}

static int launch_variant(const Variant &v, const CUtensorMap &mg, const Enc2 &P, int grid, cudaStream_t st)
{
    const int sel = (v.groups == 4 ? 16 : 0) | (v.pair ? 8 : 0) | (v.fmask ? 4 : 0) | (v.f2 ? 2 : 0) | (v.r2 ? 1 : 0);
    switch (sel) {
    case 0: return launch_one<3, false, false, false, false>(mg, P, grid, st);   // structural changes only
    case 8: return launch_one<3, true, false, false, false>(mg, P, grid, st);
    case 12: return launch_one<3, true, true, false, false>(mg, P, grid, st);
    case 13: return launch_one<3, true, true, false, true>(mg, P, grid, st);
    case 14: return launch_one<3, true, true, true, false>(mg, P, grid, st);
    case 15: return launch_one<3, true, true, true, true>(mg, P, grid, st);
    case 9: return launch_one<3, true, false, false, true>(mg, P, grid, st);
    case 16 + 14: return launch_one<4, true, true, true, false>(mg, P, grid, st);
    case 16 + 15: return launch_one<4, true, true, true, true>(mg, P, grid, st);
    case 16 + 13: return launch_one<4, true, true, false, true>(mg, P, grid, st);
    case 16 + 12: return launch_one<4, true, true, false, false>(mg, P, grid, st);
    default:
        set_error("GQ_TC2: this combination of switches is not built");
        return GQ_ERR_UNSUPPORTED;
    }
}


}  // namespace tc2

// default variant with the pipeline trace of CTA 0 (9 x 128 int64) followed by four wall-clock stamps
// per CTA (4 x grid int64); search only, or the whole one-launch encode when `tail` is given
int hsq_tc2_trace(const float *grad, int64_t n_chunks, const float *codebook, void *codes, float *u_out,
                  const int64_t *seg_start, int n_seg, uint32_t *keys, uint64_t *flag, uint32_t *barrier,
                  const Tc2Tail *tail, long long *trace, cudaStream_t st)
{
    using namespace tc2;
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0 && ((uintptr_t)codebook & 15) == 0, "TMA needs 16-byte aligned bases");
    GQ_REQUIRE(n_chunks > 0 && n_chunks < ((int64_t)1 << 31) - 256 && trace, "bad arguments");
    CUtensorMap mg;
    int e = make_map(&mg, grad, n_chunks);
    if (e) return e;
    static std::atomic<unsigned long long> counter{0x7ace000000000000ull};
    Enc2 P = {};
    P.codebook = codebook;
    P.n_chunks = (int)n_chunks;
    P.codes = (uint8_t *)codes;
    P.u_out = u_out;
    P.trace = trace;
    if (tail != nullptr) {
        P.seg_start = seg_start;
        P.n_seg = n_seg;
        P.keys = keys;
        P.flag = reinterpret_cast<unsigned long long *>(flag);
        P.id = counter.fetch_add(1) + 1;
        P.l = tail->l;
        P.lbub = tail->lbub;
        P.barrier = barrier;
        P.uniforms = tail->uniforms;
        P.seed = tail->seed;
        P.offset = tail->offset;
        P.s = (float)(1u << tail->n_bit);
        P.random = tail->random;
    }
    const int n_tiles = (int)((n_chunks + kTileM - 1) / kTileM);
    int sms = sm_count();
    if (const char *g = getenv("GQ_TC_GRID")) {
        int v = atoi(g);
        if (v > 0 && v < sms) sms = v;
    }
    const int grid = n_tiles < sms ? n_tiles : sms;
    const Variant v = pick_variant();
    auto launch = [&](auto kern, int threads, size_t smem) -> int {
        GQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GQ_CUDA(launch_pdl(kern, dim3(grid), dim3(threads), smem, st, mg, P));
        return GQ_OK;
    };
    if (v.groups == 4) e = launch(hsq_encode_tc2_kernel<4, true, true, true, true, true>, 640, Layout<4>::kSmemBytes);
    else if (v.r2) e = launch(hsq_encode_tc2_kernel<3, true, true, true, true, true>, 512, Layout<3>::kSmemBytes);
    else e = launch(hsq_encode_tc2_kernel<3, true, true, true, false, true>, 512, Layout<3>::kSmemBytes);
    if (e) return e;
    GQ_LAUNCH_CHECK("hsq_tc2_trace");
    return GQ_OK;
}

bool hsq_tc2_supported(int d, int K, int code_bytes)
{
    return (d == 8 || d == 16 || d == 32) && K == tc2::kK && code_bytes == 1;
}

bool hsq_tc2_tail_supported(int n_seg, int n_bit, int l_bytes, const void *u_out, const void *uniforms, const void *l,
                            const void *codes)
{
    return n_seg <= tc2::kTailMaxSeg && n_bit >= 1 && n_bit <= 7 && l_bytes == 1 && ((uintptr_t)u_out & 15) == 0 &&
           ((uintptr_t)uniforms & 15) == 0 && ((uintptr_t)l & 3) == 0 && ((uintptr_t)codes & 3) == 0;
}

// One-launch encode (or search only when tail == nullptr).  keys == nullptr: no min/max.  flag: 8-byte
// scratch word for the in-kernel key reset; barrier: 2 x uint32 scratch (grid barrier, delivery counter).
int hsq_encode_tc2(const float *grad, int64_t n_chunks, int d, const float *codebook, void *codes, float *u_out,
                   const int64_t *seg_start, int n_seg, uint32_t *keys, uint64_t *flag, uint32_t *barrier,
                   const Rider &rider, const Tc2Tail *tail, const Tc2Remote *remote, cudaStream_t st)
{
    using namespace tc2;
    GQ_REQUIRE(d == 8 || d == 16 || d == 32, "tcgen05 encode: chunk dimension %d (8, 16 or 32)", d);
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0 && ((uintptr_t)codebook & 15) == 0, "TMA needs 16-byte aligned bases");
    GQ_REQUIRE(n_chunks > 0 && n_chunks < ((int64_t)1 << 31) - 256, "n_chunks out of range for one tensor map");
    CUtensorMap mg;
    int e = make_map(&mg, grad, n_chunks, d);
    if (e) return e;
    static std::atomic<unsigned long long> counter{[] {
        unsigned long long seed = (unsigned long long)(uintptr_t)&seed ^ (unsigned long long)clock();
        seed = seed * 6364136223846793005ull + 1442695040888963407ull;
        return (seed >> 16) << 32;
    }()};
    Enc2 P = {};
    P.codebook = codebook;
    P.n_chunks = (int)n_chunks;
    P.codes = (uint8_t *)codes;
    P.u_out = u_out;
    P.seg_start = seg_start;
    P.n_seg = n_seg;
    P.keys = keys;
    P.flag = keys ? reinterpret_cast<unsigned long long *>(flag) : nullptr;
    P.id = counter.fetch_add(1) + 1;
    P.rider = rider;
    if (tail != nullptr) {
        GQ_REQUIRE(keys && flag && barrier, "the fused tail needs keys, flag and barrier scratch");
        P.l = tail->l;
        P.lbub = tail->lbub;
        P.barrier = barrier;
        P.uniforms = tail->uniforms;
        P.seed = tail->seed;
        P.offset = tail->offset;
        P.s = (float)(1u << tail->n_bit);
        P.random = tail->random;
        if (remote != nullptr && remote->n > 0) {
            GQ_REQUIRE(((uintptr_t)codes & 15) == 0 && ((uintptr_t)tail->l & 15) == 0,
                       "remote delivery needs 16-byte aligned codes / l sections");
            Remote &R = P.remote;
            R.n = remote->n;
            R.multicast = remote->multicast;
            for (int i = 0; i < 7; ++i) R.delta[i] = i < remote->n ? remote->delta[i] : 0;
            R.ident = remote->ident;
            R.ident_bytes = remote->ident_bytes;
            R.done = barrier + 1;
            R.n_flag = remote->n_flag;
            for (int i = 0; i < 8; ++i) R.flag[i] = i < remote->n_flag ? remote->flag[i] : nullptr;
            R.epoch = remote->epoch;
        }
    }
    const int n_tiles = (int)((n_chunks + kTileM - 1) / kTileM);
    int sms = sm_count();
    if (const char *g = getenv("GQ_TC_GRID")) {
        int v = atoi(g);
        if (v > 0 && v < sms) sms = v;
    }
    const int grid = n_tiles < sms ? n_tiles : sms;
    if (d == 8) {          // one variant each for the other chunk dimensions (the measured-best switches)
        e = launch_one<3, true, true, true, false, 8>(mg, P, grid, st);
    } else if (d == 32) {
        e = launch_one<3, true, true, false, false, 32>(mg, P, grid, st);
    } else {
        const Variant v = pick_variant();
        e = launch_variant(v, mg, P, grid, st);
    }
    if (e) return e;
    GQ_LAUNCH_CHECK("hsq_encode_tc2");
    return GQ_OK;
}

}  // namespace gq

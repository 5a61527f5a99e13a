// qsgd_sign.cu -- QSGD / TernGrad and SignSGD: HBM-bound elementwise codecs.
//   QSGD   : compressors/qsgd_compressor.py:42-71
//   SignSGD: compressors/signsgd_compressor.py:8-12
// Algorithmic bytes per gradient element: QSGD encode 4 (+4 when uniforms are
// supplied) + bits/8 + 4/dim; QSGD decode-reduce 4 + U*(bits/8 + 4/dim);
// sign encode 4 + 0.25; sign decode-reduce 4 + 0.25 U.
#include "gq_internal.cuh"

namespace gq {

static int grid_for(int64_t n, int per_block, int waves = 8)
{
    int64_t blocks = (n + per_block - 1) / per_block;
    int64_t cap = (int64_t)sm_count() * waves;
    int64_t g = blocks < cap ? blocks : cap;
    return (int)(g < 1 ? 1 : g);
}

// ------------------------------------------------------ peer-to-peer delivery ---
// The one-launch encodes below take `bool DELIVER` as a template parameter: with a remote delivery
// attached (gq_attach_remote_record) they also store every record byte they write at the peers'
// copies of the record, then run the arrival handshake; the DELIVER == false instantiations never
// touch the Remote parameter and compile to the code of an encode without delivery.  These kernels
// have no grid barrier, so
//  - a section whose 32-bit words are written by different lanes or CTAs is sent by read-back: a
//    CTA re-reads (ld.cg) what it wrote after a __syncthreads, and the words it shares with another
//    CTA are sent by the last CTA to arrive, which sees every CTA's stores (deliver_finish);
//  - the arrival counter cannot be zeroed in the prologue: the last CTA to arrive sets it back to 0.
//    The next launch that counts on it runs its atomics after griddepcontrol.wait, i.e. after this
//    grid has completed, reset included.

// Remote copy of the local bytes [p0, p1) that this CTA has written and synchronised: whole 16-byte
// words with one wide store, the 4-byte words before and after one by one.  A 32-bit word that the
// range covers only in part is left to its neighbour's owner (deliver_finish).  Block-collective.
__device__ __forceinline__ void deliver_bytes(const Remote &R, const void *p0, const void *p1)
{
    const uintptr_t a0 = ((uintptr_t)p0 + 3) & ~(uintptr_t)3, a1 = (uintptr_t)p1 & ~(uintptr_t)3;
    if (a0 >= a1) return;
    const uintptr_t v0 = min((a0 + 15) & ~(uintptr_t)15, a1), v1 = max(v0, a1 & ~(uintptr_t)15);
    const uintptr_t t = threadIdx.x, nt = blockDim.x;
    for (uintptr_t a = a0 + 4 * t; a < v0; a += 4 * nt) remote_st32(R, (void *)a, __ldcg((const uint32_t *)a));
    for (uintptr_t a = v0 + 16 * t; a < v1; a += 16 * nt) remote_st128(R, (void *)a, __ldcg((const uint4 *)a));
    for (uintptr_t a = v1 + 4 * t; a < a1; a += 4 * nt) remote_st32(R, (void *)a, __ldcg((const uint32_t *)a));
}
// the 32-bit word of the local record that holds byte p, read back and sent whole
__device__ __forceinline__ void deliver_word(const Remote &R, const void *p)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>((uintptr_t)p & ~(uintptr_t)3);
    remote_st32(R, const_cast<uint32_t *>(w), __ldcg(w));
}

// The identity section, when this launch carries it.  A rider of this launch wrote element i from grid
// thread i (mod threads), the thread that reads it back here; one written by an earlier launch is
// visible after griddepcontrol.wait.  Call after rider_run().
__device__ __forceinline__ void deliver_ident(const Remote &R)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>(R.ident);
    const int64_t nw = R.ident_bytes >> 2, nt = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += nt)
        remote_st32(R, const_cast<uint32_t *>(w + i), __ldcg(w + i));
}

// End of a delivering launch, block-collective: every CTA makes its remote stores visible system-wide
// and arrives on the counter; the last CTA to arrive runs last() (every CTA's local stores are visible
// to it), sends what that wrote, sets the counter back to 0 and stores the epoch into the n_flag flag
// words with st.release.sys (n_flag == 0: an earlier launch of a multi-launch encode, which delivers
// and leaves the announcement to the last launch).
template <typename F>
__device__ __forceinline__ void deliver_finish(const Remote &R, F &&last)
{
    __shared__ int s_last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        s_last = atomicAdd(R.done, 1u) == gridDim.x - 1;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    last();
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) *R.done = 0u;
    __syncthreads();
    if ((int)threadIdx.x < R.n_flag)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(R.flag[threadIdx.x]), "r"(R.epoch) : "memory");
}

// A PeerWait as a template-selected parameter of the fast decodes (WAIT == false: never touched).  With
// WAIT every CTA polls the flags after griddepcontrol.wait and before it reads a record byte, and the
// records are read with ld.global.cg instead of ld.global.nc: the peers write them while this grid is
// resident, and the non-coherent path is only defined for data that is read-only for the kernel's life.
template <bool WAIT>
__device__ __forceinline__ void wait_prologue(const PeerWait &w)
{
    if constexpr (WAIT) {
        if ((int)threadIdx.x < w.n) peer_wait_flag(w.flags + threadIdx.x, w.epoch, w.timeout_ns);
        __syncthreads();
    }
}
template <bool WAIT, typename T>
__device__ __forceinline__ T ld_rec(const T *p)
{
    if constexpr (WAIT) return __ldcg(p);
    else return __ldg(p);
}

__device__ __forceinline__ int64_t chunk_of(const int64_t *__restrict__ chunk_start, int64_t n_chunks,
                                            int dim, int64_t i)
{
    return chunk_start ? (int64_t)find_segment(chunk_start, (int)n_chunks, i) : i / dim;
}

// ------------------------------------------------------------ chunk L-inf ---
// norm[m] = max |v| over chunk m (qsgd_compressor.py:49).  |v| bit patterns are
// monotone as unsigned ints, so one atomicMax per warp (or lane) suffices.
__global__ void __launch_bounds__(256)
chunk_absmax_kernel(const float *__restrict__ v, int64_t n, const int64_t *__restrict__ chunk_start,
                    int64_t n_chunks, int dim, uint32_t *__restrict__ norm_bits)
{
    for (int64_t base = (int64_t)blockIdx.x * 256; base < n; base += (int64_t)gridDim.x * 256) {
        int64_t i = base + threadIdx.x;
        bool valid = i < n;
        uint32_t a = valid ? (__float_as_uint(v[i]) & 0x7fffffffu) : 0u;
        int64_t m = valid ? chunk_of(chunk_start, n_chunks, dim, i) : -1;
        int64_t m0 = __shfl_sync(0xffffffffu, m, 0);
        bool uniform = __all_sync(0xffffffffu, (m == m0) || !valid) && (m0 >= 0);
        if (uniform) {
            uint32_t w = __reduce_max_sync(0xffffffffu, a);
            if ((threadIdx.x & 31) == 0) atomicMax(norm_bits + m0, w);
        } else if (valid) {
            atomicMax(norm_bits + m, a);
        }
    }
}

// --------------------------------------------------------------- quantize ---
// level/sign of one element (qsgd_compressor.py:50-63), exact op order.
// returns level; nan_level flags the 0/0 case (reference: int cast of NaN = INT_MIN).
__device__ __forceinline__ int qsgd_level(float x, float nm, float s, int random, float r, bool &is_nan)
{
    float scaled = fabsf(__fdiv_rn(x, nm)) * s;
    is_nan = (scaled != scaled);
    if (is_nan) return 0;
    float c = fminf(fmaxf(scaled, 0.0f), s - 1.0f);
    int li = (int)c;
    if (random) {
        float prob = __fsub_rn(scaled, (float)li);
        li += (prob > r) ? 1 : 0;
    }
    return li;
}

// same, for the packed wire form (which has no room for the reference's INT_MIN level of a 0/0
// element: a NaN quotient gives level 0 through the same arithmetic -- fmaxf(NaN, 0) = 0 and
// NaN > r is false -- so no branch is needed)
__device__ __forceinline__ uint32_t qsgd_level_packed(float x, float nm, float s, int random, float r)
{
    const float scaled = fabsf(__fdiv_rn(x, nm)) * s;
    const float c = fminf(fmaxf(scaled, 0.0f), s - 1.0f);
    int li = (int)c;
    li += (random && (__fsub_rn(scaled, (float)li) > r)) ? 1 : 0;
    return (uint32_t)li;
}

template <int BITS>  // 0: no packed output; 4, 8, 16
__global__ void __launch_bounds__(256)
qsgd_quantize_kernel(const float *__restrict__ v, int64_t n, const int64_t *__restrict__ chunk_start,
                     int64_t n_chunks, int dim, float s, int random,
                     const float *__restrict__ uniforms, uint64_t seed, uint64_t offset,
                     const float *__restrict__ norm, uint8_t *__restrict__ signs,
                     int32_t *__restrict__ l, void *__restrict__ packed)
{
    const int64_t n4 = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x; q < n4; q += (int64_t)gridDim.x * 256) {
        const int64_t i0 = q * 4;
        float x[4], r[4];
        const bool full = (i0 + 3 < n);
        if (full) {
            float4 t = ld_stream_f4(reinterpret_cast<const float4 *>(v) + q);
            x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) x[t] = (i0 + t < n) ? v[i0 + t] : 0.0f;
        }
        if (random) {
            if (uniforms) {
                if (full) {
                    float4 t = ld_stream_f4(reinterpret_cast<const float4 *>(uniforms) + q);
                    r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
                } else {
#pragma unroll
                    for (int t = 0; t < 4; ++t) r[t] = (i0 + t < n) ? uniforms[i0 + t] : 0.0f;
                }
            } else if (((offset + (uint64_t)i0) & 3u) == 0) {
                uint4 w = philox4x32_10(seed, (offset + (uint64_t)i0) >> 2);
                r[0] = u01(w.x); r[1] = u01(w.y); r[2] = u01(w.z); r[3] = u01(w.w);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) r[t] = philox_uniform(seed, offset, (uint64_t)(i0 + t));
            }
        } else {
            r[0] = r[1] = r[2] = r[3] = 0.0f;
        }
        uint32_t pk[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int64_t i = i0 + t;
            if (i >= n) { pk[t] = 0; continue; }
            const int64_t m = chunk_of(chunk_start, n_chunks, dim, i);
            const float nm = __ldg(norm + m);
            bool is_nan;
            int li = qsgd_level(x[t], nm, s, random, r[t], is_nan);
            const uint32_t sg = (x[t] > 0.0f) ? 1u : 0u;
            if (signs) signs[i] = (uint8_t)sg;
            if (l) l[i] = is_nan ? (int32_t)0x80000000 : li;
            pk[t] = (BITS > 0) ? ((sg << (BITS - 1)) | (uint32_t)li) : 0u;
        }
        if (BITS == 4) {
            reinterpret_cast<uint16_t *>(packed)[q] =
                (uint16_t)(pk[0] | (pk[1] << 4) | (pk[2] << 8) | (pk[3] << 12));
        } else if (BITS == 8) {
            reinterpret_cast<uint32_t *>(packed)[q] = pk[0] | (pk[1] << 8) | (pk[2] << 16) | (pk[3] << 24);
        } else if (BITS == 16) {
            reinterpret_cast<uint2 *>(packed)[q] = make_uint2(pk[0] | (pk[1] << 16), pk[2] | (pk[3] << 16));
        }
    }
}


// ------------------------------------------------- fast encode, chunked groups ---
// dim % 4 == 0 and dim <= 2048 (every c_dim the reference is run with: 128 -> 192 -> 288 ...):
// LPC lanes own one chunk at a time and keep it in registers (NV float4 per lane), so the gradient
// is read ONCE: chunk L-inf norm by shuffles, then level / sign / packed store from the registers.
// One launch, no memset, no atomics, no per-element division for the chunk index.
template <int BITS>
__device__ __forceinline__ void qsgd_store_packed(void *__restrict__ packed, int64_t q, const uint32_t (&pk)[4])
{
    if (BITS == 4) {
        reinterpret_cast<uint16_t *>(packed)[q] = (uint16_t)(pk[0] | (pk[1] << 4) | (pk[2] << 8) | (pk[3] << 12));
    } else if (BITS == 8) {
        reinterpret_cast<uint32_t *>(packed)[q] = pk[0] | (pk[1] << 8) | (pk[2] << 16) | (pk[3] << 24);
    } else {
        reinterpret_cast<uint2 *>(packed)[q] = make_uint2(pk[0] | (pk[1] << 16), pk[2] | (pk[3] << 16));
    }
}

// four uniforms for elements i0 .. i0 + 3 (i0 % 4 == 0): caller-supplied stream or Philox
__device__ __forceinline__ void qsgd_uniforms4(int random, const float *__restrict__ uniforms, uint64_t seed,
                                               uint64_t offset, int64_t i0, float (&r)[4])
{
    r[0] = r[1] = r[2] = r[3] = 0.0f;
    if (!random) return;
    if (uniforms) {
        if ((reinterpret_cast<uintptr_t>(uniforms) & 15) == 0) {
            const float4 t = ld_stream_f4(reinterpret_cast<const float4 *>(uniforms + i0));
            r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) r[t] = uniforms[i0 + t];
        }
    } else if (((offset + (uint64_t)i0) & 3u) == 0) {
        const uint4 w = philox4x32_10(seed, (offset + (uint64_t)i0) >> 2);
        r[0] = u01(w.x); r[1] = u01(w.y); r[2] = u01(w.z); r[3] = u01(w.w);
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) r[t] = philox_uniform(seed, offset, (uint64_t)(i0 + t));
    }
}

template <int BITS, int NV, int LPC, int UNR, bool DELIVER>
__global__ void __launch_bounds__(256)
qsgd_encode_chunks_kernel(const float *__restrict__ v, int64_t n_chunks, int dim, float s, int random,
                          const float *__restrict__ uniforms, uint64_t seed, uint64_t offset,
                          float *__restrict__ norm, void *__restrict__ packed, const Rider rider, const Remote R)
{
    pdl_launch_dependents();
    const int dim4 = dim >> 2;
    const int sub = threadIdx.x & (LPC - 1);
    constexpr int SPB = 256 / LPC;   // chunk slots per CTA
    const int64_t n_slots = (int64_t)gridDim.x * SPB;
    const int64_t slot = ((int64_t)blockIdx.x * 256 + threadIdx.x) / LPC;
    const int64_t warp_slot0 = (((int64_t)blockIdx.x * 256 + threadIdx.x) & ~31ll) / LPC;
    // a delivering CTA ends every iteration with a __syncthreads: a CTA-uniform trip count
    const int64_t first_slot = DELIVER ? (int64_t)blockIdx.x * SPB : warp_slot0;
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    if constexpr (DELIVER) deliver_ident(R);
    for (int64_t base = 0; base + first_slot < n_chunks; base += n_slots * UNR) {   // warp-uniform trip count
        float4 x[UNR][NV];
        int64_t c[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            c[u] = base + (int64_t)u * n_slots + slot;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                const int j = sub + t * LPC;
                x[u][t] = (c[u] < n_chunks && j < dim4)
                              ? ld_stream_f4(reinterpret_cast<const float4 *>(v) + c[u] * dim4 + j)
                              : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            uint32_t a = 0u;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                a = max(a, __float_as_uint(x[u][t].x) & 0x7fffffffu);
                a = max(a, __float_as_uint(x[u][t].y) & 0x7fffffffu);
                a = max(a, __float_as_uint(x[u][t].z) & 0x7fffffffu);
                a = max(a, __float_as_uint(x[u][t].w) & 0x7fffffffu);
            }
#pragma unroll
            for (int o = LPC / 2; o > 0; o >>= 1) a = max(a, __shfl_xor_sync(0xffffffffu, a, o));
            const float nm = __uint_as_float(a);
            if (c[u] >= n_chunks) continue;
            if (sub == 0) norm[c[u]] = nm;
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                const int j = sub + t * LPC;
                if (j >= dim4) continue;
                const int64_t q = c[u] * dim4 + j;
                float r[4];
                qsgd_uniforms4(random, uniforms, seed, offset, q * 4, r);
                const float xe[4] = {x[u][t].x, x[u][t].y, x[u][t].z, x[u][t].w};
                uint32_t pk[4];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    pk[e] = ((xe[e] > 0.0f ? 1u : 0u) << (BITS - 1)) | qsgd_level_packed(xe[e], nm, s, random, r[e]);
                qsgd_store_packed<BITS>(packed, q, pk);
            }
        }
        if constexpr (DELIVER) {
            // this iteration's UNR runs of SPB consecutive chunks, read back: norms and packed levels
            __syncthreads();
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int64_t c0 = base + (int64_t)u * n_slots + (int64_t)blockIdx.x * SPB;
                if (c0 >= n_chunks) break;
                const int64_t c1 = min(c0 + SPB, n_chunks);
                deliver_bytes(R, norm + c0, norm + c1);
                deliver_bytes(R, static_cast<uint8_t *>(packed) + c0 * dim4 * (BITS / 2),
                              static_cast<uint8_t *>(packed) + c1 * dim4 * (BITS / 2));
            }
        }
    }
    if constexpr (DELIVER) {
        deliver_finish(R, [&] {
            // the 32-bit words two runs share (4-bit wire, dim / 4 odd: a run boundary falls mid-word),
            // and a last word that the section ends inside (sent whole: the section is padded to 4 bytes)
            if (BITS == 4 && (dim4 & 1)) {
                const int64_t n_runs = (n_chunks + SPB - 1) / SPB;
                for (int64_t k = 1 + threadIdx.x; k <= n_runs; k += blockDim.x) {
                    const int64_t b = min(k * SPB, n_chunks) * dim4 * 2;
                    if (b & 2) deliver_word(R, static_cast<uint8_t *>(packed) + b);
                }
            }
        });
    }
}

// ------------------------------------- fast encode, explicit chunk boundaries ---
// TernGrad (one chunk per tensor): every warp walks increasing addresses of one CTA-owned range, so
// the chunk of its elements changes a handful of times: running maximum in registers and one
// atomicMax per (warp, chunk) in the first kernel, one norm load per chunk change in the second.
constexpr int kRangeTable = 1023;   // tensors per group whose boundaries fit the shared-memory table
template <int UN>
__global__ void __launch_bounds__(256)
seg_absmax_ranges_kernel(const float *__restrict__ v, int64_t n, const int64_t *__restrict__ chunk_start,
                         int n_chunks, uint32_t *__restrict__ norm_bits, const Rider rider)
{
    pdl_launch_dependents();
    // every CTA owns a contiguous range, its eight warps take the spans of that range in turn (the
    // CTA streams 8 consecutive spans at a time; a warp still sees increasing addresses)
    const int lane = threadIdx.x & 31;
    const int64_t span = 128 * UN;
    const int64_t R = ((n + gridDim.x - 1) / gridDim.x + 8 * span - 1) / (8 * span) * (8 * span);
    const int64_t e_begin = (int64_t)blockIdx.x * R + (threadIdx.x >> 5) * span, e_end = min(n, (int64_t)(blockIdx.x + 1) * R);
    // (a moving front -- the whole grid on adjacent spans, a flush per iteration -- measured 53-60 us against
    //  35-39 us for the ranges; eight loads per thread instead of four: 67 us)
    // tensor boundaries in shared memory: the lookup at a boundary is a binary search of shared-memory
    // loads instead of dependent L2 round trips (the table belongs to the plan: readable before the wait)
    __shared__ int64_t s_start[kRangeTable + 1];
    const bool tab = n_chunks <= kRangeTable;
    if (tab) {
        for (int i = threadIdx.x; i <= n_chunks; i += 256) s_start[i] = __ldg(chunk_start + i);
        __syncthreads();
    }
    SegCache sc;
    int cur = -1;
    uint32_t cur_max = 0u;
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    auto flush = [&]() {
        if (cur >= 0) {
            const uint32_t w = __reduce_max_sync(0xffffffffu, cur_max);
            if (lane == 0) atomicMax(norm_bits + cur, w);
        }
        cur = -1;
        cur_max = 0u;
    };
    for (int64_t e0 = e_begin; e0 < e_end; e0 += 8 * span) {
        const int64_t e1 = min(e0 + span, e_end);
        float4 x[UN];
        if (e0 + span <= e_end) {   // whole span inside the range (warp-uniform): UN independent loads in flight
#pragma unroll
            for (int t = 0; t < UN; ++t) x[t] = ld_stream_f4(reinterpret_cast<const float4 *>(v + e0 + 4 * (lane + 32 * t)));
        } else {
#pragma unroll
            for (int t = 0; t < UN; ++t) {
                const int64_t i0 = e0 + 4 * (lane + 32 * t);
                float y[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) y[k] = (i0 + k < e1) ? v[i0 + k] : 0.0f;
                x[t] = make_float4(y[0], y[1], y[2], y[3]);
            }
        }
        const int first = tab ? cached_segment_smem(sc, s_start, n_chunks, e0) : cached_segment(sc, chunk_start, n_chunks, e0);
        if (e1 <= sc.hi) {   // the whole span lies in one chunk (warp-uniform)
            if (first != cur) { flush(); cur = first; }
#pragma unroll
            for (int t = 0; t < UN; ++t) {
                cur_max = max(cur_max, __float_as_uint(x[t].x) & 0x7fffffffu);
                cur_max = max(cur_max, __float_as_uint(x[t].y) & 0x7fffffffu);
                cur_max = max(cur_max, __float_as_uint(x[t].z) & 0x7fffffffu);
                cur_max = max(cur_max, __float_as_uint(x[t].w) & 0x7fffffffu);
            }
        } else {             // a chunk boundary inside the span: per element
            flush();
#pragma unroll
            for (int t = 0; t < UN; ++t) {
                const int64_t i0 = e0 + 4 * (lane + 32 * t);
                const float y[4] = {x[t].x, x[t].y, x[t].z, x[t].w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (i0 + k < e1)
                        atomicMax(norm_bits + (tab ? find_segment_smem(s_start, n_chunks, i0 + k)
                                                   : find_segment(chunk_start, n_chunks, i0 + k)),
                                  __float_as_uint(y[k]) & 0x7fffffffu);
            }
        }
    }
    flush();
}

template <int BITS, int UN, bool DELIVER>
__global__ void __launch_bounds__(256)
qsgd_quantize_ranges_kernel(const float *__restrict__ v, int64_t n, const int64_t *__restrict__ chunk_start,
                            int n_chunks, float s, int random, const float *__restrict__ uniforms,
                            uint64_t seed, uint64_t offset, const float *__restrict__ norm,
                            void *__restrict__ packed, const Remote rem)
{
    pdl_launch_dependents();
    // every CTA owns a contiguous range, its eight warps take the spans of that range in turn (the
    // CTA streams 8 consecutive spans at a time; a warp still sees increasing addresses)
    const int lane = threadIdx.x & 31;
    const int64_t span = 128 * UN;
    const int64_t R = ((n + gridDim.x - 1) / gridDim.x + 8 * span - 1) / (8 * span) * (8 * span);
    const int64_t e_begin = (int64_t)blockIdx.x * R + (threadIdx.x >> 5) * span, e_end = min(n, (int64_t)(blockIdx.x + 1) * R);
    __shared__ int64_t s_start[kRangeTable + 1];
    const bool tab = n_chunks <= kRangeTable;
    if (tab) {
        for (int i = threadIdx.x; i <= n_chunks; i += 256) s_start[i] = __ldg(chunk_start + i);
        __syncthreads();
    }
    SegCache sc;
    int cur = -1;
    float nm_cur = 0.0f;
    pdl_wait();
    if constexpr (DELIVER) {
        // the per-tensor norms are final once the first pass has completed (atomicMax), and so is the
        // identity section its rider wrote
        deliver_ident(rem);
        if (blockIdx.x == 0)
            for (int i = threadIdx.x; i < n_chunks; i += 256)
                remote_st32(rem, const_cast<float *>(norm) + i, __float_as_uint(__ldcg(norm + i)));
    }
    for (int64_t e0 = e_begin; e0 < e_end; e0 += 8 * span) {
        const int64_t e1 = min(e0 + span, e_end);
        float4 x[UN];
        if (e0 + span <= e_end) {   // whole span inside the range (warp-uniform): UN independent loads in flight
#pragma unroll
            for (int t = 0; t < UN; ++t) x[t] = ld_stream_f4(reinterpret_cast<const float4 *>(v + e0 + 4 * (lane + 32 * t)));
        } else {
#pragma unroll
            for (int t = 0; t < UN; ++t) {
                const int64_t i0 = e0 + 4 * (lane + 32 * t);
                float y[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) y[k] = (i0 + k < e1) ? v[i0 + k] : 0.0f;
                x[t] = make_float4(y[0], y[1], y[2], y[3]);
            }
        }
        const int first = tab ? cached_segment_smem(sc, s_start, n_chunks, e0) : cached_segment(sc, chunk_start, n_chunks, e0);
        const bool uniform = e1 <= sc.hi;
        if (uniform && first != cur) {
            cur = first;
            nm_cur = __ldcg(norm + first);
        }
#pragma unroll
        for (int t = 0; t < UN; ++t) {
            const int64_t i0 = e0 + 4 * (lane + 32 * t);
            if (i0 >= e1) continue;
            float r[4];
            if (i0 + 3 < n) {   // (always, except in the last float4 group of the gradient)
                qsgd_uniforms4(random, uniforms, seed, offset, i0, r);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    r[k] = (!random || i0 + k >= n) ? 0.0f
                           : (uniforms ? uniforms[i0 + k] : philox_uniform(seed, offset, (uint64_t)(i0 + k)));
            }
            const float y[4] = {x[t].x, x[t].y, x[t].z, x[t].w};
            uint32_t pk[4];
            if (uniform && i0 + 3 < e1) {   // the common case: four elements of one tensor, no per-element branches
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    pk[k] = ((y[k] > 0.0f ? 1u : 0u) << (BITS - 1)) | qsgd_level_packed(y[k], nm_cur, s, random, r[k]);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (i0 + k >= e1) { pk[k] = 0u; continue; }
                    const float nm = uniform ? nm_cur
                                             : __ldcg(norm + (tab ? find_segment_smem(s_start, n_chunks, i0 + k)
                                                                  : find_segment(chunk_start, n_chunks, i0 + k)));
                    pk[k] = ((y[k] > 0.0f ? 1u : 0u) << (BITS - 1)) | qsgd_level_packed(y[k], nm, s, random, r[k]);
                }
            }
            qsgd_store_packed<BITS>(packed, i0 >> 2, pk);
        }
    }
    if constexpr (DELIVER) {
        // the CTA's packed range (R is a multiple of 4096 elements: interior ends are 16-byte aligned)
        uint8_t *pb = static_cast<uint8_t *>(packed);
        const int64_t q_end = (n + 3) >> 2;
        const int64_t qa = min((int64_t)blockIdx.x * R / 4, q_end), qz = min((int64_t)(blockIdx.x + 1) * R / 4, q_end);
        __syncthreads();
        deliver_bytes(rem, pb + qa * (BITS / 2), pb + qz * (BITS / 2));
        deliver_finish(rem, [&] {
            if ((q_end * (BITS / 2)) & 3) deliver_word(rem, pb + q_end * (BITS / 2));   // the section ends mid-word
        });
    }
}

int qsgd_wire_bits(int n_bit) { return n_bit <= 2 ? 4 : (n_bit <= 6 ? 8 : 16); }

// The pending remote delivery as the kernels take it.  An identity section to mirror must be the one a
// rider of the same launch writes (thread i of the grid reads back element i), or one an earlier launch wrote.
static int device_remote(const Tc2Remote &t, const Rider &rider, Remote *R)
{
    GQ_REQUIRE(t.counter != nullptr, "a delivering sign / QSGD encode needs an arrival counter (gq_attach_delivery_counter)");
    GQ_REQUIRE(rider.n == 0 || t.ident_bytes == 0 || (const void *)rider.out == (const void *)t.ident,
               "the identity section to deliver is not the one this encode's rider writes");
    *R = Remote{};
    R->n = t.n;
    R->multicast = t.multicast;
    for (int i = 0; i < 7; ++i) R->delta[i] = i < t.n ? t.delta[i] : 0;
    R->ident = t.ident;
    R->ident_bytes = t.ident_bytes;
    R->done = t.counter;
    R->n_flag = t.n_flag;
    for (int i = 0; i < 8; ++i) R->flag[i] = i < t.n_flag ? t.flag[i] : nullptr;
    R->epoch = t.epoch;
    return GQ_OK;
}

// remote: the pending delivery (n == 0: none).  Only the one-launch chunked kernel and the TernGrad range
// kernels deliver; a call that would take another path returns GQ_ERR_UNSUPPORTED before it launches anything.
int qsgd_encode(const float *grad, int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim,
                int n_bit, int random, const float *uniforms, uint64_t seed, uint64_t offset, float *norm,
                uint8_t *signs, int32_t *l, void *packed, const Tc2Remote &remote, cudaStream_t st)
{
    const bool deliver = remote.n > 0;
    const float s = (float)(1u << n_bit);
    const bool fast_ok = packed && !signs && !l && ((uintptr_t)packed & 15) == 0 && n_chunks < (1ll << 31);
    const bool chunked = fast_ok && !chunk_start && dim % 4 == 0 && dim <= 2048;
    const bool ranges = fast_ok && chunk_start && ((uintptr_t)grad & 15) == 0;
    if (deliver && (n == 0 || !(chunked || ranges))) {
        set_error("a remote delivery is attached, but this QSGD encode takes the generic kernels (packed output only, "
                  "16-byte aligned, dim %% 4 == 0 and dim <= 2048, or explicit chunk boundaries)");
        return GQ_ERR_UNSUPPORTED;
    }
    if (n == 0) return GQ_OK;
    if (chunked) {
        // one launch: chunk norms and packed levels from registers
        const Rider rider = take_rider();   // a pending identity copy rides in this launch
        Remote R = {};
        if (deliver) GQ_CUDA_INT(device_remote(remote, rider, &R));
        const int b = qsgd_wire_bits(n_bit);
        const int dim4 = dim / 4;
        const int lpc = dim4 <= 8 ? 8 : 32;
        const int nv = lpc == 8 ? 1 : (dim4 <= 32 ? 1 : dim4 <= 64 ? 2 : dim4 <= 128 ? 4 : dim4 <= 256 ? 8 : 16);
        const int unr = nv == 1 ? 4 : (nv == 2 ? 2 : 1);
        const int64_t per_block = (int64_t)(256 / lpc) * unr;
        const int grid = grid_for(n_chunks, (int)per_block, 16);
#define GQ_E(B, NV, LPC, UNR)                                                                                           \
        GQ_CUDA(deliver ? launch_pdl(qsgd_encode_chunks_kernel<B, NV, LPC, UNR, true>, dim3(grid), dim3(256), 0, st,   \
                                     grad, n_chunks, dim, s, random, uniforms, seed, offset, norm, packed, rider, R)   \
                        : launch_pdl(qsgd_encode_chunks_kernel<B, NV, LPC, UNR, false>, dim3(grid), dim3(256), 0, st,  \
                                     grad, n_chunks, dim, s, random, uniforms, seed, offset, norm, packed, rider, R))
#define GQ_EB(B)                                                  \
        do {                                                      \
            if (lpc == 8) GQ_E(B, 1, 8, 4);                       \
            else if (nv == 1) GQ_E(B, 1, 32, 4);                  \
            else if (nv == 2) GQ_E(B, 2, 32, 2);                  \
            else if (nv == 4) GQ_E(B, 4, 32, 1);                  \
            else if (nv == 8) GQ_E(B, 8, 32, 1);                  \
            else GQ_E(B, 16, 32, 1);                              \
        } while (0)
        if (b == 4) GQ_EB(4);
        else if (b == 8) GQ_EB(8);
        else GQ_EB(16);
#undef GQ_EB
#undef GQ_E
        GQ_LAUNCH_CHECK("qsgd_encode_chunks");
        return GQ_OK;
    }
    GQ_CUDA(cudaMemsetAsync(norm, 0, (size_t)n_chunks * 4, st));
    if (ranges) {
        // explicit chunk boundaries (TernGrad): contiguous range per warp, two launches
        // one CTA-contiguous range per CTA and exactly ONE wave: the grid is the number of CTAs that are
        // resident at once (8 per SM asked for 1184 CTAs of which 5 / 4 per SM fit: a second, 60 % full wave)
        const int b = qsgd_wire_bits(n_bit);
        auto one_wave = [&](auto kern) {
            static int per_sm = 0;   // per kernel instantiation (generic lambda)
            if (per_sm == 0 &&
                (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0) != cudaSuccess || per_sm < 1))
                per_sm = 4;
            return grid_for(n, 256 * 4 * 4, per_sm);
        };
        const int grid_a = one_wave(seg_absmax_ranges_kernel<4>);
        const Rider rider = take_rider();   // a pending identity copy rides in the first pass
        Remote R = {};   // the second pass delivers (the norms are final only after the first)
        if (deliver) GQ_CUDA_INT(device_remote(remote, rider, &R));
        GQ_CUDA(launch_pdl(seg_absmax_ranges_kernel<4>, dim3(grid_a), dim3(256), 0, st, grad, n, chunk_start, (int)n_chunks,
                           reinterpret_cast<uint32_t *>(norm), rider));
#define GQ_R(B, D) GQ_CUDA(launch_pdl(qsgd_quantize_ranges_kernel<B, 4, D>, dim3(one_wave(qsgd_quantize_ranges_kernel<B, 4, D>)), dim3(256), 0, st, \
                                      grad, n, chunk_start, (int)n_chunks, s, random, uniforms, seed, offset, (const float *)norm, packed, R))
#define GQ_RB(B) do { if (deliver) GQ_R(B, true); else GQ_R(B, false); } while (0)
        if (b == 4) GQ_RB(4);
        else if (b == 8) GQ_RB(8);
        else GQ_RB(16);
#undef GQ_RB
#undef GQ_R
        GQ_LAUNCH_CHECK("qsgd_quantize_ranges");
        return GQ_OK;
    }
    chunk_absmax_kernel<<<grid_for(n, 256), 256, 0, st>>>(grad, n, chunk_start, n_chunks, dim,
                                                          reinterpret_cast<uint32_t *>(norm));
    GQ_LAUNCH_CHECK("chunk_absmax");
    const int grid = grid_for((n + 3) / 4, 256);
    const int bits = packed ? qsgd_wire_bits(n_bit) : 0;
#define GQ_Q(B) qsgd_quantize_kernel<B><<<grid, 256, 0, st>>>(grad, n, chunk_start, n_chunks, dim, s, random, uniforms, seed, offset, norm, signs, l, packed)
    if (bits == 0) GQ_Q(0);
    else if (bits == 4) GQ_Q(4);
    else if (bits == 8) GQ_Q(8);
    else GQ_Q(16);
#undef GQ_Q
    GQ_LAUNCH_CHECK("qsgd_quantize");
    return GQ_OK;
}

// ----------------------------------------------------------------- decode ---
// value = (float(l) * (2*sign - 1)) * norm / s   (qsgd_compressor.py:69-70)
__device__ __forceinline__ float qsgd_value(int li, uint32_t sg, float nm, float s)
{
    float sv = __fmul_rn((float)li, __fsub_rn(__fmul_rn(2.0f, (float)sg), 1.0f));
    return __fdiv_rn(__fmul_rn(sv, nm), s);
}

template <int BITS>
__global__ void __launch_bounds__(256)
qsgd_decode_reduce_kernel(const float *__restrict__ norm, const void *__restrict__ packed,
                          int64_t user_stride, int n_users, int64_t n,
                          const int64_t *__restrict__ chunk_start, int64_t n_chunks, int dim, float s,
                          int mean, int accumulate, float *__restrict__ out)
{
    const int64_t n4 = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x; q < n4; q += (int64_t)gridDim.x * 256) {
        const int64_t i0 = q * 4;
        int64_t m[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) m[t] = (i0 + t < n) ? chunk_of(chunk_start, n_chunks, dim, i0 + t) : 0;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int u = 0; u < n_users; ++u) {
            const char *pu = reinterpret_cast<const char *>(packed) + u * user_stride;
            const float *nu = reinterpret_cast<const float *>(reinterpret_cast<const char *>(norm) + u * user_stride);
            uint32_t pk[4];
            if (BITS == 4) {
                uint32_t w = reinterpret_cast<const uint16_t *>(pu)[q];
                pk[0] = w & 15u; pk[1] = (w >> 4) & 15u; pk[2] = (w >> 8) & 15u; pk[3] = (w >> 12) & 15u;
            } else if (BITS == 8) {
                uint32_t w = reinterpret_cast<const uint32_t *>(pu)[q];
                pk[0] = w & 255u; pk[1] = (w >> 8) & 255u; pk[2] = (w >> 16) & 255u; pk[3] = w >> 24;
            } else {
                uint2 w = reinterpret_cast<const uint2 *>(pu)[q];
                pk[0] = w.x & 0xffffu; pk[1] = w.x >> 16; pk[2] = w.y & 0xffffu; pk[3] = w.y >> 16;
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const uint32_t sg = pk[t] >> (BITS - 1);
                const int li = (int)(pk[t] & ((1u << (BITS - 1)) - 1u));
                float val = qsgd_value(li, sg, __ldg(nu + m[t]), s);
                acc[t] = (u == 0) ? val : __fadd_rn(acc[t], val);
            }
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (i0 + t >= n) continue;
            float r = acc[t];
            if (mean) r = __fdiv_rn(r, (float)n_users);
            if (accumulate) r = (accumulate == 2) ? __fsub_rn(out[i0 + t], r) : __fadd_rn(out[i0 + t], r);
            out[i0 + t] = r;
        }
    }
}

// Fast decode-and-reduce: 8 consecutive elements per thread (one 32 / 64 / 128-bit word of packed
// levels per user, two float4 stores), the chunk index from one 32-bit division per thread (or the
// thread's cached segment), "/ s" and a power-of-two "/ U" as exact multiplications by 2^-k.
template <int BITS, int U_, bool WAIT>   // U_ > 0: number of users at compile time
__global__ void __launch_bounds__(256)
qsgd_decode_reduce8_kernel(const float *__restrict__ norm, const void *__restrict__ packed, int64_t user_stride,
                           int n_users_rt, int64_t n, const int64_t *__restrict__ chunk_start, int n_chunks,
                           uint32_t dim, float inv_s, float inv_u, float div_u, int accumulate,
                           float *__restrict__ out, const Rider rider, const PeerWait wait)
{
    pdl_launch_dependents();
    const int n_users = U_ > 0 ? U_ : n_users_rt;
    const int64_t n8 = n >> 3;
    SegCache sc;
    pdl_wait();
    wait_prologue<WAIT>(wait);   // the peers' delivery flags, before any record byte is read
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 255) {
        // the last n % 8 elements, one by one
        for (int64_t i = n8 * 8; i < n; ++i) {
            const int m = chunk_start ? find_segment(chunk_start, n_chunks, i) : (int)((uint64_t)i / dim);
            float acc = 0.0f;
            for (int u = 0; u < n_users; ++u) {
                const uint8_t *pu = reinterpret_cast<const uint8_t *>(packed) + u * user_stride;
                const float *nu = reinterpret_cast<const float *>(reinterpret_cast<const char *>(norm) + u * user_stride);
                uint32_t pk;
                if (BITS == 4) pk = (pu[i >> 1] >> (4 * (i & 1))) & 15u;
                else if (BITS == 8) pk = pu[i];
                else pk = reinterpret_cast<const uint16_t *>(pu)[i];
                const uint32_t sg = pk >> (BITS - 1);
                const float lf = (float)(int)(pk & ((1u << (BITS - 1)) - 1u));
                const float val = __fmul_rn(__fmul_rn(__fmul_rn(lf, sg ? 1.0f : -1.0f), nu[m]), inv_s);
                acc = (u == 0) ? val : __fadd_rn(acc, val);
            }
            if (inv_u != 0.0f) acc = __fmul_rn(acc, inv_u);
            else if (div_u != 0.0f) acc = __fdiv_rn(acc, div_u);
            if (accumulate) acc = (accumulate == 2) ? __fsub_rn(out[i], acc) : __fadd_rn(out[i], acc);
            out[i] = acc;
        }
    }
    for (int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x; q < n8; q += (int64_t)gridDim.x * 256) {
        const int64_t i0 = q * 8;
        int m[8];
        bool uni;
        if (chunk_start) {
            m[0] = cached_segment(sc, chunk_start, n_chunks, i0);
            uni = i0 + 7 < sc.hi;
            if (!uni) {
#pragma unroll
                for (int t = 1; t < 8; ++t) m[t] = find_segment(chunk_start, n_chunks, i0 + t);
            }
        } else {
            m[0] = (int)((uint64_t)i0 / dim);
            uni = (uint32_t)((uint64_t)i0 - (uint64_t)m[0] * dim) + 7u < dim;
            if (!uni) {
#pragma unroll
                for (int t = 1; t < 8; ++t) m[t] = (int)((uint64_t)(i0 + t) / dim);
            }
        }
        float acc[8];
#pragma unroll
        for (int u = 0; u < (U_ > 0 ? U_ : 8); ++u) {
            if (u >= n_users) break;
            const char *pu = reinterpret_cast<const char *>(packed) + u * user_stride;
            const float *nu = reinterpret_cast<const float *>(reinterpret_cast<const char *>(norm) + u * user_stride);
            uint32_t pk[8];
            if (BITS == 4) {
                const uint32_t w = ld_rec<WAIT>(reinterpret_cast<const uint32_t *>(pu) + q);
#pragma unroll
                for (int t = 0; t < 8; ++t) pk[t] = (w >> (4 * t)) & 15u;
            } else if (BITS == 8) {
                const uint2 w = ld_rec<WAIT>(reinterpret_cast<const uint2 *>(pu) + q);
#pragma unroll
                for (int t = 0; t < 4; ++t) { pk[t] = (w.x >> (8 * t)) & 255u; pk[4 + t] = (w.y >> (8 * t)) & 255u; }
            } else {
                const uint4 w = ld_rec<WAIT>(reinterpret_cast<const uint4 *>(pu) + q);
                pk[0] = w.x & 0xffffu; pk[1] = w.x >> 16; pk[2] = w.y & 0xffffu; pk[3] = w.y >> 16;
                pk[4] = w.z & 0xffffu; pk[5] = w.z >> 16; pk[6] = w.w & 0xffffu; pk[7] = w.w >> 16;
            }
            const float nm0 = ld_rec<WAIT>(nu + m[0]);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const float nm = uni ? nm0 : ld_rec<WAIT>(nu + m[t]);
                const uint32_t sg = pk[t] >> (BITS - 1);
                const float lf = (float)(int)(pk[t] & ((1u << (BITS - 1)) - 1u));
                // (float(l) * (2 * sign - 1)) * norm / s, qsgd_compressor.py:69-70
                const float val = __fmul_rn(__fmul_rn(__fmul_rn(lf, sg ? 1.0f : -1.0f), nm), inv_s);
                acc[t] = (u == 0) ? val : __fadd_rn(acc[t], val);
            }
        }
        float4 o[2];
        float *of = reinterpret_cast<float *>(o);
        if (accumulate) {
            o[0] = reinterpret_cast<const float4 *>(out)[2 * q];
            o[1] = reinterpret_cast<const float4 *>(out)[2 * q + 1];
        }
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            float r = acc[t];
            if (inv_u != 0.0f) r = __fmul_rn(r, inv_u);
            else if (div_u != 0.0f) r = __fdiv_rn(r, div_u);
            if (accumulate) r = (accumulate == 2) ? __fsub_rn(of[t], r) : __fadd_rn(of[t], r);
            of[t] = r;
        }
        reinterpret_cast<float4 *>(out)[2 * q] = o[0];
        reinterpret_cast<float4 *>(out)[2 * q + 1] = o[1];
    }
}

// mean over U users: exact multiplication by 1/U when U is a power of two, IEEE division otherwise
static void mean_factors(int mean, int n_users, float *inv_u, float *div_u)
{
    *inv_u = 0.0f;
    *div_u = 0.0f;
    if (!mean) return;
    if ((n_users & (n_users - 1)) == 0) *inv_u = 1.0f / (float)n_users;
    else *div_u = (float)n_users;
}

// wait: the peers' delivery flags to poll first (n == 0: none); in the fast kernel's prologue, else in a
// one-warp kernel of its own
int qsgd_decode_reduce(const float *norm, const void *packed, int64_t user_stride, int n_users,
                       int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit,
                       int mean, int accumulate, float *out, const PeerWait &wait, cudaStream_t st)
{
    if (n == 0) {
        set_wait(wait);
        return flush_wait(st);
    }
    const float s = (float)(1u << n_bit);
    const int bits = qsgd_wire_bits(n_bit);
    const int64_t n8 = n / 8;
    if (n_users <= 8 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)packed & 15) == 0 &&
        (user_stride & 15) == 0 && n < (1ll << 40) && n_chunks < (1ll << 31)) {
        float inv_u, div_u;
        mean_factors(mean, n_users, &inv_u, &div_u);
        const int grid8 = grid_for(n8 + 1, 256, 16);
        const Rider rider = take_rider();   // a pending identity reduction rides in this launch
#define GQ_D8W(B, UU, W) GQ_CUDA(launch_pdl(qsgd_decode_reduce8_kernel<B, UU, W>, dim3(grid8), dim3(256), 0, st, norm, packed, user_stride, \
                                            n_users, n, chunk_start, (int)n_chunks, (uint32_t)(dim > 0 ? dim : 1), 1.0f / s, inv_u, div_u, accumulate, out, rider, wait))
#define GQ_D8(B, UU) do { if (wait.n > 0) GQ_D8W(B, UU, true); else GQ_D8W(B, UU, false); } while (0)
#define GQ_D8B(B) do { if (n_users == 1) GQ_D8(B, 1); else if (n_users == 2) GQ_D8(B, 2); else if (n_users == 4) GQ_D8(B, 4); \
                       else if (n_users == 8) GQ_D8(B, 8); else GQ_D8(B, 0); } while (0)
        if (bits == 4) GQ_D8B(4);
        else if (bits == 8) GQ_D8B(8);
        else GQ_D8B(16);
#undef GQ_D8B
#undef GQ_D8
#undef GQ_D8W
        GQ_LAUNCH_CHECK("qsgd_decode_reduce8");
        return GQ_OK;
    }
    set_wait(wait);
    GQ_CUDA_INT(flush_wait(st));
    const int grid = grid_for((n + 3) / 4, 256);
#define GQ_D(B) qsgd_decode_reduce_kernel<B><<<grid, 256, 0, st>>>(norm, packed, user_stride, n_users, n, chunk_start, n_chunks, dim, s, mean, accumulate, out)
    if (bits == 4) GQ_D(4);
    else if (bits == 8) GQ_D(8);
    else GQ_D(16);
#undef GQ_D
    GQ_LAUNCH_CHECK("qsgd_decode_reduce");
    return GQ_OK;
}

__global__ void __launch_bounds__(256)
qsgd_decode_unpacked_kernel(const float *__restrict__ norm, const uint8_t *__restrict__ signs,
                            const int32_t *__restrict__ l, int64_t n,
                            const int64_t *__restrict__ chunk_start, int64_t n_chunks, int dim, float s,
                            float *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const int64_t m = chunk_of(chunk_start, n_chunks, dim, i);
        out[i] = qsgd_value(l[i], (uint32_t)signs[i], __ldg(norm + m), s);
    }
}

int qsgd_decode_unpacked(const float *norm, const uint8_t *signs, const int32_t *l, int64_t n,
                         const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit, float *out,
                         cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    qsgd_decode_unpacked_kernel<<<grid_for(n, 256), 256, 0, st>>>(norm, signs, l, n, chunk_start, n_chunks,
                                                                  dim, (float)(1u << n_bit), out);
    GQ_LAUNCH_CHECK("qsgd_decode_unpacked");
    return GQ_OK;
}

// ------------------------------------------------------------------- sign ---
// torch.sign -> {-1, 0, +1}; packed: 2 bits per element (0 -> 0, 1 -> +1, 2 -> -1).
__global__ void __launch_bounds__(256)
sign_encode_kernel(const float *__restrict__ v, int64_t n, float *__restrict__ out_f32,
                   uint8_t *__restrict__ packed)
{
    const int64_t n4 = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x; q < n4; q += (int64_t)gridDim.x * 256) {
        const int64_t i0 = q * 4;
        float x[4];
        if (i0 + 3 < n) {
            float4 t = ld_stream_f4(reinterpret_cast<const float4 *>(v) + q);
            x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t) x[t] = (i0 + t < n) ? v[i0 + t] : 0.0f;
        }
        uint32_t byte = 0;
        float sg[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int pos = x[t] > 0.0f, neg = x[t] < 0.0f;
            sg[t] = (float)(pos - neg);
            byte |= (uint32_t)(pos | (neg << 1)) << (2 * t);
        }
        if (packed) packed[q] = (uint8_t)byte;
        if (out_f32) {
            if (i0 + 3 < n) {
                reinterpret_cast<float4 *>(out_f32)[q] = make_float4(sg[0], sg[1], sg[2], sg[3]);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) if (i0 + t < n) out_f32[i0 + t] = sg[t];
            }
        }
    }
}

// A warp decodes 512 elements at a time: lane L loads the L-th 32-bit word of packed signs of every
// user (one coalesced 128-byte request per user), the words are redistributed by shuffles so that lane
// L produces the float4 groups L, 32 + L, 64 + L, 96 + L of the tile: four fully coalesced 512-byte
// stores (a thread writing its own 16 consecutive elements would put half-sector writes on L2).
template <int U_, bool WAIT>
__global__ void __launch_bounds__(256)
sign_decode_reduce_kernel(const uint8_t *__restrict__ packed, int64_t user_stride, int n_users_rt,
                          int64_t n, float inv_u, float div_u, int accumulate, float *__restrict__ out, const Rider rider,
                          const PeerWait wait)
{
    pdl_launch_dependents();
    const int n_users = U_ > 0 ? U_ : n_users_rt;
    const int lane = threadIdx.x & 31;
    const int64_t n_tiles = (n + 511) / 512;
    const bool aligned = ((reinterpret_cast<uintptr_t>(out) & 15) == 0) && ((user_stride & 3) == 0) &&
                         ((reinterpret_cast<uintptr_t>(packed) & 3) == 0);
    pdl_wait();
    wait_prologue<WAIT>(wait);   // the peers' delivery flags, before any record byte is read
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    for (int64_t tile = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); tile < n_tiles; tile += (int64_t)gridDim.x * 8) {
        const int64_t e0 = tile * 512;
        const bool full = aligned && (e0 + 511 < n);   // warp-uniform
        float acc[4][4];
        for (int u = 0; u < n_users; ++u) {
            const uint8_t *pu = packed + u * user_stride + (e0 >> 2);
            uint32_t w = 0u;
            if (full) {
                w = ld_rec<WAIT>(reinterpret_cast<const uint32_t *>(pu) + lane);
            } else {
                for (int k = 0; k < 4; ++k)
                    if (e0 + 16 * lane + 4 * k < n) w |= (uint32_t)pu[4 * lane + k] << (8 * k);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const uint32_t ws = __shfl_sync(0xffffffffu, w, t * 8 + (lane >> 2));
                const uint32_t by = (ws >> (8 * (lane & 3))) & 0xffu;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t c = (by >> (2 * k)) & 3u;
                    const float val = (c & 1u) ? 1.0f : ((c & 2u) ? -1.0f : 0.0f);
                    acc[t][k] = (u == 0) ? val : __fadd_rn(acc[t][k], val);
                }
            }
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            float r[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                r[k] = acc[t][k];
                if (inv_u != 0.0f) r[k] = __fmul_rn(r[k], inv_u);
                else if (div_u != 0.0f) r[k] = __fdiv_rn(r[k], div_u);
            }
            const int64_t i = e0 + 4 * (t * 32 + lane);
            if (full) {
                float4 *op = reinterpret_cast<float4 *>(out + i);
                if (accumulate) {
                    const float4 o = *op;
                    r[0] = (accumulate == 2) ? __fsub_rn(o.x, r[0]) : __fadd_rn(o.x, r[0]);
                    r[1] = (accumulate == 2) ? __fsub_rn(o.y, r[1]) : __fadd_rn(o.y, r[1]);
                    r[2] = (accumulate == 2) ? __fsub_rn(o.z, r[2]) : __fadd_rn(o.z, r[2]);
                    r[3] = (accumulate == 2) ? __fsub_rn(o.w, r[3]) : __fadd_rn(o.w, r[3]);
                }
                *op = make_float4(r[0], r[1], r[2], r[3]);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (i + k >= n) continue;
                    float x = r[k];
                    if (accumulate) x = (accumulate == 2) ? __fsub_rn(out[i + k], x) : __fadd_rn(out[i + k], x);
                    out[i + k] = x;
                }
            }
        }
    }
}

// ------------------------------------------------- sign, base-3 wire (f4) ---
// Five ternary digits per byte (3^5 = 243 <= 256): byte = t0 + 3 t1 + 9 t2 + 27 t3 + 81 t4 with the
// same digit code as the 2-bit form (0 -> 0, 1 -> +1, 2 -> -1): 1.6 bits per element instead of 2.
// A thread owns 20 consecutive elements = one 32-bit word of the wire (little-endian bytes); the
// section holds ceil(n / 20) words, elements past n encode as 0.
template <bool DELIVER>
__global__ void __launch_bounds__(256)
sign_encode_t5_kernel(const float *__restrict__ v, int64_t n, uint32_t *__restrict__ packed, const Rider rider, const Remote R)
{
    pdl_launch_dependents();
    const int64_t n_words = (n + 19) / 20;
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    if constexpr (DELIVER) deliver_ident(R);
    for (int64_t w = (int64_t)blockIdx.x * 256 + threadIdx.x; w < n_words; w += (int64_t)gridDim.x * 256) {
        const int64_t i0 = w * 20;
        float x[20];
        if (i0 + 19 < n) {   // five 16-byte loads of 80 consecutive bytes (the other half of each sector: L1)
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                const float4 t = __ldg(reinterpret_cast<const float4 *>(v + i0) + q);
                x[4 * q] = t.x; x[4 * q + 1] = t.y; x[4 * q + 2] = t.z; x[4 * q + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int t = 0; t < 20; ++t) x[t] = (i0 + t < n) ? v[i0 + t] : 0.0f;
        }
        uint32_t word = 0u;
#pragma unroll
        for (int b = 3; b >= 0; --b) {
            uint32_t byte = 0u;
#pragma unroll
            for (int t = 4; t >= 0; --t) {
                const float e = x[5 * b + t];
                byte = byte * 3u + (e > 0.0f ? 1u : (e < 0.0f ? 2u : 0u));
            }
            word = (word << 8) | byte;
        }
        packed[w] = word;
        if constexpr (DELIVER) remote_st32(R, packed + w, word);
    }
    if constexpr (DELIVER) deliver_finish(R, [] {});
}

// A warp decodes 640 elements at a time: lane L takes word L of every user (one coalesced 128-byte
// request per user), sums its 20 values in user order, and the warp transposes the 640 results through
// shared memory so that the stores are five fully coalesced 512-byte rows (see sign_decode_reduce_kernel).
template <int U_, bool WAIT>
__global__ void __launch_bounds__(256)
sign_decode_reduce_t5_kernel(const uint32_t *__restrict__ packed, int64_t user_stride_words, int n_users_rt,
                             int64_t n, float inv_u, float div_u, int accumulate, float *__restrict__ out, const Rider rider,
                             const PeerWait wait)
{
    __shared__ float4 s_t[8][160];   // per warp: 640 floats
    pdl_launch_dependents();
    const int n_users = U_ > 0 ? U_ : n_users_rt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_tiles = (n + 639) / 640;
    const int64_t n_words = (n + 19) / 20;
    const bool aligned = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    pdl_wait();
    wait_prologue<WAIT>(wait);   // the peers' delivery flags, before any record byte is read
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    for (int64_t tile = (int64_t)blockIdx.x * 8 + warp; tile < n_tiles; tile += (int64_t)gridDim.x * 8) {
        const int64_t e0 = tile * 640;
        const int64_t w = tile * 32 + lane;
        float acc[20];
        for (int u = 0; u < n_users; ++u) {
            uint32_t word = (w < n_words) ? ld_rec<WAIT>(packed + u * user_stride_words + w) : 0u;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                uint32_t by = word & 0xffu;
                word >>= 8;
#pragma unroll
                for (int t = 0; t < 5; ++t) {
                    const uint32_t q = (by * 171u) >> 9;   // by / 3 for by < 256
                    const uint32_t c = by - 3u * q;
                    by = q;
                    const float val = (c == 1u) ? 1.0f : ((c == 2u) ? -1.0f : 0.0f);
                    acc[5 * b + t] = (u == 0) ? val : __fadd_rn(acc[5 * b + t], val);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 20; ++k) {
            if (inv_u != 0.0f) acc[k] = __fmul_rn(acc[k], inv_u);
            else if (div_u != 0.0f) acc[k] = __fdiv_rn(acc[k], div_u);
        }
        // lane L holds elements 20 L .. 20 L + 19 = float4 groups 5 L .. 5 L + 4 of the tile
#pragma unroll
        for (int q = 0; q < 5; ++q) s_t[warp][5 * lane + q] = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            float4 r = s_t[warp][32 * q + lane];
            const int64_t i = e0 + 4 * (32 * q + lane);
            if (aligned && i + 3 < n) {
                float4 *op = reinterpret_cast<float4 *>(out + i);
                if (accumulate) {
                    const float4 o = *op;
                    r.x = (accumulate == 2) ? __fsub_rn(o.x, r.x) : __fadd_rn(o.x, r.x);
                    r.y = (accumulate == 2) ? __fsub_rn(o.y, r.y) : __fadd_rn(o.y, r.y);
                    r.z = (accumulate == 2) ? __fsub_rn(o.z, r.z) : __fadd_rn(o.z, r.z);
                    r.w = (accumulate == 2) ? __fsub_rn(o.w, r.w) : __fadd_rn(o.w, r.w);
                }
                *op = r;
            } else {
                const float y[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (i + k >= n) continue;
                    float x = y[k];
                    if (accumulate) x = (accumulate == 2) ? __fsub_rn(out[i + k], x) : __fadd_rn(out[i + k], x);
                    out[i + k] = x;
                }
            }
        }
        __syncwarp();
    }
}

int sign_encode_t5(const float *grad, int64_t n, uint32_t *packed, const Tc2Remote &remote, cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    const Rider rider = take_rider();   // a pending identity copy rides in this launch
    Remote R = {};
    if (remote.n > 0) GQ_CUDA_INT(device_remote(remote, rider, &R));
    const dim3 grid(grid_for((n + 19) / 20, 256, 16));
    GQ_CUDA(remote.n > 0 ? launch_pdl(sign_encode_t5_kernel<true>, grid, dim3(256), 0, st, grad, n, packed, rider, R)
                         : launch_pdl(sign_encode_t5_kernel<false>, grid, dim3(256), 0, st, grad, n, packed, rider, R));
    GQ_LAUNCH_CHECK("sign_encode_t5");
    return GQ_OK;
}

int sign_decode_reduce_t5(const uint32_t *packed, int64_t user_stride_words, int n_users, int64_t n, int mean,
                          int accumulate, float *out, const PeerWait &wait, cudaStream_t st)
{
    if (n == 0) {
        set_wait(wait);
        return flush_wait(st);
    }
    float inv_u, div_u;
    mean_factors(mean, n_users, &inv_u, &div_u);
    const int grid = grid_for((n + 639) / 640, 8, 8);
    const Rider rider = take_rider();   // a pending identity reduction rides in this launch
#define GQ_SW(UU, W) GQ_CUDA(launch_pdl(sign_decode_reduce_t5_kernel<UU, W>, dim3(grid), dim3(256), 0, st, packed, user_stride_words, \
                                        n_users, n, inv_u, div_u, accumulate, out, rider, wait))
#define GQ_S(UU) do { if (wait.n > 0) GQ_SW(UU, true); else GQ_SW(UU, false); } while (0)
    if (n_users == 1) GQ_S(1);
    else if (n_users == 2) GQ_S(2);
    else if (n_users == 4) GQ_S(4);
    else if (n_users == 8) GQ_S(8);
    else GQ_S(0);
#undef GQ_S
#undef GQ_SW
    GQ_LAUNCH_CHECK("sign_decode_reduce_t5");
    return GQ_OK;
}

// packed output only (the fused plan): a thread owns 16 consecutive elements = one 32-bit word of the
// wire -- four 16-byte loads in flight per thread and a coalesced 128-byte store per warp instead of 32
// single bytes (21.0 -> see DESIGN.md section 8)
template <bool DELIVER>
__global__ void __launch_bounds__(256)
sign_encode_words_kernel(const float *__restrict__ v, int64_t n, uint32_t *__restrict__ packed, const Rider rider, const Remote R)
{
    pdl_launch_dependents();
    const int64_t n_words = n / 16;   // whole words; the ragged tail goes through sign_encode_kernel
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    if constexpr (DELIVER) deliver_ident(R);
    for (int64_t w = (int64_t)blockIdx.x * 256 + threadIdx.x; w < n_words; w += (int64_t)gridDim.x * 256) {
        float4 t[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) t[q] = __ldg(reinterpret_cast<const float4 *>(v) + 4 * w + q);
        uint32_t word = 0u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float x[4] = {t[q].x, t[q].y, t[q].z, t[q].w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                word |= ((x[k] > 0.0f ? 1u : 0u) | (x[k] < 0.0f ? 2u : 0u)) << (8 * q + 2 * k);
        }
        packed[w] = word;
        if constexpr (DELIVER) remote_st32(R, packed + w, word);
    }
    if constexpr (DELIVER) {
        // a delivering launch encodes the ragged tail itself (at most 15 elements: the bytes that
        // sign_encode_kernel would write), then sends that word whole -- the section is padded to 4 bytes
        const int64_t done = n_words * 16;
        if (done < n && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
            uint8_t *pb = reinterpret_cast<uint8_t *>(packed + n_words);
            for (int b = 0; 4 * b < n - done; ++b) {
                uint32_t byte = 0u;
                for (int k = 0; k < 4; ++k) {
                    const float x = (done + 4 * b + k < n) ? v[done + 4 * b + k] : 0.0f;
                    byte |= ((x > 0.0f ? 1u : 0u) | (x < 0.0f ? 2u : 0u)) << (2 * k);
                }
                pb[b] = (uint8_t)byte;
            }
            deliver_word(R, pb);
        }
        deliver_finish(R, [] {});
    }
}

// remote: the pending delivery (n == 0: none), which only the packed-words kernel makes; a call that would
// take the other kernel returns GQ_ERR_UNSUPPORTED before it launches anything
int sign_encode(const float *grad, int64_t n, float *out_f32, uint8_t *packed, const Tc2Remote &remote, cudaStream_t st)
{
    const bool words = !out_f32 && packed && ((uintptr_t)packed & 3) == 0;
    if (remote.n > 0) {
        if (!words || n == 0) {
            set_error("a remote delivery is attached, but this sign encode is not the packed-words kernel "
                      "(packed output only, 4-byte aligned, n > 0)");
            return GQ_ERR_UNSUPPORTED;
        }
        const Rider rider = take_rider();   // a pending identity copy rides in this launch
        Remote R = {};
        GQ_CUDA_INT(device_remote(remote, rider, &R));
        GQ_CUDA(launch_pdl(sign_encode_words_kernel<true>, dim3(grid_for(n / 16 + 1, 256, 16)), dim3(256), 0, st, grad, n,
                           reinterpret_cast<uint32_t *>(packed), rider, R));
        GQ_LAUNCH_CHECK("sign_encode");
        return GQ_OK;
    }
    if (n == 0) return GQ_OK;
    if (words && n >= 16) {
        const int64_t n_words = n / 16;
        const Rider rider = take_rider();   // a pending identity copy rides in this launch
        GQ_CUDA(launch_pdl(sign_encode_words_kernel<false>, dim3(grid_for(n_words, 256, 16)), dim3(256), 0, st, grad, n,
                           reinterpret_cast<uint32_t *>(packed), rider, Remote{}));
        const int64_t done = n_words * 16;
        if (done < n)   // at most 15 elements
            sign_encode_kernel<<<1, 32, 0, st>>>(grad + done, n - done, nullptr, packed + done / 4);
        GQ_LAUNCH_CHECK("sign_encode");
        return GQ_OK;
    }
    sign_encode_kernel<<<grid_for((n + 3) / 4, 256), 256, 0, st>>>(grad, n, out_f32, packed);
    GQ_LAUNCH_CHECK("sign_encode");
    return GQ_OK;
}

int sign_decode_reduce(const uint8_t *packed, int64_t user_stride, int n_users, int64_t n, int mean,
                       int accumulate, float *out, const PeerWait &wait, cudaStream_t st)
{
    if (n == 0) {
        set_wait(wait);
        return flush_wait(st);
    }
    float inv_u, div_u;
    mean_factors(mean, n_users, &inv_u, &div_u);
    const int grid = grid_for((n + 511) / 512, 8, 16);
    const Rider rider = take_rider();   // a pending identity reduction rides in this launch
#define GQ_SW(UU, W) GQ_CUDA(launch_pdl(sign_decode_reduce_kernel<UU, W>, dim3(grid), dim3(256), 0, st, packed, user_stride, n_users, n, \
                                        inv_u, div_u, accumulate, out, rider, wait))
#define GQ_S(UU) do { if (wait.n > 0) GQ_SW(UU, true); else GQ_SW(UU, false); } while (0)
    if (n_users == 1) GQ_S(1);
    else if (n_users == 2) GQ_S(2);
    else if (n_users == 4) GQ_S(4);
    else if (n_users == 8) GQ_S(8);
    else GQ_S(0);
#undef GQ_S
#undef GQ_SW
    GQ_LAUNCH_CHECK("sign_decode_reduce");
    return GQ_OK;
}

}  // namespace gq

using namespace gq;

extern "C" {

int gq_qsgd_wire_bits(int n_bit) { return qsgd_wire_bits(n_bit); }

int gq_qsgd_encode(const float *grad, int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim,
                   int n_bit, int random, const float *uniforms, uint64_t philox_seed,
                   uint64_t philox_offset, float *norm, uint8_t *signs, int32_t *l, void *packed,
                   gq_stream_t stream)
{
    const Rider pending = take_rider();   // consumed first: an early error return must not leave it armed
    const Tc2Remote remote = take_remote();   // likewise the pending delivery to the peers
    GQ_REQUIRE(n >= 0 && n_chunks >= 0, "negative size");
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 14, "n_bit %d out of range 1..14", n_bit);
    GQ_REQUIRE(chunk_start || (dim >= 1 && n_chunks * (int64_t)dim == n),
               "n (%lld) != n_chunks (%lld) * dim (%d)", (long long)n, (long long)n_chunks, dim);
    GQ_REQUIRE(n == 0 || (grad && norm), "null pointer");
    GQ_REQUIRE(packed || (signs && l), "need packed or (signs and l) outputs");
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0, "gradient must be 16-byte aligned");
    set_rider(pending);
    const int e = qsgd_encode(grad, n, chunk_start, n_chunks, dim, n_bit, random, uniforms, philox_seed,
                              philox_offset, norm, signs, l, packed, remote, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));   // no-op when the encode kernel carried it
}

int gq_qsgd_decode_reduce(const float *norm, const void *packed, int64_t user_stride_bytes, int n_users,
                          int64_t n, const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit,
                          int mean, int accumulate, float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();
    const PeerWait wait = take_wait();
    GQ_REQUIRE(n >= 0 && n_users >= 1, "bad sizes");
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 14, "n_bit %d out of range 1..14", n_bit);
    GQ_REQUIRE(chunk_start || (dim >= 1 && n_chunks * (int64_t)dim == n), "n != n_chunks * dim");
    GQ_REQUIRE(n == 0 || (norm && packed && out), "null pointer");
    set_rider(pending);
    const int e = qsgd_decode_reduce(norm, packed, user_stride_bytes, n_users, n, chunk_start, n_chunks, dim,
                                     n_bit, mean, accumulate, out, wait, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

int gq_qsgd_decode_unpacked(const float *norm, const uint8_t *signs, const int32_t *l, int64_t n,
                            const int64_t *chunk_start, int64_t n_chunks, int dim, int n_bit, float *out,
                            gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0, "bad sizes");
    GQ_REQUIRE(chunk_start || (dim >= 1 && n_chunks * (int64_t)dim == n), "n != n_chunks * dim");
    GQ_REQUIRE(n == 0 || (norm && signs && l && out), "null pointer");
    return qsgd_decode_unpacked(norm, signs, l, n, chunk_start, n_chunks, dim, n_bit, out,
                                as_stream(stream));
}

int gq_sign_encode(const float *grad, int64_t n, float *out_f32, uint8_t *packed, gq_stream_t stream)
{
    const Rider pending = take_rider();
    const Tc2Remote remote = take_remote();
    GQ_REQUIRE(n >= 0 && (n == 0 || grad), "bad arguments");
    GQ_REQUIRE(out_f32 || packed, "need at least one output");
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0, "gradient must be 16-byte aligned");
    set_rider(pending);
    const int e = sign_encode(grad, n, out_f32, packed, remote, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

int gq_sign_decode_reduce(const uint8_t *packed, int64_t user_stride_bytes, int n_users, int64_t n,
                          int mean, int accumulate, float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();
    const PeerWait wait = take_wait();
    GQ_REQUIRE(n >= 0 && n_users >= 1 && (n == 0 || (packed && out)), "bad arguments");
    set_rider(pending);
    const int e = sign_decode_reduce(packed, user_stride_bytes, n_users, n, mean, accumulate, out, wait, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

int64_t gq_sign_t5_bytes(int64_t n) { return n <= 0 ? 0 : (n + 19) / 20 * 4; }

int gq_sign_encode_t5(const float *grad, int64_t n, void *packed, gq_stream_t stream)
{
    const Rider pending = take_rider();
    const Tc2Remote remote = take_remote();
    GQ_REQUIRE(n >= 0 && (n == 0 || (grad && packed)), "bad arguments");
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0 && ((uintptr_t)packed & 3) == 0, "gradient 16-byte, wire 4-byte aligned");
    if (remote.n > 0 && n == 0) {
        set_error("a remote delivery is attached to an empty sign encode");
        return GQ_ERR_UNSUPPORTED;
    }
    set_rider(pending);
    const int e = sign_encode_t5(grad, n, reinterpret_cast<uint32_t *>(packed), remote, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

int gq_sign_decode_reduce_t5(const void *packed, int64_t user_stride_bytes, int n_users, int64_t n, int mean,
                             int accumulate, float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();
    const PeerWait wait = take_wait();
    GQ_REQUIRE(n >= 0 && n_users >= 1 && (n == 0 || (packed && out)), "bad arguments");
    GQ_REQUIRE(((uintptr_t)packed & 3) == 0 && (user_stride_bytes & 3) == 0, "wire sections are 4-byte aligned");
    set_rider(pending);
    const int e = sign_decode_reduce_t5(reinterpret_cast<const uint32_t *>(packed), user_stride_bytes / 4, n_users, n, mean,
                                        accumulate, out, wait, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

}  // extern "C"

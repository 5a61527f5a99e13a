// hsq_tail.cu -- everything of the HSQ codec after the search:
//   * per-tensor min/max of u (when the search kernel did not fold it in)
//   * n-bit norm quantization   (probabilistic_scalar_compressor.py:12-27)
//   * norm dequantization       (probabilistic_scalar_compressor.py:29-33)
//   * fused decode-and-reduce over users
//       (nearest_neighbor_compressor.py:80-90 + ps_quantizer.py:48 /
//        ring_quantizer.py:31-32)
// All HBM-bound.  Algorithmic bytes per gradient element (d = chunk dim, U users):
//   quantize: (4 u + 1 l [+4 r]) / d        decode-reduce: 4 + 2U/d (+4 if accumulate)
#include <stdlib.h>

#include <type_traits>

#include "gq_internal.cuh"

namespace gq {

// ------------------------------------------------------- segmented min/max ---
__global__ void __launch_bounds__(256)
seg_minmax_kernel(const float *__restrict__ u, int64_t n, const int64_t *__restrict__ seg_start,
                  int n_seg, uint32_t *__restrict__ keys)
{
    SegCache segc;
    for (int64_t base = (int64_t)blockIdx.x * 256; base < n; base += (int64_t)gridDim.x * 256) {
        int64_t i = base + threadIdx.x;
        bool valid = i < n;
        float x = valid ? u[i] : 0.0f;
        int seg = valid ? cached_segment(segc, seg_start, n_seg, i) : -1;
        int seg0 = __shfl_sync(0xffffffffu, seg, 0);
        bool uniform = __all_sync(0xffffffffu, (seg == seg0) || !valid) && (seg0 >= 0);
        // torch.min / torch.max propagate NaN (fminf / fmaxf drop it): it goes into the max key, above +inf
        if (valid && x != x) atomicMax(keys + 2 * seg + 1, GQ_KEY_NAN);
        if (uniform) {
            float mn = warp_min(valid ? x : INFINITY);
            float mx = warp_max(valid ? x : -INFINITY);
            if ((threadIdx.x & 31) == 0) {
                atomicMin(keys + 2 * seg0, float_to_key(mn));
                atomicMax(keys + 2 * seg0 + 1, float_to_key(mx));
            }
        } else if (valid) {
            atomicMin(keys + 2 * seg, float_to_key(x));
            atomicMax(keys + 2 * seg + 1, float_to_key(x));
        }
    }
}

// ---------------------------------------------------------- norm quantize ---
// Four consecutive chunks per thread: one float4 load of u (and of the uniforms), one
// Philox4x32-10 block for the four draws, one packed store of the four levels.
template <typename LT>
__global__ void __launch_bounds__(256)
norm_quantize_kernel(const float *__restrict__ u, int64_t n, const int64_t *__restrict__ seg_start,
                     int n_seg, float s, int random, const float *__restrict__ uniforms,
                     uint64_t seed, uint64_t offset, LT *__restrict__ l, float *__restrict__ lbub,
                     const uint32_t *__restrict__ keys)
{
    // block 0 also publishes lb/ub as floats (the reference returns them, :27)
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i < 2 * n_seg; i += 256) lbub[i] = key_to_float(keys[i]);
    }
    quantize_range<LT, false>(u, 0, n, n, (int)(blockIdx.x * 256 + threadIdx.x), (int)(gridDim.x * 256), seg_start,
                              n_seg, s, random, uniforms, seed, offset, l, keys);
}

// Same, instruction-lean (the kernel is issue-bound, not HBM-bound: 5.6 M warp instructions for
// 7 MB of traffic in its first version): 32-bit segment table and decoded (lb, ub) pairs in shared
// memory; the segment of a block's first chunk is COUNTED by the block (one __syncthreads_count
// per 256 segments) instead of binary-searched per thread; four consecutive chunks per thread =
// one float4 of u (and of the uniforms), one Philox4x32-10 block, one packed store; when all four
// lie in one tensor (almost always) lb, ub and ub - lb are fetched once.  The host sizes the grid
// so that it is ONE resident wave with `items` groups per thread, a grid-width apart (1435 blocks
// of one item each were 1.2 waves on 148 SMs: the second, nearly empty wave doubled the run
// time); the loads of the next item are issued before the current one is processed.
constexpr int kQuantMaxSeg = 1024;
template <typename LT>
__global__ void __launch_bounds__(256)
norm_quantize_smem_kernel(const float *__restrict__ u, int n, const int64_t *__restrict__ seg_start,
                          int n_seg, float s, int random, const float *__restrict__ uniforms,
                          uint64_t seed, uint64_t offset, LT *__restrict__ l, float *__restrict__ lbub,
                          const uint32_t *__restrict__ keys, int items)
{
    extern __shared__ int s_segi[];                                                  // [n_seg + 1]
    float2 *s_lbub2 = reinterpret_cast<float2 *>(s_segi + ((n_seg + 2) & ~1));      // [n_seg]
    const int tid = threadIdx.x;
    pdl_launch_dependents();
    for (int i = tid; i <= n_seg; i += 256) s_segi[i] = (int)seg_start[i];
    pdl_wait();   // keys and u come from the search kernel
    for (int i = tid; i < n_seg; i += 256) {
        const float lb = key_to_float(keys[2 * i]), ub = key_to_float(keys[2 * i + 1]);
        s_lbub2[i] = make_float2(lb, ub);
        if (blockIdx.x == 0) {   // the reference returns lb/ub (probabilistic_scalar_compressor.py:27)
            lbub[2 * i] = lb;
            lbub[2 * i + 1] = ub;
        }
    }
    const int n4 = (n + 3) >> 2;
    const int stride = gridDim.x * 256;
    int q = blockIdx.x * 256 + tid;
    float4 xv = make_float4(0.f, 0.f, 0.f, 0.f), rv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q < n4 && q * 4 + 3 < n) {
        xv = __ldg(reinterpret_cast<const float4 *>(u) + q);
        if (random && uniforms) rv = __ldg(reinterpret_cast<const float4 *>(uniforms) + q);
    }
    const bool philox = random && !uniforms;
    const bool philox_aligned = (offset & 3u) == 0;
    __syncthreads();
    for (int it = 0; it < items; ++it, q += stride) {   // uniform trip count (block-wide barriers inside)
        // segment holding the first chunk of this block's range
        const int block_i0 = (blockIdx.x * 256 + it * stride) * 4;
        int base = -1;
        for (int j0 = 0; j0 < n_seg; j0 += 256)
            base += __syncthreads_count(j0 + tid < n_seg && s_segi[j0 + tid] <= block_i0);
        if (q >= n4) continue;
        const bool full = q * 4 + 3 < n;
        const int i0 = q * 4;
        float x[4] = {xv.x, xv.y, xv.z, xv.w}, r[4] = {rv.x, rv.y, rv.z, rv.w};
        {
            const int qn = q + stride;
            if (it + 1 < items && qn < n4 && qn * 4 + 3 < n) {
                xv = __ldg(reinterpret_cast<const float4 *>(u) + qn);
                if (random && uniforms) rv = __ldg(reinterpret_cast<const float4 *>(uniforms) + qn);
            }
        }
        if (!full) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                x[t] = (i0 + t < n) ? u[i0 + t] : 0.0f;
                r[t] = (random && uniforms && i0 + t < n) ? uniforms[i0 + t] : 0.0f;
            }
        }
        if (philox) {
            if (philox_aligned) {
                const uint4 w = philox4x32_10(seed, (offset + (uint64_t)i0) >> 2);
                r[0] = u01(w.x); r[1] = u01(w.y); r[2] = u01(w.z); r[3] = u01(w.w);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) r[t] = philox_uniform(seed, offset, (uint64_t)(i0 + t));
            }
        }
        int seg = base < 0 ? 0 : base;
        int lv[4];
        psc_levels4(x, r, i0, n, s_segi, s_lbub2, seg, s, random, lv);
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

template <typename LT>
__global__ void __launch_bounds__(256)
norm_dequantize_kernel(const LT *__restrict__ l, int64_t n, const int64_t *__restrict__ seg_start,
                       int n_seg, float s, const float *__restrict__ lbub, float *__restrict__ out)
{
    SegCache segc;
    for (int64_t base = (int64_t)blockIdx.x * 256; base < n; base += (int64_t)gridDim.x * 256) {
        int64_t i = base + threadIdx.x;
        if (i >= n) continue;
        int seg = cached_segment(segc, seg_start, n_seg, i);
        out[i] = psc_value((int)l[i], __ldg(lbub + 2 * seg), __ldg(lbub + 2 * seg + 1), 1.0f / s);
    }
}

static int grid_for(int64_t n, int per_block, int waves = 8)
{
    int64_t blocks = (n + per_block - 1) / per_block;
    int64_t cap = (int64_t)sm_count() * waves;
    int64_t g = blocks < cap ? blocks : cap;
    return (int)(g < 1 ? 1 : g);
}

int launch_seg_minmax(const float *u, int64_t n, const int64_t *seg_start, int n_seg, uint32_t *keys,
                      cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    seg_minmax_kernel<<<grid_for(n, 256), 256, 0, st>>>(u, n, seg_start, n_seg, keys);
    GQ_LAUNCH_CHECK("seg_minmax");
    return GQ_OK;
}

int launch_norm_quantize(const float *u, int64_t n, const int64_t *seg_start, int n_seg, int n_bit,
                         int random, const float *uniforms, uint64_t seed, uint64_t offset, void *l,
                         int l_bytes, float *lbub, const uint32_t *keys, cudaStream_t st)
{
    const float s = (float)(1u << n_bit);
    const int64_t n4 = (n + 3) / 4;
    const bool aligned = (((uintptr_t)u & 15) == 0) && (uniforms == nullptr || ((uintptr_t)uniforms & 15) == 0) &&
                         (((uintptr_t)l & (4 * (size_t)l_bytes - 1)) == 0);
    if (n_seg <= kQuantMaxSeg && aligned && n4 > 0 && n < ((int64_t)1 << 31) - 8) {
        // tables in shared memory, 32-bit indices
        const size_t smem = (size_t)((n_seg + 2) & ~1) * 4 + (size_t)n_seg * 8;
        const int64_t blocks = (n4 + 255) / 256;
        int occ = 1;
        if (l_bytes == 1)
            GQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, norm_quantize_smem_kernel<uint8_t>, 256, smem));
        else
            GQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, norm_quantize_smem_kernel<int32_t>, 256, smem));
        const int64_t cap = (int64_t)sm_count() * (occ < 1 ? 1 : occ);
        const int items = (int)((blocks + cap - 1) / cap);                 // per thread
        const unsigned grid = (unsigned)((blocks + items - 1) / items);    // one wave, evenly loaded
        if (l_bytes == 1)
            GQ_CUDA(launch_pdl(norm_quantize_smem_kernel<uint8_t>, dim3(grid), dim3(256), smem, st, u, (int)n, seg_start,
                               n_seg, s, random, uniforms, seed, offset, (uint8_t *)l, lbub, keys, items));
        else
            GQ_CUDA(launch_pdl(norm_quantize_smem_kernel<int32_t>, dim3(grid), dim3(256), smem, st, u, (int)n, seg_start,
                               n_seg, s, random, uniforms, seed, offset, (int32_t *)l, lbub, keys, items));
        return GQ_OK;
    }
    const int grid = grid_for(n > 0 ? n4 : 1, 256);
    if (l_bytes == 1)
        norm_quantize_kernel<uint8_t><<<grid, 256, 0, st>>>(u, n, seg_start, n_seg, s, random, uniforms,
                                                            seed, offset, (uint8_t *)l, lbub, keys);
    else
        norm_quantize_kernel<int32_t><<<grid, 256, 0, st>>>(u, n, seg_start, n_seg, s, random, uniforms,
                                                            seed, offset, (int32_t *)l, lbub, keys);
    GQ_LAUNCH_CHECK("norm_quantize");
    return GQ_OK;
}

int launch_norm_dequantize(const void *l, int l_bytes, int64_t n, const int64_t *seg_start, int n_seg,
                           int n_bit, const float *lbub, float *out, cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    const float s = (float)(1u << n_bit);
    const int grid = grid_for(n, 256);
    if (l_bytes == 1)
        norm_dequantize_kernel<uint8_t><<<grid, 256, 0, st>>>((const uint8_t *)l, n, seg_start, n_seg, s, lbub, out);
    else
        norm_dequantize_kernel<int32_t><<<grid, 256, 0, st>>>((const int32_t *)l, n, seg_start, n_seg, s, lbub, out);
    GQ_LAUNCH_CHECK("norm_dequantize");
    return GQ_OK;
}

// accumulate: 0 store the reduction r, 1 out = out + r (ring: grad += previous hop's sum,
// ring_quantizer.py:31-32), 2 out = out - r (error feedback: error = grad - decompress(compress(grad)),
// ps_quantizer.py:39, with `out` holding the compensated gradient)
__device__ __forceinline__ float combine1(float o, float r, int accumulate)
{
    return accumulate == 2 ? __fsub_rn(o, r) : __fadd_rn(o, r);
}
__device__ __forceinline__ float4 combine4(float4 o, float4 r, int accumulate)
{
    return accumulate == 2 ? make_float4(__fsub_rn(o.x, r.x), __fsub_rn(o.y, r.y), __fsub_rn(o.z, r.z), __fsub_rn(o.w, r.w))
                           : make_float4(__fadd_rn(o.x, r.x), __fadd_rn(o.y, r.y), __fadd_rn(o.z, r.z), __fadd_rn(o.w, r.w));
}

// ------------------------------------------------------- decode-and-reduce ---
// One thread per float4 of the output, four independent float4 per thread (the loads of all
// four are issued before any is consumed).  A chunk of D floats is D/4 consecutive float4, so
// the D/4 lanes that share a chunk read the same code / level bytes (one coalesced request)
// and dequantize the norm redundantly -- cheaper than a shuffle phase.  The codeword comes
// from shared memory (K*d*4 <= 64 KB) or L1/L2; products are added in user order
// u = 0..U-1 with separately rounded mul and add, exactly like torch.mul +
// stack().mean(0) of the reference.
constexpr int kDecodeThreads = 256;
constexpr int kDecodeUnroll = 4;

template <int D, typename CodeT, typename LT, bool CB_SMEM>
__global__ void __launch_bounds__(kDecodeThreads)
hsq_decode_reduce_kernel(const CodeT *__restrict__ codes, const LT *__restrict__ l,
                         const float *__restrict__ lbub, const float *__restrict__ norms_f32,
                         int64_t user_stride, int n_users, int64_t n_chunks,
                         const float *__restrict__ codebook, int K,
                         const int64_t *__restrict__ seg_start, int n_seg, float s, int n_bit,
                         int mean, int accumulate, float *__restrict__ out)
{
    extern __shared__ float4 s_cbd[];
    constexpr int D4 = D / 4;  // float4 per chunk
    const float4 *cb4g = reinterpret_cast<const float4 *>(codebook);
    if (CB_SMEM) {
        for (int i = threadIdx.x; i < K * D4; i += kDecodeThreads) s_cbd[i] = __ldg(cb4g + i);
        __syncthreads();
    }
    // mean = sum / U with the reference's true division; U == 1 and powers of two are exact
    // as a multiplication by 1/U, everything else pays the IEEE division.
    const float inv_s = 1.0f / s;
    const float nu = (float)n_users;
    const bool pow2 = (n_users & (n_users - 1)) == 0;
    const float inv_nu = 1.0f / nu;
    SegCache segc;
    const int64_t n4 = n_chunks * D4;
    constexpr int64_t kSpan = (int64_t)kDecodeThreads * kDecodeUnroll;
    float4 *o4 = reinterpret_cast<float4 *>(out);
    for (int64_t base = (int64_t)blockIdx.x * kSpan; base < n4; base += (int64_t)gridDim.x * kSpan) {
        int64_t f[kDecodeUnroll], c[kDecodeUnroll];
        int part[kDecodeUnroll], seg[kDecodeUnroll];
        bool ok[kDecodeUnroll];
        float4 acc[kDecodeUnroll];
#pragma unroll
        for (int j = 0; j < kDecodeUnroll; ++j) {
            f[j] = base + j * kDecodeThreads + threadIdx.x;
            ok[j] = f[j] < n4;
            c[j] = ok[j] ? f[j] / D4 : 0;
            part[j] = (int)(f[j] % D4);
            seg[j] = (ok[j] && n_bit != 32) ? cached_segment(segc, seg_start, n_seg, c[j]) : 0;
            acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int u = 0; u < n_users; ++u) {
            const char *cu = reinterpret_cast<const char *>(codes) + u * user_stride;
            int code[kDecodeUnroll];
            float norm[kDecodeUnroll];
            if (n_bit == 32) {
                const char *nup = reinterpret_cast<const char *>(norms_f32) + u * user_stride;
#pragma unroll
                for (int j = 0; j < kDecodeUnroll; ++j) {
                    code[j] = ok[j] ? (int)reinterpret_cast<const CodeT *>(cu)[c[j]] : 0;
                    norm[j] = ok[j] ? reinterpret_cast<const float *>(nup)[c[j]] : 0.0f;
                }
            } else {
                const char *lu = reinterpret_cast<const char *>(l) + u * user_stride;
                const float *b = reinterpret_cast<const float *>(reinterpret_cast<const char *>(lbub) + u * user_stride);
                int lv[kDecodeUnroll];
#pragma unroll
                for (int j = 0; j < kDecodeUnroll; ++j) {
                    code[j] = ok[j] ? (int)reinterpret_cast<const CodeT *>(cu)[c[j]] : 0;
                    lv[j] = ok[j] ? (int)reinterpret_cast<const LT *>(lu)[c[j]] : 0;
                }
#pragma unroll
                for (int j = 0; j < kDecodeUnroll; ++j)
                    norm[j] = psc_value(lv[j], __ldg(b + 2 * seg[j]), __ldg(b + 2 * seg[j] + 1), inv_s);
            }
#pragma unroll
            for (int j = 0; j < kDecodeUnroll; ++j) {
                const float4 cw = CB_SMEM ? s_cbd[code[j] * D4 + part[j]]
                                          : __ldg(cb4g + (int64_t)code[j] * D4 + part[j]);
                float4 pr;
                pr.x = __fmul_rn(cw.x, norm[j]); pr.y = __fmul_rn(cw.y, norm[j]);
                pr.z = __fmul_rn(cw.z, norm[j]); pr.w = __fmul_rn(cw.w, norm[j]);
                if (u == 0) {
                    acc[j] = pr;
                } else {
                    acc[j].x = __fadd_rn(acc[j].x, pr.x); acc[j].y = __fadd_rn(acc[j].y, pr.y);
                    acc[j].z = __fadd_rn(acc[j].z, pr.z); acc[j].w = __fadd_rn(acc[j].w, pr.w);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kDecodeUnroll; ++j) {
            if (!ok[j]) continue;
            float4 r = acc[j];
            if (mean && n_users > 1) {
                if (pow2) {
                    r.x = __fmul_rn(r.x, inv_nu); r.y = __fmul_rn(r.y, inv_nu);
                    r.z = __fmul_rn(r.z, inv_nu); r.w = __fmul_rn(r.w, inv_nu);
                } else {
                    r.x = __fdiv_rn(r.x, nu); r.y = __fdiv_rn(r.y, nu);
                    r.z = __fdiv_rn(r.z, nu); r.w = __fdiv_rn(r.w, nu);
                }
            }
            if (accumulate) {
                const float4 o = o4[f[j]];
                r = combine4(o, r, accumulate);
            }
            o4[f[j]] = r;
        }
    }
}

// scalar fallback for chunk dims that are not a multiple of 4
template <typename CodeT, typename LT>
__global__ void __launch_bounds__(256)
hsq_decode_reduce_generic_kernel(const CodeT *__restrict__ codes, const LT *__restrict__ l,
                                 const float *__restrict__ lbub, const float *__restrict__ norms_f32,
                                 int64_t user_stride, int n_users, int64_t n_chunks, int d,
                                 const float *__restrict__ codebook,
                                 const int64_t *__restrict__ seg_start, int n_seg, float s, int n_bit,
                                 int mean, int accumulate, float *__restrict__ out)
{
    const int64_t n = n_chunks * (int64_t)d;
    for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < n; e += (int64_t)gridDim.x * 256) {
        const int64_t c = e / d;
        const int j = (int)(e % d);
        int seg = (n_bit != 32) ? find_segment(seg_start, n_seg, c) : 0;
        float acc = 0.0f;
        for (int u = 0; u < n_users; ++u) {
            const char *cu = reinterpret_cast<const char *>(codes) + u * user_stride;
            int code = (int)reinterpret_cast<const CodeT *>(cu)[c];
            float norm;
            if (n_bit == 32) {
                const char *nu = reinterpret_cast<const char *>(norms_f32) + u * user_stride;
                norm = reinterpret_cast<const float *>(nu)[c];
            } else {
                const char *lu = reinterpret_cast<const char *>(l) + u * user_stride;
                const char *bu = reinterpret_cast<const char *>(lbub) + u * user_stride;
                const float *b = reinterpret_cast<const float *>(bu);
                norm = psc_value((int)reinterpret_cast<const LT *>(lu)[c], __ldg(b + 2 * seg),
                                 __ldg(b + 2 * seg + 1), 1.0f / s);
            }
            float pr = __fmul_rn(__ldg(codebook + (int64_t)code * d + j), norm);
            acc = (u == 0) ? pr : __fadd_rn(acc, pr);
        }
        if (mean) acc = __fdiv_rn(acc, (float)n_users);
        if (accumulate) acc = combine1(out[e], acc, accumulate);
        out[e] = acc;
    }
}

// Power-of-two chunk sizes (D = 4, 8, 16): one warp owns 128 consecutive chunks per iteration,
// handled as four slots of 32 chunks (lane <-> chunk).  Per slot the code / level bytes of ALL
// users are loaded first (2U coalesced 32-byte requests in flight), the U norms are dequantized
// once, and the warp then writes the D4 rows of 32 float4 of that slot: the chunk of row r,
// lane L is q = (32 r + L) / D4 and lives in lane q of the slot, so (code, norm) arrive with
// two shuffles per user from statically indexed registers.  Users are summed in user order with
// separately rounded products (two packed mul.f32x2 per float4) and sums.
// Register use is independent of the number of users beyond the MAXU * 2 slot registers.
__device__ __forceinline__ float2 mul2(float2 a, float b)
{
    float2 r;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %4};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b));
    return r;
}
template <int D, int MAXU, typename CodeT, typename LT>
__global__ void __launch_bounds__(kDecodeThreads)
hsq_decode_reduce_warp_kernel(const CodeT *__restrict__ codes, const LT *__restrict__ l,
                              const float *__restrict__ lbub, const float *__restrict__ norms_f32,
                              const UserOffsets uoff, int n_users, int64_t n_chunks,
                              const float *__restrict__ codebook, int K,
                              const int64_t *__restrict__ seg_start, int n_seg, float s, int n_bit,
                              int mean, int accumulate, float *__restrict__ out)
{
    extern __shared__ float4 s_cbd[];
    constexpr int D4 = D / 4;
    static_assert((D4 & (D4 - 1)) == 0 && D4 <= 4, "D = 4, 8 or 16");
    const float4 *cb4g = reinterpret_cast<const float4 *>(codebook);
    pdl_launch_dependents();
    for (int i = threadIdx.x; i < K * D4; i += kDecodeThreads) s_cbd[i] = __ldg(cb4g + i);   // static codebook
    __syncthreads();
    pdl_wait();   // the packed records come from the encode kernels / the exchange
    const int lane = threadIdx.x & 31;
    constexpr int kWarps = kDecodeThreads / 32;
    const float inv_s = 1.0f / s;
    const float nu = (float)n_users;
    const bool pow2 = (n_users & (n_users - 1)) == 0;
    const float inv_nu = 1.0f / nu;
    SegCache segc;
    const int64_t n_slots = (n_chunks + 31) / 32;
    const int64_t n4 = n_chunks * D4;
    float4 *o4 = reinterpret_cast<float4 *>(out);
    for (int64_t slot = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); slot < n_slots;
         slot += (int64_t)gridDim.x * kWarps) {
        const int64_t c = slot * 32 + lane;
        const bool ok = c < n_chunks;
        int code[MAXU];
        float nrm[MAXU];
#pragma unroll
        for (int u = 0; u < MAXU; ++u) {
            code[u] = 0;
            nrm[u] = 0.0f;
            if (u < n_users && ok) {
                const char *cu = reinterpret_cast<const char *>(codes) + uoff.off[u];
                code[u] = (int)reinterpret_cast<const CodeT *>(cu)[c];
                if (n_bit == 32) {
                    const char *nf = reinterpret_cast<const char *>(norms_f32) + uoff.off[u];
                    nrm[u] = reinterpret_cast<const float *>(nf)[c];
                } else {
                    const char *lu = reinterpret_cast<const char *>(l) + uoff.off[u];
                    nrm[u] = (float)(int)reinterpret_cast<const LT *>(lu)[c];
                }
            }
        }
        if (n_bit != 32) {
            const int seg = ok ? cached_segment(segc, seg_start, n_seg, c) : 0;
#pragma unroll
            for (int u = 0; u < MAXU; ++u) {
                if (u < n_users) {
                    const float *b = reinterpret_cast<const float *>(reinterpret_cast<const char *>(lbub) + uoff.off[u]);
                    const float lb = __ldg(b + 2 * seg), ub = __ldg(b + 2 * seg + 1);
                    // l * (ub - lb) / 2^n + lb   (probabilistic_scalar_compressor.py:31-32)
                    nrm[u] = __fadd_rn(__fmul_rn(__fmul_rn(nrm[u], __fsub_rn(ub, lb)), inv_s), lb);
                }
            }
        }
        const int64_t f0 = slot * 32 * D4;
#pragma unroll
        for (int r = 0; r < D4; ++r) {
            const int fl = r * 32 + lane;
            const int owner = fl / D4;
            const int part = fl % D4;
            float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
#pragma unroll
            for (int u = 0; u < MAXU; ++u) {
                if (u < n_users) {
                    const int cd = __shfl_sync(0xffffffffu, code[u], owner);
                    const float nm = __shfl_sync(0xffffffffu, nrm[u], owner);
                    const float4 cw = s_cbd[cd * D4 + part];
                    const float2 p0 = mul2(make_float2(cw.x, cw.y), nm);
                    const float2 p1 = mul2(make_float2(cw.z, cw.w), nm);
                    if (u == 0) {
                        a0 = p0; a1 = p1;
                    } else {
                        // scalar adds: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (one
                        // rounding), which would break bit-exactness with the reference's mul-then-add
                        a0.x = __fadd_rn(a0.x, p0.x); a0.y = __fadd_rn(a0.y, p0.y);
                        a1.x = __fadd_rn(a1.x, p1.x); a1.y = __fadd_rn(a1.y, p1.y);
                    }
                }
            }
            float4 acc = make_float4(a0.x, a0.y, a1.x, a1.y);
            const int64_t f = f0 + fl;
            if (f < n4) {
                if (mean && n_users > 1) {
                    if (pow2) {
                        acc.x = __fmul_rn(acc.x, inv_nu); acc.y = __fmul_rn(acc.y, inv_nu);
                        acc.z = __fmul_rn(acc.z, inv_nu); acc.w = __fmul_rn(acc.w, inv_nu);
                    } else {
                        acc.x = __fdiv_rn(acc.x, nu); acc.y = __fdiv_rn(acc.y, nu);
                        acc.z = __fdiv_rn(acc.z, nu); acc.w = __fdiv_rn(acc.w, nu);
                    }
                }
                if (accumulate) {
                    const float4 o = o4[f];
                    acc = combine4(o, acc, accumulate);
                }
                o4[f] = acc;
            }
        }
    }
}

// Pull-and-decode for records that live in DIFFERENT buffers (one per user, typically peer GPU
// memory mapped over NVLink): d = 16, uint8 codes and levels.  Each CTA walks tiles of 1024 chunks;
// the code / level bytes of all users for the next tile are pulled with 16-byte cp.async (wide
// requests, bypassing L1) into a double-buffered shared-memory stage while the current tile is
// decoded, so every remote byte crosses NVLink exactly once and the transfer overlaps the decode:
// the exchange step needs no separate gather pass and no local copy of the peers' records.
// The lb/ub tables of all users are staged once per CTA.  The codebook is stored twice per
// codeword (128-byte slots): lanes 0-3 of a quarter-warp read the copy in bank groups 0-3, lanes
// 4-7 the copy in groups 4-7, so the two codewords a quarter-warp gathers never conflict.
constexpr int kStTile = 1024;
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc) : "memory");
}
// the first src_bytes (1..16) of the 16 come from gsrc, the rest is zero-filled
__device__ __forceinline__ void cp_async16_part(void *smem_dst, const void *gsrc, int src_bytes)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t saddr)
{
    float4 r;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(saddr));
    return r;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t saddr)
{
    uint32_t r;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"(saddr) : "memory");
    return r;
}
// QUANT (NU == 1): the record's levels are not there yet.  The search kernel left u and the per-tensor
// min/max keys behind (gq_hsq_encode_search); this kernel builds lb/ub from the keys, stages each tile's
// u in place of its level bytes, computes the tile's levels before decoding it (psc_levels4, as the
// encode's tail does), stores them over the first quarter of the staged u and into the record, and
// CTA 0 writes the lb/ub table: the record ends up complete.  The stage buffer grows from 2 KB to 5 KB,
// which keeps five CTAs per SM within the shared memory (and 48 registers) of the plain NU = 1 decode.
struct DecQuant {
    const float *u;
    const uint32_t *keys;
    const float *uniforms;   // nullptr: Philox4x32-10 (seed, offset + chunk)
    uint64_t seed, offset;
    int random;
};
// NU = exact number of users (compile time: the per-user loops are branch-free)
template <int NU, bool QUANT>
__global__ void __launch_bounds__(kDecodeThreads, QUANT ? 5 : 0)
hsq_decode_reduce_staged_kernel(const uint8_t *__restrict__ codes, uint8_t *__restrict__ l,
                                float *__restrict__ lbub, const UserOffsets uoff,
                                int64_t n_chunks, const float *__restrict__ codebook,
                                const int64_t *__restrict__ seg_start, int n_seg, float s, int mean,
                                int accumulate, float *__restrict__ out, const Rider rider, const PeerWait wait,
                                const DecQuant quant)
{
    static_assert(!QUANT || NU == 1, "levels are computed for one user's record");
    // one stage buffer: per user codes [1024] | levels [1024]; QUANT: codes [1024] | u [1024] (fp32), the
    // levels overwrite the first 1024 bytes of u
    constexpr int kBuf = NU * 2 * kStTile + (QUANT ? 3 * kStTile : 0);
    extern __shared__ float4 s_dyn[];
    float4 *s_cb = s_dyn;                                                    // [256][2][4]
    uint8_t *s_stage = reinterpret_cast<uint8_t *>(s_cb + 256 * 8);          // [2][kBuf]
    float2 *s_lbub = reinterpret_cast<float2 *>(s_stage + 2 * kBuf);         // [NU][n_seg]
    int64_t *s_seg = reinterpret_cast<int64_t *>(s_lbub + NU * n_seg);             // [n_seg + 1] tensor boundaries
    __shared__ int64_t s_off[8];
    const int tid = threadIdx.x, lane = tid & 31;
    // warp index through a shuffle: the compiler then knows it is warp-uniform, and the slot loop
    // below (with its warp shuffles) is compiled as convergent code
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    pdl_launch_dependents();
    if (tid == 0) {
#pragma unroll
        for (int u = 0; u < 8; ++u) s_off[u] = uoff.off[u];
    }
    for (int i = tid; i < 256 * 8; i += kDecodeThreads)
        s_cb[i] = __ldg(reinterpret_cast<const float4 *>(codebook) + (i >> 3) * 4 + (i & 3));
    for (int i = tid; i <= n_seg; i += kDecodeThreads) s_seg[i] = __ldg(seg_start + i);   // (a table of the plan, not of the step)
    __syncthreads();
    pdl_wait();   // the records are complete (and, across GPUs, announced by the barrier kernel)
    if (wait.n > 0) {   // ... or by the peers' encode kernels themselves: wait for every rank's delivery flag
        if (tid < wait.n) peer_wait_flag(wait.flags + tid, wait.epoch, wait.timeout_ns);
        __syncthreads();
    }
    const int64_t n_tiles = (n_chunks + kStTile - 1) / kStTile;
    auto issue = [&](int64_t tile, int buf) {
        const int64_t c0 = tile * kStTile;
        const int64_t left = n_chunks - c0;
        const int lim = (int)(left < kStTile ? left : (int64_t)kStTile);
        const int pieces = (lim + 15) >> 4;   // 16-byte pieces holding data
        if (QUANT) {   // codes, then u: 64 + 256 pieces
            for (int i = tid; i < 64 + 256; i += kDecodeThreads) {
                if (i < 64) {
                    if (i < pieces) cp_async16(s_stage + buf * kBuf + i * 16, codes + c0 + i * 16);
                } else {
                    const int p = i - 64;   // chunks 4p .. 4p + 3 of the tile
                    if (4 * p < lim)
                        cp_async16_part(s_stage + buf * kBuf + kStTile + p * 16, quant.u + c0 + 4 * p,
                                        4 * min(4, lim - 4 * p));
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            return;
        }
        for (int i = tid; i < NU * 128; i += kDecodeThreads) {
            const int u = i >> 7, which = (i >> 6) & 1, piece = i & 63;
            if (piece < pieces) {
                const char *src = (which ? reinterpret_cast<const char *>(l) : reinterpret_cast<const char *>(codes)) +
                                  s_off[u] + c0 + piece * 16;
                cp_async16(s_stage + buf * kBuf + (u * 2 + which) * kStTile + piece * 16, src);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const float inv_s = 1.0f / s;
    const float nu = (float)NU;
    constexpr bool pow2 = (NU & (NU - 1)) == 0;
    const float inv_nu = 1.0f / nu;
    // 32-bit shared-window addresses: this lane's 16-byte unit inside a codeword slot, the stage
    const uint32_t cb_lane = (uint32_t)__cvta_generic_to_shared(s_cb) + (uint32_t)(((lane >> 2) & 1) * 64 + (lane & 3) * 16);
    const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(s_stage);
    SegCache segc;
    float4 *o4 = reinterpret_cast<float4 *>(out);
    const int64_t n4 = n_chunks * 4;
    // (32-bit tile indices in the QUANT kernel: what keeps it within 48 registers without spills)
    std::conditional_t<QUANT, int, int64_t> tile = blockIdx.x;
    int buf = 0;
    if (tile < n_tiles) issue(tile, 0);
    // while the first tile is in flight: the users' (lb, ub) tables (read before the first decode,
    // i.e. after the block barrier that follows the tile's arrival) ...
    if (QUANT) {
        for (int i = tid; i < n_seg; i += kDecodeThreads) {
            const float lb = key_to_float(__ldcg(quant.keys + 2 * i)), ub = key_to_float(__ldcg(quant.keys + 2 * i + 1));
            s_lbub[i] = make_float2(lb, ub);
            if (blockIdx.x == 0) {   // the reference returns lb/ub (probabilistic_scalar_compressor.py:27)
                lbub[2 * i] = lb;
                lbub[2 * i + 1] = ub;
            }
        }
    } else {
        for (int i = tid; i < NU * n_seg; i += kDecodeThreads) {
            const int u = i / n_seg, sg = i - u * n_seg;
            const float2 *b = reinterpret_cast<const float2 *>(reinterpret_cast<const char *>(lbub) + s_off[u]);
            s_lbub[i] = __ldcv(b + sg);
        }
    }
    // ... and the attached small reduction (identity tensors)
    rider_run(rider, (int64_t)blockIdx.x * kDecodeThreads + tid, (int64_t)gridDim.x * kDecodeThreads);
    for (; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
        const auto next = tile + gridDim.x;
        if (next < n_tiles) {
            issue(next, buf ^ 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const uint32_t st = stage0 + (uint32_t)(buf * kBuf);
        const int64_t c0 = tile * kStTile;
        if (QUANT) {
            // levels of chunks c0 + 4 tid .. + 3: into the record and, once every thread has read its u,
            // over the first 1024 bytes of the staged u, where the decode below reads the level bytes
            const int i0 = (int)c0 + 4 * tid, n = (int)n_chunks;   // n_chunks < 2^31 (gq_hsq_decode_quantize)
            uint32_t packed = 0u;
            uint32_t *s_lv = reinterpret_cast<uint32_t *>(s_stage + buf * kBuf + kStTile);
            if (i0 < n) {
                const float4 xv = reinterpret_cast<const float4 *>(s_lv)[tid];
                const float x[4] = {xv.x, xv.y, xv.z, xv.w};
                float r[4] = {0.f, 0.f, 0.f, 0.f};
                if (quant.random) {
                    if (quant.uniforms != nullptr) {
                        if (i0 + 3 < n) {
                            const float4 t = __ldg(reinterpret_cast<const float4 *>(quant.uniforms + i0));
                            r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
                        } else {
#pragma unroll
                            for (int t = 0; t < 4; ++t) r[t] = (i0 + t < n) ? __ldg(quant.uniforms + i0 + t) : 0.0f;
                        }
                    } else {
                        philox_uniform4(quant.seed, quant.offset, (uint64_t)i0, r);
                    }
                }
                int seg = cached_segment_smem(segc, s_seg, n_seg, (int64_t)i0);
                int lv[4];
                psc_levels4(x, r, i0, n, s_seg, s_lbub, seg, s, quant.random, lv);
                packed = (uint32_t)lv[0] | ((uint32_t)lv[1] << 8) | ((uint32_t)lv[2] << 16) | ((uint32_t)lv[3] << 24);
                if (i0 + 3 < n) {
                    reinterpret_cast<uint32_t *>(l)[i0 >> 2] = packed;
                } else {
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        if (i0 + t < n) l[i0 + t] = (uint8_t)lv[t];
                }
            }
            __syncthreads();
            s_lv[tid] = packed;
            __syncthreads();
        }
        for (int sl = warp; sl < kStTile / 32; sl += kDecodeThreads / 32) {
            const int64_t c = c0 + sl * 32 + lane;
            if (c0 + sl * 32 >= n_chunks) break;
            const bool ok = c < n_chunks;
            const int seg = ok ? cached_segment_smem(segc, s_seg, n_seg, c) : 0;
            // Three or more users: when the whole slot lies in one tensor (almost always), a lane
            // hands (code, level) of TWO users to the writers in one shuffle and the writers
            // dequantize the norm themselves (same three rounded operations) -- the kernel is bound
            // by the LSU/shuffle pipe there, not by ALU.  Otherwise: code and norm, one shuffle each.
            constexpr bool kPack = NU >= 3;
            const int seg0 = __shfl_sync(0xffffffffu, seg, 0);
            const bool uni = kPack && __all_sync(0xffffffffu, !ok || seg == seg0);
            uint32_t code[NU];
            float nrm[NU];          // !uni: dequantized norm of this lane's chunk; uni: lb of (user, tensor)
            float den[NU];          // uni: ub - lb of (user, tensor)
            uint32_t pk[(NU + 1) / 2];
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                const uint32_t cb8 = lds_u8(st + (uint32_t)((u * 2) * kStTile + sl * 32 + lane));
                const uint32_t lv8 = lds_u8(st + (uint32_t)((u * 2 + 1) * kStTile + sl * 32 + lane));
                const float2 b = s_lbub[u * n_seg + (uni ? seg0 : seg)];
                code[u] = cb8 << 7;   // byte offset of the codeword's slot
                den[u] = __fsub_rn(b.y, b.x);
                if (uni) {
                    nrm[u] = b.x;
                    const uint32_t h = cb8 | (lv8 << 8);
                    if (u & 1) pk[u >> 1] |= h << 16; else pk[u >> 1] = h;
                } else {
                    // l * (ub - lb) / 2^n + lb   (probabilistic_scalar_compressor.py:31-32)
                    nrm[u] = __fadd_rn(__fmul_rn(__fmul_rn((float)(int)lv8, den[u]), inv_s), b.x);
                }
            }
            const int64_t f0 = (c0 + sl * 32) * 4;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int owner = r * 8 + (lane >> 2);
                float4 cw[NU];
                float nm[NU];
                if (uni) {
#pragma unroll
                    for (int j = 0; j < (NU + 1) / 2; ++j) {
                        const uint32_t w = __shfl_sync(0xffffffffu, pk[j], owner);
                        cw[2 * j] = lds128(cb_lane + ((w & 0xffu) << 7));
                        nm[2 * j] = __fadd_rn(__fmul_rn(__fmul_rn((float)(int)((w >> 8) & 0xffu), den[2 * j]), inv_s), nrm[2 * j]);
                        if (2 * j + 1 < NU) {
                            cw[2 * j + 1] = lds128(cb_lane + (((w >> 16) & 0xffu) << 7));
                            nm[2 * j + 1] = __fadd_rn(__fmul_rn(__fmul_rn((float)(int)(w >> 24), den[2 * j + 1]), inv_s), nrm[2 * j + 1]);
                        }
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < NU; ++u) {
                        const uint32_t cd = __shfl_sync(0xffffffffu, code[u], owner);
                        nm[u] = __shfl_sync(0xffffffffu, nrm[u], owner);
                        cw[u] = lds128(cb_lane + cd);
                    }
                }
                float2 a0 = mul2(make_float2(cw[0].x, cw[0].y), nm[0]);
                float2 a1 = mul2(make_float2(cw[0].z, cw[0].w), nm[0]);
#pragma unroll
                for (int u = 1; u < NU; ++u) {
                    const float2 p0 = mul2(make_float2(cw[u].x, cw[u].y), nm[u]);
                    const float2 p1 = mul2(make_float2(cw[u].z, cw[u].w), nm[u]);
                    // scalar adds: see hsq_decode_reduce_warp_kernel.  (Packed alternative that stays exact: the
                    // product as FFMA2 with a -0.0 addend from a kernel argument + FADD2 -- ptxas never fuses an
                    // fma with an add.  Measured: 46.9 us either way at U = 8; packed ops save no issue slots.)
                    a0.x = __fadd_rn(a0.x, p0.x); a0.y = __fadd_rn(a0.y, p0.y);
                    a1.x = __fadd_rn(a1.x, p1.x); a1.y = __fadd_rn(a1.y, p1.y);
                }
                float4 acc = make_float4(a0.x, a0.y, a1.x, a1.y);
                const int64_t f = f0 + r * 32 + lane;
                if (f < n4) {
                    if (mean && NU > 1) {
                        if (pow2) {
                            acc.x = __fmul_rn(acc.x, inv_nu); acc.y = __fmul_rn(acc.y, inv_nu);
                            acc.z = __fmul_rn(acc.z, inv_nu); acc.w = __fmul_rn(acc.w, inv_nu);
                        } else {
                            acc.x = __fdiv_rn(acc.x, nu); acc.y = __fdiv_rn(acc.y, nu);
                            acc.z = __fdiv_rn(acc.z, nu); acc.w = __fdiv_rn(acc.w, nu);
                        }
                    }
                    if (accumulate) {
                        const float4 o = o4[f];
                        acc = combine4(o, acc, accumulate);
                    }
                    o4[f] = acc;
                }
            }
        }
        __syncthreads();   // this stage buffer is refilled by the next iteration's prefetch
    }
}

template <int NU, bool QUANT = false>
static int launch_decode_staged(const void *codes, const void *l, const float *lbub, const UserOffsets &uoff,
                                int64_t n_chunks, const float *codebook, const int64_t *seg_start,
                                int n_seg, float s, int mean, int accumulate, float *out, cudaStream_t st,
                                const DecQuant &quant = DecQuant{})
{
    auto kern = hsq_decode_reduce_staged_kernel<NU, QUANT>;
    const size_t buf = (size_t)NU * 2 * kStTile + (QUANT ? 3 * kStTile : 0);
    const size_t smem = 256 * 128 + 2 * buf + (size_t)NU * n_seg * 8 + (size_t)(n_seg + 1) * 8;
    GQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    GQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kDecodeThreads, smem));
    const int64_t n_tiles = (n_chunks + kStTile - 1) / kStTile;
    const int64_t cap = (int64_t)sm_count() * (occ < 1 ? 1 : occ);
    // the same number of tiles for every CTA (to within one): no CTA is left with a straggler tile
    const int64_t per = (n_tiles + cap - 1) / cap;
    int64_t grid = (n_tiles + per - 1) / per;
    if (grid < 1) grid = 1;
    const Rider rider = take_rider();   // carried by this launch if one is pending
    const PeerWait wait = take_wait();  // likewise: the wait for the peers' delivery flags
    GQ_CUDA(launch_pdl(kern, dim3((unsigned)grid), dim3(kDecodeThreads), smem, st, (const uint8_t *)codes,
                       (uint8_t *)l, (float *)lbub, uoff, n_chunks, codebook, seg_start, n_seg, s, mean,
                       accumulate, out, rider, wait, quant));
    return GQ_OK;
}

int hsq_decode_quantize(const void *codes, void *l, float *lbub, const float *u, const uint32_t *keys,
                        int64_t n_chunks, const float *codebook, const int64_t *seg_start, int n_seg, int n_bit,
                        int random, const float *uniforms, uint64_t seed, uint64_t offset, int accumulate,
                        float *out, cudaStream_t st)
{
    UserOffsets uoff = {};
    const DecQuant quant = {u, keys, uniforms, seed, offset, random};
    return launch_decode_staged<1, true>(codes, l, lbub, uoff, n_chunks, codebook, seg_start, n_seg,
                                         (float)(1u << n_bit), 0, accumulate, out, st, quant);
}

template <int D, int MAXU, typename CodeT, typename LT>
static int launch_decode_warp(const void *codes, const void *l, const float *lbub, const float *norms_f32,
                              const UserOffsets &uoff, int n_users, int64_t n_chunks, const float *codebook,
                              int K, const int64_t *seg_start, int n_seg, float s, int n_bit, int mean,
                              int accumulate, float *out, cudaStream_t st)
{
    const size_t cb_bytes = (size_t)K * D * 4;
    auto kern = hsq_decode_reduce_warp_kernel<D, MAXU, CodeT, LT>;
    GQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cb_bytes));
    int occ = 1;
    GQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kDecodeThreads, cb_bytes));
    const int64_t iters = (n_chunks + 31) / 32;
    const int64_t wblocks = (iters + kDecodeThreads / 32 - 1) / (kDecodeThreads / 32);
    int64_t cap = (int64_t)sm_count() * (occ < 1 ? 1 : occ);
    int grid = (int)(wblocks < cap ? wblocks : cap);
    GQ_CUDA(launch_pdl(kern, dim3(grid < 1 ? 1 : grid), dim3(kDecodeThreads), cb_bytes, st, (const CodeT *)codes,
                       (const LT *)l, lbub, norms_f32, uoff, n_users, n_chunks, codebook, K, seg_start, n_seg, s,
                       n_bit, mean, accumulate, out));
    return GQ_OK;
}

template <int D, typename CodeT, typename LT>
static int launch_decode_d(const void *codes, const void *l, const float *lbub, const float *norms_f32,
                           int64_t user_stride, const int64_t *user_offsets, int n_users, int64_t n_chunks,
                           const float *codebook, int K, const int64_t *seg_start, int n_seg, int n_bit,
                           int mean, int accumulate, float *out, cudaStream_t st)
{
    const float s = (n_bit == 32) ? 1.0f : (float)(1u << n_bit);
    const size_t cb_bytes = (size_t)K * D * 4;
    const int64_t span = (int64_t)kDecodeThreads * kDecodeUnroll;
    const int64_t blocks = (n_chunks * (D / 4) + span - 1) / span;
    constexpr int D4c = D / 4;
    constexpr bool kWarpPath = ((D4c & (D4c - 1)) == 0) && D4c <= 4;   // D = 4, 8, 16
    constexpr int DW = kWarpPath ? D : 16;
    if (kWarpPath && cb_bytes <= 64 * 1024 && n_users <= 8) {
        UserOffsets uoff;
        for (int u = 0; u < 8; ++u)
            uoff.off[u] = (u < n_users) ? (user_offsets ? user_offsets[u] : (int64_t)u * user_stride) : 0;
        // records in separate (peer) buffers: pull-and-decode through a shared-memory stage
        // and for local records as well: measured faster than the warp kernel for every U
        // (U = 1: 23 vs 27 us, U = 8: 76 vs 83 us on the ResNet-50 record); GQ_DECODE_STAGED=0 = old path
        bool staged = true;
        if (const char *e = getenv("GQ_DECODE_STAGED")) staged = atoi(e) != 0;
        if (staged && D == 16 && K == 256 && sizeof(CodeT) == 1 && sizeof(LT) == 1 && n_bit != 32 &&
            (size_t)n_users * n_seg * 8 <= 48 * 1024) {
            bool aligned = (((uintptr_t)codes | (uintptr_t)l | (uintptr_t)lbub) & 15) == 0;
            for (int u = 0; u < n_users; ++u) aligned = aligned && ((uoff.off[u] & 15) == 0);
            if (aligned) {
#define GQ_S(MU) case MU: return launch_decode_staged<MU>(codes, l, lbub, uoff, n_chunks, codebook, seg_start, n_seg, s, mean, accumulate, out, st)
                switch (n_users) {
                    GQ_S(1); GQ_S(2); GQ_S(3); GQ_S(4); GQ_S(5); GQ_S(6); GQ_S(7); GQ_S(8);
                    default: break;
                }
#undef GQ_S
            }
        }
        GQ_CUDA_INT(flush_wait(st));
#define GQ_W(MU) return launch_decode_warp<DW, MU, CodeT, LT>(codes, l, lbub, norms_f32, uoff, n_users, n_chunks, codebook, K, seg_start, n_seg, s, n_bit, mean, accumulate, out, st)
        if (n_users == 1) GQ_W(1);
        if (n_users == 2) GQ_W(2);
        if (n_users <= 4) GQ_W(4);
        GQ_W(8);
#undef GQ_W
    }
    if (user_offsets != nullptr) {
        set_error("scattered user records need chunk dim 4/8/16, a codebook <= 64 KB and <= 8 users");
        return GQ_ERR_UNSUPPORTED;
    }
    GQ_CUDA_INT(flush_wait(st));
    if (cb_bytes <= 64 * 1024) {
        auto kern = hsq_decode_reduce_kernel<D, CodeT, LT, true>;
        GQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cb_bytes));
        // persistent: the codebook is staged once per CTA; exactly one resident wave
        int occ = 1;
        GQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kDecodeThreads, cb_bytes));
        int64_t cap = (int64_t)sm_count() * (occ < 1 ? 1 : occ);
        int grid = (int)(blocks < cap ? blocks : cap);
        kern<<<grid < 1 ? 1 : grid, kDecodeThreads, cb_bytes, st>>>(
            (const CodeT *)codes, (const LT *)l, lbub, norms_f32, user_stride, n_users, n_chunks,
            codebook, K, seg_start, n_seg, s, n_bit, mean, accumulate, out);
    } else {
        auto kern = hsq_decode_reduce_kernel<D, CodeT, LT, false>;
        int64_t cap = (int64_t)sm_count() * 8;
        int grid = (int)(blocks < cap ? blocks : cap);
        kern<<<grid < 1 ? 1 : grid, kDecodeThreads, 0, st>>>(
            (const CodeT *)codes, (const LT *)l, lbub, norms_f32, user_stride, n_users, n_chunks,
            codebook, K, seg_start, n_seg, s, n_bit, mean, accumulate, out);
    }
    GQ_LAUNCH_CHECK("hsq_decode_reduce");
    return GQ_OK;
}

template <typename CodeT, typename LT>
static int launch_decode(const void *codes, const void *l, const float *lbub, const float *norms_f32,
                         int64_t user_stride, const int64_t *user_offsets, int n_users, int64_t n_chunks, int d,
                         const float *codebook, int K, const int64_t *seg_start, int n_seg, int n_bit,
                         int mean, int accumulate, float *out, cudaStream_t st)
{
    switch (d) {
#define GQ_CASE(DD) case DD: return launch_decode_d<DD, CodeT, LT>(codes, l, lbub, norms_f32, user_stride, user_offsets, n_users, n_chunks, codebook, K, seg_start, n_seg, n_bit, mean, accumulate, out, st);
        GQ_CASE(4) GQ_CASE(8) GQ_CASE(12) GQ_CASE(16) GQ_CASE(24) GQ_CASE(32) GQ_CASE(48) GQ_CASE(64)
#undef GQ_CASE
        default: break;
    }
    if (user_offsets != nullptr) {
        set_error("scattered user records are not supported for chunk dim %d", d);
        return GQ_ERR_UNSUPPORTED;
    }
    const float s = (n_bit == 32) ? 1.0f : (float)(1u << n_bit);
    GQ_CUDA_INT(flush_wait(st));
    hsq_decode_reduce_generic_kernel<CodeT, LT><<<grid_for(n_chunks * (int64_t)d, 256), 256, 0, st>>>(
        (const CodeT *)codes, (const LT *)l, lbub, norms_f32, user_stride, n_users, n_chunks, d,
        codebook, seg_start, n_seg, s, n_bit, mean, accumulate, out);
    GQ_LAUNCH_CHECK("hsq_decode_reduce_generic");
    return GQ_OK;
}

int hsq_decode_reduce(const void *codes, int code_bytes, const void *l, int l_bytes, const float *lbub,
                      const float *norms_f32, int64_t user_stride, const int64_t *user_offsets, int n_users,
                      int64_t n_chunks, int d,
                      const float *codebook, int K, const int64_t *seg_start, int n_seg, int n_bit,
                      int mean, int accumulate, float *out, cudaStream_t st)
{
    if (n_chunks == 0) return GQ_OK;
#define GQ_GO(CT, LTT) return launch_decode<CT, LTT>(codes, l, lbub, norms_f32, user_stride, user_offsets, n_users, n_chunks, d, codebook, K, seg_start, n_seg, n_bit, mean, accumulate, out, st)
    if (code_bytes == 1 && l_bytes == 1) GQ_GO(uint8_t, uint8_t);
    if (code_bytes == 1 && l_bytes == 4) GQ_GO(uint8_t, int32_t);
    if (code_bytes == 4 && l_bytes == 1) GQ_GO(int32_t, uint8_t);
    GQ_GO(int32_t, int32_t);
#undef GQ_GO
}

// ------------------------------------------------------ fp32 user reduction ---
__global__ void __launch_bounds__(256)
f32_reduce_users_kernel(const float *__restrict__ in, int64_t user_stride, int n_users, int64_t n,
                        int mean, int accumulate, float *__restrict__ out)
{
    pdl_launch_dependents();
    pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        float acc = in[i];
        for (int u = 1; u < n_users; ++u)
            acc = __fadd_rn(acc, *reinterpret_cast<const float *>(
                                     reinterpret_cast<const char *>(in) + u * user_stride + 4 * i));
        if (mean) acc = __fdiv_rn(acc, (float)n_users);
        if (accumulate) acc = combine1(out[i], acc, accumulate);
        out[i] = acc;
    }
}

__global__ void __launch_bounds__(256)
f32_reduce_users_scattered_kernel(const float *__restrict__ in, const UserOffsets uoff, int n_users, int64_t n,
                                  int mean, int accumulate, float *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        float acc = 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (u < n_users) {
                const float x = *reinterpret_cast<const float *>(reinterpret_cast<const char *>(in) + uoff.off[u] + 4 * i);
                acc = (u == 0) ? x : __fadd_rn(acc, x);
            }
        }
        if (mean) acc = __fdiv_rn(acc, (float)n_users);
        if (accumulate) acc = combine1(out[i], acc, accumulate);
        out[i] = acc;
    }
}

int launch_f32_reduce_users(const float *in, int64_t user_stride, const int64_t *user_offsets, int n_users,
                            int64_t n, int mean, int accumulate, float *out, cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    if (user_offsets != nullptr) {
        GQ_REQUIRE(n_users <= 8, "scattered user records support at most 8 users");
        UserOffsets uoff;
        for (int u = 0; u < 8; ++u) uoff.off[u] = (u < n_users) ? user_offsets[u] : 0;
        f32_reduce_users_scattered_kernel<<<grid_for(n, 256), 256, 0, st>>>(in, uoff, n_users, n, mean, accumulate, out);
        GQ_LAUNCH_CHECK("f32_reduce_users_scattered");
        return GQ_OK;
    }
    GQ_CUDA(launch_pdl(f32_reduce_users_kernel, dim3(grid_for(n, 256)), dim3(256), 0, st, in, user_stride, n_users,
                       n, mean, accumulate, out));
    return GQ_OK;
}

// ---------------------------------------------------------- attached reduction ---
// ---- pending wait for the peers' delivery flags (fused peer-to-peer push) ----
static thread_local PeerWait g_wait = {};
void set_wait(const PeerWait &w) { g_wait = w; }
PeerWait take_wait()
{
    PeerWait w = g_wait;
    g_wait = PeerWait{};
    return w;
}
__global__ void peer_wait_kernel(const PeerWait wait)
{
    pdl_launch_dependents();
    pdl_wait();
    if ((int)threadIdx.x < wait.n) peer_wait_flag(wait.flags + threadIdx.x, wait.epoch, wait.timeout_ns);
}
int flush_wait(cudaStream_t st)
{
    const PeerWait w = take_wait();
    if (w.n <= 0) return GQ_OK;
    GQ_CUDA(launch_pdl(peer_wait_kernel, dim3(1), dim3(32), 0, st, w));
    return GQ_OK;
}

static thread_local Rider g_rider = {};

void set_rider(const Rider &r) { g_rider = r; }

Rider take_rider()
{
    Rider r = g_rider;
    g_rider = Rider{};
    return r;
}

__global__ void __launch_bounds__(256) rider_kernel(const Rider rider)
{
    pdl_launch_dependents();
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * 256 + threadIdx.x, (int64_t)gridDim.x * 256);
}

int launch_rider(const Rider &r, cudaStream_t st)
{
    if (r.n == 0) return GQ_OK;
    GQ_CUDA(launch_pdl(rider_kernel, dim3(grid_for(r.n, 256)), dim3(256), 0, st, r));
    return GQ_OK;
}

// ------------------------------------------------------------- elementwise ---
__global__ void __launch_bounds__(256)
axpy_kernel(const float *__restrict__ a, const float *__restrict__ b, float alpha, int64_t n,
            float *__restrict__ out, int sub)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        out[i] = sub ? __fsub_rn(a[i], b[i]) : __fadd_rn(a[i], __fmul_rn(alpha, b[i]));
    }
}

int launch_axpy(const float *a, const float *b, float alpha, int64_t n, float *out, int sub,
                cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    axpy_kernel<<<grid_for(n, 256), 256, 0, st>>>(a, b, alpha, n, out, sub);
    GQ_LAUNCH_CHECK("axpy");
    return GQ_OK;
}

}  // namespace gq

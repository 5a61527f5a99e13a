// abi.cu -- the extern "C" surface of libgqb200.so (see include/gqb200.h).
// Argument validation, workspace carving and kernel dispatch only; the kernels
// live in the other translation units.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "gq_internal.cuh"

namespace gq {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return GQ_OK;
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return GQ_ERR_CUDA;
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

bool pdl_enabled()
{
    static const bool on = [] { const char *f = getenv("GQ_PDL"); return !(f && atoi(f) == 0); }();
    return on;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// GQ_TC_V=1: first-generation tcgen05 search (hsq_tc.cu) + separate quantize launch; default 2 (hsq_tc2.cu).
// Read at every call so that one process can A/B the two.
int tc_generation()
{
    const char *f = getenv("GQ_TC_V");
    return (f && atoi(f) == 1) ? 1 : 2;
}

static thread_local Tc2Remote g_remote = {};
void set_remote(const Tc2Remote &r) { g_remote = r; }
Tc2Remote take_remote()
{
    Tc2Remote r = g_remote;
    g_remote = Tc2Remote{};
    return r;
}

}  // namespace gq

using namespace gq;

extern "C" {

const char *gq_last_error(void) { return g_err; }
int gq_abi_version(void) { return 1; }

int gq_device_info(int *sm, int *cc_major, int *cc_minor, size_t *total_mem)
{
    int dev = 0;
    GQ_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    GQ_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm) *sm = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = p.totalGlobalMem;
    return GQ_OK;
}

// ------------------------------------------------------------------ HSQ ---
size_t gq_hsq_encode_workspace_bytes(int64_t n_chunks, int d, int K, int n_seg)
{
    (void)d; (void)K;
    size_t keys = align_up((size_t)(n_seg > 0 ? n_seg : 1) * 2 * sizeof(uint32_t), 256);
    return keys + 256 /* grid barrier word */ + hsq_tc_workspace_bytes(n_chunks) + hsq_tck_workspace_bytes(d, K);
}

static int validate_group(const void *grad, int64_t n_chunks, int d, const void *codebook, int K,
                          const int64_t *seg_start, int n_seg)
{
    GQ_REQUIRE(n_chunks >= 0, "n_chunks %lld < 0", (long long)n_chunks);
    GQ_REQUIRE(d >= 1, "chunk dim %d < 1", d);
    GQ_REQUIRE(K >= 1, "codebook size %d < 1", K);
    GQ_REQUIRE(n_chunks == 0 || grad != nullptr, "null gradient pointer");
    GQ_REQUIRE(codebook != nullptr, "null codebook pointer");
    GQ_REQUIRE(n_seg >= 1 && seg_start != nullptr, "segment table required (n_seg >= 1)");
    return GQ_OK;
}

int gq_hsq_search(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                  void *codes, int code_bytes, float *u_out, const int64_t *seg_start, int n_seg,
                  uint32_t *minmax_keys, void *workspace, size_t workspace_bytes, int algo,
                  gq_stream_t stream)
{
    int e = validate_group(grad, n_chunks, d, codebook, K, seg_start, n_seg);
    if (e) return e;
    GQ_REQUIRE(code_bytes == 1 || code_bytes == 4, "code_bytes must be 1 or 4 (got %d)", code_bytes);
    GQ_REQUIRE(code_bytes == 4 || K <= 256, "uint8 codes need K <= 256 (K = %d)", K);
    GQ_REQUIRE(n_chunks == 0 || (codes && u_out), "null output pointer");
    GQ_REQUIRE(((uintptr_t)grad & 15) == 0, "gradient must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const bool tc_ok = tc_generation() == 2 ? hsq_tc2_supported(d, K, code_bytes) : hsq_tc_supported(d, K, code_bytes);
    const bool tck_ok = !tc_ok && hsq_tck_supported(d, K, code_bytes) && workspace != nullptr &&
                        ((uintptr_t)workspace & 255) == 0 && workspace_bytes >= hsq_tck_workspace_bytes(d, K);
    if (algo == GQ_ALGO_TC && !tc_ok && !tck_ok) {
        set_error("tcgen05 search supports d in {8, 16, 32} with K == 256 (uint8 codes) or d == 16 with K = 512..4096, a multiple of 512 "
                  "(int32 codes, workspace of gq_hsq_encode_workspace_bytes); got d=%d K=%d code_bytes=%d",
                  d, K, code_bytes);
        return GQ_ERR_UNSUPPORTED;
    }
    if (tck_ok && algo != GQ_ALGO_EXACT && n_chunks > 0)
        return hsq_search_tck(grad, n_chunks, codebook, K, codes, u_out, seg_start, n_seg, minmax_keys, workspace,
                              workspace_bytes, st);
    if (tc_ok && algo != GQ_ALGO_EXACT && n_chunks > 0) {
        if (tc_generation() == 1)
            return hsq_search_tc(grad, n_chunks, d, codebook, K, codes, code_bytes, u_out, seg_start, n_seg,
                                 minmax_keys, workspace, workspace_bytes, st);
        // keys (when given) were initialised by the caller: no in-kernel reset, no tail
        return hsq_encode_tc2(grad, n_chunks, d, codebook, codes, u_out, seg_start, n_seg, minmax_keys, nullptr, nullptr,
                              Rider{}, nullptr, nullptr, st);
    }
    return hsq_search_exact(grad, n_chunks, d, codebook, K, codes, code_bytes, u_out, seg_start, n_seg,
                            minmax_keys, st);
}

int gq_hsq_tc2_trace(const float *grad, int64_t n_chunks, const float *codebook, void *codes, float *u_out,
                     const int64_t *seg_start, int n_seg, void *l, float *lbub, void *workspace, int64_t *trace,
                     gq_stream_t stream)
{
    GQ_REQUIRE(hsq_tc_supported(16, 256, 1), "tcgen05 search needs an sm_100 device");
    if (l == nullptr)
        return hsq_tc2_trace(grad, n_chunks, codebook, codes, u_out, nullptr, 0, nullptr, nullptr, nullptr, nullptr,
                             reinterpret_cast<long long *>(trace), as_stream(stream));
    GQ_REQUIRE(seg_start && n_seg >= 1 && lbub && workspace && ((uintptr_t)workspace & 255) == 0, "bad arguments");
    uint32_t *keys = reinterpret_cast<uint32_t *>(workspace);
    uint32_t *barrier = reinterpret_cast<uint32_t *>((char *)workspace + align_up((size_t)n_seg * 8, 256));
    Tc2Tail tail = {(uint8_t *)l, lbub, nullptr, 1234u, 0u, 6, 1};
    return hsq_tc2_trace(grad, n_chunks, codebook, codes, u_out, seg_start, n_seg, keys, reinterpret_cast<uint64_t *>(barrier) + 1,
                         barrier, &tail, reinterpret_cast<long long *>(trace), as_stream(stream));
}

int gq_norm_quantize(const float *u, int64_t n, const int64_t *seg_start, int n_seg, int n_bit,
                     int random, const float *uniforms, uint64_t philox_seed, uint64_t philox_offset,
                     void *l, int l_bytes, float *lbub, uint32_t *minmax_keys, int precomputed,
                     gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && n_seg >= 1 && seg_start, "bad segment table");
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 24, "n_bit %d out of range 1..24", n_bit);
    GQ_REQUIRE(l_bytes == 1 || l_bytes == 4, "l_bytes must be 1 or 4");
    GQ_REQUIRE(l_bytes == 4 || n_bit <= 7, "uint8 norm codes need n_bit <= 7 (levels 0..2^n)");
    GQ_REQUIRE(l && lbub && minmax_keys, "null output pointer");
    cudaStream_t st = as_stream(stream);
    if (!precomputed) {
        int e = launch_minmax_init(minmax_keys, n_seg, st);
        if (e) return e;
        e = launch_seg_minmax(u, n, seg_start, n_seg, minmax_keys, st);
        if (e) return e;
    }
    return launch_norm_quantize(u, n, seg_start, n_seg, n_bit, random, uniforms, philox_seed,
                                philox_offset, l, l_bytes, lbub, minmax_keys, st);
}

int gq_norm_dequantize(const void *l, int l_bytes, int64_t n, const int64_t *seg_start, int n_seg,
                       int n_bit, const float *lbub, float *out, gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && n_seg >= 1 && seg_start, "bad segment table");
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 24, "n_bit %d out of range 1..24", n_bit);
    GQ_REQUIRE(l_bytes == 1 || l_bytes == 4, "l_bytes must be 1 or 4");
    return launch_norm_dequantize(l, l_bytes, n, seg_start, n_seg, n_bit, lbub, out, as_stream(stream));
}

int gq_hsq_encode(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                  const int64_t *seg_start, int n_seg, int n_bit, int random, const float *uniforms,
                  uint64_t philox_seed, uint64_t philox_offset, void *codes, int code_bytes, void *l,
                  int l_bytes, float *lbub, float *u_out, void *workspace, size_t workspace_bytes,
                  int algo, gq_stream_t stream)
{
    // pending attachments are consumed (hence cleared) first, whatever happens below
    const Rider rider = take_rider();   // identity copy, if any: rides in the search (tcgen05) or init kernel
    const Tc2Remote remote = take_remote();
    GQ_REQUIRE(n_bit == 32 || (n_bit >= 1 && n_bit <= 24), "n_bit %d out of range (1..24 or 32)", n_bit);
    const size_t need = gq_hsq_encode_workspace_bytes(n_chunks, d, K, n_seg);
    if (workspace_bytes < need || workspace == nullptr) {
        set_error("workspace too small: %zu < %zu", workspace_bytes, need);
        return GQ_ERR_WORKSPACE;
    }
    GQ_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = as_stream(stream);
    uint32_t *keys = reinterpret_cast<uint32_t *>(workspace);
    const size_t keys_bytes = align_up((size_t)n_seg * 2 * sizeof(uint32_t), 256);
    uint32_t *barrier = reinterpret_cast<uint32_t *>((char *)workspace + keys_bytes);
    const size_t head = keys_bytes + 256;
    int e = GQ_OK;
    // Optional single-launch encode (search + grid barrier + norm quantization inside the
    // persistent tcgen05 kernel).  Measured on B200 (ResNet-50 gradient): 93.7 us fused vs
    // 80.5 + 9.7 us as two kernels -- the quantization tail runs at 512 threads/SM inside the
    // persistent kernel -- so it is opt-in (GQ_TC_FUSED=1) until the tail is restructured.
    static const bool want_fused = [] { const char *f = getenv("GQ_TC_FUSED"); return f && atoi(f) == 1; }();
    const bool fused = want_fused && (n_bit != 32) && (l_bytes == 1) && (algo != GQ_ALGO_EXACT) && n_chunks > 0 &&
                       hsq_tc_supported(d, K, code_bytes);
    if (fused) {
        e = validate_group(grad, n_chunks, d, codebook, K, seg_start, n_seg);
        if (e) return e;
        GQ_REQUIRE(codes && l && lbub && u_out, "null output pointer");
        GQ_REQUIRE(n_bit <= 7, "uint8 norm codes need n_bit <= 7 (levels 0..2^n)");
        GQ_REQUIRE(((uintptr_t)grad & 15) == 0, "gradient must be 16-byte aligned");
        e = launch_minmax_init_rider(keys, n_seg, st, barrier, rider);
        if (e) return e;
        return hsq_encode_tc_fused(grad, n_chunks, codebook, codes, u_out, seg_start, n_seg, keys, barrier, n_bit,
                                   random, uniforms, philox_seed, philox_offset, (uint8_t *)l, lbub, st);
    }
    const bool tc2_ok = tc_generation() == 2 && algo != GQ_ALGO_EXACT && n_chunks > 0 && hsq_tc2_supported(d, K, code_bytes);
    if (remote.n > 0 && !(tc2_ok && n_bit != 32 && hsq_tc2_tail_supported(n_seg, n_bit, l_bytes, u_out, uniforms, l, codes))) {
        set_error("a remote delivery is attached, but this encode cannot run as the fused tcgen05 kernel");
        return GQ_ERR_UNSUPPORTED;
    }
    if (tc2_ok) {
        e = validate_group(grad, n_chunks, d, codebook, K, seg_start, n_seg);
        if (e) return e;
        GQ_REQUIRE(codes && u_out, "null output pointer");
        uint64_t *flag = reinterpret_cast<uint64_t *>(barrier) + 1;   // barrier word(s) at +0/+4, flag at +8
        if (n_bit == 32) {   // fp32 norms: search only, the rider still travels with it
            return hsq_encode_tc2(grad, n_chunks, d, codebook, codes, u_out, seg_start, n_seg, nullptr, nullptr, nullptr,
                                  rider, nullptr, nullptr, st);
        }
        GQ_REQUIRE(l && lbub, "null output pointer");
        if (hsq_tc2_tail_supported(n_seg, n_bit, l_bytes, u_out, uniforms, l, codes)) {
            Tc2Tail tail = {(uint8_t *)l, lbub, uniforms, philox_seed, philox_offset, n_bit, random};
            return hsq_encode_tc2(grad, n_chunks, d, codebook, codes, u_out, seg_start, n_seg, keys, flag, barrier, rider,
                                  &tail, remote.n > 0 ? &remote : nullptr, st);
        }
        e = hsq_encode_tc2(grad, n_chunks, d, codebook, codes, u_out, seg_start, n_seg, keys, flag, nullptr, rider,
                           nullptr, nullptr, st);
        if (e) return e;
        return gq_norm_quantize(u_out, n_chunks, seg_start, n_seg, n_bit, random, uniforms, philox_seed,
                                philox_offset, l, l_bytes, lbub, keys, /*precomputed=*/1, stream);
    }
    static const bool in_kernel_init = [] { const char *f = getenv("GQ_TC_INIT"); return !(f && atoi(f) == 0); }();
    if (n_bit != 32 && in_kernel_init && algo != GQ_ALGO_EXACT && n_chunks > 0 && hsq_tc_supported(d, K, code_bytes)) {
        // tcgen05 path: the search kernel resets the keys and carries the rider itself
        e = validate_group(grad, n_chunks, d, codebook, K, seg_start, n_seg);
        if (e) return e;
        GQ_REQUIRE(codes && u_out, "null output pointer");
        GQ_REQUIRE(((uintptr_t)grad & 15) == 0, "gradient must be 16-byte aligned");
        e = hsq_search_tc_prepared(grad, n_chunks, codebook, codes, u_out, seg_start, n_seg, keys,
                                   reinterpret_cast<uint64_t *>(barrier) + 1, rider, st);
        if (e) return e;
        return gq_norm_quantize(u_out, n_chunks, seg_start, n_seg, n_bit, random, uniforms, philox_seed,
                                philox_offset, l, l_bytes, lbub, keys, /*precomputed=*/1, stream);
    }
    if (n_bit != 32) {
        e = launch_minmax_init_rider(keys, n_seg, st, nullptr, rider);
        if (e) return e;
    } else {
        e = launch_rider(rider, st);
        if (e) return e;
    }
    e = gq_hsq_search(grad, n_chunks, d, codebook, K, codes, code_bytes, u_out, seg_start, n_seg,
                      n_bit != 32 ? keys : nullptr, (char *)workspace + head, workspace_bytes - head, algo,
                      stream);
    if (e) return e;
    if (n_bit == 32) return GQ_OK;
    return gq_norm_quantize(u_out, n_chunks, seg_start, n_seg, n_bit, random, uniforms, philox_seed,
                            philox_offset, l, l_bytes, lbub, keys, /*precomputed=*/1, stream);
}

int gq_hsq_encode_search(const float *grad, int64_t n_chunks, int d, const float *codebook, int K,
                         const int64_t *seg_start, int n_seg, void *codes, int code_bytes, float *u_out,
                         void *workspace, size_t workspace_bytes, gq_stream_t stream)
{
    const Rider rider = take_rider();
    const Tc2Remote remote = take_remote();
    GQ_REQUIRE(remote.n == 0, "a remote delivery needs the levels: use gq_hsq_encode");
    int e = validate_group(grad, n_chunks, d, codebook, K, seg_start, n_seg);
    if (e) return e;
    const size_t need = gq_hsq_encode_workspace_bytes(n_chunks, d, K, n_seg);
    if (workspace_bytes < need || workspace == nullptr) {
        set_error("workspace too small: %zu < %zu", workspace_bytes, need);
        return GQ_ERR_WORKSPACE;
    }
    GQ_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    GQ_REQUIRE(codes && u_out, "null output pointer");
    if (tc_generation() != 2 || n_chunks == 0 || !hsq_tc2_supported(d, K, code_bytes)) {
        set_error("gq_hsq_encode_search runs the second-generation tcgen05 search only (d in {8, 16, 32}, K == 256, "
                  "uint8 codes, n_chunks > 0); got d=%d K=%d code_bytes=%d n_chunks=%lld",
                  d, K, code_bytes, (long long)n_chunks);
        return GQ_ERR_UNSUPPORTED;
    }
    uint32_t *keys = reinterpret_cast<uint32_t *>(workspace);
    uint32_t *barrier = reinterpret_cast<uint32_t *>((char *)workspace + align_up((size_t)n_seg * 2 * sizeof(uint32_t), 256));
    return hsq_encode_tc2(grad, n_chunks, d, codebook, codes, u_out, seg_start, n_seg, keys,
                          reinterpret_cast<uint64_t *>(barrier) + 1, nullptr, rider, nullptr, nullptr, as_stream(stream));
}

static const int64_t kStageChunks = 1024;   // chunk indices of the last tile stay below 2^31
int gq_hsq_decode_quantize(const void *codes, void *l, float *lbub, const float *u, const uint32_t *minmax_keys,
                           int64_t n_chunks, int d, const float *codebook, int K, const int64_t *seg_start,
                           int n_seg, int n_bit, int random, const float *uniforms, uint64_t philox_seed,
                           uint64_t philox_offset, int accumulate, float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();   // consumed first: an early error return must not leave it armed
    int e = validate_group(out, n_chunks, d, codebook, K, seg_start, n_seg);
    if (e) return e;
    if (d != 16 || K != 256 || n_chunks == 0 || n_chunks >= ((int64_t)1 << 31) - kStageChunks || n_seg > 1024) {
        set_error("gq_hsq_decode_quantize: d == 16, K == 256, 1 <= n_seg <= 1024, 0 < n_chunks < 2^31 - 1024 "
                  "(got d=%d K=%d n_seg=%d n_chunks=%lld)", d, K, n_seg, (long long)n_chunks);
        return GQ_ERR_UNSUPPORTED;
    }
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 7, "uint8 norm codes need n_bit 1..7 (got %d)", n_bit);
    GQ_REQUIRE(accumulate >= 0 && accumulate <= 2, "accumulate must be 0, 1 or 2");
    GQ_REQUIRE(codes && l && lbub && u && minmax_keys, "null pointer");
    GQ_REQUIRE((((uintptr_t)codes | (uintptr_t)l | (uintptr_t)lbub | (uintptr_t)u | (uintptr_t)uniforms |
                 (uintptr_t)out) & 15) == 0,
               "codes, l, lbub, u, uniforms and out must be 16-byte aligned");
    set_rider(pending);
    e = hsq_decode_quantize(codes, l, lbub, u, minmax_keys, n_chunks, codebook, seg_start, n_seg, n_bit, random,
                            uniforms, philox_seed, philox_offset, accumulate, out, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));   // no-op: the decode kernel carried it
}

int gq_hsq_decode_reduce(const void *codes, int code_bytes, const void *l, int l_bytes,
                         const float *lbub, const float *norms_f32, int64_t user_stride_bytes,
                         int n_users, int64_t n_chunks, int d, const float *codebook, int K,
                         const int64_t *seg_start, int n_seg, int n_bit, int mean, int accumulate,
                         float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();   // consumed first: an early error return must not leave it armed
    int e = validate_group(out, n_chunks, d, codebook, K, seg_start, n_seg);
    if (e) return e;
    GQ_REQUIRE(n_users >= 1, "n_users %d < 1", n_users);
    GQ_REQUIRE(code_bytes == 1 || code_bytes == 4, "code_bytes must be 1 or 4");
    GQ_REQUIRE(n_bit == 32 || (n_bit >= 1 && n_bit <= 24), "n_bit %d out of range", n_bit);
    if (n_bit == 32) {
        GQ_REQUIRE(norms_f32 != nullptr, "n_bit == 32 needs norms_f32");
        l_bytes = 1;
    } else {
        GQ_REQUIRE(l && lbub, "null l / lbub");
        GQ_REQUIRE(l_bytes == 1 || l_bytes == 4, "l_bytes must be 1 or 4");
    }
    GQ_REQUIRE(n_users == 1 || (user_stride_bytes % 4) == 0, "user stride must be a multiple of 4 bytes");
    GQ_REQUIRE(((uintptr_t)out & 15) == 0, "output must be 16-byte aligned");
    set_rider(pending);
    e = hsq_decode_reduce(codes, code_bytes, l, l_bytes, lbub, norms_f32, user_stride_bytes, nullptr, n_users,
                          n_chunks, d, codebook, K, seg_start, n_seg, n_bit, mean, accumulate, out,
                          as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));   // no-op when the decode kernel carried it
}

int gq_hsq_decode_reduce_scattered(const void *codes, int code_bytes, const void *l, int l_bytes,
                                   const float *lbub, const int64_t *user_byte_offsets, int n_users,
                                   int64_t n_chunks, int d, const float *codebook, int K,
                                   const int64_t *seg_start, int n_seg, int n_bit, int mean, int accumulate,
                                   float *out, gq_stream_t stream)
{
    const Rider pending = take_rider();   // consumed first: an early error return must not leave it armed
    int e = validate_group(out, n_chunks, d, codebook, K, seg_start, n_seg);
    if (e) return e;
    GQ_REQUIRE(n_users >= 1 && n_users <= 8 && user_byte_offsets, "1..8 users with an offset table");
    GQ_REQUIRE(code_bytes == 1 || code_bytes == 4, "code_bytes must be 1 or 4");
    GQ_REQUIRE(n_bit >= 1 && n_bit <= 24 && l && lbub, "quantized norms required (n_bit 1..24)");
    GQ_REQUIRE(l_bytes == 1 || l_bytes == 4, "l_bytes must be 1 or 4");
    GQ_REQUIRE(((uintptr_t)out & 15) == 0, "output must be 16-byte aligned");
    set_rider(pending);
    e = hsq_decode_reduce(codes, code_bytes, l, l_bytes, lbub, nullptr, 0, user_byte_offsets, n_users, n_chunks,
                          d, codebook, K, seg_start, n_seg, n_bit, mean, accumulate, out, as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));   // no-op when the decode kernel carried it
}

int gq_f32_reduce_users(const float *in, int64_t user_stride_bytes, int n_users, int64_t n, int mean,
                        int accumulate, float *out, gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && n_users >= 1, "bad sizes");
    GQ_REQUIRE(n == 0 || (in && out), "null pointer");
    return launch_f32_reduce_users(in, user_stride_bytes, nullptr, n_users, n, mean, accumulate, out,
                                   as_stream(stream));
}

int gq_f32_reduce_users_scattered(const float *in, const int64_t *user_byte_offsets, int n_users, int64_t n,
                                  int mean, int accumulate, float *out, gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && n_users >= 1 && n_users <= 8 && user_byte_offsets, "1..8 users with an offset table");
    GQ_REQUIRE(n == 0 || (in && out), "null pointer");
    return launch_f32_reduce_users(in, 0, user_byte_offsets, n_users, n, mean, accumulate, out, as_stream(stream));
}

int gq_attach_f32_reduce(const float *in, int64_t user_stride_bytes, const int64_t *user_byte_offsets, int n_users,
                         int64_t n, int mean, int accumulate, float *out)
{
    GQ_REQUIRE(n >= 0 && n_users >= 1 && n_users <= 8, "1..8 users");
    GQ_REQUIRE(n == 0 || (in && out), "null pointer");
    Rider r = {};
    r.in = in;
    for (int u = 0; u < n_users; ++u) r.off[u] = user_byte_offsets ? user_byte_offsets[u] : (int64_t)u * user_stride_bytes;
    r.n_users = n_users;
    r.n = n;
    r.mean = mean;
    r.accumulate = accumulate;
    r.out = out;
    set_rider(r);
    return GQ_OK;
}

int gq_axpy(const float *a, const float *b, float alpha, int64_t n, float *out, gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && (n == 0 || (a && b && out)), "bad arguments");
    return launch_axpy(a, b, alpha, n, out, 0, as_stream(stream));
}

int gq_sub(const float *a, const float *b, int64_t n, float *out, gq_stream_t stream)
{
    GQ_REQUIRE(n >= 0 && (n == 0 || (a && b && out)), "bad arguments");
    return launch_axpy(a, b, 0.0f, n, out, 1, as_stream(stream));
}

// -------------------------------------------------- host-buffer round trip ---
static size_t host_scratch_layout(int64_t n_chunks, int d, int K, int n_seg, size_t off[6])
{
    size_t p = 0;
    off[0] = p; p += align_up((size_t)n_chunks * d * 4, 256);              // gradient / output
    off[1] = p; p += align_up((size_t)n_chunks, 256);                      // codes (u8)
    off[2] = p; p += align_up((size_t)n_chunks, 256);                      // l (u8)
    off[3] = p; p += align_up((size_t)n_seg * 2 * 4, 256);                 // lbub
    off[4] = p; p += align_up((size_t)n_chunks * 4, 256);                  // u
    off[5] = p; p += gq_hsq_encode_workspace_bytes(n_chunks, d, K, n_seg); // workspace
    return p;
}

size_t gq_hsq_host_scratch_bytes(int64_t n_chunks, int d, int K, int n_seg)
{
    size_t off[6];
    return host_scratch_layout(n_chunks, d, K, n_seg, off);
}

int gq_hsq_roundtrip_host(const float *host_grad, float *host_out, int64_t n_chunks, int d,
                          const float *dev_codebook, int K, const int64_t *dev_seg_start, int n_seg,
                          int n_bit, int random, uint64_t philox_seed, uint64_t philox_offset,
                          void *dev_scratch, size_t scratch_bytes, int algo, gq_stream_t stream)
{
    GQ_REQUIRE(K <= 256 && n_bit <= 7, "host round trip uses the uint8 wire format (K <= 256, n_bit <= 7)");
    size_t off[6];
    const size_t need = host_scratch_layout(n_chunks, d, K, n_seg, off);
    if (scratch_bytes < need || !dev_scratch) {
        set_error("scratch too small: %zu < %zu", scratch_bytes, need);
        return GQ_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    char *base = (char *)dev_scratch;
    float *g = (float *)(base + off[0]);
    const size_t bytes = (size_t)n_chunks * d * 4;
    GQ_CUDA(cudaMemcpyAsync(g, host_grad, bytes, cudaMemcpyHostToDevice, st));
    int e = gq_hsq_encode(g, n_chunks, d, dev_codebook, K, dev_seg_start, n_seg, n_bit, random, nullptr,
                          philox_seed, philox_offset, base + off[1], 1, base + off[2], 1,
                          (float *)(base + off[3]), (float *)(base + off[4]), base + off[5],
                          need - off[5], algo, stream);
    if (e) return e;
    e = gq_hsq_decode_reduce(base + off[1], 1, base + off[2], 1, (float *)(base + off[3]), nullptr, 0, 1,
                             n_chunks, d, dev_codebook, K, dev_seg_start, n_seg, n_bit, 0, 0, g, stream);
    if (e) return e;
    GQ_CUDA(cudaMemcpyAsync(host_out, g, bytes, cudaMemcpyDeviceToHost, st));
    GQ_CUDA(cudaStreamSynchronize(st));
    return GQ_OK;
}

}  // extern "C"

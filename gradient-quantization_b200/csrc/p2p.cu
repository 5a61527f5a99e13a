// p2p.cu -- peer-to-peer exchange of packed records over NVLink without a collective call.
//
// ps topology with one user per GPU: every rank encodes into a record buffer that its peers can
// read directly (CUDA IPC mapping of peer device memory), a tiny barrier kernel tells the peers
// "my record of step e is complete" with system-scope release stores into their flag arrays and
// waits for theirs, and the fused decode-and-average kernel then pulls the 2/d bytes per element
// of the other users straight out of peer HBM while it works.  Replaces the NCCL all-gather of
// quantizers/ps_quantizer.py's exchange step (3 MB per rank: latency-, not bandwidth-bound).
#include <stdlib.h>
#include <string.h>

#include "gq_internal.cuh"

using namespace gq;

namespace gq {

struct PeerFlags {
    uint32_t *p[8];
};

// flags layout on every rank: uint32 flags[8]; flags[r] = last epoch rank r has announced to me
__global__ void peer_barrier_kernel(uint32_t *local_flags, const PeerFlags peers, int rank, int n_ranks,
                                    uint32_t epoch, unsigned long long timeout_ns)
{
    const int u = threadIdx.x;
    if (u < n_ranks) {
        // everything this GPU wrote before the kernel (its packed record) becomes visible to peer u
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(peers.p[u] + rank), "r"(epoch) : "memory");
        peer_wait_flag(local_flags + u, epoch, timeout_ns);   // a peer never arrived: trap, do not hang
    }
}

// GQ_PEER_TIMEOUT_S (default 120): how long a rank waits for its peers before it traps
unsigned long long peer_timeout_ns()
{
    static const unsigned long long ns = [] {
        const char *e = getenv("GQ_PEER_TIMEOUT_S");
        double s = e ? atof(e) : 120.0;
        if (!(s > 0.0)) s = 120.0;
        return (unsigned long long)(s * 1e9);
    }();
    return ns;
}

struct PeerPtrs {
    const uint4 *p[8];
};

// pull every user's packed record out of its owner's memory into the local [U, stride] buffer:
// wide (16-byte) loads, many in flight per thread, so NVLink latency is covered by parallelism
__global__ void __launch_bounds__(256)
peer_gather_kernel(uint4 *__restrict__ dst, const PeerPtrs src, size_t n16, size_t dst_stride16)
{
    const int u = blockIdx.y;
    const uint4 *s = src.p[u];
    uint4 *d = dst + (size_t)u * dst_stride16;
    const size_t step = (size_t)gridDim.x * 256;
    size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    for (; i + 3 * step < n16; i += 4 * step) {
        const uint4 a = __ldcv(s + i), b = __ldcv(s + i + step), c = __ldcv(s + i + 2 * step),
                    e = __ldcv(s + i + 3 * step);
        d[i] = a; d[i + step] = b; d[i + 2 * step] = c; d[i + 3 * step] = e;
    }
    for (; i < n16; i += step) d[i] = __ldcv(s + i);
}

struct PeerDst {
    uint4 *p[8];
};

// push the local record into every peer's receive buffer: one local read, n_dst posted remote
// stores per 16 bytes.  Stores over NVLink are fire-and-forget, so (unlike the pull in
// peer_gather_kernel) no thread waits a round trip; the barrier kernel that follows on the stream
// publishes them with its system-scope release.
__global__ void __launch_bounds__(256)
peer_push_kernel(const uint4 *__restrict__ src, const PeerDst dst, int n_dst, size_t n16)
{
    const size_t step = (size_t)gridDim.x * 256;
    size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    for (; i + 3 * step < n16; i += 4 * step) {
        const uint4 a = src[i], b = src[i + step], c = src[i + 2 * step], e = src[i + 3 * step];
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            if (d < n_dst) {
                uint4 *o = dst.p[d];
                o[i] = a; o[i + step] = b; o[i + 2 * step] = c; o[i + 3 * step] = e;
            }
        }
    }
    for (; i < n16; i += step) {
        const uint4 a = src[i];
#pragma unroll
        for (int d = 0; d < 8; ++d)
            if (d < n_dst) dst.p[d][i] = a;
    }
    __threadfence_system();
}

// the same push through an NVSwitch multicast mapping (NVLS): ONE multimem store per 16 bytes is
// replicated by the switch into every rank's buffer, so the sender's NVLink egress is one record
// instead of (ranks - 1) records
__global__ void __launch_bounds__(256)
peer_push_mc_kernel(const uint4 *__restrict__ src, uint4 *mc_dst, size_t n16)
{
    const size_t step = (size_t)gridDim.x * 256;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n16; i += step) {
        const uint4 a = src[i];
        asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};"
                     ::"l"(mc_dst + i), "f"(__uint_as_float(a.x)), "f"(__uint_as_float(a.y)),
                       "f"(__uint_as_float(a.z)), "f"(__uint_as_float(a.w)) : "memory");
    }
    __threadfence_system();
}

}  // namespace gq

extern "C" {

// cudaMalloc'ed, zero-initialised buffer whose IPC handle (64 bytes) can be shipped to the other
// ranks of the node (e.g. with torch.distributed.all_gather_object).  Synchronous.
int gq_ipc_alloc(size_t bytes, void **dev_ptr, void *handle_out_64)
{
    GQ_REQUIRE(bytes > 0 && dev_ptr && handle_out_64, "bad arguments");
    GQ_CUDA(cudaMalloc(dev_ptr, bytes));
    GQ_CUDA(cudaMemset(*dev_ptr, 0, bytes));
    cudaIpcMemHandle_t h;
    GQ_CUDA(cudaIpcGetMemHandle(&h, *dev_ptr));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle_out_64, &h, 64);
    GQ_CUDA(cudaDeviceSynchronize());
    return GQ_OK;
}

int gq_ipc_free(void *dev_ptr)
{
    if (dev_ptr) GQ_CUDA(cudaFree(dev_ptr));
    return GQ_OK;
}

// Map a peer's buffer into this process (peer access is enabled lazily by the driver).
int gq_ipc_open(const void *handle_64, void **peer_ptr)
{
    GQ_REQUIRE(handle_64 && peer_ptr, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle_64, 64);
    GQ_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return GQ_OK;
}

int gq_ipc_close(void *peer_ptr)
{
    if (peer_ptr) GQ_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return GQ_OK;
}

// Cross-GPU barrier on `stream`: announce `epoch` to every rank's flag array and wait until every
// rank has announced it here.  flag_ptrs[r] (host array) = address of rank r's flag array as
// mapped in THIS process (flag_ptrs[rank] is the local one).  Epochs must increase by one per call.
int gq_peer_barrier(void *const *flag_ptrs, int rank, int n_ranks, uint32_t epoch, gq_stream_t stream)
{
    GQ_REQUIRE(flag_ptrs && n_ranks >= 1 && n_ranks <= 8 && rank >= 0 && rank < n_ranks, "bad arguments");
    PeerFlags pf;
    for (int r = 0; r < 8; ++r) pf.p[r] = (r < n_ranks) ? reinterpret_cast<uint32_t *>(flag_ptrs[r]) : nullptr;
    peer_barrier_kernel<<<1, 32, 0, as_stream(stream)>>>(pf.p[rank], pf, rank, n_ranks, epoch, peer_timeout_ns());
    GQ_LAUNCH_CHECK("peer_barrier");
    return GQ_OK;
}

// After gq_peer_barrier: copy n_ranks records of `bytes` each (a multiple of 16) from
// src_ptrs[r] (host array of device addresses, peer-mapped or local) to dst + r * dst_stride.
int gq_peer_gather(void *dst, void *const *src_ptrs, size_t bytes, size_t dst_stride, int n_ranks,
                   gq_stream_t stream)
{
    GQ_REQUIRE(dst && src_ptrs && n_ranks >= 1 && n_ranks <= 8, "bad arguments");
    GQ_REQUIRE(bytes % 16 == 0 && dst_stride % 16 == 0 && ((uintptr_t)dst & 15) == 0, "16-byte granularity");
    PeerPtrs pp;
    for (int r = 0; r < 8; ++r) pp.p[r] = (r < n_ranks) ? reinterpret_cast<const uint4 *>(src_ptrs[r]) : nullptr;
    const size_t n16 = bytes / 16;
    int bx = (int)((n16 + 1023) / 1024);
    const int cap = sm_count() * 4 / n_ranks + 1;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    peer_gather_kernel<<<dim3(bx, n_ranks), 256, 0, as_stream(stream)>>>(reinterpret_cast<uint4 *>(dst), pp, n16,
                                                                          dst_stride / 16);
    GQ_LAUNCH_CHECK("peer_gather");
    return GQ_OK;
}

// Before gq_peer_barrier: copy `bytes` (a multiple of 16) from the local `src` to each of the n_dst
// addresses in dst_ptrs (host array of peer-mapped device addresses).
int gq_peer_push(const void *src, void *const *dst_ptrs, size_t bytes, int n_dst, gq_stream_t stream)
{
    GQ_REQUIRE(src && dst_ptrs && n_dst >= 0 && n_dst <= 8, "bad arguments");
    GQ_REQUIRE(bytes % 16 == 0 && ((uintptr_t)src & 15) == 0, "16-byte granularity");
    if (n_dst == 0 || bytes == 0) return GQ_OK;
    PeerDst pd;
    for (int r = 0; r < 8; ++r) {
        pd.p[r] = (r < n_dst) ? reinterpret_cast<uint4 *>(dst_ptrs[r]) : nullptr;
        GQ_REQUIRE(r >= n_dst || (((uintptr_t)dst_ptrs[r] & 15) == 0 && dst_ptrs[r]), "bad destination");
    }
    const size_t n16 = bytes / 16;
    int bx = (int)((n16 + 1023) / 1024);
    const int cap = sm_count() * 2;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    peer_push_kernel<<<bx, 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint4 *>(src), pd, n_dst, n16);
    GQ_LAUNCH_CHECK("peer_push");
    return GQ_OK;
}

// Fused exchange, sending side: the NEXT encode call on this host thread (gq_hsq_encode, gq_sign_encode,
// gq_sign_encode_t5 or gq_qsgd_encode) also stores every finished section of the record it writes at
// (local address + delta[i]) for i < n_remote (peer-mapped copies of the same record row), or once through
// an NVLS multicast mapping (multicast = 1, n_remote = 1), mirrors the identity section
// [ident, ident + ident_bytes) the same way, and finally stores `epoch` into the n_flags words flag_ptrs[i]
// (this rank's slot in every rank's flag array, its own included).  n_flags == 0: deliver, do not announce
// (every launch but the last of an encode made of several calls).
// Requires a delivering kernel: the one-launch tcgen05 encode (d = 8, 16 or 32, K = 256, uint8 codes and
// levels), the packed-words sign kernel, the base-3 sign kernel, the one-launch chunked QSGD kernel or the
// TernGrad range kernels; the sign and QSGD ones also need gq_attach_delivery_counter.  Any other encode
// fails with GQ_ERR_UNSUPPORTED and nothing is sent; the pending delivery is cleared either way.
int gq_attach_remote_record(int n_remote, int multicast, const int64_t *delta, const void *ident, int64_t ident_bytes,
                            void *const *flag_ptrs, int n_flags, uint32_t epoch)
{
    GQ_REQUIRE(n_remote >= 1 && n_remote <= 7 && delta && n_flags >= 0 && n_flags <= 8 && (flag_ptrs || n_flags == 0),
               "bad arguments");
    GQ_REQUIRE(!multicast || n_remote == 1, "a multicast delivery has one destination");
    GQ_REQUIRE(ident_bytes >= 0 && ident_bytes % 16 == 0 && (ident_bytes == 0 || ((uintptr_t)ident & 15) == 0),
               "identity section must be 16-byte granular");
    Tc2Remote r = {};
    r.n = n_remote;
    r.multicast = multicast;
    for (int i = 0; i < n_remote; ++i) {
        GQ_REQUIRE(delta[i] % 16 == 0, "remote copies must keep the 16-byte alignment");
        r.delta[i] = delta[i];
    }
    r.ident = reinterpret_cast<const uint8_t *>(ident);
    r.ident_bytes = ident_bytes;
    r.n_flag = n_flags;
    for (int i = 0; i < n_flags; ++i) r.flag[i] = reinterpret_cast<uint32_t *>(flag_ptrs[i]);
    r.epoch = epoch;
    set_remote(r);
    return GQ_OK;
}

// The arrival counter of the pending delivery (after gq_attach_remote_record): a zero-initialised,
// 4-byte aligned device word that no other delivery uses at the same time.  The sign and QSGD encodes
// have no grid barrier behind which to zero one: their last CTA to arrive sets it back to 0.
int gq_attach_delivery_counter(void *counter)
{
    Tc2Remote r = take_remote();
    GQ_REQUIRE(r.n > 0, "no remote delivery is attached");
    GQ_REQUIRE(counter && ((uintptr_t)counter & 3) == 0, "bad counter address");
    r.counter = reinterpret_cast<uint32_t *>(counter);
    set_remote(r);
    return GQ_OK;
}

// Fused exchange, receiving side: the NEXT HSQ, sign or QSGD decode on this host thread first waits until
// all n_ranks words of the local flag array have reached `epoch` (inside the decode kernel's prologue
// when it is the staged HSQ kernel or a fast sign / QSGD kernel, else in a one-warp kernel launched
// before it).
int gq_attach_peer_wait(const void *local_flags, int n_ranks, uint32_t epoch)
{
    GQ_REQUIRE(local_flags && n_ranks >= 1 && n_ranks <= 8, "bad arguments");
    PeerWait w = {};
    w.flags = reinterpret_cast<const uint32_t *>(local_flags);
    w.n = n_ranks;
    w.epoch = epoch;
    w.timeout_ns = peer_timeout_ns();
    set_wait(w);
    return GQ_OK;
}

// Multicast variant: mc_dst is the address of the destination row inside an NVSwitch multicast
// mapping of the ranks' (symmetric) buffers, e.g. torch symmetric memory's multicast_ptr + offset.
int gq_peer_push_multicast(const void *src, void *mc_dst, size_t bytes, gq_stream_t stream)
{
    GQ_REQUIRE(src && mc_dst, "bad arguments");
    GQ_REQUIRE(bytes % 16 == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)mc_dst & 15) == 0, "16-byte granularity");
    if (bytes == 0) return GQ_OK;
    const size_t n16 = bytes / 16;
    int bx = (int)((n16 + 255) / 256);
    const int cap = sm_count() * 4;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    peer_push_mc_kernel<<<bx, 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint4 *>(src),
                                                           reinterpret_cast<uint4 *>(mc_dst), n16);
    GQ_LAUNCH_CHECK("peer_push_multicast");
    return GQ_OK;
}

}  // extern "C"

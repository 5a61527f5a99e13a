// topk.cu -- segmented top-k sparsification by radix select.
// Replaces TopKSparsificationCompressor.compress
// (compressors/topk_sparsification_compressor.py:18-23): per tensor keep the
// k largest |v| (ties at the cut resolved towards the lowest index -- torch.topk
// leaves the order unspecified), zero the rest.
//
// key = bit pattern of |v| (31 bits, monotone; NaN sorts above inf like torch.topk).
// The gradient is read TWICE:
//   1. histogram of the top 11 key bits of every tensor (shared-memory histograms over runs of
//      16 tiles) -> the bin b* holding the k-th largest key of each tensor;
//   2. classify: elements above b* are selected for sure, elements inside b* are candidates; both go,
//      in index order, into a per-tile entry list (a few percent of the tensor), the candidates'
//      next 10 key bits into the second histogram.
// Everything after that (third histogram, per-tile counts, per-tensor scan of the counts, the final
// (index, value) records in ascending index order with lowest-index-first ties) works on the entry
// lists only.  The previous version made five passes over the gradient (kept below for reference in
// the history; gone from the code).
#include <algorithm>

#include "gq_internal.cuh"

namespace gq {

constexpr int kTile = 1024;      // elements per tile (256 threads x 4)
constexpr int kBins = 2048;
constexpr int kSuper = 16;       // tiles per shared-memory histogram run (first pass)

struct TopkState {
    uint32_t prefix;    // key bits decided so far (aligned to the top)
    uint32_t k_rem;     // how many still to take among keys matching the prefix
    uint32_t T;         // final threshold key (after pass 3)
    uint32_t count_eq;  // number of elements with key == T
};

__device__ __forceinline__ uint32_t key_of(float x) { return __float_as_uint(x) & 0x7fffffffu; }

// tile_prefix[s] = number of tiles of segments < s (run_prefix: of 16-tile runs); also clears the
// histograms
__global__ void topk_setup_kernel(const int64_t *__restrict__ seg_start, const int64_t *__restrict__ k,
                                  int n_seg, int64_t *__restrict__ tile_prefix, int64_t *__restrict__ run_prefix,
                                  TopkState *__restrict__ state, uint32_t *__restrict__ hist, const Rider rider)
{
    pdl_launch_dependents();
    pdl_wait();
    rider_run(rider, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);   // identity tensors ride along
    if (blockIdx.x == 0 && threadIdx.x < 32) {
        // exclusive prefix sums of the tensors' tile / run counts: one warp, 32 tensors per step
        const int lane = threadIdx.x;
        int64_t acc = 0, racc = 0;
        for (int s0 = 0; s0 < n_seg; s0 += 32) {
            const int s = s0 + lane;
            const int64_t tiles = s < n_seg ? (seg_start[s + 1] - seg_start[s] + kTile - 1) / kTile : 0;
            const int64_t runs = (tiles + kSuper - 1) / kSuper;
            int64_t it = tiles, ir = runs;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t yt = __shfl_up_sync(0xffffffffu, it, o), yr = __shfl_up_sync(0xffffffffu, ir, o);
                if (lane >= o) { it += yt; ir += yr; }
            }
            if (s < n_seg) {
                tile_prefix[s] = acc + it - tiles;
                run_prefix[s] = racc + ir - runs;
            }
            acc += __shfl_sync(0xffffffffu, it, 31);
            racc += __shfl_sync(0xffffffffu, ir, 31);
        }
        if (lane == 0) {
            tile_prefix[n_seg] = acc;
            run_prefix[n_seg] = racc;
        }
    }
    const int64_t nh = (int64_t)n_seg * kBins;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nh; i += (int64_t)gridDim.x * blockDim.x)
        hist[i] = 0u;
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < n_seg; s += gridDim.x * blockDim.x) {
        TopkState st;
        st.prefix = 0;
        int64_t len = seg_start[s + 1] - seg_start[s];
        int64_t kk = k[s] < len ? k[s] : len;
        st.k_rem = (uint32_t)(kk < 0 ? 0 : kk);
        st.T = 0xffffffffu;
        st.count_eq = 0;
        state[s] = st;
    }
}

__device__ __forceinline__ bool tile_range(const int64_t *__restrict__ seg_start,
                                           const int64_t *__restrict__ tile_prefix, int n_seg,
                                           int64_t b, int &s, int64_t &lo, int64_t &hi)
{
    if (b >= tile_prefix[n_seg]) return false;
    s = find_segment(tile_prefix, n_seg, b);
    // skip empty segments sharing the same tile_prefix value
    while (s + 1 < n_seg && tile_prefix[s + 1] <= b) ++s;
    lo = seg_start[s] + (b - tile_prefix[s]) * kTile;
    hi = min(lo + (int64_t)kTile, seg_start[s + 1]);
    return true;
}

struct TopkEntry {
    uint32_t idx_flag;   // element index inside the group (31 bits) | candidate flag << 31
    float val;
};

// run_prefix[s] = number of 16-tile runs of segments < s (first-pass work units)
__device__ __forceinline__ bool run_range(const int64_t *__restrict__ seg_start,
                                          const int64_t *__restrict__ run_prefix, int n_seg, int64_t r,
                                          int &s, int64_t &lo, int64_t &hi)
{
    if (r >= run_prefix[n_seg]) return false;
    s = find_segment(run_prefix, n_seg, r);
    while (s + 1 < n_seg && run_prefix[s + 1] <= r) ++s;
    lo = seg_start[s] + (r - run_prefix[s]) * (int64_t)(kTile * kSuper);
    hi = min(lo + (int64_t)(kTile * kSuper), seg_start[s + 1]);
    return true;
}

// first pass: histogram of key bits 30..20 (2048 bins) per tensor
__global__ void __launch_bounds__(256)
topk_hist0_kernel(const float *__restrict__ v, const int64_t *__restrict__ seg_start,
                  const int64_t *__restrict__ run_prefix, int n_seg,
                  const TopkState *__restrict__ state, uint32_t *__restrict__ hist)
{
    __shared__ uint32_t s_hist[kBins];
    pdl_launch_dependents();
    pdl_wait();
    const int64_t total = run_prefix[n_seg];
    for (int64_t r = blockIdx.x; r < total; r += gridDim.x) {
        int s; int64_t lo, hi;
        if (!run_range(seg_start, run_prefix, n_seg, r, s, lo, hi)) break;
        if (state[s].k_rem == 0) continue;
        for (int i = threadIdx.x; i < kBins; i += 256) s_hist[i] = 0;
        __syncthreads();
        int64_t i = lo + threadIdx.x;
        for (; i + 768 < hi; i += 1024) {   // four independent loads in flight per thread
            const float a = v[i], b = v[i + 256], c = v[i + 512], d = v[i + 768];
            atomicAdd(&s_hist[key_of(a) >> 20], 1u);
            atomicAdd(&s_hist[key_of(b) >> 20], 1u);
            atomicAdd(&s_hist[key_of(c) >> 20], 1u);
            atomicAdd(&s_hist[key_of(d) >> 20], 1u);
        }
        for (; i < hi; i += 256) atomicAdd(&s_hist[key_of(v[i]) >> 20], 1u);
        __syncthreads();
        for (int j = threadIdx.x; j < kBins; j += 256) {
            const uint32_t c = s_hist[j];
            if (c) atomicAdd(hist + (int64_t)s * kBins + j, c);
        }
        __syncthreads();
    }
}

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t x, uint32_t *s_warp, uint32_t &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        uint32_t c = s_warp[w];
        if (w < warp) base += c;
        tot += c;
    }
    total = tot;
    return base + inc - x;
}

// one block per segment: pick the bin holding the k_rem-th largest key, update
// the state, clear the histogram for the next pass.
template <int PASS>
__global__ void __launch_bounds__(256)
topk_scan_kernel(uint32_t *__restrict__ hist, TopkState *__restrict__ state)
{
    __shared__ uint32_t s_warp[8];
    pdl_launch_dependents();
    pdl_wait();
    const int s = blockIdx.x;
    uint32_t *h = hist + (int64_t)s * kBins;
    TopkState st = state[s];
    constexpr int BINS = (PASS == 0) ? kBins : 1024;
    constexpr int PER = BINS / 256;
    if (st.k_rem == 0) return;
    uint32_t local[PER];
    uint32_t sum = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) { local[j] = h[threadIdx.x * PER + j]; sum += local[j]; }
    // count of keys in bins strictly above this thread's bins = total - (bins below) - (own bins)
    uint32_t total;
    const uint32_t below = block_exclusive_scan(sum, s_warp, total);
    const uint32_t above = total - below - sum;
    if (above < st.k_rem && above + sum >= st.k_rem) {
        uint32_t acc = above;
        for (int j = PER - 1; j >= 0; --j) {
            if (acc + local[j] >= st.k_rem) {
                const uint32_t bin = threadIdx.x * PER + j;
                TopkState ns = st;
                ns.k_rem = st.k_rem - acc;
                if (PASS == 0) ns.prefix = bin;
                else if (PASS == 1) ns.prefix = (st.prefix << 10) | bin;
                else { ns.T = (st.prefix << 10) | bin; ns.count_eq = local[j]; }
                state[s] = ns;
                break;
            }
            acc += local[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PER; ++j) h[threadIdx.x * PER + j] = 0;
}

// second pass over the gradient, one WARP per 1024-element tile: the tile's entry list (sure and
// candidate elements in index order) and the candidates' histogram of key bits 19..10; the dense
// output gets the sure elements.  Eight coalesced float4 loads per lane up front, flags as bit
// masks, list positions from ballots; every tile owns a fixed slot of the list: no allocation.
__global__ void __launch_bounds__(256)
topk_classify_kernel(const float *__restrict__ v, const int64_t *__restrict__ seg_start,
                     const int64_t *__restrict__ tile_prefix, int n_seg,
                     const TopkState *__restrict__ state, uint32_t *__restrict__ hist,
                     int32_t *__restrict__ tile_seg, uint32_t *__restrict__ tile_cnt,
                     TopkEntry *__restrict__ list, float *__restrict__ out_dense)
{
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int64_t total_tiles = tile_prefix[n_seg];
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < total_tiles; b += (int64_t)gridDim.x * 8) {
        int s; int64_t lo, hi;
        tile_range(seg_start, tile_prefix, n_seg, b, s, lo, hi);
        const TopkState st = state[s];
        const bool vec = ((reinterpret_cast<uintptr_t>(v + lo) & 15) == 0);
        float x[8][4];
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int64_t i0 = lo + it * 128 + lane * 4;
            if (vec && i0 + 3 < hi) {
                const float4 t = *reinterpret_cast<const float4 *>(v + i0);
                x[it][0] = t.x; x[it][1] = t.y; x[it][2] = t.z; x[it][3] = t.w;
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) x[it][t] = (i0 + t < hi) ? v[i0 + t] : 0.0f;
            }
        }
        uint32_t m_sure = 0u, m_cand = 0u;   // bit it * 4 + t
        if (st.k_rem > 0) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const bool in = lo + it * 128 + lane * 4 + t < hi;
                    const uint32_t bin = key_of(x[it][t]) >> 20;
                    if (in && bin > st.prefix) m_sure |= 1u << (it * 4 + t);
                    if (in && bin == st.prefix) m_cand |= 1u << (it * 4 + t);
                }
            }
        }
        const uint32_t m_any = m_sure | m_cand;
        const uint32_t tot = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(m_any));
        if (lane == 0) {
            tile_seg[b] = s;
            tile_cnt[b] = tot;
        }
        TopkEntry *tl = list + b * kTile;   // the tile's own slot (up to kTile entries): no allocation
        uint32_t base = 0u;
        if (tot) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const uint32_t f = (m_any >> (it * 4)) & 15u;
                if (__ballot_sync(0xffffffffu, f != 0u) == 0u) continue;   // warp-uniform
                const uint32_t b0 = __ballot_sync(0xffffffffu, f & 1u), b1 = __ballot_sync(0xffffffffu, f & 2u);
                const uint32_t b2 = __ballot_sync(0xffffffffu, f & 4u), b3 = __ballot_sync(0xffffffffu, f & 8u);
                uint32_t o = base + __popc(b0 & lt_mask) + __popc(b1 & lt_mask) + __popc(b2 & lt_mask) + __popc(b3 & lt_mask);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    if (f & (1u << t)) {
                        const bool c = (m_cand >> (it * 4 + t)) & 1u;
                        TopkEntry e;
                        e.idx_flag = (uint32_t)(lo + it * 128 + lane * 4 + t) | (c ? 0x80000000u : 0u);
                        e.val = x[it][t];
                        tl[o++] = e;
                        if (c) atomicAdd(hist + (int64_t)s * kBins + ((key_of(x[it][t]) >> 10) & 1023u), 1u);
                    }
                }
                base += __popc(b0) + __popc(b1) + __popc(b2) + __popc(b3);
            }
        }
        if (out_dense) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int64_t i0 = lo + it * 128 + lane * 4;
                float y[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) y[t] = __fmul_rn(x[it][t], ((m_sure >> (it * 4 + t)) & 1u) ? 1.0f : 0.0f);
                if (vec && i0 + 3 < hi && ((reinterpret_cast<uintptr_t>(out_dense + i0) & 15) == 0)) {
                    *reinterpret_cast<float4 *>(out_dense + i0) = make_float4(y[0], y[1], y[2], y[3]);
                } else {
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        if (i0 + t < hi) out_dense[i0 + t] = y[t];
                }
            }
        }
    }
}

// one warp per tile list: third histogram (key bits 9..0 of the candidates matching 21 decided bits)
__global__ void __launch_bounds__(256)
topk_list_hist2_kernel(const int64_t *__restrict__ seg_start, const int64_t *__restrict__ tile_prefix, int n_seg,
                       const TopkState *__restrict__ state, const int32_t *__restrict__ tile_seg,
                       const uint32_t *__restrict__ tile_cnt, const TopkEntry *__restrict__ list,
                       uint32_t *__restrict__ hist)
{
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t total_tiles = tile_prefix[n_seg];
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < total_tiles; b += (int64_t)gridDim.x * 8) {
        const uint32_t cnt = tile_cnt[b];
        if (cnt == 0) continue;
        const int s = tile_seg[b];
        const TopkState st = state[s];
        if (st.k_rem == 0) continue;
        const TopkEntry *e = list + b * kTile;
        for (uint32_t j = lane; j < cnt; j += 32) {
            const TopkEntry en = e[j];
            const uint32_t key = key_of(en.val);
            if ((en.idx_flag & 0x80000000u) && (key >> 10) == st.prefix)
                atomicAdd(hist + (int64_t)s * kBins + (key & 1023u), 1u);
        }
    }
}

// one warp per tile list: number of selected-for-sure entries (key > T) and of entries with key == T
__global__ void __launch_bounds__(256)
topk_list_count_kernel(const int64_t *__restrict__ seg_start, const int64_t *__restrict__ tile_prefix, int n_seg,
                       const TopkState *__restrict__ state, const int32_t *__restrict__ tile_seg,
                       const uint32_t *__restrict__ tile_cnt, const TopkEntry *__restrict__ list,
                       uint32_t *__restrict__ tile_gt, uint32_t *__restrict__ tile_eq)
{
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t total_tiles = tile_prefix[n_seg];
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < total_tiles; b += (int64_t)gridDim.x * 8) {
        const uint32_t cnt = tile_cnt[b];
        uint32_t gt = 0, eq = 0;
        if (cnt) {
            const uint32_t T = state[tile_seg[b]].T;
            const TopkEntry *e = list + b * kTile;
            for (uint32_t j = lane; j < cnt; j += 32) {
                const TopkEntry en = e[j];
                const uint32_t key = key_of(en.val);
                const bool c = (en.idx_flag & 0x80000000u) != 0u;
                gt += (!c || key > T) ? 1u : 0u;
                eq += (c && key == T) ? 1u : 0u;
            }
        }
        gt = __reduce_add_sync(0xffffffffu, gt);
        eq = __reduce_add_sync(0xffffffffu, eq);
        if (lane == 0) {
            tile_gt[b] = gt;
            tile_eq[b] = eq;
        }
    }
}

// one block per segment: exclusive scan of its tiles' counts (in place)
__global__ void __launch_bounds__(256)
topk_tilescan_kernel(const int64_t *__restrict__ tile_prefix, uint32_t *__restrict__ tile_gt,
                     uint32_t *__restrict__ tile_eq)
{
    __shared__ uint32_t s_warp[8];
    pdl_launch_dependents();
    pdl_wait();
    const int s = blockIdx.x;
    const int64_t t0 = tile_prefix[s], t1 = tile_prefix[s + 1];
    uint32_t carry_gt = 0, carry_eq = 0;
    for (int64_t base = t0; base < t1; base += 256) {
        const int64_t t = base + threadIdx.x;
        uint32_t g = t < t1 ? tile_gt[t] : 0u;
        uint32_t e = t < t1 ? tile_eq[t] : 0u;
        uint32_t tg, te;
        uint32_t xg = block_exclusive_scan(g, s_warp, tg);
        uint32_t xe = block_exclusive_scan(e, s_warp, te);
        if (t < t1) { tile_gt[t] = carry_gt + xg; tile_eq[t] = carry_eq + xe; }
        carry_gt += tg;
        carry_eq += te;
    }
}

// one warp per tile list: the final (index, value) records in ascending index order; the dense
// output gets the candidates that made it
__global__ void __launch_bounds__(256)
topk_list_write_kernel(const int64_t *__restrict__ seg_start, const int64_t *__restrict__ k_prefix,
                       const int64_t *__restrict__ tile_prefix, int n_seg, const TopkState *__restrict__ state,
                       const int32_t *__restrict__ tile_seg, const uint32_t *__restrict__ tile_cnt,
                       const TopkEntry *__restrict__ list, const uint32_t *__restrict__ tile_gt,
                       const uint32_t *__restrict__ tile_eq, float *__restrict__ out_dense,
                       int32_t *__restrict__ out_idx, float *__restrict__ out_val)
{
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int64_t total_tiles = tile_prefix[n_seg];
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < total_tiles; b += (int64_t)gridDim.x * 8) {
        const uint32_t cnt = tile_cnt[b];
        if (cnt == 0) continue;
        const int s = tile_seg[b];
        const TopkState st = state[s];
        if (st.k_rem == 0) continue;
        const uint32_t gt_before = tile_gt[b], eq_before = tile_eq[b];
        uint32_t eq_seen = eq_before;
        int64_t o = (k_prefix ? k_prefix[s] : 0) + gt_before + (eq_before < st.k_rem ? eq_before : st.k_rem);
        const TopkEntry *e = list + b * kTile;
        for (uint32_t j0 = 0; j0 < cnt; j0 += 32) {
            const uint32_t j = j0 + lane;
            TopkEntry en;
            en.idx_flag = 0u;
            en.val = 0.0f;
            bool have = j < cnt;
            if (have) en = e[j];
            const uint32_t key = key_of(en.val);
            const bool c = (en.idx_flag & 0x80000000u) != 0u;
            const bool is_eq = have && c && key == st.T;
            const uint32_t eq_ball = __ballot_sync(0xffffffffu, is_eq);
            const uint32_t my_eq_rank = eq_seen + __popc(eq_ball & lt_mask);
            const bool take = have && (!c || key > st.T || (is_eq && my_eq_rank < st.k_rem));
            const uint32_t tk_ball = __ballot_sync(0xffffffffu, take);
            if (take) {
                const int64_t dst = o + __popc(tk_ball & lt_mask);
                const uint32_t idx = en.idx_flag & 0x7fffffffu;
                if (out_idx) out_idx[dst] = (int32_t)idx;
                if (out_val) out_val[dst] = en.val;
                if (out_dense && c) out_dense[idx] = en.val;
            }
            o += __popc(tk_ball);
            eq_seen += __popc(eq_ball);
        }
    }
}

struct TopkWorkspace {
    int64_t *tile_prefix;
    int64_t *run_prefix;
    TopkState *state;
    uint32_t *hist;
    uint32_t *tile_gt;
    uint32_t *tile_eq;
    int32_t *tile_seg;
    uint32_t *tile_cnt;
    TopkEntry *list;
    size_t bytes;
};

static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

static TopkWorkspace carve(void *base, int64_t n, int n_seg)
{
    TopkWorkspace w;
    const int64_t max_tiles = n / kTile + n_seg + 1;
    size_t p = 0;
    char *b = (char *)base;
    w.tile_prefix = (int64_t *)(b + p); p += align256((size_t)(n_seg + 1) * 8);
    w.run_prefix = (int64_t *)(b + p);  p += align256((size_t)(n_seg + 1) * 8);
    w.state = (TopkState *)(b + p);     p += align256((size_t)n_seg * sizeof(TopkState));
    w.hist = (uint32_t *)(b + p);       p += align256((size_t)n_seg * kBins * 4);
    w.tile_gt = (uint32_t *)(b + p);    p += align256((size_t)max_tiles * 4);
    w.tile_eq = (uint32_t *)(b + p);    p += align256((size_t)max_tiles * 4);
    w.tile_seg = (int32_t *)(b + p);    p += align256((size_t)max_tiles * 4);
    w.tile_cnt = (uint32_t *)(b + p);   p += align256((size_t)max_tiles * 4);
    // every tile owns a slot of kTile entries (worst case: every element in the threshold bin)
    w.list = (TopkEntry *)(b + p);      p += align256((size_t)max_tiles * kTile * sizeof(TopkEntry));
    w.bytes = p;
    return w;
}

size_t topk_workspace_bytes(int64_t n, int n_seg) { return carve(nullptr, n, n_seg).bytes; }

int topk_select(const float *grad, int64_t n, const int64_t *seg_start, const int64_t *k,
                const int64_t *k_prefix, int n_seg, float *out_dense, int32_t *out_idx, float *out_val,
                void *workspace, cudaStream_t st)
{
    if (n == 0 || n_seg == 0) return GQ_OK;
    TopkWorkspace w = carve(workspace, n, n_seg);
    const int64_t max_tiles = n / kTile + n_seg + 1;
    const int64_t cap = (int64_t)sm_count() * 8;
    const int grid = (int)(max_tiles < cap ? max_tiles : cap);
    const int64_t max_runs = n / (kTile * kSuper) + n_seg + 1;
    const int grid_runs = (int)(max_runs < cap ? max_runs : cap);
    const int64_t warp_blocks = (max_tiles + 7) / 8;
    // (one warp per tile, a chain of dependent loads per tile: as many warps in flight as fit)
    const int grid_lists = (int)(warp_blocks < 2 * cap ? warp_blocks : 2 * cap);
    const int grid_setup = (int)std::min<int64_t>(((int64_t)n_seg * kBins + 255) / 256, cap);
    const Rider rider = take_rider();   // a pending identity copy rides in the first launch
    GQ_CUDA(launch_pdl(topk_setup_kernel, dim3(grid_setup), dim3(256), 0, st, seg_start, k, n_seg, w.tile_prefix,
                       w.run_prefix, w.state, w.hist, rider));
    GQ_CUDA(launch_pdl(topk_hist0_kernel, dim3(grid_runs), dim3(256), 0, st, grad, seg_start, (const int64_t *)w.run_prefix,
                       n_seg, (const TopkState *)w.state, w.hist));
    GQ_CUDA(launch_pdl(topk_scan_kernel<0>, dim3(n_seg), dim3(256), 0, st, w.hist, w.state));
    GQ_CUDA(launch_pdl(topk_classify_kernel, dim3(grid_lists), dim3(256), 0, st, grad, seg_start, (const int64_t *)w.tile_prefix,
                       n_seg, (const TopkState *)w.state, w.hist, w.tile_seg, w.tile_cnt, w.list, out_dense));
    GQ_CUDA(launch_pdl(topk_scan_kernel<1>, dim3(n_seg), dim3(256), 0, st, w.hist, w.state));
    GQ_CUDA(launch_pdl(topk_list_hist2_kernel, dim3(grid_lists), dim3(256), 0, st, seg_start, (const int64_t *)w.tile_prefix,
                       n_seg, (const TopkState *)w.state, (const int32_t *)w.tile_seg, (const uint32_t *)w.tile_cnt,
                       (const TopkEntry *)w.list, w.hist));
    GQ_CUDA(launch_pdl(topk_scan_kernel<2>, dim3(n_seg), dim3(256), 0, st, w.hist, w.state));
    GQ_CUDA(launch_pdl(topk_list_count_kernel, dim3(grid_lists), dim3(256), 0, st, seg_start, (const int64_t *)w.tile_prefix,
                       n_seg, (const TopkState *)w.state, (const int32_t *)w.tile_seg, (const uint32_t *)w.tile_cnt,
                       (const TopkEntry *)w.list, w.tile_gt, w.tile_eq));
    GQ_CUDA(launch_pdl(topk_tilescan_kernel, dim3(n_seg), dim3(256), 0, st, (const int64_t *)w.tile_prefix, w.tile_gt,
                       w.tile_eq));
    GQ_CUDA(launch_pdl(topk_list_write_kernel, dim3(grid_lists), dim3(256), 0, st, seg_start, k_prefix,
                       (const int64_t *)w.tile_prefix, n_seg, (const TopkState *)w.state, (const int32_t *)w.tile_seg,
                       (const uint32_t *)w.tile_cnt, (const TopkEntry *)w.list, (const uint32_t *)w.tile_gt,
                       (const uint32_t *)w.tile_eq, out_dense, out_idx, out_val));
    GQ_LAUNCH_CHECK("topk_select");
    return GQ_OK;
}

// ------------------------------------------------------- scatter + reduce ---
__global__ void __launch_bounds__(256)
fill_kernel(float *__restrict__ out, int64_t n, float val, const Rider rider)
{
    rider_run(rider, (int64_t)blockIdx.x * 256 + threadIdx.x, (int64_t)gridDim.x * 256);   // identity tensors ride along
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        out[i] = val;
}
// one user's sparse entries: indices are unique inside a user, so plain RMW is race-free
__global__ void __launch_bounds__(256)
scatter_add_kernel(const int32_t *__restrict__ idx, const float *__restrict__ val, int64_t k,
                   float *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < k; i += (int64_t)gridDim.x * 256) {
        const int32_t j = idx[i];
        out[j] = __fadd_rn(out[j], val[i]);
    }
}
__global__ void __launch_bounds__(256)
scale_div_kernel(float *__restrict__ out, int64_t n, float denom)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        out[i] = __fdiv_rn(out[i], denom);
}

static int grid_for(int64_t n)
{
    int64_t blocks = (n + 255) / 256;
    int64_t cap = (int64_t)sm_count() * 8;
    int64_t g = blocks < cap ? blocks : cap;
    return (int)(g < 1 ? 1 : g);
}

int topk_scatter_reduce(const int32_t *idx, const float *val, int64_t user_stride, int n_users,
                        int64_t k_total, int64_t n, int mean, int accumulate, float *out, cudaStream_t st)
{
    if (n == 0) return GQ_OK;
    // mean with accumulate: out + (sum)/U needs a scratch-free formulation only when U == 1
    if (!accumulate) {
        const Rider rider = take_rider();   // a pending identity reduction rides in the fill
        fill_kernel<<<grid_for(n), 256, 0, st>>>(out, n, 0.0f, rider);
    }
    for (int u = 0; u < n_users; ++u) {
        const int32_t *iu = reinterpret_cast<const int32_t *>(reinterpret_cast<const char *>(idx) + u * user_stride);
        const float *vu = reinterpret_cast<const float *>(reinterpret_cast<const char *>(val) + u * user_stride);
        if (k_total > 0) scatter_add_kernel<<<grid_for(k_total), 256, 0, st>>>(iu, vu, k_total, out);
    }
    if (mean && n_users > 1) scale_div_kernel<<<grid_for(n), 256, 0, st>>>(out, n, (float)n_users);
    GQ_LAUNCH_CHECK("topk_scatter_reduce");
    return GQ_OK;
}

}  // namespace gq

using namespace gq;

extern "C" {

size_t gq_topk_workspace_bytes(int64_t n, int n_seg) { return topk_workspace_bytes(n, n_seg > 0 ? n_seg : 1); }

int gq_topk_select(const float *grad, int64_t n, const int64_t *seg_start, const int64_t *k,
                   const int64_t *k_prefix, int n_seg, float *out_dense, int32_t *out_idx, float *out_val,
                   void *workspace, size_t workspace_bytes, gq_stream_t stream)
{
    const Rider pending = take_rider();   // consumed first: an early error return must not leave it armed
    if (take_remote().n > 0) {            // the record is written by the last of ten launches: no delivery
        set_error("a remote delivery is attached, but top-k has no delivering encode");
        return GQ_ERR_UNSUPPORTED;
    }
    GQ_REQUIRE(n >= 0 && n_seg >= 1, "bad sizes");
    GQ_REQUIRE(n < ((int64_t)1 << 31), "top-k group larger than 2^31 elements");
    GQ_REQUIRE(grad && seg_start && k, "null pointer");
    GQ_REQUIRE(out_dense || (out_idx && out_val), "need dense or (idx, val) outputs");
    GQ_REQUIRE(!(out_idx || out_val) || k_prefix, "wire output needs k_prefix");
    if (!workspace || workspace_bytes < topk_workspace_bytes(n, n_seg)) {
        set_error("workspace too small: %zu < %zu", workspace_bytes, topk_workspace_bytes(n, n_seg));
        return GQ_ERR_WORKSPACE;
    }
    set_rider(pending);
    const int e = topk_select(grad, n, seg_start, k, k_prefix, n_seg, out_dense, out_idx, out_val, workspace,
                              as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));   // no-op when the setup kernel carried it
}

int gq_topk_scatter_reduce(const int32_t *idx, const float *val, int64_t user_stride_bytes, int n_users,
                           int64_t k_total, int64_t n, int mean, int accumulate, float *out,
                           gq_stream_t stream)
{
    const Rider pending = take_rider();
    GQ_REQUIRE(n >= 0 && k_total >= 0 && n_users >= 1, "bad sizes");
    GQ_REQUIRE(!(mean && accumulate && n_users > 1), "mean + accumulate is not defined for top-k scatter");
    GQ_REQUIRE(k_total == 0 || (idx && val), "null pointer");
    set_rider(pending);
    const int e = topk_scatter_reduce(idx, val, user_stride_bytes, n_users, k_total, n, mean, accumulate, out,
                                      as_stream(stream));
    const Rider left = take_rider();
    if (e) return e;
    return launch_rider(left, as_stream(stream));
}

}  // extern "C"

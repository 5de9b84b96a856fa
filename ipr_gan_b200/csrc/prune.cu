// prune.cu -- the two weight perturbations of the IPR-GAN robustness experiments, on the device.
//
// ipr_prune_magnitude_f32: exact global magnitude pruning over a list of arena segments -- the removal attack of the
// reference's prune.py (torch.nn.utils.prune.global_unstructured with L1Unstructured, SURVEY.md 2.1 row 34).  The
// k-th smallest key |w| is found by a three-pass radix select (11 / 10 / 10 bits of the 31-bit key), every pass a
// histogram over the segments and a one-CTA bin scan; the ties at the threshold are ranked in arena order by
// per-tile counts, one scan over the tiles and an in-tile ballot scan.  No value comes back to the host, so the
// launch sequence is CUDA-graph capturable.
//
// ipr_negate_indexed_f32: the ambiguity attack's sign flip of normalisation gammas (sign_flip.py:59-77).
#include "ipr_common.cuh"

namespace {

constexpr int kTile = 1024;                 // virtual entries per tile = threads per CTA of the tile passes
constexpr int kBins = 2048;                 // widest radix digit (11 bits)

struct PruneState {
    long long rank;                         // rank (0-based) still sought inside the current digit's bin
    long long need;                         // ties at the threshold to prune (lowest arena index first)
    unsigned prefix;                        // key bits decided so far
};

struct Workspace {
    PruneState *state;
    unsigned *hist;                         // kBins
    int *tile_ties;                         // ntiles
    long long *tile_base;                   // ntiles: ties in earlier tiles
};

__host__ __device__ inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

__host__ __device__ inline Workspace carve(void *ws, long long ntiles)
{
    char *p = static_cast<char *>(ws);
    Workspace w;
    w.state = reinterpret_cast<PruneState *>(p);
    p += align256(sizeof(PruneState));
    w.hist = reinterpret_cast<unsigned *>(p);
    p += align256(kBins * sizeof(unsigned));
    w.tile_ties = reinterpret_cast<int *>(p);
    p += align256((size_t)ntiles * sizeof(int));
    w.tile_base = reinterpret_cast<long long *>(p);
    return w;
}

// |w| as an order-preserving 31-bit key: +-0 share 0, every NaN maps to one key above +inf (topk's order).
__device__ __forceinline__ unsigned magnitude_key(float w)
{
    const unsigned k = __float_as_uint(w) & 0x7fffffffu;
    return k > 0x7f800000u ? 0x7fffffffu : k;
}

// The segment table in shared memory: seg_off[s] arena offset, seg_pre[s] first virtual index of segment s.
struct SegSmem {
    long long off[IPR_PRUNE_MAX_SEGMENTS];
    long long pre[IPR_PRUNE_MAX_SEGMENTS + 1];
};

__device__ void load_segments(SegSmem &sm, const long long *seg, int n_seg)
{
    for (int s = threadIdx.x; s < n_seg; s += blockDim.x) {
        sm.off[s] = seg[2 * s];
        sm.pre[s + 1] = seg[2 * s + 1];         // count, prefix-summed below
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        sm.pre[0] = 0;
        for (int s = 0; s < n_seg; s++) sm.pre[s + 1] += sm.pre[s];
    }
    __syncthreads();
}

// virtual index v (< pre[n_seg]) -> arena index
__device__ __forceinline__ long long arena_index(const SegSmem &sm, int n_seg, long long v)
{
    int lo = 0, hi = n_seg - 1;                 // last s with pre[s] <= v
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sm.pre[mid] <= v) lo = mid; else hi = mid - 1;
    }
    return sm.off[lo] + (v - sm.pre[lo]);
}

__global__ void __launch_bounds__(1024)
prune_init_kernel(PruneState *st, unsigned *hist, long long k)
{
    for (int i = threadIdx.x; i < kBins; i += blockDim.x) hist[i] = 0;
    if (threadIdx.x == 0) {
        st->rank = k - 1;
        st->need = 0;
        st->prefix = 0;
    }
}

// histogram of digit (key >> shift) & (2^bits - 1) over the keys whose bits above shift + bits equal state->prefix
__global__ void __launch_bounds__(kTile)
prune_hist_kernel(const float *__restrict__ arena, const long long *__restrict__ seg, int n_seg, long long n_total,
                  const PruneState *__restrict__ st, unsigned *__restrict__ hist, int shift, int bits)
{
    __shared__ SegSmem sm;
    __shared__ unsigned h[kBins];
    const int nb = 1 << bits;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) h[i] = 0;
    load_segments(sm, seg, n_seg);
    const unsigned prefix = st->prefix;
    const int hi_shift = shift + bits;
    for (long long v = (long long)blockIdx.x * kTile + threadIdx.x; v < n_total; v += (long long)gridDim.x * kTile) {
        const unsigned key = magnitude_key(arena[arena_index(sm, n_seg, v)]);
        if (hi_shift >= 32 || (key >> hi_shift) == prefix) atomicAdd(&h[(key >> shift) & (nb - 1)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x)
        if (h[i]) atomicAdd(&hist[i], h[i]);
}

// one CTA: the bin holding state->rank; narrows prefix / rank to it and clears the histogram for the next pass.
// After the last digit, prefix is the threshold key T and rank + 1 the number of ties at T to prune.
__global__ void __launch_bounds__(1024)
prune_select_kernel(PruneState *st, unsigned *hist, int bits, int last)
{
    __shared__ long long warp_tot[32];
    const long long rank = st->rank;            // read before the barriers: one thread rewrites it after them
    const unsigned prefix = st->prefix;
    const int nb = 1 << bits;
    const int per = nb / blockDim.x;            // 1 or 2 bins per thread, consecutive
    const int b0 = threadIdx.x * per;
    long long mine = 0;
    for (int j = 0; j < per; j++) mine += hist[b0 + j];
    // block-wide inclusive scan of `mine`
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    if (wid == 0) {
        const int nw = blockDim.x >> 5;
        long long t = lane < nw ? warp_tot[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t += y;
        }
        warp_tot[lane] = t;                     // inclusive over warps
    }
    __syncthreads();
    long long excl = x - mine + (wid > 0 ? warp_tot[wid - 1] : 0);
    for (int j = 0; j < per; j++) {
        const long long c = hist[b0 + j];
        if (excl <= rank && rank < excl + c) {  // exactly one bin of the grid holds the rank
            st->prefix = (prefix << bits) | (unsigned)(b0 + j);
            st->rank = rank - excl;
            if (last) st->need = rank - excl + 1;
        }
        excl += c;
    }
    __syncthreads();
    for (int j = 0; j < per; j++) hist[b0 + j] = 0;
}

__device__ __forceinline__ bool is_tie(const float *arena, const SegSmem &sm, int n_seg, long long v, long long n_total,
                                       unsigned T)
{
    return v < n_total && magnitude_key(arena[arena_index(sm, n_seg, v)]) == T;
}

__global__ void __launch_bounds__(kTile)
prune_tie_count_kernel(const float *__restrict__ arena, const long long *__restrict__ seg, int n_seg,
                       long long n_total, long long ntiles, const PruneState *__restrict__ st, int *__restrict__ tile_ties)
{
    __shared__ SegSmem sm;
    __shared__ int red[32];
    load_segments(sm, seg, n_seg);
    const unsigned T = st->prefix;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const bool tie = is_tie(arena, sm, n_seg, t * kTile + threadIdx.x, n_total, T);
        const int c = __popc(__ballot_sync(0xffffffffu, tie));
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x < 32) {
            const int s = ipr_warp_sum_i(red[threadIdx.x]);
            if (threadIdx.x == 0) tile_ties[t] = s;
        }
        __syncthreads();
    }
}

// one CTA: tile_base[t] = sum of tile_ties[0 .. t)  (contiguous chunk per thread, then a scan of the chunk sums)
__global__ void __launch_bounds__(1024)
prune_tile_scan_kernel(const int *__restrict__ tile_ties, long long *__restrict__ tile_base, long long ntiles)
{
    __shared__ long long warp_tot[32];
    const long long per = (ntiles + blockDim.x - 1) / blockDim.x;
    const long long lo = min(ntiles, threadIdx.x * per), hi = min(ntiles, lo + per);
    long long mine = 0;
    for (long long t = lo; t < hi; t++) mine += tile_ties[t];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    if (wid == 0) {
        long long t = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t += y;
        }
        warp_tot[lane] = t;
    }
    __syncthreads();
    long long run = x - mine + (wid > 0 ? warp_tot[wid - 1] : 0);
    for (long long t = lo; t < hi; t++) {
        tile_base[t] = run;
        run += tile_ties[t];
    }
}

// w <- w * 0 for every key < T, and for the first `need` keys == T in arena order
__global__ void __launch_bounds__(kTile)
prune_apply_kernel(float *__restrict__ arena, const long long *__restrict__ seg, int n_seg, long long n_total,
                   long long ntiles, const PruneState *__restrict__ st, const long long *__restrict__ tile_base)
{
    __shared__ SegSmem sm;
    __shared__ int warp_excl[32];
    load_segments(sm, seg, n_seg);
    const unsigned T = st->prefix;
    const long long need = st->need;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long v = t * kTile + threadIdx.x;
        long long a = -1;
        unsigned key = 0xffffffffu;
        float w = 0.0f;
        if (v < n_total) {
            a = arena_index(sm, n_seg, v);
            w = arena[a];
            key = magnitude_key(w);
        }
        const bool tie = key == T;
        const unsigned ball = __ballot_sync(0xffffffffu, tie);
        if (lane == 0) warp_excl[wid] = __popc(ball);
        __syncthreads();
        if (wid == 0) {                         // exclusive scan of the 32 warp counts
            const int c = warp_excl[lane];
            int x = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            warp_excl[lane] = x - c;
        }
        __syncthreads();
        const long long rank = tile_base[t] + warp_excl[wid] + __popc(ball & ((1u << lane) - 1u));
        if (key < T || (tie && rank < need)) arena[a] = w * 0.0f;   // weight_orig * weight_mask: -w stays -0, NaN NaN
        __syncthreads();                        // warp_excl is reused by the next tile
    }
}

__global__ void negate_indexed_kernel(float *__restrict__ arena, const long long *__restrict__ idx, long long n)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long a = idx[i];
        arena[a] = -arena[a];
    }
}

int grid_for(long long ntiles)
{
    const long long cap = 2LL * ipr_sm_count();
    return (int)(ntiles < cap ? ntiles : cap);
}

}  // namespace

extern "C" size_t ipr_prune_workspace_bytes(int64_t n_total)
{
    if (n_total < 1) return 0;
    const long long ntiles = (n_total + kTile - 1) / kTile;
    return align256(sizeof(PruneState)) + align256(kBins * sizeof(unsigned)) + align256((size_t)ntiles * sizeof(int)) +
           (size_t)ntiles * sizeof(long long);
}

extern "C" int ipr_prune_magnitude_f32(float *arena, const int64_t *segments, int n_segments, int64_t n_total,
                                       int64_t k, void *workspace, size_t workspace_bytes, ipr_stream_t stream)
{
    IPR_REQUIRE(arena && segments && workspace, IPR_E_NULL);
    IPR_REQUIRE(n_segments >= 1 && n_total >= 1 && k >= 0 && k <= n_total, IPR_E_SHAPE);
    IPR_REQUIRE(n_segments <= IPR_PRUNE_MAX_SEGMENTS, IPR_E_UNSUPPORTED);
    IPR_REQUIRE(workspace_bytes >= ipr_prune_workspace_bytes(n_total), IPR_E_WORKSPACE);
    IPR_REQUIRE(((uintptr_t)workspace & 255u) == 0 && ((uintptr_t)segments & 7u) == 0, IPR_E_ALIGN);
    if (k == 0) return IPR_OK;                  // nothing to zero: no launch
    cudaStream_t st = ipr_cu(stream);
    const long long ntiles = (n_total + kTile - 1) / kTile;
    const Workspace w = carve(workspace, ntiles);
    const long long *seg = reinterpret_cast<const long long *>(segments);
    const int grid = grid_for(ntiles);
    prune_init_kernel<<<1, 1024, 0, st>>>(w.state, w.hist, (long long)k);
    IPR_LAUNCH_CHECK();
    const int shifts[3] = {20, 10, 0}, widths[3] = {11, 10, 10};
    for (int p = 0; p < 3; p++) {
        prune_hist_kernel<<<grid, kTile, 0, st>>>(arena, seg, n_segments, (long long)n_total, w.state, w.hist,
                                                  shifts[p], widths[p]);
        IPR_LAUNCH_CHECK();
        prune_select_kernel<<<1, 1024, 0, st>>>(w.state, w.hist, widths[p], p == 2);
        IPR_LAUNCH_CHECK();
    }
    prune_tie_count_kernel<<<grid, kTile, 0, st>>>(arena, seg, n_segments, (long long)n_total, ntiles, w.state,
                                                   w.tile_ties);
    IPR_LAUNCH_CHECK();
    prune_tile_scan_kernel<<<1, 1024, 0, st>>>(w.tile_ties, w.tile_base, ntiles);
    IPR_LAUNCH_CHECK();
    prune_apply_kernel<<<grid, kTile, 0, st>>>(arena, seg, n_segments, (long long)n_total, ntiles, w.state,
                                               w.tile_base);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

extern "C" int ipr_negate_indexed_f32(float *arena, const int64_t *index, int64_t n, ipr_stream_t stream)
{
    IPR_REQUIRE(n >= 0, IPR_E_SHAPE);
    if (n == 0) return IPR_OK;
    IPR_REQUIRE(arena && index, IPR_E_NULL);
    const long long blocks = (n + 255) / 256;
    const int grid = (int)(blocks < 4LL * ipr_sm_count() ? blocks : 4LL * ipr_sm_count());
    negate_indexed_kernel<<<grid, 256, 0, ipr_cu(stream)>>>(arena, reinterpret_cast<const long long *>(index),
                                                           (long long)n);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

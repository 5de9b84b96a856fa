// tapfold.cu -- the 3-output-channel 3x3 layers (G's ConvTranspose2d(64,3,3,1,1)+Tanh, D's first-layer input gradient)
// as ONE launch: the tap GEMM to 27 (tap, channel) columns and the nine-tap fold, with the tap tensor kept on chip.
//
// The unfused path writes T[pixel][32] fp32 from the GEMM (67 MB at batch 512) and reads it back in col2im3, because
// the fold needs taps of neighbouring pixels that a 128-row tile does not hold.  Here one persistent CTA owns whole
// images: every 128-row sub-tile of an image gets its own M=128, N=32 TMEM accumulator (8 x 32 columns for 32 x 32),
// two images are in flight (epilogue of image i overlaps the TMA / MMA of image i+1), and the epilogue writes the
// scaled taps into a zero-haloed shared-memory copy of the image and folds them from there.
//
// Larger images (64 x 64: a 505 KB staged image) run in BANDS: a work item is (image, R output rows), whose fold
// needs the taps of input rows r0-1 .. r0+R.  The band stages them into a zero-haloed (R+2) x (W+2) buffer by
// computing whole, GEMM-aligned sub-tiles: the ones covering the band plus, inside the image, the aligned sub-tile
// above and the one below, of which only the row next to the band is kept.  A whole image is the band case with
// R = height (one band, no halo sub-tiles), so both entry points launch the same kernel.
//
// Bit-identical to tapgemm_kernel<32, ..., IPR_EPI_LINEAR_F32> + col2im3_kernel: every sub-tile issues the same four
// K=16 MMAs with the same accumulate flags on the same TMA box (starting at a multiple of 128 / width rows, as in
// the GEMM), the accumulator is scaled by the same expression, and the nine taps are summed in col2im3's order
// (from 0.f, kh outer, kw inner, halo taps +0.f), then tanhf.
#include "ipr_common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int TF_K = 64;                             // input channels = one 128-byte swizzle row
constexpr int TF_N = 32;                             // 27 (tap, channel) columns stored 32 wide
constexpr int TF_ROWS = 128;                         // rows of one sub-tile (one accumulator)
constexpr int TF_STAGES = 4;
constexpr int TF_A_BYTES = TF_ROWS * TF_K * 2;       // 16 KB
constexpr int TF_B_BYTES = TF_N * TF_K * 2;          // 4 KB, resident
constexpr int TF_PITCH = 29;                         // floats per staged pixel (27 used; odd => conflict-free)
constexpr int TF_EPI_WARPS = 8;
constexpr int TF_EPI_THREADS = TF_EPI_WARPS * 32;
constexpr int TF_THREADS = TF_EPI_THREADS + 64;      // + TMA producer warp + MMA issuer warp
constexpr int TF_MAX_SUBS = 8;                       // sub-tiles per work item: 2 items x 8 x 32 = 512 TMEM columns
constexpr int TF_SMEM_LIMIT = 227 * 1024;

struct TfParams {
    int n_img, h, w, tile_h;
    int band_rows, n_bands;                          // R output rows per work item, ceil(h / R) items per image
    int subs;                                        // most sub-tiles (accumulators) one work item uses
    uint32_t tmem_cols;
    const float *sigma;
    float *out;
    int tanh_out;
};

// the staged taps of one work item: `rows` output rows plus a halo row above and below, halo columns left and right
__host__ __device__ constexpr size_t tf_img_bytes(int rows, int w) {   // rounded up: the mbarriers follow it
    return ((size_t)(rows + 2) * (w + 2) * TF_PITCH * 4 + 15) & ~(size_t)15;
}
__host__ __device__ constexpr size_t tf_bar_bytes() { return 128; }
// 1024 bytes of slack for the SWIZZLE_128B alignment of the A stages
__host__ __device__ constexpr size_t tf_smem_bytes(int rows, int w) {
    return 1024 + (size_t)TF_STAGES * TF_A_BYTES + TF_B_BYTES + tf_img_bytes(rows, w) + tf_bar_bytes();
}

// Work item -> output rows [r0, r1) of image img and the aligned sub-tiles [sub_lo, sub_hi) that hold their taps and
// the taps of the rows next to them (rows r0-1 and r1, where they are inside the image).
struct TfItem {
    int img, r0, r1, sub_lo, sub_hi;
};
__device__ __forceinline__ TfItem tf_item(const TfParams &p, int wi) {
    TfItem t;
    t.img = wi / p.n_bands;
    t.r0 = (wi - t.img * p.n_bands) * p.band_rows;
    t.r1 = min(p.h, t.r0 + p.band_rows);
    t.sub_lo = max(t.r0 - 1, 0) / p.tile_h;
    t.sub_hi = (min(t.r1 + 1, p.h) + p.tile_h - 1) / p.tile_h;
    return t;
}

__device__ __forceinline__ void epi_bar_sync() {     // the epilogue warps only (named barrier 1)
    asm volatile("bar.sync 1, %0;" ::"n"(TF_EPI_THREADS) : "memory");
}

__global__ void __launch_bounds__(TF_THREADS, 1)
tapfold3_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TfParams p)
{
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = smem_base;
    const uint32_t sB = sA + TF_STAGES * TF_A_BYTES;
    float *img_sm = reinterpret_cast<float *>(smem_raw + (smem_base - smem_u32(smem_raw)) + TF_STAGES * TF_A_BYTES + TF_B_BYTES);
    const int hw = p.h * p.w, pitch_w = p.w + 2, n_items = p.n_img * p.n_bands;
    const uint32_t bar_full = sB + TF_B_BYTES + (uint32_t)tf_img_bytes(p.band_rows, p.w);
    const uint32_t bar_empty = bar_full + TF_STAGES * 8;
    const uint32_t bar_acc_full = bar_empty + TF_STAGES * 8;    // 2 x 8
    const uint32_t bar_acc_empty = bar_acc_full + 2 * 8;        // 2 x 8
    const uint32_t bar_bres = bar_acc_empty + 2 * 8;
    const uint32_t tmem_slot = bar_bres + 8;
    const uint32_t buf_cols = (uint32_t)p.subs * TF_N;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int WARP_TMA = TF_EPI_WARPS, WARP_MMA = TF_EPI_WARPS + 1;
    if (warp == WARP_TMA && lane == 0) {
        tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB);
        for (int s = 0; s < TF_STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(bar_acc_full + 8 * b, 1); mbar_init(bar_acc_empty + 8 * b, TF_EPI_WARPS); }
        mbar_init(bar_bres, 1);
        mbar_fence_init();
    }
    if (warp == WARP_MMA) tmem_alloc(tmem_slot, p.tmem_cols);
    // the halo columns stay zero for the whole launch (only interior pixels are ever written); so do the halo rows of
    // a whole image, while a band stages image rows there and clears them again at the top and bottom of an image
    for (int i = threadIdx.x; i < (p.band_rows + 2) * pitch_w * TF_PITCH; i += TF_THREADS) img_sm[i] = 0.0f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    ipr_pdl_wait();
    ipr_pdl_trigger();

    if (warp == WARP_TMA) {
        // ===================== TMA producer: B once, then each item's sub-tiles (4-D box: 64 ch x W x tile_h x 1)
        if (lane == 0) {
            mbar_expect_tx(bar_bres, TF_B_BYTES);
            tma_load_2d(sB, &mapB, bar_bres, 0, 0);
            uint32_t g = 0;
            for (int wi = blockIdx.x; wi < n_items; wi += gridDim.x) {
                const TfItem t = tf_item(p, wi);
                for (int sub = t.sub_lo; sub < t.sub_hi; sub++, g++) {
                    const int s = g % TF_STAGES;
                    const uint32_t par = (g / TF_STAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, par ^ 1u);
                    mbar_expect_tx(bar_full + 8 * s, TF_A_BYTES);
                    tma_load_4d(sA + s * TF_A_BYTES, &mapA, bar_full + 8 * s, 0, 0, sub * p.tile_h, t.img);
                }
            }
        }
        __syncwarp();
    } else if (warp == WARP_MMA) {
        // ===================== MMA issuer: per sub-tile exactly the tap GEMM's sequence (one k-block, 4 x K=16)
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(TF_ROWS, TF_N);
            mbar_wait(bar_bres, 0);
            tc_fence_after();
            const uint64_t db = umma_desc_sw128(sB, 0, 1024);
            uint32_t g = 0, it = 0;
            for (int wi = blockIdx.x; wi < n_items; wi += gridDim.x, it++) {
                const TfItem t = tf_item(p, wi);
                const uint32_t buf = it & 1u;
                mbar_wait(bar_acc_empty + 8 * buf, ((it >> 1) & 1u) ^ 1u);
                tc_fence_after();
                for (int sub = t.sub_lo; sub < t.sub_hi; sub++, g++) {
                    const int s = g % TF_STAGES;
                    const uint32_t par = (g / TF_STAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, par);
                    tc_fence_after();
                    const uint32_t acc = tmem_base + buf * buf_cols + (sub - t.sub_lo) * TF_N;
#pragma unroll
                    for (int k = 0; k < TF_K / 16; k++) {
                        const uint64_t da = umma_desc_sw128(sA + s * TF_A_BYTES, 0, 1024);
                        umma_bf16(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, k != 0 ? 1u : 0u);
                    }
                    umma_commit(bar_empty + 8 * s);
                }
                umma_commit(bar_acc_full + 8 * buf);
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue (warps 0..7): TMEM -> scaled taps in the haloed band -> fold -> NCHW
        const int q = warp & 3, half = warp >> 2;     // TMEM lane quarter; the two warps of a quarter split the sub-tiles
        const int row = q * 32 + lane;
        const float inv_sigma = p.sigma ? 1.0f / __ldg(p.sigma) : 1.0f;
        const int tid = threadIdx.x;
        uint32_t it = 0;
        for (int wi = blockIdx.x; wi < n_items; wi += gridDim.x, it++) {
            const TfItem t = tf_item(p, wi);
            const int band_px = (t.r1 - t.r0) * p.w;
            if (p.n_bands > 1) {
                // a halo row outside the image reads as zero; an earlier band may have staged image rows there
                const int line = pitch_w * TF_PITCH;
                if (t.r0 == 0)
                    for (int i = tid; i < line; i += TF_EPI_THREADS) img_sm[i] = 0.0f;
                if (t.r1 == p.h)
                    for (int i = tid; i < line; i += TF_EPI_THREADS) img_sm[(t.r1 - t.r0 + 1) * line + i] = 0.0f;
            }
            const uint32_t buf = it & 1u;
            mbar_wait_backoff(bar_acc_full + 8 * buf, (it >> 1) & 1u);
            tc_fence_after();
            for (int sub = t.sub_lo + half; sub < t.sub_hi; sub += 2) {
                uint32_t raw[32];
                tmem_ld_32x32(tmem_base + buf * buf_cols + (sub - t.sub_lo) * TF_N + ((uint32_t)(q * 32) << 16), raw);
                tmem_ld_wait();
                float v[TF_N];
#pragma unroll
                for (int j = 0; j < TF_N; j++) v[j] = __uint_as_float(raw[j]);
                if (p.sigma) {
#pragma unroll
                    for (int j = 0; j < TF_N; j++) v[j] *= inv_sigma;
                }
                // image row y -> staged row y - r0 + 1; a halo sub-tile contributes only the row next to the band
                const int m = sub * TF_ROWS + row, y = m / p.w, x = m - y * p.w, ys = y - t.r0 + 1;
                if (ys >= 0 && ys <= t.r1 - t.r0 + 1) {
                    float *dst = img_sm + (ys * pitch_w + (x + 1)) * TF_PITCH;
#pragma unroll
                    for (int j = 0; j < 27; j++) dst[j] = v[j];
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_acc_empty + 8 * buf);     // TMEM of this item is free for item i+2
            epi_bar_sync();                                         // every tap of the band is staged
            float *ob = p.out + (size_t)t.img * 3 * hw + (size_t)t.r0 * p.w;
            for (int pix = tid; pix < band_px; pix += TF_EPI_THREADS) {
                const int y = pix / p.w, x = pix - y * p.w;
                float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
                for (int kh = 0; kh < 3; kh++) {
#pragma unroll
                    for (int kw = 0; kw < 3; kw++) {
                        // source pixel (y+1-kh, x+1-kw) -> halo coordinates (y+2-kh, x+2-kw)
                        const float *src = img_sm + ((y + 2 - kh) * pitch_w + (x + 2 - kw)) * TF_PITCH + (kh * 3 + kw) * 3;
                        a0 += src[0]; a1 += src[1]; a2 += src[2];
                    }
                }
                if (p.tanh_out) { a0 = tanhf(a0); a1 = tanhf(a1); a2 = tanhf(a2); }
                ob[pix] = a0; ob[hw + pix] = a1; ob[2 * hw + pix] = a2;
            }
            epi_bar_sync();                                         // the staging buffer may be overwritten
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WARP_MMA) tmem_dealloc(tmem_base, p.tmem_cols);
}

// Launch over work items of band_rows output rows (band_rows = height: whole images).  The caller has checked the
// pointers, the shape and that the item fits TMEM (subs <= TF_MAX_SUBS) and shared memory.
int tf_launch(const void *a, const void *b, const float *sigma, float *out, int64_t batch, int height, int width,
              int band_rows, int tanh_out, ipr_stream_t stream)
{
    TfParams p;
    p.n_img = (int)batch; p.h = height; p.w = width; p.tile_h = TF_ROWS / width;
    p.band_rows = band_rows; p.n_bands = (height + band_rows - 1) / band_rows;
    p.subs = p.n_bands == 1 ? height / p.tile_h : band_rows / p.tile_h + 2;
    uint32_t cols = 32;
    while (cols < 2u * p.subs * TF_N) cols <<= 1;                   // tcgen05.alloc: a power of two >= 32
    p.tmem_cols = cols;
    p.sigma = sigma; p.out = out; p.tanh_out = tanh_out ? 1 : 0;

    CUtensorMap ma, mb;
    {
        const uint64_t C = TF_K, W = width, H = height, N = batch;
        const uint64_t dims[4] = {C, W, H, N};
        const uint64_t str[3] = {C * 2, W * C * 2, H * W * C * 2};
        const uint32_t box[4] = {(uint32_t)TF_K, (uint32_t)width, (uint32_t)p.tile_h, 1u};
        int rc = make_tmap_bf16(&ma, a, 4, dims, str, box);
        if (rc) return rc;
    }
    {
        const uint64_t dims[2] = {TF_K, TF_N};
        const uint64_t str[1] = {TF_K * 2};
        const uint32_t box[2] = {(uint32_t)TF_K, (uint32_t)TF_N};
        int rc = make_tmap_bf16(&mb, b, 2, dims, str, box);
        if (rc) return rc;
    }
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(tapfold3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TF_SMEM_LIMIT);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const long long items = (long long)p.n_img * p.n_bands;
    const int ctas = items < ipr_sm_count() ? (int)items : ipr_sm_count();
    IPR_LAUNCH_PDL((tapfold3_kernel), ctas, TF_THREADS, tf_smem_bytes(band_rows, width), ipr_cu(stream), ma, mb, p);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

// Rows per band for a (height, width) image: the largest multiple of 128 / width whose sub-tiles, with the halo
// sub-tile above and below, fit two items in TMEM (<= TF_MAX_SUBS) and whose staged taps fit in shared memory.
// 64 x 64: 12 rows (6 + 2 sub-tiles, 107 KB staged), 6 bands an image, 384 items at batch 64 for 148 SMs;
// 128 x 128: 6 rows; 32 x 32: 24 rows.  0 if no band fits.
int tf_band_rows(int height, int width)
{
    const int tile_h = TF_ROWS / width;
    int r = (TF_MAX_SUBS - 2) * tile_h;
    while (r >= tile_h && tf_smem_bytes(r, width) > (size_t)TF_SMEM_LIMIT) r -= tile_h;
    if (r < tile_h) return 0;
    return r < height ? r : height;
}

}  // namespace

extern "C" int ipr_tapfold3_f32(const void *a, const void *b, const float *sigma, float *out, int64_t batch, int height,
                                int width, int tanh_out, ipr_stream_t stream)
{
    IPR_REQUIRE(a && b && out, IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && batch <= INT32_MAX && height > 0 && width > 0, IPR_E_SHAPE);
    IPR_REQUIRE(ipr_aligned16(a) && ipr_aligned16(b) && ((uintptr_t)out & 3u) == 0, IPR_E_ALIGN);
    // whole images of whole 128-row sub-tiles (a sub-tile is 128 / width full rows), at most 8 sub-tiles per image
    const long long hw = (long long)height * width;
    IPR_REQUIRE(hw % TF_ROWS == 0 && hw <= TF_ROWS * TF_MAX_SUBS && width <= TF_ROWS && TF_ROWS % width == 0,
                IPR_E_UNSUPPORTED);
    IPR_REQUIRE(tf_smem_bytes(height, width) <= (size_t)TF_SMEM_LIMIT, IPR_E_UNSUPPORTED);
    return tf_launch(a, b, sigma, out, batch, height, width, height, tanh_out, stream);
}

extern "C" int ipr_tapfold3_band_f32(const void *a, const void *b, const float *sigma, float *out, int64_t batch,
                                     int height, int width, int tanh_out, ipr_stream_t stream)
{
    IPR_REQUIRE(a && b && out, IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && batch <= INT32_MAX && height > 0 && width > 0, IPR_E_SHAPE);
    IPR_REQUIRE(ipr_aligned16(a) && ipr_aligned16(b) && ((uintptr_t)out & 3u) == 0, IPR_E_ALIGN);
    // whole 128-row sub-tiles of whole image rows (a sub-tile is 128 / width rows; then height is a multiple of it)
    const long long hw = (long long)height * width;
    IPR_REQUIRE(hw % TF_ROWS == 0 && width <= TF_ROWS && TF_ROWS % width == 0 && hw <= INT32_MAX / 3,
                IPR_E_UNSUPPORTED);
    const int rows = tf_band_rows(height, width);
    IPR_REQUIRE(rows > 0, IPR_E_UNSUPPORTED);
    IPR_REQUIRE(batch * ((height + rows - 1) / rows) <= INT32_MAX, IPR_E_SHAPE);    // work items are ints
    return tf_launch(a, b, sigma, out, batch, height, width, rows, tanh_out, stream);
}

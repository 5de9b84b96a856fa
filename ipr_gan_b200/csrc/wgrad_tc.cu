// wgrad_tc.cu -- weight gradients of the tap-GEMM layers on tcgen05 tensor cores.
//
//   dW[p][n][t*Cx + c] = sum_{pixels m} Y[pixel(m)][n] * X[pixel(m) + tap_t][c]
//
// The reduction runs over PIXELS, which are the strided dimension of both NHWC operands, so both
// MMA operands are MN-major: a TMA box (64 channels x 64 pixels) lands in shared memory as 64 rows of
// 128 swizzled bytes, i.e. exactly the canonical MN-major SWIZZLE_128B atom layout
// (leading-dimension byte offset = one 64-channel block = 8 KB, stride byte offset = 8 pixel rows = 1 KB),
// and the instruction descriptor carries a_major = b_major = MN.  No transposed copy is ever made.
//
// CTA tile: 128 output channels (two 64-channel boxes of Y) x 64 * X_UNITS columns (X_UNITS (tap, 64-channel) units
// of X, each its own shifted TMA box with zero fill at the borders) x a slice of the pixel range (split-K).
// Partial tiles go to an fp32 workspace [split][phase][n][t*Cx + c]; ipr_wgrad_reduce_f32 adds the splits
// in a fixed order (deterministic) and scatters into the parameter's own (reference) layout.
#include "ipr_common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int KB_PIX = 64;                    // pixels per k-block
constexpr int UNIT_BYTES = KB_PIX * 128;      // one 64-channel x 64-pixel box
constexpr int NUM_THREADS = 192;
constexpr int UMMA_K = 16;

struct WgParams {
    int n_imgs, q_h, q_w, kb_rows, kb_imgs, kb_per_img, total_kb, kb_per_split;
    int y_c, x_c, x_chunks, n_units, n_taps, k_total, n_pad;
    int8_t y_map[IPR_TG_MAX_PHASES];
    int8_t tap_map[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t tap_dh[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t tap_dw[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    float *ws;
    int n_phases;
};

struct Maps { CUtensorMap y[4]; CUtensorMap x[4]; };

template <int X_UNITS, int STAGES>
__global__ void __launch_bounds__(NUM_THREADS)
wgrad_kernel(const __grid_constant__ Maps maps, const WgParams p)
{
    constexpr int STAGE_BYTES = (2 + X_UNITS) * UNIT_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = smem_base + STAGES * STAGE_BYTES;
    const uint32_t bar_empty = bar_full + STAGES * 8;
    const uint32_t bar_tmem = bar_empty + STAGES * 8;
    const uint32_t tmem_slot = bar_tmem + 8;
    constexpr uint32_t TMEM_COLS = X_UNITS == 2 ? 128 : 256;    // power of two >= 64 * X_UNITS

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = (p.n_units + X_UNITS - 1) / X_UNITS;
    const int m_blk = blockIdx.x / n_tiles, n_tile = blockIdx.x - m_blk * n_tiles;
    const int split = blockIdx.y, phase = blockIdx.z;
    const int kb0 = split * p.kb_per_split;
    const int kb1 = min(p.total_kb, kb0 + p.kb_per_split);
    const int num_kb = max(0, kb1 - kb0);
    const int unit0 = X_UNITS * n_tile;
    const int units_here = min(X_UNITS, p.n_units - unit0);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_tmem, 1);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    ipr_pdl_wait();                 // prologue above overlapped the previous kernel's tail (PDL)
    ipr_pdl_trigger();

    if (warp == 0) {
        if (lane == 0) {
            const CUtensorMap *my = &maps.y[p.y_map[phase]];
            for (int i = 0; i < num_kb; i++) {
                const int kb = kb0 + i;
                const int s = i % STAGES;
                const uint32_t par = (uint32_t)((i / STAGES) & 1);
                int img0, h0;
                if (p.kb_imgs == 1) { img0 = kb / p.kb_per_img; h0 = (kb - img0 * p.kb_per_img) * p.kb_rows; }
                else { img0 = kb * p.kb_imgs; h0 = 0; }
                mbar_wait(bar_empty + 8 * s, par ^ 1u);
                mbar_expect_tx(bar_full + 8 * s, (2 + units_here) * UNIT_BYTES);
                const uint32_t st = smem_base + s * STAGE_BYTES;
                tma_load_4d(st, my, bar_full + 8 * s, (2 * m_blk) * 64, 0, h0, img0);
                tma_load_4d(st + UNIT_BYTES, my, bar_full + 8 * s, (2 * m_blk + 1) * 64, 0, h0, img0);
                for (int u = 0; u < units_here; u++) {
                    const int unit = unit0 + u;
                    const int tap = unit / p.x_chunks, cc = unit - tap * p.x_chunks;
                    const CUtensorMap *mx = &maps.x[p.tap_map[phase][tap]];
                    tma_load_4d(st + (2 + u) * UNIT_BYTES, mx, bar_full + 8 * s, cc * 64, (int)p.tap_dw[phase][tap],
                                h0 + (int)p.tap_dh[phase][tap], img0);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(128, 64 * X_UNITS, /*a_major=MN*/ 1, /*b_major=MN*/ 1);
            for (int i = 0; i < num_kb; i++) {
                const int s = i % STAGES;
                const uint32_t par = (uint32_t)((i / STAGES) & 1);
                mbar_wait(bar_full + 8 * s, par);
                tc_fence_after();
                const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
                for (int k = 0; k < KB_PIX / UMMA_K; k++) {
                    // 16 pixel rows per MMA = 2048 bytes along K; 64-channel blocks are UNIT_BYTES apart (LBO)
                    const uint64_t da = umma_desc_sw128(st + k * UMMA_K * 128, UNIT_BYTES, 1024);
                    const uint64_t db = umma_desc_sw128(st + 2 * UNIT_BYTES + k * UMMA_K * 128, UNIT_BYTES, 1024);
                    umma_bf16(tmem_base, da, db, idesc, (i | k) != 0 ? 1u : 0u);
                }
                umma_commit(bar_empty + 8 * s);
            }
            umma_commit(bar_tmem);
        }
        __syncwarp();
    } else {
        const int q = warp & 3;
        const int n = m_blk * 128 + q * 32 + lane;        // output channel (row of dW)
        float *dst_row = p.ws + (((size_t)split * p.n_phases + phase) * p.n_pad + n) * p.k_total;
        if (num_kb > 0) { mbar_wait_backoff(bar_tmem, 0); tc_fence_after(); }
#pragma unroll 1
        for (int c0 = 0; c0 < 64 * X_UNITS; c0 += 32) {
            const int unit = unit0 + (c0 >> 6);
            if (unit >= p.n_units) break;
            if (unit * 64 + (c0 & 63) >= p.k_total) break;      // narrow single-tap layers: columns past x_c are zero fill
            uint32_t raw[32];
            if (num_kb > 0) {
                tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, raw);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; j++) raw[j] = 0u;
            }
            float4 *dst = reinterpret_cast<float4 *>(dst_row + (size_t)unit * 64 + (c0 & 63));
#pragma unroll
            for (int g = 0; g < 8; g++)
                dst[g] = make_float4(__uint_as_float(raw[4 * g]), __uint_as_float(raw[4 * g + 1]),
                                     __uint_as_float(raw[4 * g + 2]), __uint_as_float(raw[4 * g + 3]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// grad[row(n)*s_n + dst_off[p*k_total + k]] (+)= scale * sum_splits ws[split][p][n][k]   (dst_off < 0: padding column)
// One thread per (p, n, k): coalesced reads along k, 8 independent loads in flight over the splits (fixed summation
// order), scattered 4-byte writes into the parameter's own layout (the output is tiny compared with the partials).
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float *__restrict__ ws, int splits, int phases, int n_rows, int n_pad, int k_total,
                    const int *__restrict__ dst_off, const int *__restrict__ row_map, long long s_n,
                    float *__restrict__ grad, int accumulate, float scale)
{
    ipr_pdl_wait();
    ipr_pdl_trigger();
    const long long total = (long long)phases * n_rows * k_total;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int k = (int)(e % k_total);
    const long long t = e / k_total;
    const int n = (int)(t % n_rows);
    const int ph = (int)(t / n_rows);
    const int off = __ldg(dst_off + (size_t)ph * k_total + k);
    if (off < 0) return;
    const size_t split_stride = (size_t)phases * n_pad * k_total;
    const float *src = ws + ((size_t)ph * n_pad + n) * k_total + k;
    float acc = 0.0f;
    int s = 0;
    for (; s + 8 <= splits; s += 8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = src[(size_t)(s + j) * split_stride];
#pragma unroll
        for (int j = 0; j < 8; j++) acc += v[j];
    }
    for (; s < splits; s++) acc += src[(size_t)s * split_stride];
    const int rn = row_map ? __ldg(row_map + n) : n;
    if (rn < 0) return;                                  // padding row of the GEMM (N padded to a multiple of 16)
    float *dst = grad + (size_t)rn * s_n + off;
    *dst = accumulate ? *dst + acc * scale : acc * scale;
}

// Same reduction for plain convolution weights, destination-major: one thread per (row n, input channel c) gathers the
// kk = kh*kw taps of that weight slice from the partials (coalesced along c) and writes them as ONE contiguous run
// grad[n*s_n + c*s_c + 0..kk) -- Conv2d (O,I,kh,kw): s_n = I*kk, s_c = kk; ConvTranspose2d (I,O,kh,kw): s_n = kk,
// s_c = O*kk.  The element-major kernel above scatters 4-byte read-modify-writes (57 us for the 512->256 k4 layer).
struct TapOf { int v[16]; };                      // destination tap j -> phase * n_taps + tap

__global__ void __launch_bounds__(256)
wgrad_reduce_taps_kernel(const float *__restrict__ ws, int splits, int phases, int n_rows, int n_pad, int n_taps, int x_c,
                         TapOf tap_of, int kk, long long s_n, long long s_c, float *__restrict__ grad, int accumulate,
                         float scale)
{
    ipr_pdl_wait();
    ipr_pdl_trigger();
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)n_rows * x_c) return;
    const int c = (int)(e % x_c), n = (int)(e / x_c);
    const int k_total = n_taps * x_c;
    const size_t split_stride = (size_t)phases * n_pad * k_total;
    float *dst = grad + (size_t)n * s_n + (size_t)c * s_c;
    float out[16];
    size_t src_off[16];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        const int pt = tap_of.v[j < kk ? j : 0], ph = pt / n_taps, t = pt - ph * n_taps;
        src_off[j] = ((size_t)ph * n_pad + n) * k_total + (size_t)t * x_c + c;
        out[j] = 0.0f;
    }
    for (int sp = 0; sp < splits; sp++) {             // 16 independent loads in flight per split, fixed summation order
        const float *base = ws + (size_t)sp * split_stride;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = j < kk ? base[src_off[j]] : 0.0f;
#pragma unroll
        for (int j = 0; j < 16; j++) out[j] += v[j];
    }
#pragma unroll
    for (int j = 0; j < 16; j++) out[j] *= scale;
    if (kk == 16 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        float4 *d4 = reinterpret_cast<float4 *>(dst);
#pragma unroll
        for (int g = 0; g < 4; g++) {
            float4 v = make_float4(out[4 * g], out[4 * g + 1], out[4 * g + 2], out[4 * g + 3]);
            if (accumulate) { const float4 o = d4[g]; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
            d4[g] = v;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; j++)
            if (j < kk) dst[j] = accumulate ? dst[j] + out[j] : out[j];
    }
}

// Tile configuration: X_UNITS (tap, 64-channel) units of X per CTA tile, i.e. N = 64 * X_UNITS, and as many smem stages
// of (2 + X_UNITS) * 8 KB as fit in about 200 KB: <2, 6>, <3, 5> or <4, 4>, one CTA per SM.  X_UNITS is the widest of
// {4, 3, 2} that divides the layer's unit count (9-tap layers -> 3, 16-tap / 4-tap layers -> 4): the kernel is paced by
// TMA requests per MAC, which fall by 25 % going from N = 128 to N = 192 / 256 (measured: 1027 -> 1248 cycles per
// k-block for twice the MACs), provided no tile is left partly empty.
int wgrad_x_units(int n_units) {
    if (n_units % 4 == 0) return 4;
    if (n_units % 3 == 0) return 3;
    return 2;
}

template <int X_UNITS, int STAGES>
int launch_wgrad(const Maps &maps, const WgParams &p, dim3 grid, cudaStream_t st)
{
    constexpr size_t smem = (size_t)STAGES * (2 + X_UNITS) * UNIT_BYTES + (2 * STAGES + 2) * 8 + 1024 + 64;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(wgrad_kernel<X_UNITS, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    IPR_LAUNCH_PDL((wgrad_kernel<X_UNITS, STAGES>), grid, NUM_THREADS, smem, st, maps, p);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

int geometry(const ipr_wgrad_t *d, WgParams &p)
{
    const int per_img = d->q_h * d->q_w;
    IPR_REQUIRE(per_img > 0 && d->q_w <= KB_PIX, IPR_E_UNSUPPORTED);
    if (per_img >= KB_PIX) {
        IPR_REQUIRE(KB_PIX % d->q_w == 0, IPR_E_UNSUPPORTED);
        p.kb_rows = KB_PIX / d->q_w;
        IPR_REQUIRE(d->q_h % p.kb_rows == 0, IPR_E_UNSUPPORTED);
        p.kb_imgs = 1;
        p.kb_per_img = d->q_h / p.kb_rows;
        p.total_kb = d->n_imgs * p.kb_per_img;
    } else {
        IPR_REQUIRE(KB_PIX % per_img == 0, IPR_E_UNSUPPORTED);
        p.kb_rows = d->q_h;
        p.kb_imgs = KB_PIX / per_img;
        p.kb_per_img = 1;
        p.total_kb = (d->n_imgs + p.kb_imgs - 1) / p.kb_imgs;
    }
    p.n_pad = ((d->y_c + 127) / 128) * 128;
    p.k_total = d->n_taps * d->x_c;
    return IPR_OK;
}

int make_maps(const void *base, int C, int H, int W, int N, int parity, const uint32_t *box, CUtensorMap *out)
{
    const uint64_t c = C, w = W, h = H, n = N;
    if (!parity) {
        const uint64_t dims[4] = {c, w, h, n};
        const uint64_t str[3] = {c * 2, w * c * 2, h * w * c * 2};
        int rc = make_tmap_bf16(&out[0], base, 4, dims, str, box);
        if (rc) return rc;
        out[1] = out[2] = out[3] = out[0];
        return 0;
    }
    const uint64_t dims[4] = {c, w / 2, h / 2, n};
    const uint64_t str[3] = {2 * c * 2, 2 * w * c * 2, h * w * c * 2};
    for (int ph = 0; ph < 2; ph++)
        for (int pw = 0; pw < 2; pw++) {
            int rc = make_tmap_bf16(&out[ph * 2 + pw], (const char *)base + ((size_t)ph * w + pw) * c * 2, 4, dims, str, box);
            if (rc) return rc;
        }
    return 0;
}

}  // namespace

extern "C" size_t ipr_wgrad_workspace_bytes(const ipr_wgrad_t *d)
{
    if (!d) return 0;
    WgParams p;
    if (geometry(d, p) != IPR_OK) return 0;
    return (size_t)d->splits * d->n_phases * p.n_pad * p.k_total * sizeof(float);
}

extern "C" int ipr_wgrad_total_kblocks(const ipr_wgrad_t *d)
{
    if (!d) return IPR_E_NULL;
    WgParams p;
    int rc = geometry(d, p);
    return rc != IPR_OK ? rc : p.total_kb;
}

extern "C" int ipr_wgrad_bf16(const ipr_wgrad_t *d, ipr_stream_t stream)
{
    IPR_REQUIRE(d, IPR_E_NULL);
    IPR_REQUIRE(d->y && d->x && d->workspace, IPR_E_NULL);
    IPR_REQUIRE(d->n_imgs > 0 && d->y_c > 0 && d->x_c > 0 && d->splits > 0, IPR_E_SHAPE);
    // X channels are consumed in 64-wide units; a single-tap layer may store fewer (TMA zero-fills the rest)
    IPR_REQUIRE((d->x_c % 64 == 0 || (d->n_taps == 1 && d->x_c % 8 == 0)) && d->y_c % 8 == 0, IPR_E_UNSUPPORTED);
    IPR_REQUIRE(d->n_taps >= 1 && d->n_taps <= IPR_TG_MAX_TAPS && d->n_phases >= 1 && d->n_phases <= IPR_TG_MAX_PHASES,
                IPR_E_SHAPE);
    IPR_REQUIRE(ipr_aligned16(d->y) && ipr_aligned16(d->x) && ipr_aligned16(d->workspace), IPR_E_ALIGN);
    WgParams p;
    int rc = geometry(d, p);
    if (rc != IPR_OK) return rc;
    p.n_imgs = d->n_imgs; p.q_h = d->q_h; p.q_w = d->q_w;
    p.y_c = d->y_c; p.x_c = d->x_c; p.x_chunks = (d->x_c + 63) / 64; p.n_taps = d->n_taps;
    p.n_units = d->n_taps * p.x_chunks; p.n_phases = d->n_phases;
    p.kb_per_split = (p.total_kb + d->splits - 1) / d->splits;
    p.ws = d->workspace;
    for (int ph = 0; ph < IPR_TG_MAX_PHASES; ph++) {
        p.y_map[ph] = d->y_map[ph];
        for (int t = 0; t < IPR_TG_MAX_TAPS; t++) {
            p.tap_map[ph][t] = d->tap_map[ph][t]; p.tap_dh[ph][t] = d->tap_dh[ph][t]; p.tap_dw[ph][t] = d->tap_dw[ph][t];
        }
    }
    Maps maps;
    const uint32_t box[4] = {64u, (uint32_t)d->q_w, (uint32_t)p.kb_rows, (uint32_t)p.kb_imgs};
    const int yh = d->y_parity ? 2 * d->q_h : d->q_h, yw = d->y_parity ? 2 * d->q_w : d->q_w;
    const int xh = d->x_parity ? 2 * d->q_h : d->q_h, xw = d->x_parity ? 2 * d->q_w : d->q_w;
    rc = make_maps(d->y, d->y_c, yh, yw, d->n_imgs, d->y_parity, box, maps.y);
    if (rc) return rc;
    rc = make_maps(d->x, d->x_c, xh, xw, d->n_imgs, d->x_parity, box, maps.x);
    if (rc) return rc;

    const int xu = wgrad_x_units(p.n_units);
    const int n_tiles = (p.n_units + xu - 1) / xu;
    dim3 grid((unsigned)((p.n_pad / 128) * n_tiles), (unsigned)d->splits, (unsigned)d->n_phases);
    switch (xu) {
        case 4:  return launch_wgrad<4, 4>(maps, p, grid, ipr_cu(stream));
        case 3:  return launch_wgrad<3, 5>(maps, p, grid, ipr_cu(stream));
        default: return launch_wgrad<2, 6>(maps, p, grid, ipr_cu(stream));
    }
}

extern "C" int ipr_wgrad_tiles(const ipr_wgrad_t *d)
{
    if (!d) return IPR_E_NULL;
    const int n_units = d->n_taps * ((d->x_c + 63) / 64);
    const int xu = wgrad_x_units(n_units);
    return ((d->y_c + 127) / 128) * ((n_units + xu - 1) / xu) * d->n_phases;
}

extern "C" int ipr_wgrad_reduce_taps_f32(const float *workspace, int splits, int phases, int n_rows, int n_taps, int x_c,
                                         const int32_t *tap_of_host, int kk, int64_t s_n, int64_t s_c, float *grad,
                                         int accumulate, float scale, ipr_stream_t stream)
{
    IPR_REQUIRE(workspace && tap_of_host && grad, IPR_E_NULL);
    IPR_REQUIRE(splits > 0 && phases > 0 && n_rows > 0 && n_taps > 0 && x_c > 0 && kk > 0 && kk <= 16 &&
                kk == phases * n_taps, IPR_E_SHAPE);
    TapOf t;
    for (int j = 0; j < 16; j++) t.v[j] = j < kk ? tap_of_host[j] : 0;
    for (int j = 0; j < kk; j++) IPR_REQUIRE(t.v[j] >= 0 && t.v[j] < phases * n_taps, IPR_E_SHAPE);
    const int n_pad = ((n_rows + 127) / 128) * 128;
    const long long total = (long long)n_rows * x_c;
    IPR_LAUNCH_PDL((wgrad_reduce_taps_kernel), (unsigned)((total + 255) / 256), 256, 0, ipr_cu(stream), workspace, splits, phases,
                   n_rows, n_pad, n_taps, x_c, t, kk, (long long)s_n, (long long)s_c, grad, accumulate, scale);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

extern "C" int ipr_wgrad_reduce_f32(const float *workspace, int splits, int phases, int n_rows, int k_total,
                                    const int32_t *dst_off, const int32_t *row_map, int64_t s_n, float *grad,
                                    int accumulate, float scale, ipr_stream_t stream)
{
    IPR_REQUIRE(workspace && dst_off && grad, IPR_E_NULL);
    IPR_REQUIRE(splits > 0 && phases > 0 && n_rows > 0 && k_total > 0, IPR_E_SHAPE);
    const int n_pad = ((n_rows + 127) / 128) * 128;
    const long long total = (long long)phases * n_rows * k_total;
    IPR_LAUNCH_PDL((wgrad_reduce_kernel), (unsigned)((total + 255) / 256), 256, 0, ipr_cu(stream), workspace, splits, phases, n_rows, n_pad,
                                                                                   k_total, dst_off, row_map,
                                                                                   (long long)s_n, grad, accumulate, scale);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

// trigger.cu -- black-box trigger path: watermark / noise-patch paste, crop (apply_mask),
// latent bit-mask scatter, TransformDist, TransformVar.  All are single-pass, coalesced,
// 128-bit vectorised where alignment allows; HBM-bound (read x + write y).
//
// Bit-exactness: the paste is two separately rounded steps (x*bg, then + (1-bg)*fg) exactly like the
// reference's two in-place tensor ops, so FMA contraction is disabled with explicit _rn intrinsics.
#include "ipr_common.cuh"

namespace {

__device__ __forceinline__ float paste_one(float x, float bg, float fg) {
    // y *= bg ; y += (1 - bg) * fg      (tools/paste_watermark.py:50-51)
    float t = __fmul_rn(x, bg);
    float u = __fmul_rn(__fsub_rn(1.0f, bg), fg);
    return __fadd_rn(t, u);
}

__device__ __forceinline__ float tdist_one(float z) {
    // 0.5 * (1 + erf(z / sqrt(2))) * sqrt(2 pi)      (tools/transform_dist.py:10-11)
    float t = __fdiv_rn(z, 0x1.6a09e6p+0f);
    float y = __fmul_rn(0.5f, __fadd_rn(1.0f, erff(t)));
    return __fmul_rn(y, 0x1.40d932p+1f);
}

struct PasteGeom {
    int C, H, W, s, row0, col0;
};

// One thread per 4 consecutive pixels of a row (W % 4 == 0, 16B-aligned bases).
__global__ void __launch_bounds__(256)
paste_vec4_kernel(const float4 *__restrict__ x, float4 *__restrict__ y, const float *__restrict__ fg,
                  const float *__restrict__ bg, long long n_vec, PasteGeom g,
                  const float4 *__restrict__ z, float4 *__restrict__ xwm, long long z_vec)
{
    ipr_pdl_wait();
    ipr_pdl_trigger();
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int w4 = g.W >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
        float4 v = ipr_ldg_stream4(x + i);
        const int col = (int)(i % w4) << 2;
        const long long rowid = i / w4;
        const int h = (int)(rowid % g.H);
        const int hh = h - g.row0;
        if (hh >= 0 && hh < g.s && col + 3 >= g.col0 && col < g.col0 + g.s) {
            const int c = (int)((rowid / g.H) % g.C);
            const float *fgr = fg + ((size_t)c * g.s + hh) * g.s;
            const float *bgr = bg + (size_t)hh * g.s;
            float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int cc = col + k - g.col0;
                if (cc >= 0 && cc < g.s) e[k] = paste_one(e[k], __ldg(bgr + cc), __ldg(fgr + cc));
            }
            v = make_float4(e[0], e[1], e[2], e[3]);
        }
        ipr_stg_stream4(y + i, v);
    }
    // fused latent transform (optional second stream of work in the same launch)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < z_vec; i += stride) {
        float4 v = __ldg(z + i);
        v.x = tdist_one(v.x); v.y = tdist_one(v.y); v.z = tdist_one(v.z); v.w = tdist_one(v.w);
        xwm[i] = v;
    }
}

__global__ void __launch_bounds__(256)
paste_scalar_kernel(const float *__restrict__ x, float *__restrict__ y, const float *__restrict__ fg,
                    const float *__restrict__ bg, long long n, PasteGeom g,
                    const float *__restrict__ z, float *__restrict__ xwm, long long zn)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v = x[i];
        const int col = (int)(i % g.W);
        const long long rowid = i / g.W;
        const int hh = (int)(rowid % g.H) - g.row0;
        const int cc = col - g.col0;
        if (hh >= 0 && hh < g.s && cc >= 0 && cc < g.s) {
            const int c = (int)((rowid / g.H) % g.C);
            v = paste_one(v, bg[(size_t)hh * g.s + cc], fg[((size_t)c * g.s + hh) * g.s + cc]);
        }
        y[i] = v;
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < zn; i += stride)
        xwm[i] = tdist_one(z[i]);
}

// POST: the evaluation loop's post-processing fused in.
//   CROP_PLAIN    apply_mask's result as is
//   CROP_SIGNED   out = (clamp(crop, -1, 1) + 1) / 2 for normalized=True outputs (experiments/image_generation.py:141-149
//                 `postproc`): same three fp32 operations, same order, so the uint8 conversion downstream sees
//                 bit-identical values
//   CROP_UNIT     out = clamp(crop, 0, 1) for normalized=False outputs, already in data range 1 (SRGAN)
enum CropPost { CROP_PLAIN = 0, CROP_SIGNED = 1, CROP_UNIT = 2 };

template <int POST>
__global__ void __launch_bounds__(256)
crop_kernel(const float *__restrict__ x, float *__restrict__ out, const float *__restrict__ bg,
            long long n_out, PasteGeom g)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += stride) {
        const int cc = (int)(i % g.s);
        const long long t = i / g.s;
        const int hh = (int)(t % g.s);
        const long long plane = t / g.s;                       // n * C + c
        const float b = __ldg(bg + (size_t)hh * g.s + cc);
        const float v = x[((size_t)plane * g.H + (hh + g.row0)) * g.W + (cc + g.col0)];
        // y = ones * bg ; y += (1 - bg) * crop      (tools/paste_watermark.py:58-60)
        float r = __fadd_rn(__fmul_rn(1.0f, b), __fmul_rn(__fsub_rn(1.0f, b), v));
        // torch.clamp propagates NaN; fminf / fmaxf would drop it
        if (POST == CROP_SIGNED) {
            r = (r != r) ? r : fminf(fmaxf(r, -1.0f), 1.0f);
            r = __fmul_rn(__fadd_rn(r, 1.0f), 0.5f);
        } else if (POST == CROP_UNIT) {
            // torch.clamp's min(max(v, lo), hi) with the comparisons spelled out: NaN passes, -0 stays -0
            r = (r < 0.0f) ? 0.0f : r;
            r = (r > 1.0f) ? 1.0f : r;
        }
        out[i] = r;
    }
}

// One CTA handles a slab of rows; the mask is expanded into a shared per-column flag table first.
__global__ void __launch_bounds__(256)
bitmask_kernel(const float *__restrict__ z, float *__restrict__ out, const long long *__restrict__ mask,
               long long batch, int z_dim, int n, float constant)
{
    extern __shared__ unsigned char flag[];
    for (int i = threadIdx.x; i < z_dim; i += blockDim.x) flag[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) flag[(int)mask[i]] = 1;
    __syncthreads();
    const long long total = batch * z_dim;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int d = (int)(i % z_dim);
        out[i] = flag[d] ? constant : z[i];
    }
}

__global__ void __launch_bounds__(256)
tdist_kernel(const float *__restrict__ z, float *__restrict__ out, long long n)
{
    ipr_pdl_wait();
    ipr_pdl_trigger();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = tdist_one(z[i]);
}

__global__ void __launch_bounds__(256)
tvar_kernel(const float *__restrict__ z, float *__restrict__ out, const float *__restrict__ a,
            const float *__restrict__ w, long long n, int dim)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = (int)(i % dim);
        const float av = __ldg(a + d), wv = __ldg(w + d);
        // z * (1 - a) + a * w      (tools/transform_var.py:13)
        out[i] = __fadd_rn(__fmul_rn(z[i], __fsub_rn(1.0f, av)), __fmul_rn(av, wv));
    }
}

inline int grid_for(long long work_items, int threads, int max_waves = 8) {
    long long blocks = (work_items + threads - 1) / threads;
    long long cap = (long long)ipr_sm_count() * max_waves;   // multiple of the SM count
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

int paste_impl(const float *x, float *y, const float *fg, const float *bg, int64_t batch, int C, int H, int W,
               int s, int row0, int col0, const float *z, float *xwm, int64_t zn, cudaStream_t st)
{
    IPR_REQUIRE(x && y && fg && bg, IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && C > 0 && H > 0 && W > 0 && s > 0, IPR_E_SHAPE);
    IPR_REQUIRE(row0 >= 0 && col0 >= 0 && row0 + s <= H && col0 + s <= W, IPR_E_SHAPE);
    IPR_REQUIRE(zn == 0 || (z && xwm), IPR_E_NULL);
    PasteGeom g{C, H, W, s, row0, col0};
    const long long n = (long long)batch * C * H * W;
    const bool vec = (W % 4 == 0) && ipr_aligned16(x) && ipr_aligned16(y) &&
                     (zn == 0 || (zn % 4 == 0 && ipr_aligned16(z) && ipr_aligned16(xwm)));
    if (vec) {
        IPR_LAUNCH_PDL((paste_vec4_kernel), grid_for(n / 4, 256), 256, 0, st, 
            (const float4 *)x, (float4 *)y, fg, bg, n / 4, g, (const float4 *)z, (float4 *)xwm, zn / 4);
    } else {
        paste_scalar_kernel<<<grid_for(n, 256), 256, 0, st>>>(x, y, fg, bg, n, g, z, xwm, zn);
    }
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

}  // namespace

extern "C" int ipr_paste_patch_f32(const float *x, float *y, const float *fg, const float *bg,
                                   int64_t batch, int channels, int height, int width,
                                   int size, int row0, int col0, ipr_stream_t stream)
{
    return paste_impl(x, y, fg, bg, batch, channels, height, width, size, row0, col0, nullptr, nullptr, 0,
                      ipr_cu(stream));
}

extern "C" int ipr_trigger_pair_f32(const float *x, float *ywm, const float *fg, const float *bg,
                                    int64_t batch, int channels, int height, int width, int size, int row0,
                                    int col0, const float *z, float *xwm, int64_t z_numel, ipr_stream_t stream)
{
    IPR_REQUIRE(z && xwm, IPR_E_NULL);
    IPR_REQUIRE(z_numel > 0, IPR_E_SHAPE);
    return paste_impl(x, ywm, fg, bg, batch, channels, height, width, size, row0, col0, z, xwm, z_numel,
                      ipr_cu(stream));
}

namespace {

template <int POST>
int crop_impl(const float *x, float *out, const float *bg, int64_t batch, int channels, int height, int width,
              int size, int row0, int col0, cudaStream_t st)
{
    IPR_REQUIRE(x && out && bg, IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && channels > 0 && height > 0 && width > 0 && size > 0, IPR_E_SHAPE);
    IPR_REQUIRE(row0 >= 0 && col0 >= 0 && row0 + size <= height && col0 + size <= width, IPR_E_SHAPE);
    PasteGeom g{channels, height, width, size, row0, col0};
    const long long n = (long long)batch * channels * size * size;
    crop_kernel<POST><<<grid_for(n, 256), 256, 0, st>>>(x, out, bg, n, g);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

}  // namespace

extern "C" int ipr_crop_patch_f32(const float *x, float *out, const float *bg,
                                  int64_t batch, int channels, int height, int width,
                                  int size, int row0, int col0, ipr_stream_t stream)
{
    return crop_impl<CROP_PLAIN>(x, out, bg, batch, channels, height, width, size, row0, col0, ipr_cu(stream));
}

extern "C" int ipr_crop_postproc_f32(const float *x, float *out, const float *bg,
                                     int64_t batch, int channels, int height, int width,
                                     int size, int row0, int col0, ipr_stream_t stream)
{
    return crop_impl<CROP_SIGNED>(x, out, bg, batch, channels, height, width, size, row0, col0, ipr_cu(stream));
}

extern "C" int ipr_crop_clamp01_f32(const float *x, float *out, const float *bg,
                                    int64_t batch, int channels, int height, int width,
                                    int size, int row0, int col0, ipr_stream_t stream)
{
    return crop_impl<CROP_UNIT>(x, out, bg, batch, channels, height, width, size, row0, col0, ipr_cu(stream));
}

extern "C" int ipr_bitmask_scatter_f32(const float *z, float *out, const int64_t *mask,
                                       int64_t batch, int z_dim, int n, float constant, ipr_stream_t stream)
{
    IPR_REQUIRE(z && out && (mask || n == 0), IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && z_dim > 0 && n >= 0 && n <= z_dim, IPR_E_SHAPE);
    IPR_REQUIRE(z_dim <= 48 * 1024, IPR_E_UNSUPPORTED);
    bitmask_kernel<<<grid_for((long long)batch * z_dim, 256), 256, (size_t)z_dim, ipr_cu(stream)>>>(
        z, out, (const long long *)mask, batch, z_dim, n, constant);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

extern "C" int ipr_transform_dist_f32(const float *z, float *out, int64_t numel, ipr_stream_t stream)
{
    IPR_REQUIRE(z && out, IPR_E_NULL);
    IPR_REQUIRE(numel > 0, IPR_E_SHAPE);
    IPR_LAUNCH_PDL((tdist_kernel), grid_for(numel, 256), 256, 0, ipr_cu(stream), z, out, numel);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

extern "C" int ipr_transform_var_f32(const float *z, float *out, const float *a, const float *w,
                                     int64_t batch, int dim, ipr_stream_t stream)
{
    IPR_REQUIRE(z && out && a && w, IPR_E_NULL);
    IPR_REQUIRE(batch > 0 && dim > 0, IPR_E_SHAPE);
    tvar_kernel<<<grid_for((long long)batch * dim, 256), 256, 0, ipr_cu(stream)>>>(z, out, a, w,
                                                                                 (long long)batch * dim, dim);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

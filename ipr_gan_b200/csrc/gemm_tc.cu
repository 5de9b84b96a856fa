// gemm_tc.cu -- "tap GEMM": implicit-GEMM convolution / transposed convolution / linear layers on the
// 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, operands staged by TMA).
//
//   acc[m, n] = sum_taps sum_c A[pixel(m) + tap offset, c] * B[n, tap*C + c]
//
// * A tiles are fetched straight from the NHWC bf16 activation tensor by 4-D TMA boxes
//   (channels x width x rows x images); a tap is just a shifted box, and the zero padding of the
//   convolution is TMA's out-of-bounds fill -- no im2col buffer ever exists in HBM.
// * stride-2 convolutions address the input through its four (row, column) parity sub-grids, each
//   described by its own tensor map; k4s2 transposed convolutions run as four output-parity phases of
//   2x2 taps (blockIdx.z), so no multiplication by an inserted zero is ever issued.
// * 128-byte swizzled K-major smem tiles feed tcgen05.mma (M=128, N=BLOCK_N, K=16 per instruction);
//   one elected thread issues, tcgen05.commit releases smem stages / signals the epilogue.
// * warp roles: warps 0..EW-1 epilogue (EW = 4 or 8, chosen per launch), then the TMA producer and the MMA issuer
//   (+ TMEM allocator) on the two highest warp ids.  Epilogue: tcgen05.ld 32 lanes x 32 columns, fused 1/sigma, bias,
//   LeakyReLU / activation-gradient mask / tanh, bf16 pack, per-column sum and sum-of-squares (BatchNorm statistics,
//   bias gradients) accumulated per CTA and warp.
// * persistent: one CTA per SM walks the tile list; the accumulator is double-buffered in TMEM (2 x BLOCK_N columns)
//   so the epilogue of tile i overlaps the TMA/MMA main loop of tile i+1, and the TMA producer never drains between
//   tiles (6-8 smem stages, ~190 KB).
#include "ipr_common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;          // bf16 elements = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;
// EW epilogue warps (template parameter): 4 = one per TMEM lane quarter, 8 = two per quarter that split the tile's
// column chunks.  Measured on B200: 8 is faster when the epilogue does per-element work (bias + LeakyReLU, activation
// mask, column statistics), 4 is faster for plain stores (more registers, fewer warps competing for issue slots).
// The warp scheduler prefers the highest warp id among eligible warps (B300_MICROARCH.md): the single-thread TMA and
// MMA issuers take the two highest ids so that polling / draining epilogue warps never delay them.

struct TgParams {
    int a_n, q_h, q_w, tile_h, tile_imgs, tiles_per_img, m_tiles;
    int a_c, c_chunks, n_taps, n_total, n_phases;
    int8_t tap_map[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t tap_dh[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t tap_dw[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int epi_mode;
    float slope;
    const float *sigma;
    const float *bias;
    const float *scale;
    const __nv_bfloat16 *mask;
    void *out;
    int out_h, out_w, out_c, out_sh, out_sw;
    int8_t out_oh[IPR_TG_MAX_PHASES], out_ow[IPR_TG_MAX_PHASES];
    int n_valid;
    float *stats;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}

// TG = 2 ("tile groups"): the 8 epilogue warps form two groups of four that drain ALTERNATE tiles, each group with its
// own pair of TMEM accumulators (4 in all).  A 128 x 64 tile has a main loop of a few hundred cycles but its read-out
// (tcgen05.ld of 32 KB, then bias / activation / pack / store at ~0.4 instructions per cycle and scheduler) takes
// ~1 900 (per-tile clock64 stamps); with all eight warps on the SAME tile the TMEM read-out and the arithmetic run
// strictly one after the other.  Two groups on different tiles overlap one group's tcgen05.ld with the other's math.
// EPI / ST: the epilogue mode and "column statistics wanted" as COMPILE-TIME values for the hot combinations (-1 = read
// them from the launch parameters).  The generic epilogue executes ~430 instructions per 32-column chunk, most of them
// mode dispatch, register moves for the paths not taken and their address arithmetic (ncu source view, profiles/
// r2_linear_case_generic_epilogue_full.txt); the low-K layers are paced by exactly that instruction stream.
template <int BLOCK_N, int STAGES, bool RES, int EPI_WARPS, int TG = 1, int EPI = -1, int ST = -1>
__global__ void __launch_bounds__(64 + EPI_WARPS * 32, 1)
tapgemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
               const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapA3,
               const __grid_constant__ CUtensorMap mapB, const TgParams p)
{
    constexpr int B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;
    constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
    constexpr uint32_t ACC_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;     // TMEM columns of one accumulator
    constexpr int NBUF = 2 * TG;                                     // accumulators in flight (two per tile group)
    constexpr uint32_t TMEM_COLS = NBUF * ACC_COLS;                  // multi-buffered: epilogue(i) overlaps mainloop(i+1..)
    static_assert(TMEM_COLS <= 512, "TMEM budget");
    static_assert(TG == 1 || (EPI_WARPS == 8 && TG == 2), "tile groups: two groups of four warps");
    constexpr int CH = BLOCK_N >= 32 ? 32 : 16;                      // columns per tcgen05.ld
    constexpr int N_CHUNKS = BLOCK_N / CH;
    constexpr int WARP_TMA = EPI_WARPS, WARP_MMA = EPI_WARPS + 1;
    constexpr int WPG = EPI_WARPS / TG;                              // warps per tile group
    constexpr int EPI_GROUPS = WPG / 4;                              // warps per TMEM lane quarter (within a tile group)
    constexpr int EPI_ACTIVE_PG = N_CHUNKS >= EPI_GROUPS ? WPG : 4;  // warps of a group that have columns to drain
    constexpr int EPI_ACTIVE = TG == 1 ? EPI_ACTIVE_PG : EPI_WARPS;
    constexpr int CH_PER_WARP = N_CHUNKS >= EPI_GROUPS ? N_CHUNKS / EPI_GROUPS : 1;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B needs 1024-byte alignment
    const uint32_t sA = smem_base;
    const uint32_t sB = smem_base + STAGES * A_STAGE_BYTES;
    // RES: the whole weight matrix of this layer (all taps, all phases; one N block) stays resident in shared memory
    // for the lifetime of the persistent CTA, so only A tiles are streamed -- the kernel is paced by TMA row requests
    // (128 A rows + BLOCK_N B rows per k-block), and high-resolution layers have small weights
    const uint32_t b_region = RES ? (uint32_t)(p.n_phases * p.n_taps * p.c_chunks) * B_STAGE_BYTES
                                  : (uint32_t)STAGES * B_STAGE_BYTES;
    const uint32_t bar_full = sB + b_region;                               // STAGES x 8 bytes
    const uint32_t bar_empty = bar_full + STAGES * 8;
    const uint32_t bar_acc_full = bar_empty + STAGES * 8;                 // NBUF x 8
    const uint32_t bar_acc_empty = bar_acc_full + NBUF * 8;               // NBUF x 8
    const uint32_t bar_bres = bar_acc_empty + NBUF * 8;
    const uint32_t tmem_slot = bar_bres + 8;

    // per-warp running column statistics [epilogue warp][sum | sumsq][CH_PER_WARP * CH] floats (after the mbarriers)
    float *stat_sm = reinterpret_cast<float *>(smem_raw + (smem_base - smem_u32(smem_raw)) + STAGES * A_STAGE_BYTES + b_region + 256);
    // per-epilogue-warp staging (2 KB each) for the transposed bf16 store: behind the statistics slots, 16-byte aligned
    uint8_t *stage_sm = reinterpret_cast<uint8_t *>(stat_sm) + TG * 8 * BLOCK_N * 4;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_kb = p.n_taps * p.c_chunks;
    const int n_blks = p.n_total / BLOCK_N;
    const int tiles_per_phase = p.m_tiles * n_blks;
    const int total_tiles = tiles_per_phase * p.n_phases;

    if (warp == WARP_TMA && lane == 0) {
        tma_prefetch_desc(&mapA0); tma_prefetch_desc(&mapB);
        for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < NBUF; b++) { mbar_init(bar_acc_full + 8 * b, 1); mbar_init(bar_acc_empty + 8 * b, EPI_ACTIVE_PG); }
        mbar_init(bar_bres, 1);
        mbar_fence_init();
    }
    if (warp == WARP_MMA) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    // everything above overlapped the previous kernel's tail (PDL); from here on its results are needed
    ipr_pdl_wait();
    ipr_pdl_trigger();

    // persistent: CTA c processes tiles c, c + grid, c + 2 grid, ...   tile -> (phase, m_tile, n_blk), n_blk fastest
    if (warp == WARP_TMA) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t g = 0;                                            // running k-block counter across tiles
            if (RES) {
                mbar_expect_tx(bar_bres, b_region);
                for (int ph = 0; ph < p.n_phases; ph++)
                    for (int kb = 0; kb < num_kb; kb++)
                        tma_load_2d(sB + (ph * num_kb + kb) * B_STAGE_BYTES, &mapB, bar_bres, kb * BLOCK_K, ph * p.n_total);
            }
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int phase = tile / tiles_per_phase, rem = tile - phase * tiles_per_phase;
                const int m_tile = rem / n_blks, n_blk = rem - m_tile * n_blks;
                int img0, h0;
                if (p.tile_imgs == 1) { img0 = m_tile / p.tiles_per_img; h0 = (m_tile - img0 * p.tiles_per_img) * p.tile_h; }
                else { img0 = m_tile * p.tile_imgs; h0 = 0; }
                for (int kb = 0; kb < num_kb; kb++, g++) {
                    const int s = g % STAGES;
                    const uint32_t par = (g / STAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, par ^ 1u);
                    mbar_expect_tx(bar_full + 8 * s, RES ? A_STAGE_BYTES : STAGE_BYTES);
                    const int tap = kb / p.c_chunks, cc = kb - tap * p.c_chunks;
                    const int mi = p.tap_map[phase][tap];
                    const CUtensorMap *ma = mi == 0 ? &mapA0 : (mi == 1 ? &mapA1 : (mi == 2 ? &mapA2 : &mapA3));
                    tma_load_4d(sA + s * A_STAGE_BYTES, ma, bar_full + 8 * s, cc * BLOCK_K, (int)p.tap_dw[phase][tap],
                                h0 + (int)p.tap_dh[phase][tap], img0);
                    if (!RES)
                        tma_load_2d(sB + s * B_STAGE_BYTES, &mapB, bar_full + 8 * s, tap * p.a_c + cc * BLOCK_K,
                                    phase * p.n_total + n_blk * BLOCK_N);
                }
            }
        }
        __syncwarp();
    } else if (warp == WARP_MMA) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BLOCK_M, BLOCK_N);
            uint32_t g = 0, it = 0;
            if (RES) { mbar_wait(bar_bres, 0); tc_fence_after(); }
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, it++) {
                const int phase_m = tile / tiles_per_phase;
                const uint32_t buf = it % NBUF;
                mbar_wait(bar_acc_empty + 8 * buf, ((it / NBUF) & 1u) ^ 1u);    // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t acc = tmem_base + buf * ACC_COLS;
                for (int kb = 0; kb < num_kb; kb++, g++) {
                    const int s = g % STAGES;
                    const uint32_t par = (g / STAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, par);
                    tc_fence_after();
                    const uint64_t da = umma_desc_sw128(sA + s * A_STAGE_BYTES, 0, 1024);
                    const uint64_t db = umma_desc_sw128(RES ? sB + (phase_m * num_kb + kb) * B_STAGE_BYTES
                                                            : sB + s * B_STAGE_BYTES, 0, 1024);
                    // advance 32 bytes (16 bf16) along K inside the swizzle atom: +2 in the (addr >> 4) field
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; k++)
                        umma_bf16(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_commit(bar_empty + 8 * s);           // smem stage reusable once these MMAs retire
                }
                umma_commit(bar_acc_full + 8 * buf);          // accumulator complete
            }
        }
        __syncwarp();
    } else if (warp < EPI_ACTIVE) {
        // ===================== epilogue (warps 0..EPI_ACTIVE-1) =====================
        const int grp = warp / WPG, wg = warp - grp * WPG;   // tile group, warp within the group
        const int q = warp & 3;                           // TMEM lane quarter this warp may access (WPG is a multiple of 4)
        const int c_begin = (wg >> 2) * CH_PER_WARP * CH, c_end = c_begin + CH_PER_WARP * CH;   // this warp's columns
        const int row = q * 32 + lane;                    // row of the 128-row tile
        const int per_img = p.tile_h * p.q_w;
        const int i_img = row / per_img, rem_r = row - i_img * per_img;
        const int i_row = rem_r / p.q_w, i_col = rem_r - i_row * p.q_w;
        const float inv_sigma = p.sigma ? 1.0f / __ldg(p.sigma) : 1.0f;
        // EPI_MASK reads one activation row per thread and chunk.  Those loads miss to L2/HBM (~1 us): issued after
        // the accumulator wait they serialise every chunk behind a full memory round trip.  A walker therefore runs two
        // chunks ahead of the (tile, chunk) sequence and keeps their mask words in a register FIFO, so the loads
        // for the next tile are in flight while this warp still waits for that tile's MMAs.
        constexpr int MQ = CH / 8;                         // uint4 per thread and chunk
        uint4 mq0[MQ], mq1[MQ];
        // Tile coordinates advance by gridDim.x every iteration: (phase, m_tile, n_blk) are stepped incrementally and the
        // pixel of a row is (per-tile uniform part) + (per-thread constant part) -- no division in the tile loop.
        const int t_step = TG * (int)gridDim.x;           // a group's next tile
        const int g_q = t_step / n_blks, g_r = t_step - g_q * n_blks;
        const int tpi_shift = (p.tiles_per_img & (p.tiles_per_img - 1)) == 0 ? 31 - __clz(p.tiles_per_img) : -1;
        const int thr_pix = (i_img * p.out_h + i_row * p.out_sh) * p.out_w + i_col * p.out_sw;
        struct TileIt { int tile, phase, m_tile, n_blk; };
        auto it_init = [&](TileIt &t) {
            t.tile = blockIdx.x + grp * gridDim.x;
            t.phase = t.tile / tiles_per_phase;
            const int rm = t.tile - t.phase * tiles_per_phase;
            t.m_tile = rm / n_blks; t.n_blk = rm - t.m_tile * n_blks;
        };
        auto it_next = [&](TileIt &t) {
            t.tile += t_step; t.n_blk += g_r; t.m_tile += g_q;
            if (t.n_blk >= n_blks) { t.n_blk -= n_blks; t.m_tile++; }
            while (t.m_tile >= p.m_tiles) { t.m_tile -= p.m_tiles; t.phase++; }
        };
        // -> pixel index of this thread's row in tile t, or -1 when the row is outside the tensor
        auto row_pix = [&](const TileIt &t) -> long long {
            int im0, hh0;
            if (p.tile_imgs == 1) {
                im0 = tpi_shift >= 0 ? (t.m_tile >> tpi_shift) : t.m_tile / p.tiles_per_img;
                hh0 = (t.m_tile - im0 * p.tiles_per_img) * p.tile_h;
            } else { im0 = t.m_tile * p.tile_imgs; hh0 = 0; }
            if (im0 + i_img >= p.a_n) return -1;
            return (long long)(im0 * p.out_h + hh0 * p.out_sh + p.out_oh[t.phase]) * p.out_w + p.out_ow[t.phase] + thr_pix;
        };
        TileIt wt;                                         // the walker's position
        int w_c0 = c_begin;
        const __nv_bfloat16 *w_base = nullptr;             // mask row of the walker's tile, nullptr when masked out
        auto w_locate = [&]() {
            w_base = nullptr;
            if (wt.tile >= total_tiles) return;
            const long long px = row_pix(wt);
            if (px >= 0) w_base = p.mask + px * p.out_c + wt.n_blk * BLOCK_N;
        };
        auto w_fetch = [&](uint4 (&dst)[MQ]) {
            if (w_base) {
#pragma unroll
                for (int g = 0; g < MQ; g++) dst[g] = __ldg(reinterpret_cast<const uint4 *>(w_base + w_c0) + g);
            }
            w_c0 += CH;
            if (w_c0 >= c_end) {
                w_c0 = c_begin;
                it_next(wt);
                w_locate();
            }
        };
        const int epi_mode = EPI >= 0 ? EPI : p.epi_mode;
        const bool has_stats = ST >= 0 ? (ST == 1) : (p.stats != nullptr);
        const bool masked = epi_mode == IPR_EPI_MASK;
        const bool bias_vec = p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15u) == 0;
        const bool want_sq = epi_mode != IPR_EPI_MASK;   // masked data gradients only need column sums (bias grad)
        // column statistics: with a single N block every tile of this CTA covers the same columns, so each warp keeps
        // running sums in its own shared-memory slots (no barrier, fixed order) and writes ONE row at the end:
        // stats rows = 4 * CTAs instead of 4 * tiles.
        const bool cta_stats = has_stats && n_blks == 1;
        float *my_stat = stat_sm + warp * 2 * CH_PER_WARP * CH;
        if (cta_stats) {
            for (int c = lane; c < 2 * CH_PER_WARP * CH; c += 32) my_stat[c] = 0.0f;
            __syncwarp();
        }
        if (masked) { it_init(wt); w_locate(); w_fetch(mq0); w_fetch(mq1); }
        uint32_t it = grp;                                // position in the CTA's tile sequence: grp, grp + TG, ...
        TileIt ct;
        it_init(ct);
        for (; ct.tile < total_tiles; it_next(ct), it += TG) {
            const int phase = ct.phase, m_tile = ct.m_tile, n_blk = ct.n_blk;
            const uint32_t buf = it % NBUF;
            // bias (and eval-BatchNorm scale) of the tile's FIRST chunk: fetched before the accumulator wait, so the loads
            // are in flight while the main loop of this tile still runs (they used to stall the first FADDs)
            constexpr bool PRE = EPI == IPR_EPI_BIAS_LRELU;     // only where the mode is known at compile time (registers)
            float4 bpre[PRE ? CH / 4 : 1], spre[PRE ? CH / 4 : 1];
            const bool pre_bias = PRE && bias_vec;
            if (pre_bias) {
#pragma unroll
                for (int j4 = 0; j4 < (PRE ? CH / 4 : 1); j4++) bpre[j4] = __ldg(reinterpret_cast<const float4 *>(p.bias + n_blk * BLOCK_N + c_begin) + j4);
                if (p.scale) {
#pragma unroll
                    for (int j4 = 0; j4 < (PRE ? CH / 4 : 1); j4++) spre[j4] = __ldg(reinterpret_cast<const float4 *>(p.scale + n_blk * BLOCK_N + c_begin) + j4);
                }
            }
            mbar_wait_backoff(bar_acc_full + 8 * buf, (it / NBUF) & 1u);
            tc_fence_after();
            const long long pix_s = row_pix(ct);
            const bool valid = pix_s >= 0;
            const size_t pix = (size_t)pix_s;
#pragma unroll 1
            for (int c0 = c_begin; c0 < c_end; c0 += CH) {
                uint32_t raw[32];
                uint4 mcur[MQ];
                if (masked) {                              // pop this chunk's mask words, refill the FIFO two chunks ahead
#pragma unroll
                    for (int g = 0; g < MQ; g++) { mcur[g] = mq0[g]; mq0[g] = mq1[g]; }
                    w_fetch(mq1);
                }
                const uint32_t taddr = tmem_base + buf * ACC_COLS + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
                if constexpr (CH == 32) tmem_ld_32x32(taddr, raw);
                else tmem_ld_32x16(taddr, *reinterpret_cast<uint32_t(*)[16]>(&raw));
                tmem_ld_wait();
                if (c0 + CH >= c_end) {
                    // last chunk is in registers: hand the accumulator back to the MMA warp before the slow part
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acc_empty + 8 * buf);
                }
                const int n0 = n_blk * BLOCK_N + c0;
                float v[CH];
#pragma unroll
                for (int j = 0; j < CH; j++) v[j] = __uint_as_float(raw[j]);
                if (p.sigma) {                             // (uniform) spectral norm: W / sigma applied to the accumulator
#pragma unroll
                    for (int j = 0; j < CH; j++) v[j] *= inv_sigma;
                }

                if (epi_mode == IPR_EPI_BIAS_LRELU) {
                    const bool first = pre_bias && c0 == c_begin;
                    if (p.scale) {                         // eval-mode BatchNorm folded into the layer: per-column factor
#pragma unroll
                        for (int j4 = 0; j4 < CH / 4; j4++) {
                            const float4 s4 = first ? spre[PRE ? j4 : 0] : __ldg(reinterpret_cast<const float4 *>(p.scale + n0) + j4);
                            v[4 * j4 + 0] *= s4.x; v[4 * j4 + 1] *= s4.y; v[4 * j4 + 2] *= s4.z; v[4 * j4 + 3] *= s4.w;
                        }
                    }
                    if (bias_vec) {                        // 8 broadcast 128-bit loads instead of 32 scalar ones
#pragma unroll
                        for (int j4 = 0; j4 < CH / 4; j4++) {
                            const float4 b4 = first ? bpre[PRE ? j4 : 0] : __ldg(reinterpret_cast<const float4 *>(p.bias + n0) + j4);
                            v[4 * j4 + 0] += b4.x; v[4 * j4 + 1] += b4.y; v[4 * j4 + 2] += b4.z; v[4 * j4 + 3] += b4.w;
                        }
                    } else if (p.bias) {
#pragma unroll
                        for (int j = 0; j < CH; j++) v[j] += __ldg(p.bias + n0 + j);
                    }
#pragma unroll
                    for (int j = 0; j < CH; j++) v[j] = v[j] > 0.0f ? v[j] : v[j] * p.slope;
                } else if (epi_mode == IPR_EPI_MASK) {
                    if (valid) {
#pragma unroll
                        for (int gq = 0; gq < CH / 8; gq++) {
                            const uint4 mv = mcur[gq];
                            const uint32_t w[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
                            for (int h = 0; h < 4; h++) {
                                const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162 *>(&w[h]);
                                const float2 f2 = __bfloat1622float2(b2);
                                v[gq * 8 + 2 * h] *= f2.x > 0.0f ? 1.0f : p.slope;
                                v[gq * 8 + 2 * h + 1] *= f2.y > 0.0f ? 1.0f : p.slope;
                            }
                        }
                    }
                } else if (epi_mode == IPR_EPI_TANH_NCHW) {
#pragma unroll
                    for (int j = 0; j < CH; j++) v[j] = tanhf(v[j]);
                }

                if (has_stats) {
                    // per-column sum / sum of squares over this warp's 32 rows: 31-step transposing butterfly
                    float s1[CH], s2[CH];
#pragma unroll
                    for (int j = 0; j < CH; j++) { const float t = valid ? v[j] : 0.0f; s1[j] = t; s2[j] = t * t; }
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
                        const bool up = (lane & off) != 0;
                        if (off < CH) {
#pragma unroll
                            for (int i = 0; i < off; i++) {
                                const float snd1 = up ? s1[i] : s1[i + off], kp1 = up ? s1[i + off] : s1[i];
                                s1[i] = kp1 + __shfl_xor_sync(0xffffffffu, snd1, off);
                            }
                            if (want_sq) {
#pragma unroll
                                for (int i = 0; i < off; i++) {
                                    const float snd2 = up ? s2[i] : s2[i + off], kp2 = up ? s2[i + off] : s2[i];
                                    s2[i] = kp2 + __shfl_xor_sync(0xffffffffu, snd2, off);
                                }
                            }
                        } else {   // CH == 16 and off == 16: plain pairwise sum, both halves keep all 16 columns
#pragma unroll
                            for (int i = 0; i < CH; i++) {
                                s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], off);
                                if (want_sq) s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], off);
                            }
                        }
                    }
                    if (lane < CH && m_tile < p.m_tiles) { // lane L now holds column (L mod CH)
                        if (cta_stats) {                   // one N block: keep a running sum per CTA and warp (own slots only)
                            my_stat[c0 - c_begin + lane] += s1[0];
                            if (want_sq) my_stat[CH_PER_WARP * CH + c0 - c_begin + lane] += s2[0];
                        } else {                           // several N blocks: one stats row per tile and warp
                            float *dst = p.stats + (((size_t)phase * p.m_tiles + m_tile) * 4 + q) * 2 * p.n_total + n0 + lane;
                            dst[0] = s1[0];
                            dst[p.n_total] = want_sq ? s2[0] : 0.0f;
                        }
                    }
                }

                if (epi_mode == IPR_EPI_TANH_NCHW || epi_mode == IPR_EPI_LINEAR_NCHW) {
                    if (!valid) continue;
                    const size_t hw = (size_t)p.out_h * p.out_w, img = pix / hw, inner = pix - img * hw;
                    float *o = reinterpret_cast<float *>(p.out) + img * p.out_c * hw + inner;
#pragma unroll
                    for (int j = 0; j < CH; j++) {
                        const int n = n0 + j;
                        if (n < p.n_valid) o[(size_t)n * hw] = v[j];
                    }
                } else if (epi_mode == IPR_EPI_LINEAR_F32) {
                    if (!valid) continue;
                    float *o = reinterpret_cast<float *>(p.out) + pix * p.out_c + n0;
                    if (n0 + CH <= p.n_valid && (p.out_c & 3) == 0) {
#pragma unroll
                        for (int j4 = 0; j4 < CH / 4; j4++)
                            reinterpret_cast<float4 *>(o)[j4] = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < CH; j++) if (n0 + j < p.n_valid) o[j] = v[j];
                    }
                } else {
                    __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(p.out) + pix * p.out_c + n0;
                    if (n0 + CH <= p.n_valid) {            // (warp-uniform)
                        uint4 pk[CH / 8];
#pragma unroll
                        for (int gq = 0; gq < CH / 8; gq++) {
                            pk[gq].x = pack_bf16x2(v[gq * 8 + 0], v[gq * 8 + 1]); pk[gq].y = pack_bf16x2(v[gq * 8 + 2], v[gq * 8 + 3]);
                            pk[gq].z = pack_bf16x2(v[gq * 8 + 4], v[gq * 8 + 5]); pk[gq].w = pack_bf16x2(v[gq * 8 + 6], v[gq * 8 + 7]);
                        }
                        if constexpr (CH == 32) {
                            // Every thread owns one output row (64 bytes of it per chunk).  Storing it as four 16-byte
                            // pieces makes each store instruction touch 32 different lines; transposed through a 2 KB
                            // per-warp staging area (XOR-swizzled 16-byte slots: conflict-free both ways) one
                            // instruction writes 8 rows x 64 contiguous bytes: a quarter of the line touches.
                            // Measured: neutral for the step (patch GEMM 48.0 -> 46.6 us) -- disabling the stores
                            // altogether changes nothing either; the epilogue is paced by its instruction stream, see
                            // the EPI / ST template parameters.
                            uint8_t *stg = stage_sm + warp * 2048;
#pragma unroll
                            for (int gq = 0; gq < 4; gq++)
                                *reinterpret_cast<uint4 *>(stg + lane * 64 + ((gq ^ ((lane >> 1) & 3)) << 4)) = pk[gq];
                            __syncwarp();
                            const unsigned long long optr = valid ? reinterpret_cast<unsigned long long>(o) : 0ull;
#pragma unroll
                            for (int jj = 0; jj < 4; jj++) {
                                const int R = 8 * jj + (lane >> 2), pz = lane & 3;
                                const uint4 val = *reinterpret_cast<const uint4 *>(stg + R * 64 + ((pz ^ ((R >> 1) & 3)) << 4));
                                const unsigned long long rp = __shfl_sync(0xffffffffu, optr, R);
                                if (rp) *reinterpret_cast<uint4 *>(rp + pz * 16) = val;
                            }
                            __syncwarp();
                        } else {
                            if (valid) {
#pragma unroll
                                for (int gq = 0; gq < CH / 8; gq++) reinterpret_cast<uint4 *>(o)[gq] = pk[gq];
                            }
                        }
                    } else if (valid) {
#pragma unroll
                        for (int j = 0; j < CH; j++) if (n0 + j < p.n_valid) o[j] = __float2bfloat16(v[j]);
                    }
                }
            }
        }
        if (cta_stats) {
            __syncwarp();
            float *dst = p.stats + (((size_t)blockIdx.x * TG + grp) * 4 + q) * 2 * p.n_total + c_begin;
            for (int c = lane; c < CH_PER_WARP * CH; c += 32) {
                dst[c] = my_stat[c];
                dst[p.n_total + c] = want_sq ? my_stat[CH_PER_WARP * CH + c] : 0.0f;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WARP_MMA) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int BLOCK_N, int STAGES, bool RES, int EW, int TG = 1, int EPI = -1, int ST = -1>
int launch_ew(const CUtensorMap *ma, const CUtensorMap &mb, const TgParams &p, dim3 grid, cudaStream_t st)
{
    const size_t b_region = RES ? (size_t)p.n_phases * p.n_taps * p.c_chunks * BLOCK_N * BLOCK_K * 2
                                : (size_t)STAGES * BLOCK_N * BLOCK_K * 2;
    const size_t smem = (size_t)STAGES * A_STAGE_BYTES + b_region + 256 + TG * 8 * BLOCK_N * 4 + 8 * 2048 + 1024 + 64;
    if (smem > (size_t)227 * 1024) return IPR_E_UNSUPPORTED;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(tapgemm_kernel<BLOCK_N, STAGES, RES, EW, TG, EPI, ST>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const int total = (int)(grid.x * grid.y * grid.z);
    const int ctas = total < ipr_sm_count() ? total : ipr_sm_count();       // persistent: one CTA per SM
    IPR_LAUNCH_PDL((tapgemm_kernel<BLOCK_N, STAGES, RES, EW, TG, EPI, ST>), ctas, 64 + EW * 32, smem, st, ma[0], ma[1], ma[2], ma[3], mb, p);
    IPR_LAUNCH_CHECK();
    return IPR_OK;
}

// The kernel variant of one launch, chosen from the descriptor and the tile count alone: ipr_tapgemm_bf16 launches it
// and ipr_tapgemm_stats_rows sizes the statistics from it.  The smem stages follow from BLOCK_N and RES (see launch).
struct Variant {
    bool resident;        // RES
    int epi_warps;        // EW
    int tile_groups;      // TG
    int epi, stats;       // EPI, ST: -1 = the generic epilogue, which reads them from the launch parameters
};

Variant pick_variant(const ipr_tapgemm_t *d, int m_tiles, bool stats)
{
    const int num_kb = d->n_taps * ((d->a_c + BLOCK_K - 1) / BLOCK_K);
    const long long tiles = (long long)m_tiles * (d->n_total / d->block_n) * d->n_phases;
    const long long sms = ipr_sm_count();
    Variant v;
    // weights resident in shared memory: one N block, everything (all phases x taps) fits beside 4 A stages, and every
    // CTA has at least two tiles to amortise the one-off weight load over
    const size_t b_all = (size_t)d->n_phases * num_kb * d->block_n * BLOCK_K * 2;
    v.resident = d->block_n <= 128 && d->n_total == d->block_n && b_all <= 132 * 1024 && tiles >= 2 * sms;
    const bool heavy = d->epi_mode == IPR_EPI_BIAS_LRELU || d->epi_mode == IPR_EPI_MASK || stats;
    v.epi_warps = heavy ? 8 : 4;
    v.tile_groups = 1;
    v.epi = v.stats = -1;
    if (!heavy) {
        if (d->epi_mode == IPR_EPI_LINEAR || d->epi_mode == IPR_EPI_LINEAR_F32) { v.epi = d->epi_mode; v.stats = 0; }
        return v;
    }
    if (d->epi_mode == IPR_EPI_BIAS_LRELU && !stats) { v.epi = IPR_EPI_BIAS_LRELU; v.stats = 0; }
    else if (d->epi_mode == IPR_EPI_MASK) { v.epi = IPR_EPI_MASK; v.stats = stats ? 1 : 0; }
    else if (d->epi_mode == IPR_EPI_LINEAR && stats) { v.epi = IPR_EPI_LINEAR; v.stats = 1; }
    // Two tile groups need every CTA to have at least four tiles.  Measured (batch 512): the single-k-block patch GEMM
    // gains (32->64 bias+LeakyReLU 46.3 -> 40.6 us); layers with a real main loop do not (convT4s2 128->64 79 -> 82 us,
    // conv3_dgrad 128->64 44.5 -> 46.6 us), so the groups are used for main loops of at most two k-blocks.  Of the
    // specialised epilogues only bias + LeakyReLU has a tile-group version.
    if ((v.epi == -1 || v.epi == IPR_EPI_BIAS_LRELU) && d->block_n >= 32 && d->block_n <= 128 && tiles >= 4 * sms &&
        num_kb <= 2)
        v.tile_groups = 2;
    return v;
}

template <int BLOCK_N, bool RES>
int launch(const Variant &v, const CUtensorMap *ma, const CUtensorMap &mb, const TgParams &p, dim3 grid, cudaStream_t st)
{
    // smem stages: 4 A stages beside a resident weight matrix, otherwise as many A + B stages as fit in ~190 KB
    constexpr int S = RES ? 4 : (BLOCK_N <= 64 ? 8 : (BLOCK_N == 128 ? 6 : 4));
    if (v.epi_warps == 4) {
        if (v.epi == IPR_EPI_LINEAR) return launch_ew<BLOCK_N, S, RES, 4, 1, IPR_EPI_LINEAR, 0>(ma, mb, p, grid, st);
        if (v.epi == IPR_EPI_LINEAR_F32) return launch_ew<BLOCK_N, S, RES, 4, 1, IPR_EPI_LINEAR_F32, 0>(ma, mb, p, grid, st);
        return launch_ew<BLOCK_N, S, RES, 4>(ma, mb, p, grid, st);
    }
    if constexpr (BLOCK_N >= 32 && BLOCK_N <= 128) {
        if (v.tile_groups == 2)
            return v.epi == IPR_EPI_BIAS_LRELU ? launch_ew<BLOCK_N, S, RES, 8, 2, IPR_EPI_BIAS_LRELU, 0>(ma, mb, p, grid, st)
                                               : launch_ew<BLOCK_N, S, RES, 8, 2>(ma, mb, p, grid, st);
    }
    if (v.epi == IPR_EPI_BIAS_LRELU) return launch_ew<BLOCK_N, S, RES, 8, 1, IPR_EPI_BIAS_LRELU, 0>(ma, mb, p, grid, st);
    if (v.epi == IPR_EPI_MASK)
        return v.stats ? launch_ew<BLOCK_N, S, RES, 8, 1, IPR_EPI_MASK, 1>(ma, mb, p, grid, st)
                       : launch_ew<BLOCK_N, S, RES, 8, 1, IPR_EPI_MASK, 0>(ma, mb, p, grid, st);
    if (v.epi == IPR_EPI_LINEAR) return launch_ew<BLOCK_N, S, RES, 8, 1, IPR_EPI_LINEAR, 1>(ma, mb, p, grid, st);
    return launch_ew<BLOCK_N, S, RES, 8>(ma, mb, p, grid, st);
}

int tile_geometry(const ipr_tapgemm_t *d, TgParams &p)
{
    const int per_img = d->q_h * d->q_w;
    IPR_REQUIRE(per_img > 0 && d->q_w <= 128, IPR_E_UNSUPPORTED);
    if (per_img >= BLOCK_M) {
        IPR_REQUIRE(BLOCK_M % d->q_w == 0, IPR_E_UNSUPPORTED);
        p.tile_h = BLOCK_M / d->q_w;
        IPR_REQUIRE(d->q_h % p.tile_h == 0, IPR_E_UNSUPPORTED);
        p.tile_imgs = 1;
        p.tiles_per_img = d->q_h / p.tile_h;
        p.m_tiles = d->a_n * p.tiles_per_img;
    } else {
        IPR_REQUIRE(BLOCK_M % per_img == 0, IPR_E_UNSUPPORTED);
        p.tile_h = d->q_h;
        p.tile_imgs = BLOCK_M / per_img;
        p.tiles_per_img = 1;
        p.m_tiles = (d->a_n + p.tile_imgs - 1) / p.tile_imgs;
    }
    return IPR_OK;
}

}  // namespace

extern "C" int ipr_tapgemm_stats_rows(const ipr_tapgemm_t *d)
{
    if (!d) return IPR_E_NULL;
    TgParams p;
    int rc = tile_geometry(d, p);
    if (rc != IPR_OK) return rc;
    IPR_REQUIRE(d->block_n > 0 && d->n_total % d->block_n == 0 && d->n_phases >= 1, IPR_E_SHAPE);
    const long long tiles = (long long)p.m_tiles * d->n_phases;
    if (d->n_total != d->block_n) return (int)(4 * tiles);          // 4 rows per tile
    // one N block: 4 rows per CTA and tile group
    const long long ctas = tiles < ipr_sm_count() ? tiles : ipr_sm_count();
    return (int)(4 * pick_variant(d, p.m_tiles, true).tile_groups * ctas);
}

extern "C" int ipr_tapgemm_m_tiles(const ipr_tapgemm_t *d)
{
    if (!d) return IPR_E_NULL;
    TgParams p;
    int rc = tile_geometry(d, p);
    return rc != IPR_OK ? rc : p.m_tiles;
}

extern "C" int ipr_tapgemm_bf16(const ipr_tapgemm_t *d, ipr_stream_t stream)
{
    IPR_REQUIRE(d, IPR_E_NULL);
    IPR_REQUIRE(d->a && d->b && d->out, IPR_E_NULL);
    IPR_REQUIRE(d->a_n > 0 && d->a_h > 0 && d->a_w > 0 && d->a_c > 0, IPR_E_SHAPE);
    // channels are consumed in 64-wide boxes; a single-tap layer may store fewer (a multiple of 8): the rest of the box
    // is TMA out-of-bounds zero fill on both operands (the 27-column patch matrices are stored 32 wide)
    IPR_REQUIRE(d->a_c % BLOCK_K == 0 || (d->n_taps == 1 && d->a_c % 8 == 0), IPR_E_UNSUPPORTED);
    IPR_REQUIRE(d->n_taps >= 1 && d->n_taps <= IPR_TG_MAX_TAPS && d->n_phases >= 1 && d->n_phases <= IPR_TG_MAX_PHASES,
                IPR_E_SHAPE);
    IPR_REQUIRE(d->block_n == 16 || d->block_n == 32 || d->block_n == 64 || d->block_n == 128 || d->block_n == 256,
                IPR_E_UNSUPPORTED);
    IPR_REQUIRE(d->n_total > 0 && d->n_total % d->block_n == 0, IPR_E_SHAPE);
    IPR_REQUIRE(ipr_aligned16(d->a) && ipr_aligned16(d->b) && ipr_aligned16(d->out), IPR_E_ALIGN);
    IPR_REQUIRE(d->epi_mode >= 0 && d->epi_mode <= 5, IPR_E_SHAPE);
    IPR_REQUIRE(d->epi_mode != IPR_EPI_MASK || (d->mask && ipr_aligned16(d->mask)), IPR_E_NULL);
    if (d->epi_mode == IPR_EPI_LINEAR || d->epi_mode == IPR_EPI_BIAS_LRELU || d->epi_mode == IPR_EPI_MASK)
        IPR_REQUIRE(d->out_c % 8 == 0, IPR_E_ALIGN);
    if (d->a_parity) IPR_REQUIRE(d->a_h % 2 == 0 && d->a_w % 2 == 0 && d->a_c % 8 == 0, IPR_E_UNSUPPORTED);

    TgParams p;
    int rc = tile_geometry(d, p);
    if (rc != IPR_OK) return rc;
    p.a_n = d->a_n; p.q_h = d->q_h; p.q_w = d->q_w;
    p.a_c = d->a_c; p.c_chunks = (d->a_c + BLOCK_K - 1) / BLOCK_K; p.n_taps = d->n_taps; p.n_total = d->n_total;
    p.n_phases = d->n_phases;
    for (int ph = 0; ph < IPR_TG_MAX_PHASES; ph++) {
        for (int t = 0; t < IPR_TG_MAX_TAPS; t++) {
            p.tap_map[ph][t] = d->tap_map[ph][t]; p.tap_dh[ph][t] = d->tap_dh[ph][t]; p.tap_dw[ph][t] = d->tap_dw[ph][t];
            if (ph < d->n_phases && t < d->n_taps)
                IPR_REQUIRE(d->tap_map[ph][t] >= 0 && d->tap_map[ph][t] < (d->a_parity ? 4 : 1), IPR_E_SHAPE);
        }
        p.out_oh[ph] = d->out_oh[ph]; p.out_ow[ph] = d->out_ow[ph];
    }
    p.epi_mode = d->epi_mode; p.slope = d->slope; p.sigma = d->sigma; p.bias = d->bias; p.scale = d->scale;
    IPR_REQUIRE(!d->scale || (d->epi_mode == IPR_EPI_BIAS_LRELU && ipr_aligned16(d->scale)), IPR_E_ALIGN);
    p.mask = (const __nv_bfloat16 *)d->mask; p.out = d->out;
    p.out_h = d->out_h; p.out_w = d->out_w; p.out_c = d->out_c; p.out_sh = d->out_sh; p.out_sw = d->out_sw;
    p.n_valid = d->n_valid > 0 ? d->n_valid : d->n_total; p.stats = d->stats;

    // ---- tensor maps (host-encoded, passed by value as kernel parameters: graph-capturable)
    CUtensorMap ma[4], mb;
    const uint64_t C = d->a_c, W = d->a_w, H = d->a_h, N = d->a_n;
    const uint32_t box[4] = {(uint32_t)BLOCK_K, (uint32_t)d->q_w, (uint32_t)p.tile_h, (uint32_t)p.tile_imgs};
    if (!d->a_parity) {
        IPR_REQUIRE(d->q_w == d->a_w && d->q_h == d->a_h, IPR_E_SHAPE);
        const uint64_t dims[4] = {C, W, H, N};
        const uint64_t str[3] = {C * 2, W * C * 2, H * W * C * 2};
        rc = make_tmap_bf16(&ma[0], d->a, 4, dims, str, box);
        if (rc) return rc;
        ma[1] = ma[2] = ma[3] = ma[0];
    } else {
        IPR_REQUIRE(d->q_w == d->a_w / 2 && d->q_h == d->a_h / 2, IPR_E_SHAPE);
        const uint64_t dims[4] = {C, W / 2, H / 2, N};
        const uint64_t str[3] = {2 * C * 2, 2 * W * C * 2, H * W * C * 2};
        for (int ph = 0; ph < 2; ph++)
            for (int pw = 0; pw < 2; pw++) {
                const char *base = (const char *)d->a + ((size_t)ph * W + pw) * C * 2;
                rc = make_tmap_bf16(&ma[ph * 2 + pw], base, 4, dims, str, box);
                if (rc) return rc;
            }
    }
    {
        const uint64_t K = (uint64_t)d->n_taps * C;
        const uint64_t dims[2] = {K, (uint64_t)d->n_phases * d->n_total};
        const uint64_t str[1] = {K * 2};
        const uint32_t bbox[2] = {(uint32_t)BLOCK_K, (uint32_t)d->block_n};
        rc = make_tmap_bf16(&mb, d->b, 2, dims, str, bbox);
        if (rc) return rc;
    }
    dim3 grid((unsigned)p.m_tiles, (unsigned)(d->n_total / d->block_n), (unsigned)d->n_phases);
    cudaStream_t st = ipr_cu(stream);
    const Variant v = pick_variant(d, p.m_tiles, d->stats != nullptr);
    switch (d->block_n) {
        case 16:  return v.resident ? launch<16, true>(v, ma, mb, p, grid, st) : launch<16, false>(v, ma, mb, p, grid, st);
        case 32:  return v.resident ? launch<32, true>(v, ma, mb, p, grid, st) : launch<32, false>(v, ma, mb, p, grid, st);
        case 64:  return v.resident ? launch<64, true>(v, ma, mb, p, grid, st) : launch<64, false>(v, ma, mb, p, grid, st);
        case 128: return v.resident ? launch<128, true>(v, ma, mb, p, grid, st) : launch<128, false>(v, ma, mb, p, grid, st);
        default:  return launch<256, false>(v, ma, mb, p, grid, st);
    }
}

// conv3d weight gradient on tcgen05 (algo 2, pass 2):  dw[co, ci, tap] = sum_voxels dy[v, co] * x[src(v, tap), ci].
//
// GEMM view: for each tap, D[M = co][N = ci] accumulates over K = voxels.  Both operands are "MN-major" in shared memory: the TMA
// drops a line of voxels as [voxel rows][channels] tiles, which is exactly the transposed (MN-major) canonical layout of tcgen05.
//
// Two B200-specific tricks (both verified by tools/tc_probe on hardware, profiles/r01_tc_probe*.txt):
//  * all kw taps of a (kd, kh) pair in ONE MMA: the x operand is a halo line of (voxels + kw - 1) rows; its N index runs over kw
//    row-shifted windows of that single buffer by setting the descriptor's leading-dimension byte offset to ONE ROW, N = kw * chunk;
//  * split-bf16 in 2 MMAs instead of 3: the dy operand's M = 128 rows are [dy_hi | dy_lo] (the two bf16 planes sit in adjacent
//    shared-memory chunks), so one MMA against x_hi and one against x_lo produce hi*hi + hi*lo in TMEM lanes [0, co) and
//    lo*hi + lo*lo in lanes [co_p, co_p + co); the epilogue adds both halves into dw.  (Used when 2 * co_p <= 128; otherwise 3 MMAs.)
//
// Work decomposition: a CTA owns up to CB "column blocks" (kd, kh, ci-chunk) whose accumulators fill its 512 TMEM columns, and a
// strided share of the output lines; it streams dy lines + x halo lines through a 2-stage TMA ring and finally dumps its accumulators
// (real channels only, no padding lanes / columns) to its slot of a partial buffer; wgrad_reduce_kernel adds the slots in a fixed order
// (deterministic; the first version's fp32 red.global.add cost more than the MMAs).  The number of lines per CTA is bounded by the
// accumulator chain limit (kMaxChain MMAs, see wg_splits): the tensor core's fp32 accumulation is not round-to-nearest.
#include "conv3d_common.cuh"
#include "tc_common.cuh"
#include <cstdlib>

namespace mdt {
using namespace tc;

__global__ void split_rows_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, long long rows, int C, int Cp, int planes, int inter_w,
                                  const float *__restrict__ relu_of, float *__restrict__ masked_out, float *__restrict__ colsum);
int conv_tc_kpad(int channels);        // channels of the global split layout (multiple of 16)
int conv_tc_kpad_smem(int channels);   // channels staged in shared memory (TMA zero-fills past the global extent)
int conv_tc_run(const ConvGeom &g, int pass, const float *src, const float *w, const float *bias, const float *residual, float *dst, int relu,
                int precision, void *ws, size_t ws_bytes, cudaStream_t st, const __nv_bfloat16 *presplit, __nv_bfloat16 *out_split);
size_t conv_tc_workspace_bytes(const ConvGeom &g, int pass, int precision);

struct TcWgradParams {
    int NB, OD, OH, OW, D, H, W;
    int KD, KH, KW, sd, sh, pd, ph, pw;
    int cin, cout, T;
    int seg, segs, ksteps;           // voxels per work unit (<= 128), units per line, K16 steps
    int swy, chunky, nmc, co_p;      // dy: swizzle bytes, channels per chunk, chunks in one M tile, padded cout
    int mtrick;
    int swx, chunkx, nxc;            // x: swizzle bytes, channels per chunk, number of ci chunks
    int ncb_total, CB, groups, splits;
    int planes, stages, tmem_cols, slot_cols;
    int y_chunk_bytes, y_plane_bytes, x_plane_bytes, x_buf_bytes, stage_bytes;
    int y_tx_bytes, x_tx_bytes;      // bytes one TMA box delivers
    int y_stride, x_base, x_stride;  // shared-memory placement: dy of stage s at s * y_stride, x at x_base + s * x_stride
    long long units;                 // NB * OD * OH * segs
    float *partial;                  // [split][group][mtile][128 lanes][512 cols] fp32 accumulator dumps (reduced by wgrad_reduce_kernel)
    int mtiles;
    int skip;                        // diagnostics (MDT_WG_SKIP): 1 = no MMAs (TMA pipeline alone), 2 = no TMA loads (MMAs alone); results are garbage
};

constexpr int kWgThreads = 192;
constexpr int kWgMaxStages = 2;

__device__ __forceinline__ void wg_decode_cb(const TcWgradParams &p, int cb, int &kd, int &kh, int &xc) {
    xc = cb % p.nxc;
    const int pair = cb / p.nxc;
    kh = pair % p.KH;
    kd = pair / p.KH;
}

__global__ void __launch_bounds__(kWgThreads, 1)
conv_tc_wgrad_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmX, const TcWgradParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full[kWgMaxStages], empty[kWgMaxStages], accum_full;
    __shared__ uint32_t tmem_base_s, s_started;
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = blockIdx.x % p.groups, split = blockIdx.x / p.groups;
    const int mt = blockIdx.y;                       // M tile (128 rows of co) when co_p > 128
    const int cb0 = group * p.CB;
    const int ncb = min(p.CB, p.ncb_total - cb0);
    const int ncols = p.KW * p.chunkx;               // accumulator columns per column block

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(&accum_full, 1);
        s_started = 0;
        fence_barrier_init();
        prefetch_tmap(&tmY);
        prefetch_tmap(&tmX);
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    // unit -> (n, od, oh, seg)
    auto decode_unit = [&](long long u, int &n, int &od, int &oh, int &ow0) {
        const int sg = (int)(u % p.segs); u /= p.segs;
        oh = (int)(u % p.OH); u /= p.OH;
        od = (int)(u % p.OD);
        n = (int)(u / p.OD);
        ow0 = sg * p.seg;
    };

    if (warp == 0) {
        if (elect_one()) {
            int it = 0;
            for (long long u = split; u < p.units; u += p.splits, ++it) {
                int n, od, oh, ow0;
                decode_unit(u, n, od, oh, ow0);
                const int s = it % p.stages;
                mbar_wait(&empty[s], ((it / p.stages) & 1) ^ 1);
                uint8_t *st = smem + (size_t)s * p.y_stride;
                // which column blocks have their source line inside the image
                uint32_t bytes = p.planes * p.nmc * p.y_tx_bytes;
                for (int b = 0; b < ncb; ++b) {
                    int kd, kh, xc;
                    wg_decode_cb(p, cb0 + b, kd, kh, xc);
                    const int d = od * p.sd - p.pd + kd, h = oh * p.sh - p.ph + kh;
                    if (d >= 0 && d < p.D && h >= 0 && h < p.H) bytes += p.planes * p.x_tx_bytes;
                }
                if (p.skip == 2) { mbar_arrive(&full[s]); continue; }
                mbar_arrive_expect_tx(&full[s], bytes);
                for (int pl = 0; pl < p.planes; ++pl)
                    for (int mc = 0; mc < p.nmc; ++mc)
                        tma_load_5d(st + (size_t)pl * p.y_plane_bytes + (size_t)mc * p.y_chunk_bytes, &tmY, &full[s], (mt * p.nmc + mc) * p.chunky, ow0,
                                    pl, oh, n * p.OD + od);
                uint8_t *xb = smem + p.x_base + (size_t)s * p.x_stride;
                for (int b = 0; b < ncb; ++b) {
                    int kd, kh, xc;
                    wg_decode_cb(p, cb0 + b, kd, kh, xc);
                    const int d = od * p.sd - p.pd + kd, h = oh * p.sh - p.ph + kh;
                    if (d < 0 || d >= p.D || h < 0 || h >= p.H) continue;
                    for (int pl = 0; pl < p.planes; ++pl)
                        tma_load_5d(xb + (size_t)b * p.x_buf_bytes + (size_t)pl * p.x_plane_bytes, &tmX, &full[s], xc * p.chunkx, ow0 - p.pw, pl, h,
                                    n * p.D + d);
                }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            const uint32_t idesc = make_idesc_bf16(128, ncols, 1, 1);
            const uint32_t lty = layout_type_for_swizzle_bytes(p.swy), ltx = layout_type_for_swizzle_bytes(p.swx);
            // descriptor templates (everything but the 14-bit start address); the x descriptor's LBO is ONE ROW: next N chunk = next kw shift
            const uint64_t ytmpl = make_smem_desc(0, p.y_chunk_bytes, 8 * p.swy, lty), xtmpl = make_smem_desc(0, p.swx, 8 * p.swx, ltx);
            const uint64_t ystep = (uint64_t)((16 * p.swy) >> 4), xstep = (uint64_t)((16 * p.swx) >> 4);
            uint32_t started = 0;
            int it = 0;
            for (long long u = split; u < p.units; u += p.splits, ++it) {
                int n, od, oh, ow0;
                decode_unit(u, n, od, oh, ow0);
                const int s = it % p.stages;
                mbar_wait(&full[s], (it / p.stages) & 1);
                tc_fence_after();
                const uint32_t y_hi = smem_u32(smem + (size_t)s * p.y_stride);
                const uint32_t x0 = smem_u32(smem + p.x_base + (size_t)s * p.x_stride);
                // (measured: interleaving the column blocks inside the K loop does not help — the accumulate dependency is not the limiter, the
                //  single-thread issue rate is — so keep the order with the fewest instructions per MMA: descriptors advance by integer adds)
                for (int b = 0; b < ncb; ++b) {
                    int kd, kh, xc;
                    wg_decode_cb(p, cb0 + b, kd, kh, xc);
                    const int d = od * p.sd - p.pd + kd, h = oh * p.sh - p.ph + kh;
                    if (d < 0 || d >= p.D || h < 0 || h >= p.H) continue;
                    const uint32_t dcol = tmem + b * ncols;
                    uint64_t dyh = ytmpl | (uint64_t)((y_hi >> 4) & 0x3FFF);
                    uint64_t dyl = ytmpl | (uint64_t)(((y_hi + p.y_plane_bytes) >> 4) & 0x3FFF);
                    uint64_t dxh = xtmpl | (uint64_t)(((x0 + b * p.x_buf_bytes) >> 4) & 0x3FFF);
                    uint64_t dxl = xtmpl | (uint64_t)(((x0 + b * p.x_buf_bytes + p.x_plane_bytes) >> 4) & 0x3FFF);
                    uint32_t acc = (started >> b) & 1u;
                    for (int k = 0; k < (p.skip == 1 ? 1 : p.ksteps); ++k) {
                        umma_bf16(dcol, dyh, dxh, idesc, acc);
                        if (p.planes > 1) {
                            umma_bf16(dcol, dyh, dxl, idesc, 1);
                            if (!p.mtrick) umma_bf16(dcol, dyl, dxh, idesc, 1);
                        }
                        acc = 1;
                        dyh += ystep; dyl += ystep; dxh += xstep; dxl += xstep;     // 16 voxel rows further along K
                    }
                    started |= 1u << b;
                }
                umma_commit(&empty[s]);
            }
            *(volatile uint32_t *)&s_started = started;
            __threadfence_block();
            if (started) umma_commit(&accum_full);
            else mbar_arrive(&accum_full);
        }
    }
    if (warp >= 2) {
        // epilogue: dump this CTA's accumulators (TMEM lanes x used columns) to its slot of the partial buffer — plain coalesced-ish
        // stores, no atomics; the cross-CTA (split-K) reduction is a separate streaming kernel
        mbar_wait(&accum_full, 0);
        tc_fence_after();
        const uint32_t started = *(volatile uint32_t *)&s_started;
        const int q = warp & 3;
        const int m = q * 32 + lane;
        float *slot = p.partial + (((size_t)split * p.groups + group) * p.mtiles + mt) * (size_t)(128 * p.slot_cols) + (size_t)m * p.slot_cols;
        // only the lanes / columns that hold real (co, ci) pairs are written: the reduction never reads the channel padding (36 of 64 lanes per
        // half and 48 of 64 columns per tap for the 36-channel layers: 58 % of the dump traffic)
        const bool lane_used = p.mtrick ? (m < 2 * p.co_p && (m % p.co_p) < p.cout) : (mt * 128 + m < p.cout);
        if (__ballot_sync(0xffffffffu, lane_used) == 0u) goto dumped;
        for (int b = 0; b < ncb; ++b) {
            const bool live = (started >> b) & 1u;
            int kd_, kh_, xc_;
            wg_decode_cb(p, cb0 + b, kd_, kh_, xc_);
            for (int c0 = 0; c0 < ncols; c0 += 16) {
                if (xc_ * p.chunkx + (c0 % p.chunkx) >= p.cin) continue;
                float v[16];
                if (live) {
                    tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + b * ncols + c0, v);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = 0.f;
                }
                if (!lane_used) continue;
                float4 *dst = reinterpret_cast<float4 *>(slot + b * ncols + c0);
                dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                dst[2] = make_float4(v[8], v[9], v[10], v[11]);
                dst[3] = make_float4(v[12], v[13], v[14], v[15]);
            }
        }
    dumped:;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, p.tmem_cols);
}

// dw[co, ci, tap] = sum over splits (and over the hi / lo lane halves in mtrick mode) of the partial accumulators
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(TcWgradParams p, float *__restrict__ dw) {
    const int ncols = p.KW * p.chunkx;
    const long long total = (long long)p.cout * p.ncb_total * ncols;     // (co, column block, col)
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int col = (int)(i % ncols);
        const int cb = (int)((i / ncols) % p.ncb_total);
        const int co = (int)(i / ((long long)ncols * p.ncb_total));
        int kd, kh, xc;
        wg_decode_cb(p, cb, kd, kh, xc);
        const int kw = col / p.chunkx, ci = xc * p.chunkx + col % p.chunkx;
        if (ci >= p.cin) continue;
        const int group = cb / p.CB, b = cb % p.CB;
        const int mt = p.mtrick ? 0 : co / 128, m = p.mtrick ? co : co % 128;
        float acc = 0.f;
        for (int sp = 0; sp < p.splits; ++sp) {
            const float *slot = p.partial + (((size_t)sp * p.groups + group) * p.mtiles + mt) * (size_t)(128 * p.slot_cols) + b * ncols + col;
            acc += slot[(size_t)m * p.slot_cols];
            if (p.mtrick && p.planes > 1) acc += slot[(size_t)(m + p.co_p) * p.slot_cols];
        }
        dw[((size_t)co * p.cin + ci) * p.T + (kd * p.KH + kh) * p.KW + kw] = acc;
    }
}

// ------------------------------------------------------------------------------------------------ host
struct WgPlan {
    bool ok = false;
    int co_p, swy, chunky, nmc, mtiles, mtrick;
    int ci_p, swx, chunkx, nxc;
    int seg, segs, ksteps, rows_y, rows_x, rows_x_pad;
    int ncb_total, CB, groups, stages, waves;
};

static WgPlan make_wg_plan(const ConvGeom &g) {
    WgPlan w;
    if (g.sw != 1) return w;
    // x (N side): one chunk spans all of ci when ci <= 64, so that all kw taps of a pair fit one MMA
    w.ci_p = conv_tc_kpad_smem(g.cin);
    w.chunkx = w.ci_p < 64 ? w.ci_p : 64;
    w.swx = w.chunkx * 2;
    w.nxc = w.ci_p / w.chunkx;
    if (g.kw * w.chunkx > 256) return w;
    // dy (M side)
    w.co_p = conv_tc_kpad_smem(g.cout);
    w.swy = w.co_p >= 64 ? 128 : w.co_p * 2;
    w.chunky = w.swy / 2;
    w.mtrick = (2 * w.co_p <= 128) ? 1 : 0;
    if (w.mtrick) { w.nmc = w.co_p / w.chunky; w.mtiles = 1; }
    else {
        // M tiles of 128 rows (2 chunks of 64 channels); the tensor keeps conv_tc_kpad(cout) channels, chunks past it are TMA zero fill
        w.swy = 128; w.chunky = 64;
        w.nmc = 2; w.mtiles = ceil_div(w.co_p, 128);
    }
    w.seg = g.ow >= 128 ? 128 : g.ow;
    w.segs = ceil_div(g.ow, w.seg);
    w.ksteps = ceil_div(w.seg, 16);
    w.rows_y = w.ksteps * 16;
    w.rows_x = w.ksteps * 16 + g.kw - 1;
    w.rows_x_pad = ceil_div(w.rows_x, 8) * 8;
    if (w.rows_x > 256) return w;
    w.ncb_total = g.kd * g.kh * w.nxc;
    w.CB = 512 / (g.kw * w.chunkx);
    if (w.CB > 32) w.CB = 32;
    if (w.CB > w.ncb_total) w.CB = w.ncb_total;
    // Narrow x operands (<= 32 channels: small N per MMA, issue-bound) run best as many small co-resident CTAs — one column block and a
    // small TMEM/shared-memory footprint each; wide ones (64-channel chunks, tensor-bound N = kw*64) as one big CTA per SM.  Measured sweep:
    // profiles/r01_wgrad_sweep.txt.
    w.waves = 1;
    if (w.chunkx <= 32) { w.CB = 1; w.waves = 2; }
    if (const char *e = getenv("MDT_WG_CB")) { const int v = atoi(e); if (v >= 1 && v < w.CB) w.CB = v; }   // experiment knobs
    if (const char *e = getenv("MDT_WG_WAVES")) { const int v = atoi(e); if (v >= 1 && v <= 8) w.waves = v; }
    // shared memory: 2 stages of (dy planes + CB x buffers)
    auto stage_bytes = [&](int cb, int planes) { return planes * w.nmc * w.rows_y * w.swy + cb * planes * w.rows_x_pad * w.swx; };
    w.stages = kWgMaxStages;
    if (const char *e = getenv("MDT_WG_STAGES")) { const int v = atoi(e); if (v >= 1 && v <= kWgMaxStages) w.stages = v; }
    while (w.CB > 1 && w.stages * stage_bytes(w.CB, 2) > 200 * 1024) --w.CB;
    if (w.stages * stage_bytes(w.CB, 2) > 200 * 1024) return w;
    w.groups = ceil_div(w.ncb_total, w.CB);
    w.ok = true;
    return w;
}

bool conv_tc_wgrad_supported(const ConvGeom &g) { return make_wg_plan(g).ok && tmap_encode_fn() != nullptr; }

static size_t wg_align(size_t v) { return (v + 1023) / 1024 * 1024; }

// split-K factor.  Lower bound: a full wave of CTAs.  Upper bound on the work per CTA: the tensor core's fp32 accumulation is not
// round-to-nearest — measured on B200 (tools/wgrad_precision.py, profiles/r01_wgrad_precision.txt) the error of a TMEM accumulator grows
// LINEARLY with the number of MMAs chained into it (~1.9e-7 of the result per MMA: 3.3e-4 after the 1771 steps a 2 x 128^3 layer gives one
// CTA per SM).  Chains are therefore cut at kMaxChain MMAs (measured <= 1e-5 at every size) and the partial sums are combined in IEEE fp32 by wgrad_reduce_kernel.
constexpr int kMaxChain = 512;

static int wg_splits(const ConvGeom &g, const WgPlan &w) {
    const long long units = (long long)g.n * g.od * g.oh * w.segs;
    const int mmas_per_unit = w.ksteps * 2;                         // two MMAs per K step go into the same accumulator (x_hi, x_lo)
    long long max_units = (getenv("MDT_WG_CHAIN") ? atoi(getenv("MDT_WG_CHAIN")) : kMaxChain) / mmas_per_unit;   // MDT_WG_CHAIN: experiment knob
    if (max_units < 1) max_units = 1;
    const long long min_splits = ceil_div<long long>(units, max_units);
    long long splits = (long long)num_sms() * w.waves / ((long long)w.groups * w.mtiles);   // w.waves CTAs per SM, co-resident
    if (splits < min_splits) splits = min_splits;
    if (splits < 1) splits = 1;
    if (splits > units) splits = units;
    return (int)splits;
}

static int wg_slot_cols(const ConvGeom &g, const WgPlan &w) { return ceil_div(w.CB * g.kw * w.chunkx, 16) * 16; }

size_t conv_tc_wgrad_workspace_bytes(const ConvGeom &g, int precision) {
    const WgPlan w = make_wg_plan(g);
    if (!w.ok) return 0;
    const int planes = precision == 1 ? 1 : 2;
    const size_t rows_y = (size_t)g.n * g.od * g.oh * g.ow, rows_x = (size_t)g.n * g.d * g.h * g.w;
    const size_t partial = (size_t)wg_splits(g, w) * w.groups * w.mtiles * 128 * wg_slot_cols(g, w) * sizeof(float);
    const size_t b = wg_align(planes * rows_y * conv_tc_kpad(g.cout) * 2) + wg_align(planes * rows_x * conv_tc_kpad(g.cin) * 2) + wg_align(partial) + 2048;
    const size_t bias = conv_bias_grad_workspace_bytes(g);
    return b > bias ? b : bias;
}

// dy_presplit != nullptr: dy is already split (interleaved layout, conv_tc_kpad(cout) channels); then db must have been produced by the caller
static int conv_tc_wgrad_impl(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, int precision, void *ws, size_t ws_bytes,
                              cudaStream_t st, const __nv_bfloat16 *dy_presplit, const __nv_bfloat16 *x_presplit = nullptr) {
    const WgPlan w = make_wg_plan(g);
    if (!w.ok) return MDT_EUNSUPPORTED;
    if (ws_bytes < conv_tc_wgrad_workspace_bytes(g, precision)) return MDT_EWORKSPACE;
    const int planes = precision == 1 ? 1 : 2;
    const int T = g.kd * g.kh * g.kw;
    const long long rows_y = (long long)g.n * g.od * g.oh * g.ow, rows_x = (long long)g.n * g.d * g.h * g.w;
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    __nv_bfloat16 *ys = dy_presplit ? const_cast<__nv_bfloat16 *>(dy_presplit) : reinterpret_cast<__nv_bfloat16 *>(base);
    const int co_g = conv_tc_kpad(g.cout), ci_g = conv_tc_kpad(g.cin);   // channel extents of the split planes in global memory
    __nv_bfloat16 *xs = x_presplit ? const_cast<__nv_bfloat16 *>(x_presplit)
                                   : reinterpret_cast<__nv_bfloat16 *>(base + wg_align((size_t)planes * rows_y * co_g * 2));
    auto split = [&](const float *src, __nv_bfloat16 *dst, long long rows, int C, int Cp, int line_w) {
        long long blocks = ceil_div<long long>(rows * (Cp / 8), 256);
        if (blocks > (long long)num_sms() * 32) blocks = (long long)num_sms() * 32;
        split_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, dst, rows, C, Cp, planes, line_w, nullptr, nullptr, nullptr);
        return launch_status();
    };
    int rc = MDT_OK;
    if (!dy_presplit && (rc = split(dy, ys, rows_y, g.cout, co_g, g.ow))) return rc;
    if (!x_presplit && (rc = split(x, xs, rows_x, g.cin, ci_g, g.w))) return rc;

    TcWgradParams p{};
    p.NB = g.n; p.OD = g.od; p.OH = g.oh; p.OW = g.ow; p.D = g.d; p.H = g.h; p.W = g.w;
    p.KD = g.kd; p.KH = g.kh; p.KW = g.kw; p.sd = g.sd; p.sh = g.sh; p.pd = g.pd; p.ph = g.ph; p.pw = g.pw;
    p.cin = g.cin; p.cout = g.cout; p.T = T;
    p.seg = w.seg; p.segs = w.segs; p.ksteps = w.ksteps;
    p.swy = w.swy; p.chunky = w.chunky; p.nmc = w.nmc; p.co_p = w.co_p; p.mtrick = w.mtrick;
    p.swx = w.swx; p.chunkx = w.chunkx; p.nxc = w.nxc;
    p.ncb_total = w.ncb_total; p.CB = w.CB; p.groups = w.groups;
    p.planes = planes;
    p.stages = w.stages;
    p.tmem_cols = 32;
    while (p.tmem_cols < w.CB * g.kw * w.chunkx) p.tmem_cols <<= 1;
    p.y_chunk_bytes = w.rows_y * w.swy;
    p.y_plane_bytes = w.nmc * p.y_chunk_bytes;
    p.x_plane_bytes = w.rows_x_pad * w.swx;
    p.x_buf_bytes = planes * p.x_plane_bytes;
    p.stage_bytes = (int)wg_align((size_t)planes * p.y_plane_bytes + (size_t)w.CB * p.x_buf_bytes);
    p.y_tx_bytes = w.rows_y * w.swy;
    p.x_tx_bytes = w.rows_x * w.swx;
    p.units = (long long)g.n * g.od * g.oh * w.segs;
    p.splits = wg_splits(g, w);
    p.mtiles = w.mtiles;
    p.skip = getenv("MDT_WG_SKIP") ? atoi(getenv("MDT_WG_SKIP")) : 0;
    p.slot_cols = wg_slot_cols(g, w);
    p.partial = reinterpret_cast<float *>(base + wg_align((size_t)planes * rows_y * co_g * 2) + wg_align((size_t)planes * rows_x * ci_g * 2));

    CUtensorMap tmY, tmX;
    {
        const uint64_t yl = (uint64_t)g.ow * co_g * 2;   // one W line of one plane
        const uint64_t dims[5] = {(uint64_t)co_g, (uint64_t)g.ow, (uint64_t)planes, (uint64_t)g.oh, (uint64_t)g.n * g.od};
        const uint64_t str[4] = {(uint64_t)co_g * 2, yl, yl * planes, yl * planes * g.oh};
        const uint32_t box[5] = {(uint32_t)w.chunky, (uint32_t)w.rows_y, 1u, 1u, 1u};
        if (!encode_bf16_tmap(&tmY, ys, 5, dims, str, box, w.swy)) return MDT_EDRIVER;
        const uint64_t xl = (uint64_t)g.w * ci_g * 2;
        const uint64_t xd[5] = {(uint64_t)ci_g, (uint64_t)g.w, (uint64_t)planes, (uint64_t)g.h, (uint64_t)g.n * g.d};
        const uint64_t xs_[4] = {(uint64_t)ci_g * 2, xl, xl * planes, xl * planes * g.h};
        const uint32_t xbox[5] = {(uint32_t)w.chunkx, (uint32_t)w.rows_x, 1u, 1u, 1u};
        if (!encode_bf16_tmap(&tmX, xs, 5, xd, xs_, xbox, w.swx)) return MDT_EDRIVER;
    }
    // the M = 128 dy descriptor walks 128 / chunky chunk slots from the stage base (rows past the real dy chunks are ignored by the
    // epilogue); make sure that walk stays inside the allocation for the last stage too
    const size_t walk = (size_t)(128 / w.chunky) * w.rows_y * w.swy;
    const size_t tail = walk > (size_t)p.stage_bytes ? walk - p.stage_bytes : 0;
    size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + tail;
    if (smem > 218 * 1024) return MDT_EUNSUPPORTED;
    p.y_stride = p.stage_bytes; p.x_base = planes * p.y_plane_bytes; p.x_stride = p.stage_bytes;
    // placement experiment (tools/mma_major_probe: the cost of an MMA depends on how far apart its two shared-memory operands lie):
    // MDT_WG_LAYOUT=1 groups the dy buffers of all stages in front of the x buffers, MDT_WG_GAP (KiB) moves the x region further up
    if (const char *e = getenv("MDT_WG_LAYOUT")) {
        if (atoi(e) == 1) {
            const size_t yreg = wg_align((size_t)planes * p.y_plane_bytes), xreg = wg_align((size_t)w.CB * p.x_buf_bytes);
            size_t gap = getenv("MDT_WG_GAP") ? (size_t)atoi(getenv("MDT_WG_GAP")) * 1024 : 0;
            auto total = [&](size_t g_) {
                const size_t a = p.stages * yreg + g_ + p.stages * xreg, b = (p.stages - 1) * yreg + walk;   // the M = 128 walk from the last dy stage
                return (a > b ? a : b) + 1024;
            };
            size_t need = total(gap);
            if (need > 218 * 1024) { gap = 0; need = total(0); }
            if (need <= 218 * 1024) {
                p.y_stride = (int)yreg; p.x_base = (int)(p.stages * yreg + gap); p.x_stride = (int)xreg;
                smem = need;
            }
        }
    }
    static bool attr[kMaxDevices] = {};
    if (!ensure_smem_attr(conv_tc_wgrad_kernel, 220 * 1024, attr)) return MDT_EDRIVER;
    dim3 grid((unsigned)(w.groups * p.splits), w.mtiles);
    conv_tc_wgrad_kernel<<<grid, kWgThreads, smem, st>>>(tmY, tmX, p);
    if ((rc = launch_status())) return rc;
    {
        const long long total = (long long)g.cout * w.ncb_total * g.kw * w.chunkx;
        wgrad_reduce_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(p, dw);
        if ((rc = launch_status())) return rc;
    }
    if (db && !dy_presplit) return conv_bias_grad(g, dy, db, ws, ws_bytes, st);   // the workspace is free again once the reduction has run
    return MDT_OK;
}

int conv_tc_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, int precision, void *ws, size_t ws_bytes,
                  cudaStream_t st) {
    return conv_tc_wgrad_impl(g, x, dy, dw, db, precision, ws, ws_bytes, st, nullptr);
}

// ------------------------------------------------------------------------------------------------ fused backward
// One streaming pass over dy produces everything both gradient kernels need: the split planes (shared by dgrad and wgrad), the ReLU
// mask of a fused-ReLU conv, the bias gradient, and (on request) the masked fp32 gradient for a fused residual input.
bool conv_tc_backward_supported(const ConvGeom &g, bool need_dx) {
    return conv_tc_wgrad_supported(g) && (!need_dx || conv_tc_supported(g, 1)) && g.cout <= 256;
}

// grid of the split pass over dy; with a bias gradient a thread must stay on the same 8-channel group across its grid-stride steps (its column
// sums live in registers), i.e. gridDim * 256 must be a multiple of co_p / 8 (6 groups for 36 -> 48 channels)
static long long backward_split_blocks(const ConvGeom &g, bool with_bias) {
    const int co_p = conv_tc_kpad(g.cout);
    const long long rows_y = (long long)g.n * g.od * g.oh * g.ow;
    long long blocks = ceil_div<long long>(rows_y * (co_p / 8), 256);
    if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
    if (with_bias) {
        const long long groups = co_p / 8;
        long long unit = groups;
        for (long long a = groups, b = 256; b;) { const long long t = a % b; a = b; b = t; unit = groups / a; }   // groups / gcd(groups, 256)
        blocks = blocks > unit ? blocks / unit * unit : unit;
    }
    return blocks;
}

size_t conv_tc_backward_workspace_bytes(const ConvGeom &g, bool need_dx, int precision) {
    const int planes = precision == 1 ? 1 : 2;
    const size_t rows_y = (size_t)g.n * g.od * g.oh * g.ow;
    const size_t ys = wg_align(planes * rows_y * conv_tc_kpad(g.cout) * 2);
    size_t inner = conv_tc_wgrad_workspace_bytes(g, precision);
    if (need_dx) { const size_t d = conv_tc_workspace_bytes(g, 1, precision); if (d > inner) inner = d; }
    const size_t colsum = sizeof(float) * (size_t)backward_split_blocks(g, true) * g.cout;   // per-block bias-gradient partials
    if (colsum > inner) inner = colsum;
    return ys + inner + 4096;
}

int conv_tc_backward(const ConvGeom &g, const float *x, const float *dy, const float *relu_of, const float *w, float *dx, float *dw, float *db,
                     float *dy_masked_out, int precision, void *ws, size_t ws_bytes, cudaStream_t st, const void *x_split) {
    if (!conv_tc_backward_supported(g, dx != nullptr)) return MDT_EUNSUPPORTED;
    if (ws_bytes < conv_tc_backward_workspace_bytes(g, dx != nullptr, precision)) return MDT_EWORKSPACE;
    const int planes = precision == 1 ? 1 : 2;
    const int co_p = conv_tc_kpad(g.cout);
    const long long rows_y = (long long)g.n * g.od * g.oh * g.ow;
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    __nv_bfloat16 *ys = reinterpret_cast<__nv_bfloat16 *>(base);
    uint8_t *inner = base + wg_align((size_t)planes * rows_y * co_p * 2);
    const size_t inner_bytes = ws_bytes - (size_t)(inner - reinterpret_cast<uint8_t *>(ws));
    const long long blocks = backward_split_blocks(g, db != nullptr);
    // bias gradient: per-block column sums go to the (not yet used) inner workspace and are combined in a fixed order before dgrad / wgrad
    // reuse that memory
    float *colsum = db ? reinterpret_cast<float *>(inner) : nullptr;
    split_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(dy, ys, rows_y, g.cout, co_p, planes, g.ow, relu_of, dy_masked_out, colsum);
    int rc = launch_status();
    if (rc) return rc;
    if (db && (rc = reduce_partials(colsum, (int)blocks, g.cout, db, st))) return rc;
    if (dx && (rc = conv_tc_run(g, 1, nullptr, w, nullptr, nullptr, dx, 0, precision, inner, inner_bytes, st, ys, nullptr))) return rc;
    return conv_tc_wgrad_impl(g, x, nullptr, dw, nullptr, precision, inner, inner_bytes, st, ys, reinterpret_cast<const __nv_bfloat16 *>(x_split));
}

// ---- canonical split form of an activation tensor [N, D, H, W, C]: it depends on the tensor alone (C -> conv_tc_kpad(C), W), so one split can
// serve every consumer (sibling convs in the forward pass, the weight gradient in the backward pass)
size_t conv_tc_split_bytes(long long rows, int channels, int precision) {
    return wg_align((size_t)(precision == 1 ? 1 : 2) * rows * conv_tc_kpad(channels) * 2);
}

int conv_tc_split(const float *x, long long rows, int channels, int line_w, int precision, void *out, cudaStream_t st) {
    const int planes = precision == 1 ? 1 : 2, cp = conv_tc_kpad(channels);
    long long blocks = ceil_div<long long>(rows * (cp / 8), 256);
    if (blocks > (long long)num_sms() * 32) blocks = (long long)num_sms() * 32;
    split_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, reinterpret_cast<__nv_bfloat16 *>(out), rows, channels, cp, planes, line_w, nullptr, nullptr, nullptr);
    return launch_status();
}

}  // namespace mdt

// conv3d on the 5th-generation tensor cores (algo 2): implicit GEMM with TMA-staged operands, tcgen05.mma, TMEM accumulators.
//
// Replaces the cuDNN conv3d behind nn.Conv3d in the reference (utils/model_utils.py:762; models/backbone.py:27-206, heads in
// models/retina_unet.py:40-119, models/mrcnn.py:40-169).
//
// GEMM view (fprop): rows M = output voxels, columns N = Cout, reduction K = taps x Cin.   dgrad: rows = input voxels, N = Cin, K = taps x Cout.
//
// fp32-faithful arithmetic on a bf16 tensor pipe ("split-bf16 x3"): every fp32 operand v is stored as two bf16 planes hi = rn(v),
// lo = rn(v - hi) (|v - hi - lo| <= 2^-17 |v|); the kernel issues three MMAs per K step — A_hi*B_hi + A_hi*B_lo + A_lo*B_hi — into ONE fp32
// TMEM accumulator, dropping only the lo*lo term (~2^-18).  precision = 1 issues the first MMA only (plain bf16 inputs).
//
// Data movement (the part that decides the roofline): a tile is 128 consecutive output voxels along the innermost spatial axis (the
// reference's z).  For every (kd, kh) the TMA loads ONE halo line of 128 + kw - 1 voxels x a 16/32/64-channel chunk into a
// hardware-swizzled shared-memory buffer, and the kw taps are issued as tcgen05.mma on row-SHIFTED windows of that buffer (the shared
// memory matrix descriptor start address moves by kw rows; verified on B200 by tools/tc_probe, profiles/r01_tc_probe.txt).  Each input
// element is therefore fetched kd*kh times per tile instead of kd*kh*kw times.  Zero padding = TMA out-of-bounds fill.  Tiles that are not
// one full line (W < 128) use a box of BH lines x BW voxels per tap instead (generic mode).
// Weights stream through their own ring as [Np x chunk] K-major tiles per tap.
//
// Warp roles (192 threads): warp 0 TMA producer (one lane), warp 1 TMEM allocator + MMA issuer (one lane), warps 2-5 epilogue
// (TMEM -> registers -> bias / residual / ReLU -> global fp32 NDHWC).
#include "conv3d_common.cuh"
#include "tc_common.cuh"
#include "conv3d_tc_plan.cuh"
#include <cstdlib>

namespace mdt {
using namespace tc;

// ------------------------------------------------------------------------------------------------ operand preparation kernels
// fp32 [rows, C] -> bf16 planes (hi, lo), channels zero-padded to Cp (multiple of 16).
//   inter_w = 0: plane-major  [plane][rows][Cp]                       (wgrad operands)
//   inter_w > 0: line-interleaved [line][plane][inter_w voxels][Cp]   (fprop/dgrad A operand: both planes of a W-line are adjacent, so ONE
//                TMA box {chunk, voxels, 2 planes} fetches the hi and lo halo line together); rows = lines * inter_w
__global__ void __launch_bounds__(256) split_rows_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, long long rows, int C,
                                                        int Cp, int planes, int inter_w, const float *__restrict__ relu_of,
                                                        float *__restrict__ masked_out, float *__restrict__ colsum) {
    // backward-pass extras, all fused into this one streaming pass over dy:
    //   relu_of    : forward output y of a conv with fused ReLU -> the element is zeroed where y <= 0 (threshold_backward)
    //   masked_out : fp32 copy of the masked gradient (needed when it is also the gradient of a fused residual input)
    //   colsum     : [gridDim.x][C] per-block column sums (bias-gradient partials, combined by reduce_partials); needs gridDim * 256 to be a
    //                multiple of Cp / 8, so that a thread keeps the same 8 channels for all its rows and sums them in registers
    __shared__ float s_part[256][8];
    const int groups = Cp / 8;  // 8 channels (16 bytes of bf16) per thread
    const long long total = rows * groups;
    const long long plane_stride = inter_w > 0 ? (long long)inter_w * Cp : rows * Cp;
    const bool vec4 = (C & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(relu_of) | reinterpret_cast<uintptr_t>(masked_out)) & 15) == 0;
    float rs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / groups;
        const int c0 = (int)(i % groups) * 8;
        float v[8];
        if (vec4) {
            // 128-bit loads / stores: a row is C * 4 bytes with C % 4 == 0 and c0 % 8 == 0, so every 4-channel piece is 16-byte aligned
#pragma unroll
            for (int h = 0; h < 8; h += 4) {
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c0 + h < C) {
                    t = __ldg(reinterpret_cast<const float4 *>(src + r * C + c0 + h));
                    if (relu_of) {
                        const float4 y = __ldg(reinterpret_cast<const float4 *>(relu_of + r * C + c0 + h));
                        if (!(y.x > 0.f)) t.x = 0.f;
                        if (!(y.y > 0.f)) t.y = 0.f;
                        if (!(y.z > 0.f)) t.z = 0.f;
                        if (!(y.w > 0.f)) t.w = 0.f;
                    }
                    if (masked_out) *reinterpret_cast<float4 *>(masked_out + r * C + c0 + h) = t;
                }
                v[h] = t.x; v[h + 1] = t.y; v[h + 2] = t.z; v[h + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float t = (c0 + k < C) ? __ldg(src + r * C + c0 + k) : 0.f;
                if (relu_of && c0 + k < C && !(__ldg(relu_of + r * C + c0 + k) > 0.f)) t = 0.f;
                v[k] = t;
            }
            if (masked_out) {
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (c0 + k < C) masked_out[r * C + c0 + k] = v[k];
            }
        }
        if (colsum) {
#pragma unroll
            for (int k = 0; k < 8; ++k) rs[k] += v[k];
        }
        __align__(16) __nv_bfloat16 hi[8], lo[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            hi[k] = __float2bfloat16_rn(v[k]);
            lo[k] = __float2bfloat16_rn(v[k] - __bfloat162float(hi[k]));
        }
        long long off;
        if (inter_w > 0) { const long long line = r / inter_w; const int w = (int)(r % inter_w); off = (line * planes * inter_w + w) * Cp + c0; }
        else off = r * Cp + c0;
        *reinterpret_cast<uint4 *>(dst + off) = *reinterpret_cast<const uint4 *>(hi);
        if (planes > 1) *reinterpret_cast<uint4 *>(dst + off + plane_stride) = *reinterpret_cast<const uint4 *>(lo);
    }
    if (colsum) {
        // thread t holds the sums of group (blockIdx.x * blockDim.x + t) % groups; channel c adds its threads up in increasing t
#pragma unroll
        for (int k = 0; k < 8; ++k) s_part[threadIdx.x][k] = rs[k];
        __syncthreads();
        const int base = (int)((blockIdx.x * (long long)blockDim.x) % groups);
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            float t = 0.f;
            for (int u = ((c / 8 - base) % groups + groups) % groups; u < (int)blockDim.x; u += groups) t += s_part[u][c % 8];
            colsum[(long long)blockIdx.x * C + c] = t;
        }
    }
}

// weights [Cout, Cin, T] fp32 -> bf16 planes [planes][T][Nrows][Kp]  (K contiguous)
//   mode 0 (fprop): Nrows = Cout (padded Np), K = Cin:  B[t][co][ci] = w[co][ci][t]
//   mode 1 (dgrad): Nrows = Cin  (padded Np), K = Cout: B[t][ci][co] = w[co][ci][t]
// The packed tensor is written `reps` times: every CTA of the conv kernel streams the SAME weight tiles at about the same time, and a
// single copy makes all SMs hit the same few L2 slices in lockstep; CTAs pick replica blockIdx.x % reps, spreading the load.
__global__ void __launch_bounds__(256) pack_weights_tc_kernel(const float *__restrict__ w, __nv_bfloat16 *__restrict__ dst, int cout, int cin, int T,
                                                             int Np, int Kp, int planes, int mode, int reps) {
    const long long total = (long long)T * Np * Kp;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % Kp);
        const int n = (int)((i / Kp) % Np);
        const int t = (int)(i / ((long long)Kp * Np));
        float v = 0.f;
        if (mode == 0) { if (n < cout && k < cin) v = w[((size_t)n * cin + k) * T + t]; }
        else           { if (n < cin && k < cout) v = w[((size_t)k * cin + n) * T + t]; }
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
        // layout [T][plane][Np][Kp]: the planes of a tap are adjacent, so one TMA box {chunk, NT, planes, taps} fetches a whole stage
        const long long per_tap = (long long)Np * Kp;
        const long long o = ((long long)t * planes) * per_tap + (long long)n * Kp + k;
        dst[o] = hi;
        if (planes > 1) dst[o + per_tap] = lo;
        (void)reps;
    }
}

// ------------------------------------------------------------------------------------------------ the implicit-GEMM kernel
// source line (d_src, h_src) feeding tile row-line (rd, rh0) through tap (kd, kh); false = this tap contributes nothing to the tile
__device__ __forceinline__ bool tc_step_coords(const TcConvParams &p, int rd, int rh0, int kd, int kh, int &d_src, int &h_src) {
    if (!p.dgrad) {
        d_src = rd * p.sd - p.pd + kd;
        h_src = rh0 * p.sh - p.ph + kh;              // generic mode (BH > 1) is only planned for sh == 1
    } else {
        const int td = rd + p.pd - kd;
        if (td < 0 || td % p.sd != 0) return false;
        d_src = td / p.sd;
        const int th = rh0 + p.ph - kh;
        if (p.BH == 1) {
            if (th < 0 || th % p.sh != 0) return false;
            h_src = th / p.sh;
        } else {
            h_src = th;                              // sh == 1
        }
    }
    if (d_src < 0 || d_src >= p.SD) return false;   // whole line outside the source: zeros
    if (h_src + p.BH <= 0 || h_src >= p.SH) return false;
    return true;
}

// Pipeline stage = one (kd, kh) x a group of CPS K-chunks: the A halo line(s) of those chunks + the B tiles of the TPS taps sharing it.
// One full / one empty mbarrier per stage; the MMA thread waits once, issues TPS * CPS * (swz/32) * {1|2} MMAs back to back, commits once.
// Split-bf16 uses N-stacking: the hi and lo weight planes of a tile are adjacent in shared memory, so  A_hi x [B_hi ; B_lo]  is ONE
// MMA with N = 2*NT (accumulator columns [0,NT) += hi*hi, [NT,2NT) += hi*lo) followed by  A_lo x B_hi  (N = NT); the epilogue adds the
// two column halves.  2 MMAs and 2 A reads per K step instead of 3.
__global__ void __launch_bounds__(kTcThreads, 5)   // <= 68 registers: residency (CTAs per SM) is what hides the per-stage latency
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcConvParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ uint64_t full[kTcMaxStages], empty[kTcMaxStages], accum_full;
    __shared__ uint32_t tmem_base_s;
    __shared__ uint32_t s_have_acc;
    __shared__ uint32_t s_n1, s_n2;   // accumulators actually written, per MMA type
    __shared__ float s_bias[128];

    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int t = blockIdx.x;
    const int tw = t % p.tiles_w; t /= p.tiles_w;
    const int th = t % p.tiles_h; t /= p.tiles_h;
    const int rd = t % p.RD;
    const int nb = t / p.RD;
    const int rw0 = tw * p.BW, rh0 = th * p.BH;
    const int n0 = blockIdx.y * p.NT;
    const int chunk_elems = p.swz >> 1;
    const int ngroups = (p.nchunks + p.CPS - 1) / p.CPS;

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.D; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(&accum_full, 1);
        s_have_acc = 1;
        fence_barrier_init();
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmB);
    }
    if (threadIdx.x >= 64) {
        const int c = threadIdx.x - 64;
        s_bias[c] = (p.bias && n0 + c < p.Cn) ? __ldg(p.bias + n0 + c) : 0.f;
    }
    // Q independent accumulator chains per MMA type (see the MMA issuer): type-1 accumulators are acc1_cols wide, type-2 (split-bf16 only) NT wide
    const int acc1_cols = p.planes > 1 ? 2 * p.NT : p.NT;
    const int Q = p.Q;
    const int acc2_base = Q * acc1_cols;
    const int acc_total = acc2_base;   // no separate type-2 accumulators: keeps TMEM at 2*NT columns so that up to 4 CTAs fit in the SM's 512
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < acc_total) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (warp == 0) {
        // =============================================================== TMA producer
        if (elect_one()) {
            int s = 0;
            uint32_t ph = 1;   // parity to wait for on `empty` (fresh barrier: the "previous" phase counts as complete)
                    for (int kd = 0; kd < p.KD; ++kd)
                for (int kh = 0; kh < p.KH; ++kh) {
                    int d_src, h_src;
                    if (!tc_step_coords(p, rd, rh0, kd, kh, d_src, h_src)) continue;
                    for (int g = 0; g < ngroups; ++g) {
                        const int c_lo = g * p.CPS, cn = min(p.CPS, p.nchunks - c_lo);
                        for (int kw0 = 0; kw0 < p.KW; kw0 += p.TPS) {
                            mbar_wait(&empty[s], ph);
                            uint8_t *st = smem + (size_t)s * p.stage_bytes;
                            // halo mode, single stage: the A halo of this (kd, kh, chunk group) is fetched with the FIRST tap group only and stays
                            // in place while the later tap groups stream their weight tiles through the B area
                            const bool load_a = !(p.halo && p.D == 1) || kw0 == 0;
                            mbar_arrive_expect_tx(&full[s], (uint32_t)(cn * p.planes * ((load_a ? p.a_tx_bytes : 0) + p.TPS * p.b_plane_bytes)));
                            int w_start;
                            if (p.halo) w_start = p.dgrad ? rw0 + p.pw - (p.KW - 1) : rw0 - p.pw;
                            else        w_start = p.dgrad ? rw0 + p.pw - kw0 : rw0 - p.pw + kw0;
                            const int tap0 = (kd * p.KH + kh) * p.KW + kw0;
                            for (int c = 0; c < cn; ++c) {
                                uint8_t *ab = st + (size_t)c * p.a_chunk_bytes;
                                if (p.halo) {   // one box = both planes of the halo line: {chunk, voxels, planes, 1, 1}
                                    if (load_a) tma_load_5d(ab, &tmA, &full[s], (c_lo + c) * chunk_elems, w_start, 0, h_src, nb * p.SD + d_src);
                                } else {
                                    for (int pl = 0; pl < p.planes; ++pl)
                                        tma_load_5d(ab + (size_t)pl * p.a_plane_bytes, &tmA, &full[s], (c_lo + c) * chunk_elems, w_start, pl, h_src,
                                                    nb * p.SD + d_src);
                                }
                                // one box = all taps of the stage x both planes: {chunk, NT, planes, TPS}
                                tma_load_4d(st + p.a_region_bytes + (size_t)c * p.b_chunk_bytes, &tmB, &full[s], (c_lo + c) * chunk_elems, n0, 0, tap0);
                            }
                            if (++s == p.D) { s = 0; ph ^= 1; }
                        }
                    }
                }
        }
    } else if (warp == 1) {
        // =============================================================== MMA issuer
        if (elect_one()) {
            const uint32_t idesc1 = make_idesc_bf16(128, p.NT, 0, 0);
            const uint32_t idesc2 = make_idesc_bf16(128, 2 * p.NT, 0, 0);
            // descriptor template: everything but the start address (low 14 bits of the low word)
            const uint64_t dtmpl = make_smem_desc(0, 16, 8u * p.swz, layout_type_for_swizzle_bytes(p.swz));
            const int ksteps = p.swz / 32;
            const uint32_t smem_base = smem_u32(smem);
            // A chain of tcgen05.mma into ONE accumulator is latency-bound for the small N of these layers (each MMA must see the previous
            // result; measured: a CTA ran ~5x below the tensor-pipe rate and only co-resident CTAs overlapped).  So successive MMAs rotate over
            // Q independent accumulators per type (type 1: A_hi x [B_hi;B_lo], 2*NT columns; type 2: A_lo x B_hi, NT columns) and the epilogue
            // adds them up.
            int s = 0;
            uint32_t ph = 0;
            uint32_t n1 = 0, n2 = 0;          // MMAs issued per type
            uint32_t q1 = 0;                  // round-robin cursor
            for (int kd = 0; kd < p.KD; ++kd)
                for (int kh = 0; kh < p.KH; ++kh) {
                    int d_src, h_src;
                    if (!tc_step_coords(p, rd, rh0, kd, kh, d_src, h_src)) continue;
                    for (int g = 0; g < ngroups; ++g) {
                        const int cn = min(p.CPS, p.nchunks - g * p.CPS);
                        for (int kw0 = 0; kw0 < p.KW; kw0 += p.TPS) {
                            mbar_wait(&full[s], ph);
                            tc_fence_after();
                            const uint32_t st = smem_base + s * p.stage_bytes;
                            const int ktaps = min(p.TPS, p.KW - kw0);   // the last tap group of a line may be short
                            for (int k = 0; k < ktaps; ++k) {
                                const int shift = p.halo ? (p.dgrad ? p.KW - 1 - (kw0 + k) : kw0 + k) : 0;
                                for (int c = 0; c < cn; ++c) {
                                    const uint32_t a_hi = st + c * p.a_chunk_bytes + shift * p.swz;
                                    const uint32_t b_hi = st + p.a_region_bytes + c * p.b_chunk_bytes + (k * p.planes) * p.b_plane_bytes;
                                    uint64_t da = dtmpl | (uint64_t)((a_hi >> 4) & 0x3FFF);
                                    uint64_t db = dtmpl | (uint64_t)((b_hi >> 4) & 0x3FFF);
                                    uint64_t dal = dtmpl | (uint64_t)(((a_hi + p.a_plane_bytes) >> 4) & 0x3FFF);
                                    for (int j = 0; j < ksteps; ++j) {
                                        umma_bf16(tmem + q1 * acc1_cols, da, db, p.planes > 1 ? idesc2 : idesc1, n1 >= (uint32_t)Q);
                                        const uint32_t qprev = q1;
                                        ++n1;
                                        if (++q1 == (uint32_t)Q) q1 = 0;
                                        if (p.planes > 1)   // A_lo x B_hi accumulates into the hi*hi columns of the same accumulator (in-order after MMA 1)
                                            umma_bf16(tmem + qprev * acc1_cols, dal, db, idesc1, 1);
                                        da += 2; db += 2; dal += 2;          // +32 bytes along K
                                    }
                                }
                            }
                            umma_commit(&empty[s]);
                            if (++s == p.D) { s = 0; ph ^= 1; }
                        }
                    }
                }
            const uint32_t acc = n1;
            *(volatile uint32_t *)&s_n1 = n1 < (uint32_t)Q ? n1 : (uint32_t)Q;
            *(volatile uint32_t *)&s_n2 = n2 < (uint32_t)Q ? n2 : (uint32_t)Q;
            __threadfence_block();
            if (acc) {
                umma_commit(&accum_full);
            } else {   // no tap contributed (e.g. a dgrad row of a strided conv that no output touches): the result is bias / zero only
                *(volatile uint32_t *)&s_have_acc = 0;
                mbar_arrive(&accum_full);   // release: orders the flag write before the epilogue's acquire wait
            }
        }
    }
    if (warp >= 2) {
        // =============================================================== epilogue
        mbar_wait(&accum_full, 0);
        tc_fence_after();
        const bool have_acc = (*(volatile uint32_t *)&s_have_acc) != 0u;
        const uint32_t n1_used = *(volatile uint32_t *)&s_n1, n2_used = *(volatile uint32_t *)&s_n2;
        const int q = warp & 3;              // TMEM lane quarter this warp may access
        const int r = q * 32 + lane;
        const int hi_ = r / p.BW, wi = r % p.BW;
        const int rh = rh0 + hi_, rw = rw0 + wi;
        const bool valid = rh < p.RH && rw < p.RW;
        const size_t row_off = ((((size_t)nb * p.RD + rd) * p.RH + rh) * p.RW + rw) * (size_t)p.Cn;
        const bool vec4 = (p.Cn % 4 == 0);
        for (int c0 = 0; c0 < p.NT; c0 += 16) {
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = 0.f;
            if (have_acc) {
                const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
                float u[16];
                for (uint32_t a = 0; a < n1_used; ++a) {
                    tmem_ld16(lane_base + a * acc1_cols + c0, u);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] += u[j];
                    if (p.planes > 1) {
                        tmem_ld16(lane_base + a * acc1_cols + p.NT + c0, u);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] += u[j];
                    }
                }
                for (uint32_t a = 0; a < n2_used; ++a) {
                    tmem_ld16(lane_base + acc2_base + a * p.NT + c0, u);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] += u[j];
                }
            }
            if (!valid) continue;
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
                const int col = n0 + c0 + j;
                if (col >= p.Cn && !(p.out_split && col < p.out_kg)) break;
                float o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) o[k] = v[j + k] + s_bias[c0 + j + k];
                if (col < p.Cn) {
                    if (vec4) {
                        if (p.residual) {
                            const float4 rr = __ldg(reinterpret_cast<const float4 *>(p.residual + row_off + col));
                            o[0] += rr.x; o[1] += rr.y; o[2] += rr.z; o[3] += rr.w;
                        }
                        if (p.relu) { o[0] = fmaxf(o[0], 0.f); o[1] = fmaxf(o[1], 0.f); o[2] = fmaxf(o[2], 0.f); o[3] = fmaxf(o[3], 0.f); }
                        *reinterpret_cast<float4 *>(p.out + row_off + col) = make_float4(o[0], o[1], o[2], o[3]);
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (col + k >= p.Cn) break;
                            float x = o[k];
                            if (p.residual) x += __ldg(p.residual + row_off + col + k);
                            if (p.relu) x = fmaxf(x, 0.f);
                            p.out[row_off + col + k] = x;
                            o[k] = x;
                        }
                    }
                }
                if (p.out_split && col < p.out_kg) {
                    // the same values as (hi, lo) bf16 planes for the next conv: [line][plane][w][out_kg]; channels >= Cn are written as zeros
                    __align__(8) __nv_bfloat16 hi[4], lo[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float x = (col + k < p.Cn) ? o[k] : 0.f;
                        hi[k] = __float2bfloat16_rn(x);
                        lo[k] = __float2bfloat16_rn(x - __bfloat162float(hi[k]));
                    }
                    const size_t line = ((size_t)nb * p.RD + rd) * p.RH + rh;
                    const size_t so = ((line * p.planes) * (size_t)p.RW + rw) * (size_t)p.out_kg + col;
                    *reinterpret_cast<uint2 *>(p.out_split + so) = *reinterpret_cast<const uint2 *>(hi);
                    if (p.planes > 1) *reinterpret_cast<uint2 *>(p.out_split + so + (size_t)p.RW * p.out_kg) = *reinterpret_cast<const uint2 *>(lo);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, tmem_cols);
}

// ------------------------------------------------------------------------------------------------ host side
// channels of the canonical split layout in GLOBAL memory: padded to 16 only (36 -> 48).  Kernels that stage wider chunks in shared memory
// (conv_tc_kpad_smem) let the TMA box run past the tensor's channel extent: out-of-bounds elements arrive as zeros.
int conv_tc_kpad(int channels) { return ceil_div(channels, 16) * 16; }
int conv_tc_kpad_smem(int channels) { return channels <= 16 ? 16 : channels <= 32 ? 32 : ceil_div(channels, 64) * 64; }

bool conv_tcw_supported(const ConvGeom &g, int pass);
size_t conv_tcw_workspace_bytes(const ConvGeom &g, int pass, int precision);
int conv_tcw_run(const ConvGeom &g, int pass, const float *src, const float *w, const float *bias, const float *residual, float *dst, int relu,
                 int precision, void *ws, size_t ws_bytes, cudaStream_t st, const __nv_bfloat16 *presplit, __nv_bfloat16 *out_split);

bool conv_tc_wgrad_supported(const ConvGeom &g);
size_t conv_tc_wgrad_workspace_bytes(const ConvGeom &g, int precision);

bool conv_tc_supported(const ConvGeom &g, int pass) {
    if (pass == 2) return conv_tc_wgrad_supported(g);
    if (conv_tcw_supported(g, pass)) return true;
    const TcPlan pl = make_plan(g, pass);
    int a, b, c, d;
    return pl.ok && plan_stages(pl, g.kw, 2, a, b, c, d) && tmap_encode_fn() != nullptr;
}


// number of weight replicas: as many as fit in ~16 MB, at most 16
static int weight_reps(const TcPlan &pl, int T, int planes) {
    const size_t one = (size_t)planes * T * pl.Np * pl.Kp * 2;
    (void)one;
    return 1;   // measured on B200: replication does not change the kernel time (the weight tiles are not an L2 hot spot); kept for experiments
}

size_t conv_tc_workspace_bytes(const ConvGeom &g, int pass, int precision) {
    if (pass == 2) return conv_tc_wgrad_workspace_bytes(g, precision);
    const size_t tcw = conv_tcw_workspace_bytes(g, pass, precision);
    const TcPlan pl = make_plan(g, pass);
    if (!pl.ok) return tcw;
    const int planes = precision == 1 ? 1 : 2;
    const int T = g.kd * g.kh * g.kw;
    const size_t old = align_up((size_t)planes * pl.src_rows * pl.Kg * 2, 1024) + align_up((size_t)weight_reps(pl, T, planes) * planes * T * pl.Np * pl.Kp * 2, 1024) + 2048;
    return old > tcw ? old : tcw;
}

// presplit != nullptr: the A operand is already in split form (layout of split_rows_kernel with inter_w = SW) and `src` is ignored
int conv_tc_run(const ConvGeom &g, int pass, const float *src, const float *w, const float *bias, const float *residual, float *dst,
                int relu, int precision, void *ws, size_t ws_bytes, cudaStream_t st, const __nv_bfloat16 *presplit, __nv_bfloat16 *out_split) {
    if (conv_tcw_supported(g, pass))   // the tap-stacked kernel (conv3d_tcw.cu) where it wins
        return conv_tcw_run(g, pass, src, w, bias, residual, dst, relu, precision, ws, ws_bytes, st, presplit, out_split);
    const TcPlan pl = make_plan(g, pass);
    if (!pl.ok) return MDT_EUNSUPPORTED;
    if (ws_bytes < conv_tc_workspace_bytes(g, pass, precision)) return MDT_EWORKSPACE;
    const int planes = precision == 1 ? 1 : 2;
    const int T = g.kd * g.kh * g.kw;
    const bool dgrad = pass == 1;
    uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~uintptr_t(1023));
    __nv_bfloat16 *xs = presplit ? const_cast<__nv_bfloat16 *>(presplit) : reinterpret_cast<__nv_bfloat16 *>(base);
    __nv_bfloat16 *wp = reinterpret_cast<__nv_bfloat16 *>(base + align_up((size_t)planes * pl.src_rows * pl.Kg * 2, 1024));

    {   // operand preparation
        const long long total = pl.src_rows * (pl.Kg / 8);
        long long blocks = ceil_div<long long>(total, 256);
        if (blocks > (long long)num_sms() * 32) blocks = (long long)num_sms() * 32;
        if (!presplit) split_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, xs, pl.src_rows, pl.Kc, pl.Kg, planes, pl.SW, nullptr, nullptr, nullptr);
        int rc = launch_status();
        if (rc) return rc;
        const long long wt = (long long)T * pl.Np * pl.Kp;
        pack_weights_tc_kernel<<<(unsigned)ceil_div<long long>(wt, 256), 256, 0, st>>>(w, wp, g.cout, g.cin, T, pl.Np, pl.Kp, planes, dgrad ? 1 : 0,
                                                                                      weight_reps(pl, T, planes));
        if ((rc = launch_status())) return rc;
    }

    TcConvParams p{};
    p.NB = g.n; p.RD = pl.RD; p.RH = pl.RH; p.RW = pl.RW; p.SD = pl.SD; p.SH = pl.SH;
    p.KD = g.kd; p.KH = g.kh; p.KW = g.kw; p.sd = g.sd; p.sh = g.sh; p.pd = g.pd; p.ph = g.ph; p.pw = g.pw;
    p.dgrad = dgrad ? 1 : 0;
    p.Cn = pl.Nc; p.Np = pl.Np; p.NT = pl.NT; p.nchunks = pl.nchunks; p.swz = pl.swz; p.planes = planes;
    p.BW = pl.BW; p.BH = pl.BH; p.halo = pl.halo;
    p.tiles_w = ceil_div(pl.RW, pl.BW); p.tiles_h = ceil_div(pl.RH, pl.BH);
    const int rows_loaded = a_rows_loaded(pl, g.kw);
    p.a_plane_bytes = rows_loaded * pl.swz;                       // plane 1 follows plane 0 directly (one TMA box delivers both)
    p.a_chunk_bytes = a_chunk_bytes_of(pl, g.kw, planes);
    p.b_plane_bytes = pl.NT * pl.swz;
    if (!plan_stages(pl, g.kw, planes, p.CPS, p.TPS, p.D, p.stage_bytes)) return MDT_EUNSUPPORTED;
    p.b_chunk_bytes = (int)align_up((size_t)p.TPS * planes * p.b_plane_bytes, 1024);
    p.a_region_bytes = p.CPS * p.a_chunk_bytes;
    p.relu = relu; p.bias = bias; p.residual = residual; p.out = dst;
    p.out_split = out_split; p.out_kg = conv_tc_kpad(pl.Nc);
    // Accumulator chains.  For speed one chain is enough (the accumulate dependency is not the limiter), but the tensor core's fp32 accumulation
    // truncates: the error of a TMEM accumulator grows ~1e-7 of the result per chained MMA (tools/wgrad_precision.py).  3x3x3 layers chain
    // <= 216 MMAs (2e-5); the 7x7x7 stem conv would chain 1372, so its MMAs rotate over Q accumulators that the epilogue adds in IEEE fp32.
    {
        const int chain = g.kd * g.kh * g.kw * pl.nchunks * (pl.swz / 32) * (planes > 1 ? 2 : 1);
        p.Q = (chain + 511) / 512;
        const int acc1 = (planes > 1 ? 2 : 1) * pl.NT;
        while (p.Q > 1 && p.Q * acc1 > 128) --p.Q;   // keep the TMEM footprint at <= 128 columns (4 CTAs per SM)
        if (p.Q < 1) p.Q = 1;
    }
    if (const char *e = getenv("MDT_TC_Q")) { const int v = atoi(e); if (v >= 1 && v <= p.Q) p.Q = v; }
    p.wreps = weight_reps(pl, T, planes);

    // tensor maps.  A: bf16 [N*SD][SH][plane][SW][Kg] (N and D merged: out-of-range d taps are skipped explicitly, never fetched; channel
    //               chunks past Kg are TMA zero fill);
    //               B: bf16 [T][plane][Np][Kp]
    CUtensorMap tmA, tmB;
    {
        const uint64_t line = (uint64_t)pl.SW * pl.Kg * 2;
        const uint64_t dims[5] = {(uint64_t)pl.Kg, (uint64_t)pl.SW, (uint64_t)planes, (uint64_t)pl.SH, (uint64_t)g.n * pl.SD};
        const uint64_t strides[4] = {(uint64_t)pl.Kg * 2, line, line * planes, line * planes * pl.SH};
        const uint32_t box[5] = {(uint32_t)(pl.swz / 2), (uint32_t)(pl.halo ? rows_loaded : pl.BW), (uint32_t)(pl.halo ? planes : 1), (uint32_t)pl.BH, 1u};
        if (!encode_bf16_tmap(&tmA, xs, 5, dims, strides, box, pl.swz)) return MDT_EDRIVER;
        const uint64_t bdims[4] = {(uint64_t)pl.Kp, (uint64_t)pl.Np, (uint64_t)planes, (uint64_t)T};
        const uint64_t bstr[3] = {(uint64_t)pl.Kp * 2, (uint64_t)pl.Np * pl.Kp * 2, (uint64_t)planes * pl.Np * pl.Kp * 2};
        const uint32_t bbox[4] = {(uint32_t)(pl.swz / 2), (uint32_t)pl.NT, (uint32_t)planes, (uint32_t)p.TPS};
        if (!encode_bf16_tmap(&tmB, wp, 4, bdims, bstr, bbox, pl.swz)) return MDT_EDRIVER;
    }
    p.a_tx_bytes = rows_loaded * pl.swz;   // per plane; expect_tx must equal the bytes the TMA boxes deliver

    const size_t smem = (size_t)p.D * p.stage_bytes + 1024;
    static bool attr[kMaxDevices] = {};
    if (!ensure_smem_attr(conv_tc_kernel, 220 * 1024, attr)) return MDT_EDRIVER;
    dim3 grid((unsigned)((long long)g.n * pl.RD * p.tiles_h * p.tiles_w), pl.n_tiles_n);
    conv_tc_kernel<<<grid, kTcThreads, smem, st>>>(tmA, tmB, p);
    return launch_status();
}

int conv_tc_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, const float *residual, float *y, int relu, int precision,
                  void *ws, size_t ws_bytes, cudaStream_t st) {
    return conv_tc_run(g, 0, x, w, bias, residual, y, relu, precision, ws, ws_bytes, st, nullptr, nullptr);
}
int conv_tc_fprop_presplit(const ConvGeom &g, const void *x_split, const float *w, const float *bias, const float *residual, float *y, int relu,
                           int precision, void *ws, size_t ws_bytes, cudaStream_t st, void *y_split) {
    return conv_tc_run(g, 0, nullptr, w, bias, residual, y, relu, precision, ws, ws_bytes, st, reinterpret_cast<const __nv_bfloat16 *>(x_split),
                       reinterpret_cast<__nv_bfloat16 *>(y_split));
}
int conv_tc_dgrad(const ConvGeom &g, const float *dy, const float *w, float *dx, int precision, void *ws, size_t ws_bytes, cudaStream_t st) {
    return conv_tc_run(g, 1, dy, w, nullptr, nullptr, dx, 0, precision, ws, ws_bytes, st, nullptr, nullptr);
}

}  // namespace mdt

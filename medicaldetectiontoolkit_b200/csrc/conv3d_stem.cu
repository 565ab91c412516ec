// Direct kernels for the network stem (Cin <= 4, e.g. the 1-channel image -> 18 feature maps 3x3x3 conv of models/backbone.py:48):
// with one input channel the GEMM view has K = 27 — padding it to tensor-core shape wastes 94 % of every MMA and the operand split writes
// 16x the input — so this layer is bandwidth-bound SIMT work: each output voxel reads its 27*Cin neighbours (L1/L2 hits) and writes Cout
// floats.  fprop: one thread per voxel, weights broadcast from shared memory, the warp's 32 x Cout outputs staged through shared memory
// for fully coalesced stores.  wgrad: one block per output line, dy line + x halo lines in shared memory, each thread owns a few
// (cout, tap) accumulators, block-level partials combined with one atomicAdd per element per block.
#include "conv3d_common.cuh"
#include <cstdlib>

namespace mdt {

constexpr int kStemMaxCout = 32, kStemMaxTaps = 27, kStemMaxCin = 4;

__global__ void __launch_bounds__(256) stem_fprop_kernel(ConvGeom g, const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ bias,
                                                        float *__restrict__ y, int relu) {
    __shared__ float s_w[kStemMaxTaps * kStemMaxCin * kStemMaxCout];   // [tap][ci][co]
    __shared__ float s_b[kStemMaxCout];
    __shared__ float s_out[8][32 * kStemMaxCout];
    const int T = g.kd * g.kh * g.kw;
    for (int i = threadIdx.x; i < T * g.cin * g.cout; i += blockDim.x) {
        const int co = i % g.cout, ci = (i / g.cout) % g.cin, t = i / (g.cout * g.cin);
        s_w[i] = w[((size_t)co * g.cin + ci) * T + t];
    }
    if ((int)threadIdx.x < g.cout) s_b[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
    __syncthreads();
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * 256; base < M; base += (long long)gridDim.x * 256) {
        const long long m = base + threadIdx.x;
        float acc[kStemMaxCout];
#pragma unroll
        for (int c = 0; c < kStemMaxCout; ++c) acc[c] = 0.f;
        if (m < M) {
            int ow = m % g.ow; long long r = m / g.ow;
            int oh = r % g.oh; r /= g.oh;
            int od = r % g.od;
            const int n = (int)(r / g.od);
            for (int kd = 0; kd < g.kd; ++kd) {
                const int d = od * g.sd - g.pd + kd;
                if (d < 0 || d >= g.d) continue;
                for (int kh = 0; kh < g.kh; ++kh) {
                    const int h = oh * g.sh - g.ph + kh;
                    if (h < 0 || h >= g.h) continue;
                    for (int kw = 0; kw < g.kw; ++kw) {
                        const int ww = ow * g.sw - g.pw + kw;
                        if (ww < 0 || ww >= g.w) continue;
                        const float *px = x + ((((long long)n * g.d + d) * g.h + h) * g.w + ww) * g.cin;
                        const float *pw = s_w + ((kd * g.kh + kh) * g.kw + kw) * g.cin * g.cout;
                        for (int ci = 0; ci < g.cin; ++ci) {
                            const float xv = __ldg(px + ci);
#pragma unroll
                            for (int c = 0; c < kStemMaxCout; ++c)
                                if (c < g.cout) acc[c] = fmaf(xv, pw[ci * g.cout + c], acc[c]);
                        }
                    }
                }
            }
        }
        // stage the warp's 32 x cout outputs and store them as one contiguous run
        float *so = s_out[warp];
#pragma unroll
        for (int c = 0; c < kStemMaxCout; ++c)
            if (c < g.cout) {
                float v = acc[c] + s_b[c];
                so[lane * g.cout + c] = relu ? fmaxf(v, 0.f) : v;
            }
        __syncwarp();
        const long long wbase = base + warp * 32;
        const long long nvalid = (M - wbase) < 32 ? (M - wbase) : 32;
        if (nvalid > 0)
            for (int i = lane; i < (int)nvalid * g.cout; i += 32) y[wbase * g.cout + i] = so[i];
        __syncwarp();
    }
}

// one block per (n, od, oh) output line; requires sw == 1.  partial[block][co][ci][tap]: the weight gradient of the block's lines
__global__ void __launch_bounds__(256) stem_wgrad_kernel(ConvGeom g, const float *__restrict__ x, const float *__restrict__ dy, float *__restrict__ partial,
                                                        long long lines_per_block) {
    extern __shared__ float smem[];
    const int T = g.kd * g.kh * g.kw;
    const int XW = g.ow + g.kw - 1;                       // halo line length
    float *s_dy = smem;                                   // [ow][cout]
    float *s_x = smem + (size_t)g.ow * g.cout;            // [kd*kh][XW][cin]
    const int npairs = g.cout * g.cin * T;
    constexpr int kPer = 8;                               // (cout, ci, tap) accumulators per thread: supports up to 2048 weights
    float acc[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) acc[q] = 0.f;
    const long long nlines = (long long)g.n * g.od * g.oh;
    const long long l0 = (long long)blockIdx.x * lines_per_block, l1 = min(nlines, l0 + lines_per_block);
    for (long long line = l0; line < l1; ++line) {
        const int oh = line % g.oh; long long r = line / g.oh;
        const int od = r % g.od;
        const int n = (int)(r / g.od);
        __syncthreads();
        for (int i = threadIdx.x; i < g.ow * g.cout; i += blockDim.x) s_dy[i] = __ldg(dy + line * g.ow * g.cout + i);
        for (int i = threadIdx.x; i < g.kd * g.kh * XW * g.cin; i += blockDim.x) {
            const int ci = i % g.cin; int t = i / g.cin;
            const int xw = t % XW; t /= XW;
            const int kh = t % g.kh, kd = t / g.kh;
            const int d = od * g.sd - g.pd + kd, h = oh * g.sh - g.ph + kh, ww = xw - g.pw;
            s_x[i] = (d >= 0 && d < g.d && h >= 0 && h < g.h && ww >= 0 && ww < g.w)
                         ? __ldg(x + ((((long long)n * g.d + d) * g.h + h) * g.w + ww) * g.cin + ci) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kPer; ++q) {
            const int pidx = threadIdx.x + q * 256;
            if (pidx >= npairs) break;
            const int t = pidx % T, ci = (pidx / T) % g.cin, co = pidx / (T * g.cin);
            const int kw = t % g.kw, kdh = t / g.kw;
            const float *px = s_x + ((size_t)kdh * XW + kw) * g.cin + ci;
            float a = 0.f;
            for (int v = 0; v < g.ow; ++v) a = fmaf(s_dy[v * g.cout + co], px[(size_t)v * g.cin], a);
            acc[q] += a;
        }
    }
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const int pidx = threadIdx.x + q * 256;
        if (pidx < npairs) partial[(long long)blockIdx.x * npairs + pidx] = acc[q];   // dw layout [co][ci][tap] == pidx order
    }
}

// ---- specialisations for the layer that actually is the stem of every BASELINE config: Cin = 1, 3x3x3, stride 1, pad 1 (models/backbone.py:48).
// The generic kernels above are instruction-bound (ncu: issue 87 % / 60 %, 0.61 / 0.96 ms for 2x128^3): one shared-memory load per FMA.
//
// fprop: taps fully unrolled, weights padded to a multiple of 4 output channels and read as 128-bit broadcasts (0.25 loads per FMA).
template <int CP>   // padded cout (multiple of 4)
__global__ void __launch_bounds__(256) stem_fprop_c1k3_kernel(ConvGeom g, const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ bias,
                                                             float *__restrict__ y, int relu) {
    __shared__ __align__(16) float s_w[27 * CP];   // [tap][co padded]
    __shared__ float s_b[CP];
    __shared__ float s_out[8][32 * CP];
    for (int i = threadIdx.x; i < 27 * CP; i += blockDim.x) {
        const int co = i % CP, t = i / CP;
        s_w[i] = co < g.cout ? w[(size_t)co * 27 + t] : 0.f;
    }
    if ((int)threadIdx.x < CP) s_b[threadIdx.x] = (bias && (int)threadIdx.x < g.cout) ? bias[threadIdx.x] : 0.f;
    __syncthreads();
    const long long M = (long long)g.n * g.d * g.h * g.w;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * 256; base < M; base += (long long)gridDim.x * 256) {
        const long long m = base + threadIdx.x;
        float acc[CP];
#pragma unroll
        for (int c = 0; c < CP; ++c) acc[c] = 0.f;
        if (m < M) {
            const int ow = (int)(m % g.w); long long r = m / g.w;
            const int oh = (int)(r % g.h); r /= g.h;
            const int od = (int)(r % g.d);
            const int n = (int)(r / g.d);
            const float *xn = x + (long long)n * g.d * g.h * g.w;
#pragma unroll
            for (int kd = 0; kd < 3; ++kd) {
                const int d = od - 1 + kd;
                const bool okd = d >= 0 && d < g.d;
#pragma unroll
                for (int kh = 0; kh < 3; ++kh) {
                    const int h = oh - 1 + kh;
                    const bool okh = okd && h >= 0 && h < g.h;
                    const float *row = xn + ((long long)(okh ? d : 0) * g.h + (okh ? h : 0)) * g.w;
#pragma unroll
                    for (int kw = 0; kw < 3; ++kw) {
                        const int ww = ow - 1 + kw;
                        const float xv = (okh && ww >= 0 && ww < g.w) ? __ldg(row + ww) : 0.f;
                        const float4 *pw = reinterpret_cast<const float4 *>(s_w + ((kd * 3 + kh) * 3 + kw) * CP);
#pragma unroll
                        for (int q = 0; q < CP / 4; ++q) {
                            const float4 wv = pw[q];
                            acc[4 * q] = fmaf(xv, wv.x, acc[4 * q]);
                            acc[4 * q + 1] = fmaf(xv, wv.y, acc[4 * q + 1]);
                            acc[4 * q + 2] = fmaf(xv, wv.z, acc[4 * q + 2]);
                            acc[4 * q + 3] = fmaf(xv, wv.w, acc[4 * q + 3]);
                        }
                    }
                }
            }
        }
        float *so = s_out[warp];
#pragma unroll
        for (int c = 0; c < CP; ++c)
            if (c < g.cout) {
                const float v = acc[c] + s_b[c];
                so[lane * g.cout + c] = relu ? fmaxf(v, 0.f) : v;
            }
        __syncwarp();
        const long long wbase = base + warp * 32;
        const long long nvalid = (M - wbase) < 32 ? (M - wbase) : 32;
        if (nvalid > 0)
            for (int i = lane; i < (int)nvalid * g.cout; i += 32) y[wbase * g.cout + i] = so[i];
        __syncwarp();
    }
}

// wgrad: dw[co][tap] = sum_v dy[v][co] * x[v + tap].  A block works on kStemWgLines output lines at once; within a line a thread owns a
// 3 (co) x 3 (kw) register tile of one (kd, kh) pair and slides along the line: per voxel 3 dy loads + 1 new x value feed 9 FMAs (the generic
// kernel: 2 loads per FMA).  Partials are kept in registers over all lines of the block; the kStemWgLines threads of an element are summed
// in shared memory in line order and written to partial[block][co][tap].
constexpr int kStemWgLines = 4, kStemWgCoT = 3;
__global__ void __launch_bounds__(256) stem_wgrad_c1k3_kernel(ConvGeom g, const float *__restrict__ x, const float *__restrict__ dy, float *__restrict__ partial,
                                                             long long groups_per_block) {
    extern __shared__ float smem[];
    const int W = g.w, XW = W + 2;
    const int cog = ceil_div(g.cout, kStemWgCoT);            // co groups (6 for 18 channels)
    const int per_line = cog * 9;                            // threads per line: (co group, kd*3 + kh)
    float *s_dy = smem;                                      // [line][W][cout]
    float *s_x = smem + (size_t)kStemWgLines * W * g.cout;   // [line][9][XW]
    const int lt = threadIdx.x / per_line, li = threadIdx.x % per_line;   // which line of the group, which tile inside the line
    const bool active = lt < kStemWgLines;
    const int cg = li / 9, kdh = li % 9;
    float acc[kStemWgCoT][3];
#pragma unroll
    for (int a = 0; a < kStemWgCoT; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) acc[a][b] = 0.f;
    const long long nlines = (long long)g.n * g.d * g.h;
    const long long ngroups = ceil_div<long long>(nlines, kStemWgLines);
    const long long g0 = (long long)blockIdx.x * groups_per_block, g1 = min(ngroups, g0 + groups_per_block);
    for (long long grp = g0; grp < g1; ++grp) {
        __syncthreads();
        // stage dy lines (contiguous in memory: lines are consecutive) and the 9 x halo lines of each output line
        const long long line0 = grp * kStemWgLines;
        const long long left_ = nlines - line0;
        const int nl = left_ < kStemWgLines ? (int)left_ : kStemWgLines;
        for (int i = threadIdx.x; i < nl * W * g.cout; i += blockDim.x) s_dy[i] = __ldg(dy + line0 * W * g.cout + i);
        for (int i = threadIdx.x; i < nl * 9 * XW; i += blockDim.x) {
            const int xw = i % XW; int t = i / XW;
            const int kh = t % 3; t /= 3;
            const int kd = t % 3; const int l = t / 3;
            const long long line = line0 + l;
            const int oh = (int)(line % g.h); const long long r = line / g.h;
            const int od = (int)(r % g.d); const int n = (int)(r / g.d);
            const int d = od - 1 + kd, h = oh - 1 + kh, ww = xw - 1;
            s_x[i] = (d >= 0 && d < g.d && h >= 0 && h < g.h && ww >= 0 && ww < W) ? __ldg(x + (((long long)n * g.d + d) * g.h + h) * W + ww) : 0.f;
        }
        __syncthreads();
        if (active && lt < nl) {
            const float *py = s_dy + (size_t)lt * W * g.cout + cg * kStemWgCoT;
            const float *px = s_x + ((size_t)lt * 9 + kdh) * XW;
            const int c1 = min(kStemWgCoT, g.cout - cg * kStemWgCoT);
            float x0 = px[0], x1 = px[1];
            for (int v = 0; v < W; ++v) {
                const float x2 = px[v + 2];
#pragma unroll
                for (int a = 0; a < kStemWgCoT; ++a) {
                    const float d_ = a < c1 ? py[(size_t)v * g.cout + a] : 0.f;
                    acc[a][0] = fmaf(d_, x0, acc[a][0]);
                    acc[a][1] = fmaf(d_, x1, acc[a][1]);
                    acc[a][2] = fmaf(d_, x2, acc[a][2]);
                }
                x0 = x1; x1 = x2;
            }
        }
    }
    __syncthreads();
    float *s_red = smem;                                     // [line][per_line][kStemWgCoT * 3]
    if (active) {
#pragma unroll
        for (int a = 0; a < kStemWgCoT; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) s_red[((size_t)lt * per_line + li) * (kStemWgCoT * 3) + a * 3 + b] = acc[a][b];
    }
    __syncthreads();
    if ((int)threadIdx.x < per_line) {
#pragma unroll
        for (int a = 0; a < kStemWgCoT; ++a) {
            const int co = cg * kStemWgCoT + a;
            if (co >= g.cout) continue;
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                float t = 0.f;
                for (int l = 0; l < kStemWgLines; ++l) t += s_red[((size_t)l * per_line + li) * (kStemWgCoT * 3) + a * 3 + b];
                partial[(long long)blockIdx.x * g.cout * 27 + (size_t)co * 27 + kdh * 3 + b] = t;   // dw [co][1][kd][kh][kw]
            }
        }
    }
}

static bool stem_c1k3(const ConvGeom &g) {
    return g.cin == 1 && g.kd == 3 && g.kh == 3 && g.kw == 3 && g.sd == 1 && g.sh == 1 && g.sw == 1 && g.pd == 1 && g.ph == 1 && g.pw == 1 && g.cout <= 32;
}

bool conv_stem_supported(const ConvGeom &g, int pass) {
    if (g.cin > kStemMaxCin || g.cout > kStemMaxCout || g.kd * g.kh * g.kw > kStemMaxTaps) return false;
    if (pass == 0) return true;
    if (pass == 2) {
        const size_t smem = ((size_t)g.ow * g.cout + (size_t)g.kd * g.kh * (g.ow + g.kw - 1) * g.cin) * sizeof(float);
        return g.sw == 1 && g.cout * g.cin * g.kd * g.kh * g.kw <= 2048 && smem <= 96 * 1024;
    }
    return false;   // dgrad of the stem is never needed (the image has no gradient); generic kernels cover it if it is
}

int conv_stem_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, float *y, int relu, cudaStream_t st) {
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    long long blocks = ceil_div<long long>(M, 256);
    if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
    if (stem_c1k3(g) && !getenv("MDT_STEM_GENERIC")) {
        const int cp = ceil_div(g.cout, 4) * 4;
        if (cp <= 20) stem_fprop_c1k3_kernel<20><<<(unsigned)blocks, 256, 0, st>>>(g, x, w, bias, y, relu);
        else stem_fprop_c1k3_kernel<32><<<(unsigned)blocks, 256, 0, st>>>(g, x, w, bias, y, relu);
        return launch_status();
    }
    stem_fprop_kernel<<<(unsigned)blocks, 256, 0, st>>>(g, x, w, bias, y, relu);
    return launch_status();
}

// launch shape of the weight gradient: the c1k3 kernel (c1k3 = true) or the generic one, its block count and dynamic shared memory
struct StemWgradPlan {
    bool c1k3;
    long long blocks, per_block;
    size_t smem;
};

static StemWgradPlan stem_wgrad_plan(const ConvGeom &g) {
    StemWgradPlan p;
    const long long nlines = (long long)g.n * g.od * g.oh;
    const int per_line = ceil_div(g.cout, kStemWgCoT) * 9;
    const size_t stage3 = (size_t)kStemWgLines * ((size_t)g.w * g.cout + 9 * (g.w + 2)) * sizeof(float);
    const size_t red3 = (size_t)kStemWgLines * per_line * kStemWgCoT * 3 * sizeof(float);   // the final per-block combination reuses the buffer
    p.smem = stage3 > red3 ? stage3 : red3;
    p.c1k3 = stem_c1k3(g) && per_line * kStemWgLines <= 256 && p.smem <= 96 * 1024 && !getenv("MDT_STEM_GENERIC");
    if (p.c1k3) {
        const long long ngroups = ceil_div<long long>(nlines, kStemWgLines);
        p.blocks = (long long)num_sms() * 4;
        if (p.blocks > ngroups) p.blocks = ngroups;
        p.per_block = ceil_div<long long>(ngroups, p.blocks);
    } else {
        p.blocks = (long long)num_sms() * 8;
        if (p.blocks > nlines) p.blocks = nlines;
        p.per_block = ceil_div<long long>(nlines, p.blocks);
        p.smem = ((size_t)g.ow * g.cout + (size_t)g.kd * g.kh * (g.ow + g.kw - 1) * g.cin) * sizeof(float);
    }
    return p;
}

size_t conv_stem_wgrad_workspace_bytes(const ConvGeom &g) {
    const StemWgradPlan p = stem_wgrad_plan(g);
    const size_t w = sizeof(float) * (size_t)p.blocks * g.cout * g.cin * g.kd * g.kh * g.kw, b = conv_bias_grad_workspace_bytes(g);
    return w > b ? w : b;
}

int conv_stem_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (!ws || ws_bytes < conv_stem_wgrad_workspace_bytes(g)) return MDT_EWORKSPACE;
    const StemWgradPlan p = stem_wgrad_plan(g);
    float *partial = reinterpret_cast<float *>(ws);
    if (p.c1k3) {
        static bool attr3[kMaxDevices] = {};
        if (!ensure_smem_attr(stem_wgrad_c1k3_kernel, 96 * 1024, attr3)) return MDT_EDRIVER;
        stem_wgrad_c1k3_kernel<<<(unsigned)p.blocks, 256, p.smem, st>>>(g, x, dy, partial, p.per_block);
    } else {
        static bool attr[kMaxDevices] = {};
        if (!ensure_smem_attr(stem_wgrad_kernel, 96 * 1024, attr)) return MDT_EDRIVER;
        stem_wgrad_kernel<<<(unsigned)p.blocks, 256, p.smem, st>>>(g, x, dy, partial, p.per_block);
    }
    int rc = launch_status();
    if (rc) return rc;
    if ((rc = reduce_partials(partial, (int)p.blocks, (long long)g.cout * g.cin * g.kd * g.kh * g.kw, dw, st))) return rc;
    if (db) return conv_bias_grad(g, dy, db, ws, ws_bytes, st);   // reuses the workspace after the reduction (same stream)
    return MDT_OK;
}

}  // namespace mdt

// conv3d fp32 SIMT kernels (algo 1): generic implicit-GEMM forward / data-gradient and split-K weight-gradient for NDHWC activations.
//
// This is the shape-complete path (any kernel size, stride, padding, channel count): it serves the layers the tcgen05 path does not
// cover (Cin = 1 stem, strided 1x1x1 / k7 convs, > 256 channels) and is the in-library numerical cross-check of the tensor-core path.
// It replaces the cuDNN conv3d the reference reaches through nn.Conv3d (utils/model_utils.py:762; call sites models/backbone.py:27-206).
//
// GEMM view (fprop): M = N*Do*Ho*Wo output voxels, N = Cout, K = taps*Cin;  y[m, co] = sum_{tap, ci} x[src(m, tap), ci] * w[co, ci, tap].
// dgrad is the same kernel with the gather `src = (o + p - k) / s` (valid iff divisible) and the roles of Cin/Cout swapped.
// wgrad: dw[co, ci, tap] = sum_m dy[m, co] * x[src(m, tap), ci], split over m across CTAs, reduced with fp32 atomics.
#include "conv3d_common.cuh"
#include <algorithm>

namespace mdt {

// ---------------------------------------------------------------- weight packing: [Cout, Cin, T] -> B[tap][K][N] with N contiguous
// mode 0 (fprop): K = Cin,  N = Cout, B[t][ci][co] = w[co][ci][t]
// mode 1 (dgrad): K = Cout, N = Cin,  B[t][co][ci] = w[co][ci][t]   (the tap is NOT mirrored: the dgrad gather handles the geometry)
__global__ void pack_weights_simt(const float *__restrict__ w, float *__restrict__ out, int cout, int cin, int taps, int mode) {
    const int total = cout * cin * taps;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int t, k, n;
        if (mode == 0) { n = i % cout; k = (i / cout) % cin; t = i / (cout * cin); out[i] = w[((size_t)n * cin + k) * taps + t]; }
        else           { n = i % cin;  k = (i / cin) % cout; t = i / (cout * cin); out[i] = w[((size_t)k * cin + n) * taps + t]; }
    }
}

constexpr int BM = 128, BN = 64, BK = 8, TM = 8, TN = 4;  // 256 threads, each TM x TN outputs

// DGRAD = false: rows are output voxels of the forward conv, gather reads x.   DGRAD = true: rows are INPUT voxels, gather reads dy.
template <bool DGRAD>
__global__ void __launch_bounds__(256) conv_igemm_simt(ConvGeom g, const float *__restrict__ src, const float *__restrict__ wpk,
                                                      const float *__restrict__ bias, const float *__restrict__ residual,
                                                      float *__restrict__ dst, int relu) {
    // rows: (n, a, b, c) over the "row space" RD x RH x RW; K channels CK; N channels CN
    const int RD = DGRAD ? g.d : g.od, RH = DGRAD ? g.h : g.oh, RW = DGRAD ? g.w : g.ow;
    const int SD = DGRAD ? g.od : g.d, SH = DGRAD ? g.oh : g.h, SW = DGRAD ? g.ow : g.w;  // source extent
    const int CK = DGRAD ? g.cout : g.cin, CN = DGRAD ? g.cin : g.cout;
    const long long M = (long long)g.n * RD * RH * RW;
    const int taps = g.kd * g.kh * g.kw;

    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN];
    __shared__ int row_n[BM], row_a[BM], row_b[BM], row_c[BM];

    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int tid = threadIdx.x;
    if (tid < BM) {
        long long m = m0 + tid;
        if (m < M) {
            int c = m % RW; long long r = m / RW;
            int b = r % RH; r /= RH;
            int a = r % RD; r /= RD;
            row_n[tid] = (int)r; row_a[tid] = a; row_b[tid] = b; row_c[tid] = c;
        } else {
            row_n[tid] = -1; row_a[tid] = row_b[tid] = row_c[tid] = 0;
        }
    }
    __syncthreads();

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    const int tx = tid % 16, ty = tid / 16;       // tx -> N (4 cols each), ty -> M (8 rows each)
    const int a_row = tid / 2, a_k = (tid % 2) * 4;  // A loader: 128 rows x 8 k, 4 consecutive k per thread
    const int b_k = tid / 32, b_n = (tid % 32) * 2;  // B loader: 8 k x 64 n, 2 consecutive n per thread

    for (int t = 0; t < taps; ++t) {
        const int kw_ = t % g.kw, kh_ = (t / g.kw) % g.kh, kd_ = t / (g.kw * g.kh);
        // source voxel of this thread's A row for this tap
        long long src_off = -1;
        {
            const int n = row_n[a_row];
            if (n >= 0) {
                int sa, sb, sc; bool ok = true;
                if (!DGRAD) {
                    sa = row_a[a_row] * g.sd - g.pd + kd_; sb = row_b[a_row] * g.sh - g.ph + kh_; sc = row_c[a_row] * g.sw - g.pw + kw_;
                } else {
                    const int ta = row_a[a_row] + g.pd - kd_, tb = row_b[a_row] + g.ph - kh_, tc = row_c[a_row] + g.pw - kw_;
                    ok = (ta % g.sd == 0) && (tb % g.sh == 0) && (tc % g.sw == 0) && ta >= 0 && tb >= 0 && tc >= 0;
                    sa = ta / g.sd; sb = tb / g.sh; sc = tc / g.sw;
                }
                if (ok && sa >= 0 && sa < SD && sb >= 0 && sb < SH && sc >= 0 && sc < SW)
                    src_off = ((((long long)n * SD + sa) * SH + sb) * SW + sc) * CK;
            }
        }
        const float *wt = wpk + (size_t)t * CK * CN;
        for (int k0 = 0; k0 < CK; k0 += BK) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = k0 + a_k + q;
                As[a_k + q][a_row] = (src_off >= 0 && k < CK) ? __ldg(src + src_off + k) : 0.f;
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int k = k0 + b_k, n = n0 + b_n + q;
                Bs[b_k][b_n + q] = (k < CK && n < CN) ? __ldg(wt + (size_t)k * CN + n) : 0.f;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < BK; ++k) {
                float a[TM], b[TN];
#pragma unroll
                for (int i = 0; i < TM; ++i) a[i] = As[k][ty * TM + i];
#pragma unroll
                for (int j = 0; j < TN; ++j) b[j] = Bs[k][tx * TN + j];
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            __syncthreads();
        }
    }
    // epilogue: bias, residual, ReLU
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const long long m = m0 + ty * TM + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int n = n0 + tx * TN + j;
            if (n >= CN) continue;
            float v = acc[i][j];
            if (bias) v += __ldg(bias + n);
            if (residual) v += __ldg(residual + m * CN + n);
            if (relu) v = fmaxf(v, 0.f);
            dst[m * CN + n] = v;
        }
    }
}

// wgrad: grid (tap, m-split, ci-tile * co-tile).  Tile 32 (ci) x 64 (co), BKW voxels per step, 256 threads each 2 x 4.
constexpr int WCI = 32, WCO = 64, BKW = 32;

// partial[split][co][ci][tap]: the weight gradient of the rows of one split (blockIdx.y); reduce_partials sums the splits
__global__ void __launch_bounds__(256) conv_wgrad_simt(ConvGeom g, const float *__restrict__ x, const float *__restrict__ dy,
                                                      float *__restrict__ partial, long long rows_per_split) {
    const int taps = g.kd * g.kh * g.kw;
    const int t = blockIdx.x;
    const int kw_ = t % g.kw, kh_ = (t / g.kw) % g.kh, kd_ = t / (g.kw * g.kh);
    const int co_tiles = ceil_div(g.cout, WCO);
    const int ci0 = (blockIdx.z / co_tiles) * WCI, co0 = (blockIdx.z % co_tiles) * WCO;
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    const long long m_begin = (long long)blockIdx.y * rows_per_split;
    const long long m_end = min(M, m_begin + rows_per_split);

    __shared__ float Xs[BKW][WCI + 1];
    __shared__ float Ys[BKW][WCO];
    __shared__ long long xoff[BKW];

    const int tid = threadIdx.x;
    const int tci = (tid / 16) * 2, tco = (tid % 16) * 4;
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};

    for (long long mb = m_begin; mb < m_end; mb += BKW) {
        if (tid < BKW) {
            const long long m = mb + tid;
            long long off = -1;
            if (m < m_end) {
                int c = m % g.ow; long long r = m / g.ow;
                int b = r % g.oh; r /= g.oh;
                int a = r % g.od; r /= g.od;
                const int sa = a * g.sd - g.pd + kd_, sb = b * g.sh - g.ph + kh_, sc = c * g.sw - g.pw + kw_;
                if (sa >= 0 && sa < g.d && sb >= 0 && sb < g.h && sc >= 0 && sc < g.w)
                    off = ((((long long)r * g.d + sa) * g.h + sb) * g.w + sc) * g.cin;
            }
            xoff[tid] = off;
        }
        __syncthreads();
        for (int i = tid; i < BKW * WCI; i += 256) {
            const int r = i / WCI, c = i % WCI;
            Xs[r][c] = (xoff[r] >= 0 && ci0 + c < g.cin) ? __ldg(x + xoff[r] + ci0 + c) : 0.f;
        }
        for (int i = tid; i < BKW * WCO; i += 256) {
            const int r = i / WCO, c = i % WCO;
            const long long m = mb + r;
            Ys[r][c] = (m < m_end && co0 + c < g.cout) ? __ldg(dy + m * g.cout + co0 + c) : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < BKW; ++k) {
            const float x0 = Xs[k][tci], x1 = Xs[k][tci + 1];
            const float4 yv = *reinterpret_cast<const float4 *>(&Ys[k][tco]);
            acc[0][0] = fmaf(x0, yv.x, acc[0][0]); acc[0][1] = fmaf(x0, yv.y, acc[0][1]);
            acc[0][2] = fmaf(x0, yv.z, acc[0][2]); acc[0][3] = fmaf(x0, yv.w, acc[0][3]);
            acc[1][0] = fmaf(x1, yv.x, acc[1][0]); acc[1][1] = fmaf(x1, yv.y, acc[1][1]);
            acc[1][2] = fmaf(x1, yv.z, acc[1][2]); acc[1][3] = fmaf(x1, yv.w, acc[1][3]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ci = ci0 + tci + i, co = co0 + tco + j;
            if (ci < g.cin && co < g.cout) partial[(size_t)blockIdx.y * g.cout * g.cin * taps + ((size_t)co * g.cin + ci) * taps + t] = acc[i][j];
        }
}

// db[co] = sum_m dy[m, co].  dy is read as a FLAT array: the block walks it in strides of S = (256 / cout) * cout elements, so thread t always
// owns channel t % cout and a warp's loads are 32 consecutive floats (fully coalesced, no idle channel lanes); 4 independent accumulators
// keep 4 loads in flight per thread.  Shared-memory tree over the row lanes; partial[block][co] is the sum of the block's rows.
__global__ void __launch_bounds__(256) bias_grad_kernel(const float *__restrict__ dy, float *__restrict__ partial, long long M, int cout,
                                                       long long rows_per_block) {
    __shared__ float red[256];
    const long long m0 = (long long)blockIdx.x * rows_per_block, m1 = min(M, m0 + rows_per_block);
    if (cout <= 256) {
        const int nrl = 256 / cout, active = nrl * cout;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        if ((int)threadIdx.x < active) {
            const long long e1 = m1 * cout;
            long long e = m0 * cout + threadIdx.x;
            for (; e + 3LL * active < e1; e += 4LL * active) {
                s0 += __ldg(dy + e); s1 += __ldg(dy + e + active); s2 += __ldg(dy + e + 2LL * active); s3 += __ldg(dy + e + 3LL * active);
            }
            for (; e < e1; e += active) s0 += __ldg(dy + e);
        }
        red[threadIdx.x] = (s0 + s1) + (s2 + s3);
        __syncthreads();
        if ((int)threadIdx.x < cout) {
            float t = 0.f;
            for (int r = 0; r < nrl; ++r) t += red[r * cout + threadIdx.x];
            partial[(long long)blockIdx.x * cout + threadIdx.x] = t;
        }
    } else {
        for (int c = threadIdx.x; c < cout; c += 256) {
            float s = 0.f;
            for (long long m = m0; m < m1; ++m) s += __ldg(dy + m * cout + c);
            partial[(long long)blockIdx.x * cout + c] = s;
        }
    }
}

int conv_simt_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, const float *residual, float *y, int relu, void *ws,
                    cudaStream_t st) {
    const int taps = g.kd * g.kh * g.kw;
    float *wpk = reinterpret_cast<float *>(ws);
    pack_weights_simt<<<ceil_div(g.cout * g.cin * taps, 256), 256, 0, st>>>(w, wpk, g.cout, g.cin, taps, 0);
    int rc = launch_status();
    if (rc) return rc;
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    dim3 grid((unsigned)ceil_div<long long>(M, BM), ceil_div(g.cout, BN));
    conv_igemm_simt<false><<<grid, 256, 0, st>>>(g, x, wpk, bias, residual, y, relu);
    return launch_status();
}

int conv_simt_dgrad(const ConvGeom &g, const float *dy, const float *w, float *dx, void *ws, cudaStream_t st) {
    const int taps = g.kd * g.kh * g.kw;
    float *wpk = reinterpret_cast<float *>(ws);
    pack_weights_simt<<<ceil_div(g.cout * g.cin * taps, 256), 256, 0, st>>>(w, wpk, g.cout, g.cin, taps, 1);
    int rc = launch_status();
    if (rc) return rc;
    const long long M = (long long)g.n * g.d * g.h * g.w;
    dim3 grid((unsigned)ceil_div<long long>(M, BM), ceil_div(g.cin, BN));
    conv_igemm_simt<true><<<grid, 256, 0, st>>>(g, dy, wpk, nullptr, nullptr, dx, 0);
    return launch_status();
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const float *__restrict__ partial, int nb, long long n, float *__restrict__ out) {
    // one warp per output element: lane l sums partials l, l + 32, ... in order, then a fixed butterfly combines the 32 lane sums
    const long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    if (e >= n) return;   // warp-uniform
    float s = 0.f;
    for (int b = lane; b < nb; b += 32) s += __ldg(partial + (long long)b * n + e);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[e] = s;
}

int reduce_partials(const float *partial, int nb, long long n, float *out, cudaStream_t st) {
    reduce_partials_kernel<<<(unsigned)ceil_div<long long>(n * 32, 256), 256, 0, st>>>(partial, nb, n, out);
    return launch_status();
}

static int bias_grad_blocks(const ConvGeom &g) {
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    // rows per block: 1024 for the full-resolution maps, down to 32 for the small deep maps — the wide (cout > 256) path walks its rows
    // serially per thread and took 113-146 us on 1-4 blocks for 1-5 MB tensors (profiles/r02_ncu_launches.csv)
    long long blocks = ceil_div<long long>(M, g.cout > 256 ? 32 : (M >= 262144 ? 1024 : 128));
    if (blocks > (long long)num_sms() * 8) blocks = (long long)num_sms() * 8;
    return (int)blocks;
}

size_t conv_bias_grad_workspace_bytes(const ConvGeom &g) { return sizeof(float) * (size_t)bias_grad_blocks(g) * g.cout; }

int conv_bias_grad(const ConvGeom &g, const float *dy, float *db, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (!ws || ws_bytes < conv_bias_grad_workspace_bytes(g)) return MDT_EWORKSPACE;
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    const int blocks = bias_grad_blocks(g);
    float *partial = reinterpret_cast<float *>(ws);
    bias_grad_kernel<<<blocks, 256, 0, st>>>(dy, partial, M, g.cout, ceil_div<long long>(M, blocks));
    const int rc = launch_status();
    if (rc) return rc;
    return reduce_partials(partial, blocks, g.cout, db, st);
}

// rows of M per split (a multiple of BKW) and the number of splits of the SIMT weight gradient
static void simt_wgrad_splits(const ConvGeom &g, long long &splits, long long &rows) {
    const int taps = g.kd * g.kh * g.kw;
    const long long M = (long long)g.n * g.od * g.oh * g.ow;
    const int tiles = ceil_div(g.cin, WCI) * ceil_div(g.cout, WCO);
    // enough CTAs to fill the machine a few times over, but at least 4 * BKW rows each
    splits = ceil_div<long long>((long long)num_sms() * 16, (long long)taps * tiles);
    if (splits > ceil_div<long long>(M, 4 * BKW)) splits = ceil_div<long long>(M, 4 * BKW);
    if (splits < 1) splits = 1;
    if (splits > 65535) splits = 65535;
    rows = ceil_div<long long>(ceil_div<long long>(M, splits), BKW) * BKW;
    splits = ceil_div<long long>(M, rows);
}

size_t conv_simt_wgrad_workspace_bytes(const ConvGeom &g) {
    long long splits, rows;
    simt_wgrad_splits(g, splits, rows);
    const size_t w = sizeof(float) * (size_t)splits * g.cout * g.cin * g.kd * g.kh * g.kw, b = conv_bias_grad_workspace_bytes(g);
    return w > b ? w : b;
}

int conv_simt_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (!ws || ws_bytes < conv_simt_wgrad_workspace_bytes(g)) return MDT_EWORKSPACE;
    const int taps = g.kd * g.kh * g.kw;
    const int tiles = ceil_div(g.cin, WCI) * ceil_div(g.cout, WCO);
    long long splits, rows;
    simt_wgrad_splits(g, splits, rows);
    float *partial = reinterpret_cast<float *>(ws);
    dim3 grid(taps, (unsigned)splits, tiles);
    conv_wgrad_simt<<<grid, 256, 0, st>>>(g, x, dy, partial, rows);
    int rc = launch_status();
    if (rc) return rc;
    if ((rc = reduce_partials(partial, (int)splits, (long long)g.cout * g.cin * taps, dw, st))) return rc;
    if (db) return conv_bias_grad(g, dy, db, ws, ws_bytes, st);   // reuses the workspace after the reduction (same stream)
    return MDT_OK;
}

}  // namespace mdt

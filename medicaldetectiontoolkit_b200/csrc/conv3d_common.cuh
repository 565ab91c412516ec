// Shared conv3d geometry + internal entry points (SIMT and tcgen05 implementations).
#pragma once
#include "mdt_common.cuh"

namespace mdt {

struct ConvGeom {
    int n, d, h, w, cin, cout;
    int kd, kh, kw, sd, sh, sw, pd, ph, pw;
    int od, oh, ow;
};

inline bool make_geom(const mdt_conv3d_desc *c, ConvGeom &g) {
    if (!c) return false;
    g = ConvGeom{c->n, c->d, c->h, c->w, c->cin, c->cout, c->kd, c->kh, c->kw, c->sd, c->sh, c->sw, c->pd, c->ph, c->pw, 0, 0, 0};
    if (g.n <= 0 || g.d <= 0 || g.h <= 0 || g.w <= 0 || g.cin <= 0 || g.cout <= 0 || g.kd <= 0 || g.kh <= 0 || g.kw <= 0 || g.sd <= 0 ||
        g.sh <= 0 || g.sw <= 0 || g.pd < 0 || g.ph < 0 || g.pw < 0)
        return false;
    g.od = (g.d + 2 * g.pd - g.kd) / g.sd + 1;
    g.oh = (g.h + 2 * g.ph - g.kh) / g.sh + 1;
    g.ow = (g.w + 2 * g.pw - g.kw) / g.sw + 1;
    return g.od > 0 && g.oh > 0 && g.ow > 0;
}

// SIMT (conv3d_simt.cu)
int conv_simt_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, const float *residual, float *y, int relu, void *ws,
                    cudaStream_t st);
int conv_simt_dgrad(const ConvGeom &g, const float *dy, const float *w, float *dx, void *ws, cudaStream_t st);
int conv_simt_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, void *ws, size_t ws_bytes, cudaStream_t st);
size_t conv_simt_wgrad_workspace_bytes(const ConvGeom &g);
int conv_bias_grad(const ConvGeom &g, const float *dy, float *db, void *ws, size_t ws_bytes, cudaStream_t st);
size_t conv_bias_grad_workspace_bytes(const ConvGeom &g);
// out[e] = sum over b = 0 .. nb-1 of partial[b * n + e], always in the same order: the per-block partial sums of a reduction are combined
// here instead of with float atomics, so gradients are bitwise reproducible from run to run
int reduce_partials(const float *partial, int nb, long long n, float *out, cudaStream_t st);

// direct stem kernels, Cin <= 4 (conv3d_stem.cu)
bool conv_stem_supported(const ConvGeom &g, int pass);
int conv_stem_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, float *y, int relu, cudaStream_t st);
int conv_stem_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, void *ws, size_t ws_bytes, cudaStream_t st);
size_t conv_stem_wgrad_workspace_bytes(const ConvGeom &g);

// pointwise 1x1x1 stride-1 fp32 streaming kernels (conv3d_pw.cu)
bool conv_pw_supported(const ConvGeom &g, int pass);
bool conv_pw_preferred(const ConvGeom &g);   // `auto` picks the pointwise kernels only where they measured faster than tcgen05
size_t conv_pw_workspace_bytes(const ConvGeom &g, int pass);
int conv_pw_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, const float *residual, float *y, int relu, int precision,
                  void *y_split, cudaStream_t st);
int conv_pw_dgrad(const ConvGeom &g, const float *dy, const float *relu_of, const float *w, float *dx, float *dy_masked_out, cudaStream_t st);
int conv_pw_wgrad(const ConvGeom &g, const float *x, const float *dy, const float *relu_of, float *dw, float *db, void *ws, size_t ws_bytes,
                  cudaStream_t st, float *dy_masked_out = nullptr);

// tcgen05 (conv3d_tc.cu; conv3d_tcw.cu for the tap-stacked variant)
bool conv_tc_supported(const ConvGeom &g, int pass);
bool conv_tcw_supported(const ConvGeom &g, int pass);
size_t conv_tc_workspace_bytes(const ConvGeom &g, int pass, int precision);
int conv_tc_fprop(const ConvGeom &g, const float *x, const float *w, const float *bias, const float *residual, float *y, int relu, int precision,
                  void *ws, size_t ws_bytes, cudaStream_t st);
int conv_tc_dgrad(const ConvGeom &g, const float *dy, const float *w, float *dx, int precision, void *ws, size_t ws_bytes, cudaStream_t st);
int conv_tc_wgrad(const ConvGeom &g, const float *x, const float *dy, float *dw, float *db, int precision, void *ws, size_t ws_bytes,
                  cudaStream_t st);

// fused backward (conv3d_tc_wgrad.cu)
bool conv_tc_backward_supported(const ConvGeom &g, bool need_dx);
size_t conv_tc_backward_workspace_bytes(const ConvGeom &g, bool need_dx, int precision);
int conv_tc_backward(const ConvGeom &g, const float *x, const float *dy, const float *relu_of, const float *w, float *dx, float *dw, float *db,
                     float *dy_masked_out, int precision, void *ws, size_t ws_bytes, cudaStream_t st, const void *x_split);
size_t conv_tc_split_bytes(long long rows, int channels, int precision);
int conv_tc_split(const float *x, long long rows, int channels, int line_w, int precision, void *out, cudaStream_t st);
int conv_tc_fprop_presplit(const ConvGeom &g, const void *x_split, const float *w, const float *bias, const float *residual, float *y, int relu,
                           int precision, void *ws, size_t ws_bytes, cudaStream_t st, void *y_split = nullptr);

}  // namespace mdt

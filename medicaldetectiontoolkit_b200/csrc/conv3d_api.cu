// C-ABI of the conv3d path: algorithm selection (tcgen05 implicit GEMM vs fp32 SIMT) + workspace accounting.
#include "conv3d_common.cuh"

namespace mdt {
int conv_tcw_read_prof(unsigned long long *out16);
// 1 = fp32 SIMT (generic implicit GEMM, or the direct stem kernels when Cin <= 4), 2 = tcgen05, 4 = pointwise fp32 streaming (1x1x1, stride 1)
static int pick_algo(const mdt_conv3d_desc *c, const ConvGeom &g, int pass) {
    if (c->algo == 1) return 1;
    if (c->algo == 4) return conv_pw_supported(g, pass) ? 4 : 0;
    if (c->algo == 0 && conv_pw_preferred(g) && conv_pw_supported(g, pass)) return 4;   // HBM-bound: read the fp32 rows once instead of split + MMA + epilogue
    if (c->algo == 0 && conv_stem_supported(g, pass)) return 1;   // bandwidth-bound stem: direct kernels beat a 94 %-padded MMA
    const bool tc = conv_tc_supported(g, pass);
    if (c->algo == 2) return tc ? 2 : 0;
    return tc ? 2 : 1;
}
static bool pw_backward(const mdt_conv3d_desc *c, const ConvGeom &g, bool need_dx) {
    return (c->algo == 4 || (c->algo == 0 && conv_pw_preferred(g))) && conv_pw_supported(g, 2) && (!need_dx || conv_pw_supported(g, 1));
}
static size_t simt_ws(const ConvGeom &g, int pass, int algo) {
    if (algo == 4) return conv_pw_workspace_bytes(g, pass);
    if (pass == 2) return conv_stem_supported(g, 2) ? conv_stem_wgrad_workspace_bytes(g) : conv_simt_wgrad_workspace_bytes(g);
    return sizeof(float) * (size_t)g.cout * g.cin * g.kd * g.kh * g.kw;
}
}  // namespace mdt

extern "C" {

int mdt_conv3d_algo(const mdt_conv3d_desc *c, int pass) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || pass < 0 || pass > 2) return MDT_EINVAL;
    return mdt::pick_algo(c, g, pass);
}

int mdt_debug_conv_tcw_prof(unsigned long long *out16) { return out16 ? mdt::conv_tcw_read_prof(out16) : MDT_EINVAL; }

int mdt_conv3d_variant(const mdt_conv3d_desc *c, int pass) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || pass < 0 || pass > 2) return MDT_EINVAL;
    const int algo = mdt::pick_algo(c, g, pass);
    if (algo != 2) return algo;
    return (pass < 2 && mdt::conv_tcw_supported(g, pass)) ? 3 : 2;
}

size_t mdt_conv3d_workspace_bytes(const mdt_conv3d_desc *c, int pass) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || pass < 0 || pass > 2) return 0;
    const int algo = mdt::pick_algo(c, g, pass);
    size_t b = algo == 2 ? mdt::conv_tc_workspace_bytes(g, pass, c->precision) : mdt::simt_ws(g, pass, algo);
    return b + 256;
}

int mdt_conv3d_fprop(const mdt_conv3d_desc *c, const float *x, const float *w, const float *bias, const float *residual, float *y, void *ws,
                     size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x || !w || !y) return MDT_EINVAL;
    if (ws_bytes < mdt_conv3d_workspace_bytes(c, 0) || !ws) return MDT_EWORKSPACE;
    const int algo = mdt::pick_algo(c, g, 0);
    if (algo == 0) return MDT_EUNSUPPORTED;
    if (algo == 2) return mdt::conv_tc_fprop(g, x, w, bias, residual, y, c->relu, c->precision, ws, ws_bytes, mdt::as_stream(stream));
    if (algo == 4) return mdt::conv_pw_fprop(g, x, w, bias, residual, y, c->relu, c->precision, nullptr, mdt::as_stream(stream));
    if (!residual && mdt::conv_stem_supported(g, 0)) return mdt::conv_stem_fprop(g, x, w, bias, y, c->relu, mdt::as_stream(stream));
    return mdt::conv_simt_fprop(g, x, w, bias, residual, y, c->relu, ws, mdt::as_stream(stream));
}

int mdt_conv3d_dgrad(const mdt_conv3d_desc *c, const float *dy, const float *w, float *dx, void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !dy || !w || !dx) return MDT_EINVAL;
    if (ws_bytes < mdt_conv3d_workspace_bytes(c, 1) || !ws) return MDT_EWORKSPACE;
    const int algo = mdt::pick_algo(c, g, 1);
    if (algo == 0) return MDT_EUNSUPPORTED;
    if (algo == 2) return mdt::conv_tc_dgrad(g, dy, w, dx, c->precision, ws, ws_bytes, mdt::as_stream(stream));
    if (algo == 4) return mdt::conv_pw_dgrad(g, dy, nullptr, w, dx, nullptr, mdt::as_stream(stream));
    return mdt::conv_simt_dgrad(g, dy, w, dx, ws, mdt::as_stream(stream));
}

int mdt_conv3d_wgrad(const mdt_conv3d_desc *c, const float *x, const float *dy, float *dw, float *db, void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x || !dy || !dw) return MDT_EINVAL;
    if (ws_bytes < mdt_conv3d_workspace_bytes(c, 2)) return MDT_EWORKSPACE;
    const int algo = mdt::pick_algo(c, g, 2);
    if (algo == 0) return MDT_EUNSUPPORTED;
    if (algo == 2) return mdt::conv_tc_wgrad(g, x, dy, dw, db, c->precision, ws, ws_bytes, mdt::as_stream(stream));
    if (algo == 4) return mdt::conv_pw_wgrad(g, x, dy, nullptr, dw, db, ws, ws_bytes, mdt::as_stream(stream));
    if (mdt::conv_stem_supported(g, 2)) return mdt::conv_stem_wgrad(g, x, dy, dw, db, ws, ws_bytes, mdt::as_stream(stream));
    return mdt::conv_simt_wgrad(g, x, dy, dw, db, ws, ws_bytes, mdt::as_stream(stream));
}

/* fused backward: 1 if the tcgen05 fused path (one pass over dy shared by dgrad + wgrad, ReLU mask and bias gradient folded in) applies */
int mdt_conv3d_backward_fused(const mdt_conv3d_desc *c, int need_dx) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g)) return 0;
    if (c->algo == 1) return 0;
    if (mdt::pw_backward(c, g, need_dx != 0)) return 1;
    if (c->algo == 4) return 0;
    if (c->algo == 0 && mdt::conv_stem_supported(g, 2)) return 0;   // stem: direct kernels
    return mdt::conv_tc_backward_supported(g, need_dx != 0) ? 1 : 0;
}

size_t mdt_conv3d_backward_workspace_bytes(const mdt_conv3d_desc *c, int need_dx) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g)) return 0;
    if (mdt::pw_backward(c, g, need_dx != 0)) return mdt::conv_pw_workspace_bytes(g, 2) + 256;
    return mdt::conv_tc_backward_workspace_bytes(g, need_dx != 0, c->precision) + 256;
}

size_t mdt_conv3d_split_bytes(const mdt_conv3d_desc *c) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g)) return 0;
    return mdt::conv_tc_split_bytes((long long)g.n * g.d * g.h * g.w, g.cin, c->precision);
}

int mdt_conv3d_split(const mdt_conv3d_desc *c, const float *x, void *x_split, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x || !x_split) return MDT_EINVAL;
    return mdt::conv_tc_split(x, (long long)g.n * g.d * g.h * g.w, g.cin, g.w, c->precision, x_split, mdt::as_stream(stream));
}

int mdt_conv3d_fprop_presplit(const mdt_conv3d_desc *c, const void *x_split, const float *w, const float *bias, const float *residual, float *y,
                              void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x_split || !w || !y) return MDT_EINVAL;
    if (mdt::pick_algo(c, g, 0) != 2) return MDT_EUNSUPPORTED;
    if (ws_bytes < mdt_conv3d_workspace_bytes(c, 0) || !ws) return MDT_EWORKSPACE;
    return mdt::conv_tc_fprop_presplit(g, x_split, w, bias, residual, y, c->relu, c->precision, ws, ws_bytes, mdt::as_stream(stream));
}

int mdt_conv3d_fprop_presplit_out(const mdt_conv3d_desc *c, const void *x_split, const float *w, const float *bias, const float *residual, float *y,
                                  void *y_split, void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x_split || !w || !y || !y_split) return MDT_EINVAL;
    if (mdt::pick_algo(c, g, 0) != 2) return MDT_EUNSUPPORTED;
    if (ws_bytes < mdt_conv3d_workspace_bytes(c, 0) || !ws) return MDT_EWORKSPACE;
    return mdt::conv_tc_fprop_presplit(g, x_split, w, bias, residual, y, c->relu, c->precision, ws, ws_bytes, mdt::as_stream(stream), y_split);
}

int mdt_conv3d_fprop_out(const mdt_conv3d_desc *c, const float *x, const float *w, const float *bias, const float *residual, float *y, void *y_split,
                         void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || !x || !w || !y || !y_split) return MDT_EINVAL;
    if (mdt::pick_algo(c, g, 0) != 4) return MDT_EUNSUPPORTED;
    return mdt::conv_pw_fprop(g, x, w, bias, residual, y, c->relu, c->precision, y_split, mdt::as_stream(stream));
}

size_t mdt_conv3d_out_split_bytes(const mdt_conv3d_desc *c) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g)) return 0;
    return mdt::conv_tc_split_bytes((long long)g.n * g.od * g.oh * g.ow, g.cout, c->precision);
}

int mdt_conv3d_backward(const mdt_conv3d_desc *c, const float *x, const void *x_split, const float *dy, const float *y_relu, const float *w,
                        float *dx, float *dw, float *db, float *dy_masked_out, void *ws, size_t ws_bytes, void *stream) {
    mdt::ConvGeom g;
    if (!mdt::make_geom(c, g) || (!x && !x_split) || !dy || !w || !dw) return MDT_EINVAL;
    if (!mdt_conv3d_backward_fused(c, dx != nullptr)) return MDT_EUNSUPPORTED;
    if (!ws || ws_bytes < mdt_conv3d_backward_workspace_bytes(c, dx != nullptr)) return MDT_EWORKSPACE;
    if (mdt::pw_backward(c, g, dx != nullptr)) {
        // pointwise conv: dgrad (masks dy by the forward output on load, writes the masked copy if asked) + wgrad (reads the masked copy when
        // there is one, else masks on load); both stream fp32 rows once
        if (!x) return MDT_EINVAL;
        int rc = MDT_OK;
        if (dx && (rc = mdt::conv_pw_dgrad(g, dy, y_relu, w, dx, dy_masked_out, mdt::as_stream(stream)))) return rc;
        const bool have_masked = dx && y_relu && dy_masked_out;
        return mdt::conv_pw_wgrad(g, x, have_masked ? dy_masked_out : dy, have_masked ? nullptr : y_relu, dw, db, ws, ws_bytes,
                                  mdt::as_stream(stream), have_masked ? nullptr : dy_masked_out);
    }
    return mdt::conv_tc_backward(g, x, dy, y_relu, w, dx, dw, db, dy_masked_out, c->precision, ws, ws_bytes, mdt::as_stream(stream), x_split);
}

}  // extern "C"

// C-ABI entry points of the masked conv / linear path: argument validation and
// the shape dispatch between the tcgen05 implicit-GEMM kernels (igemm_tc.cu)
// and the CUDA-core kernels (conv_simt.cu).
#include <stdlib.h>

#include "common.cuh"
#include "conv_common.cuh"

namespace rigl {

static int g_force_simt = -1;

static bool force_simt() {
  if (g_force_simt < 0) {
    const char* e = getenv("RIGL_FORCE_SIMT");
    g_force_simt = (e && e[0] == '1') ? 1 : 0;
  }
  return g_force_simt == 1;
}

int geom_from_desc(const rigl_conv_desc* d, ConvGeom* g) {
  RIGL_REQUIRE(d != nullptr, "null conv desc");
  RIGL_REQUIRE(d->batch > 0 && d->in_h > 0 && d->in_w > 0 && d->cin > 0 && d->cout > 0 && d->ksize > 0 &&
                   d->stride > 0 && d->pad >= 0,
               "conv desc: non-positive dimension");
  // `pad` is the padding BEFORE the image; windows may overrun the far edge (implicit zero
  // padding there), which covers TF 'SAME' (asymmetric for stride 2), explicit fixed padding
  // and 'VALID'.  Every window must start inside the padded image.
  RIGL_REQUIRE(d->pad < d->ksize && d->out_h > 0 && d->out_w > 0 &&
                   (d->out_h - 1) * d->stride - d->pad < d->in_h && (d->out_w - 1) * d->stride - d->pad < d->in_w,
               "conv desc: output %dx%d inconsistent with input %dx%d, k=%d, stride=%d, pad=%d", d->out_h,
               d->out_w, d->in_h, d->in_w, d->ksize, d->stride, d->pad);
  g->batch = d->batch; g->in_h = d->in_h; g->in_w = d->in_w; g->cin = d->cin;
  g->out_h = d->out_h; g->out_w = d->out_w; g->cout = d->cout;
  g->ksize = d->ksize; g->stride = d->stride; g->pad = d->pad;
  g->cin_pad = round_up8(d->cin); g->cout_pad = round_up8(d->cout);
  g->x_pitch = d->x_pitch > 0 ? d->x_pitch : d->cin;
  RIGL_REQUIRE(g->x_pitch >= d->cin, "conv desc: x_pitch %d < cin %d", g->x_pitch, d->cin);
  return RIGL_OK;
}

}  // namespace rigl

using namespace rigl;

extern "C" int rigl_im2col_nhwc(const rigl_conv_desc* d, const void* x, void* out, int64_t out_pitch,
                                void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && out && out_pitch >= (int64_t)g.taps() * g.cin, "rigl_im2col_nhwc: bad arguments");
  return simt_im2col(g, x, out, out_pitch, (cudaStream_t)stream);
}

// ---- small-Cin (stem) convs: zero-bordered 8-channel input + window tensor maps ----
// ---- space-to-depth stem (experimental, see stem_s2d.cuh) ----
extern "C" int rigl_stem_s2d_supported(const rigl_conv_desc* d) {
  ConvGeom g;
  if (geom_from_desc(d, &g) != RIGL_OK) return 0;
  return s2d_supported(g) && !force_simt() ? 1 : 0;
}
extern "C" size_t rigl_stem_s2d_folded_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? s2d_folded_bytes(g) : 0;
}
extern "C" size_t rigl_stem_s2d_packed_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? s2d_packed_bytes(g) : 0;
}
extern "C" size_t rigl_stem_s2d_workspace_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? s2d_workspace_bytes(g) : 0;
}
extern "C" int rigl_stem_s2d_fold_input(const rigl_conv_desc* d, const void* x, void* xs, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && xs && s2d_supported(g) && aligned16(xs), "rigl_stem_s2d_fold_input: bad arguments");
  return s2d_fold(g, x, xs, (cudaStream_t)stream);
}
extern "C" int rigl_stem_s2d_pack_weights(const rigl_conv_desc* d, const float* w_hwio, const uint32_t* mask_bits,
                                          void* packed, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(w_hwio && mask_bits && packed && s2d_supported(g), "rigl_stem_s2d_pack_weights: bad arguments");
  return s2d_pack(g, w_hwio, mask_bits, packed, (cudaStream_t)stream);
}
extern "C" int rigl_stem_s2d_fprop(const rigl_conv_desc* d, const void* xs, const void* packed, void* y,
                                   void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(xs && packed && y && s2d_supported(g), "rigl_stem_s2d_fprop: bad arguments");
  return s2d_fprop(g, xs, packed, y, (cudaStream_t)stream);
}
extern "C" int rigl_stem_s2d_wgrad(const rigl_conv_desc* d, const void* xs, const void* dy, float* dw, float beta,
                                   void* ws, size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(xs && dy && dw && s2d_supported(g), "rigl_stem_s2d_wgrad: bad arguments");
  return s2d_wgrad(g, xs, dy, dw, beta, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int rigl_smallc_supported(const rigl_conv_desc* d) {
  ConvGeom g;
  if (geom_from_desc(d, &g) != RIGL_OK) return 0;
  return smallc_supported(g) && !force_simt() ? 1 : 0;
}
extern "C" size_t rigl_smallc_padded_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? smallc_padded_bytes(g) : 0;
}
extern "C" size_t rigl_smallc_packed_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? smallc_packed_bytes(g) : 0;
}
extern "C" size_t rigl_smallc_workspace_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  return geom_from_desc(d, &g) == RIGL_OK ? smallc_wgrad_ws_bytes(g) : 0;
}
extern "C" int rigl_smallc_pad_input(const rigl_conv_desc* d, const void* x, void* xp, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && xp && smallc_supported(g) && aligned16(xp), "rigl_smallc_pad_input: bad arguments");
  return smallc_pad_input(g, x, xp, (cudaStream_t)stream);
}
extern "C" int rigl_smallc_pack_weights(const rigl_conv_desc* d, const float* w_hwio, const uint32_t* mask_bits,
                                        void* packed, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(w_hwio && mask_bits && packed && smallc_supported(g), "rigl_smallc_pack_weights: bad arguments");
  return smallc_pack(g, w_hwio, mask_bits, packed, (cudaStream_t)stream);
}
extern "C" int rigl_smallc_fprop(const rigl_conv_desc* d, const void* xp, const void* packed, void* y,
                                 void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(xp && packed && y && smallc_supported(g), "rigl_smallc_fprop: bad arguments");
  return smallc_fprop(g, xp, packed, y, (cudaStream_t)stream);
}
extern "C" int rigl_smallc_wgrad(const rigl_conv_desc* d, const void* xp, const void* dy, float* dw, float beta,
                                 void* ws, size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(xp && dy && dw && smallc_supported(g), "rigl_smallc_wgrad: bad arguments");
  return smallc_wgrad(g, xp, dy, dw, beta, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int rigl_set_force_simt(int on) {
  g_force_simt = on ? 1 : 0;
  return RIGL_OK;
}

extern "C" size_t rigl_conv_workspace_bytes(const rigl_conv_desc* d) {
  ConvGeom g;
  if (geom_from_desc(d, &g) != RIGL_OK) return 0;
  return tc_workspace_bytes(g);
}

extern "C" int rigl_masked_conv2d_fprop(const rigl_conv_desc* d, const void* x, const void* packed,
                                        void* y_bf16, float* y_f32, const float* bias, void* ws,
                                        size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && packed && (y_bf16 || y_f32), "rigl_masked_conv2d_fprop: null tensor");
  const PackedLayout L = packed_layout(g.taps(), g.cin, g.cout);
  if (!force_simt() && tc_supported(g, 0))
    return tc_fprop(g, x, packed, y_bf16, y_f32, bias, ws, ws_bytes, (cudaStream_t)stream);
  return simt_fprop(g, x, static_cast<const uint8_t*>(packed) + L.off_dgrad, y_bf16, y_f32, bias,
                    (cudaStream_t)stream);
}

extern "C" int rigl_bn_partial_rows(void) { return tc_max_ctas(); }

extern "C" int rigl_set_bn_stats_always(int on) {
  tc_set_bn_stats_always(on != 0);
  tc_set_bn_stats_debug(on >> 4);       // (development: bits 4.. select partial variants of the statistics code)
  return RIGL_OK;
}

extern "C" int rigl_masked_conv2d_fprop_bnstats(const rigl_conv_desc* d, const void* x, const void* packed,
                                                void* y_bf16, float* bn_partial, int* bn_rows_out, void* ws,
                                                size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && packed && y_bf16 && bn_partial && bn_rows_out, "rigl_masked_conv2d_fprop_bnstats: null argument");
  if (force_simt() || !tc_supported(g, 0)) {
    set_error("rigl_masked_conv2d_fprop_bnstats: shape not on the tensor-core path");
    return RIGL_ERR_UNSUPPORTED;
  }
  return tc_fprop(g, x, packed, y_bf16, nullptr, nullptr, ws, ws_bytes, (cudaStream_t)stream, bn_partial, bn_rows_out);
}

extern "C" int rigl_masked_conv2d_fprop_affine(const rigl_conv_desc* d, const void* x, const void* packed,
                                               const float* scale, const float* shift, const void* residual,
                                               int relu, void* y_bf16, void* ws, size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && packed && y_bf16, "rigl_masked_conv2d_fprop_affine: null tensor");
  RIGL_REQUIRE(aligned16(y_bf16) && aligned16(scale) && aligned16(shift) && aligned16(residual),
               "rigl_masked_conv2d_fprop_affine: y, scale, shift and residual must be 16-byte aligned");
  const AffineEpi epi = {scale, shift, residual, relu ? 1 : 0};
  const PackedLayout L = packed_layout(g.taps(), g.cin, g.cout);
  if (!force_simt() && tc_supported(g, 0))
    return tc_fprop(g, x, packed, y_bf16, nullptr, nullptr, ws, ws_bytes, (cudaStream_t)stream, nullptr, nullptr, &epi);
  return simt_fprop(g, x, static_cast<const uint8_t*>(packed) + L.off_dgrad, y_bf16, nullptr, nullptr,
                    (cudaStream_t)stream, &epi);
}

extern "C" int rigl_masked_conv2d_dgrad(const rigl_conv_desc* d, const void* dy, const void* packed,
                                        void* dx, void* ws, size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(dy && packed && dx, "rigl_masked_conv2d_dgrad: null tensor");
  const PackedLayout L = packed_layout(g.taps(), g.cin, g.cout);
  if (!force_simt() && tc_supported(g, 1))
    return tc_dgrad(g, dy, packed, dx, ws, ws_bytes, (cudaStream_t)stream);
  return simt_dgrad(g, dy, static_cast<const uint8_t*>(packed) + L.off_fprop, dx, (cudaStream_t)stream);
}

extern "C" int rigl_conv2d_wgrad_dense(const rigl_conv_desc* d, const void* x, const void* dy, float* dw,
                                       float beta, void* ws, size_t ws_bytes, void* stream) {
  ConvGeom g;
  int rc = geom_from_desc(d, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && dy && dw, "rigl_conv2d_wgrad_dense: null tensor");
  RIGL_REQUIRE(beta == 0.f || beta == 1.f, "rigl_conv2d_wgrad_dense: beta must be 0 or 1");
  if (!force_simt() && tc_supported(g, 2))
    return tc_wgrad(g, x, dy, dw, beta, ws, ws_bytes, (cudaStream_t)stream);
  return simt_wgrad(g, x, dy, dw, beta, (cudaStream_t)stream);
}

// Geometry and packed-operand layout shared by the conv / linear kernels.
#pragma once
#include <stdint.h>
#include <stddef.h>

#include "../../include/rigl_b200.h"

namespace rigl {

struct ConvGeom {
  int batch, in_h, in_w, cin;
  int out_h, out_w, cout;
  int ksize, stride, pad;
  int cin_pad, cout_pad;     // rounded up to multiples of 8 (16-byte bf16 rows)
  int x_pitch;               // elements between pixels of x (>= cin)
  __host__ __device__ int64_t out_pixels() const { return (int64_t)batch * out_h * out_w; }
  __host__ __device__ int64_t in_pixels() const { return (int64_t)batch * in_h * in_w; }
  __host__ __device__ int taps() const { return ksize * ksize; }
};

inline int round_up8(int v) { return (v + 7) / 8 * 8; }

// Packed masked-weight blob written by rigl_pack_masked_weights:
//   [ w_fprop bf16 [taps][cout][cin_pad] | w_dgrad bf16 [taps][cin][cout_pad] |
//     tile_nnz u32 [taps][ceil(cout/64)][ceil(cin/64)] ]   (each section 256B aligned)
struct PackedLayout {
  size_t off_fprop, off_dgrad, off_nnz, total;
  int cin_pad, cout_pad, n_tiles, k_tiles;
};

inline PackedLayout packed_layout(int taps, int cin, int cout) {
  PackedLayout L;
  L.cin_pad = round_up8(cin);
  L.cout_pad = round_up8(cout);
  L.n_tiles = (cout + 63) / 64;
  L.k_tiles = (cin + 63) / 64;
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  L.off_fprop = 0;
  L.off_dgrad = up((size_t)taps * cout * L.cin_pad * 2);
  L.off_nnz = L.off_dgrad + up((size_t)taps * cin * L.cout_pad * 2);
  L.total = L.off_nnz + up((size_t)taps * L.n_tiles * L.k_tiles * 4);
  return L;
}

int geom_from_desc(const rigl_conv_desc* d, ConvGeom* g);   // validates; sets last error

// Inference epilogue of rigl_masked_conv2d_fprop_affine: y = [relu](acc * scale[c] + shift[c] (+ residual)).
struct AffineEpi {
  const float* scale;        // [cout] or null (1)
  const float* shift;        // [cout] or null (0)
  const void* residual;      // bf16, the output's shape, or null
  int relu;
};

// SIMT path (conv_simt.cu)
int simt_fprop(const ConvGeom& g, const void* x, const void* w_dgrad, void* y, float* y_f32,
               const float* bias, cudaStream_t s, const AffineEpi* epi = nullptr);
int simt_dgrad(const ConvGeom& g, const void* dy, const void* w_fprop, void* dx, cudaStream_t s);
int simt_wgrad(const ConvGeom& g, const void* x, const void* dy, float* dw, float beta, cudaStream_t s);
int simt_im2col(const ConvGeom& g, const void* x, void* out, int64_t out_pitch, cudaStream_t s);

// tcgen05 path (igemm_tc.cu)
bool tc_supported(const ConvGeom& g, int which /*0 fprop, 1 dgrad, 2 wgrad*/);
size_t tc_workspace_bytes(const ConvGeom& g);
int tc_fprop(const ConvGeom& g, const void* x, const void* packed, void* y, float* y_f32,
             const float* bias, void* ws, size_t ws_bytes, cudaStream_t s, float* bn_partial = nullptr,
             int* bn_rows = nullptr, const AffineEpi* epi = nullptr);
int tc_max_ctas();
void tc_set_bn_stats_always(bool on);
void tc_set_bn_stats_debug(int v);
int tc_dgrad(const ConvGeom& g, const void* dy, const void* packed, void* dx, void* ws,
             size_t ws_bytes, cudaStream_t s);
int tc_wgrad(const ConvGeom& g, const void* x, const void* dy, float* dw, float beta, void* ws,
             size_t ws_bytes, cudaStream_t s);

// small-Cin (stem) path (igemm_tc.cu)
// Space-to-depth stem (stem_s2d.cuh) -- experimental, opt-in
bool s2d_supported(const ConvGeom& g);
size_t s2d_folded_bytes(const ConvGeom& g);
size_t s2d_packed_bytes(const ConvGeom& g);
size_t s2d_workspace_bytes(const ConvGeom& g);
int s2d_fold(const ConvGeom& g, const void* x, void* xs, cudaStream_t s);
int s2d_pack(const ConvGeom& g, const float* w, const uint32_t* bits, void* packed, cudaStream_t s);
int s2d_fprop(const ConvGeom& g, const void* xs, const void* packed, void* y, cudaStream_t s);
int s2d_wgrad(const ConvGeom& g, const void* xs, const void* dy, float* dw, float beta, void* ws, size_t ws_bytes,
              cudaStream_t s);
bool smallc_supported(const ConvGeom& g);
size_t smallc_padded_bytes(const ConvGeom& g);
size_t smallc_packed_bytes(const ConvGeom& g);
size_t smallc_wgrad_ws_bytes(const ConvGeom& g);
int smallc_pad_input(const ConvGeom& g, const void* x, void* xp, cudaStream_t s);
int smallc_pack(const ConvGeom& g, const float* w, const uint32_t* bits, void* packed, cudaStream_t s);
int smallc_fprop(const ConvGeom& g, const void* xp, const void* packed, void* y, cudaStream_t s);
int smallc_wgrad(const ConvGeom& g, const void* xp, const void* dy, float* dw, float beta, void* ws,
                 size_t ws_bytes, cudaStream_t s);

}  // namespace rigl

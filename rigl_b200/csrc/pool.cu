// Max pooling for NHWC bf16 activations (the stem's 3x3/2 pool), HBM-bound streaming kernels.
// Replaces tf.layers.max_pooling2d(pool_size=3, strides=2, padding='SAME')
// (rigl/imagenet_resnet/resnet_model.py:636-642) with TF's SAME rule: pad_total =
// max((out-1)*s + k - in, 0), pad_before = pad_total / 2 (so 112 -> 56 pads only at the end).
// Forward stores the window-relative argmax (first maximum in (kh,kw) scan order) as one byte
// per output element; backward is a deterministic gather over the <= ceil(k/s)^2 windows that
// cover an input pixel.  One thread = 8 channels (16-byte vectors), channels innermost.
#include <cuda_bf16.h>

#include "common.cuh"

namespace rigl {

struct PoolGeom {
  int n, h, w, c, oh, ow, k, s, pad;
};

// kArg = false: inference (no backward pass follows), the argmax bytes are not written.
template <bool kArg>
__global__ void __launch_bounds__(256)
k_maxpool_fwd(PoolGeom g, const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
              uint8_t* __restrict__ idx) {
  // grid = (column tiles, output rows, images), block = (8 channel vectors, 32 columns): no index
  // divisions in the kernel (they cost more than the window loads).
  const int V = g.c >> 3;
  const int ow = blockIdx.x * blockDim.y + threadIdx.y, oh = blockIdx.y, n = blockIdx.z;
  if (ow >= g.ow) return;
  const long long p = ((long long)n * g.oh + oh) * g.ow + ow;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float best[8];
    uint8_t arg[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { best[e] = -INFINITY; arg[e] = 0; }
    for (int kh = 0; kh < g.k; ++kh) {
      const int hi = oh * g.s + kh - g.pad;
      if (hi < 0 || hi >= g.h) continue;
      for (int kw = 0; kw < g.k; ++kw) {
        const int wi = ow * g.s + kw - g.pad;
        if (wi < 0 || wi >= g.w) continue;
        const uint4 raw = *reinterpret_cast<const uint4*>(x + (((long long)n * g.h + hi) * g.w + wi) * g.c + 8 * v);
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __bfloat1622float2(h2[e]);
          if (f.x > best[2 * e]) { best[2 * e] = f.x; arg[2 * e] = (uint8_t)(kh * g.k + kw); }
          if (f.y > best[2 * e + 1]) { best[2 * e + 1] = f.y; arg[2 * e + 1] = (uint8_t)(kh * g.k + kw); }
        }
      }
    }
    uint4 o;
    __nv_bfloat162* oh2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) oh2[e] = __floats2bfloat162_rn(best[2 * e], best[2 * e + 1]);
    *reinterpret_cast<uint4*>(y + p * g.c + 8 * v) = o;
    if constexpr (kArg) {
      uint2 a;
      a.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | ((uint32_t)arg[3] << 24);
      a.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | ((uint32_t)arg[7] << 24);
      *reinterpret_cast<uint2*>(idx + p * g.c + 8 * v) = a;
    }
  }
}

__global__ void __launch_bounds__(256)
k_maxpool_bwd(PoolGeom g, const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
              __nv_bfloat16* __restrict__ dx) {
  const int V = g.c >> 3;
  const int wi = blockIdx.x * blockDim.y + threadIdx.y, hi = blockIdx.y, n = blockIdx.z;
  if (wi >= g.w) return;
  const long long q = ((long long)n * g.h + hi) * g.w + wi;
  // outputs oh with oh*s - pad <= hi <= oh*s - pad + k - 1
  const int oh_lo = max(0, (hi + g.pad - g.k + g.s) / g.s), oh_hi = min(g.oh - 1, (hi + g.pad) / g.s);
  const int ow_lo = max(0, (wi + g.pad - g.k + g.s) / g.s), ow_hi = min(g.ow - 1, (wi + g.pad) / g.s);
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    for (int oh = oh_lo; oh <= oh_hi; ++oh)
      for (int ow = ow_lo; ow <= ow_hi; ++ow) {
        const int rel = (hi - (oh * g.s - g.pad)) * g.k + (wi - (ow * g.s - g.pad));
        const long long p = ((long long)n * g.oh + oh) * g.ow + ow;
        const uint2 a = *reinterpret_cast<const uint2*>(idx + p * g.c + 8 * v);
        const uint4 raw = *reinterpret_cast<const uint4*>(dy + p * g.c + 8 * v);
        const __nv_bfloat16* d = reinterpret_cast<const __nv_bfloat16*>(&raw);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const uint32_t ai = ((e < 4 ? a.x : a.y) >> (8 * (e & 3))) & 0xFFu;
          if ((int)ai == rel) acc[e] += __bfloat162float(d[e]);
        }
      }
    uint4 o;
    __nv_bfloat162* o2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) o2[e] = __floats2bfloat162_rn(acc[2 * e], acc[2 * e + 1]);
    *reinterpret_cast<uint4*>(dx + q * g.c + 8 * v) = o;
  }
}

// The stem's case (3x3 window, stride 2, no leading pad, even extents): a 2x2 quad of input pixels is covered by the
// same four windows (oh-1|oh) x (ow-1|ow), nine (pixel, window) visits in all.  One thread = one quad x 8 channels:
// it loads the four outputs once (2.25 -> 1 window loads per input pixel) and writes the four pixels as two 32-byte
// runs.  Same accumulation order as the generic gather (oh ascending, then ow): bit-identical results.
__global__ void __launch_bounds__(256)
k_maxpool_bwd_3x3s2(PoolGeom g, const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
                    __nv_bfloat16* __restrict__ dx) {
  const int V = g.c >> 3;
  const int qw = blockIdx.x * blockDim.y + threadIdx.y, qh = blockIdx.y, n = blockIdx.z;
  if (qw >= (g.w >> 1)) return;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float acc[4][8];            // pixels (0,0) (0,1) (1,0) (1,1) of the quad
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[p][e] = 0.f;
    uint2 a[4];
    uint4 d[4];
    bool ok[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {           // windows in the generic kernel's visiting order
      const int oh = qh - 1 + (j >> 1), ow = qw - 1 + (j & 1);
      ok[j] = oh >= 0 && ow >= 0 && oh < g.oh && ow < g.ow;
      a[j] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
      d[j] = make_uint4(0u, 0u, 0u, 0u);
      if (ok[j]) {
        const long long p = (((long long)n * g.oh + oh) * g.ow + ow) * g.c + 8 * v;
        a[j] = *reinterpret_cast<const uint2*>(idx + p);
        d[j] = *reinterpret_cast<const uint4*>(dy + p);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat16* dv = reinterpret_cast<const __nv_bfloat16*>(&d[j]);
      const int dh = 2 - 2 * (j >> 1), dw = 2 - 2 * (j & 1);   // window-relative position of pixel (0,0)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int ai = (int)(((e < 4 ? a[j].x : a[j].y) >> (8 * (e & 3))) & 0xFFu);
        const float f = __bfloat162float(dv[e]);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const int rh = dh + (p >> 1), rw = dw + (p & 1);
          if (rh < 3 && rw < 3 && ai == rh * 3 + rw) acc[p][e] += f;
        }
      }
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      uint4 o;
      __nv_bfloat162* o2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
      for (int e = 0; e < 4; ++e) o2[e] = __floats2bfloat162_rn(acc[p][2 * e], acc[p][2 * e + 1]);
      const long long q = ((long long)n * g.h + 2 * qh + (p >> 1)) * g.w + 2 * qw + (p & 1);
      *reinterpret_cast<uint4*>(dx + q * g.c + 8 * v) = o;
    }
  }
}

static int pool_geom(int n, int h, int w, int c, int k, int s, PoolGeom* g) {
  RIGL_REQUIRE(n > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0 && k > 0 && s > 0 && k * k <= 255,
               "maxpool: bad geometry (channels must be a multiple of 8)");
  g->n = n; g->h = h; g->w = w; g->c = c; g->k = k; g->s = s;
  g->oh = (h + s - 1) / s; g->ow = (w + s - 1) / s;                       // TF 'SAME'
  const int pad_total = max((g->oh - 1) * s + k - h, 0);
  g->pad = pad_total / 2;
  return RIGL_OK;
}

}  // namespace rigl

using namespace rigl;

extern "C" int rigl_maxpool_same_forward(const void* x, int n, int h, int w, int c, int ksize, int stride,
                                         void* y, uint8_t* argmax, void* stream) {
  PoolGeom g;
  int rc = pool_geom(n, h, w, c, ksize, stride, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(x && y, "rigl_maxpool_same_forward: null tensor");
  RIGL_REQUIRE(g.oh <= 65535 && n <= 65535, "rigl_maxpool_same_forward: extent too large");
  const dim3 block(8, 32), grid((unsigned)((g.ow + 31) / 32), (unsigned)g.oh, (unsigned)n);
  if (argmax)
    k_maxpool_fwd<true><<<grid, block, 0, (cudaStream_t)stream>>>(g, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, argmax);
  else
    k_maxpool_fwd<false><<<grid, block, 0, (cudaStream_t)stream>>>(g, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, nullptr);
  RIGL_LAUNCH_CHECK("k_maxpool_fwd");
  return RIGL_OK;
}

extern "C" int rigl_maxpool_same_backward(const void* dy, const uint8_t* argmax, int n, int h, int w, int c,
                                          int ksize, int stride, void* dx, void* stream) {
  PoolGeom g;
  int rc = pool_geom(n, h, w, c, ksize, stride, &g);
  if (rc != RIGL_OK) return rc;
  RIGL_REQUIRE(dy && dx && argmax, "rigl_maxpool_same_backward: null tensor");
  RIGL_REQUIRE(g.h <= 65535 && n <= 65535, "rigl_maxpool_same_backward: extent too large");
  if (g.k == 3 && g.s == 2 && g.pad == 0 && (g.h & 1) == 0 && (g.w & 1) == 0) {
    const dim3 block(8, 32), grid((unsigned)((g.w / 2 + 31) / 32), (unsigned)(g.h / 2), (unsigned)n);
    k_maxpool_bwd_3x3s2<<<grid, block, 0, (cudaStream_t)stream>>>(g, (const __nv_bfloat16*)dy, argmax,
                                                                   (__nv_bfloat16*)dx);
    RIGL_LAUNCH_CHECK("k_maxpool_bwd_3x3s2");
    return RIGL_OK;
  }
  const dim3 block(8, 32), grid((unsigned)((g.w + 31) / 32), (unsigned)g.h, (unsigned)n);
  k_maxpool_bwd<<<grid, block, 0, (cudaStream_t)stream>>>(g, (const __nv_bfloat16*)dy, argmax, (__nv_bfloat16*)dx);
  RIGL_LAUNCH_CHECK("k_maxpool_bwd");
  return RIGL_OK;
}

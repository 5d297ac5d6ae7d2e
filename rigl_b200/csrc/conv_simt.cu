// CUDA-core (SIMT) masked conv / linear kernels: the shape-agnostic path.
//
// Used (a) for shapes the TMA/tcgen05 path cannot address (channel counts that
// are not multiples of 8, i.e. row pitches that are not 16-byte multiples: the
// 7x7x3 stem, 10-way logits, unit-test layers) and (b) as the on-device
// cross-check of the tcgen05 kernels (RIGL_FORCE_SIMT=1).  bf16 operands, fp32
// accumulation, same packed masked-weight operands as the tensor-core path.
#include <cuda_bf16.h>

#include "common.cuh"
#include "conv_common.cuh"

namespace rigl {

// y[p, co] = sum_{tap, ci} x[pix(p, tap), ci] * wd[tap][ci][co]      (wd = w_dgrad layout)
// grid: (ceil(pixels/4), ceil(cout/64)); block (64, 4)
// AFF: inference epilogue y = [relu](acc * scale[co] + shift[co] (+ residual[p, co])), one bf16 rounding.
template <bool AFF>
__global__ void k_simt_fprop(ConvGeom g, const __nv_bfloat16* __restrict__ x,
                             const __nv_bfloat16* __restrict__ wd, __nv_bfloat16* __restrict__ y,
                             float* __restrict__ y_f32, const float* __restrict__ bias,
                             const float* __restrict__ scale, const float* __restrict__ shift,
                             const __nv_bfloat16* __restrict__ residual, int relu) {
  const int co = blockIdx.y * 64 + threadIdx.x;
  const int64_t p = (int64_t)blockIdx.x * 4 + threadIdx.y;
  if (p >= g.out_pixels() || co >= g.cout) return;
  const int wo = (int)(p % g.out_w);
  const int ho = (int)((p / g.out_w) % g.out_h);
  const int n = (int)(p / ((int64_t)g.out_w * g.out_h));
  float acc = bias ? bias[co] : 0.f;
  for (int kh = 0; kh < g.ksize; ++kh) {
    const int hi = ho * g.stride + kh - g.pad;
    if (hi < 0 || hi >= g.in_h) continue;
    for (int kw = 0; kw < g.ksize; ++kw) {
      const int wi = wo * g.stride + kw - g.pad;
      if (wi < 0 || wi >= g.in_w) continue;
      const __nv_bfloat16* xr = x + (((int64_t)n * g.in_h + hi) * g.in_w + wi) * g.x_pitch;
      const __nv_bfloat16* wr = wd + (int64_t)(kh * g.ksize + kw) * g.cin * g.cout_pad + co;
      for (int ci = 0; ci < g.cin; ++ci)
        acc = fmaf(__bfloat162float(xr[ci]), __bfloat162float(wr[(int64_t)ci * g.cout_pad]), acc);
    }
  }
  if constexpr (AFF) {
    acc = fmaf(acc, scale ? scale[co] : 1.f, shift ? shift[co] : 0.f);
    if (residual) acc += __bfloat162float(residual[p * g.cout + co]);
    if (relu) acc = fmaxf(acc, 0.f);
  }
  if (y) y[p * g.cout + co] = __float2bfloat16(acc);
  if (y_f32) y_f32[p * g.cout + co] = acc;
}

// dx[q, ci] = sum_{tap, co} dy[pix_out(q, tap), co] * wf[tap][co][ci]   (wf = w_fprop layout)
// grid: (ceil(in_pixels/4), ceil(cin/64)); block (64, 4)
__global__ void k_simt_dgrad(ConvGeom g, const __nv_bfloat16* __restrict__ dy,
                             const __nv_bfloat16* __restrict__ wf, __nv_bfloat16* __restrict__ dx) {
  const int ci = blockIdx.y * 64 + threadIdx.x;
  const int64_t q = (int64_t)blockIdx.x * 4 + threadIdx.y;
  if (q >= g.in_pixels() || ci >= g.cin) return;
  const int wi = (int)(q % g.in_w);
  const int hi = (int)((q / g.in_w) % g.in_h);
  const int n = (int)(q / ((int64_t)g.in_w * g.in_h));
  float acc = 0.f;
  for (int kh = 0; kh < g.ksize; ++kh) {
    const int hn = hi + g.pad - kh;
    if (hn < 0 || hn % g.stride) continue;
    const int ho = hn / g.stride;
    if (ho >= g.out_h) continue;
    for (int kw = 0; kw < g.ksize; ++kw) {
      const int wn = wi + g.pad - kw;
      if (wn < 0 || wn % g.stride) continue;
      const int wo = wn / g.stride;
      if (wo >= g.out_w) continue;
      const __nv_bfloat16* dr = dy + (((int64_t)n * g.out_h + ho) * g.out_w + wo) * g.cout;
      const __nv_bfloat16* wr = wf + (int64_t)(kh * g.ksize + kw) * g.cout * g.cin_pad + ci;
      for (int co = 0; co < g.cout; ++co)
        acc = fmaf(__bfloat162float(dr[co]), __bfloat162float(wr[(int64_t)co * g.cin_pad]), acc);
    }
  }
  dx[q * g.x_pitch + ci] = __float2bfloat16(acc);
}

// dw[tap][ci][co] += sum_{p in chunk} x[pix(p,tap), ci] * dy[p, co]
// grid: (ceil(taps*cin*cout/256), ceil(pixels/chunk)); block 256; fp32 atomics.
__global__ void k_simt_wgrad(ConvGeom g, const __nv_bfloat16* __restrict__ x,
                             const __nv_bfloat16* __restrict__ dy, float* __restrict__ dw, int chunk) {
  const int64_t o = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int64_t total = (int64_t)g.ksize * g.ksize * g.cin * g.cout;
  if (o >= total) return;
  const int co = (int)(o % g.cout);
  const int ci = (int)((o / g.cout) % g.cin);
  const int tap = (int)(o / ((int64_t)g.cout * g.cin));
  const int kh = tap / g.ksize, kw = tap % g.ksize;
  const int64_t p0 = (int64_t)blockIdx.y * chunk;
  const int64_t p1 = min(p0 + chunk, g.out_pixels());
  float acc = 0.f;
  for (int64_t p = p0; p < p1; ++p) {
    const int wo = (int)(p % g.out_w);
    const int ho = (int)((p / g.out_w) % g.out_h);
    const int n = (int)(p / ((int64_t)g.out_w * g.out_h));
    const int hi = ho * g.stride + kh - g.pad, wi = wo * g.stride + kw - g.pad;
    if (hi < 0 || hi >= g.in_h || wi < 0 || wi >= g.in_w) continue;
    acc = fmaf(__bfloat162float(x[(((int64_t)n * g.in_h + hi) * g.in_w + wi) * g.x_pitch + ci]),
               __bfloat162float(dy[p * g.cout + co]), acc);
  }
  atomicAdd(dw + o, acc);
}

// Patch matrix: out[p][(kh*k+kw)*cin + ci] = x[pix(p, kh, kw), ci].
// One block = kTP consecutive output pixels of one output row: the k input rows they touch
// are staged in shared memory with coalesced reads, then every thread emits 16-byte chunks
// of the output rows, so the (large) write stream is fully coalesced.
constexpr int kTP = 64;
__global__ void __launch_bounds__(256)
k_im2col(ConvGeom g, const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int64_t out_pitch) {
  extern __shared__ __nv_bfloat16 sm[];
  const int segs = (g.out_w + kTP - 1) / kTP;
  const int seg = blockIdx.x % segs;
  const int ho = (blockIdx.x / segs) % g.out_h;
  const int n = blockIdx.x / (segs * g.out_h);
  const int wo0 = seg * kTP;
  const int npix = min(kTP, g.out_w - wo0);
  const int span = (kTP - 1) * g.stride + g.ksize;
  const int rowlen = span * g.cin;
  const int wi0 = wo0 * g.stride - g.pad;
  const __nv_bfloat16 zero = __float2bfloat16(0.f);
  for (int idx = threadIdx.x; idx < g.ksize * rowlen; idx += blockDim.x) {
    const int kh = idx / rowlen, r = idx - kh * rowlen;
    const int wi = wi0 + r / g.cin, c = r % g.cin;
    const int hi = ho * g.stride + kh - g.pad;
    __nv_bfloat16 v = zero;
    if (hi >= 0 && hi < g.in_h && wi >= 0 && wi < g.in_w)
      v = x[(((int64_t)n * g.in_h + hi) * g.in_w + wi) * g.x_pitch + c];
    sm[idx] = v;
  }
  // source offset (inside the staged rows, for pixel 0) of every output column: no divisions
  // in the streaming loop
  const int kc = g.ksize * g.cin;                 // elements per kh segment
  const int K = g.ksize * kc;
  int* src_off = reinterpret_cast<int*>(sm + ((g.ksize * rowlen + 7) & ~7));
  for (int kk = threadIdx.x; kk < (int)out_pitch; kk += blockDim.x) {
    const int kh = kk / kc;
    src_off[kk] = kk < K ? kh * rowlen + (kk - kh * kc) : -1;
  }
  __syncthreads();
  const int cpr = (int)(out_pitch / 8);           // 16-byte chunks per output row
  const int pstep = g.stride * g.cin;
  const int64_t p0 = ((int64_t)n * g.out_h + ho) * g.out_w + wo0;
  for (int q = threadIdx.x; q < npix * cpr; q += blockDim.x) {
    const int pl = q / cpr, j = q - pl * cpr;
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int so = src_off[8 * j + e];
      v[e] = so >= 0 ? sm[so + pl * pstep] : zero;
    }
    *reinterpret_cast<uint4*>(out + (p0 + pl) * out_pitch + 8 * j) = *reinterpret_cast<const uint4*>(v);
  }
}

int simt_im2col(const ConvGeom& g, const void* x, void* out, int64_t out_pitch, cudaStream_t s) {
  RIGL_REQUIRE(out_pitch % 8 == 0 && aligned16(out), "rigl_im2col_nhwc: out_pitch must be a multiple of 8");
  const int segs = (g.out_w + kTP - 1) / kTP;
  const int span = (kTP - 1) * g.stride + g.ksize;
  const size_t smem = (((size_t)g.ksize * span * g.cin + 7) & ~(size_t)7) * sizeof(__nv_bfloat16) +
                      (size_t)out_pitch * sizeof(int);
  RIGL_REQUIRE(smem <= 48 * 1024, "rigl_im2col_nhwc: patch rows too large for shared memory (%zu B)", smem);
  const int64_t blocks = (int64_t)g.batch * g.out_h * segs;
  k_im2col<<<(unsigned)blocks, 256, smem, s>>>(g, (const __nv_bfloat16*)x, (__nv_bfloat16*)out, out_pitch);
  RIGL_LAUNCH_CHECK("k_im2col");
  return RIGL_OK;
}

int simt_fprop(const ConvGeom& g, const void* x, const void* w_dgrad, void* y, float* y_f32,
               const float* bias, cudaStream_t s, const AffineEpi* epi) {
  dim3 grid((unsigned)((g.out_pixels() + 3) / 4), (g.cout + 63) / 64), block(64, 4);
  if (epi != nullptr)
    k_simt_fprop<true><<<grid, block, 0, s>>>(g, (const __nv_bfloat16*)x, (const __nv_bfloat16*)w_dgrad,
                                              (__nv_bfloat16*)y, y_f32, bias, epi->scale, epi->shift,
                                              (const __nv_bfloat16*)epi->residual, epi->relu);
  else
    k_simt_fprop<false><<<grid, block, 0, s>>>(g, (const __nv_bfloat16*)x, (const __nv_bfloat16*)w_dgrad,
                                               (__nv_bfloat16*)y, y_f32, bias, nullptr, nullptr, nullptr, 0);
  RIGL_LAUNCH_CHECK("k_simt_fprop");
  return RIGL_OK;
}

int simt_dgrad(const ConvGeom& g, const void* dy, const void* w_fprop, void* dx, cudaStream_t s) {
  dim3 grid((unsigned)((g.in_pixels() + 3) / 4), (g.cin + 63) / 64), block(64, 4);
  k_simt_dgrad<<<grid, block, 0, s>>>(g, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)w_fprop,
                                      (__nv_bfloat16*)dx);
  RIGL_LAUNCH_CHECK("k_simt_dgrad");
  return RIGL_OK;
}

int simt_wgrad(const ConvGeom& g, const void* x, const void* dy, float* dw, float beta, cudaStream_t s) {
  const int64_t total = (int64_t)g.ksize * g.ksize * g.cin * g.cout;
  if (beta == 0.f) RIGL_CUDA(cudaMemsetAsync(dw, 0, total * sizeof(float), s));
  int chunk = 2048;
  while ((g.out_pixels() + chunk - 1) / chunk > 65535) chunk *= 2;
  dim3 grid((unsigned)((total + 255) / 256), (unsigned)((g.out_pixels() + chunk - 1) / chunk));
  k_simt_wgrad<<<grid, 256, 0, s>>>(g, (const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, dw, chunk);
  RIGL_LAUNCH_CHECK("k_simt_wgrad");
  return RIGL_OK;
}

}  // namespace rigl

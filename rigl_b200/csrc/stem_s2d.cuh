// Space-to-depth stem kernels (layers.STEM_S2D_PATH, default on; validated on B200 in round 2 by
// tools/umma_sw32_probe.cu and tests/test_conv_gpu.py::test_conv_stem_s2d_path).  Design: DESIGN.md 3.7.
//
// The 7x7 / stride-2 / 3-channel stem without a patch matrix.  The zero-padded input is folded
// 2x2 -> channels ("space to depth"): xs[n, hs, ws, (dy*2+dx)*3 + c] = xpad[n, 2hs+dy, 2ws+dx, c],
// 16 bf16 = 32 bytes per folded pixel (slots 12..15 zero).  The conv becomes a 4x4 / stride-1
// conv over 16 channels (taps (th, tw), weights of the non-existent kh = 7 / kw = 7 zero), i.e.
// exactly ONE K = 16 tcgen05.mma per tap, and the halo trick of halo3x3.cuh applies with
// 32-byte rows: one halo tile of (R+3) folded rows x 128 columns (TMA, SWIZZLE_32B, OOB zero fill)
// feeds all 16 taps through row-shifted descriptors (tap (th,tw): +th*128 + tw rows).  An M tile
// is one output row (128 positions, 112 valid); the 32 KB weight operand stays resident.
//
// wgrad: A = the same halo tile read MN-major (row = position = K index, 32 B = 16 folded channels):
// M = 128 is EIGHT 16-channel atoms LBO = 32 B apart = eight horizontally neighbouring taps
// (tw = 0..7, the last four unused), so one MMA per th accumulates a whole filter row; B = the dY
// tile (MN-major, SWIZZLE_128B, padding columns zero-filled by TMA).  Four accumulators of 64
// columns; per-CTA fp32 partials [th][tw*16 + k16][co], then k_stem_s2d_reduce scatters them into
// the dense HWIO gradient in CTA order (deterministic).
//
// Open hardware questions (tools/umma_sw32_probe.cu): row-shifted descriptors under SWIZZLE_32B,
// and 8 MN atoms addressed through LBO.
//
// Included by igemm_tc.cu inside namespace rigl.
#pragma once

struct S2dParams {
  int H, W;                     // output extents (conv output = in/2)
  int NB;
  int HS, WS;                   // folded input extents: (in + 2*pad) / 2
  int R;                        // output rows per strip (= M tiles per strip)
  int nbuf;
  int strips_per_image, total_strips;
  int N;                        // output channels (<= 64)
  uint32_t a_buf_bytes;         // halo tile incl. slack rows, multiple of 1024
  uint32_t a_tx_bytes;
  float* wgrad_out;             // wgrad: [gridDim.x][4][128][64] fp32
};

constexpr int kS2dWp = 128;                               // halo pitch (positions per M tile)
constexpr uint32_t kS2dBTapBytes = 64 * 16 * 2;           // one tap of the weight operand: 64 rows x 32 B
constexpr uint32_t kS2dSwz32 = 6;                         // UMMA descriptor layout type: SWIZZLE_32B

__device__ __forceinline__ uint64_t make_smem_desc_swz(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t swz) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)swz << 61;
  return d;
}

// ---- input fold: x [N,H,W,cin<=3] (pitch x_pitch) -> xs [N,HS,WS,16] ----
__global__ void __launch_bounds__(256)
k_stem_s2d_fold(ConvGeom g, int hs, int ws, const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ xs) {
  const long long total = (long long)g.batch * hs * ws;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int wx = (int)(i % ws), hy = (int)((i / ws) % hs), n = (int)(i / ((long long)ws * hs));
    __align__(16) __nv_bfloat16 v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = __float2bfloat16(0.f);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int hi = 2 * hy + dy - g.pad, wi = 2 * wx + dx - g.pad;
        if (hi >= 0 && hi < g.in_h && wi >= 0 && wi < g.in_w) {
          const __nv_bfloat16* src = x + (((long long)n * g.in_h + hi) * g.in_w + wi) * g.x_pitch;
          for (int c = 0; c < g.cin; ++c) v[(dy * 2 + dx) * 3 + c] = src[c];
        }
      }
    uint4* dst = reinterpret_cast<uint4*>(xs + i * 16);
    dst[0] = reinterpret_cast<const uint4*>(v)[0];
    dst[1] = reinterpret_cast<const uint4*>(v)[1];
  }
}

// ---- weights: fp32 HWIO [7][7][cin][cout] + bitmap -> bf16 [16 taps][cout][16] (mask fused) ----
__global__ void __launch_bounds__(256)
k_stem_s2d_pack(ConvGeom g, const float* __restrict__ w, const uint32_t* __restrict__ bits,
                __nv_bfloat16* __restrict__ out) {
  const int total = 16 * g.cout * 16;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k16 = i % 16, co = (i / 16) % g.cout, tap = i / (16 * g.cout);
  const int th = tap / 4, tw = tap % 4, q = k16 / 3, c = k16 % 3;
  const int kh = 2 * th + (q >> 1), kw = 2 * tw + (q & 1);
  float v = 0.f;
  if (k16 < 12 && c < g.cin && kh < g.ksize && kw < g.ksize) {
    const long long flat = (((long long)kh * g.ksize + kw) * g.cin + c) * g.cout + co;
    if ((bits[flat >> 5] >> (flat & 31)) & 1u) v = w[flat];
  }
  out[i] = __float2bfloat16(v);
}

// ---- forward ----
__global__ void __launch_bounds__(kThreads, 1)
k_stem_s2d_fprop(const __grid_constant__ CUtensorMap amap, const __grid_constant__ CUtensorMap bmap,
                 const __grid_constant__ CUtensorMap omap, const S2dParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kIdesc = make_idesc_bf16(128, 64, 0, 0);
  constexpr uint32_t kSlab = 128 * 64 * 2;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_base = smem_base;                                   // 16 taps x 2 KB
  const uint32_t a_base = b_base + 16 * kS2dBTapBytes;
  const uint32_t out_base = a_base + p.nbuf * p.a_buf_bytes;
  const uint32_t bar_base = out_base + 2 * kSlab;
  const uint32_t b_full = bar_base;
  auto a_full = [&](int b) { return bar_base + 8u * (1 + b); };
  auto a_empty = [&](int b) { return bar_base + 8u * (5 + b); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (9 + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (11 + a); };
  const uint32_t tmem_slot = bar_base + 8u * 13;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&amap); prefetch_tmap(&bmap); prefetch_tmap(&omap);
    mbar_init(b_full, 1);
    for (int b = 0; b < p.nbuf; ++b) { mbar_init(a_full(b), 1); mbar_init(a_empty(b), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (elect_one()) {
      mbar_arrive_expect_tx(b_full, 16 * kS2dBTapBytes);
      for (int t = 0; t < 16; ++t) tma_load_3d(b_base + t * kS2dBTapBytes, &bmap, b_full, 0, 0, t);
      int buf = 0; uint32_t phase = 0;
      for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
        const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
        mbar_wait(a_empty(buf), phase ^ 1u);
        mbar_arrive_expect_tx(a_full(buf), p.a_tx_bytes);
        tma_load_4d(a_base + buf * p.a_buf_bytes, &amap, a_full(buf), 0, 0, h0, n);   // folded rows h0 .. h0+R+2
        if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    mbar_wait(b_full, 0);
    int buf = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    const uint64_t b_desc0 = make_smem_desc_swz(b_base, 16, 256, kS2dSwz32);
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      mbar_wait(a_full(buf), phase);
      tc_fence_after();
      const uint64_t a_desc0 = make_smem_desc_swz(a_base + buf * p.a_buf_bytes, 16, 256, kS2dSwz32);
      for (int t = 0; t < p.R; ++t) {                        // M tile t = output row h0 + t
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 64);
        if (elect_one()) {
#pragma unroll
          for (int tap = 0; tap < 16; ++tap) {               // rows of 32 B = 2 address units each
            const int row = (t + (tap >> 2)) * kS2dWp + (tap & 3);
            umma_bf16(d_tmem, a_desc0 + (uint64_t)(row * 2), b_desc0 + (uint64_t)(tap * (kS2dBTapBytes >> 4)), kIdesc,
                      tap == 0 ? 0u : 1u);
          }
          umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      if (elect_one()) umma_commit(a_empty(buf));
      __syncwarp();
      if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
    }
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const bool issuer = (warp == 2 && lane == 0);
    int acc = 0; uint32_t acc_phase = 0;
    uint32_t slab_ctr = 0;
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
      for (int t = 0; t < p.R; ++t) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t slab = out_base + (slab_ctr & 1u) * kSlab;
        if (issuer) tma_store_wait_read<1>();
        named_bar_sync(1, 128);
        uint32_t r0[32], r1[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 64), r0);
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 64 + 32), r1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        stage_row_bf16(slab, row, r0, r1, false);
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (issuer) {                                        // columns >= W and rows >= H are clipped by TMA
          tma_store_4d(&omap, slab, 0, 0, h0 + t, n);
          tma_store_commit();
        }
        ++slab_ctr;
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    if (issuer) tma_store_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

// ---- wgrad ----
__global__ void __launch_bounds__(kThreads, 1)
k_stem_s2d_wgrad(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ CUtensorMap dymap,
                 const S2dParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kIdesc = make_idesc_bf16(128, 64, 1, 1);
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t dy_bytes = (uint32_t)(p.R * kS2dWp) * 128u;
  const uint32_t stage_bytes = p.a_buf_bytes + dy_bytes;               // [x halo | dy]
  const uint32_t bar_base = smem_base + p.nbuf * stage_bytes;
  auto full_bar = [&](int b) { return bar_base + 8u * b; };
  auto empty_bar = [&](int b) { return bar_base + 8u * (4 + b); };
  const uint32_t tfull = bar_base + 8u * 8;
  const uint32_t tmem_slot = bar_base + 8u * 9;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&xmap); prefetch_tmap(&dymap);
    for (int b = 0; b < p.nbuf; ++b) { mbar_init(full_bar(b), 1); mbar_init(empty_bar(b), 1); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  {   // slack rows behind each halo tile are read against zero dY columns: they must be finite
    const uint32_t slack = p.a_buf_bytes - p.a_tx_bytes;
    for (int b = 0; b < p.nbuf; ++b)
      for (uint32_t i = threadIdx.x * 16u; i < slack; i += kThreads * 16u)
        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(smem_base + b * stage_bytes + p.a_tx_bytes + i), "r"(0u)
                     : "memory");
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (elect_one()) {
      int buf = 0; uint32_t phase = 0;
      for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
        const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
        mbar_wait(empty_bar(buf), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(buf), p.a_tx_bytes + dy_bytes);
        const uint32_t x_dst = smem_base + buf * stage_bytes;
        tma_load_4d(x_dst, &xmap, full_bar(buf), 0, 0, h0, n);
        tma_load_4d(x_dst + p.a_buf_bytes, &dymap, full_bar(buf), 0, 0, h0, n);
        if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    int buf = 0; uint32_t phase = 0;
    bool first = true;
    const int ksteps = p.R * kS2dWp / 16;
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      mbar_wait(full_bar(buf), phase);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t x_src = smem_base + buf * stage_bytes;
        const uint64_t db0 = make_smem_desc_swz(x_src + p.a_buf_bytes, 8192, 1024, 2);          // dY: 128-byte rows
        uint64_t da0[4];
#pragma unroll
        for (int th = 0; th < 4; ++th)       // 8 atoms of 16 channels, one 32-byte row apart: taps (th, tw = 0..7)
          da0[th] = make_smem_desc_swz(x_src + (uint32_t)(th * kS2dWp) * 32u, 32, 256, kS2dSwz32);
#pragma unroll 2
        for (int k = 0; k < ksteps; ++k) {                   // 16 positions: +512 B of x rows, +2048 B of dY rows
#pragma unroll
          for (int th = 0; th < 4; ++th)
            umma_bf16(tmem_base + (uint32_t)(th * 64), da0[th] + (uint64_t)(32 * k), db0 + (uint64_t)(128 * k), kIdesc,
                      (first && k == 0) ? 0u : 1u);
        }
        umma_commit(empty_bar(buf));
      }
      __syncwarp();
      first = false;
      if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
    }
    if (elect_one()) umma_commit(tfull);
    __syncwarp();
  } else {
    const int quad = warp & 3;
    mbar_wait(tfull, 0);
    tc_fence_after();
    float* part = p.wgrad_out + (size_t)blockIdx.x * 4 * 128 * 64;
#pragma unroll 1
    for (int th = 0; th < 4; ++th) {
      float* dst_row = part + ((size_t)th * 128 + quad * 32 + lane) * 64;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r32[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(th * 64 + c0), r32);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 32; q += 4)
          *reinterpret_cast<float4*>(dst_row + c0 + q) =
              make_float4(__uint_as_float(r32[q]), __uint_as_float(r32[q + 1]), __uint_as_float(r32[q + 2]),
                          __uint_as_float(r32[q + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// dw[kh][kw][c][co] = beta * dw + sum over CTAs of partial[cta][kh/2][(kw/2)*16 + ((kh&1)*2 + (kw&1))*3 + c][co]
__global__ void __launch_bounds__(256)
k_stem_s2d_reduce(ConvGeom g, const float* __restrict__ part, int nparts, float* __restrict__ dw, float beta) {
  const int total = g.ksize * g.ksize * g.cin * g.cout;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int co = i % g.cout, c = (i / g.cout) % g.cin, kw = (i / (g.cout * g.cin)) % g.ksize, kh = i / (g.cout * g.cin * g.ksize);
  const int th = kh >> 1, row = (kw >> 1) * 16 + ((kh & 1) * 2 + (kw & 1)) * 3 + c;
  const float* src = part + ((size_t)th * 128 + row) * 64 + co;
  float a = beta != 0.f ? beta * dw[i] : 0.f;
  for (int s = 0; s < nparts; ++s) a += src[(size_t)s * 4 * 128 * 64];
  dw[i] = a;
}

// ---------------------------------------------------------------------------- host side
static bool s2d_geom(const ConvGeom& g, S2dParams* p, bool wgrad) {
  if (g.ksize != 7 || g.stride != 2 || g.pad != 3 || g.cin > 3 || g.cin < 1) return false;
  if ((g.in_h & 1) || (g.in_w & 1) || g.cout > 64 || (g.cout % 8)) return false;
  if (g.out_h != g.in_h / 2 || g.out_w != g.in_w / 2 || g.out_w + 3 > kS2dWp) return false;
  p->H = g.out_h; p->W = g.out_w; p->NB = g.batch;
  p->HS = (g.in_h + 2 * g.pad) / 2; p->WS = (g.in_w + 2 * g.pad) / 2;
  p->R = wgrad ? 4 : 8;
  p->nbuf = wgrad ? 2 : 3;
  if (p->R > g.out_h) p->R = g.out_h;
  p->strips_per_image = (g.out_h + p->R - 1) / p->R;
  p->total_strips = p->strips_per_image * g.batch;
  p->N = g.cout;
  p->a_tx_bytes = (uint32_t)((p->R + 3) * kS2dWp) * 32u;
  p->a_buf_bytes = (uint32_t)(((size_t)((p->R + 3) * kS2dWp + 8) * 32 + 1023) / 1024 * 1024);
  p->wgrad_out = nullptr;
  return true;
}

bool s2d_supported(const ConvGeom& g) {
  S2dParams p;
  return s2d_geom(g, &p, false);
}
size_t s2d_folded_bytes(const ConvGeom& g) {
  S2dParams p;
  if (!s2d_geom(g, &p, false)) return 0;
  return (size_t)g.batch * p.HS * p.WS * 32;
}
size_t s2d_packed_bytes(const ConvGeom& g) { return (size_t)16 * g.cout * 32; }
static int s2d_wgrad_grid(const S2dParams& p) {
  ensure_driver();
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  return p.total_strips < sms ? p.total_strips : sms;
}
size_t s2d_workspace_bytes(const ConvGeom& g) {
  S2dParams p;
  if (!s2d_geom(g, &p, true)) return 0;
  return (size_t)s2d_wgrad_grid(p) * 4 * 128 * 64 * sizeof(float) + 256;
}

int s2d_fold(const ConvGeom& g, const void* x, void* xs, cudaStream_t s) {
  S2dParams p;
  if (!s2d_geom(g, &p, false)) { set_error("rigl_stem_s2d: unsupported geometry"); return RIGL_ERR_UNSUPPORTED; }
  k_stem_s2d_fold<<<148 * 16, 256, 0, s>>>(g, p.HS, p.WS, (const __nv_bfloat16*)x, (__nv_bfloat16*)xs);
  RIGL_LAUNCH_CHECK("k_stem_s2d_fold");
  return RIGL_OK;
}

int s2d_pack(const ConvGeom& g, const float* w, const uint32_t* bits, void* packed, cudaStream_t s) {
  const int total = 16 * g.cout * 16;
  k_stem_s2d_pack<<<(total + 255) / 256, 256, 0, s>>>(g, w, bits, (__nv_bfloat16*)packed);
  RIGL_LAUNCH_CHECK("k_stem_s2d_pack");
  return RIGL_OK;
}

// folded-input view (16, WS, HS, N) with 32-byte rows
static int s2d_x_map(CUtensorMap* out, const void* xs, const S2dParams& p, int box_rows) {
  const uint64_t dims[4] = {16, (uint64_t)p.WS, (uint64_t)p.HS, (uint64_t)p.NB};
  const uint64_t strides[3] = {32, (uint64_t)p.WS * 32, (uint64_t)p.HS * p.WS * 32};
  const uint32_t box[4] = {16, (uint32_t)kS2dWp, (uint32_t)box_rows, 1};
  return make_tmap_swz(out, xs, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

int s2d_fprop(const ConvGeom& g, const void* xs, const void* packed, void* y, cudaStream_t s) {
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  S2dParams p;
  if (!s2d_geom(g, &p, false)) { set_error("rigl_stem_s2d_fprop: unsupported geometry"); return RIGL_ERR_UNSUPPORTED; }
  CUtensorMap amap, bmap, omap;
  rc = s2d_x_map(&amap, xs, p, p.R + 3);
  if (rc != RIGL_OK) return rc;
  const uint64_t bdims[3] = {16, (uint64_t)g.cout, 16};
  const uint64_t bstr[2] = {32, (uint64_t)g.cout * 32};
  const uint32_t bbox[3] = {16, 64, 1};
  rc = make_tmap_swz(&bmap, packed, 3, bdims, bstr, bbox, CU_TENSOR_MAP_SWIZZLE_32B);
  if (rc != RIGL_OK) return rc;
  const uint32_t obox[4] = {64, (uint32_t)kS2dWp, 1, 1};
  rc = make_act_map(&omap, y, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, obox);
  if (rc != RIGL_OK) return rc;
  const size_t smem = 16 * kS2dBTapBytes + p.nbuf * (size_t)p.a_buf_bytes + 2 * (128 * 64 * 2) + 1024 + 256;
  static size_t configured = 0;
  if (smem > configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_stem_s2d_fprop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  const int grid = p.total_strips < sms ? p.total_strips : sms;
  k_stem_s2d_fprop<<<grid, kThreads, smem, s>>>(amap, bmap, omap, p);
  RIGL_LAUNCH_CHECK("k_stem_s2d_fprop");
  return RIGL_OK;
}

int s2d_wgrad(const ConvGeom& g, const void* xs, const void* dy, float* dw, float beta, void* ws, size_t ws_bytes,
              cudaStream_t s) {
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  S2dParams p;
  if (!s2d_geom(g, &p, true)) { set_error("rigl_stem_s2d_wgrad: unsupported geometry"); return RIGL_ERR_UNSUPPORTED; }
  const int grid = s2d_wgrad_grid(p);
  const size_t need = (size_t)grid * 4 * 128 * 64 * sizeof(float);
  if (ws == nullptr || ws_bytes < need + 256) {
    set_error("rigl_stem_s2d_wgrad: workspace %zu < required %zu", ws_bytes, need + 256);
    return RIGL_ERR_WORKSPACE;
  }
  p.wgrad_out = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  CUtensorMap xmap, dymap;
  rc = s2d_x_map(&xmap, xs, p, p.R + 3);
  if (rc != RIGL_OK) return rc;
  const uint32_t dbox[4] = {64, (uint32_t)kS2dWp, (uint32_t)p.R, 1};
  rc = make_act_map(&dymap, dy, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, dbox);
  if (rc != RIGL_OK) return rc;
  const size_t smem = p.nbuf * ((size_t)p.a_buf_bytes + (size_t)p.R * kS2dWp * 128) + 1024 + 256;
  static size_t configured = 0;
  if (smem > configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_stem_s2d_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  k_stem_s2d_wgrad<<<grid, kThreads, smem, s>>>(xmap, dymap, p);
  RIGL_LAUNCH_CHECK("k_stem_s2d_wgrad");
  const int total = g.ksize * g.ksize * g.cin * g.cout;
  k_stem_s2d_reduce<<<(total + 255) / 256, 256, 0, s>>>(g, p.wgrad_out, grid, dw, beta);
  RIGL_LAUNCH_CHECK("k_stem_s2d_reduce");
  return RIGL_OK;
}

// 3x3 / stride 1 / pad 1 convolutions with at most 64 reduction channels ("halo" kernels).
//
// The generic implicit-GEMM kernels fetch one shifted TMA box per filter tap, so a 3x3 layer
// reads its input NINE times from L2; at 64 channels there is so little math per byte that the
// chip-wide L2 -> SM bandwidth (~6300 B/clk) is what bounds them (200 us for 59 GFLOP).
// Here a CTA loads ONE halo tile -- (R+2) image rows, each padded to a power-of-two pitch Wp
// >= W+2 by TMA out-of-bounds zero fill -- and feeds all nine taps from it: the UMMA shared
// memory descriptor of tap (dh, dw) simply starts (dh+1)*Wp + (dw+1) rows (128 B each) further
// down the tile.  SWIZZLE_128B is a function of the absolute shared-memory address, so a start
// address that is not 1024-byte aligned addresses the same swizzled bytes TMA wrote (verified on
// B200 by tools/umma_shift_probe.cu for every row shift, K-major and MN-major).
//
//   position q = r*Wp + c   (r = row inside the strip, c = column, c >= W is padding)
//   fprop/dgrad: D[q, n]   = sum_tap sum_k  X[q + off(tap), k] * Wt[tap][n, k]     (K-major A)
//   wgrad:       D[tap][ci, co] = sum_q X[q + off(tap), ci] * dY[q, co]            (MN-major A, B)
// Padding columns of the OUTPUT are clipped by the TMA store (fprop/dgrad) or multiply dY zeros
// (wgrad: the dY tile is loaded with the same pitch, its padding columns zero-filled).
//
// Included by igemm_tc.cu (uses its tensor-map helpers).
#pragma once
// (textually included inside namespace rigl)

struct HaloParams {
  int W, H, NB;                 // image extents (input == output)
  int Wp;                       // halo row pitch in pixels: power of two, W + 2 <= Wp <= 128
  int R;                        // output rows per strip (multiple of 128 / Wp)
  int T;                        // 128-position M tiles per strip (R * Wp / 128)
  int nbuf;                     // halo tiles in flight (2..4)
  int strips_per_image, total_strips;
  int N;                        // fprop/dgrad: output channels.  wgrad: co
  int ci;                       // wgrad: input channels (<= 64)
  int row_off[9];               // halo row offset of each tap: (dh+1)*Wp + (dw+1)
  uint32_t a_buf_bytes;         // halo tile incl. slack rows, multiple of 1024
  uint32_t a_tx_bytes;          // bytes the halo TMA box delivers
  float* wgrad_out;             // wgrad: [gridDim.x][9][ci][N] fp32 partials
};

constexpr uint32_t kHaloBTapBytes = 64 * 64 * 2;        // one tap of the resident weight tile: 8 KB
constexpr uint32_t kHaloSlabBytes = 128 * 64 * 2;       // output staging slab: 16 KB

// ----------------------------------------------------------------------------
// fprop / dgrad: weights of this CTA's 64-channel N tile stay resident in shared memory.
// grid = (CTAs over strips, N tiles).  warp 0: TMA, warp 1: MMA, warps 2-5: epilogue.
// ----------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
k_halo3x3_kmajor(const __grid_constant__ CUtensorMap amap, const __grid_constant__ CUtensorMap bmap,
                 const __grid_constant__ CUtensorMap omap, const HaloParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kIdesc = make_idesc_bf16(128, 64, 0, 0);
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_base = smem_base;                                   // 9 taps x 8 KB
  const uint32_t a_base = b_base + 9 * kHaloBTapBytes;                 // nbuf halo tiles
  const uint32_t out_base = a_base + p.nbuf * p.a_buf_bytes;           // 2 staging slabs
  const uint32_t bar_base = out_base + 2 * kHaloSlabBytes;
  const uint32_t b_full = bar_base;
  auto a_full = [&](int b) { return bar_base + 8u * (1 + b); };
  auto a_empty = [&](int b) { return bar_base + 8u * (5 + b); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (9 + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (11 + a); };
  const uint32_t tmem_slot = bar_base + 8u * 13;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tile = blockIdx.y;
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
  const int rt = 128 / p.Wp;                              // image rows per M tile

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(b_full, 9 * kHaloBTapBytes);
      for (int t = 0; t < 9; ++t) tma_load_3d(b_base + t * kHaloBTapBytes, &bmap, b_full, 0, n_tile * 64, t);
      int buf = 0; uint32_t phase = 0;
      for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
        const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
        mbar_wait(a_empty(buf), phase ^ 1u);
        mbar_arrive_expect_tx(a_full(buf), p.a_tx_bytes);
        tma_load_4d(a_base + buf * p.a_buf_bytes, &amap, a_full(buf), 0, -1, h0 - 1, n);
        if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // The whole warp runs the loop converged; one elected lane issues (see ptx::elect_one).
    mbar_wait(b_full, 0);
    int buf = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    const uint64_t b_desc0 = make_smem_desc(b_base, 16, 1024);
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      mbar_wait(a_full(buf), phase);
      tc_fence_after();
      const uint64_t a_desc0 = make_smem_desc(a_base + buf * p.a_buf_bytes, 16, 1024);
      for (int t = 0; t < p.T; ++t) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 64);
        if (elect_one()) {
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {              // descriptor start addresses are in 16-byte units
            const uint64_t da = a_desc0 + (uint64_t)((t * 128 + p.row_off[tap]) * 8);
            const uint64_t db = b_desc0 + (uint64_t)(tap * (kHaloBTapBytes >> 4));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, da + 2 * k, db + 2 * k, kIdesc, (tap == 0 && k == 0) ? 0u : 1u);
          }
          umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      if (elect_one()) umma_commit(a_empty(buf));          // halo tile reusable once its MMAs retire
      __syncwarp();
      if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
    }
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;                      // position inside the M tile
    const bool issuer = (warp == 2 && lane == 0);
    int acc = 0; uint32_t acc_phase = 0;
    uint32_t slab_ctr = 0;
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
      for (int t = 0; t < p.T; ++t) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t slab = out_base + (slab_ctr & 1u) * kHaloSlabBytes;
        if (issuer) tma_store_wait_read<1>();
        named_bar_sync(1, 128);
        uint32_t r0[32], r1[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 64), r0);
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 64 + 32), r1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));       // accumulator drained into registers
        stage_row_bf16(slab, row, r0, r1, false);
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (issuer) {                                      // columns >= W and rows >= H are clipped by TMA
          tma_store_4d(&omap, slab, n_tile * 64, 0, h0 + t * rt, n);
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

// ----------------------------------------------------------------------------
// wgrad: every CTA accumulates all nine taps over its strips in TMEM (five 128 x 64
// accumulators: two taps per MMA, the taps being the two 64-channel M atoms of an MN-major A
// operand whose atom stride (LBO) is the distance between the taps' halo rows), then writes one
// fp32 partial [9][ci][co]; k_splitk_reduce sums the partials in CTA order (deterministic).
// ----------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
k_halo3x3_wgrad(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ CUtensorMap dymap,
                const HaloParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kIdesc = make_idesc_bf16(128, 64, 1, 1);
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t dy_bytes = (uint32_t)(p.R * p.Wp) * 128u;
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
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  // The slack rows behind each halo tile are read (against zero dY columns): they must be finite.
  {
    const uint32_t halo_rows_bytes = p.a_tx_bytes;
    const uint32_t slack = p.a_buf_bytes - halo_rows_bytes;
    for (int b = 0; b < p.nbuf; ++b)
      for (uint32_t i = threadIdx.x * 16u; i < slack; i += kThreads * 16u)
        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(smem_base + b * stage_bytes + halo_rows_bytes + i), "r"(0u)
                     : "memory");
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int buf = 0; uint32_t phase = 0;
      for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
        const int n = strip / p.strips_per_image, h0 = (strip % p.strips_per_image) * p.R;
        mbar_wait(empty_bar(buf), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(buf), p.a_tx_bytes + dy_bytes);
        const uint32_t x_dst = smem_base + buf * stage_bytes;
        tma_load_4d(x_dst, &xmap, full_bar(buf), 0, -1, h0 - 1, n);
        tma_load_4d(x_dst + p.a_buf_bytes, &dymap, full_bar(buf), 0, 0, h0, n);
        if (++buf == p.nbuf) { buf = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    int buf = 0; uint32_t phase = 0;                       // converged warp, one elected lane issues
    bool first = true;
    const int ksteps = p.R * p.Wp / 16;
    for (int strip = blockIdx.x; strip < p.total_strips; strip += gridDim.x) {
      mbar_wait(full_bar(buf), phase);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t x_src = smem_base + buf * stage_bytes;
        const uint64_t db0 = make_smem_desc(x_src + p.a_buf_bytes, 8192, 1024);
        uint64_t da0[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          // accumulator j holds taps (2j, 2j+1); the last one pairs (7, 8): tap 7 is computed twice
          const int t0 = j < 4 ? 2 * j : 7, t1 = t0 + 1;
          da0[j] = make_smem_desc(x_src + (uint32_t)p.row_off[t0] * 128u,
                                  (uint32_t)(p.row_off[t1] - p.row_off[t0]) * 128u, 1024);
        }
#pragma unroll 2
        for (int k = 0; k < ksteps; ++k) {                 // 16 positions = +128 in the 16-byte address field
#pragma unroll
          for (int j = 0; j < 5; ++j)
            umma_bf16(tmem_base + (uint32_t)(j * 64), da0[j] + (uint64_t)(128 * k), db0 + (uint64_t)(128 * k), kIdesc,
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
    const int ci = (quad & 1) * 32 + lane;
    float* part = p.wgrad_out + (size_t)blockIdx.x * 9 * p.ci * p.N;
#pragma unroll 1
    for (int j = 0; j < 5; ++j) {
      const int t0 = j < 4 ? 2 * j : 7;
      const int tap = t0 + (quad >> 1);
      const bool dup = (j == 4 && (quad >> 1) == 0);       // second copy of tap 7
      float* dst_row = part + ((size_t)tap * p.ci + ci) * p.N;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r32[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(j * 64 + c0), r32);
        tmem_ld_wait();
        if (!dup && ci < p.ci && c0 < p.N) {
#pragma unroll
          for (int q = 0; q < 32; q += 4) {
            if (c0 + q + 4 <= p.N) {
              *reinterpret_cast<float4*>(dst_row + c0 + q) =
                  make_float4(__uint_as_float(r32[q]), __uint_as_float(r32[q + 1]), __uint_as_float(r32[q + 2]),
                              __uint_as_float(r32[q + 3]));
            } else {
              for (int t = 0; t < 4 && c0 + q + t < p.N; ++t) dst_row[c0 + q + t] = __uint_as_float(r32[q + t]);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ----------------------------------------------------------------------------
// Host side
// ----------------------------------------------------------------------------

// Geometry the halo kernels cover; `kred` = reduction channels per tap (cin for fprop, cout for dgrad).
static bool halo_geom(const ConvGeom& g, int kred, HaloParams* p, size_t smem_fixed, int dy_tile) {
  if (!g_halo || g.ksize != 3 || g.stride != 1 || g.pad != 1) return false;
  if (g.in_h != g.out_h || g.in_w != g.out_w || kred > 64 || kred % 8) return false;
  int wp = 8;
  while (wp < g.in_w + 2) wp *= 2;
  if (wp > 128 || g.in_w * 4 < wp * 3) return false;          // < 75 % useful positions: not worth it
  const int rt = 128 / wp;
  // Strip height R = rt*T and the number of halo tiles in flight.  One TMA box per strip means the
  // load pipeline is only as deep as the buffers: prefer >= 3 buffers (measured: the kernels are
  // load-latency bound with 2), then the tallest strip (smallest halo overhead (R+2)/R).
  int best_t = 0, best_nbuf = 0; long long best_cost = 0;
  for (int nbuf = 2; nbuf <= 4; ++nbuf)
    for (int t = 1; t <= 8; ++t) {
      const int r = rt * t;
      const size_t a_buf = ((size_t)((r + 2) * wp + 8) * 128 + 1023) / 1024 * 1024;
      const size_t need = smem_fixed + nbuf * (a_buf + (dy_tile ? (size_t)r * wp * 128 : 0)) + 2048;
      if (need > 227 * 1024) break;
      const long long strips = (g.in_h + r - 1) / r;
      // rows fetched + rows computed per image, scaled by a pipeline-depth penalty
      long long cost = (strips * (r + 2) + strips * r) * 16 + strips * 8;
      if (nbuf == 2) cost = cost * 3 / 2;
      if (best_t == 0 || cost < best_cost) { best_t = t; best_nbuf = nbuf; best_cost = cost; }
      if (r >= g.in_h) break;
    }
  if (best_t == 0) return false;
  p->W = g.in_w; p->H = g.in_h; p->NB = g.batch; p->Wp = wp;
  p->T = best_t; p->R = rt * best_t; p->nbuf = best_nbuf;
  p->strips_per_image = (g.in_h + p->R - 1) / p->R;
  p->total_strips = p->strips_per_image * g.batch;
  p->a_tx_bytes = (uint32_t)((p->R + 2) * wp) * 128u;
  p->a_buf_bytes = (uint32_t)(((size_t)((p->R + 2) * wp + 8) * 128 + 1023) / 1024 * 1024);
  return true;
}

static bool halo_fprop_ok(const ConvGeom& g, HaloParams* p) {
  return g.cout % 8 == 0 && g.x_pitch % 8 == 0 && halo_geom(g, g.cin, p, 9 * kHaloBTapBytes + 2 * kHaloSlabBytes, 0);
}
static bool halo_dgrad_ok(const ConvGeom& g, HaloParams* p) {
  return g.cin % 8 == 0 && g.x_pitch % 8 == 0 && halo_geom(g, g.cout, p, 9 * kHaloBTapBytes + 2 * kHaloSlabBytes, 0);
}
static bool halo_wgrad_ok(const ConvGeom& g, HaloParams* p) {
  return g.cout <= 64 && g.cout % 8 == 0 && g.x_pitch % 8 == 0 && halo_geom(g, g.cin, p, 0, 1);
}
static int halo_wgrad_grid(const HaloParams& p) {
  ensure_driver();
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  return p.total_strips < sms ? p.total_strips : sms;
}
static size_t halo_wgrad_ws_elems(const ConvGeom& g, const HaloParams& p) {
  return (size_t)halo_wgrad_grid(p) * 9 * g.cin * g.cout;
}

// in: activations [NB,H,W,kred] (pitch in_pitch); out: [NB,H,W,n_out] (pitch out_pitch);
// wts: packed [tap][n_out][kpad] K-major bf16; flip = dgrad (tap (kh,kw) reads the pixel at (1-kh, 1-kw)).
static int halo_launch_kmajor(HaloParams p, const void* in, int kred, int in_pitch, const void* wts, int kpad,
                              int n_out, void* out, int out_pitch, bool flip, cudaStream_t s) {
  for (int kh = 0; kh < 3; ++kh)
    for (int kw = 0; kw < 3; ++kw) {
      const int t = kh * 3 + kw;
      const int dh = flip ? 1 - kh : kh - 1, dw = flip ? 1 - kw : kw - 1;
      p.row_off[t] = (dh + 1) * p.Wp + (dw + 1);
    }
  p.N = n_out;
  CUtensorMap amap, bmap, omap;
  const uint32_t abox[4] = {64, (uint32_t)p.Wp, (uint32_t)(p.R + 2), 1};
  int rc = make_act_map(&amap, in, p.NB, p.H, p.W, kred, in_pitch, 1, 0, 0, abox);
  if (rc != RIGL_OK) return rc;
  const uint64_t bdims[3] = {(uint64_t)kpad, (uint64_t)n_out, 9};
  const uint64_t bstr[2] = {(uint64_t)kpad * 2, (uint64_t)n_out * kpad * 2};
  const uint32_t bbox[3] = {64, 64, 1};
  rc = make_tmap(&bmap, wts, 3, bdims, bstr, bbox);
  if (rc != RIGL_OK) return rc;
  const uint32_t obox[4] = {64, (uint32_t)p.Wp, (uint32_t)(128 / p.Wp), 1};
  rc = make_act_map(&omap, out, p.NB, p.H, p.W, n_out, out_pitch, 1, 0, 0, obox);
  if (rc != RIGL_OK) return rc;
  const size_t smem = 9 * kHaloBTapBytes + p.nbuf * (size_t)p.a_buf_bytes + 2 * kHaloSlabBytes + 1024 + 256;
  static size_t configured = 0;
  if (smem > configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_halo3x3_kmajor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  const int n_tiles = (n_out + 63) / 64;
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  int gx = sms / n_tiles;
  if (gx < 1) gx = 1;
  if (gx > p.total_strips) gx = p.total_strips;
  k_halo3x3_kmajor<<<dim3((unsigned)gx, (unsigned)n_tiles), kThreads, smem, s>>>(amap, bmap, omap, p);
  RIGL_LAUNCH_CHECK("k_halo3x3_kmajor");
  return RIGL_OK;
}

static int halo_launch_wgrad(HaloParams p, const ConvGeom& g, const void* x, const void* dy, float* partials,
                             cudaStream_t s) {
  for (int kh = 0; kh < 3; ++kh)
    for (int kw = 0; kw < 3; ++kw) {
      p.row_off[kh * 3 + kw] = kh * p.Wp + kw;
    }
  p.N = g.cout; p.ci = g.cin; p.wgrad_out = partials;
  CUtensorMap xmap, dymap;
  const uint32_t xbox[4] = {64, (uint32_t)p.Wp, (uint32_t)(p.R + 2), 1};
  int rc = make_act_map(&xmap, x, p.NB, p.H, p.W, g.cin, g.x_pitch, 1, 0, 0, xbox);
  if (rc != RIGL_OK) return rc;
  const uint32_t dbox[4] = {64, (uint32_t)p.Wp, (uint32_t)p.R, 1};
  rc = make_act_map(&dymap, dy, p.NB, p.H, p.W, g.cout, g.cout, 1, 0, 0, dbox);
  if (rc != RIGL_OK) return rc;
  const size_t smem = p.nbuf * ((size_t)p.a_buf_bytes + (size_t)p.R * p.Wp * 128) + 1024 + 256;
  static size_t configured = 0;
  if (smem > configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_halo3x3_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  k_halo3x3_wgrad<<<(unsigned)halo_wgrad_grid(p), kThreads, smem, s>>>(xmap, dymap, p);
  RIGL_LAUNCH_CHECK("k_halo3x3_wgrad");
  return RIGL_OK;
}


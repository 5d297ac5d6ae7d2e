// Masked conv2d / linear as implicit GEMM on the 5th-gen tensor cores (sm_100a).
//
//   fprop : y[pix, co]  = sum_{tap, ci} x[pix (+) tap, ci] * Wm[tap][co][ci]
//   dgrad : dx[pix, ci] = sum_{tap, co} dy[pix (-) tap, co] * Wm[tap][ci][co]
//   wgrad : dW[tap][ci][co] = sum_{pix} x[pix (+) tap, ci] * dy[pix, co]      (dense, fp32)
// Wm = mask * W is produced once per step by pack.cu; its per-tile survivor counts
// gate the weight-tile loads (an all-zero 64x64 weight tile costs no TMA and no MMA).
//
// No im2col buffer (except the 3-channel stem's patch matrix, conv_simt.cu): an M tile is a BOX of 128 output pixels
// (bw x bh x bn over width, height, batch) and, for filter tap (kh,kw), the A
// operand is the same box shifted by the tap offset, fetched by ONE 4-D TMA
// (cp.async.bulk.tensor.4d) whose out-of-bounds zero fill implements the padding.
// Stride-2 convs read through four parity sub-grid tensor maps (same trick,
// element strides doubled), so every conv shape in ResNet/WRN is a plain loop of
// TMA boxes + tcgen05.mma with fp32 accumulators in TMEM.
//
// Kernel organisation (persistent, one CTA per SM, 192 threads):
//   warp 0    : TMA producer (converged warp, one elect.sync lane issues)   smem ring, full/empty mbarriers
//   warp 1    : TMEM allocator + MMA issuer (same pattern): tcgen05.mma kind::f16, M = 128 per CTA
//   warps 2-5 : epilogue: tcgen05.ld 32x32b -> bf16 -> swizzled smem slab -> TMA store (or direct
//               fp32/bias stores), double-buffered accumulators so the epilogue of tile i overlaps
//               the main loop of tile i+1.
// Variants: k_igemm_kmajor (one CTA per tile, optional 2-CTA weight multicast, optional fused BN
// statistics), k_igemm_kmajor2 (default for fprop/dgrad: CTA pair, tcgen05 cta_group::2, M = 256),
// k_igemm_wgrad, and -- textually included below -- halo3x3.cuh (3x3/s1 layers with <= 64 channels:
// one smem halo tile feeds all nine taps) and stem_s2d.cuh (experimental).  Measured limits that
// shape these kernels (TMA ingest 54 B/clk/SM, cycles per MMA by N): DESIGN.md 3.2 / 3.7.
// fprop/dgrad use K-major operands; wgrad reduces over pixels, so both operands are
// MN-major views of the NHWC tensors (no transposes are materialised) and the
// pixel range is split across CTAs (deterministic two-pass split-K).
#include <cuda.h>
#include <cuda_bf16.h>

#include <stdio.h>
#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace rigl {

using namespace ptx;

constexpr int kMaxTaps = 9;
constexpr int kBM = 128;            // UMMA M
constexpr int kBK = 64;             // K block: 64 bf16 = one 128B swizzle row
constexpr int kThreads = 192;

struct TapInfo {
  int8_t map_id, dh, dw, pad;
  int32_t b_tap;                    // tap index into the packed weights
};

struct IgemmParams {
  int ntaps;
  TapInfo taps[kMaxTaps];
  int kblks;                        // K blocks per tap
  int GW, GH, NB;                   // pixel grid covered by this launch
  int bw, bh, bn;                   // pixel box of one M tile (bw*bh*bn == 128)
  int tiles_w, tiles_h, tiles_n;    // boxes per dimension
  int n_tiles;                      // tiles along the output-channel dim
  int N;                            // output channels
  __nv_bfloat16* out_bf16;
  float* out_f32;
  const float* bias;
  long long o_off, o_sn, o_sh, o_sw;   // element offsets of pixel (n,h,w) in the output
  const uint32_t* nnz;              // survivor counts per 64x64 weight tile (or null)
  int nnz_tap_stride, nnz_n_stride, nnz_k_stride;
  int tma_store;                    // 1: epilogue stages bf16 tiles in smem and TMA-stores them
  float* bn_partial;                // optional [gridDim.x][2][N]: per-CTA column sums / sums of squares of D
  int pair_local;                   // CTA-pair kernel: each CTA's TMA completes on its OWN barrier (see k_igemm_kmajor2)
  int stats_dbg;                    // development: 1 = statistics without the global REDs, 2 = without the smem pass
  // Inference epilogue (kernel variant AFF = true): y = [relu](acc * scale[c] + shift[c] (+ residual[pixel, c])).
  const float* ep_scale;            // [N] or null (1)
  const float* ep_shift;            // [N] or null (0)
  const __nv_bfloat16* ep_res;      // same shape and pixel offsets as the output, or null
  int ep_relu;
};

struct TMaps4 {
  CUtensorMap a[4];
};

__device__ __forceinline__ bool weight_block_live(const IgemmParams& p, int tap_idx, int n_tile, int kb, int bn64) {
  if (p.nnz == nullptr) return true;
  const uint32_t* base = p.nnz + (long long)p.taps[tap_idx].b_tap * p.nnz_tap_stride + (long long)kb * p.nnz_k_stride;
  uint32_t s = 0;
  for (int j = 0; j < bn64; ++j) {
    const int nt = n_tile * bn64 + j;
    if ((long long)nt * 64 < p.N) s += __ldg(base + (long long)nt * p.nnz_n_stride);
  }
  return s != 0;
}


// Liveness of every (tap, K block) of one N tile as a bitmask in shared memory, computed by a
// whole warp at the start of a tile (one round of parallel loads) instead of by the issuing
// thread once per K block: the single-thread TMA / MMA issue loops are instruction-latency bound
// (about 900 clk per stage with the survivor-table loads inline, which hid the TMA and tensor
// limits), so everything that can leave them does.  Block 0 is always live (it initialises D).
constexpr int kLiveWords = 10;        // 320 (tap, K block) pairs; longer reductions run without skipping
template <int kBN64>
__device__ __forceinline__ bool build_live_mask(const IgemmParams& p, int n_tile, int lane, uint32_t* mask_smem) {
  const int nkb = p.ntaps * p.kblks;
  if (p.nnz == nullptr || nkb > kLiveWords * 32) return false;       // no table (or too long): everything is live
  for (int w = 0; w * 32 < nkb; ++w) {
    const int j = w * 32 + lane;
    bool live = true;
    if (j > 0 && j < nkb) live = weight_block_live(p, j / p.kblks, n_tile, j % p.kblks, kBN64);
    const uint32_t m = __ballot_sync(0xffffffffu, live);
    if (lane == 0) mask_smem[w] = m;
  }
  __syncwarp();
  return true;
}

// ----------------------------------------------------------------------------
// fprop / dgrad kernel: D[128 pixels, BN] += A[128, 64] * B[BN, 64]^T per (tap, k block)
// ----------------------------------------------------------------------------
// Batch-norm statistics of one staged output slab (128 pixel rows x 64 channels, bf16, 128-byte rows with the
// 16-byte chunks XOR-swizzled by row & 7 -- exactly what the TMA store is about to read): column sums and sums of
// squares of the values AS STORED (bf16-rounded), added to this CTA's row of the partial table.
//   warp q (0..3) owns channels 16q..16q+15 (chunks 2q, 2q+1); lane = (row group g = lane >> 3, channel pair
//   cp = lane & 7); group g walks rows 32g + ((i + 2g) & 31), i = 0..31: the four groups then sit on four different
//   swizzle phases, so the 32 lanes of every LDS.32 hit 32 different banks.
// 32 LDS + ~130 FP ops per thread per slab, two shuffles per statistic, and ONE RED per (slab, channel, statistic):
// each table entry is only ever touched by one lane of one warp, in tile order, so the fp32 sums are deterministic.
// Rows outside the pixel grid are written as zeros by their owner (see the staging loops), so they do not count.
__device__ __forceinline__ void slab_bn_stats(uint32_t slab, int quad, int lane, float* __restrict__ bn_row, int co0,
                                              int n, int dbg) {
  const int cp = lane & 7, g = lane >> 3;
  const uint32_t chunk = (uint32_t)(2 * quad + (cp >> 2));
  const uint32_t word = (uint32_t)(cp & 3) * 4u;
  float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
  const int n_it = (dbg & 2) ? 0 : 32;
#pragma unroll 8
  for (int i = 0; i < n_it; ++i) {
    const uint32_t row = (uint32_t)(32 * g + ((i + 2 * g) & 31));
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(slab + row * 128u + (((chunk ^ (row & 7u)) << 4) | word)));
    const float a = __uint_as_float(v << 16), b = __uint_as_float(v & 0xffff0000u);
    s0 += a; s1 += b;
    q0 = fmaf(a, a, q0); q1 = fmaf(b, b, q1);
  }
#pragma unroll
  for (int o = 8; o <= 16; o <<= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    q0 += __shfl_xor_sync(0xffffffffu, q0, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o);
  }
  const int co = co0 + 16 * quad + 2 * cp;
  if (g == 0 && co < n && !(dbg & 1)) {          // (n is a multiple of 8 on this path, so co + 1 < n as well)
    atomicAdd(bn_row + co, s0); atomicAdd(bn_row + co + 1, s1);
    atomicAdd(bn_row + n + co, q0); atomicAdd(bn_row + n + co + 1, q1);
  }
}

// Inference epilogue on one thread's 64 fp32 accumulators of a staged slab (one pixel row, channels co0..co0+63),
// in place: the folded batch norm, the residual add and the ReLU happen before the single bf16 rounding.  N is a
// multiple of 8 on this path, so an 8-channel chunk is either wholly inside the output or wholly outside; the scale,
// shift (16-byte aligned, checked by the caller) and residual row (16-byte loads) are read only for chunks inside it.
__device__ __forceinline__ void slab_affine(const IgemmParams& p, uint32_t (&r0)[32], uint32_t (&r1)[32], int co0,
                                            long long o_pix, bool pix_ok) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int co = co0 + 8 * j;
    if (co >= p.N) break;
    float sc[8], sh[8], rs[8];
    if (p.ep_scale) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p.ep_scale + co));
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.ep_scale + co) + 1);
      sc[0] = a.x; sc[1] = a.y; sc[2] = a.z; sc[3] = a.w; sc[4] = b.x; sc[5] = b.y; sc[6] = b.z; sc[7] = b.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) sc[e] = 1.f;
    }
    if (p.ep_shift) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p.ep_shift + co));
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.ep_shift + co) + 1);
      sh[0] = a.x; sh[1] = a.y; sh[2] = a.z; sh[3] = a.w; sh[4] = b.x; sh[5] = b.y; sh[6] = b.z; sh[7] = b.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) sh[e] = 0.f;
    }
    uint4 rv = make_uint4(0u, 0u, 0u, 0u);
    if (p.ep_res && pix_ok) rv = __ldg(reinterpret_cast<const uint4*>(p.ep_res + o_pix + co));
    const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { rs[2 * e] = __uint_as_float(rw[e] << 16); rs[2 * e + 1] = __uint_as_float(rw[e] & 0xffff0000u); }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int i = 8 * j + e;
      float z = fmaf(__uint_as_float(i < 32 ? r0[i] : r1[i - 32]), sc[e], sh[e]);
      if (p.ep_res) z += rs[e];
      if (p.ep_relu) z = fmaxf(z, 0.f);
      if (i < 32) r0[i] = __float_as_uint(z); else r1[i - 32] = __float_as_uint(z);
    }
  }
}

// The same transform for one element (the direct-store epilogues: RIGL_TMA_STORE=0).
__device__ __forceinline__ float elem_affine(const IgemmParams& p, float a, int co, long long o) {
  float z = fmaf(a, p.ep_scale ? __ldg(p.ep_scale + co) : 1.f, p.ep_shift ? __ldg(p.ep_shift + co) : 0.f);
  if (p.ep_res) z += __bfloat162float(p.ep_res[o]);
  return p.ep_relu ? fmaxf(z, 0.f) : z;
}

// CL = CTAs per cluster (1 or 2).  With CL == 2 the two CTAs work on the two M tiles of a tile
// PAIR that share the weight tile: each loads HALF of B and multicasts it into both CTAs'
// shared memory, which cuts the L2->smem bytes per FLOP by a third (these kernels are bound
// by that traffic, not by the tensor pipe).  A stage is recycled only when BOTH consumers
// have released it (empty barriers count CL arrivals; tcgen05.commit multicasts them).
// AFF: the inference epilogue (slab_affine / elem_affine) is compiled in; AFF = false is the training kernel.
template <int BN, int STAGES, int CL, bool AFF>
__global__ void __launch_bounds__(kThreads, 1)
k_igemm_kmajor(const __grid_constant__ TMaps4 amaps, const __grid_constant__ CUtensorMap bmap,
               const __grid_constant__ CUtensorMap omap, const IgemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kABytes = kBM * kBK * 2;        // 16 KB
  constexpr uint32_t kBBytes = BN * kBK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  constexpr uint32_t kIdesc = make_idesc_bf16(kBM, BN, 0, 0);

  constexpr uint32_t kSlabBytes = kBM * 64 * 2;       // one 128-pixel x 64-channel output slab
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t out_base = smem_base + STAGES * kStageBytes;          // 2 staging slabs (1024B aligned)
  const uint32_t bar_base = out_base + 2 * kSlabBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  __shared__ uint32_t live_prod[kLiveWords], live_mma[kLiveWords];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) prefetch_tmap(&amaps.a[i]);
    prefetch_tmap(&bmap);
    if (p.tma_store) prefetch_tmap(&omap);
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), CL); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  if (CL > 1) cluster_sync_all(); else __syncthreads();       // peers' barriers are live before any multicast
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // Tile schedule: a "pair" = CL consecutive M tiles x one N tile; pairs are dealt round-robin to
  // clusters, N fastest (neighbouring clusters reuse the same activation tiles in L2).
  const uint32_t cta_rank = CL > 1 ? cluster_ctarank() : 0u;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int m_pairs = (m_tiles + CL - 1) / CL;
  const int total_pairs = m_pairs * p.n_tiles;
  const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;
  constexpr int kBN64 = (BN + 63) / 64;
  constexpr uint16_t kMcMask = (uint16_t)((1u << CL) - 1u);

  if (warp == 0) {
    // ===================== TMA producer (converged warp, one elected lane issues) =====================
    {
      int stage = 0; uint32_t phase = 0;
      for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
        const int n_tile = pair % p.n_tiles;
        const int m_tile = (pair / p.n_tiles) * CL + (int)cta_rank;   // may exceed m_tiles: loads zero-fill, stores clip
        const int tw = m_tile % p.tiles_w;
        const int th = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const bool masked = build_live_mask<kBN64>(p, n_tile, lane, live_prod);
        int j = 0;
        for (int t = 0; t < p.ntaps; ++t) {
          const TapInfo tap = p.taps[t];
          for (int kb = 0; kb < p.kblks; ++kb, ++j) {
            if (masked && !((live_prod[j >> 5] >> (j & 31)) & 1u)) continue;
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (elect_one()) {
              const uint32_t a_dst = smem_base + stage * kStageBytes;
              const uint32_t b_dst = a_dst + kABytes;
              mbar_arrive_expect_tx(full_bar(stage), kStageBytes);
              tma_load_4d(a_dst, &amaps.a[tap.map_id], full_bar(stage), kb * kBK, tw * p.bw + tap.dw,
                          th * p.bh + tap.dh, tn * p.bn);
              if (CL > 1) {     // my half of the weight tile, multicast to every CTA of the cluster
                tma_load_3d_mc(b_dst + cta_rank * (uint32_t)(BN / CL) * 128u, &bmap, full_bar(stage), kb * kBK,
                               n_tile * BN + (int)cta_rank * (BN / CL), tap.b_tap, kMcMask);
              } else {
                tma_load_3d(b_dst, &bmap, full_bar(stage), kb * kBK, n_tile * BN, tap.b_tap);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs the loop converged and ONE ELECTED lane issues: with an elect.sync
    // predicate the descriptors stay in uniform registers (a `lane == 0` test costs ~13 extra
    // instructions per MMA, more than a 128 x 64 x 16 MMA takes to execute).
    {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
        const int n_tile = pair % p.n_tiles;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);       // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        const bool masked = build_live_mask<kBN64>(p, n_tile, lane, live_mma);
        bool first = true;
        const int nkb = p.ntaps * p.kblks;
        for (int j = 0; j < nkb; ++j) {
          if (masked && !((live_mma[j >> 5] >> (j & 31)) & 1u)) continue;
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t da = make_smem_desc(smem_base + stage * kStageBytes, 16, 1024);
            const uint64_t db = make_smem_desc(smem_base + stage * kStageBytes + kABytes, 16, 1024);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)          // +32 bytes along K = +2 in the 16-byte address field
              umma_bf16(d_tmem, da + 2 * k, db + 2 * k, kIdesc, (first && k == 0) ? 0u : 1u);
            if (CL > 1) umma_commit_mc(empty_bar(stage), kMcMask);   // release the slot in BOTH CTAs
            else umma_commit(empty_bar(stage));          // frees the smem slot when the MMAs retire
          }
          __syncwarp();
          first = false;
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) umma_commit(tfull_bar(acc));      // accumulator complete
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int quad = warp & 3;                            // TMEM lane quadrant this warp may read
    const int row = quad * 32 + lane;                     // pixel index inside the box
    int acc = 0; uint32_t acc_phase = 0;
    uint32_t slab_ctr = 0;
    float* bn_row = p.bn_partial ? p.bn_partial + (size_t)blockIdx.x * 2 * p.N : nullptr;
    if (bn_row) {            // this CTA's row of the batch-norm partial sums starts at zero
      for (int i = (warp - 2) * 32 + lane; i < 2 * p.N; i += 128) bn_row[i] = 0.f;
      __threadfence_block();
      named_bar_sync(1, 128);
    }
    for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
      const int n_tile = pair % p.n_tiles;
      const int m_tile = (pair / p.n_tiles) * CL + (int)cta_rank;
      const int tw = m_tile % p.tiles_w;
      const int th = (m_tile / p.tiles_w) % p.tiles_h;
      const int tn = m_tile / (p.tiles_w * p.tiles_h);
      const int pw = tw * p.bw + row % p.bw;
      const int ph = th * p.bh + (row / p.bw) % p.bh;
      const int pn = tn * p.bn + row / (p.bw * p.bh);
      const bool pix_ok = pw < p.GW && ph < p.GH && pn < p.NB;
      const long long o_pix = p.o_off + pn * p.o_sn + ph * p.o_sh + pw * p.o_sw;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      if (p.tma_store) {
        // ---- stage 64-channel slabs in smem (128B-swizzled rows) and TMA-store them ----
        const bool issuer = (warp == 2 && lane == 0);
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 64) {
          const int co0 = n_tile * BN + c0;
          if (co0 >= p.N) break;                                   // uniform: whole slab out of range
          const uint32_t slab = out_base + (uint32_t)(slab_ctr & 1) * kSlabBytes;
          if (issuer) tma_store_wait_read<1>();                    // the store that last used this slab is done reading
          named_bar_sync(1, 128);
          uint32_t r0[32], r1[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0), r0);
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0 + 32), r1);
          tmem_ld_wait();
          if constexpr (AFF) slab_affine(p, r0, r1, co0, o_pix, pix_ok);
          const uint32_t row_addr = slab + (uint32_t)row * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            uint32_t pk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int e = 8 * j + 2 * q;
              const float a = __uint_as_float(e < 32 ? r0[e] : r1[e - 32]);
              const float b = __uint_as_float(e + 1 < 32 ? r0[e + 1] : r1[e + 1 - 32]);
              __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
              pk[q] = pix_ok ? *reinterpret_cast<uint32_t*>(&h) : 0u;   // rows outside the grid: clipped by the
            }                                                           // store, must be zero for the statistics
            const uint32_t dst = row_addr + (uint32_t)((j ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]),
                         "r"(pk[3])
                         : "memory");
          }
          fence_proxy_async_smem();
          named_bar_sync(1, 128);
          if (issuer) {
            tma_store_4d(&omap, slab, co0, tw * p.bw, th * p.bh, tn * p.bn);
            tma_store_commit();
          }
          if (bn_row) slab_bn_stats(slab, quad, lane, bn_row, co0, p.N, p.stats_dbg);   // next to the bulk store's own read
          ++slab_ctr;
        }
      } else {
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0), r);
        tmem_ld_wait();
        const int co0 = n_tile * BN + c0;
        if (pix_ok && co0 < p.N) {
          if (p.out_bf16) {
            __nv_bfloat16* dst = p.out_bf16 + o_pix + co0;
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              if (co0 + j + 8 <= p.N) {
                uint32_t pk[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float a = __uint_as_float(r[j + 2 * q]), b = __uint_as_float(r[j + 2 * q + 1]);
                  if (p.bias) { a += __ldg(p.bias + co0 + j + 2 * q); b += __ldg(p.bias + co0 + j + 2 * q + 1); }
                  if constexpr (AFF) {
                    a = elem_affine(p, a, co0 + j + 2 * q, o_pix + co0 + j + 2 * q);
                    b = elem_affine(p, b, co0 + j + 2 * q + 1, o_pix + co0 + j + 2 * q + 1);
                  }
                  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
                  pk[q] = *reinterpret_cast<uint32_t*>(&h);
                }
                *reinterpret_cast<uint4*>(dst + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
              } else {
                for (int q = 0; q < 8 && co0 + j + q < p.N; ++q) {
                  float a = __uint_as_float(r[j + q]);
                  if (p.bias) a += __ldg(p.bias + co0 + j + q);
                  if constexpr (AFF) a = elem_affine(p, a, co0 + j + q, o_pix + co0 + j + q);
                  dst[j + q] = __float2bfloat16(a);
                }
              }
            }
          }
          if (p.out_f32) {
            float* dst = p.out_f32 + o_pix + co0;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (co0 + j + 4 <= p.N) {
                float4 v = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                       __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                if (p.bias) {
                  v.x += __ldg(p.bias + co0 + j); v.y += __ldg(p.bias + co0 + j + 1);
                  v.z += __ldg(p.bias + co0 + j + 2); v.w += __ldg(p.bias + co0 + j + 3);
                }
                *reinterpret_cast<float4*>(dst + j) = v;
              } else {
                for (int q = 0; q < 4 && co0 + j + q < p.N; ++q) {
                  float a = __uint_as_float(r[j + q]);
                  if (p.bias) a += __ldg(p.bias + co0 + j + q);
                  dst[j + q] = a;
                }
              }
            }
          }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (p.tma_store && warp == 2 && lane == 0) tma_store_wait_all();   // smem must outlive the bulk stores
  }
  tc_fence_before();
  if (CL > 1) cluster_sync_all(); else __syncthreads();    // no CTA exits while a peer may still signal it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ----------------------------------------------------------------------------
// wgrad kernel: D[128 ci, BN co] += X^T[ci, 64 pix] * dY[64 pix, co]  (both MN-major)
// ----------------------------------------------------------------------------
struct WgradParams {
  int ntaps;
  TapInfo taps[kMaxTaps];
  int GW, GH, NB;                   // output pixel grid (the reduction domain)
  int bw, bh, bn;                   // pixel box of one K block (bw*bh*bn == 64)
  int tiles_w, tiles_h, tiles_n;
  int pblocks, splits, pblocks_per_split;
  int ci, co;                       // M and N extents
  int m_tiles, n_tiles;
  float* out;                       // [splits][taps][ci][co] partials (or dw itself when splits == 1)
  long long split_stride;           // elements between split slices
  int* counters;                    // split-K fix-up: arrivals per output tile (zeroed by the launcher), or null
  float* dw;                        // fix-up target [taps][ci][co]
  float beta;                       // dw <- beta * dw + sum of the partials
};

// ----------------------------------------------------------------------------
// CTA-pair version of the fprop / dgrad kernel: tcgen05.mma.cta_group::2, M = 256.
// A single SM cannot feed its tensor core from shared memory at full rate with a 128 x N x 64
// tile (per K block it writes A+B once and reads them once: ~190 B/clk against a 128 B/clk smem
// port).  With cta_group::2 the two SMs of a TPC compute ONE 256 x N tile: each holds its own
// 128 pixel rows of A and only HALF of the weight tile, so the per-SM smem traffic per FLOP drops
// by a third and the instruction count halves.  Protocol (as CUTLASS / the Blackwell guide):
//   * both CTAs' TMA loads (.cta_group::2) complete on the LEADER's full barrier
//     (count 2: leader's arrive.expect_tx for both halves + the peer's remote arrive);
//   * only the leader issues MMAs; tcgen05.commit.cta_group::2 multicasts the "slot free" and
//     "accumulator ready" arrivals to both CTAs;
//   * each CTA's epilogue drains its own 128 TMEM lanes and arrives on the leader's
//     "accumulator free" barrier (count 8).
// ----------------------------------------------------------------------------
template <int BN, int STAGES, bool AFF>
__global__ void __launch_bounds__(kThreads, 1)
k_igemm_kmajor2(const __grid_constant__ TMaps4 amaps, const __grid_constant__ CUtensorMap bmap,
                const __grid_constant__ CUtensorMap omap, const IgemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kABytes = kBM * kBK * 2;              // my 128 pixel rows: 16 KB
  constexpr uint32_t kBBytes = (BN / 2) * kBK * 2;          // my half of the weight tile
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  constexpr uint32_t kIdesc = make_idesc_bf16(2 * kBM, BN, 0, 0);
  constexpr uint32_t kSlabBytes = kBM * 64 * 2;
  constexpr uint16_t kPairMask = 0x3;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t out_base = smem_base + STAGES * kStageBytes;
  const uint32_t bar_base = out_base + 2 * kSlabBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  auto peer_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 6 + s); };   // leader: the peer's tile has landed
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  __shared__ uint32_t live_prod[kLiveWords], live_mma[kLiveWords];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) prefetch_tmap(&amaps.a[i]);
    prefetch_tmap(&bmap);
    if (p.tma_store) prefetch_tmap(&omap);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), p.pair_local ? 1 : 2); mbar_init(empty_bar(s), 1); mbar_init(peer_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2cta(tmem_slot, kTmemCols);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int m_pairs = (m_tiles + 1) / 2;
  const int total_pairs = m_pairs * p.n_tiles;
  const int cluster_id = blockIdx.x / 2, n_clusters = gridDim.x / 2;
  constexpr int kBN64 = (BN + 63) / 64;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs; converged warp, one elected lane issues) =====================
    {
      int stage = 0; uint32_t phase = 0;
      for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
        const int n_tile = pair % p.n_tiles;
        const int m_tile = (pair / p.n_tiles) * 2 + (int)cta_rank;
        const int tw = m_tile % p.tiles_w;
        const int th = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const bool masked = build_live_mask<kBN64>(p, n_tile, lane, live_prod);
        int j = 0;
        for (int t = 0; t < p.ntaps; ++t) {
          const TapInfo tap = p.taps[t];
          for (int kb = 0; kb < p.kblks; ++kb, ++j) {
            if (masked && !((live_prod[j >> 5] >> (j & 31)) & 1u)) continue;
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (elect_one()) {
              const uint32_t a_dst = smem_base + stage * kStageBytes;
              const uint32_t b_dst = a_dst + kABytes;
              if (p.pair_local) {
                // Each CTA's bytes complete on its OWN barrier; the peer's idle MMA warp forwards ONE
                // cluster-scope arrive per stage to the leader.  (With the loads of both CTAs signalling the
                // leader's barrier the peer's TMA stream only reached ~33 of the 54 B/clk a lone SM ingests.)
                mbar_arrive_expect_tx(full_bar(stage), kStageBytes);
                tma_load_4d(a_dst, &amaps.a[tap.map_id], full_bar(stage), kb * kBK, tw * p.bw + tap.dw,
                            th * p.bh + tap.dh, tn * p.bn);
                tma_load_3d(b_dst, &bmap, full_bar(stage), kb * kBK, n_tile * BN + (int)cta_rank * (BN / 2), tap.b_tap);
              } else {
                if (leader) mbar_arrive_expect_tx(full_bar(stage), 2 * kStageBytes);   // both CTAs' bytes land here
                else mbar_arrive_leader(full_bar(stage));
                tma_load_4d_2cta(a_dst, &amaps.a[tap.map_id], full_bar(stage), kb * kBK, tw * p.bw + tap.dw,
                                 th * p.bh + tap.dh, tn * p.bn);
                tma_load_3d_2cta(b_dst, &bmap, full_bar(stage), kb * kBK, n_tile * BN + (int)cta_rank * (BN / 2),
                                 tap.b_tap);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only; converged warp, one elected lane) =====================
    if (leader) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
        const int n_tile = pair % p.n_tiles;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);       // both epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        const bool masked = build_live_mask<kBN64>(p, n_tile, lane, live_mma);
        bool first = true;
        const int nkb = p.ntaps * p.kblks;
        for (int j = 0; j < nkb; ++j) {
          if (masked && !((live_mma[j >> 5] >> (j & 31)) & 1u)) continue;
          mbar_wait(full_bar(stage), phase);
          if (p.pair_local) mbar_wait_cluster(peer_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t da = make_smem_desc(smem_base + stage * kStageBytes, 16, 1024);
            const uint64_t db = make_smem_desc(smem_base + stage * kStageBytes + kABytes, 16, 1024);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              umma_bf16_2cta(d_tmem, da + 2 * k, db + 2 * k, kIdesc, (first && k == 0) ? 0u : 1u);
            umma_commit_2cta_mc(empty_bar(stage), kPairMask);     // slot free in BOTH CTAs
          }
          __syncwarp();
          first = false;
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) umma_commit_2cta_mc(tfull_bar(acc), kPairMask);   // accumulator ready in BOTH CTAs
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    else if (p.pair_local) {
      // ===== peer CTA: forward "my tile of this stage has landed" to the leader, one arrive per stage =====
      int stage = 0; uint32_t phase = 0;
      for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
        const int n_tile = pair % p.n_tiles;
        const bool masked = build_live_mask<kBN64>(p, n_tile, lane, live_mma);
        const int nkb = p.ntaps * p.kblks;
        for (int j = 0; j < nkb; ++j) {
          if (masked && !((live_mma[j >> 5] >> (j & 31)) & 1u)) continue;
          mbar_wait(full_bar(stage), phase);
          if (elect_one()) mbar_arrive_leader_release(peer_bar(stage));
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..5 of both CTAs) =====================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    uint32_t slab_ctr = 0;
    float* bn_row = p.bn_partial ? p.bn_partial + (size_t)blockIdx.x * 2 * p.N : nullptr;
    if (bn_row) {            // this CTA's row of the batch-norm partial sums starts at zero
      for (int i = (warp - 2) * 32 + lane; i < 2 * p.N; i += 128) bn_row[i] = 0.f;
      __threadfence_block();
      named_bar_sync(1, 128);
    }
    for (int pair = cluster_id; pair < total_pairs; pair += n_clusters) {
      const int n_tile = pair % p.n_tiles;
      const int m_tile = (pair / p.n_tiles) * 2 + (int)cta_rank;
      const int tw = m_tile % p.tiles_w;
      const int th = (m_tile / p.tiles_w) % p.tiles_h;
      const int tn = m_tile / (p.tiles_w * p.tiles_h);
      const int pw = tw * p.bw + row % p.bw;
      const int ph = th * p.bh + (row / p.bw) % p.bh;
      const int pn = tn * p.bn + row / (p.bw * p.bh);
      const bool pix_ok = pw < p.GW && ph < p.GH && pn < p.NB;
      const long long o_pix = p.o_off + pn * p.o_sn + ph * p.o_sh + pw * p.o_sw;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const bool issuer = (warp == 2 && lane == 0);
      if (p.tma_store) {
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 64) {
          const int co0 = n_tile * BN + c0;
          if (co0 >= p.N) break;
          const uint32_t slab = out_base + (uint32_t)(slab_ctr & 1) * kSlabBytes;
          if (issuer) tma_store_wait_read<1>();
          named_bar_sync(1, 128);
          uint32_t r0[32], r1[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0), r0);
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0 + 32), r1);
          tmem_ld_wait();
          if constexpr (AFF) slab_affine(p, r0, r1, co0, o_pix, pix_ok);
          const uint32_t row_addr = slab + (uint32_t)row * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            uint32_t pk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int e = 8 * j + 2 * q;
              const float a = __uint_as_float(e < 32 ? r0[e] : r1[e - 32]);
              const float b = __uint_as_float(e + 1 < 32 ? r0[e + 1] : r1[e + 1 - 32]);
              __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
              pk[q] = pix_ok ? *reinterpret_cast<uint32_t*>(&h) : 0u;   // rows outside the grid: clipped by the
            }                                                           // store, must be zero for the statistics
            const uint32_t dst = row_addr + (uint32_t)((j ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]),
                         "r"(pk[3])
                         : "memory");
          }
          fence_proxy_async_smem();
          named_bar_sync(1, 128);
          if (issuer) {
            tma_store_4d(&omap, slab, co0, tw * p.bw, th * p.bh, tn * p.bn);
            tma_store_commit();
          }
          if (bn_row) slab_bn_stats(slab, quad, lane, bn_row, co0, p.N, p.stats_dbg);   // next to the bulk store's own read
          ++slab_ctr;
        }
      } else {
        // direct global stores (fp32 output / bias: the dense layer); static register indexing only
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0), r);
          tmem_ld_wait();
          const int co0 = n_tile * BN + c0;
          if (pix_ok && co0 < p.N) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (co0 + j < p.N) {
                float a = __uint_as_float(r[j]);
                if (p.bias) a += __ldg(p.bias + co0 + j);
                if constexpr (AFF) a = elem_affine(p, a, co0 + j, o_pix + co0 + j);
                if (p.out_bf16) p.out_bf16[o_pix + co0 + j] = __float2bfloat16(a);
                if (p.out_f32) p.out_f32[o_pix + co0 + j] = a;
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(tempty_bar(acc));
        else mbar_arrive_leader(tempty_bar(acc));
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (p.tma_store && warp == 2 && lane == 0) tma_store_wait_all();
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, kTmemCols);
  }
}

// CL = CTAs per cluster (1 or 2).  The dY tile depends only on (pixel block, N tile), so with
// CL == 2 two work units that differ in (tap, M tile) share it: each CTA fetches half of the dY
// boxes and multicasts them to both (same protocol as k_igemm_kmajor).
template <int BN, int STAGES, int CL>
__global__ void __launch_bounds__(kThreads, 1)
k_igemm_wgrad(const __grid_constant__ TMaps4 xmaps, const __grid_constant__ CUtensorMap dymap,
              const WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr uint32_t kABytes = kBM * kBK * 2;        // two 64-channel boxes of 64 pixels: 16 KB
  constexpr uint32_t kBBytes = BN * kBK * 2;
  constexpr uint32_t kStageBytes = kABytes + kBBytes;
  constexpr uint32_t kBox = 64 * 64 * 2;             // 8 KB: 64 pixels x 64 channels
  constexpr uint32_t kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  constexpr uint32_t kIdesc = make_idesc_bf16(kBM, BN, 1, 1);
  constexpr int kBBoxes = BN / 64;
  static_assert(CL == 1 || kBBoxes % CL == 0, "multicast splits the dY boxes between the CTAs");
  constexpr uint16_t kMcMask = (uint16_t)((1u << CL) - 1u);

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  __shared__ int s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) prefetch_tmap(&xmaps.a[i]);
    prefetch_tmap(&dymap);
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), CL); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  if (CL > 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // Work units: (split, N tile, M index) with M index = tap * m_tiles + m_tile; a cluster takes
  // CL consecutive M indices of one (split, N tile).  Indices past the end are idle partners:
  // their x boxes are requested out of bounds (zero fill) and nothing is stored.
  const uint32_t cta_rank = CL > 1 ? cluster_ctarank() : 0u;
  const int mcount = p.ntaps * p.m_tiles;
  const int m_groups = (mcount + CL - 1) / CL;
  const int groups_per_split = m_groups * p.n_tiles;
  const int total_groups = groups_per_split * p.splits;
  const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;

  if (warp == 0) {
    {                                                      // converged warp, one elected lane issues
      int stage = 0; uint32_t phase = 0;
      for (int q = cluster_id; q < total_groups; q += n_clusters) {
        const int split = q / groups_per_split;
        const int r = q % groups_per_split;
        const int n_tile = r % p.n_tiles;
        const int mi = (r / p.n_tiles) * CL + (int)cta_rank;
        const bool live = mi < mcount;
        const TapInfo tap = p.taps[live ? mi / p.m_tiles : 0];
        const int c_base = live ? (mi % p.m_tiles) * kBM : (1 << 28);     // idle partner: out of bounds
        const int pb0 = split * p.pblocks_per_split;
        const int pb1 = min(pb0 + p.pblocks_per_split, p.pblocks);
        int tw = pb0 % p.tiles_w, th = (pb0 / p.tiles_w) % p.tiles_h, tn = pb0 / (p.tiles_w * p.tiles_h);
        for (int pb = pb0; pb < pb1; ++pb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          if (elect_one()) {
            const uint32_t a_dst = smem_base + stage * kStageBytes;
            const uint32_t b_dst = a_dst + kABytes;
            mbar_arrive_expect_tx(full_bar(stage), kStageBytes);
#pragma unroll
            for (int h = 0; h < kBM / 64; ++h)
              tma_load_4d(a_dst + h * kBox, &xmaps.a[tap.map_id], full_bar(stage), c_base + h * 64,
                          tw * p.bw + tap.dw, th * p.bh + tap.dh, tn * p.bn);
            if (CL > 1) {
#pragma unroll
              for (int hh = 0; hh < kBBoxes / CL; ++hh) {
                const int h = (int)cta_rank * (kBBoxes / CL) + hh;
                tma_load_4d_mc(b_dst + h * kBox, &dymap, full_bar(stage), n_tile * BN + h * 64, tw * p.bw,
                               th * p.bh, tn * p.bn, kMcMask);
              }
            } else {
#pragma unroll
              for (int h = 0; h < kBBoxes; ++h)
                tma_load_4d(b_dst + h * kBox, &dymap, full_bar(stage), n_tile * BN + h * 64, tw * p.bw,
                            th * p.bh, tn * p.bn);
            }
          }
          __syncwarp();
          if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++tn; } }   // next pixel block (no divisions)
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    {                                                      // converged warp, one elected lane issues
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int q = cluster_id; q < total_groups; q += n_clusters) {
        const int split = q / groups_per_split;
        const int pb0 = split * p.pblocks_per_split;
        const int pb1 = min(pb0 + p.pblocks_per_split, p.pblocks);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int pb = pb0; pb < pb1; ++pb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t da = make_smem_desc(smem_base + stage * kStageBytes, kBox, 1024);
            const uint64_t db = make_smem_desc(smem_base + stage * kStageBytes + kABytes, kBox, 1024);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)            // 16 pixels = 16 rows of 128 B = +128 address units
              umma_bf16(d_tmem, da + 128 * k, db + 128 * k, kIdesc, (pb == pb0 && k == 0) ? 0u : 1u);
            if (CL > 1) umma_commit_mc(empty_bar(stage), kMcMask);
            else umma_commit(empty_bar(stage));
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) umma_commit(tfull_bar(acc));
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    for (int q = cluster_id; q < total_groups; q += n_clusters) {
      const int split = q / groups_per_split;
      const int r = q % groups_per_split;
      const int n_tile = r % p.n_tiles;
      const int mi = (r / p.n_tiles) * CL + (int)cta_rank;
      const bool live = mi < mcount;
      const int tap_idx = live ? mi / p.m_tiles : 0;
      const int ci = live ? (mi % p.m_tiles) * kBM + row : p.ci;          // idle partner stores nothing
      float* dst_row = p.out + (long long)split * p.split_stride +
                       ((long long)p.taps[tap_idx].b_tap * p.ci + ci) * p.co;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r32[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0), r32);
        tmem_ld_wait();
        const int co0 = n_tile * BN + c0;
        if (ci < p.ci && co0 < p.co) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (co0 + j + 4 <= p.co) {
              *reinterpret_cast<float4*>(dst_row + co0 + j) =
                  make_float4(__uint_as_float(r32[j]), __uint_as_float(r32[j + 1]), __uint_as_float(r32[j + 2]),
                              __uint_as_float(r32[j + 3]));
            } else {
              for (int t = 0; t < 4 && co0 + j + t < p.co; ++t) dst_row[co0 + j + t] = __uint_as_float(r32[j + t]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      if (p.counters != nullptr) {
        // ---- split-K fix-up inside the kernel: the unit that arrives LAST at an output tile sums the partial
        // tiles of all splits in split order (deterministic) while they are still in L2, and writes dw.  Replaces
        // one k_splitk_reduce launch per layer.
        __threadfence();                                   // my part of this unit's partial tile is visible
        named_bar_sync(2, 128);
        if (warp == 2 && lane == 0) {
          int last = 0;
          if (live) {
            int* ctr = p.counters + (mi * p.n_tiles + n_tile);
            last = (atomicAdd(ctr, 1) == p.splits - 1) ? 1 : 0;
            if (last) *ctr = 0;                            // every split has arrived: re-arm for the next launch
          }
          s_last = last;
        }
        named_bar_sync(2, 128);
        if (s_last) {
          __threadfence();
          const int m0 = (mi % p.m_tiles) * kBM;
          const long long tap_off = (long long)p.taps[tap_idx].b_tap * p.ci;
          for (int rr = warp - 2; rr < kBM && m0 + rr < p.ci; rr += 4) {       // warp per row, lanes over columns
            const long long row_off = (tap_off + m0 + rr) * p.co;
            for (int c = 4 * lane; c < BN; c += 128) {
              const int co = n_tile * BN + c;
              if (co >= p.co) break;
              float4 a = p.beta != 0.f ? *reinterpret_cast<const float4*>(p.dw + row_off + co)
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
              for (int sp = 0; sp < p.splits; ++sp) {
                const float4 v = __ldcg(reinterpret_cast<const float4*>(p.out + (long long)sp * p.split_stride + row_off + co));
                a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
              }
              *reinterpret_cast<float4*>(p.dw + row_off + co) = a;
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  if (CL > 1) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// dw = beta * dw + sum_s partial[s]   (fixed summation order => deterministic)
__global__ void k_splitk_reduce(const float* __restrict__ part, long long split_stride, int splits,
                                float* __restrict__ dw, long long n, float beta) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (i + 3 < n) {
    float4 acc = beta != 0.f ? *reinterpret_cast<const float4*>(dw + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < splits; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(part + (long long)s * split_stride + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(dw + i) = acc;
  } else {
    for (long long j = i; j < n; ++j) {
      float a = beta != 0.f ? dw[j] : 0.f;
      for (int s = 0; s < splits; ++s) a += part[(long long)s * split_stride + j];
      dw[j] = a;
    }
  }
}

// ----------------------------------------------------------------------------
// Host side
// ----------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn g_encode = nullptr;
static bool g_tma_store = true;     // RIGL_TMA_STORE=0 falls back to per-thread global stores
static bool g_cta_pair = true;      // RIGL_CTA_PAIR=0: single-CTA MMA (M = 128) everywhere
static bool g_pair_local = false;   // RIGL_PAIR_LOCALBAR=1: per-CTA full barriers + a forwarded arrive (measured 2.5x SLOWER than signalling the leader directly; kept as a documented negative result)
// RIGL_WGRAD_FIXUP=1: the last-arriving CTA of an output tile sums the split-K partials inside the wgrad kernel
// instead of a separate k_splitk_reduce launch.  MEASURED SLOWER on ResNet-50 b256 (wgrad 4.3 -> 10.7 ms per step):
// the layers with few output tiles run 100-300 splits, and one CTA then sums 20 MB that the separate kernel
// spreads over the whole grid.  Kept opt-in as a documented negative result.
static bool g_wgrad_fixup = false;
static bool g_bn_stats_always = false;   // RIGL_BN_STATS_ALWAYS=1: epilogue statistics for every supported shape (tests)
static bool g_affine_always = false;     // RIGL_AFFINE_ALWAYS=1: inference epilogue for every supported shape (measurement)
static bool g_halo = true;          // RIGL_HALO3X3=0: 3x3/s1 layers with <= 64 channels use the generic kernels
static int g_halo_t = 0, g_halo_nbuf = 0;   // RIGL_HALO_CFG=T,NBUF: tuning override for the halo kernels
static bool g_cluster_mc = false;   // RIGL_CLUSTER_MC=1 enables the 2-CTA multicast clusters (measured neutral
                                    // on ResNet-50 b256: the main loops are not L2-bandwidth bound)
static int g_num_sms = 0;
static std::once_flag g_once;
static int g_init_status = RIGL_OK;

static void init_driver() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled not available from the driver (%s)", cudaGetErrorString(e));
    g_init_status = RIGL_ERR_DRIVER;
    return;
  }
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  if (const char* e = getenv("RIGL_TMA_STORE")) g_tma_store = !(e[0] == '0');
  if (const char* e = getenv("RIGL_CLUSTER_MC")) g_cluster_mc = (e[0] == '1');
  if (const char* e = getenv("RIGL_CTA_PAIR")) g_cta_pair = !(e[0] == '0');
  if (const char* e = getenv("RIGL_HALO3X3")) g_halo = !(e[0] == '0');
  if (const char* e = getenv("RIGL_BN_STATS_ALWAYS")) g_bn_stats_always = (e[0] == '1');
  if (const char* e = getenv("RIGL_AFFINE_ALWAYS")) g_affine_always = (e[0] == '1');
  if (const char* e = getenv("RIGL_WGRAD_FIXUP")) g_wgrad_fixup = (e[0] == '1');
  if (const char* e = getenv("RIGL_PAIR_LOCALBAR")) g_pair_local = (e[0] == '1');
  if (const char* e = getenv("RIGL_HALO_CFG")) sscanf(e, "%d,%d", &g_halo_t, &g_halo_nbuf);
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  if (g_num_sms <= 0) g_num_sms = 148;
}

static int ensure_driver() {
  // The driver entry point needs a CUDA context current on THIS thread (autograd runs
  // backward on worker threads that may not have touched the runtime yet).
  static thread_local bool ctx_ready = false;
  if (!ctx_ready) {
    cudaFree(0);
    ctx_ready = true;
  }
  std::call_once(g_once, init_driver);
  return g_init_status;
}

// bf16 tensor map over `rank` dims (dim 0 innermost, contiguous), 128B swizzle, zero OOB fill.
static int make_tmap_swz(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box, CUtensorMapSwizzle swz) {
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim,
                        gstr, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu,%llu,%llu,%llu] box [%u,%u,%u,%u]", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
              rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return RIGL_ERR_DRIVER;
  }
  return RIGL_OK;
}
static int make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box) {
  return make_tmap_swz(out, base, rank, dims, strides_bytes, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

// Activation view (C, W_r, H_r, N) of an NHWC tensor sub-sampled by `s` at parity (rh, rw).
static int make_act_map(CUtensorMap* out, const void* base, int nb, int h, int w, int c, int pitch, int s, int rh,
                        int rw, const uint32_t box[4]) {
  const uint64_t hr = (h - rh + s - 1) / s, wr = (w - rw + s - 1) / s;
  const uint64_t dims[4] = {(uint64_t)c, wr, hr, (uint64_t)nb};
  const uint64_t strides[3] = {(uint64_t)s * pitch * 2, (uint64_t)s * w * pitch * 2, (uint64_t)h * w * pitch * 2};
  const uint8_t* p = static_cast<const uint8_t*>(base) + ((size_t)rh * w + rw) * pitch * 2;
  return make_tmap(out, p, 4, dims, strides, box);
}

// Smallest-waste factorisation bw*bh*bn == total (powers of two) for a GW x GH x NB pixel grid.
static void choose_box(int gw, int gh, int nb, int total, int* bw, int* bh, int* bn) {
  long long best = -1;
  for (int w = 1; w <= total; w *= 2)
    for (int h = 1; w * h <= total; h *= 2) {
      const int n = total / (w * h);
      const long long padded = (long long)((gw + w - 1) / w * w) * ((gh + h - 1) / h * h) * ((nb + n - 1) / n * n);
      // prefer less padding; then longer contiguous runs (larger w, then larger h)
      const long long score = padded * 1024 - w * 16 - h;
      if (best < 0 || score < best) { best = score; *bw = w; *bh = h; *bn = n; }
    }
}

static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
static inline int posmod(int a, int b) { return ((a % b) + b) % b; }

int tc_max_ctas() {
  ensure_driver();
  return g_num_sms > 0 ? g_num_sms : 148;
}

bool tc_supported(const ConvGeom& g, int which) {
  if (g.x_pitch % 8 || g.cout % 8) return false;     // 16-byte row pitches for TMA
  if (which == 1 && g.cin % 8) return false;         // dgrad stores 8 channels at a time
  if (g.stride != 1 && g.stride != 2) return false;
  if (g.ksize * g.ksize > kMaxTaps) return false;
  (void)which;
  return true;
}

static size_t wgrad_ws_elems(const ConvGeom& g, int* splits_out, int* bps_out, int bw, int bh, int bn, int bn_tile) {
  const int tiles_w = (g.out_w + bw - 1) / bw, tiles_h = (g.out_h + bh - 1) / bh, tiles_n = (g.batch + bn - 1) / bn;
  const int pblocks = tiles_w * tiles_h * tiles_n;
  const int out_tiles = g.taps() * ((g.cin + kBM - 1) / kBM) * ((g.cout + bn_tile - 1) / bn_tile);
  const int sms = g_num_sms > 0 ? g_num_sms : 148;
  int splits = (2 * sms + out_tiles - 1) / out_tiles;
  if (splits > pblocks) splits = pblocks;
  if (splits < 1) splits = 1;
  const int bps = (pblocks + splits - 1) / splits;
  splits = (pblocks + bps - 1) / bps;
  if (splits_out) *splits_out = splits;
  if (bps_out) *bps_out = bps;
  return (size_t)splits * g.taps() * g.cin * g.cout;
}

static size_t wgrad_counter_bytes(const ConvGeom& g, int bn_tile) {
  const size_t tiles = (size_t)g.taps() * ((g.cin + kBM - 1) / kBM + 1) * ((g.cout + bn_tile - 1) / bn_tile);
  return (tiles * sizeof(int) + 255) / 256 * 256;
}

// Wider N tiles halve the L2->smem bytes per FLOP (the wgrad main loop is L2-bandwidth bound:
// K blocks are only 64 pixels deep).
static int wgrad_bn_tile(const ConvGeom& g) {
  if (g.cout >= 256 && g.cin >= 256) return 256;      // (measured: narrow-Cin layers prefer more, smaller units)
  return g.cout >= 128 ? 128 : 64;
}

#include "halo3x3.cuh"
#include "stem_s2d.cuh"

size_t tc_workspace_bytes(const ConvGeom& g) {
  if (!tc_supported(g, 2)) return 0;
  int bw, bh, bn;
  choose_box(g.out_w, g.out_h, g.batch, 64, &bw, &bh, &bn);
  size_t elems = wgrad_ws_elems(g, nullptr, nullptr, bw, bh, bn, wgrad_bn_tile(g));
  HaloParams hp;
  if (halo_wgrad_ok(g, &hp)) { const size_t e = halo_wgrad_ws_elems(g, hp); if (e > elems) elems = e; }
  return elems * sizeof(float) + wgrad_counter_bytes(g, wgrad_bn_tile(g)) + 256;
}

// With the 2-CTA multicast each CTA fetches half of the weight tile (B box = bn_tile/2 rows).
static bool kmajor_use_pair(const IgemmParams& p) {      // CTA-pair (cta_group::2) kernel
  return g_cta_pair && p.tiles_w * p.tiles_h * p.tiles_n >= 2;
}
static bool kmajor_use_mc(const IgemmParams& p) {
  return !kmajor_use_pair(p) && g_cluster_mc && p.tiles_w * p.tiles_h * p.tiles_n >= 2;
}
static int kmajor_b_rows(const IgemmParams& p, int bn_tile) {
  return (kmajor_use_mc(p) || kmajor_use_pair(p)) ? bn_tile / 2 : bn_tile;
}

static int kmajor_grid(const IgemmParams& p) {         // CTAs the K-major launcher will use (p.n_tiles set)
  const int cl = (kmajor_use_mc(p) || kmajor_use_pair(p)) ? 2 : 1;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int pairs = ((m_tiles + cl - 1) / cl) * p.n_tiles;
  int clusters = g_num_sms / cl;
  if (pairs < clusters) clusters = pairs;
  return clusters * cl;
}

template <int BN, int STAGES, int CL, bool AFF>
static int launch_kmajor(const TMaps4& amaps, const CUtensorMap& bmap, const CUtensorMap& omap, const IgemmParams& p,
                         cudaStream_t s) {
  constexpr size_t smem = (size_t)STAGES * (kBM * kBK * 2 + BN * kBK * 2) + 2 * (kBM * 64 * 2) + 1024 + 256;
  static bool configured = false;
  if (!configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_igemm_kmajor<BN, STAGES, CL, AFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int pairs = ((m_tiles + CL - 1) / CL) * p.n_tiles;
  int clusters = g_num_sms / CL;
  if (pairs < clusters) clusters = pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * CL));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (CL == 1) {
    k_igemm_kmajor<BN, STAGES, CL, AFF><<<cfg.gridDim, cfg.blockDim, smem, s>>>(amaps, bmap, omap, p);
  } else {
    RIGL_CUDA(cudaLaunchKernelEx(&cfg, k_igemm_kmajor<BN, STAGES, CL, AFF>, amaps, bmap, omap, p));
  }
  RIGL_LAUNCH_CHECK("k_igemm_kmajor");
  return RIGL_OK;
}

template <int BN, int STAGES, bool AFF>
static int launch_kmajor2(const TMaps4& amaps, const CUtensorMap& bmap, const CUtensorMap& omap, const IgemmParams& p,
                          cudaStream_t s) {
  constexpr size_t smem = (size_t)STAGES * (kBM * kBK * 2 + (BN / 2) * kBK * 2) + 2 * (kBM * 64 * 2) + 1024 + 512;
  static bool configured = false;
  if (!configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_igemm_kmajor2<BN, STAGES, AFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int pairs = ((m_tiles + 1) / 2) * p.n_tiles;
  int clusters = g_num_sms / 2;
  if (pairs < clusters) clusters = pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * 2));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  RIGL_CUDA(cudaLaunchKernelEx(&cfg, k_igemm_kmajor2<BN, STAGES, AFF>, amaps, bmap, omap, p));
  RIGL_LAUNCH_CHECK("k_igemm_kmajor2");
  return RIGL_OK;
}

template <bool AFF>
static int dispatch_kmajor_t(int n_out, const TMaps4& amaps, const CUtensorMap& bmap, const CUtensorMap& omap,
                             IgemmParams& p, int bn_tile, cudaStream_t s) {
  p.n_tiles = (n_out + bn_tile - 1) / bn_tile;
  if (kmajor_use_pair(p)) {               // CTA-pair MMA (M = 256); bmap was built with bn_tile/2 rows
    p.pair_local = g_pair_local ? 1 : 0;
    if (bn_tile == 64) return launch_kmajor2<64, 9, AFF>(amaps, bmap, omap, p, s);
    if (bn_tile == 128) return launch_kmajor2<128, 8, AFF>(amaps, bmap, omap, p, s);
    return launch_kmajor2<256, 6, AFF>(amaps, bmap, omap, p, s);
  }
  const bool mc = kmajor_use_mc(p);                        // multicast needs a partner M tile
  if (bn_tile == 64) return mc ? launch_kmajor<64, 8, 2, AFF>(amaps, bmap, omap, p, s) : launch_kmajor<64, 8, 1, AFF>(amaps, bmap, omap, p, s);
  if (bn_tile == 128) return mc ? launch_kmajor<128, 6, 2, AFF>(amaps, bmap, omap, p, s) : launch_kmajor<128, 6, 1, AFF>(amaps, bmap, omap, p, s);
  return mc ? launch_kmajor<256, 4, 2, AFF>(amaps, bmap, omap, p, s) : launch_kmajor<256, 4, 1, AFF>(amaps, bmap, omap, p, s);
}

// affine: the inference-epilogue kernel variant (p.ep_*), a separate instantiation of every K-major kernel.
static int dispatch_kmajor(int n_out, const TMaps4& amaps, const CUtensorMap& bmap, const CUtensorMap& omap,
                           IgemmParams& p, int bn_tile, cudaStream_t s, bool affine = false) {
  return affine ? dispatch_kmajor_t<true>(n_out, amaps, bmap, omap, p, bn_tile, s)
                : dispatch_kmajor_t<false>(n_out, amaps, bmap, omap, p, bn_tile, s);
}

static int pick_bn(int n_out, long long m_tiles) {
  // Keep at least ~1 wave of CTAs busy; otherwise prefer the widest tile (fewest A re-reads).
  if (n_out > 128 && m_tiles * ((n_out + 255) / 256) >= 148) return 256;
  if (n_out > 64) return 128;
  return 64;
}

void tc_set_bn_stats_always(bool on) { g_bn_stats_always = on; }
static int g_stats_dbg = 0;
void tc_set_bn_stats_debug(int v) { g_stats_dbg = v; }

// Measured on B200 (ResNet-50 and MobileNet-v1 at b256, profiles/r03_inference_shapes.md), fused call against the plain
// call + rigl_bn_apply: with a residual the per-thread 16-byte loads of the shortcut rows make the epilogue the
// bottleneck, 1.52-1.79x on every ResNet-50 shape that has one; without a residual the fused call takes 0.73-0.92x,
// except the short-K, wide output on a small pixel grid (7x7 512->1024, K = 512: 1.065x, runs within 1 %).
static bool affine_profitable(const ConvGeom& g, const AffineEpi& e) {
  if (e.residual != nullptr) return false;
  const int K = g.taps() * g.cin;
  return !(K <= 512 && g.cout >= 2 * K && g.out_pixels() <= 12544);
}

int tc_fprop(const ConvGeom& g, const void* x, const void* packed, void* y, float* y_f32, const float* bias,
             void* ws, size_t ws_bytes, cudaStream_t s, float* bn_partial, int* bn_rows, const AffineEpi* epi) {
  (void)ws; (void)ws_bytes;
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  const PackedLayout L = packed_layout(g.taps(), g.cin, g.cout);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  {
    HaloParams hp = {};
    if (y != nullptr && y_f32 == nullptr && bias == nullptr && halo_fprop_ok(g, &hp)) {
      if (bn_partial != nullptr) {        // the halo kernels have no statistics epilogue: the caller runs the plain
        set_error("fused BN statistics: layer runs on the halo kernels");   // call + the stats pass instead
        return RIGL_ERR_UNSUPPORTED;
      }
      if (epi != nullptr) {               // nor an inference epilogue: plain call + rigl_bn_apply
        set_error("fused inference epilogue: layer runs on the halo kernels");
        return RIGL_ERR_UNSUPPORTED;
      }
      return halo_launch_kmajor(hp, x, g.cin, g.x_pitch, pk + L.off_fprop, L.cin_pad, g.cout, y, g.cout, false, s);
    }
  }
  if (bn_partial != nullptr && !g_bn_stats_always) {
    // Measured on B200 (ResNet-50 b256, profiles/r02_bn_stats_epilogue.md): the statistics are free when the tile's
    // main loop is long enough to hide them (reduction length K = taps * cin >= 512), and cost about what the
    // separate stats pass costs -- or more -- for the short-K / wide-output layers whose epilogue is the
    // bottleneck (1x1 convs with K <= 128; K = 256 with more than 128 output channels).
    const int K = g.taps() * g.cin;
    if (!(K >= 512 || (K >= 256 && g.cout <= 128))) {
      set_error("fused BN statistics: not profitable for this shape (K = %d, cout = %d)", K, g.cout);
      return RIGL_ERR_UNSUPPORTED;
    }
  }
  if (epi != nullptr && !g_affine_always && !affine_profitable(g, *epi)) {
    set_error("fused inference epilogue: not profitable for this shape (K = %d, cout = %d, residual %d)",
              g.taps() * g.cin, g.cout, epi->residual != nullptr);
    return RIGL_ERR_UNSUPPORTED;
  }
  IgemmParams p = {};
  choose_box(g.out_w, g.out_h, g.batch, 128, &p.bw, &p.bh, &p.bn);
  p.GW = g.out_w; p.GH = g.out_h; p.NB = g.batch;
  p.tiles_w = (p.GW + p.bw - 1) / p.bw; p.tiles_h = (p.GH + p.bh - 1) / p.bh; p.tiles_n = (p.NB + p.bn - 1) / p.bn;
  p.kblks = (g.cin + kBK - 1) / kBK;
  p.N = g.cout;
  p.out_bf16 = static_cast<__nv_bfloat16*>(y); p.out_f32 = y_f32; p.bias = bias;
  if (epi != nullptr) {
    p.ep_scale = epi->scale; p.ep_shift = epi->shift; p.ep_relu = epi->relu;
    p.ep_res = static_cast<const __nv_bfloat16*>(epi->residual);
  }
  p.o_off = 0; p.o_sw = g.cout; p.o_sh = (long long)g.out_w * g.cout; p.o_sn = (long long)g.out_h * g.out_w * g.cout;
  p.nnz = reinterpret_cast<const uint32_t*>(pk + L.off_nnz);
  p.nnz_tap_stride = L.n_tiles * L.k_tiles; p.nnz_n_stride = L.k_tiles; p.nnz_k_stride = 1;
  p.bn_partial = bn_partial;            // (decides the kernel variant, hence the B box: set before the maps)
  p.stats_dbg = g_stats_dbg;
  TMaps4 amaps;
  const uint32_t abox[4] = {(uint32_t)kBK, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};
  bool made[4] = {false, false, false, false};
  p.ntaps = 0;
  for (int kh = 0; kh < g.ksize; ++kh)
    for (int kw = 0; kw < g.ksize; ++kw) {
      const int rh = posmod(kh - g.pad, g.stride), rw = posmod(kw - g.pad, g.stride);
      const int id = rh * g.stride + rw;
      if (!made[id]) {
        rc = make_act_map(&amaps.a[id], x, g.batch, g.in_h, g.in_w, g.cin, g.x_pitch, g.stride, rh, rw, abox);
        if (rc != RIGL_OK) return rc;
        made[id] = true;
      }
      TapInfo& t = p.taps[p.ntaps++];
      t.map_id = (int8_t)id; t.dh = (int8_t)floordiv(kh - g.pad, g.stride); t.dw = (int8_t)floordiv(kw - g.pad, g.stride);
      t.b_tap = kh * g.ksize + kw;
    }
  for (int i = 0; i < 4; ++i) if (!made[i]) amaps.a[i] = amaps.a[p.taps[0].map_id];
  const int bn_tile = pick_bn(g.cout, (long long)p.tiles_w * p.tiles_h * p.tiles_n);
  CUtensorMap bmap;
  const uint64_t bdims[3] = {(uint64_t)L.cin_pad, (uint64_t)g.cout, (uint64_t)g.taps()};
  const uint64_t bstr[2] = {(uint64_t)L.cin_pad * 2, (uint64_t)g.cout * L.cin_pad * 2};
  const uint32_t bbox[3] = {(uint32_t)kBK, (uint32_t)kmajor_b_rows(p, bn_tile), 1};
  rc = make_tmap(&bmap, pk + L.off_fprop, 3, bdims, bstr, bbox);
  if (rc != RIGL_OK) return rc;
  CUtensorMap omap = bmap;
  p.tma_store = (y != nullptr && y_f32 == nullptr && bias == nullptr && g_tma_store) ? 1 : 0;
  if (p.tma_store) {
    rc = make_act_map(&omap, y, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, abox);
    if (rc != RIGL_OK) return rc;
  }
  if (bn_partial) {
    if (!p.tma_store) {
      set_error("fused BN statistics need the bf16 TMA-store epilogue");
      return RIGL_ERR_UNSUPPORTED;
    }
    p.bn_partial = bn_partial;
    p.n_tiles = (g.cout + bn_tile - 1) / bn_tile;
    if (bn_rows) *bn_rows = kmajor_grid(p);
  }
  return dispatch_kmajor(g.cout, amaps, bmap, omap, p, bn_tile, s, epi != nullptr);
}

int tc_dgrad(const ConvGeom& g, const void* dy, const void* packed, void* dx, void* ws, size_t ws_bytes,
             cudaStream_t s) {
  (void)ws; (void)ws_bytes;
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  const PackedLayout L = packed_layout(g.taps(), g.cin, g.cout);
  const uint8_t* pk = static_cast<const uint8_t*>(packed);
  const int st = g.stride;
  {
    HaloParams hp = {};
    if (halo_dgrad_ok(g, &hp))
      return halo_launch_kmajor(hp, dy, g.cout, g.cout, pk + L.off_dgrad, L.cout_pad, g.cin, dx, g.x_pitch, true, s);
  }
  // classes of input pixels by parity; each class is one launch over its sub-grid
  bool need_zero = false;
  for (int ph = 0; ph < st && !need_zero; ++ph)
    for (int pw = 0; pw < st; ++pw) {
      int n = 0;
      for (int kh = 0; kh < g.ksize; ++kh)
        for (int kw = 0; kw < g.ksize; ++kw)
          if (posmod(ph + g.pad - kh, st) == 0 && posmod(pw + g.pad - kw, st) == 0) ++n;
      if (n == 0) need_zero = true;
    }
  if (need_zero) RIGL_CUDA(cudaMemsetAsync(dx, 0, (size_t)g.in_pixels() * g.x_pitch * 2, s));
  for (int ph = 0; ph < st; ++ph)
    for (int pw = 0; pw < st; ++pw) {
      IgemmParams p = {};
      p.GH = (g.in_h - ph + st - 1) / st; p.GW = (g.in_w - pw + st - 1) / st; p.NB = g.batch;
      if (p.GH <= 0 || p.GW <= 0) continue;
      p.ntaps = 0;
      for (int kh = 0; kh < g.ksize; ++kh)
        for (int kw = 0; kw < g.ksize; ++kw)
          if (posmod(ph + g.pad - kh, st) == 0 && posmod(pw + g.pad - kw, st) == 0) {
            TapInfo& t = p.taps[p.ntaps++];
            t.map_id = 0; t.dh = (int8_t)((ph + g.pad - kh) / st); t.dw = (int8_t)((pw + g.pad - kw) / st);
            t.b_tap = kh * g.ksize + kw;
          }
      if (p.ntaps == 0) continue;
      choose_box(p.GW, p.GH, p.NB, 128, &p.bw, &p.bh, &p.bn);
      p.tiles_w = (p.GW + p.bw - 1) / p.bw; p.tiles_h = (p.GH + p.bh - 1) / p.bh; p.tiles_n = (p.NB + p.bn - 1) / p.bn;
      p.kblks = (g.cout + kBK - 1) / kBK;
      p.N = g.cin;
      p.out_bf16 = static_cast<__nv_bfloat16*>(dx);
      p.o_off = ((long long)ph * g.in_w + pw) * g.x_pitch;
      p.o_sw = (long long)st * g.x_pitch; p.o_sh = (long long)st * g.in_w * g.x_pitch;
      p.o_sn = (long long)g.in_h * g.in_w * g.x_pitch;
      // survivor table indexed [tap][co/64][ci/64]: here N = ci, K = co
      p.nnz = reinterpret_cast<const uint32_t*>(pk + L.off_nnz);
      p.nnz_tap_stride = L.n_tiles * L.k_tiles; p.nnz_n_stride = 1; p.nnz_k_stride = L.k_tiles;
      TMaps4 amaps;
      const uint32_t abox[4] = {(uint32_t)kBK, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};
      rc = make_act_map(&amaps.a[0], dy, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, abox);
      if (rc != RIGL_OK) return rc;
      for (int i = 1; i < 4; ++i) amaps.a[i] = amaps.a[0];
      const int bn_tile = pick_bn(g.cin, (long long)p.tiles_w * p.tiles_h * p.tiles_n);
      CUtensorMap bmap;
      const uint64_t bdims[3] = {(uint64_t)L.cout_pad, (uint64_t)g.cin, (uint64_t)g.taps()};
      const uint64_t bstr[2] = {(uint64_t)L.cout_pad * 2, (uint64_t)g.cin * L.cout_pad * 2};
      const uint32_t bbox[3] = {(uint32_t)kBK, (uint32_t)kmajor_b_rows(p, bn_tile), 1};
      rc = make_tmap(&bmap, pk + L.off_dgrad, 3, bdims, bstr, bbox);
      if (rc != RIGL_OK) return rc;
      CUtensorMap omap = bmap;
      p.tma_store = g_tma_store ? 1 : 0;
      if (p.tma_store) {                 // dx viewed through the parity sub-grid of this launch
        rc = make_act_map(&omap, dx, g.batch, g.in_h, g.in_w, g.cin, g.x_pitch, st, ph, pw, abox);
        if (rc != RIGL_OK) return rc;
      }
      rc = dispatch_kmajor(g.cin, amaps, bmap, omap, p, bn_tile, s);
      if (rc != RIGL_OK) return rc;
    }
  return RIGL_OK;
}

template <int BN, int STAGES, int CL>
static int launch_wgrad_cl(const TMaps4& xmaps, const CUtensorMap& dymap, const WgradParams& p, cudaStream_t s) {
  constexpr size_t smem = (size_t)STAGES * (kBM * kBK * 2 + BN * kBK * 2) + 1024 + 256;
  static bool configured = false;
  if (!configured) {
    RIGL_CUDA(cudaFuncSetAttribute(k_igemm_wgrad<BN, STAGES, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int mcount = p.ntaps * p.m_tiles;
  const int groups = ((mcount + CL - 1) / CL) * p.n_tiles * p.splits;
  int clusters = g_num_sms / CL;
  if (groups < clusters) clusters = groups;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * CL));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (CL == 1) {
    k_igemm_wgrad<BN, STAGES, CL><<<cfg.gridDim, cfg.blockDim, smem, s>>>(xmaps, dymap, p);
  } else {
    RIGL_CUDA(cudaLaunchKernelEx(&cfg, k_igemm_wgrad<BN, STAGES, CL>, xmaps, dymap, p));
  }
  RIGL_LAUNCH_CHECK("k_igemm_wgrad");
  return RIGL_OK;
}

template <int BN, int STAGES>
static int launch_wgrad(const TMaps4& xmaps, const CUtensorMap& dymap, const WgradParams& p, cudaStream_t s) {
  if constexpr (BN >= 128) {
    if (g_cluster_mc && p.ntaps * p.m_tiles >= 2) return launch_wgrad_cl<BN, STAGES, 2>(xmaps, dymap, p, s);
  }
  return launch_wgrad_cl<BN, STAGES, 1>(xmaps, dymap, p, s);
}

int tc_wgrad(const ConvGeom& g, const void* x, const void* dy, float* dw, float beta, void* ws, size_t ws_bytes,
             cudaStream_t s) {
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  {
    HaloParams hp = {};
    if (halo_wgrad_ok(g, &hp)) {
      const size_t need = halo_wgrad_ws_elems(g, hp) * sizeof(float);
      float* wsf = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
      if (ws == nullptr || ws_bytes < need + 256) {
        set_error("rigl_conv2d_wgrad_dense: workspace %zu < required %zu", ws_bytes, need + 256);
        return RIGL_ERR_WORKSPACE;
      }
      rc = halo_launch_wgrad(hp, g, x, dy, wsf, s);
      if (rc != RIGL_OK) return rc;
      const long long n_w9 = (long long)9 * g.cin * g.cout;
      const long long threads = (n_w9 + 3) / 4;
      k_splitk_reduce<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(wsf, n_w9, halo_wgrad_grid(hp), dw, n_w9, beta);
      RIGL_LAUNCH_CHECK("k_splitk_reduce");
      return RIGL_OK;
    }
  }
  WgradParams p = {};
  choose_box(g.out_w, g.out_h, g.batch, 64, &p.bw, &p.bh, &p.bn);
  p.GW = g.out_w; p.GH = g.out_h; p.NB = g.batch;
  p.tiles_w = (p.GW + p.bw - 1) / p.bw; p.tiles_h = (p.GH + p.bh - 1) / p.bh; p.tiles_n = (p.NB + p.bn - 1) / p.bn;
  p.pblocks = p.tiles_w * p.tiles_h * p.tiles_n;
  const int bn_tile = wgrad_bn_tile(g);
  const size_t elems = wgrad_ws_elems(g, &p.splits, &p.pblocks_per_split, p.bw, p.bh, p.bn, bn_tile);
  p.ci = g.cin; p.co = g.cout;
  p.m_tiles = (g.cin + kBM - 1) / kBM; p.n_tiles = (g.cout + bn_tile - 1) / bn_tile;
  const long long n_w = (long long)g.taps() * g.cin * g.cout;
  const bool direct = (p.splits == 1 && beta == 0.f);
  if (!direct) {
    const size_t need = elems * sizeof(float);
    const size_t ctr_bytes = wgrad_counter_bytes(g, bn_tile);
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    if (ws == nullptr || ws_bytes < need + ctr_bytes + 256) {
      set_error("rigl_conv2d_wgrad_dense: workspace %zu < required %zu", ws_bytes, need + ctr_bytes + 256);
      return RIGL_ERR_WORKSPACE;
    }
    p.out = reinterpret_cast<float*>(base + ctr_bytes); p.split_stride = n_w;
    if (g_wgrad_fixup) {
      p.counters = reinterpret_cast<int*>(base); p.dw = dw; p.beta = beta;
      RIGL_CUDA(cudaMemsetAsync(p.counters, 0, ctr_bytes, s));     // (the kernel re-arms them, but the scratch is the caller's)
    }
  } else {
    p.out = dw; p.split_stride = 0;
  }
  TMaps4 xmaps;
  const uint32_t box[4] = {64, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};
  bool made[4] = {false, false, false, false};
  p.ntaps = 0;
  for (int kh = 0; kh < g.ksize; ++kh)
    for (int kw = 0; kw < g.ksize; ++kw) {
      const int rh = posmod(kh - g.pad, g.stride), rw = posmod(kw - g.pad, g.stride);
      const int id = rh * g.stride + rw;
      if (!made[id]) {
        rc = make_act_map(&xmaps.a[id], x, g.batch, g.in_h, g.in_w, g.cin, g.x_pitch, g.stride, rh, rw, box);
        if (rc != RIGL_OK) return rc;
        made[id] = true;
      }
      TapInfo& t = p.taps[p.ntaps++];
      t.map_id = (int8_t)id; t.dh = (int8_t)floordiv(kh - g.pad, g.stride); t.dw = (int8_t)floordiv(kw - g.pad, g.stride);
      t.b_tap = kh * g.ksize + kw;
    }
  for (int i = 0; i < 4; ++i) if (!made[i]) xmaps.a[i] = xmaps.a[p.taps[0].map_id];
  CUtensorMap dymap;
  rc = make_act_map(&dymap, dy, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, box);
  if (rc != RIGL_OK) return rc;
  rc = (bn_tile == 256)   ? launch_wgrad<256, 4>(xmaps, dymap, p, s)
       : (bn_tile == 128) ? launch_wgrad<128, 6>(xmaps, dymap, p, s)
                          : launch_wgrad<64, 8>(xmaps, dymap, p, s);
  if (rc != RIGL_OK) return rc;
  if (!direct && p.counters == nullptr) {
    const long long threads = (n_w + 3) / 4;
    k_splitk_reduce<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(p.out, p.split_stride, p.splits, dw, n_w, beta);
    RIGL_LAUNCH_CHECK("k_splitk_reduce");
  }
  return RIGL_OK;
}

// ----------------------------------------------------------------------------
// Small-Cin convs (the 7x7x3 stem) without a patch matrix.
// The input is copied once into a zero-bordered, 8-channel-padded buffer xp[N,Hp,Wp,8]; for
// filter row kh the K slice (kw, c) of an output pixel is then 64 CONTIGUOUS bf16 (8 pixels x
// 8 channels) starting at pixel (s*wo, s*ho + kh): a tensor map whose W dimension has a
// stride of s pixels (32 bytes for s = 2: overlapping windows) presents exactly that to TMA,
// so the conv runs on the same k_igemm_kmajor / k_igemm_wgrad kernels with k "taps" of K = 64
// and weights packed as [kh][co][kw*8 + c].  No im2col buffer, 216 MB instead of 1 GB of traffic.
// ----------------------------------------------------------------------------
struct SmallCGeom {
  int hp, wp;        // padded input extents
};

static SmallCGeom smallc_geom(const ConvGeom& g) {
  SmallCGeom q;
  q.hp = (g.out_h - 1) * g.stride + g.ksize;
  q.wp = (g.out_w - 1) * g.stride + 8;
  return q;
}

__global__ void k_smallc_pad(ConvGeom g, int hp, int wp, const __nv_bfloat16* __restrict__ x,
                             __nv_bfloat16* __restrict__ xp) {
  const long long total = (long long)g.batch * hp * wp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(i % wp), h = (int)((i / wp) % hp), n = (int)(i / ((long long)wp * hp));
    const int hi = h - g.pad, wi = w - g.pad;
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = __float2bfloat16(0.f);
    if (hi >= 0 && hi < g.in_h && wi >= 0 && wi < g.in_w) {
      const __nv_bfloat16* src = x + (((long long)n * g.in_h + hi) * g.in_w + wi) * g.x_pitch;
      for (int c = 0; c < g.cin; ++c) v[c] = src[c];
    }
    reinterpret_cast<uint4*>(xp)[i] = *reinterpret_cast<const uint4*>(v);
  }
}

// packed[kh][co][kw*8 + c] = mask ? w[kh,kw,c,co] : 0   (zero for c >= cin, kw >= k)
__global__ void k_smallc_pack(ConvGeom g, const float* __restrict__ w, const uint32_t* __restrict__ bits,
                              __nv_bfloat16* __restrict__ out) {
  const int total = g.ksize * g.cout * 64;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int kk = i % 64, co = (i / 64) % g.cout, kh = i / (64 * g.cout);
  const int kw = kk >> 3, c = kk & 7;
  float v = 0.f;
  if (kw < g.ksize && c < g.cin) {
    const long long e = (((long long)kh * g.ksize + kw) * g.cin + c) * g.cout + co;
    if ((bits[e >> 5] >> (e & 31)) & 1u) v = w[e];
  }
  out[i] = __float2bfloat16(v);
}

// dw_hwio[kh,kw,c,co] = beta*dw + sum_s part[s][kh][kw*8+c][co]
__global__ void k_smallc_unpack(ConvGeom g, const float* __restrict__ part, long long split_stride, int splits,
                                float* __restrict__ dw, float beta) {
  const long long total = (long long)g.ksize * g.ksize * g.cin * g.cout;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int co = (int)(e % g.cout), c = (int)((e / g.cout) % g.cin);
  const int kw = (int)((e / ((long long)g.cout * g.cin)) % g.ksize), kh = (int)(e / ((long long)g.cout * g.cin * g.ksize));
  const long long src = ((long long)kh * 64 + kw * 8 + c) * g.cout + co;
  float a = beta != 0.f ? dw[e] : 0.f;
  for (int s = 0; s < splits; ++s) a += part[(long long)s * split_stride + src];
  dw[e] = a;
}

bool smallc_supported(const ConvGeom& g) {
  return g.cin <= 8 && g.ksize <= 8 && g.ksize >= 2 && g.cout % 8 == 0 && (g.stride == 1 || g.stride == 2);
}

size_t smallc_padded_bytes(const ConvGeom& g) {
  const SmallCGeom q = smallc_geom(g);
  return (size_t)g.batch * q.hp * q.wp * 16;
}

size_t smallc_packed_bytes(const ConvGeom& g) { return (size_t)g.ksize * g.cout * 64 * 2; }

int smallc_pad_input(const ConvGeom& g, const void* x, void* xp, cudaStream_t s) {
  const SmallCGeom q = smallc_geom(g);
  k_smallc_pad<<<148 * 16, 256, 0, s>>>(g, q.hp, q.wp, (const __nv_bfloat16*)x, (__nv_bfloat16*)xp);
  RIGL_LAUNCH_CHECK("k_smallc_pad");
  return RIGL_OK;
}

int smallc_pack(const ConvGeom& g, const float* w, const uint32_t* bits, void* packed, cudaStream_t s) {
  const int total = g.ksize * g.cout * 64;
  k_smallc_pack<<<(total + 255) / 256, 256, 0, s>>>(g, w, bits, (__nv_bfloat16*)packed);
  RIGL_LAUNCH_CHECK("k_smallc_pack");
  return RIGL_OK;
}

// Window view of xp for filter rows kh == parity (mod stride): dims (64, out_w, rows, N).
static int make_window_map(CUtensorMap* out, const void* xp, const ConvGeom& g, const SmallCGeom& q, int parity,
                           const uint32_t box[4]) {
  const uint64_t rows = (q.hp - parity + g.stride - 1) / g.stride;
  const uint64_t dims[4] = {64, (uint64_t)g.out_w, rows, (uint64_t)g.batch};
  const uint64_t strides[3] = {(uint64_t)g.stride * 16, (uint64_t)g.stride * q.wp * 16, (uint64_t)q.hp * q.wp * 16};
  const uint8_t* base = static_cast<const uint8_t*>(xp) + (size_t)parity * q.wp * 16;
  return make_tmap(out, base, 4, dims, strides, box);
}

int smallc_fprop(const ConvGeom& g, const void* xp, const void* packed, void* y, cudaStream_t s) {
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  const SmallCGeom q = smallc_geom(g);
  IgemmParams p = {};
  choose_box(g.out_w, g.out_h, g.batch, 128, &p.bw, &p.bh, &p.bn);
  p.GW = g.out_w; p.GH = g.out_h; p.NB = g.batch;
  p.tiles_w = (p.GW + p.bw - 1) / p.bw; p.tiles_h = (p.GH + p.bh - 1) / p.bh; p.tiles_n = (p.NB + p.bn - 1) / p.bn;
  p.kblks = 1;
  p.N = g.cout;
  p.out_bf16 = static_cast<__nv_bfloat16*>(y);
  p.o_off = 0; p.o_sw = g.cout; p.o_sh = (long long)g.out_w * g.cout; p.o_sn = (long long)g.out_h * g.out_w * g.cout;
  p.nnz = nullptr;
  TMaps4 amaps;
  const uint32_t abox[4] = {64, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};
  for (int par = 0; par < g.stride; ++par) {
    rc = make_window_map(&amaps.a[par], xp, g, q, par, abox);
    if (rc != RIGL_OK) return rc;
  }
  for (int i = g.stride; i < 4; ++i) amaps.a[i] = amaps.a[0];
  p.ntaps = g.ksize;
  for (int kh = 0; kh < g.ksize; ++kh) {
    TapInfo& t = p.taps[kh];
    t.map_id = (int8_t)(kh % g.stride); t.dh = (int8_t)(kh / g.stride); t.dw = 0; t.b_tap = kh;
  }
  const int bn_tile = pick_bn(g.cout, (long long)p.tiles_w * p.tiles_h * p.tiles_n);
  CUtensorMap bmap;
  const uint64_t bdims[3] = {64, (uint64_t)g.cout, (uint64_t)g.ksize};
  const uint64_t bstr[2] = {128, (uint64_t)g.cout * 128};
  const uint32_t bbox[3] = {64, (uint32_t)kmajor_b_rows(p, bn_tile), 1};
  rc = make_tmap(&bmap, packed, 3, bdims, bstr, bbox);
  if (rc != RIGL_OK) return rc;
  CUtensorMap omap = bmap;
  p.tma_store = g_tma_store ? 1 : 0;
  if (p.tma_store) {
    rc = make_act_map(&omap, y, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, abox);
    if (rc != RIGL_OK) return rc;
  }
  return dispatch_kmajor(g.cout, amaps, bmap, omap, p, bn_tile, s);
}

static ConvGeom smallc_as_gemm(const ConvGeom& g) {     // the wgrad work decomposition sees k taps of 64 "channels"
  ConvGeom v = g;
  v.ksize = 1; v.cin = 64;
  return v;
}

size_t smallc_wgrad_ws_bytes(const ConvGeom& g) {
  int bw, bh, bn;
  choose_box(g.out_w, g.out_h, g.batch, 64, &bw, &bh, &bn);
  ConvGeom v = smallc_as_gemm(g);
  return wgrad_ws_elems(v, nullptr, nullptr, bw, bh, bn, wgrad_bn_tile(g)) * g.ksize * sizeof(float) + 256;
}

int smallc_wgrad(const ConvGeom& g, const void* xp, const void* dy, float* dw, float beta, void* ws, size_t ws_bytes,
                 cudaStream_t s) {
  int rc = ensure_driver();
  if (rc != RIGL_OK) return rc;
  const SmallCGeom q = smallc_geom(g);
  WgradParams p = {};
  choose_box(g.out_w, g.out_h, g.batch, 64, &p.bw, &p.bh, &p.bn);
  p.GW = g.out_w; p.GH = g.out_h; p.NB = g.batch;
  p.tiles_w = (p.GW + p.bw - 1) / p.bw; p.tiles_h = (p.GH + p.bh - 1) / p.bh; p.tiles_n = (p.NB + p.bn - 1) / p.bn;
  p.pblocks = p.tiles_w * p.tiles_h * p.tiles_n;
  const int bn_tile = wgrad_bn_tile(g);
  const int out_tiles = g.ksize * ((g.cout + bn_tile - 1) / bn_tile);
  int splits = (2 * g_num_sms + out_tiles - 1) / out_tiles;
  if (splits > p.pblocks) splits = p.pblocks;
  if (splits < 1) splits = 1;
  p.pblocks_per_split = (p.pblocks + splits - 1) / splits;
  p.splits = (p.pblocks + p.pblocks_per_split - 1) / p.pblocks_per_split;
  p.ci = 64; p.co = g.cout;
  p.m_tiles = 1; p.n_tiles = (g.cout + bn_tile - 1) / bn_tile;
  const long long n_part = (long long)g.ksize * 64 * g.cout;
  const size_t need = (size_t)p.splits * n_part * sizeof(float);
  if (ws == nullptr || ws_bytes < need + 256) {
    set_error("rigl_smallc_wgrad: workspace %zu < required %zu", ws_bytes, need + 256);
    return RIGL_ERR_WORKSPACE;
  }
  p.out = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  p.split_stride = n_part;
  TMaps4 xmaps;
  const uint32_t box[4] = {64, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};
  for (int par = 0; par < g.stride; ++par) {
    rc = make_window_map(&xmaps.a[par], xp, g, q, par, box);
    if (rc != RIGL_OK) return rc;
  }
  for (int i = g.stride; i < 4; ++i) xmaps.a[i] = xmaps.a[0];
  p.ntaps = g.ksize;
  for (int kh = 0; kh < g.ksize; ++kh) {
    TapInfo& t = p.taps[kh];
    t.map_id = (int8_t)(kh % g.stride); t.dh = (int8_t)(kh / g.stride); t.dw = 0; t.b_tap = kh;
  }
  CUtensorMap dymap;
  rc = make_act_map(&dymap, dy, g.batch, g.out_h, g.out_w, g.cout, g.cout, 1, 0, 0, box);
  if (rc != RIGL_OK) return rc;
  rc = (bn_tile == 256)   ? launch_wgrad<256, 4>(xmaps, dymap, p, s)
       : (bn_tile == 128) ? launch_wgrad<128, 6>(xmaps, dymap, p, s)
                          : launch_wgrad<64, 8>(xmaps, dymap, p, s);
  if (rc != RIGL_OK) return rc;
  const long long total = (long long)g.ksize * g.ksize * g.cin * g.cout;
  k_smallc_unpack<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(g, p.out, p.split_stride, p.splits, dw, beta);
  RIGL_LAUNCH_CHECK("k_smallc_unpack");
  return RIGL_OK;
}

}  // namespace rigl

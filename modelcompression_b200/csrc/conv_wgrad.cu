// conv_wgrad.cu — weight gradient of the Darknet-19 convolutions on tcgen05/TMEM, fed by TMA.
//
// Replaces the conv weight-gradient that autograd computes for MaskedConv2d.forward = F.conv2d(x, weight*mask)
// (src/pruning/weightPruning/layers.py:53-64) inside loss.backward() of the retrain step (src/train.py:229-233):
//     dW[o, c, r, s] = mask[o, c, r, s] * sum_{b,y,x} dZ[b, o, y, x] * A[b, c, y+r-1, x+s-1]
//
// Formulation.  With PNHWC activations (include/mcb200.h) both operands are 2-D matrices over the same row index p
// (pixel incl. pad rows): dZ [rows, O] and A [rows, C], and a tap is a constant row offset of A.  Per tap
//     dW_tap[o, c] = sum_p dZ[p, o] * A[p + off(tap), c]
// is a GEMM whose REDUCTION dimension is the row index, i.e. both operands are "MN-major" for the tensor core: a TMA box
// [64 rows x 64 columns] with 128-byte swizzle lands in shared memory exactly as the canonical MN-major SWIZZLE_128B
// atom (8 k-rows x 128 B, atoms 1024 B apart along k, 64-column blocks 8 KB apart), so no transpose is ever materialised.
// Pad rows of dZ are zero (the BatchNorm backward writes them so) and pad rows of A are zero, so the shifted product
// needs no bounds logic; rows before/after the buffer are TMA out-of-bounds zero fill.
//
// The reduction is very long (B*(H+1)*(W+1) rows: 2.8 M for conv2) and the output tiny for the early layers, so the row
// range is split over CTAs; each CTA writes its partial tile [tap][o][c] to the workspace with plain vector stores and
// a reduction kernel (wgrad_reduce_rows_kernel, or wgrad_reduce_small_kernel for small filter banks cut into many
// splits; plan_wgrad picks it) sums the splits, applies the mask and emits the PyTorch layout [O, C, kh, kw].
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "ptx_sm100.cuh"
#include "tmap.cuh"

namespace {

constexpr int BLOCK_M = 128;         // output channels (rows of dW) per CTA
constexpr int BLOCK_K = 64;          // pixel rows per pipeline stage
constexpr int BOX_BYTES = 64 * 128;  // one TMA box: 64 rows x 64 bf16
constexpr int BBOX_ROWS = 72;          // 3x3: activation box of a filter row = 64 k-rows + halo, serves dx = -1, 0, +1
constexpr int BBOX_BYTES = BBOX_ROWS * 128;  // 9,216 B landed by TMA
constexpr int BBOX_STRIDE = 10 * 1024;       // pitch of the 64-column blocks (1024-byte aligned for the swizzle)
constexpr int MAX_STAGES = 8;
constexpr int NUM_THREADS = 192;

struct WgradParams {
  int num_kb;       // ceil(rows / 64)
  int nsplit;       // CTAs along the reduction
  int m_tiles, n_tiles, ntaps;
  int block_n, nb64;  // N tile (multiple of 16, <= 256) and its number of 64-column boxes
  int stages, tmem_cols;
  int Wp;
  int share3;       // 3x3: one CTA = one filter row (dy), three accumulators, the activation box shared by its 3 taps
  int merge3;       // share3 with <= 64 input channels: the three dx taps are ONE instruction of N = 192 (see the issuer)
  uint32_t idesc3;  // instruction descriptor of that N = 192 instruction
  int Opad, Cpad;   // workspace tile pitch: m_tiles*128, n_tiles*block_n
  int O;            // real output channels
  uint32_t idesc;
  float* ws;        // [nsplit][ntaps][Opad][Cpad]
};

// MN-major operand tile, 128-byte swizzle: 64-element (128 B) rows of the MN dimension, 8 k-rows per 1024-byte atom
// (SBO), next 64 MN elements one whole box further (LBO).  Descriptor version 1 (Blackwell).
__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);  // start address, bits [0,14)
  d |= (uint64_t)(BOX_BYTES >> 4) << 16;        // leading byte offset: next 64-column block
  d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset: next group of 8 k-rows
  d |= (uint64_t)1 << 46;                       // version
  d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
  return d;
}

__device__ __forceinline__ int m_tile_of(int block, const WgradParams& p) { return (block / p.n_tiles) % p.m_tiles; }

__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_wgrad_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_dz, const __grid_constant__ CUtensorMap tmap_a,
                          const WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  {
    uint32_t a = ptx::smem_u32(smem);
    smem += (1024u - (a & 1023u)) & 1023u;
  }
  const uint32_t b_blk = p.share3 ? (uint32_t)BBOX_STRIDE : (uint32_t)BOX_BYTES;  // pitch of a 64-column block of B
  const uint32_t stage_bytes = 2u * BOX_BYTES + (uint32_t)p.nb64 * b_blk;
  // <= 64 output channels left in this M tile: the second 64-column dZ box would be pure zero fill, and TMA time follows
  // the box area.  It is not loaded; accumulator rows 64..127 then hold products of stale shared memory, which land in
  // workspace rows >= O that the reduction never reads.
  const bool a_half = (m_tile_of(blockIdx.x, p) * BLOCK_M + 64 >= p.O);
  const uint32_t tx_bytes = (a_half ? 1u : 2u) * BOX_BYTES +
                            (uint32_t)p.nb64 * (p.share3 ? (uint32_t)BBOX_BYTES : (uint32_t)BOX_BYTES);
  uint8_t* tiles = smem;
  uint8_t* aux = tiles + (size_t)p.stages * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tmem_full_bar = empty_bar + MAX_STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // work unit: blockIdx.x -> (split, tap, m_tile, n_tile); n fastest so neighbouring CTAs share the dZ tile in L2
  int u = blockIdx.x;
  const int n_tile = u % p.n_tiles;
  u /= p.n_tiles;
  const int m_tile = u % p.m_tiles;
  u /= p.m_tiles;
  const int ngroups = p.share3 ? 3 : p.ntaps;  // share3: a work unit is a filter ROW (3 taps)
  const int tap = u % ngroups;                 // share3: dy
  const int split = u / ngroups;
  const int kb0 = (int)(((long long)p.num_kb * split) / p.nsplit);
  const int kb1 = (int)(((long long)p.num_kb * (split + 1)) / p.nsplit);
  const int m0 = m_tile * BLOCK_M, n0 = n_tile * p.block_n;
  // 3x3: first row of the box, tap dx reads it dx rows further down; 1x1: no offset
  const int row_off = p.share3 ? (tap - 1) * p.Wp - 1 : 0;

  if (warp_idx == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_dz);
    ptx::prefetch_tensormap(&tmap_a);
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(tmem_full_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp_idx == 1) {
    ptx::tmem_alloc(tmem_ptr_smem, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp_idx == 0) {
    if (lane == 0) {  // ===================== TMA producer =====================
      int s = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        ptx::mbar_wait(&empty_bar[s], phase ^ 1u);
        uint8_t* a_dst = tiles + (size_t)s * stage_bytes;
        uint8_t* b_dst = a_dst + 2 * BOX_BYTES;
        ptx::mbar_arrive_expect_tx(&full_bar[s], tx_bytes);
        ptx::tma_load_2d(a_dst, &tmap_dz, &full_bar[s], m0, kb * BLOCK_K);
        if (!a_half) ptx::tma_load_2d(a_dst + BOX_BYTES, &tmap_dz, &full_bar[s], m0 + 64, kb * BLOCK_K);
        for (int j = 0; j < p.nb64; ++j)
          ptx::tma_load_2d(b_dst + (size_t)j * b_blk, &tmap_a, &full_bar[s], n0 + j * 64, kb * BLOCK_K + row_off);
        if (++s == p.stages) { s = 0; phase ^= 1u; }
      }
    }
  } else if (warp_idx == 1) {
    {  // ===================== MMA issuer: the whole warp walks the loop, one elected lane issues (see conv_tcgen05.cu)
      int s = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        ptx::mbar_wait(&full_bar[s], phase);
        ptx::tc_fence_after();
        const uint32_t a_addr = ptx::smem_u32(tiles + (size_t)s * stage_bytes);
        const uint64_t adesc = make_sw128_mnmajor_desc(a_addr);
        if (ptx::elect_one()) {
        if (p.merge3) {
          // <= 64 input channels: the B tile of a tap is ONE 64-column block, and tap dx is the same block one pixel row
          // (128 B) further down.  An MN-major descriptor reaches the next 64-column block through its leading byte
          // offset, so LBO = 128 B makes the three taps the three column blocks of a single N = 192 operand: 4 instead
          // of 12 instructions per 64 pixel rows (the narrow layers were bound by the COUNT of narrow MMAs).
          uint64_t bdesc = make_sw128_mnmajor_desc(a_addr + 2 * BOX_BYTES);
          bdesc = (bdesc & ~((uint64_t)0x3FFF << 16)) | ((uint64_t)(128 >> 4) << 16);
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k)
            ptx::umma_bf16_ss(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), p.idesc3,
                              (kb > kb0 || k > 0) ? 1u : 0u);
        } else if (p.share3) {
          // tap dx = rows dx .. dx+63 of the 72-row box: start dx*128 B into it (the swizzle is applied to the absolute
          // shared-memory address, so an un-aligned start needs no base offset — see conv_tcgen05.cu); 64-column blocks
          // are BBOX_STRIDE apart (LBO)
          for (int dx = 0; dx < 3; ++dx) {
            uint64_t bdesc = make_sw128_mnmajor_desc(a_addr + 2 * BOX_BYTES + (uint32_t)dx * 128u);
            bdesc = (bdesc & ~((uint64_t)0x3FFF << 16)) | ((uint64_t)(BBOX_STRIDE >> 4) << 16);
#pragma unroll
            for (int k = 0; k < BLOCK_K / 16; ++k)
              ptx::umma_bf16_ss(tmem_base + (uint32_t)(dx * p.block_n), adesc + (uint64_t)(128 * k),
                                bdesc + (uint64_t)(128 * k), p.idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
        } else {
          const uint64_t bdesc = make_sw128_mnmajor_desc(a_addr + 2 * BOX_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) {
            // 16 k-rows = two 1024-byte atoms: +2048 B = +128 in the (addr >> 4) field
            ptx::umma_bf16_ss(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), p.idesc,
                              (kb > kb0 || k > 0) ? 1u : 0u);
          }
        }
        ptx::umma_commit(&empty_bar[s]);
        if (kb == kb1 - 1) ptx::umma_commit(tmem_full_bar);
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; phase ^= 1u; }
      }
      if (kb1 <= kb0 && ptx::elect_one()) ptx::umma_commit(tmem_full_bar);  // empty split: nothing to wait for
      __syncwarp();
    }
  } else {
    // ===================== epilogue: warps 2..5 -> partial tile to the workspace =====================
    const int quarter = warp_idx & 3;
    const int o = m0 + quarter * 32 + lane;
    ptx::mbar_wait(tmem_full_bar, 0);
    ptx::tc_fence_after();
    const uint32_t taddr_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int naccs = p.share3 ? 3 : 1;
    for (int acc = 0; acc < naccs; ++acc) {
      const int tap_out = p.share3 ? tap * 3 + acc : tap;
      float* dst = p.ws + ((((size_t)split * p.ntaps + tap_out) * p.Opad + o) * p.Cpad + n0);
      for (int c0 = 0; c0 < p.block_n; c0 += 16) {
        uint32_t r[16];
        ptx::tmem_ld_32x32b_x16(taddr_row + (uint32_t)(acc * (p.merge3 ? 64 : p.block_n) + c0), r);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 v;
          v.x = __uint_as_float(r[4 * q + 0]);
          v.y = __uint_as_float(r[4 * q + 1]);
          v.z = __uint_as_float(r[4 * q + 2]);
          v.w = __uint_as_float(r[4 * q + 3]);
          *reinterpret_cast<float4*>(dst + c0 + 4 * q) = v;
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp_idx == 1) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// Large filter banks, few splits: a warp owns 32 consecutive input channels of one filter for ALL taps.  Per tap the
// lanes read one coalesced 128-byte run of every split; the taps * 32 results — which are contiguous in dW's [O, C, kh, kw]
// layout — go through shared memory so that the mask read and the dW write are coalesced runs as well (one thread per
// (o, c) writing all taps wrote 36-byte pieces 36 bytes apart and took 75 us for the 190 MB of the 1280 -> 1024 layer).
template <int TAPS>
__global__ void __launch_bounds__(256) wgrad_reduce_rows_kernel(const float* __restrict__ ws, int nsplit, int Opad, int Cpad,
                                                                int O, int C, const float* __restrict__ mask,
                                                                float* __restrict__ dw, int accumulate) {
  __shared__ float s_t[8][32 * TAPS + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cchunks = (C + 31) / 32;
  const long long items = (long long)O * cchunks;
  const long long item = (long long)blockIdx.x * 8 + warp;
  if (item >= items) return;  // (no block barrier below: warps are independent)
  const int o = (int)(item / cchunks), c0 = (int)(item % cchunks) * 32;
  const int c = c0 + lane;
  const size_t sstride = (size_t)TAPS * Opad * Cpad;
  if (c < C) {
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
      const float* src = ws + ((size_t)t * Opad + o) * Cpad + c;
      float acc = 0.f;
      for (int sp = 0; sp < nsplit; ++sp) acc += src[(size_t)sp * sstride];
      s_t[warp][lane * TAPS + t] = acc;
    }
  }
  __syncwarp();
  const int run = min(32, C - c0) * TAPS;  // contiguous outputs of this item
  const size_t d0 = ((size_t)o * C + c0) * TAPS;
#pragma unroll
  for (int k = 0; k < TAPS; ++k) {
    const int j = k * 32 + lane;
    if (j < run) {
      float v = s_t[warp][j];
      if (mask) v *= mask[d0 + j];
      dw[d0 + j] = accumulate ? dw[d0 + j] + v : v;
    }
  }
}

// Same sum for SMALL filter banks (the stem: 2 K .. 32 K (o, c) pairs summed over up to 99 splits).  One thread per
// (o, c) left 4-32 blocks walking 9 x nsplit dependent loads each (93 us for conv2's 18 K outputs); here a warp owns 32
// consecutive c of one (tap, o), G warps share the splits of that item (split s goes to group s % G, partial sums are
// combined in group order through shared memory: the result does not depend on scheduling) and a block holds 8 / G
// items, so the grid is ntaps * O * ceil(C / 32) / (8 / G) blocks.
template <int G>
__global__ void __launch_bounds__(256) wgrad_reduce_small_kernel(const float* __restrict__ ws, int nsplit, int ntaps,
                                                                 int Opad, int Cpad, int O, int C,
                                                                 const float* __restrict__ mask, float* __restrict__ dw,
                                                                 int accumulate) {
  constexpr int R = 8 / G;
  __shared__ float part[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = warp % G, r = warp / G;
  const int cchunks = (C + 31) / 32;
  const long long items = (long long)ntaps * O * cchunks;
  const long long item = (long long)blockIdx.x * R + r;
  // item -> (o, chunk, tap) with the tap fastest: the 9 taps of a weight are 36 contiguous bytes of dW
  const int t = (int)(item % ntaps);
  const long long oc = item / ntaps;
  const int cc = (int)(oc % cchunks), o = (int)(oc / cchunks);
  const int c = cc * 32 + lane;
  const bool valid = item < items && c < C;
  float acc = 0.f;
  if (valid) {
    const float* src = ws + ((size_t)t * Opad + o) * Cpad + c;
    const size_t sstride = (size_t)ntaps * Opad * Cpad;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int s = g;
    for (; s + 3 * G < nsplit; s += 4 * G) {
      a0 += src[(size_t)s * sstride];
      a1 += src[(size_t)(s + G) * sstride];
      a2 += src[(size_t)(s + 2 * G) * sstride];
      a3 += src[(size_t)(s + 3 * G) * sstride];
    }
    for (; s < nsplit; s += G) a0 += src[(size_t)s * sstride];
    acc = (a0 + a1) + (a2 + a3);
  }
  if (G > 1) {
    part[warp][lane] = acc;
    __syncthreads();
    if (g != 0) return;
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < G; ++k) acc += part[r * G + k][lane];
  }
  if (valid) {
    const size_t di = ((size_t)o * C + c) * ntaps + t;
    if (mask) acc *= mask[di];
    dw[di] = accumulate ? dw[di] + acc : acc;
  }
}

// Reduction kernel of the split partial tiles (the numbering is the one mc_conv_wgrad_plan reports).
enum WgradReduce { RED_ROWS9 = 1, RED_ROWS1 = 2, RED_SMALL1 = 3, RED_SMALL4 = 4, RED_SMALL8 = 5 };

struct WgradPlan {
  int block_n, nb64, n_tiles, m_tiles, ntaps, num_kb, nsplit, stages, tmem_cols, Opad, Cpad, share3, merge3, reduce;
  size_t smem_bytes, ws_bytes;
};

int plan_wgrad(WgradPlan* pl, int B, int H, int W, int C, int O, int ksize) {
  const long long rows = (long long)B * (H + 1) * (W + 1);
  if (rows >= (1ll << 31) - 64) return mc_set_error(MC_ERR_SHAPE, "mc_conv_wgrad: too many rows");
  pl->ntaps = ksize * ksize;
  pl->num_kb = (int)((rows + BLOCK_K - 1) / BLOCK_K);
  pl->m_tiles = (O + BLOCK_M - 1) / BLOCK_M;
  const int c16 = (C + 15) / 16 * 16;
  pl->share3 = ksize == 3 ? 1 : 0;
  const int max_n = pl->share3 ? 128 : 256;  // share3: three accumulators must fit the 512 TMEM columns
  pl->n_tiles = (c16 + max_n - 1) / max_n;
  pl->block_n = ((c16 + pl->n_tiles - 1) / pl->n_tiles + 15) / 16 * 16;
  pl->nb64 = (pl->block_n + 63) / 64;
  pl->Opad = pl->m_tiles * BLOCK_M;
  pl->Cpad = pl->n_tiles * pl->block_n;
  const int tiles = pl->m_tiles * pl->n_tiles * (pl->share3 ? 3 : pl->ntaps);
  // Split count.  The ring takes ~200 KB of shared memory, so ONE CTA is resident per SM and the grid runs in waves of
  // num_sms CTAs: "about two CTAs per SM" used to give grids like 297 or 300 (two waves plus a third one of 1-4 CTAs,
  // i.e. 1.5x the time).  Pick the split that minimises   waves * (k-blocks per CTA + fixed) + reduction traffic
  // (a k-block costs its TMA bytes at ~46 B/ns per SM — measured 0.30 us for the 17 KB stages of a 32 -> 64 layer and
  // 0.75 us for the 34 KB stages of 1024 -> 1024 —, ~3 us of set-up / partial-tile store per CTA, partial tiles written
  // and re-read at ~3 TB/s); at least 8 pipeline steps per CTA.
  const int sms = mc_num_sms();
  const int max_split = pl->num_kb / 8 > 0 ? pl->num_kb / 8 : 1;
  const double tile_bytes = 128.0 * pl->block_n * (pl->share3 ? 3 : 1) * 4.0;
  const int nb64_ = (pl->block_n + 63) / 64;
  const double kb_us = ((O <= 64 ? 1 : 2) * (double)BOX_BYTES + nb64_ * (double)(pl->share3 ? BBOX_BYTES : BOX_BYTES)) *
                       2.18e-5;
  int nsplit = 1;
  double best = 1e30;
  for (int sp = 1; sp <= max_split && (long long)sp * tiles <= 6ll * sms; ++sp) {
    const int waves = (sp * tiles + sms - 1) / sms;
    const double t = waves * ((double)pl->num_kb / sp * kb_us + 3.0) + (sp > 1 ? 2.0 * sp * tiles * tile_bytes / 3.0e6 : 0.0);
    if (t < best) { best = t; nsplit = sp; }
  }
  pl->nsplit = nsplit;
  const int stage_bytes = 2 * BOX_BYTES + pl->nb64 * (pl->share3 ? BBOX_STRIDE : BOX_BYTES);
  int stages = (200 * 1024) / stage_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  pl->stages = stages;
  pl->smem_bytes = (size_t)stages * stage_bytes + 256 + 1024;
  pl->merge3 = (pl->share3 && pl->nb64 == 1 && pl->n_tiles == 1) ? 1 : 0;
  int tc = 32;
  while (tc < (pl->merge3 ? 192 : (pl->share3 ? 3 : 1) * pl->block_n)) tc <<= 1;
  pl->tmem_cols = tc;
  pl->ws_bytes = (size_t)nsplit * pl->ntaps * pl->Opad * pl->Cpad * sizeof(float);
  // few outputs, many splits: parallel over taps and split groups; otherwise a warp per 32 channels of a filter
  if ((long long)O * C < 65536 && nsplit > 1)
    pl->reduce = nsplit >= 32 ? RED_SMALL8 : nsplit >= 8 ? RED_SMALL4 : RED_SMALL1;
  else
    pl->reduce = pl->ntaps == 9 ? RED_ROWS9 : RED_ROWS1;
  return 0;
}

}  // namespace

extern "C" size_t mc_workspace_bytes_conv_wgrad(int B, int H, int W, int C, int O, int ksize) {
  WgradPlan pl;
  if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || O <= 0 || (ksize != 1 && ksize != 3)) return 0;
  if (plan_wgrad(&pl, B, H, W, C, O, ksize)) return 0;
  return pl.ws_bytes;
}

extern "C" int mc_conv_wgrad_plan(int B, int H, int W, int C, int O, int ksize, int info[8]) {
  MC_CHECK_ARG(info != nullptr, "mc_conv_wgrad_plan: null info");
  MC_CHECK_ARG(ksize == 1 || ksize == 3, "mc_conv_wgrad_plan: ksize must be 1 or 3 (got %d)", ksize);
  MC_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && O > 0, "mc_conv_wgrad_plan: bad dims");
  WgradPlan pl;
  const int rc = plan_wgrad(&pl, B, H, W, C, O, ksize);
  if (rc) return rc;
  info[0] = pl.nsplit;
  info[1] = pl.m_tiles;
  info[2] = pl.n_tiles;
  info[3] = pl.block_n;
  info[4] = pl.share3;
  info[5] = pl.merge3;
  info[6] = pl.reduce;
  info[7] = pl.num_kb;
  return 0;
}

extern "C" int mc_conv_wgrad(const void* d_a, int lda, int C, const void* d_dz, int ld_dz, int O, int B, int H, int W,
                             int ksize, const float* d_mask, float* d_dw, int accumulate, void* d_ws, size_t ws_bytes,
                             void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_a && d_dz && d_dw && d_ws, "mc_conv_wgrad: null pointer");
  MC_CHECK_ARG(ksize == 1 || ksize == 3, "mc_conv_wgrad: ksize must be 1 or 3 (got %d)", ksize);
  MC_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && O > 0, "mc_conv_wgrad: bad dims");
  MC_CHECK_ARG((lda % 8) == 0 && C <= lda && (ld_dz % 8) == 0 && O <= ld_dz,
               "mc_conv_wgrad: pitches must be multiples of 8 covering the channels");
  MC_CHECK_ARG(((uintptr_t)d_a & 15) == 0 && ((uintptr_t)d_dz & 15) == 0 && ((uintptr_t)d_ws & 15) == 0,
               "mc_conv_wgrad: pointers must be 16-byte aligned");
  WgradPlan pl;
  int rc = plan_wgrad(&pl, B, H, W, C, O, ksize);
  if (rc) return rc;
  if (ws_bytes < pl.ws_bytes) return mc_set_error(MC_ERR_WS, "mc_conv_wgrad: workspace %zu < required %zu", ws_bytes, pl.ws_bytes);
  MC_CHECK_ARG(pl.smem_bytes <= 227 * 1024, "mc_conv_wgrad: smem %zu too large", pl.smem_bytes);
  const long long rows = (long long)B * (H + 1) * (W + 1);

  CUtensorMap tm_dz, tm_a;
  rc = mc_make_tmap_2d_bf16(&tm_dz, d_dz, (uint64_t)rows, (uint64_t)O, (uint64_t)ld_dz, BLOCK_K);
  if (rc) return rc;
  rc = mc_make_tmap_2d_bf16(&tm_a, d_a, (uint64_t)rows, (uint64_t)C, (uint64_t)lda, pl.share3 ? BBOX_ROWS : BLOCK_K);
  if (rc) return rc;

  WgradParams p;
  p.num_kb = pl.num_kb;
  p.nsplit = pl.nsplit;
  p.m_tiles = pl.m_tiles;
  p.n_tiles = pl.n_tiles;
  p.ntaps = pl.ntaps;
  p.block_n = pl.block_n;
  p.nb64 = pl.nb64;
  p.stages = pl.stages;
  p.tmem_cols = pl.tmem_cols;
  p.Wp = W + 1;
  p.share3 = pl.share3;
  p.merge3 = pl.merge3;
  p.Opad = pl.Opad;
  p.Cpad = pl.Cpad;
  p.O = O;
  // c=f32, a=b=bf16, both operands MN-major (bits 15/16), N>>3 at [17,23), M>>4 at [24,29)
  p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(pl.block_n >> 3) << 17) |
            ((uint32_t)(BLOCK_M >> 4) << 24);
  p.idesc3 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(192 >> 3) << 17) |
             ((uint32_t)(BLOCK_M >> 4) << 24);
  p.ws = reinterpret_cast<float*>(d_ws);

  static bool attr_set = false;
  if (!attr_set) {
    MC_CUDA(cudaFuncSetAttribute(conv_wgrad_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int grid = pl.m_tiles * pl.n_tiles * (pl.share3 ? 3 : pl.ntaps) * pl.nsplit;
  conv_wgrad_tcgen05_kernel<<<grid, NUM_THREADS, pl.smem_bytes, stream>>>(tm_dz, tm_a, p);
  MC_LAUNCH_CHECK("conv_wgrad_tcgen05_kernel");
  if (pl.reduce == RED_ROWS9 || pl.reduce == RED_ROWS1) {
    const long long items = (long long)O * ((C + 31) / 32);
    const unsigned g = (unsigned)((items + 7) / 8);
    if (pl.reduce == RED_ROWS9)
      wgrad_reduce_rows_kernel<9><<<g, 256, 0, stream>>>(p.ws, pl.nsplit, pl.Opad, pl.Cpad, O, C, d_mask, d_dw, accumulate);
    else
      wgrad_reduce_rows_kernel<1><<<g, 256, 0, stream>>>(p.ws, pl.nsplit, pl.Opad, pl.Cpad, O, C, d_mask, d_dw, accumulate);
    MC_LAUNCH_CHECK("wgrad_reduce_rows_kernel");
    return 0;
  }
  const long long items = (long long)pl.ntaps * O * ((C + 31) / 32);
  if (pl.reduce == RED_SMALL8) {
    wgrad_reduce_small_kernel<8><<<(unsigned)items, 256, 0, stream>>>(p.ws, pl.nsplit, pl.ntaps, pl.Opad, pl.Cpad, O, C,
                                                                      d_mask, d_dw, accumulate);
  } else if (pl.reduce == RED_SMALL4) {
    wgrad_reduce_small_kernel<4><<<(unsigned)((items + 1) / 2), 256, 0, stream>>>(p.ws, pl.nsplit, pl.ntaps, pl.Opad,
                                                                                  pl.Cpad, O, C, d_mask, d_dw, accumulate);
  } else {
    wgrad_reduce_small_kernel<1><<<(unsigned)((items + 7) / 8), 256, 0, stream>>>(p.ws, pl.nsplit, pl.ntaps, pl.Opad,
                                                                                  pl.Cpad, O, C, d_mask, d_dw, accumulate);
  }
  MC_LAUNCH_CHECK("wgrad_reduce_small_kernel");
  return 0;
}

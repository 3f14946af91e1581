// conv_window.cu — 3x3 conv (+ folded BN + leaky + optional 2x2/2 max-pool) for THIN inputs on tcgen05 with NO im2col
// build: the tensor core reads overlapping receptive-field windows straight out of a shared-memory pixel patch.
//
// Replaces the same reference call sites as conv_tcgen05.cu (MaskedConv2d.forward / BatchNorm2d / LeakyReLU / MaxPool2d,
// src/pruning/weightPruning/layers.py:53-64, src/nets.py:802,809,821) for the network's stem: the 3-channel first
// layer and the <= 8-channel layers of a filter-pruned network.
//
// Idea.  A K-major, un-swizzled UMMA operand is made of "core matrices" of 8 rows x 16 bytes; the descriptor gives the
// byte distance between 8-row groups (SBO) and between the two 16-byte K chunks of an instruction (LBO), and rows inside
// a group are 16 bytes apart.  With pixels stored 16 bytes apart in a patch [rows][pixels], GEMM row (ty, tx) of a
// 16 x 8 output tile starts at   patch + ty*SBO + tx*16   and its K chunks are 16-byte pixels of its window, reached
// through the descriptor START address (tap offset) and LBO (distance to the second tap of the instruction):
//     P8  (bf16 PNHWC input, 8-channel pixels = 16 B):  SBO = patch row pitch; 9 taps = 5 instructions (tap pairs,
//          the last one against a zero weight chunk); the patch is ONE dense 2-D TMA box (18 rows x 160 B) per tile.
//     IMG (fp32 / uint8 NCHW image, 3 channels -> 4-channel pixels = 8 B, 2x2 max-pool fused as a pool-window GEMM:
//          GEMM row = pool window, K = its 4x4x4 input patch, N = 4 window positions x filters, see
//          conv_im2col_tc.cu): a 16-byte chunk is TWO pixels, windows advance by 2 pixels = 16 B, SBO = 2 patch rows,
//          LBO = 16; 4 instructions (one per patch row of the window).  The raw image box is staged by TMA and converted
//          once per pixel to bf16 by the CTA's threads — the old kernel gathered every pixel 4 times into explicit
//          im2col rows, and ncu showed its LSU pipe as the limiter.
//          uint8 pixels enter the GEMM as the exact bf16 integers 0..255 (two integer instructions per value, no
//          rounding at all) and ToTensor's 1/255 is folded into the fp32 epilogue scale: closer to the reference's fp32
//          arithmetic than rounding x/255 to bf16 first.
// No thread touches an A operand in P8 mode; per tile the SM does one TMA box, 5 tcgen05.mma and the epilogue.
// The 2x2 max-pool of a P8 layer is taken in the epilogue across lanes: the window partners of row (ty, tx) are lanes
// +-1 (x) and +-8 (y) of the same warp.
//
// These layers are bound by instruction issue in the epilogue (ncu: 21,632 tiles of 128 pixels, a few real channels
// each), so the epilogue works on the REAL channel count in groups of 4 columns, keeps scale/shift in registers for the
// narrow cases, walks tile coordinates incrementally (every CTA owns a contiguous tile range), and stages pixels wider
// than 16 bytes through shared memory so that global stores are whole coalesced segments.
#include <cuda.h>
#include <string.h>
#include "common.cuh"
#include "ptx_sm100.cuh"
#include "tmap.cuh"

namespace {

constexpr int WTY = 16, WTX = 8;  // GEMM rows of a tile: (ty, tx), row = ty*8 + tx = TMEM lane
// CTA = FRONT warps (P8: TMA producer + MMA issuer; IMG: 4 warps that load + convert the image, warp 0 also issues the MMAs)
// + 4 epilogue warps (one per TMEM lane quarter)

struct WinParams {
  const void* in;
  const __nv_bfloat16* w;  // P8: [nb_pad][80] column tap*8+c (taps 9 = zero); IMG: [nb_pad][64] column (py*4+px)*4+c
  void* out;
  const float* scale;
  const float* shift;
  int B, H, W;        // conv resolution
  int Cin;
  int N, npos, nb;    // valid outputs; IMG: per-position column stride; UMMA N (multiple of 16)
  int ldc, leaky, pool;
  int nsc;            // entries of scale/shift that may be read
  int stage_pitch;    // > 0: bytes per staged pixel row (epilogue goes through shared memory)
  int tiles_x, tiles_y, total_tiles;
  int tmem_cols, acc_stages, acc_shift;  // accumulator stages in TMEM (power of two, 1..8) and log2 of it
  uint32_t idesc;
};

// K-major operand without swizzle: 8-row core matrices, rows 16 B apart, groups `sbo` bytes apart, the instruction's
// second K chunk `lbo` bytes after the first.
__device__ __forceinline__ uint64_t make_nosw_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell); layout type bits [61,64) = 0: no swizzle
  return d;
}

__device__ __forceinline__ void tmem_ld16f(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  ptx::tmem_ld_32x32b_x16(taddr, r);
  ptx::tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
}

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

struct TileIter {
  int b, ty, tx;
  __device__ __forceinline__ void init(unsigned int tile, unsigned int txy, int tiles_x) {
    b = (int)(tile / txy);
    const unsigned int rem = tile - (unsigned)b * txy;
    ty = (int)(rem / (unsigned)tiles_x);
    tx = (int)(rem - (unsigned)ty * (unsigned)tiles_x);
  }
  __device__ __forceinline__ void next(int tiles_x, int tiles_y) {
    if (++tx == tiles_x) {
      tx = 0;
      if (++ty == tiles_y) { ty = 0; ++b; }
    }
  }
};

// KIND: 0 = P8 (bf16 PNHWC input, pitch 8), 1 = fp32 NCHW image, 2 = uint8 NCHW image (x/255 like ToTensor)
template <int KIND>
struct WinGeom {
  static constexpr bool IMG = KIND != 0;
  static constexpr int NCHUNK = IMG ? 8 : 10;                 // 16-byte K chunks of the weight matrix
  static constexpr int NMMA = IMG ? 4 : 5;
  static constexpr int PROWS = IMG ? 2 * WTY + 2 : WTY + 2;    // patch rows
  static constexpr int PPITCH = IMG ? 208 : (WTX + 2) * 16;    // patch row pitch in bytes (IMG: 26 pixels of 8 B)
  static constexpr int PBYTES = PROWS * PPITCH;
  static constexpr int PSTRIDE = (PBYTES + 16 + 127) & ~127;   // + one chunk of slack (the zero-weight partner of tap 8)
  static constexpr int NPATCH = IMG ? 4 : 8;                   // patch ring depth
  static constexpr int NRAW = 0;                               // (no raw staging: image pixels are loaded by the threads)
  static constexpr int FRONT_WARPS = IMG ? 4 : 2;
  static constexpr int FRONT = FRONT_WARPS * 32;
  static constexpr int THREADS = FRONT + 128;
  static constexpr int REL = KIND == 2 ? 1 : 4;
  static constexpr int RSTRIDE = 0;
  static constexpr int KW = NCHUNK * 8;                        // weight matrix columns
};

// These layers are LATENCY bound (clock64 traces: per tile and CTA the epilogue chain accumulator-ready -> tcgen05.ld ->
// math -> stores -> hand-back takes ~1,900 cycles whatever the channel count), so the kernel is built for occupancy:
// 6 warps per CTA, <= 42 registers (8 CTAs = 32 epilogue warps per SM) unless the tile is WIDE (> 16 output columns).
// p is __grid_constant__ so that its fields are read from parameter space where they are used: passed by value, the
// compiler loads the whole struct into registers at entry, and the image kernels then spill under their 64-register cap.
template <int KIND, bool WIDE>
__global__ void __launch_bounds__(WinGeom<KIND>::THREADS, WIDE ? 4 : (KIND == 0 ? 6 : 4))
conv_window_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ WinParams p) {
  using G = WinGeom<KIND>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  smem += (128u - (ptx::smem_u32(smem) & 127u)) & 127u;
  const int nb_pad = p.nb;
  uint8_t* bsm = smem;                                           // [NCHUNK][nb_pad][16 B]
  uint8_t* patch0 = bsm + (((size_t)G::NCHUNK * nb_pad * 16 + 127) & ~(size_t)127);
  uint8_t* raw0 = patch0 + (size_t)G::NPATCH * G::PSTRIDE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(raw0 + (size_t)G::NRAW * G::RSTRIDE);
  uint64_t* in_full = bars;                    // [8] TMA landed (P8: the patch itself, NPATCH used; IMG: the raw box, NRAW used)
  uint64_t* patch_free = bars + 8;             // [8] tcgen05.commit: the MMAs that read patch[s] have retired (NPATCH used)
  uint64_t* tmem_full = bars + 16;             // [8] (acc_stages used)
  uint64_t* tmem_free = bars + 24;             // [8] 4 epilogue warps
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 32);
  float* s_sc = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);  // [256] scale, [256] shift
  float* s_sh = s_sc + 256;
  uint8_t* s_stage = reinterpret_cast<uint8_t*>(s_sh + 256);     // [4 lane quarters][32 pixels][stage_pitch]

  const int t = threadIdx.x;
  const int warp_idx = t >> 5;
  const int lane = t & 31;
  if (t == 0) {
    if constexpr (!G::IMG) ptx::prefetch_tensormap(&tmap_in);
    for (int i = 0; i < 8; ++i) {
      ptx::mbar_init(&in_full[i], 1);
      ptx::mbar_init(&patch_free[i], 1);
    }
    for (int i = 0; i < 8; ++i) {
      ptx::mbar_init(&tmem_full[i], 1);
      ptx::mbar_init(&tmem_free[i], 4);
    }
    ptx::fence_barrier_init();
  }
  if (warp_idx == 0) {
    ptx::tmem_alloc(tmem_ptr_smem, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  // weights -> chunk layout; patches zeroed once (slack chunks and never-written margin pixels must stay finite)
  for (int i = t; i < nb_pad * G::NCHUNK; i += G::THREADS) {
    const int n = i / G::NCHUNK, q = i - n * G::NCHUNK;
    *reinterpret_cast<uint4*>(bsm + ((size_t)q * nb_pad + n) * 16) =
        *reinterpret_cast<const uint4*>(p.w + (size_t)n * G::KW + q * 8);
  }
  for (int i = t; i < G::NPATCH * G::PSTRIDE / 16; i += G::THREADS)
    reinterpret_cast<uint4*>(patch0)[i] = make_uint4(0, 0, 0, 0);
  for (int i = t; i < 256; i += G::THREADS) {
    const bool ok = i < p.nsc;
    float sc = ok ? __ldg(p.scale + i) : 0.f;
    // uint8 image: the GEMM runs on the integers 0..255; ToTensor's 1/255 (src/nets2_utils.py:346-352) is applied here
    if constexpr (KIND == 2) sc = __fdiv_rn(sc, 255.0f);
    s_sc[i] = sc;
    s_sh[i] = ok ? __ldg(p.shift + i) : 0.f;
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t acc_stride = (uint32_t)((nb_pad + 31) & ~31);
  const unsigned int tiles_xy = (unsigned)(p.tiles_x * p.tiles_y);
  const int Hout = (G::IMG || p.pool) ? p.H / 2 : p.H, Wout = (G::IMG || p.pool) ? p.W / 2 : p.W;
  // CTA c owns the contiguous tile range [c*T/G, (c+1)*T/G): neighbouring tiles share their halo in L2, and every role
  // walks (b, ty, tx) incrementally instead of dividing per tile
  const unsigned int tile_lo = (unsigned int)(((unsigned long long)blockIdx.x * (unsigned)p.total_tiles) / gridDim.x);
  const unsigned int tile_hi = (unsigned int)(((unsigned long long)(blockIdx.x + 1) * (unsigned)p.total_tiles) / gridDim.x);

  auto issue_in = [&](const TileIter& ti, int buf) {  // P8: one dense TMA box per tile
    const int iy0 = ti.ty * WTY - 1, ix0 = ti.tx * WTX - 1;
    ptx::mbar_arrive_expect_tx(&in_full[buf], (uint32_t)G::PBYTES);
    ptx::tma_load_2d(patch0 + (size_t)buf * G::PSTRIDE, &tmap_in, &in_full[buf], ix0 * 8, ti.b * (p.H + 1) + iy0);
  };
  // Descriptors are loop invariants: one A descriptor per instruction for patch stage 0 (stage s adds s*PSTRIDE to the
  // 16-byte-unit address field) and one B descriptor per instruction.  The issuing WARP walks its loop warp-uniformly and
  // one elected lane issues: inside `if (lane == 0)` the compiler wraps every tcgen05.mma in a vote / R2UR loop and
  // re-derives 64-bit descriptors per tile, which made that single thread the slowest stage of the pipeline.
  uint64_t adesc0[G::NMMA], bdesc[G::NMMA];
  {
    const uint32_t pa = ptx::smem_u32(patch0), ba = ptx::smem_u32(bsm);
#pragma unroll
    for (int i = 0; i < G::NMMA; ++i) {
      if constexpr (G::IMG) {
        // window row i: pixels (2tx .. 2tx+3) of patch row 2ty + i; the window's first pixel is patch pixel 4 (32 B)
        adesc0[i] = make_nosw_desc(pa + (uint32_t)i * G::PPITCH + 32u, 16u, 2u * G::PPITCH);
      } else {
        const int ta = 2 * i, tb = 2 * i + 1;  // taps of this instruction (tap 9 = zero weights: any finite chunk)
        const uint32_t oa = (uint32_t)((ta / 3) * (WTX + 2) + ta % 3) * 16u;
        const uint32_t ob = tb < 9 ? (uint32_t)((tb / 3) * (WTX + 2) + tb % 3) * 16u : oa + 16u;
        adesc0[i] = make_nosw_desc(pa + oa, ob - oa, (uint32_t)G::PPITCH);
      }
      bdesc[i] = make_nosw_desc(ba + (uint32_t)(2 * i) * (uint32_t)nb_pad * 16u, (uint32_t)nb_pad * 16u, 128u);
    }
  }
  auto issue_mma = [&](int ps, uint32_t tacc) {  // called by ONE elected lane
    const uint64_t soff = (uint64_t)((uint32_t)ps * (uint32_t)(G::PSTRIDE >> 4));
#pragma unroll
    for (int i = 0; i < G::NMMA; ++i) ptx::umma_bf16_ss(tacc, adesc0[i] + soff, bdesc[i], p.idesc, i > 0 ? 1u : 0u);
  };

  if (warp_idx < G::FRONT_WARPS) {
    if constexpr (G::IMG) {
      // ============ image mode: 128 threads load + convert the tile's pixels, warp 0 issues the MMAs ============
      // A tile needs 34 image rows x 18 pixels of each channel.  Quad q = (row r, 4-pixel group k) covers the word-aligned
      // pixels x0-4+4k .. x0-1+4k (k < 6): 204 quads per tile, thread t owns quads t and t+128 for the whole launch.  The
      // pixels come straight from global memory (one 32-bit word / one float4 per channel and quad, through L1: the tiles
      // of a CTA are consecutive along x, so 7 of 8 tiles find their 128-byte lines already there) — clock64 traces showed
      // TMA boxes with 48-byte rows delivering only ~10 bytes per clock and SM.  The words of tile i+1 are requested right
      // after tile i is converted, so their latency overlaps the barrier, the MMA issue and the other CTAs of the SM.
      constexpr int NQ = G::PROWS * 6;
      constexpr int EL = G::REL;
      int qr[2], qk[2];
      bool qok[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int q = t + j * G::FRONT;
        qok[j] = q < NQ;
        qr[j] = qok[j] ? q / 6 : 0;
        qk[j] = qok[j] ? q - qr[j] * 6 : 0;
      }
      uint32_t wd[2][3];   // uint8: the quad's 4 pixels of each channel
      float4 fq[2][3];     // fp32
      const uint8_t* img = reinterpret_cast<const uint8_t*>(p.in);
      const long long plane = (long long)p.H * p.W * EL;
      auto load_tile = [&](const TileIter& ti) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int y = 2 * ti.ty * WTY - 1 + qr[j], x = 2 * ti.tx * WTX - 4 + 4 * qk[j];
          const bool ok = qok[j] && y >= 0 && y < p.H && x >= 0 && x + 4 <= p.W;
          const uint8_t* src = img + (long long)ti.b * 3 * plane + ((long long)y * p.W + x) * EL;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if constexpr (KIND == 2) wd[j][c] = ok ? __ldg(reinterpret_cast<const uint32_t*>(src + c * plane)) : 0u;
            else fq[j][c] = ok ? __ldg(reinterpret_cast<const float4*>(src + c * plane)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      };
      TileIter tin;
      tin.init(tile_lo, tiles_xy, p.tiles_x);
      if (tile_lo < tile_hi) load_tile(tin);
      int it = 0;
      for (unsigned int tile = tile_lo; tile < tile_hi; ++tile, ++it) {
        const int s = it & (G::NPATCH - 1);
        const uint32_t ph = (uint32_t)((it / G::NPATCH) & 1);
        ptx::mbar_wait(&patch_free[s], ph ^ 1u);  // MMAs of tile it-2 have read patch[s]
        uint8_t* patch = patch0 + (size_t)s * G::PSTRIDE;
        // quad k of row r -> patch pixels 4k+1 .. 4k+4 of patch row r, each pixel = (c0 c1 | c2 0) in bf16
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (!qok[j]) continue;
          uint32_t px[4][2];
          if constexpr (KIND == 2) {
#pragma unroll
            for (int sx = 0; sx < 4; ++sx) {
              // byte -> float exactly: bits(2^23 + x) = 0x4B000000 | x, minus 2^23; the upper half of the fp32 IS the
              // bf16 (x has <= 8 significant bits), so two values pack with one byte permute
              uint32_t f[3];
#pragma unroll
              for (int c = 0; c < 3; ++c)
                f[c] = __float_as_uint(__uint_as_float(__byte_perm(wd[j][c], 0x4B000000u, 0x7650u + (uint32_t)sx)) - 8388608.0f);
              px[sx][0] = __byte_perm(f[0], f[1], 0x7632u);
              px[sx][1] = f[2] >> 16;
            }
          } else {
            px[0][0] = pack2(fq[j][0].x, fq[j][1].x); px[0][1] = pack2(fq[j][2].x, 0.f);
            px[1][0] = pack2(fq[j][0].y, fq[j][1].y); px[1][1] = pack2(fq[j][2].y, 0.f);
            px[2][0] = pack2(fq[j][0].z, fq[j][1].z); px[2][1] = pack2(fq[j][2].z, 0.f);
            px[3][0] = pack2(fq[j][0].w, fq[j][1].w); px[3][1] = pack2(fq[j][2].w, 0.f);
          }
          uint8_t* dst = patch + qr[j] * G::PPITCH + (1 + 4 * qk[j]) * 8;
#pragma unroll
          for (int sx = 0; sx < 4; ++sx) *reinterpret_cast<uint2*>(dst + sx * 8) = make_uint2(px[sx][0], px[sx][1]);
        }
        if (tile + 1u < tile_hi) {  // request the next tile's pixels
          tin.next(p.tiles_x, p.tiles_y);
          load_tile(tin);
        }
        ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
        asm volatile("bar.sync 1, 128;" ::: "memory");  // patch[s] complete
        if (warp_idx == 0) {
          const int a = it & (p.acc_stages - 1);
          ptx::mbar_wait(&tmem_free[a], (uint32_t)(((it >> p.acc_shift) & 1) ^ 1));  // epilogue drained TMEM[a]
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            issue_mma(s, tmem_base + (uint32_t)a * acc_stride);
            ptx::umma_commit(&patch_free[s]);
            ptx::umma_commit(&tmem_full[a]);
          }
          __syncwarp();
        }
      }
    } else {
      // ============ P8 mode: one thread feeds TMA boxes, one thread issues the MMAs ============
      if (warp_idx == 0) {
        TileIter tin;
        tin.init(tile_lo, tiles_xy, p.tiles_x);
        int it = 0;
        for (unsigned int tile = tile_lo; tile < tile_hi; ++tile, ++it) {
          const int s = it & (G::NPATCH - 1);
          const uint32_t ph = (uint32_t)((it / G::NPATCH) & 1);
          ptx::mbar_wait(&patch_free[s], ph ^ 1u);
          if (ptx::elect_one()) issue_in(tin, s);
          __syncwarp();
          tin.next(p.tiles_x, p.tiles_y);
        }
      } else if (warp_idx == 1) {
        int it = 0;
        for (unsigned int tile = tile_lo; tile < tile_hi; ++tile, ++it) {
          const int s = it & (G::NPATCH - 1), a = it & (p.acc_stages - 1);
          ptx::mbar_wait(&in_full[s], (uint32_t)((it / G::NPATCH) & 1));
          ptx::mbar_wait(&tmem_free[a], (uint32_t)(((it >> p.acc_shift) & 1) ^ 1));
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            issue_mma(s, tmem_base + (uint32_t)a * acc_stride);
            ptx::umma_commit(&patch_free[s]);
            ptx::umma_commit(&tmem_full[a]);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ============================== epilogue warps 4..7 ==============================
    const int quarter = warp_idx & 3;       // the TMEM lane quarter a warp may access is warp_idx % 4
    const int et = quarter * 32 + lane;     // TMEM lane == GEMM row
    const int ty = et >> 3, tx = et & 7;
    const bool pool8 = !G::IMG && p.pool != 0;
    const int N = p.N, ldc = p.ldc;
    const int n4 = (N + 3) & ~3;            // real columns, in groups of 4
    const bool staged = p.stage_pitch > 0;
    uint8_t* wstage = s_stage + (size_t)quarter * 32 * p.stage_pitch;
    // pixels a warp holds after pooling: IMG / un-pooled P8: 32 (4 rows x 8); pooled P8: 8 (2 rows x 4)
    const int wpx_cols = pool8 ? 4 : 8, wpx = pool8 ? 8 : 32;
    const int my_px = pool8 ? ((ty & 3) >> 1) * 4 + (tx >> 1) : (ty & 3) * 8 + tx;   // index inside the warp's pixels
    const bool my_store = !pool8 || (((ty | tx) & 1) == 0);
    // narrow IMG layers: scale / shift of the <= 8 filters live in registers for the whole launch
    float rsc[8], rsh[8];
#pragma unroll
    for (int n = 0; n < 8; ++n) { rsc[n] = s_sc[n]; rsh[n] = s_sh[n]; }
    // staged copy-out: lane l handles chunks l, l+32, ... of the warp's [pixel][chunk] list (no division per chunk)
    const int co_cpr = ((n4 + 7) >> 3) > 0 ? ((n4 + 7) >> 3) : 1;
    const int co_px0 = lane / co_cpr, co_c0 = lane - co_px0 * co_cpr, co_dpx = 32 / co_cpr, co_dc = 32 - co_dpx * co_cpr;
    TileIter ti;
    ti.init(tile_lo, tiles_xy, p.tiles_x);
    int it = 0;
    for (unsigned int tile = tile_lo; tile < tile_hi; ++tile, ++it, ti.next(p.tiles_x, p.tiles_y)) {
      const int a = it & (p.acc_stages - 1);
      const uint32_t aph = (uint32_t)((it >> p.acc_shift) & 1);
      // output pixel of this lane, and of the warp's first pixel
      const int gy = ti.ty * WTY + ty, gx = ti.tx * WTX + tx;          // GEMM-row coordinates (conv px, or pool window)
      const int oy = pool8 ? gy >> 1 : gy, ox = pool8 ? gx >> 1 : gx;
      const bool valid = oy < Hout && ox < Wout && my_store;
      __nv_bfloat16* dst =
          reinterpret_cast<__nv_bfloat16*>(p.out) + (((long long)ti.b * (Hout + 1) + oy) * (Wout + 1) + ox) * ldc;
      ptx::mbar_wait(&tmem_full[a], aph);
      ptx::tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)a * acc_stride;

      // ---- the lane's pixel: up to N activated values, produced 16 accumulator columns at a time
      auto emit = [&](int n0, const float* v) {  // 16 values for channels [n0, n0+16): 4-column groups below n4 are real
        if (staged) {
          if (my_store) {
            uint8_t* row = wstage + (size_t)my_px * p.stage_pitch + n0 * 2;
#pragma unroll
            for (int g = 0; g < 2; ++g)
              if (n0 + g * 8 < n4)
                *reinterpret_cast<uint4*>(row + g * 16) = make_uint4(pack2(v[g * 8], v[g * 8 + 1]), pack2(v[g * 8 + 2], v[g * 8 + 3]),
                                                                     pack2(v[g * 8 + 4], v[g * 8 + 5]), pack2(v[g * 8 + 6], v[g * 8 + 7]));
          }
        } else if (valid) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            const int c0 = n0 + g * 8;
            if (c0 >= N) continue;
            if ((ldc & 7) == 0 && c0 + 8 <= ldc) {
              *reinterpret_cast<uint4*>(dst + c0) = make_uint4(pack2(v[g * 8], v[g * 8 + 1]), pack2(v[g * 8 + 2], v[g * 8 + 3]),
                                                               pack2(v[g * 8 + 4], v[g * 8 + 5]), pack2(v[g * 8 + 6], v[g * 8 + 7]));
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (c0 + j < N) dst[c0 + j] = __float2bfloat16_rn(v[g * 8 + j]);
            }
          }
        }
      };

      if constexpr (G::IMG) {
        const int np = p.npos;
        if (!WIDE && np == 4) {
          // all four window positions of the 4 filters in ONE 16-column load
          float v[16], m[16];
          tmem_ld16f(trow, v);
#pragma unroll
          for (int n = 0; n < 16; ++n) m[n] = 0.f;
#pragma unroll
          for (int n = 0; n < 4; ++n) {
            float r = fmaf(v[n], rsc[n], rsh[n]);
#pragma unroll
            for (int pos = 1; pos < 4; ++pos) r = fmaxf(r, fmaf(v[pos * 4 + n], rsc[n], rsh[n]));
            if (p.leaky) r = fmaxf(r, 0.1f * r);
            m[n] = n < N ? r : 0.f;
          }
          emit(0, m);
        } else if (!WIDE && np == 8) {
          float v0[16], v1[16], m[16];
          tmem_ld16f(trow, v0);
          tmem_ld16f(trow + 16, v1);
#pragma unroll
          for (int n = 0; n < 16; ++n) m[n] = 0.f;
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            float r = fmaf(v0[n], rsc[n], rsh[n]);
            r = fmaxf(r, fmaf(v0[8 + n], rsc[n], rsh[n]));
            r = fmaxf(r, fmaf(v1[n], rsc[n], rsh[n]));
            r = fmaxf(r, fmaf(v1[8 + n], rsc[n], rsh[n]));
            if (p.leaky) r = fmaxf(r, 0.1f * r);
            m[n] = n < N ? r : 0.f;
          }
          emit(0, m);
        } else if (WIDE) {
          for (int n0 = 0; n0 < np; n0 += 16) {
            // the four window positions of 16 filters: four loads in flight, ONE wait (a tcgen05.ld round trip is ~300
            // cycles; eight serial ones made this epilogue 2,600 cycles per tile)
            uint32_t r[4][16];
#pragma unroll
            for (int pos = 0; pos < 4; ++pos) ptx::tmem_ld_32x32b_x16(trow + (uint32_t)(pos * np + n0), r[pos]);
            ptx::tmem_ld_wait();
            float m[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 sc = *reinterpret_cast<const float4*>(s_sc + n0 + 4 * q), sh = *reinterpret_cast<const float4*>(s_sh + n0 + 4 * q);
              const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float x = fmaf(__uint_as_float(r[0][4 * q + j]), scv[j], shv[j]);
#pragma unroll
                for (int pos = 1; pos < 4; ++pos) x = fmaxf(x, fmaf(__uint_as_float(r[pos][4 * q + j]), scv[j], shv[j]));
                if (p.leaky) x = fmaxf(x, 0.1f * x);
                m[4 * q + j] = (n0 + 4 * q + j < N) ? x : 0.f;
              }
            }
            emit(n0, m);
          }
        }
      } else {
        for (int n0 = 0; n0 < n4; n0 += 16) {
          float v[16];
          tmem_ld16f(trow + n0, v);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (n0 + 4 * q < n4) {  // warp-uniform: only the column groups that hold real channels are processed
              const float4 sc = *reinterpret_cast<const float4*>(s_sc + n0 + 4 * q), sh = *reinterpret_cast<const float4*>(s_sh + n0 + 4 * q);
              v[4 * q + 0] = fmaf(v[4 * q + 0], sc.x, sh.x); v[4 * q + 1] = fmaf(v[4 * q + 1], sc.y, sh.y);
              v[4 * q + 2] = fmaf(v[4 * q + 2], sc.z, sh.z); v[4 * q + 3] = fmaf(v[4 * q + 3], sc.w, sh.w);
#pragma unroll
              for (int j = 4 * q; j < 4 * q + 4; ++j) {
                if (pool8) {
                  // 2x2 window partners: lane ^ 1 (x) and lane ^ 8 (y) of this warp (tile rows are 8 lanes apart)
                  v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 1));
                  v[j] = fmaxf(v[j], __shfl_xor_sync(0xffffffffu, v[j], 8));
                }
                if (p.leaky) v[j] = fmaxf(v[j], 0.1f * v[j]);
                if (n0 + j >= N) v[j] = 0.f;
              }
            } else {
              v[4 * q + 0] = v[4 * q + 1] = v[4 * q + 2] = v[4 * q + 3] = 0.f;
            }
          }
          emit(n0, v);
        }
      }
      // the accumulator stage is drained: hand it back before the (possibly staged) copy-out
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_free[a]);

      if (staged) {
        // the warp's pixels sit in shared memory [pixel][stage_pitch]; consecutive lanes write consecutive 16-byte
        // chunks of consecutive pixels: whole coalesced segments instead of 16-byte pieces one pixel pitch apart
        const int cpr = (n4 + 7) >> 3;  // 16-byte chunks per pixel that hold real channels
        const int wy0 = (pool8 ? (ti.ty * WTY + quarter * 4) >> 1 : ti.ty * WTY + quarter * 4);
        const int wx0 = pool8 ? (ti.tx * WTX) >> 1 : ti.tx * WTX;
        __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + (((long long)ti.b * (Hout + 1) + wy0) * (Wout + 1) + wx0) * ldc;
        const int rows_ok = Hout - wy0, cols_ok = Wout - wx0;
        int px = co_px0, c = co_c0;
        while (px < wpx) {
          const int py = pool8 ? px >> 2 : px >> 3, pxx = pool8 ? px & 3 : px & 7;
          if (py < rows_ok && pxx < cols_ok)
            *reinterpret_cast<uint4*>(obase + ((long long)py * (Wout + 1) + pxx) * ldc + c * 8) =
                *reinterpret_cast<const uint4*>(wstage + (size_t)px * p.stage_pitch + c * 16);
          px += co_dpx; c += co_dc;
          if (c >= cpr) { c -= cpr; ++px; }
        }
        __syncwarp();  // the staging rows are rewritten by the next tile
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp_idx == 0) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

template <int KIND>
size_t window_smem_bytes(int nb_pad, int stage_pitch) {
  using G = WinGeom<KIND>;
  return (((size_t)G::NCHUNK * nb_pad * 16 + 127) & ~(size_t)127) + (size_t)G::NPATCH * G::PSTRIDE +
         (size_t)G::NRAW * G::RSTRIDE + 512 + 2048 + (size_t)128 * stage_pitch + 128;
}

template <int KIND, bool WIDE>
int launch_window(const WinParams& p, cudaStream_t stream) {
  using G = WinGeom<KIND>;
  const size_t smem = window_smem_bytes<KIND>(p.nb, p.stage_pitch);
  if (smem > 200 * 1024) return mc_set_error(MC_ERR_SHAPE, "mc_conv_window_fwd: %zu B of shared memory", smem);
  CUtensorMap tm_in;
  int rc;
  if (G::IMG) {  // the image is read with plain loads: word-aligned quads need W % 4 == 0
    if (p.W % 4 != 0) return mc_set_error(MC_ERR_SHAPE, "mc_conv_window_fwd: image width must be a multiple of 4 (got %d)", p.W);
    memset(&tm_in, 0, sizeof(tm_in));
    rc = 0;
  } else {       // bf16 PNHWC pitch 8 viewed as [B*(H+1)][(W+1)*8], box [PROWS][(WTX+2)*8]
    const uint64_t dims[2] = {(uint64_t)(p.W + 1) * 8, (uint64_t)p.B * (p.H + 1)};
    const uint64_t strides[1] = {(uint64_t)(p.W + 1) * 16};
    const uint32_t box[2] = {(uint32_t)(WTX + 2) * 8, (uint32_t)G::PROWS};
    rc = mc_make_tmap(&tm_in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p.in, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
  }
  if (rc) return rc;
  auto kern = conv_window_kernel<KIND, WIDE>;
  static size_t attr_smem = 0;  // per template instantiation
  if (smem > attr_smem) {
    MC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem = smem;
  }
  int per_sm = (int)((220 * 1024) / (smem + 1024));
  const int tmem_lim = 512 / p.tmem_cols;
  if (per_sm > tmem_lim) per_sm = tmem_lim;
  const int cta_cap = WIDE ? 4 : (KIND == 0 ? 6 : 4);
  if (per_sm > cta_cap) per_sm = cta_cap;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)mc_num_sms() * per_sm;
  if (grid > p.total_tiles) grid = p.total_tiles;
  kern<<<(int)grid, G::THREADS, smem, stream>>>(tm_in, p);
  MC_LAUNCH_CHECK("conv_window_kernel");
  return 0;
}

}  // namespace

// in_kind: 0 = bf16 PNHWC with pitch 8 (Cin <= 8), 1 = fp32 NCHW image, 2 = uint8 NCHW image (Cin <= 3, pool required)
extern "C" int mc_conv_window_supported(int Cin, int in_kind, int N, int pool) {
  if (Cin < 1 || N < 1) return 0;
  if (in_kind == 0) return (Cin <= 8 && N <= 128) ? 1 : 0;
  if (in_kind != 1 && in_kind != 2) return 0;
  if (Cin > 3 || !pool) return 0;
  const int npos = (N <= 4) ? 4 : (N <= 8) ? 8 : ((N + 15) & ~15);
  return 4 * npos <= 256 ? 1 : 0;
}

extern "C" int mc_conv_window_geometry(int Cin, int in_kind, int N, int pool, int* npos, int* nb, int* kcols) {
  if (!mc_conv_window_supported(Cin, in_kind, N, pool)) return mc_set_error(MC_ERR_SHAPE, "mc_conv_window: unsupported shape");
  int np, n;
  if (in_kind == 0) {
    np = (N + 15) & ~15;
    n = np;
  } else {
    np = (N <= 4) ? 4 : (N <= 8) ? 8 : ((N + 15) & ~15);
    n = (4 * np + 15) & ~15;
  }
  if (npos) *npos = np;
  if (nb) *nb = n;
  if (kcols) *kcols = in_kind == 0 ? 80 : 64;
  return 0;
}

extern "C" int mc_conv_window_fwd(const void* d_in, int in_kind, const void* d_w, const float* d_scale,
                                  const float* d_shift, void* d_out, int B, int H, int W, int Cin, int N, int ldc,
                                  int leaky, int pool, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_in && d_w && d_scale && d_shift && d_out, "mc_conv_window_fwd: null pointer");
  MC_CHECK_ARG(B > 0 && H > 0 && W > 0, "mc_conv_window_fwd: bad dims");
  int npos, nb, kcols;
  int rc = mc_conv_window_geometry(Cin, in_kind, N, pool, &npos, &nb, &kcols);
  if (rc) return rc;
  MC_CHECK_ARG(ldc >= N, "mc_conv_window_fwd: ldc < N");
  if (pool) MC_CHECK_ARG((H % 2) == 0 && (W % 2) == 0, "mc_conv_window_fwd: pooling needs even H,W");
  MC_CHECK_ARG(((uintptr_t)d_w & 15) == 0 && ((uintptr_t)d_in & 15) == 0 && ((uintptr_t)d_out & 15) == 0,
               "mc_conv_window_fwd: pointers must be 16-byte aligned");
  WinParams p;
  p.in = d_in;
  p.w = reinterpret_cast<const __nv_bfloat16*>(d_w);
  p.out = d_out;
  p.scale = d_scale;
  p.shift = d_shift;
  p.B = B; p.H = H; p.W = W;
  p.Cin = Cin;
  p.N = N; p.npos = npos; p.nb = nb;
  p.ldc = ldc; p.leaky = leaky; p.pool = pool;
  p.nsc = in_kind == 0 ? nb : ((npos + 15) & ~15);
  // pixels wider than one 16-byte chunk go through shared memory (coalesced copy-out); the pitch needs ldc % 8 == 0
  const int n4 = (N + 3) & ~3;
  p.stage_pitch = (n4 > 8 && (ldc & 7) == 0) ? (((n4 + 7) & ~7) * 2 + 16) : 0;
  if (in_kind == 0) {
    p.tiles_x = (W + WTX - 1) / WTX;
    p.tiles_y = (H + WTY - 1) / WTY;
  } else {
    p.tiles_x = (W / 2 + WTX - 1) / WTX;
    p.tiles_y = (H / 2 + WTY - 1) / WTY;
  }
  p.total_tiles = B * p.tiles_x * p.tiles_y;
  // Accumulator stages.  The hand-offs (tcgen05.commit -> epilogue, epilogue -> MMA issuer) each take ~1,000 cycles
  // (clock64 traces), far longer than a tile's 5 MMAs, so narrow tiles keep up to 8 accumulators in flight; the widest
  // tiles take what 512 TMEM columns / 4 CTAs allow.
  {
    const int stride = (nb + 31) & ~31;
    int st = 8;
    while (st > 1 && st * stride > 128) st >>= 1;
    p.acc_stages = st;
    p.acc_shift = st == 8 ? 3 : (st == 4 ? 2 : (st == 2 ? 1 : 0));
    int tc = 32;
    while (tc < st * stride) tc <<= 1;
    p.tmem_cols = tc;
  }
  p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(nb >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const bool wide = in_kind == 0 ? n4 > 16 : npos > 8;
  if (in_kind == 2) return wide ? launch_window<2, true>(p, stream) : launch_window<2, false>(p, stream);
  if (in_kind == 1) return wide ? launch_window<1, true>(p, stream) : launch_window<1, false>(p, stream);
  return wide ? launch_window<0, true>(p, stream) : launch_window<0, false>(p, stream);
}

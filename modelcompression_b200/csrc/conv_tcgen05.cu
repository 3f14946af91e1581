// conv_tcgen05.cu — Darknet-19 conv + folded-BN + leaky-ReLU as an implicit GEMM on tcgen05/TMEM, fed by TMA.
//
// Replaces: MaskedConv2d.forward -> F.conv2d (src/pruning/weightPruning/layers.py:53-64) followed by
// nn.BatchNorm2d (eval) and nn.LeakyReLU(0.1) (src/nets.py:802,809), the Reorg module (src/nets.py:648-667)
// and the route concat (src/nets.py:735-746), which are folded into the store addressing of the epilogue.
//
// Formulation.  Activations live in "PNHWC" (see include/mcb200.h): a 2-D bf16 matrix [rows, C] in which a
// 3x3 tap (dy,dx) is the constant row offset dy*(W+1)+dx and out-of-image reads hit zero rows/columns (or TMA
// out-of-bounds zero fill at the ends of the buffer).  So
//     Y[p, n] = sum_{tap} sum_{c} X[p + off(tap), c] * Wt[n, tap*Kc + c]
// is a plain GEMM whose A-tile row coordinate is shifted per k-block: no im2col buffer, no bounds logic.
// M tile = 128 rows (UMMA M=128, cta_group::1), N tile = block_n (16..256), K block = 64 bf16 = one
// 128-byte swizzle row (or 32 bf16 / 64-byte swizzle for <= 32 input channels).  Warp roles: warp0 = TMA producer,
// warp1 = TMEM owner + MMA issuer (warp-uniform loop, one elected lane issues), warps 2..5 = epilogue (TMEM -> regs ->
// scale/shift/leaky -> bf16/fp32 stores, through TMA-store slabs for PNHWC tiles >= 64 wide).
// Two kernels share this file, and with it the shared-memory carve-up and barrier set-up, the shared-activation-box
// mainloop (produce_box_groups / mma_box_unit) and the per-tile epilogue (epi_tile_begin / epilogue_tile):
//   conv_gemm_tcgen05_kernel<MINB>   persistent, 1..3 CTAs per SM (MINB = register budget), every layer shape;
//   conv_gemm_tcgen05_pair_kernel    cluster of 2 CTAs, tcgen05 cta_group::2: 256-row tiles, each CTA loads half of every
//                                    weight tile — the wide 3x3 layers (block_n >= 192, >= 36 k-blocks), with a
//                                    stream-K tail and the chained launch of several layers (mc_conv_chain_fwd).
// mc_conv_fwd picks kernel, tile width, ring depth and CTAs per SM (mc_conv_last_plan reports the choice).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "ptx_sm100.cuh"
#include "tmap.cuh"
#include "decode_math.cuh"

namespace {

constexpr int BLOCK_M = 128;  // k-block: 64 bf16 (128-byte swizzle rows) or 32 bf16 (64-byte swizzle rows), per launch
constexpr int MAX_STAGES = 8;
constexpr int MAX_A_STAGES = 3;  // activation-box ring: 3 boxes with one CTA per SM, 2 with several
constexpr int A_BOX_ROWS = BLOCK_M + 8;          // rows m0-1 .. m0+134: the dx = -1, 0, +1 windows of a 128-row tile
constexpr int A_BOX_BYTES = A_BOX_ROWS * 128;   // 17,408 B landed by TMA
constexpr int A_BOX_STRIDE = 18 * 1024;         // ring pitch (1024-byte aligned for the 128-byte swizzle)
constexpr int ACC_STAGES = 2;  // accumulator stages in TMEM: the MMA issuer runs this many tiles ahead of the epilogue
constexpr int NUM_THREADS = 192;
constexpr int WORK_SLOTS = 4;  // work ring of the CTA-pair kernel's chained launch (see PairRing)

struct ConvKParams {
  int M_rows;      // B*(H+1)*(W+1)
  int N;           // valid output channels
  int Npad;        // length of scale/shift arrays
  int num_kb;      // ntaps * kb_per_tap
  int kb_per_tap;  // Kc / block_k
  int block_k;     // 64 or 32
  int ksize;       // 1 or 3
  int Wp, Hp, W, H;  // Wp = W+1, Hp = H+1
  int block_n, stages, tmem_cols, acc_stride;  // acc_stride: TMEM columns between accumulator stages
  int out_pitch;   // > 0: PNHWC epilogue stages each warp's 32 rows in shared memory (row pitch in bytes) and writes them out coalesced
  int out_chunk;   // columns staged at a time (= block_n: see epilogue_loop)
  int tma_bufs;    // > 0: PNHWC epilogue writes whole 64-column chunks with TMA stores from this many 4 KB slabs per warp
  float* stat_sum;    // training forward: per-channel sum / sum of squares of the STORED (bf16-rounded) outputs are
  float* stat_sumsq;  // accumulated from the TMA-store slabs (the batch statistics of BatchNorm); nullptr: off
  unsigned int wp_mul, wp_shr, hp_mul, hp_shr;  // magic-number division by Wp and Hp (row -> x, y, b)
  int last_ksteps;  // UMMA K steps (16 channels) that hold real channels in the LAST channel block of a tap
  int share_dx, a_stages;  // 3x3 only: one A box (136 rows) serves the three dx taps of a filter row; separate A / B rings
  int m_tiles, n_tiles;
  uint32_t idesc;
  const float* scale;
  const float* shift;
  void* out;
  int ldc, ch_off, epi_mode, leaky;
  // stream-K tail of the CTA-pair kernel (sk_units > 0): the units of the last, partial wave are cut along K into equal
  // spans, one per cluster; spans that do not end a unit leave their fp32 accumulator in the workspace
  int sk_first, sk_units;        // first stream-K unit (the units before it run one per cluster and round), their number
  int sk_gper, sk_total_g;       // K groups (one activation box = 3 taps) per unit; sk_units * sk_gper
  int sk_clusters;               // clusters that take a stream-K span (<= 3 * sk_units: a unit has at most 4 pieces)
  unsigned int* sk_count;        // [sk_units] arrivals of partial writers (8 epilogue warps each), zeroed per launch
  float* sk_part;                // [sk_units][3][block_n / 4][256 rows][4] partial accumulators
  // MC_EPI_DECODE (region decode fused into the head's epilogue)
  float* dec_boxes;
  float* dec_cls;
  float* dec_head;
  int dec_A, dec_nc, dec_only_obj;
  float dec_thresh;
  McAnchors dec_anc;
  unsigned long long* dbg;  // mc_debug_conv_trace: globaltimer stamps, 32 slots per CTA (nullptr: no tracing)
};

// Timeline stamps of both kernels (slot layout in tools/trace_conv.py)
__device__ __forceinline__ void conv_stamp(const ConvKParams& p, int slot) {
  if (p.dbg != nullptr && slot < 32) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[(size_t)blockIdx.x * 32 + slot] = t;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Shared memory and its barriers.  PAIR: the CTA-pair kernel, which always shares the activation box, loads half of
// every B tile per CTA and adds the work ring of its chained launch.
struct ConvSmem {
  uint8_t* tiles;     // shared box: [a_stages x activation box] then b_ring; else [stages x (A tile | B tile)]
  uint8_t* b_ring;    // shared box: [stages x B tile]
  uint64_t* full_bar;        // [MAX_STAGES]  B tile (or A | B stage) landed
  uint64_t* empty_bar;       // [MAX_STAGES]  its MMAs retired
  uint64_t* tmem_full_bar;   // [ACC_STAGES]  accumulator complete
  uint64_t* tmem_empty_bar;  // [ACC_STAGES]  accumulator drained by the epilogue
  uint64_t* afull_bar;       // [MAX_A_STAGES] activation box landed
  uint64_t* aempty_bar;      // [MAX_A_STAGES] its three taps retired
  uint32_t* tmem_ptr;
  uint64_t* work_full;       // (PAIR) [WORK_SLOTS] work ring, see PairRing
  uint64_t* work_empty;      // (PAIR) [WORK_SLOTS]
  int* work_val;             // (PAIR) [WORK_SLOTS]
  float* s_ss;    // [2 acc stages][scale|shift][256]
  uint8_t* s_out;  // staged epilogue: [4 warps][32 rows][out_pitch]; TMA-store slabs [4 warps][tma_bufs][4 KB]
                   // (1024-byte aligned: swizzle pattern), then the batch-statistics accumulators; decode: logits
};

// box_stride: pitch of the activation-box ring; b_bytes: one B tile (of this CTA); stage_bytes: one A | B stage of the
// ring without a shared box.  The host reserves 5 KB for aux (barriers, scale/shift) plus 1 KB of alignment slack.
template <bool PAIR>
__device__ __forceinline__ ConvSmem carve_smem(uint8_t* smem, const ConvKParams& p, uint32_t box_stride,
                                               uint32_t b_bytes, uint32_t stage_bytes) {
  {  // dynamic smem base is only guaranteed 16B aligned: align up to 1024 (host adds 1 KB of slack)
    uint32_t a = ptx::smem_u32(smem);
    smem += (1024u - (a & 1023u)) & 1023u;
  }
  ConvSmem m;
  m.tiles = smem;
  m.b_ring = smem + (size_t)p.a_stages * box_stride;
  uint8_t* aux = (PAIR || p.share_dx) ? m.b_ring + (size_t)p.stages * b_bytes : smem + (size_t)p.stages * stage_bytes;
  m.full_bar = reinterpret_cast<uint64_t*>(aux);
  m.empty_bar = m.full_bar + MAX_STAGES;
  m.tmem_full_bar = m.empty_bar + MAX_STAGES;
  m.tmem_empty_bar = m.tmem_full_bar + ACC_STAGES;
  m.afull_bar = m.tmem_empty_bar + ACC_STAGES;
  m.aempty_bar = m.afull_bar + MAX_A_STAGES;
  m.tmem_ptr = reinterpret_cast<uint32_t*>(m.aempty_bar + MAX_A_STAGES);
  m.work_full = reinterpret_cast<uint64_t*>(aux + 256);
  m.work_empty = m.work_full + WORK_SLOTS;
  m.work_val = reinterpret_cast<int*>(m.work_empty + WORK_SLOTS);
  m.s_ss = reinterpret_cast<float*>(aux + 512);
  m.s_out = aux + 5120;
  return m;
}

// Barrier initialisation (thread 0) and TMEM allocation (warp 1), published to the block — PAIR: to both CTAs of the
// cluster, whose barriers must be initialised before any remote arrival / complete_tx.  Returns the TMEM base.
template <bool PAIR>
__device__ __forceinline__ uint32_t block_setup(const ConvSmem& m, const ConvKParams& p) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&m.full_bar[s], 1);
      ptx::mbar_init(&m.empty_bar[s], 1);
    }
    for (int a = 0; a < ACC_STAGES; ++a) {
      ptx::mbar_init(&m.tmem_full_bar[a], 1);
      ptx::mbar_init(&m.tmem_empty_bar[a], PAIR ? 8 : 4);  // one arrive per epilogue warp (PAIR: of each CTA)
    }
    for (int a = 0; a < MAX_A_STAGES; ++a) {
      ptx::mbar_init(&m.afull_bar[a], 1);
      ptx::mbar_init(&m.aempty_bar[a], 1);
    }
    if (PAIR) {
      for (int s = 0; s < WORK_SLOTS; ++s) {
        ptx::mbar_init(&m.work_full[s], 1);
        ptx::mbar_init(&m.work_empty[s], 10);  // leader: MMA warp + 4 epilogue warps; peer: producer + 4 epilogue warps
      }
    }
    ptx::fence_barrier_init();
  }
  if ((threadIdx.x >> 5) == 1) {
    if (PAIR) {
      ptx::tmem_alloc_pair(m.tmem_ptr, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(m.tmem_ptr, (uint32_t)p.tmem_cols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (PAIR) ptx::cluster_sync_all();
  else __syncthreads();
  ptx::tc_fence_after();
  return *m.tmem_ptr;
}

// ---------------------------------------------------------------------------------------------------------------
// Shared-activation-box mainloop (3x3 layers).  K group g = (filter row dy, channel block cb) of a tile: one 136-row
// activation box serves the three dx taps, which read it at row offsets 0, 1, 2, so the activations cross
// L2 -> smem 3 times per tile instead of 9; the B tile of every tap comes through its own ring.

// Ring positions and phases: B tiles (s), activation boxes (sa), accumulator stages (as)
struct Pipe {
  int stages, a_stages;
  int s = 0, sa = 0, as = 0;
  uint32_t phase = 0, pha = 0, aphase = 0;
  __device__ __forceinline__ Pipe(int stages_, int a_stages_) : stages(stages_), a_stages(a_stages_) {}
  __device__ __forceinline__ void next_b() { if (++s == stages) { s = 0; phase ^= 1u; } }
  __device__ __forceinline__ void next_box() { if (++sa == a_stages) { sa = 0; pha ^= 1u; } }
  __device__ __forceinline__ void next_acc() { if (++as == ACC_STAGES) { as = 0; aphase ^= 1u; } }
};

// Producer (one thread) of K groups [g0, g1) of the tile at rows m0, B rows n0.  box_bytes: one box (136 rows of one
// k-block row); b_bytes: one B tile of this CTA.  PAIR: every CTA loads its own box and its half of the B tile, and the
// leader's barriers count the bytes of both CTAs.
template <bool PAIR>
__device__ __forceinline__ void produce_box_groups(const ConvKParams& p, const ConvSmem& m, const CUtensorMap* tm_abox,
                                                   const CUtensorMap* tm_b, int m0, int n0, int g0, int g1,
                                                   uint32_t box_stride, uint32_t box_bytes, uint32_t b_bytes,
                                                   bool leader, Pipe& pp) {
  const int block_k = PAIR ? 64 : p.block_k;
  for (int g = g0; g < g1; ++g) {
    const int dy = g / p.kb_per_tap, cb = g - dy * p.kb_per_tap;
    ptx::mbar_wait(&m.aempty_bar[pp.sa], pp.pha ^ 1u);
    if (leader) ptx::mbar_arrive_expect_tx(&m.afull_bar[pp.sa], PAIR ? 2 * box_bytes : box_bytes);
    uint8_t* box = m.tiles + (size_t)pp.sa * box_stride;
    const int box_row = m0 + (dy - 1) * p.Wp - 1;
    if (PAIR) ptx::tma_load_2d_pair(box, tm_abox, &m.afull_bar[pp.sa], cb * block_k, box_row);
    else ptx::tma_load_2d(box, tm_abox, &m.afull_bar[pp.sa], cb * block_k, box_row);
    pp.next_box();
    for (int dx = 0; dx < 3; ++dx) {
      const int kb = (dy * 3 + dx) * p.kb_per_tap + cb;
      ptx::mbar_wait(&m.empty_bar[pp.s], pp.phase ^ 1u);
      if (leader) ptx::mbar_arrive_expect_tx(&m.full_bar[pp.s], PAIR ? 2 * b_bytes : b_bytes);
      uint8_t* b_dst = m.b_ring + (size_t)pp.s * b_bytes;
      if (PAIR) ptx::tma_load_2d_pair(b_dst, tm_b, &m.full_bar[pp.s], kb * block_k, n0);
      else ptx::tma_load_2d(b_dst, tm_b, &m.full_bar[pp.s], kb * block_k, n0);
      pp.next_b();
    }
  }
}

template <bool PAIR>
__device__ __forceinline__ void umma_commit_both(uint64_t* bar) {  // PAIR: on this barrier in both CTAs
  if (PAIR) ptx::umma_commit_pair(bar);
  else ptx::umma_commit(bar);
}

// MMA issue of one tile, K groups [g0, g1), into the next accumulator stage (ti: tiles this CTA issued before, for
// tracing).  The WHOLE warp walks the loop (warp-uniform control flow and operands, so descriptors live in uniform
// registers) and one elected lane issues the tcgen05 instructions.  With the loop inside `if (lane == 0)` the compiler
// wraps every UTCHMMA in a vote/R2UR.BROADCAST loop (~25 instructions), and that single thread's issue rate — not the
// tensor pipe — bounds the k-block time.
template <bool PAIR>
__device__ __forceinline__ void mma_box_unit(const ConvKParams& p, const ConvSmem& m, uint32_t tmem_base, int g0,
                                             int g1, uint32_t box_stride, uint32_t b_bytes, Pipe& pp, int ti) {
  const int lane = threadIdx.x & 31;
  ptx::mbar_wait(&m.tmem_empty_bar[pp.as], pp.aphase ^ 1u);  // the epilogue has drained this accumulator stage
  ptx::tc_fence_after();
  const uint32_t tmem_acc = tmem_base + (uint32_t)(pp.as * p.acc_stride);
  const bool k64 = PAIR || p.block_k == 64;
  // (copied out of the parameters once: the asm statements below clobber memory, which would reload them per MMA)
  const int kbt = p.kb_per_tap, lks = p.last_ksteps;
  const uint32_t idesc = p.idesc;
  for (int g = g0; g < g1; ++g) {
    // K steps beyond the layer's real channels multiply TMA zero fill by zero weights: not issued
    const int nk = (g % kbt == kbt - 1) ? lks : (k64 ? 4 : 2);
    ptx::mbar_wait(&m.afull_bar[pp.sa], pp.pha);
    if (ti == 0 && g == g0 && lane == 0) conv_stamp(p, 4);
    const uint32_t a_addr = ptx::smem_u32(m.tiles + (size_t)pp.sa * box_stride);
    for (int dx = 0; dx < 3; ++dx) {
      ptx::mbar_wait(&m.full_bar[pp.s], pp.phase);
      ptx::tc_fence_after();
      const uint32_t b_addr = ptx::smem_u32(m.b_ring + (size_t)pp.s * b_bytes);
      // the window of tap dx starts dx rows (dx * 128 B) into the box.  The start is then not aligned to the
      // 1024-byte swizzle pattern; measured on B200: the tensor core applies the 128-byte swizzle to the absolute
      // shared-memory address (as TMA did when it wrote the box), so the descriptor's base-offset field must stay
      // 0 — setting it to dx (or 8-dx) reads garbage (tools/debug_share.py)
      // (32-wide k-blocks: the same holds for the 64-byte swizzle — rows of 64 B, window dx starts dx * 64 B in)
      const uint64_t adesc = k64 ? ptx::make_sw128_kmajor_desc(a_addr + (uint32_t)dx * 128u)
                                 : ptx::make_sw64_kmajor_desc(a_addr + (uint32_t)dx * 64u);
      const uint64_t bdesc = k64 ? ptx::make_sw128_kmajor_desc(b_addr) : ptx::make_sw64_kmajor_desc(b_addr);
      if (ptx::elect_one()) {
        // (compile-time trip count with a per-step predicate: this issue loop is on the critical path, a
        //  run-time trip count costs the narrow-Cin layers ~4 us each)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          // advance 16 bf16 = 32 B along K inside the swizzle row: +2 in the (addr>>4) field
          const uint32_t acc = (g > g0 || dx > 0 || k > 0) ? 1u : 0u;
          if (k < nk) {
            if (PAIR) ptx::umma_bf16_ss_pair(tmem_acc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, acc);
            else ptx::umma_bf16_ss(tmem_acc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, acc);
          }
        }
        umma_commit_both<PAIR>(&m.empty_bar[pp.s]);
        if (dx == 2) umma_commit_both<PAIR>(&m.aempty_bar[pp.sa]);  // the box may be refilled once its three taps retire
        if (dx == 2 && g == g1 - 1) umma_commit_both<PAIR>(&m.tmem_full_bar[pp.as]);
      }
      __syncwarp();
      pp.next_b();
    }
    pp.next_box();
  }
  if (lane == 0 && ti < 6) conv_stamp(p, 5 + ti);
  pp.next_acc();
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogue of one accumulator tile (warps 2..5: warp w owns TMEM lanes / tile rows 32*(w & 3) .. +31).

// 16 accumulator columns of one row: y = acc*scale + shift (-> leaky) ; rows outside the image become 0.
template <bool LEAKY>
__device__ __forceinline__ void scale_act16(const uint32_t (&r)[16], const float* __restrict__ sc,
                                            const float* __restrict__ sh, bool interior, float (&v)[16]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 a = *reinterpret_cast<const float4*>(sc + 4 * q);  // same address in every lane: smem broadcast
    const float4 b = *reinterpret_cast<const float4*>(sh + 4 * q);
    v[4 * q + 0] = fmaf(__uint_as_float(r[4 * q + 0]), a.x, b.x);
    v[4 * q + 1] = fmaf(__uint_as_float(r[4 * q + 1]), a.y, b.y);
    v[4 * q + 2] = fmaf(__uint_as_float(r[4 * q + 2]), a.z, b.z);
    v[4 * q + 3] = fmaf(__uint_as_float(r[4 * q + 3]), a.w, b.w);
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    if (LEAKY) v[j] = fmaxf(v[j], 0.1f * v[j]);
    v[j] = interior ? v[j] : 0.f;
  }
}

// 8 fp32 -> 8 bf16 (round to nearest even) in one 16-byte word
__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(v[0], v[1]);
  const __nv_bfloat162 h1 = __floats2bfloat162_rn(v[2], v[3]);
  const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[4], v[5]);
  const __nv_bfloat162 h3 = __floats2bfloat162_rn(v[6], v[7]);
  return make_uint4(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1),
                    *reinterpret_cast<const uint32_t*>(&h2), *reinterpret_cast<const uint32_t*>(&h3));
}

template <int MODE>
__device__ __forceinline__ void store16(const ConvKParams& p, const float (&v)[16], int nbase, long long out_row_base,
                                        bool vec_ok) {
  if (MODE == MC_EPI_NCHW_F32 || MODE == MC_EPI_DECODE) {
    float* out_f = reinterpret_cast<float*>(p.out);
    const long long hw = (long long)p.H * p.W;
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (nbase + j < p.N) out_f[out_row_base + (long long)(nbase + j) * hw] = v[j];
  } else {
    __nv_bfloat16* out_bf = reinterpret_cast<__nv_bfloat16*>(p.out) + out_row_base;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const int n = nbase + g * 8;
      if (n >= p.N) continue;
      // channels >= N of a PNHWC row are zero padding up to the pitch: a partial 8-group is still written as one
      // 16-byte store (zeros there) when it fits inside the pitch
      const bool full = n + 8 <= p.N;
      if (vec_ok && (full || (MODE == MC_EPI_PNHWC && p.ch_off + n + 8 <= p.ldc))) {
        float w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = (full || n + j < p.N) ? v[g * 8 + j] : 0.f;
        *reinterpret_cast<uint4*>(out_bf + n) = pack8_bf16(w);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (n + j < p.N) out_bf[n + j] = __float2bfloat16_rn(v[g * 8 + j]);
      }
    }
  }
}

// 16 fp32 -> 16 bf16 -> two 16-byte shared-memory stores
__device__ __forceinline__ void pack16_to_smem(const float (&v)[16], uint8_t* dst) {
#pragma unroll
  for (int g = 0; g < 2; ++g) *reinterpret_cast<uint4*>(dst + g * 16) = pack8_bf16(v + g * 8);
}

// 16 fp32 -> 16 bf16 -> the two 16-byte chunks (index chunk, chunk + 1) of this lane's 128-byte row of a TMA store
// slab.  The slab has the tensor map's 128-byte swizzle: chunk j of row r sits at chunk position j ^ (r & 7).
__device__ __forceinline__ void pack16_to_slab(const float (&v)[16], uint8_t* row, int chunk, int lane) {
#pragma unroll
  for (int g = 0; g < 2; ++g)
    *reinterpret_cast<uint4*>(row + (((chunk + g) ^ (lane & 7)) << 4)) = pack8_bf16(v + g * 8);
}

// Batch statistics from a finished 32-row x 64-column slab: lane L owns columns 2L, 2L+1 (one 4-byte word per row: the
// 32 lanes read 32 different words of a 128-byte row, conflict-free) and adds the 32 rows into this warp's private
// shared-memory accumulators acc[0][col] (sum) / acc[1][col] (sum of squares); pad rows hold zeros.
__device__ __forceinline__ void slab_stats(const uint8_t* sb, float* acc /*[2][256]*/, int col0, int lane) {
  float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
  const int j = lane >> 2, w = lane & 3;
#pragma unroll 8
  for (int r = 0; r < 32; ++r) {
    const uint32_t u = *reinterpret_cast<const uint32_t*>(sb + r * 128 + ((j ^ (r & 7)) << 4) + w * 4);
    const float a = __uint_as_float(u << 16), b = __uint_as_float(u & 0xffff0000u);
    s0 += a; s1 += b;
    q0 = fmaf(a, a, q0); q1 = fmaf(b, b, q1);
  }
  acc[col0 + 2 * lane] += s0;
  acc[col0 + 2 * lane + 1] += s1;
  acc[256 + col0 + 2 * lane] += q0;
  acc[256 + col0 + 2 * lane + 1] += q1;
}
// the warp's accumulated statistics of N tile n0 -> global (one atomic per column, statistic and warp), then zero
__device__ __forceinline__ void flush_stats(const ConvKParams& p, float* acc, int n0, int lane) {
  for (int c = lane; c < p.block_n; c += 32) {
    if (n0 + c < p.N) {
      atomicAdd(p.stat_sum + n0 + c, acc[c]);
      atomicAdd(p.stat_sumsq + n0 + c, acc[256 + c]);
    }
    acc[c] = 0.f;
    acc[256 + c] = 0.f;
  }
  __syncwarp();
}

// scale/shift of columns [n0, n0 + block_n) -> dst[i] / dst[256 + i], zeros beyond Npad (the 128 epilogue threads)
__device__ __forceinline__ void stage_scale_shift(const ConvKParams& p, float* dst, int n0) {
  for (int i = (int)threadIdx.x - 64; i < p.block_n; i += 128) {
    const bool ok = (n0 + i) < p.Npad;
    dst[i] = ok ? __ldg(p.scale + n0 + i) : 0.f;
    dst[256 + i] = ok ? __ldg(p.shift + n0 + i) : 0.f;
  }
}

// this warp has finished reading the accumulator stage: hand it back to the MMA issuer (PAIR: on the leader CTA's
// barrier, where the MMA issuer waits for the epilogues of both CTAs)
template <bool PAIR>
__device__ __forceinline__ void release_acc_stage(uint64_t* empty_bar) {
  ptx::tc_fence_before();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) {
    if (PAIR) ptx::mbar_arrive_leader(empty_bar);
    else ptx::mbar_arrive(empty_bar);
  }
}

// Start of an epilogue loop.  Batch statistics: zero this warp's accumulators behind the TMA-store slabs (returned;
// flushed whenever the N tile changes and at the end).  One N tile: every tile of the launch uses the same
// scale/shift slice, staged once (a narrow layer's epilogue is otherwise a chain of global-load latency + barrier per
// 128 rows).
template <int MODE>
__device__ __forceinline__ float* epilogue_begin(const ConvKParams& p, const ConvSmem& m, bool one_n_tile) {
  float* stat_acc = nullptr;
  if (MODE == MC_EPI_PNHWC && p.tma_bufs > 0 && p.stat_sum != nullptr) {
    stat_acc = reinterpret_cast<float*>(m.s_out + (size_t)4 * p.tma_bufs * 4096) + ((threadIdx.x >> 5) & 3) * 512;
    for (int c = threadIdx.x & 31; c < 512; c += 32) stat_acc[c] = 0.f;
    __syncwarp();
  }
  if (one_n_tile) {
    stage_scale_shift(p, m.s_ss, 0);
    asm volatile("bar.sync 1, 128;" ::: "memory");
  }
  return stat_acc;
}

template <int MODE>
__device__ __forceinline__ void epilogue_end(const ConvKParams& p, float* stat_acc, int stat_n0) {
  const int lane = threadIdx.x & 31;
  if (stat_acc != nullptr && stat_n0 >= 0) flush_stats(p, stat_acc, stat_n0, lane);
  if (MODE == MC_EPI_PNHWC && p.tma_bufs > 0 && lane == 0) ptx::bulk_wait_group_read<0>();  // slabs read before the CTA exits
}

// One accumulator tile as this thread sees it: its row, its pixel and where its outputs go
struct EpiTile {
  const float* sc;   // scale of the tile's columns in shared memory; the shift follows at sc + 256
  uint32_t taddr;    // TMEM address of this warp's 32 lanes in the accumulator stage
  int n0, row0;      // first column; first row of this warp's 32
  int x, y, b;       // this thread's pixel (x >= W or y >= H: pad row)
  bool in_buf, interior, do_store;
  long long out_row_base;
};

// Start of one tile in the epilogue: stage its scale/shift (unless staged once for the launch), decode the row ->
// (b, y, x) by magic-number division, address the output for the store mode and wait for the accumulator stage `as`.
// ti: tiles this CTA's epilogue did before (tracing).
template <int MODE>
__device__ __forceinline__ EpiTile epi_tile_begin(const ConvKParams& p, const ConvSmem& m, uint32_t tmem_base,
                                                  bool one_n_tile, int m0, int n0, int as, uint32_t aphase, int ti) {
  const int quarter = (threadIdx.x >> 5) & 3;  // TMEM lane quarter this warp may access
  EpiTile t;
  float* sc = m.s_ss + (one_n_tile ? 0 : as * 512);
  if (!one_n_tile) stage_scale_shift(p, sc, n0);
  t.sc = sc;
  t.n0 = n0;
  t.row0 = m0 + quarter * 32;
  const int row = t.row0 + (threadIdx.x & 31);
  const int q = (int)(__umulhi((unsigned int)row, p.wp_mul) >> p.wp_shr);  // row / Wp
  t.x = row - q * p.Wp;
  t.b = (int)(__umulhi((unsigned int)q, p.hp_mul) >> p.hp_shr);            // (row / Wp) / Hp
  t.y = q - t.b * p.Hp;
  t.in_buf = row < p.M_rows;
  t.interior = t.in_buf && (t.x < p.W) && (t.y < p.H);
  if (MODE == MC_EPI_PNHWC) {
    t.out_row_base = (long long)row * p.ldc + p.ch_off;
    t.do_store = t.in_buf;  // pad rows are written as zeros to keep the layout invariant
  } else if (MODE == MC_EPI_REORG2) {
    const int Wo = p.W / 2 + 1, Ho = p.H / 2 + 1;
    const long long orow = ((long long)t.b * Ho + (t.y >> 1)) * Wo + (t.x >> 1);
    t.out_row_base = orow * p.ldc + p.ch_off + ((t.y & 1) * 2 + (t.x & 1)) * p.N;
    t.do_store = t.interior;
  } else {  // MC_EPI_NCHW_F32 (+ n*H*W); MC_EPI_DECODE addresses its outputs itself
    t.out_row_base = ((long long)t.b * p.N * p.H + t.y) * p.W + t.x;
    t.do_store = t.interior;
  }
  if (!one_n_tile) asm volatile("bar.sync 1, 128;" ::: "memory");  // scale/shift of this tile visible to the 4 warps

  ptx::mbar_wait(&m.tmem_full_bar[as], aphase);
  ptx::tc_fence_after();
  if (threadIdx.x == 64 && ti < 8) conv_stamp(p, 12 + 2 * ti);
  t.taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * p.acc_stride);
  return t;
}

// Direct stores of accumulator columns [c_begin, block_n), 32 at a time: a thread writes its own row.  add(r, col)
// runs on the raw accumulator first (a stream-K finisher adds the partial accumulators there; otherwise a no-op).
template <int MODE, bool LEAKY, typename AddFn>
__device__ __forceinline__ void store_cols_direct(const ConvKParams& p, const EpiTile& t, int c_begin, bool vec_ok,
                                                  AddFn& add) {
  const float* sc = t.sc;
  const float* sh = t.sc + 256;
  for (int c0 = c_begin; c0 < p.block_n; c0 += 32) {
    uint32_t r0[16], r1[16];
    const bool two = c0 + 16 < p.block_n;
    ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)c0, r0);
    if (two) ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(c0 + 16), r1);
    ptx::tmem_ld_wait();
    if (!t.do_store) continue;
    add(r0, c0);
    if (two) add(r1, c0 + 16);
    float v[16];
    scale_act16<LEAKY>(r0, sc + c0, sh + c0, t.interior, v);
    store16<MODE>(p, v, t.n0 + c0, t.out_row_base, vec_ok);
    if (two) {
      scale_act16<LEAKY>(r1, sc + c0 + 16, sh + c0 + 16, t.interior, v);
      store16<MODE>(p, v, t.n0 + c0 + 16, t.out_row_base, vec_ok);
    }
  }
}

// PNHWC epilogue of one accumulator tile through TMA stores.  A warp owns 32 rows; every whole 64-column chunk of the
// tile is converted into the warp's 4 KB slab (32 rows x 128 B, swizzled like the tensor map of the output) and leaves
// as ONE bulk tensor store — 128-byte rows, issued by one lane, asynchronous — instead of 16-byte pieces one row pitch
// apart per thread (measured: ~38 cycles per output column and tile, 4..7.6 us for a 208..256-wide tile, which
// throttles short-K layers and is exposed after the last tile of every CTA).  With two slabs per warp the conversion of
// chunk i+1 overlaps the store of chunk i.  The tile's last block_n % 64 columns take direct stores; rows and columns
// outside the output tensor are clipped by TMA.
template <bool LEAKY, bool WIDE_LD, typename AddFn>
__device__ __forceinline__ void epilogue_tile_tma(const ConvKParams& p, const CUtensorMap* tm_out, const EpiTile& t,
                                                  bool vec_ok, uint8_t* slab, int& buf, AddFn& add, float* stat_acc) {
  const int lane = threadIdx.x & 31;
  const float* sc = t.sc;
  const float* sh = t.sc + 256;
  int cols_valid = ((p.N - t.n0 + 7) >> 3) << 3;  // whole 8-groups up to the last one holding a real channel
  if (cols_valid > p.block_n) cols_valid = p.block_n;
  const int full_cols = p.block_n & ~63;
  for (int cc = 0; cc < full_cols && cc < cols_valid; cc += 64) {
    uint8_t* sb = slab + (size_t)buf * 4096;
    if (lane == 0) {  // the store that last read this slab has finished reading it
      if (p.tma_bufs >= 2) ptx::bulk_wait_group_read<1>();
      else ptx::bulk_wait_group_read<0>();
    }
    __syncwarp();
    uint8_t* mine = sb + lane * 128;
    if (WIDE_LD) {
      // all 64 columns of the chunk in flight before the one wait (register budget of the 1-CTA-per-SM variants)
      uint32_t r[4][16];
#pragma unroll
      for (int q = 0; q < 4; ++q) ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(cc + 16 * q), r[q]);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        add(r[q], cc + 16 * q);
        float v[16];
        scale_act16<LEAKY>(r[q], sc + cc + 16 * q, sh + cc + 16 * q, t.interior, v);
        pack16_to_slab(v, mine, 2 * q, lane);
      }
    } else {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r0[16], r1[16];
        ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(cc + 32 * h), r0);
        ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(cc + 32 * h + 16), r1);
        ptx::tmem_ld_wait();
        add(r0, cc + 32 * h);
        add(r1, cc + 32 * h + 16);
        float v[16];
        scale_act16<LEAKY>(r0, sc + cc + 32 * h, sh + cc + 32 * h, t.interior, v);
        pack16_to_slab(v, mine, 4 * h, lane);
        scale_act16<LEAKY>(r1, sc + cc + 32 * h + 16, sh + cc + 32 * h + 16, t.interior, v);
        pack16_to_slab(v, mine, 4 * h + 2, lane);
      }
    }
    ptx::fence_proxy_async_smem();  // this lane's slab writes -> visible to the TMA (async proxy)
    __syncwarp();
    if (lane == 0) {
      ptx::tma_store_2d(tm_out, sb, t.n0 + cc, t.row0);
      ptx::bulk_commit_group();
    }
    if (stat_acc != nullptr) slab_stats(sb, stat_acc, cc, lane);
    if (p.tma_bufs >= 2) buf ^= 1;
  }
  store_cols_direct<MC_EPI_PNHWC, LEAKY>(p, t, full_cols, vec_ok, add);
}

// Scale/shift/leaky and store of one accumulator tile in both kernels — TMA stores (PNHWC, p.tma_bufs > 0) or direct
// stores — then the stage goes back to the MMA issuer.  add(r, col): see store_cols_direct.  slab_buf, stat_acc and
// stat_n0 are the warp's TMA-store slab and batch-statistics state across tiles.
template <int MODE, bool LEAKY, bool PAIR, bool WIDE_LD, typename AddFn>
__device__ __forceinline__ void epilogue_tile(const ConvKParams& p, const CUtensorMap* tm_out, const ConvSmem& m,
                                              const EpiTile& t, bool vec_ok, uint64_t* empty_bar, int& slab_buf,
                                              float* stat_acc, int& stat_n0, AddFn add) {
  if (MODE == MC_EPI_PNHWC && p.tma_bufs > 0) {
    if (stat_acc != nullptr && t.n0 != stat_n0) {
      if (stat_n0 >= 0) flush_stats(p, stat_acc, stat_n0, threadIdx.x & 31);
      stat_n0 = t.n0;
    }
    uint8_t* slab = m.s_out + (size_t)((threadIdx.x >> 5) & 3) * p.tma_bufs * 4096;
    epilogue_tile_tma<LEAKY, WIDE_LD>(p, tm_out, t, vec_ok, slab, slab_buf, add, stat_acc);
  } else {
    store_cols_direct<MODE, LEAKY>(p, t, 0, vec_ok, add);
  }
  release_acc_stage<PAIR>(empty_bar);
}

// Epilogue warps (threads 64..191) of the single-CTA kernel: tiles blockIdx.x, + gridDim.x, ...  Besides the TMA-store
// and direct paths of epilogue_tile, PNHWC tiles without TMA stores take the staged store where the planner gave them a
// staging buffer (p.out_pitch > 0), and the head takes the decode.
template <int MODE, bool LEAKY, bool WIDE_LD = false>
__device__ __forceinline__ void epilogue_loop(const ConvKParams& p, const ConvSmem& m, uint32_t tmem_base,
                                              const CUtensorMap* tm_out) {
  const int lane = threadIdx.x & 31;
  const int quarter = (threadIdx.x >> 5) & 3;
  const int total_tiles = p.m_tiles * p.n_tiles;
  const bool vec_ok = ((p.ldc | p.ch_off) & 7) == 0 && (MODE != MC_EPI_REORG2 || (p.N & 7) == 0);
  const bool one_n_tile = p.n_tiles == 1;
  float* stat_acc = epilogue_begin<MODE>(p, m, one_n_tile);
  int stat_n0 = -1;
  int slab_buf = 0;  // (TMA-store epilogue) slab of this warp the next chunk goes to
  int as = 0;
  uint32_t aphase = 0;
  int ti = 0;  // (tracing) tiles done by this CTA
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++ti) {
    const int n0 = (tile % p.n_tiles) * p.block_n;
    const int m0 = (tile / p.n_tiles) * BLOCK_M;
    const EpiTile t = epi_tile_begin<MODE>(p, m, tmem_base, one_n_tile, m0, n0, as, aphase, ti);

    if (MODE == MC_EPI_PNHWC && p.tma_bufs == 0 && p.out_pitch > 0) {
      // Staged store: a thread owns one output ROW, so direct stores are 16-byte pieces one row pitch apart (32 half-
      // filled sectors per warp instruction: measured ~38 cycles per output column and tile).  Instead the warp parks
      // its 32 rows x block_n bf16 in shared memory (pitch +16 B: conflict-free), hands the TMEM stage back at once,
      // and writes the rows out with consecutive lanes on consecutive 16-byte chunks.  The planner stages only the 32-
      // and 48-wide tiles (wider aligned tiles take the TMA stores), so out_chunk == block_n and the chunk loop runs
      // once; written as one pass instead, the kernel spills more (ptxas, kernel<3>: 248 / 432 B of spill stores /
      // loads instead of 224 / 328 B).
      const int pitch = p.out_pitch;
      const int chunk = p.out_chunk;
      uint8_t* wbuf = m.s_out + (size_t)quarter * 32 * pitch;
      uint8_t* mine = wbuf + (size_t)lane * pitch;
      int cols_left = ((p.N - n0 + 7) >> 3) << 3;  // whole 8-groups up to the last one holding a real channel
      if (cols_left > p.block_n) cols_left = p.block_n;
      for (int cc = 0; cc < p.block_n; cc += chunk) {
        const int cw = (p.block_n - cc < chunk) ? p.block_n - cc : chunk;
        for (int c0 = 0; c0 < cw; c0 += 32) {
          uint32_t r0[16], r1[16];
          const bool two = c0 + 16 < cw;
          ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(cc + c0), r0);
          if (two) ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(cc + c0 + 16), r1);
          ptx::tmem_ld_wait();
          float v[16];
          scale_act16<LEAKY>(r0, t.sc + cc + c0, t.sc + 256 + cc + c0, t.interior, v);
          pack16_to_smem(v, mine + c0 * 2);
          if (two) {
            scale_act16<LEAKY>(r1, t.sc + cc + c0 + 16, t.sc + 256 + cc + c0 + 16, t.interior, v);
            pack16_to_smem(v, mine + (c0 + 16) * 2);
          }
        }
        if (cc + chunk >= p.block_n) release_acc_stage<false>(&m.tmem_empty_bar[as]);  // before the copy-out
        else __syncwarp();
        int cols_w = cols_left - cc;
        if (cols_w > cw) cols_w = cw;
        if (cols_w > 0) {
          const int cpr = cols_w >> 3;  // 16-byte chunks per row
          int r = lane / cpr, c = lane - r * cpr;
          const int dr = 32 / cpr, dc = 32 - dr * cpr;
          __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out) + p.ch_off + n0 + cc;
          while (r < 32) {
            if (t.row0 + r < p.M_rows)
              *reinterpret_cast<uint4*>(obase + (long long)(t.row0 + r) * p.ldc + c * 8) =
                  *reinterpret_cast<const uint4*>(wbuf + (size_t)r * pitch + c * 16);
            r += dr; c += dc;
            if (c >= cpr) { c -= cpr; ++r; }
          }
        }
        __syncwarp();  // wbuf is rewritten by the next chunk / tile
      }
    } else if (MODE == MC_EPI_DECODE) {
      // Region decode in the epilogue (get_region_boxes, src/nets2_utils.py:158-205).  The thread owns pixel (b, y, x):
      // its A*(5+nc) logits (= acc*scale + shift, the head's bias) are parked in the warp's shared-memory rows (row
      // pitch block_n+1 floats: lanes hit different banks), the TMEM stage goes back to the MMA issuer at once, and the
      // thread then decodes its A anchors from shared memory with the arithmetic of decode_math.cuh.
      const int pitch_f = p.block_n + 1;
      float* mine = reinterpret_cast<float*>(m.s_out) + (size_t)(quarter * 32 + lane) * pitch_f;
      for (int c0 = 0; c0 < p.block_n; c0 += 16) {
        uint32_t r0[16];
        ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)c0, r0);
        ptx::tmem_ld_wait();
        float v[16];
        scale_act16<LEAKY>(r0, t.sc + c0, t.sc + 256 + c0, true, v);
#pragma unroll
        for (int j = 0; j < 16; ++j) mine[c0 + j] = v[j];
      }
      release_acc_stage<false>(&m.tmem_empty_bar[as]);
      if (t.interior) {
        const int x = t.x, y = t.y, b = t.b;
        const int A = p.dec_A, nc = p.dec_nc, F = 5 + p.dec_nc;
        const long long P = (long long)p.H * p.W * A;
        const long long slot0 = (long long)(y * p.W + x) * A;
        if (p.dec_head != nullptr) {
          float* hd = p.dec_head + ((long long)b * p.N * p.H + y) * p.W + x;
          const long long hw = (long long)p.H * p.W;
          for (int n = 0; n < p.N; ++n) hd[n * hw] = mine[n];
        }
        for (int a = 0; a < A; ++a) {
          const float* row = mine + a * F;
          const McDecoded d = mc_decode_anchor([row](int f) { return row[f]; }, nc, x, y, p.W, p.H, p.dec_anc.w[a],
                                               p.dec_anc.h[a], p.dec_thresh, p.dec_only_obj);
          float* dst = p.dec_boxes + ((long long)b * P + slot0 + a) * 8;
          reinterpret_cast<float4*>(dst)[0] = make_float4(d.bx, d.by, d.bw, d.bh);
          reinterpret_cast<float4*>(dst)[1] =
              make_float4(d.conf, d.cmax, (float)d.cid, d.cand ? (float)(slot0 + a) : -1.0f);
          if (d.cand && p.dec_cls != nullptr) {
            float* cd = p.dec_cls + ((long long)b * P + slot0 + a) * nc;
            for (int c = 0; c < nc; ++c) cd[c] = __fdiv_rn(expf(__fsub_rn(row[5 + c], d.cls_max_logit)), d.cls_sum);
          }
        }
      }
      __syncwarp();  // the rows are rewritten by the next tile
    } else {
      epilogue_tile<MODE, LEAKY, false, WIDE_LD>(p, tm_out, m, t, vec_ok, &m.tmem_empty_bar[as], slab_buf, stat_acc,
                                                 stat_n0, [](uint32_t (&)[16], int) {});
    }
    if (MODE != MC_EPI_DECODE && threadIdx.x == 64 && ti < 8) conv_stamp(p, 13 + 2 * ti);
    if (++as == ACC_STAGES) { as = 0; aphase ^= 1u; }
  }
  epilogue_end<MODE>(p, stat_acc, stat_n0);
}

// Persistent: grid = min(#tiles, #SMs); CTA c works on tiles c, c+grid, ...  The smem ring runs across tiles, and the
// accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// MINB (resident CTAs per SM the register budget allows): 1 for the wide compute-bound tiles; 3 for narrow layers
// (few output channels / short K), whose per-tile chain TMA -> MMA -> commit -> epilogue -> TMEM hand-back is latency
// bound inside one CTA — several CTAs per SM (each with its own small smem ring and TMEM slice) overlap those chains.
template <int MINB>
__global__ void __launch_bounds__(NUM_THREADS, MINB)
conv_gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ CUtensorMap tmap_abox, const __grid_constant__ CUtensorMap tmap_out,
                         const ConvKParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t a_tile_bytes = (uint32_t)(BLOCK_M * p.block_k * 2);
  const uint32_t b_tile_bytes = (uint32_t)(p.block_n * p.block_k * 2);
  const uint32_t stage_bytes = a_tile_bytes + b_tile_bytes;
  // shared activation box: 136 rows of one k-block row (128 B with 64-wide k-blocks / 128-byte swizzle, 64 B with 32-wide
  // k-blocks / 64-byte swizzle); ring pitch 18 KB / 9 KB keeps every box 1024-byte aligned
  const uint32_t box_bytes = (uint32_t)A_BOX_ROWS * (uint32_t)p.block_k * 2u;
  const uint32_t box_stride = p.block_k == 64 ? (uint32_t)A_BOX_STRIDE : (uint32_t)A_BOX_STRIDE / 2u;
  const ConvSmem m = carve_smem<false>(smem_raw, p, box_stride, b_tile_bytes, stage_bytes);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.m_tiles * p.n_tiles;
  if (threadIdx.x == 0) {
    conv_stamp(p, 0);
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_b);
    ptx::prefetch_tensormap(&tmap_abox);
    if (p.tma_bufs > 0) ptx::prefetch_tensormap(&tmap_out);
  }
  const uint32_t tmem_base = block_setup<false>(m, p);
  if (threadIdx.x == 0) conv_stamp(p, 1);

  if (warp_idx == 0) {
    // ===================== TMA producer (one thread) =====================
    if (lane == 0) {
      if (p.share_dx) {
        Pipe pp(p.stages, p.a_stages);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
          const int n0 = (tile % p.n_tiles) * p.block_n;
          const int m0 = (tile / p.n_tiles) * BLOCK_M;
          produce_box_groups<false>(p, m, &tmap_abox, &tmap_b, m0, n0, 0, 3 * p.kb_per_tap, box_stride, box_bytes,
                                    b_tile_bytes, true, pp);
        }
      } else {
        int s = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
          const int n0 = (tile % p.n_tiles) * p.block_n;
          const int m0 = (tile / p.n_tiles) * BLOCK_M;
          for (int kb = 0; kb < p.num_kb; ++kb) {
            const int tap = kb / p.kb_per_tap;
            const int cb = kb - tap * p.kb_per_tap;
            int row_off = 0;
            if (p.ksize == 3) row_off = (tap / 3 - 1) * p.Wp + (tap % 3 - 1);
            ptx::mbar_wait(&m.empty_bar[s], phase ^ 1u);
            uint8_t* a_dst = m.tiles + (size_t)s * stage_bytes;
            uint8_t* b_dst = a_dst + a_tile_bytes;
            ptx::mbar_arrive_expect_tx(&m.full_bar[s], stage_bytes);
            ptx::tma_load_2d(a_dst, &tmap_a, &m.full_bar[s], cb * p.block_k, m0 + row_off);
            ptx::tma_load_2d(b_dst, &tmap_b, &m.full_bar[s], kb * p.block_k, n0);
            if (++s == p.stages) { s = 0; phase ^= 1u; }
          }
        }
      }
      conv_stamp(p, 3);
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer (whole warp, one elected lane issues: see mma_box_unit) =====================
    if (p.share_dx) {
      Pipe pp(p.stages, p.a_stages);
      int ti = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++ti)
        mma_box_unit<false>(p, m, tmem_base, 0, 3 * p.kb_per_tap, box_stride, b_tile_bytes, pp, ti);
    } else {
      // one A | B stage per k-block, the A tile already shifted to the tap
      int s = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      int ti = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++ti) {
        ptx::mbar_wait(&m.tmem_empty_bar[as], aphase ^ 1u);  // epilogue has drained this accumulator stage
        ptx::tc_fence_after();
        const uint32_t tmem_acc = tmem_base + (uint32_t)(as * p.acc_stride);
        int cb_i = 0;  // channel block inside the tap
        for (int kb = 0; kb < p.num_kb; ++kb) {
          ptx::mbar_wait(&m.full_bar[s], phase);
          ptx::tc_fence_after();
          if (ti == 0 && kb == 0 && lane == 0) conv_stamp(p, 4);
          const uint32_t a_addr = ptx::smem_u32(m.tiles + (size_t)s * stage_bytes);
          const bool k64 = p.block_k == 64;
          const uint64_t adesc = k64 ? ptx::make_sw128_kmajor_desc(a_addr) : ptx::make_sw64_kmajor_desc(a_addr);
          const uint64_t bdesc = k64 ? ptx::make_sw128_kmajor_desc(a_addr + a_tile_bytes)
                                     : ptx::make_sw64_kmajor_desc(a_addr + a_tile_bytes);
          const int ksteps = (cb_i == p.kb_per_tap - 1) ? p.last_ksteps : p.block_k / 16;
          if (++cb_i == p.kb_per_tap) cb_i = 0;
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              // advance 16 bf16 = 32 B along K inside the swizzle row: +2 in the (addr>>4) field
              if (k < ksteps)
                ptx::umma_bf16_ss(tmem_acc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), p.idesc,
                                  (kb > 0 || k > 0) ? 1u : 0u);
            }
            ptx::umma_commit(&m.empty_bar[s]);  // frees the smem slot when these MMAs retire
            if (kb == p.num_kb - 1) ptx::umma_commit(&m.tmem_full_bar[as]);  // accumulator complete
          }
          __syncwarp();
          if (++s == p.stages) { s = 0; phase ^= 1u; }
        }
        if (lane == 0 && ti < 6) conv_stamp(p, 5 + ti);
        if (++as == ACC_STAGES) { as = 0; aphase ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue: warps 2..5 =====================
    if (p.epi_mode == MC_EPI_PNHWC) {
      if (p.leaky) epilogue_loop<MC_EPI_PNHWC, true, MINB == 1>(p, m, tmem_base, &tmap_out);
      else epilogue_loop<MC_EPI_PNHWC, false, MINB == 1>(p, m, tmem_base, &tmap_out);
    } else if (p.epi_mode == MC_EPI_REORG2) {
      if (p.leaky) epilogue_loop<MC_EPI_REORG2, true>(p, m, tmem_base, &tmap_out);
      else epilogue_loop<MC_EPI_REORG2, false>(p, m, tmem_base, &tmap_out);
    } else if (p.epi_mode == MC_EPI_DECODE) {
      epilogue_loop<MC_EPI_DECODE, false>(p, m, tmem_base, &tmap_out);
    } else {
      if (p.leaky) epilogue_loop<MC_EPI_NCHW_F32, true>(p, m, tmem_base, &tmap_out);
      else epilogue_loop<MC_EPI_NCHW_F32, false>(p, m, tmem_base, &tmap_out);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) conv_stamp(p, 30);
  if (warp_idx == 1) ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// Work items of one cluster of the CTA-pair kernel: whole units first (cluster c: units c, c+G, ... < sk_first), then
// its stream-K span.  Stream-K: the sk_units units of the partial last wave hold sk_total_g K groups; cluster c (of the
// first G' = min(G, 3 * sk_units) clusters) owns groups [c*T/G', (c+1)*T/G') of the unit-major sequence, i.e. the END of
// one unit and / or the START of the next (a span is shorter than a unit, so it touches at most two; a unit is cut into
// at most four pieces).  The START piece runs first and leaves its accumulator in the workspace; the END piece is the
// unit's finisher: it adds the (at most three) earlier pieces and runs the epilogue.  The
// earlier pieces were the FIRST thing their clusters did, so the finisher practically never waits.
struct PairWork {
  int layer;   // entry of the layer table (chained launch; 0 otherwise)
  int unit;    // unit index (m-pair, n-tile) inside the layer
  int g0, g1;  // K groups [g0, g1) of the unit
  int kind;    // 0 whole unit, 1 partial (dump to slot), 2 finisher (add n partials)
  int aux;     // kind 1: slot; kind 2: number of partial pieces to add
};

struct PairWorkIter {
  int next_full, step, sk_first;
  int sk_state;  // 0: stream-K pieces not started, 1: first piece done, 2: finished
  int c, G, gper, T, units;
  __device__ __forceinline__ void init(const ConvKParams& p, int cluster_id, int num_clusters) {
    next_full = cluster_id;
    step = num_clusters;
    sk_first = p.sk_first;
    c = cluster_id; G = p.sk_clusters; gper = p.sk_gper; T = p.sk_total_g; units = p.sk_units;
    sk_state = (p.sk_units > 0 && c < G) ? 0 : 2;
  }
  __device__ __forceinline__ int span_begin(int cl) const { return (int)(((long long)cl * T) / G); }
  __device__ __forceinline__ void describe(int u, int a, int b, PairWork& w) const {  // groups [a,b) of stream-K unit u
    w.unit = sk_first + u;
    w.g0 = a;
    w.g1 = b;
    // first cluster whose span reaches into unit u
    int cf = c;
    while (cf > 0 && span_begin(cf) > u * gper) --cf;
    if (b == gper) {
      w.kind = (a == 0) ? 0 : 2;
      w.aux = c - cf;
    } else {
      w.kind = 1;
      w.aux = c - cf;
    }
  }
  __device__ __forceinline__ bool next(PairWork& w) {
    w.layer = 0;
    if (next_full < sk_first) {
      w.unit = next_full; w.g0 = 0; w.g1 = -1; w.kind = 0; w.aux = 0;  // g1 < 0: the whole K range
      next_full += step;
      return true;
    }
    if (sk_state == 2) return false;
    const int r0 = span_begin(c), r1 = span_begin(c + 1);
    if (r1 <= r0) { sk_state = 2; return false; }
    const int u0 = r0 / gper, u1 = (r1 - 1) / gper;
    if (u0 == u1) {
      sk_state = 2;
      describe(u0, r0 - u0 * gper, r1 - u0 * gper, w);
      return true;
    }
    if (sk_state == 0) {  // the START piece of the later unit first
      sk_state = 1;
      describe(u1, 0, r1 - u1 * gper, w);
      return true;
    }
    sk_state = 2;
    describe(u0, r0 - u0 * gper, gper, w);
    return true;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// Layer table of the CTA-pair kernel.  One entry: today's launch (static schedule above, stream-K tail).  2..4 entries
// (mc_conv_chain_fwd): a chain of 3x3 layers in which layer i+1 reads layer i's output, run as ONE persistent launch so
// that the idle clusters of one layer's partial last wave start the next layer's first units and the layer boundaries
// need no drain / launch / set-up / pipeline fill.  The entries share B, H, W, tile width, ring depth and epilogue.
constexpr int MAX_CHAIN = 4;
constexpr unsigned long long CHAIN_POLL_NS = 1000000000ull;  // bound of one readiness wait (then: status word, go on)
enum { CHAIN_TICKET = 0, CHAIN_DONE = 1, CHAIN_STATUS = 2, CHAIN_COUNTERS = 4 };  // words of the chain workspace

struct PairLayer {
  CUtensorMap tmap_b, tmap_abox, tmap_out;
  ConvKParams p;
  int unit_end;  // tickets [unit_end of the previous entry, unit_end) are this layer's (m-pair, n-tile) units, m-major
  int cnt_off;   // this layer's first readiness counter (one per m-pair) after CHAIN_COUNTERS
};
struct PairParams {
  PairLayer layer[MAX_CHAIN];
  int n_layers;
  unsigned int* chain_ws;  // n_layers >= 2: ticket, clusters done, status, pad, then the readiness counters
};

// Work ring (chained launch): the leader CTA's producer lane claims a ticket, waits until the unit's inputs are
// complete and publishes it into the ring of BOTH CTAs; the peer's producer, the MMA warp and the 8 epilogue warps take
// their units from there (10 arrivals free a slot on the leader's empty barrier).  A ticket < 0 ends the launch.
struct PairRing {
  uint64_t* full;
  uint64_t* empty;
  int* val;
  int slot;
  uint32_t phase;
};

__device__ __forceinline__ void chain_decode(const PairParams& P, int t, PairWork& w) {
  int l = 0;
  while (l + 1 < P.n_layers && t >= P.layer[l].unit_end) ++l;
  w.layer = l;
  w.unit = t - (l > 0 ? P.layer[l - 1].unit_end : 0);
  w.g0 = 0; w.g1 = -1; w.kind = 0; w.aux = 0;
}

__device__ __forceinline__ bool ring_take(const PairParams& P, PairRing& r, PairWork& w, bool whole_warp) {
  ptx::mbar_wait_cluster(&r.full[r.slot], r.phase);
  const int t = *reinterpret_cast<volatile int*>(&r.val[r.slot]);
  if (whole_warp) __syncwarp();  // every lane has read the slot before it is handed back
  if ((threadIdx.x & 31) == 0) ptx::mbar_arrive_leader(&r.empty[r.slot]);
  if (++r.slot == WORK_SLOTS) { r.slot = 0; r.phase ^= 1u; }
  if (t < 0) return false;
  chain_decode(P, t, w);
  return true;
}

// Readiness of a unit of layer l >= 1 at m-pair i: its activation boxes cover rows [256i - Wp - 1, 256i + 264 + Wp) of
// layer l-1's output (3x3 halo around two 128-row tiles), i.e. the m-pairs of layer l-1 over those rows must have all
// n_tiles units stored.  A counter is complete at n_tiles x 8 arrivals (every epilogue warp of both CTAs, per unit).
__device__ __noinline__ void chain_wait_inputs(const PairParams& P, const PairWork& w) {
  const PairLayer& prev = P.layer[w.layer - 1];
  const int mp = w.unit / P.layer[w.layer].p.n_tiles;
  int r0 = 256 * mp - prev.p.Wp - 1, r1 = 256 * mp + 264 + prev.p.Wp;
  if (r0 < 0) r0 = 0;
  if (r1 > prev.p.M_rows) r1 = prev.p.M_rows;
  const unsigned int need = 8u * (unsigned int)prev.p.n_tiles;
  const unsigned int* cnt = P.chain_ws + CHAIN_COUNTERS + prev.cnt_off;
  const unsigned long long t0 = ptx::globaltimer();
  for (int j = r0 / 256; j <= (r1 - 1) / 256; ++j) {
    while (ptx::ld_acquire_gpu(cnt + j) < need) {
      if (ptx::globaltimer() - t0 > CHAIN_POLL_NS) {  // never expected: report it and run on instead of hanging
        atomicExch(P.chain_ws + CHAIN_STATUS, 1u);
        return;
      }
    }
  }
}

// Leader producer: claim the next ticket (increasing, one atomic), wait for its inputs, publish it to both CTAs.
// Deadlock-free: a unit depends only on smaller tickets, tickets are claimed in order and only by running clusters,
// and a cluster's producer claims its next ticket only after issuing every load of its previous one, so the smallest
// unfinished ticket always has complete inputs and a pipeline that drains.
__device__ __forceinline__ bool ring_claim(const PairParams& P, PairRing& r, PairWork& w) {
  ptx::mbar_wait_cluster(&r.empty[r.slot], r.phase ^ 1u);
  int t = (int)atomicAdd(P.chain_ws + CHAIN_TICKET, 1u);
  if (t >= P.layer[P.n_layers - 1].unit_end) {
    t = -1;
  } else {
    chain_decode(P, t, w);
    if (w.layer > 0) chain_wait_inputs(P, w);
    // the inputs were written by TMA stores (async proxy) of other SMs and published by their red.release; our
    // ld.acquire made them visible to this thread's generic proxy, and this fence extends that to the TMA loads this
    // thread issues next (PTX ISA, memory consistency model: proxies — a proxy fence is needed on BOTH sides)
    ptx::fence_proxy_async_global();
  }
  for (uint32_t rk = 0; rk < 2; ++rk) {
    ptx::st_cluster_u32(ptx::mapa_shared(&r.val[r.slot], rk), (uint32_t)t);
    ptx::mbar_arrive_cluster(ptx::mapa_shared(&r.full[r.slot], rk));  // release.cluster: the value above first
  }
  if (++r.slot == WORK_SLOTS) { r.slot = 0; r.phase ^= 1u; }
  return t >= 0;
}

// Writer side of the readiness protocol, per epilogue warp and unit (after the accumulator stage went back): the TMA
// stores of this warp must be COMPLETE (wait_group, not .read), the async-proxy writes are then ordered before the
// generic-proxy release by a proxy fence, and the release-add publishes them at GPU scope.
__device__ __forceinline__ void chain_arrive(const PairParams& P, const PairWork& w, int lane) {
  __threadfence();  // (direct stores of a last chunk narrower than 64 columns, by every lane)
  __syncwarp();
  if (lane == 0) {
    ptx::bulk_wait_group_all();
    ptx::fence_proxy_async_global();
    const PairLayer& L = P.layer[w.layer];
    ptx::red_release_gpu_add(P.chain_ws + CHAIN_COUNTERS + L.cnt_off + w.unit / L.p.n_tiles, 1u);
  }
}

// Epilogue warps of the CTA-pair kernel: one pass per work item, this CTA's 128 rows of the 256-row unit.  Whole units
// and finishers run epilogue_tile (a finisher first waits for the partial accumulators of the unit's earlier K spans and
// adds them there); partial pieces park their raw fp32 accumulator in the workspace and count themselves in.
template <int MODE, bool LEAKY>
__device__ __forceinline__ void epilogue_loop_pair(const PairParams& P, const ConvSmem& m, uint32_t tmem_base,
                                                   int cluster_id, int num_clusters, int pair_rank, PairRing ring) {
  const int lane = threadIdx.x & 31;
  const int quarter = (threadIdx.x >> 5) & 3;
  const ConvKParams& p0 = P.layer[0].p;
  const bool chain = P.n_layers > 1;
  const bool one_n_tile = !chain && p0.n_tiles == 1;
  float* stat_acc = epilogue_begin<MODE>(p0, m, one_n_tile);
  int stat_n0 = -1;
  int slab_buf = 0;
  int as = 0;
  uint32_t aphase = 0;
  PairWorkIter it;
  it.init(p0, cluster_id, num_clusters);
  PairWork w;
  int ti = -1;
  while (chain ? ring_take(P, ring, w, true) : it.next(w)) {
    ++ti;
    const ConvKParams& p = P.layer[w.layer].p;
    const bool vec_ok = ((p.ldc | p.ch_off) & 7) == 0 && (MODE != MC_EPI_REORG2 || (p.N & 7) == 0);
    const int n0 = (w.unit % p.n_tiles) * p.block_n;
    const int m0 = (2 * (w.unit / p.n_tiles) + pair_rank) * BLOCK_M;
    const EpiTile t = epi_tile_begin<MODE>(p, m, tmem_base, one_n_tile, m0, n0, as, aphase, ti);
    const int u_sk = w.unit - p.sk_first;  // (stream-K pieces only)
    // partial tiles are stored [slot][column / 4][256 rows][4 floats]: a warp instruction (32 rows, one float4 each) is one
    // contiguous 512-byte segment, for the writers and for the finisher that reads them back with the same mapping
    const int prow = pair_rank * 128 + quarter * 32 + lane;
    const size_t slot_stride = (size_t)256 * p.block_n;
    float* part_unit = p.sk_part + (size_t)(u_sk < 0 ? 0 : u_sk) * 3 * slot_stride;
    auto part_ptr = [&](int slot, int col) -> float* {  // col multiple of 4
      return part_unit + (size_t)slot * slot_stride + ((size_t)(col >> 2) * 256 + prow) * 4;
    };
    if (w.kind == 1) {
      // partial piece: raw accumulator -> workspace slot, then count this warp in (release)
      for (int c0 = 0; c0 < p.block_n; c0 += 32) {
        uint32_t r0[16], r1[16];
        const bool two = c0 + 16 < p.block_n;
        ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)c0, r0);
        if (two) ptx::tmem_ld_32x32b_x16(t.taddr + (uint32_t)(c0 + 16), r1);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<uint4*>(part_ptr(w.aux, c0 + 4 * q)) = make_uint4(r0[4 * q], r0[4 * q + 1], r0[4 * q + 2], r0[4 * q + 3]);
        if (two) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(part_ptr(w.aux, c0 + 16 + 4 * q)) = make_uint4(r1[4 * q], r1[4 * q + 1], r1[4 * q + 2], r1[4 * q + 3]);
        }
      }
      ptx::tc_fence_before();
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        atomicAdd(p.sk_count + u_sk, 1u);
        ptx::mbar_arrive_leader(&m.tmem_empty_bar[as]);
      }
    } else {
      const int nparts = w.kind == 2 ? w.aux : 0;
      if (nparts > 0) {
        // the earlier K spans of this unit were the first thing their clusters computed: normally long finished
        if (lane == 0) {
          const unsigned int want = 8u * (unsigned int)nparts;
          unsigned int spins = 0;
          while (*reinterpret_cast<volatile unsigned int*>(p.sk_count + u_sk) < want) {
            if (++spins > (1u << 24)) __trap();
          }
          // every writer has arrived and all 8 finisher warps must see that: the LAST finisher warp to get here puts the
          // counter back to zero (second counter = finisher warps done), so the workspace needs no per-launch memset
          if (atomicAdd(p.sk_count + 256 + u_sk, 1u) == 7u) {
            p.sk_count[256 + u_sk] = 0u;
            p.sk_count[u_sk] = 0u;
          }
        }
        __syncwarp();
        __threadfence();
      }
      epilogue_tile<MODE, LEAKY, true, true>(p, &P.layer[w.layer].tmap_out, m, t, vec_ok, &m.tmem_empty_bar[as],
                                             slab_buf, stat_acc, stat_n0, [&](uint32_t (&r)[16], int col) {
        for (int s2 = 0; s2 < nparts; ++s2) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 a = __ldcg(reinterpret_cast<const float4*>(part_ptr(s2, col + 4 * q)));
            r[4 * q] = __float_as_uint(__uint_as_float(r[4 * q]) + a.x);
            r[4 * q + 1] = __float_as_uint(__uint_as_float(r[4 * q + 1]) + a.y);
            r[4 * q + 2] = __float_as_uint(__uint_as_float(r[4 * q + 2]) + a.z);
            r[4 * q + 3] = __float_as_uint(__uint_as_float(r[4 * q + 3]) + a.w);
          }
        }
      });
      if (chain) chain_arrive(P, w, lane);
    }
    if (threadIdx.x == 64 && ti < 8) conv_stamp(p, 13 + 2 * ti);
    if (++as == ACC_STAGES) { as = 0; aphase ^= 1u; }
  }
  epilogue_end<MODE>(p0, stat_acc, stat_n0);
}

// ---------------------------------------------------------------------------------------------------------------
// CTA-pair variant for the wide 3x3 layers (tcgen05 cta_group::2): two CTAs on the two SMs of a TPC compute a
// 256 x block_n tile together.  Each CTA loads its own 128-row activation boxes but only HALF of every weight tile
// (block_n/2 rows); the tensor cores of both SMs read both halves.  Why: the single-CTA kernel is bound by the
// chip-wide L2 -> shared-memory TMA rate (measured ~50 B/clk/SM; a 128x256 tile needs 5.7 KB of A + 32 KB of B per
// 512 MMA cycles = 74 B/clk) — halving B per SM (5.7 + 16 KB -> 42 B/clk) puts the layer back under the tensor pipe.
// Barriers: TMA of both CTAs counts bytes on the LEADER's full barriers (only the leader issues MMAs); MMA completion
// is multicast to the empty / accumulator-full barriers of both CTAs; the epilogues of both CTAs hand the
// accumulator stage back on the leader's barrier (8 arrivals).
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_gemm_tcgen05_pair_kernel(const __grid_constant__ PairParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // every entry of the layer table shares the fields read here (tile width, ring depths, epilogue slabs)
  const ConvKParams& p0 = P.layer[0].p;
  const bool chain = P.n_layers > 1;
  const uint32_t b_half_bytes = (uint32_t)(p0.block_n / 2 * 128);
  const ConvSmem m = carve_smem<true>(smem_raw, p0, A_BOX_STRIDE, b_half_bytes, 0);
  PairRing ring;
  ring.full = m.work_full;
  ring.empty = m.work_empty;
  ring.val = m.work_val;
  ring.slot = 0;
  ring.phase = 0;

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = (int)ptx::cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  if (threadIdx.x == 0) {
    conv_stamp(p0, 0);
    for (int l = 0; l < P.n_layers; ++l) {
      ptx::prefetch_tensormap(&P.layer[l].tmap_b);
      ptx::prefetch_tensormap(&P.layer[l].tmap_abox);
      if (p0.tma_bufs > 0) ptx::prefetch_tensormap(&P.layer[l].tmap_out);
    }
  }
  const uint32_t tmem_base = block_setup<true>(m, p0);
  if (threadIdx.x == 0) conv_stamp(p0, 1);

  if (warp_idx == 0) {
    // ===================== TMA producer (one thread per CTA) =====================
    if (lane == 0) {
      Pipe pp(p0.stages, p0.a_stages);
      PairWorkIter it;
      it.init(p0, cluster_id, num_clusters);
      PairWork w;
      while (!chain ? it.next(w) : (rank == 0 ? ring_claim(P, ring, w) : ring_take(P, ring, w, false))) {
        const PairLayer& L = P.layer[w.layer];
        const ConvKParams& p = L.p;
        // (chain, peer CTA) the leader acquired this unit's inputs; the mbarrier hand-over carries that to this
        // thread, and the proxy fence to the TMA loads it issues (see ring_claim)
        if (chain && rank != 0) ptx::fence_proxy_async_global();
        const int n0 = (w.unit % p.n_tiles) * p.block_n + rank * (p.block_n / 2);
        const int m0 = (2 * (w.unit / p.n_tiles) + rank) * BLOCK_M;
        produce_box_groups<true>(p, m, &L.tmap_abox, &L.tmap_b, m0, n0, w.g0, w.g1 < 0 ? 3 * p.kb_per_tap : w.g1,
                                 A_BOX_STRIDE, A_BOX_BYTES, b_half_bytes, rank == 0, pp);
      }
      conv_stamp(p0, 3);
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer (warp 1 of the leader CTA; one elected lane issues) =====================
    if (rank == 0) {
      Pipe pp(p0.stages, p0.a_stages);
      PairWorkIter it;
      it.init(p0, cluster_id, num_clusters);
      PairWork w;
      int ti = -1;
      while (chain ? ring_take(P, ring, w, true) : it.next(w)) {
        ++ti;
        const ConvKParams& p = P.layer[w.layer].p;
        mma_box_unit<true>(p, m, tmem_base, w.g0, w.g1 < 0 ? 3 * p.kb_per_tap : w.g1, A_BOX_STRIDE, b_half_bytes, pp, ti);
      }
    }
  } else {
    // ===================== epilogue: warps 2..5 of both CTAs =====================
    if (p0.epi_mode == MC_EPI_PNHWC) {
      if (p0.leaky) epilogue_loop_pair<MC_EPI_PNHWC, true>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
      else epilogue_loop_pair<MC_EPI_PNHWC, false>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
    } else if (p0.epi_mode == MC_EPI_REORG2) {
      if (p0.leaky) epilogue_loop_pair<MC_EPI_REORG2, true>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
      else epilogue_loop_pair<MC_EPI_REORG2, false>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
    } else {
      if (p0.leaky) epilogue_loop_pair<MC_EPI_NCHW_F32, true>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
      else epilogue_loop_pair<MC_EPI_NCHW_F32, false>(P, m, tmem_base, cluster_id, num_clusters, rank, ring);
    }
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // the peer may still read this CTA's smem / signal its barriers until both are done
  if (warp_idx == 1) ptx::tmem_dealloc_pair(tmem_base, (uint32_t)p0.tmem_cols);
  if (threadIdx.x == 0) conv_stamp(p0, 30);
  if (chain && rank == 0 && threadIdx.x == 0) {
    // every unit of this cluster is stored and counted (cluster barrier above).  The LAST cluster out puts the tickets
    // and counters back to zero, so every launch leaves the workspace as it found it (graph replays need no memset)
    __threadfence();
    if (atomicAdd(P.chain_ws + CHAIN_DONE, 1u) == (unsigned int)num_clusters - 1u) {
      __threadfence();
      const PairLayer& last = P.layer[P.n_layers - 1];
      const int n_cnt = last.cnt_off + (last.p.m_tiles + 1) / 2;
      for (int i = 0; i < n_cnt; ++i) P.chain_ws[CHAIN_COUNTERS + i] = 0u;
      P.chain_ws[CHAIN_TICKET] = 0u;
      P.chain_ws[CHAIN_DONE] = 0u;
    }
  }
}

// Tile-width heuristic.  One 64-wide k-block of a 128 x bn tile costs max(2*bn, 128+bn) SM cycles: 2*bn is the
// tcgen05 issue floor (128*bn*64 MACs at 4096 MAC/clk), 128+bn is the shared-memory read of the A (16 KB) and
// B (bn*128 B) tiles at 128 B/clk.  Cost = waves over the SMs x (k-blocks x that + a fixed prologue/epilogue).
int pick_block_n(int Npad, int m_tiles, int num_kb, int num_sms, bool share_dx) {
  int best = 16;
  double best_cost = 1e30;
  for (int bn = 16; bn <= 256; bn += 16) {  // every legal UMMA N for M=128
    const int n_tiles = (Npad + bn - 1) / bn;
    const long long tiles = (long long)n_tiles * m_tiles;
    const long long rounds = (tiles + num_sms - 1) / num_sms;  // persistent CTAs: tiles per CTA
    // per 64-wide k-block: tcgen05 issue floor 2*bn cycles; smem operand read (16 KB + bn*128 B at 128 B/clk);
    // operand FEED from L2 through TMA, measured on B200 at ~13.3 cycles per KB per SM when all SMs stream
    // (128x256 tiles run at ~80% tensor-active = 640 cycles per k-block for 48 KB)
    double per_kb = 2.0 * bn;
    if (128.0 + bn > per_kb) per_kb = 128.0 + bn;
    // (with the shared activation box a tap's k-block brings 17/3 KB of A instead of 16 KB)
    const double feed = 13.3 * ((share_dx ? 17.0 / 3.0 : 16.0) + bn / 8.0);
    if (feed > per_kb) per_kb = feed;
    // one epilogue (~12 cycles per column) is exposed at the end; the others overlap the next tile's MMAs unless
    // they are longer than the mainloop
    const double main = per_kb * num_kb, epi = 12.0 * bn + 400.0;
    const double cost = (double)rounds * (main > epi ? main : epi) + epi + 2500.0;
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best = bn;
    }
  }
  return best;
}

}  // namespace

static thread_local int g_last_plan[8] = {0, 0, 0, 0, 0, 0, 0, 0};
static unsigned long long* g_conv_dbg = nullptr;

// Debug: timeline stamps of the conv GEMM kernels (32 x uint64 per CTA, globaltimer ns) into d_buf, which must hold
// 32 * 8 * grid bytes; NULL switches tracing off again.  tools/trace_conv.py and tools/trace_chain.py print the timelines.
extern "C" int mc_debug_conv_trace(void* d_buf) {
  g_conv_dbg = reinterpret_cast<unsigned long long*>(d_buf);
  return 0;
}

extern "C" int mc_conv_last_plan(int info[8]) {
  MC_CHECK_ARG(info != nullptr, "mc_conv_last_plan: null pointer");
  for (int i = 0; i < 8; ++i) info[i] = g_last_plan[i];
  return 0;
}

// Workspace the stream-K tail of the CTA-pair kernel can use for this layer (0: the layer never takes that path).  Upper
// bound over every tile width the planner may pick: up to 148/2 stream-K units x 3 partial slots x 256 rows x 256 columns
// of fp32, plus 2 KB of counters.  The counters must be ZERO before the first launch; every launch leaves them zero.
extern "C" size_t mc_workspace_bytes_conv_fwd(const mc_conv_desc* d) {
  if (d == nullptr || d->ksize != 3 || d->Cin <= 32 || d->Npad < 192) return 0;
  const int clusters = mc_num_sms() / 2;
  return (size_t)2048 + (size_t)clusters * 3 * 256 * 256 * sizeof(float);
}

// Clusters of the CTA-pair kernel that fit on the device at once (queried once)
static int pair_max_clusters(int* out) {
  static int max_clusters = -1;
  if (max_clusters < 0) {
    MC_CUDA(cudaFuncSetAttribute(conv_gemm_tcgen05_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * (mc_num_sms() / 2));
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = 222 * 1024;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, conv_gemm_tcgen05_pair_kernel, &cfg) != cudaSuccess || n < 1) {
      cudaGetLastError();
      n = mc_num_sms() / 2;
    }
    max_clusters = n;
  }
  *out = max_clusters;
  return 0;
}

// Everything mc_conv_fwd decides for one layer: kernel (CTA pair or single CTA), tile width, ring depth, CTAs per SM,
// stream-K tail, tensor maps and kernel parameters.  mc_conv_chain_fwd plans its members with the same function, so a
// chained layer computes exactly what its own mc_conv_fwd launch would.
struct ConvPlan {
  bool use_pair;
  int ctas;        // single-CTA kernel: resident CTAs per SM
  int grid;        // CTAs
  int units;       // CTA pair: (m-pair, n-tile) units
  size_t smem_bytes;
  CUtensorMap tm_a, tm_b, tm_abox, tm_out;
  ConvKParams p;
};

static int conv_plan(const mc_conv_desc* d, ConvPlan* L) {
  MC_CHECK_ARG(d != nullptr, "mc_conv_fwd: null descriptor");
  MC_CHECK_ARG(d->d_in && d->d_wpack && d->d_scale && d->d_shift && (d->d_out || d->epi_mode == MC_EPI_DECODE),
               "mc_conv_fwd: null pointer");
  MC_CHECK_ARG(d->ksize == 1 || d->ksize == 3, "mc_conv_fwd: ksize must be 1 or 3 (got %d)", d->ksize);
  MC_CHECK_ARG(d->B > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->N > 0, "mc_conv_fwd: bad dims");
  MC_CHECK_ARG((d->Cin_ld % 8) == 0 && d->Cin <= d->Cin_ld, "mc_conv_fwd: Cin_ld must be a multiple of 8 >= Cin");
  MC_CHECK_ARG((d->Npad % 16) == 0 && d->Npad >= d->N, "mc_conv_fwd: Npad must be a multiple of 16 >= N");
  MC_CHECK_ARG(((uintptr_t)d->d_in & 15) == 0 && ((uintptr_t)d->d_wpack & 15) == 0 && ((uintptr_t)d->d_out & 15) == 0,
               "mc_conv_fwd: pointers must be 16-byte aligned");
  MC_CHECK_ARG(d->epi_mode == MC_EPI_PNHWC || d->epi_mode == MC_EPI_REORG2 || d->epi_mode == MC_EPI_NCHW_F32 ||
                   d->epi_mode == MC_EPI_DECODE,
               "mc_conv_fwd: unsupported epilogue mode %d", d->epi_mode);
  const bool decode = d->epi_mode == MC_EPI_DECODE;
  if (decode) {
    const mc_decode_params* q = d->decode;
    MC_CHECK_ARG(q != nullptr && q->d_boxes != nullptr, "mc_conv_fwd: MC_EPI_DECODE needs decode parameters with d_boxes");
    MC_CHECK_ARG(q->A > 0 && q->A <= MC_MAX_ANCHORS && q->nc > 0 && q->A * (5 + q->nc) == d->N,
                 "mc_conv_fwd: decode needs N == A*(5+nc) (N %d, A %d, nc %d)", d->N, q->A, q->nc);
    MC_CHECK_ARG(d->Npad <= 256 && d->leaky == 0, "mc_conv_fwd: decode needs a linear head of <= 256 channels");
    MC_CHECK_ARG(((uintptr_t)q->d_boxes & 15) == 0, "mc_conv_fwd: d_boxes must be 16-byte aligned");
  }
  if (d->epi_mode == MC_EPI_REORG2) MC_CHECK_ARG((d->H % 2) == 0 && (d->W % 2) == 0, "mc_conv_fwd: reorg needs even H,W");

  const int ntaps = d->ksize * d->ksize;
  const int BLOCK_K = d->block_k == 32 ? 32 : 64;
  MC_CHECK_ARG(d->block_k == 0 || d->block_k == 32 || d->block_k == 64, "mc_conv_fwd: block_k must be 0, 32 or 64");
  const int A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;
  const int Kc = ((d->Cin + BLOCK_K - 1) / BLOCK_K) * BLOCK_K;
  const long long M_rows = (long long)d->B * (d->H + 1) * (d->W + 1);
  MC_CHECK_ARG(M_rows < (1ll << 31), "mc_conv_fwd: too many rows");
  const int m_tiles = (int)((M_rows + BLOCK_M - 1) / BLOCK_M);

  // 3x3 with 64-wide k-blocks: share one activation box among the three dx taps.
  // 32-wide k-blocks share the box only on long, feed-bound launches (dense conv2: 21,841 tiles, 306 -> 262 us); short
  // ones lose a little to the two-ring pipeline (shrunk conv13, 365 tiles: 18 -> 21 us)
  const int share_dx = (d->ksize == 3 && (BLOCK_K == 64 || m_tiles >= 2048)) ? 1 : 0;
  const int a_box_stride = BLOCK_K == 64 ? A_BOX_STRIDE : A_BOX_STRIDE / 2;
  int block_n = d->block_n;
  // (the operand-feed term keeps the un-shared 16 KB A tile: with the shared-box figure the model picks narrower tiles
  //  that measured 4 % slower end to end on B200)
  if (decode) block_n = d->Npad;  // every logit of a cell in ONE accumulator row
  if (block_n <= 0) block_n = pick_block_n(d->Npad, m_tiles, (ntaps * Kc + 63) / 64, mc_num_sms(), false);  // 64-wide k-block units
  const bool want_stats = d->d_stat_sum != nullptr || d->d_stat_sumsq != nullptr;
  if (want_stats) {
    // batch statistics come from the TMA-store slabs: every column of a tile must leave in a whole 64-column chunk
    MC_CHECK_ARG(d->d_stat_sum != nullptr && d->d_stat_sumsq != nullptr, "mc_conv_fwd: d_stat_sum and d_stat_sumsq go together");
    MC_CHECK_ARG(d->epi_mode == MC_EPI_PNHWC && ((d->ldc | d->ch_off) & 7) == 0 && d->N >= 33,
                 "mc_conv_fwd: statistics need the PNHWC epilogue, 8-aligned pitch / offset and more than 32 channels");
    block_n = (block_n + 63) / 64 * 64;
    if (block_n > 256) block_n = 256;
  }
  MC_CHECK_ARG(block_n >= 16 && block_n <= 256 && (block_n % 16) == 0, "mc_conv_fwd: block_n %d invalid", block_n);
  const int n_tiles = (d->Npad + block_n - 1) / block_n;

  const int stage_bytes = A_TILE_BYTES + block_n * BLOCK_K * 2;
  const long long total_tiles = (long long)n_tiles * m_tiles;
  const int acc_stride = block_n == 16 ? 16 : ((block_n + 31) / 32) * 32;
  int tmem_cols = 32;
  while (tmem_cols < ACC_STAGES * acc_stride) tmem_cols <<= 1;
  const int num_kb = ntaps * (Kc / BLOCK_K);
  constexpr size_t AUX_BYTES = 5120 + 1024;  // barriers (512), scale/shift staging (4096), pad to 1 KB; 1024-byte alignment slack

  // TMA-store epilogue (tiles >= 64 wide): whole 64-column chunks leave as bulk tensor stores from 4 KB slabs per
  // epilogue warp — two slabs per warp when the CTA has the SM to itself, one (16 KB per CTA) when several CTAs share
  // it (measured: dense conv4/conv6 at 104x104 run 113 us with 2 CTAs per SM + one slab, 158 us with one CTA + two
  // slabs, 125 us with the staged epilogue).
  const bool tma_out = d->epi_mode == MC_EPI_PNHWC && block_n >= 64 && ((d->ldc | d->ch_off) & 7) == 0;
  auto tma_bufs_for = [&](int ctas_) -> int { return tma_out ? (ctas_ == 1 ? 2 : 1) : 0; };
  // staged epilogue (the aligned PNHWC tiles the TMA stores do not take: 32 and 48 wide): 128 rows x (block_n bf16 +
  // 16 B) of shared memory (measured: dense conv2 396 -> 300 us; 16-wide rows are two stores either way)
  const bool stage_out = !tma_out && d->epi_mode == MC_EPI_PNHWC && block_n >= 32 && ((d->ldc | d->ch_off) & 7) == 0;
  const int out_pitch = stage_out ? block_n * 2 + 16 : 0;
  // (decode epilogue: 128 rows x (block_n + 1) floats of logits)
  auto out_stage_for = [&](int ctas_) -> size_t {
    return decode ? (size_t)128 * (block_n + 1) * 4
                  : (tma_out ? (size_t)tma_bufs_for(ctas_) * 4 * 4096 + (want_stats ? 4 * 512 * sizeof(float) : 0)
                             : (size_t)128 * out_pitch);
  };
  // smem ring of one CTA when `ctas` CTAs share an SM (each CTA also costs 1 KB of reserved shared memory)
  auto plan_ring = [&](int ctas, int* st, int* ast, size_t* bytes) -> bool {
    const size_t out_stage_bytes = out_stage_for(ctas);
    const long long cap = (ctas == 1 ? 220 * 1024 - (long long)AUX_BYTES : (227 * 1024) / ctas - 1024 - (long long)AUX_BYTES) - (long long)out_stage_bytes;
    if (share_dx) {
      const int b_bytes = block_n * BLOCK_K * 2;
      int a = ctas == 1 ? MAX_A_STAGES : 2;
      long long stg = (cap - (long long)a * a_box_stride) / b_bytes;
      if (stg > MAX_STAGES) stg = MAX_STAGES;
      if (stg < 3) return false;
      *st = (int)stg; *ast = a;
      *bytes = (size_t)a * a_box_stride + (size_t)stg * b_bytes + AUX_BYTES + out_stage_bytes;
    } else {
      long long stg = cap / stage_bytes;
      if (stg > MAX_STAGES) stg = MAX_STAGES;
      if (stg > num_kb * 4) stg = num_kb * 4;  // a ring deeper than four tiles' worth of k-blocks buys nothing
      if (stg < (ctas == 1 ? 1 : 3)) return false;
      *st = (int)stg; *ast = 0;
      *bytes = (size_t)stg * stage_bytes + AUX_BYTES + out_stage_bytes;
    }
    return true;
  };
  // CTAs per SM.  Wide, long-K tiles are tensor-bound: one CTA with the deepest ring.  Narrow layers are bound by the
  // per-tile latency chain, which only more CTAs (or tiles) in flight hide: up to 3 when the rings and the TMEM
  // slices fit and every CTA still gets at least one tile (measured: one beats two by 0.5 % on the shrunk step, the
  // 365-tile 26x26 layers get 2 CTAs per SM).
  int ctas = 1;
  {
    const double main_cycles = (double)num_kb * (BLOCK_K / 64.0) * (2.0 * block_n > 128.0 + block_n ? 2.0 * block_n : 128.0 + block_n);
    const bool narrow = main_cycles < 6000.0;
    for (int c = 3; c >= 2 && narrow; --c) {
      int st, ast;
      size_t bytes;
      if (c * tmem_cols > 512 || total_tiles < (long long)c * mc_num_sms() || !plan_ring(c, &st, &ast, &bytes)) continue;
      ctas = c;
      break;
    }
  }
  int stages = d->stages;
  int a_stages = 0;
  size_t smem_bytes;
  if (stages <= 0) {
    MC_CHECK_ARG(plan_ring(ctas, &stages, &a_stages, &smem_bytes), "mc_conv_fwd: no shared-memory ring fits block_n %d", block_n);
  } else {
    ctas = 1;
    if (share_dx) {
      a_stages = MAX_A_STAGES;
      MC_CHECK_ARG(stages >= 2 && stages <= MAX_STAGES, "mc_conv_fwd: stages %d invalid", stages);
      smem_bytes = (size_t)a_stages * a_box_stride + (size_t)stages * block_n * BLOCK_K * 2 + AUX_BYTES + out_stage_for(1);
    } else {
      MC_CHECK_ARG(stages >= 1 && stages <= MAX_STAGES, "mc_conv_fwd: stages %d invalid", stages);
      smem_bytes = (size_t)stages * stage_bytes + AUX_BYTES + out_stage_for(1);
    }
  }
  MC_CHECK_ARG(smem_bytes <= 227 * 1024, "mc_conv_fwd: smem %zu too large", smem_bytes);

  // CTA pair (cta_group::2) for the wide 3x3 layers
  const bool pair_legal = share_dx && BLOCK_K == 64 && d->stages <= 0 && (block_n % 16) == 0 && block_n >= 64 && m_tiles >= 2;
  const bool use_pair = !decode && pair_legal && block_n >= 192 && num_kb >= 36;
  if (use_pair) {
    ctas = 1;
    a_stages = MAX_A_STAGES;
    const int b_half = block_n / 2 * 128;
    const int slab_bytes = tma_bufs_for(1) * 4 * 4096 + (want_stats ? 4 * 512 * (int)sizeof(float) : 0);
    stages = (220 * 1024 - a_stages * A_BOX_STRIDE - slab_bytes) / b_half;
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    smem_bytes = (size_t)a_stages * A_BOX_STRIDE + (size_t)stages * b_half + AUX_BYTES + slab_bytes;
  }

  CUtensorMap tm_a, tm_b, tm_abox;
  MC_CHECK_ARG(d->in_cols == 0 || (d->in_cols >= d->Cin && d->in_cols <= d->Cin_ld), "mc_conv_fwd: in_cols %d outside [Cin, Cin_ld]", d->in_cols);
  const uint64_t in_cols = d->in_cols ? (uint64_t)d->in_cols : (uint64_t)d->Cin;
  int rc = mc_make_tmap_2d_bf16_k(&tm_a, d->d_in, (uint64_t)M_rows, in_cols, (uint64_t)d->Cin_ld, BLOCK_M, BLOCK_K);
  if (rc) return rc;
  tm_abox = tm_a;
  if (share_dx) {
    rc = mc_make_tmap_2d_bf16_k(&tm_abox, d->d_in, (uint64_t)M_rows, in_cols, (uint64_t)d->Cin_ld, A_BOX_ROWS, BLOCK_K);
    if (rc) return rc;
  }
  // weights: [n_tiles*block_n >= Npad rows (OOB rows zero-filled), ntaps*Kc]
  rc = mc_make_tmap_2d_bf16_k(&tm_b, d->d_wpack, (uint64_t)d->Npad, (uint64_t)ntaps * Kc, (uint64_t)ntaps * Kc,
                              (uint32_t)(use_pair ? block_n / 2 : block_n), BLOCK_K);
  if (rc) return rc;

  CUtensorMap tm_out = tm_a;
  const int tma_bufs = tma_bufs_for(use_pair ? 1 : ctas);
  if (tma_bufs) {
    // output slice [ch_off, ch_off + N rounded up to 8) of the PNHWC rows: stores are clipped there, so a chunk that
    // reaches past the layer's channels never touches the neighbouring concat slice; channels N .. 8-multiple get zeros
    uint64_t ocols = (uint64_t)((d->N + 7) / 8 * 8);
    if (ocols > (uint64_t)(d->ldc - d->ch_off)) ocols = (uint64_t)(d->ldc - d->ch_off);
    rc = mc_make_tmap_2d_bf16_k(&tm_out, reinterpret_cast<const __nv_bfloat16*>(d->d_out) + d->ch_off, (uint64_t)M_rows, ocols,
                                (uint64_t)d->ldc, 32, 64);
    if (rc) return rc;
  }

  ConvKParams p;
  p.M_rows = (int)M_rows;
  p.N = d->N;
  p.Npad = d->Npad;
  p.kb_per_tap = Kc / BLOCK_K;
  p.block_k = BLOCK_K;
  p.num_kb = ntaps * p.kb_per_tap;
  p.ksize = d->ksize;
  p.W = d->W;
  p.H = d->H;
  p.Wp = d->W + 1;
  p.Hp = d->H + 1;
  p.block_n = block_n;
  p.stages = stages;
  p.share_dx = share_dx;
  {
    const int rem = d->Cin - (Kc / BLOCK_K - 1) * BLOCK_K;  // channels in the last channel block of a tap
    p.last_ksteps = (rem + 15) / 16;
  }
  p.a_stages = a_stages;
  p.out_pitch = use_pair ? 0 : out_pitch;
  p.out_chunk = block_n;
  p.tma_bufs = tma_bufs;
  p.stat_sum = d->d_stat_sum;
  p.stat_sumsq = d->d_stat_sumsq;
  {
    auto magic = [](unsigned int dv, unsigned int* mul, unsigned int* shr) {
      unsigned int l = 0;
      while ((1u << l) < dv) ++l;
      const unsigned long long pw = 31ull + l;
      *mul = (unsigned int)((((unsigned long long)1 << pw) + dv - 1) / dv);
      *shr = (unsigned int)(pw - 32);
    };
    magic((unsigned int)(d->W + 1), &p.wp_mul, &p.wp_shr);
    magic((unsigned int)(d->H + 1), &p.hp_mul, &p.hp_shr);
  }
  p.acc_stride = acc_stride;
  p.tmem_cols = tmem_cols;
  p.m_tiles = m_tiles;
  p.n_tiles = n_tiles;
  p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(block_n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
  p.scale = d->d_scale;
  p.shift = d->d_shift;
  p.out = d->d_out;
  p.ldc = d->ldc;
  p.ch_off = d->ch_off;
  p.epi_mode = d->epi_mode;
  p.leaky = d->leaky;
  p.sk_first = 0; p.sk_units = 0; p.sk_gper = 0; p.sk_total_g = 0; p.sk_clusters = 0; p.sk_count = nullptr; p.sk_part = nullptr;
  p.dbg = g_conv_dbg;
  p.dec_boxes = p.dec_cls = p.dec_head = nullptr;
  p.dec_A = p.dec_nc = p.dec_only_obj = 0;
  p.dec_thresh = 0.f;
  if (decode) {
    const mc_decode_params* q = d->decode;
    p.dec_boxes = q->d_boxes;
    p.dec_cls = q->d_cls;
    p.dec_head = q->d_head;
    p.dec_A = q->A;
    p.dec_nc = q->nc;
    p.dec_only_obj = q->only_objectness;
    p.dec_thresh = q->conf_thresh;
    for (int a = 0; a < MC_MAX_ANCHORS; ++a) {
      p.dec_anc.w[a] = a < q->A ? q->anchors[2 * a] : 0.f;
      p.dec_anc.h[a] = a < q->A ? q->anchors[2 * a + 1] : 0.f;
    }
  }

  if (use_pair) {
    p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(block_n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
    p.acc_stride = ((block_n + 31) / 32) * 32;
    p.tmem_cols = 32;
    while (p.tmem_cols < ACC_STAGES * p.acc_stride) p.tmem_cols <<= 1;
    int max_clusters = 0;
    int rc2 = pair_max_clusters(&max_clusters);
    if (rc2) return rc2;
    const int m_pairs = (m_tiles + 1) / 2;
    const long long units = (long long)m_pairs * n_tiles;
    const int clusters = (int)(units < max_clusters ? units : max_clusters);
    // Stream-K for a SHORT partial last wave (at most half a wave of units left over, e.g. batch 32: 100 units over 74
    // clusters — without it the 26 left-over units cost a whole second round).  Measured on B200 for the bench shapes
    // (196 units = 2.65 waves): no gain, 0.8556 vs 0.8584 ms per step — the 48 clusters of a two-thirds-full last wave
    // run their units faster because the operand feed from L2 is shared by fewer SMs, so whole tiles are kept there.
    // Needs the caller's workspace.
    p.sk_first = (int)units;
    p.sk_units = 0;
    p.sk_gper = 3 * p.kb_per_tap;
    p.sk_total_g = 0;
    p.sk_clusters = 0;
    p.sk_count = nullptr;
    p.sk_part = nullptr;
    {
      const long long full = units / clusters, rem = units % clusters;
      const size_t need = mc_workspace_bytes_conv_fwd(d);
      if (full >= 1 && rem > 0 && rem * 2 <= (long long)clusters && d->d_ws != nullptr && need > 0 &&
          d->ws_bytes >= need && ((uintptr_t)d->d_ws & 255) == 0) {
        p.sk_first = (int)(full * clusters);
        p.sk_units = (int)rem;
        p.sk_total_g = (int)rem * p.sk_gper;
        p.sk_clusters = (int)(3 * rem < clusters ? 3 * rem : clusters);
        p.sk_count = reinterpret_cast<unsigned int*>(d->d_ws);  // [256] writer arrivals, [256] finisher warps done
        p.sk_part = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(d->d_ws) + 2048);
      }
    }
    L->use_pair = true;
    L->ctas = 1;
    L->grid = 2 * clusters;
    L->units = (int)units;
  } else {
    const long long max_ctas = (long long)mc_num_sms() * ctas;
    L->use_pair = false;
    L->ctas = ctas;
    L->grid = (int)(total_tiles < max_ctas ? total_tiles : max_ctas);
    L->units = 0;
  }
  L->smem_bytes = smem_bytes;
  L->tm_a = tm_a; L->tm_b = tm_b; L->tm_abox = tm_abox; L->tm_out = tm_out;
  L->p = p;
  return 0;
}

// one layer of the CTA-pair kernel's table from its plan
static void pair_layer(const ConvPlan& L, PairLayer* e) {
  e->tmap_b = L.tm_b;
  e->tmap_abox = L.tm_abox;
  e->tmap_out = L.tm_out;
  e->p = L.p;
  e->unit_end = L.units;
  e->cnt_off = 0;
}

extern "C" int mc_conv_fwd(const mc_conv_desc* d, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ConvPlan L;
  int rc = conv_plan(d, &L);
  if (rc) return rc;
  const ConvKParams& p = L.p;
  if (L.use_pair) {
    g_last_plan[0] = 1; g_last_plan[1] = p.block_n; g_last_plan[2] = 1; g_last_plan[3] = p.sk_units; g_last_plan[4] = 1;
    g_last_plan[5] = p.stages; g_last_plan[6] = L.grid; g_last_plan[7] = p.block_k;
    PairParams P;
    memset(&P, 0, sizeof(P));
    pair_layer(L, &P.layer[0]);
    P.n_layers = 1;
    P.chain_ws = nullptr;
    conv_gemm_tcgen05_pair_kernel<<<L.grid, NUM_THREADS, L.smem_bytes, stream>>>(P);
    MC_LAUNCH_CHECK("conv_gemm_tcgen05_pair_kernel");
    return 0;
  }

  static bool attr_set = false;
  if (!attr_set) {
    MC_CUDA(cudaFuncSetAttribute(conv_gemm_tcgen05_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    MC_CUDA(cudaFuncSetAttribute(conv_gemm_tcgen05_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024));
    MC_CUDA(cudaFuncSetAttribute(conv_gemm_tcgen05_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    attr_set = true;
  }
  g_last_plan[0] = 0; g_last_plan[1] = p.block_n; g_last_plan[2] = L.ctas; g_last_plan[3] = 0;
  g_last_plan[4] = p.share_dx; g_last_plan[5] = p.stages; g_last_plan[6] = L.grid; g_last_plan[7] = p.block_k;
  if (L.ctas >= 3)
    conv_gemm_tcgen05_kernel<3><<<L.grid, NUM_THREADS, L.smem_bytes, stream>>>(L.tm_a, L.tm_b, L.tm_abox, L.tm_out, p);
  else if (L.ctas == 2)
    conv_gemm_tcgen05_kernel<2><<<L.grid, NUM_THREADS, L.smem_bytes, stream>>>(L.tm_a, L.tm_b, L.tm_abox, L.tm_out, p);
  else
    conv_gemm_tcgen05_kernel<1><<<L.grid, NUM_THREADS, L.smem_bytes, stream>>>(L.tm_a, L.tm_b, L.tm_abox, L.tm_out, p);
  MC_LAUNCH_CHECK("conv_gemm_tcgen05_kernel");
  return 0;
}

extern "C" int mc_conv_fwd_plan(const mc_conv_desc* d, int info[16]) {
  MC_CHECK_ARG(info != nullptr, "mc_conv_fwd_plan: null pointer");
  ConvPlan L;
  const int rc = conv_plan(d, &L);
  if (rc) return rc;
  const ConvKParams& p = L.p;
  const bool pnhwc = p.epi_mode == MC_EPI_PNHWC;
  info[0] = L.use_pair ? 1 : 0;
  info[1] = L.ctas;
  info[2] = p.block_n;
  info[3] = p.block_k;
  info[4] = p.stages;
  info[5] = p.a_stages;
  info[6] = p.share_dx;
  info[7] = L.grid;
  info[8] = p.m_tiles;
  info[9] = p.n_tiles;
  info[10] = p.sk_units;
  info[11] = p.tma_bufs > 0 ? 2 : (p.out_pitch > 0 ? 1 : 0);
  info[12] = p.tma_bufs;
  info[13] = (pnhwc && (L.use_pair || L.ctas == 1)) ? 1 : 0;  // as the kernels instantiate epilogue_tile
  info[14] = (((p.ldc | p.ch_off) & 7) == 0 && (p.epi_mode != MC_EPI_REORG2 || (p.N & 7) == 0)) ? 1 : 0;
  info[15] = p.last_ksteps;
  return 0;
}

// Words of the chain workspace: ticket, clusters done, status, pad, one readiness counter per (member, m-pair)
static size_t chain_ws_words(const mc_conv_desc* descs, int n) {
  size_t words = CHAIN_COUNTERS;
  for (int i = 0; i < n; ++i) {
    const long long rows = (long long)descs[i].B * (descs[i].H + 1) * (descs[i].W + 1);
    words += (size_t)(((rows + BLOCK_M - 1) / BLOCK_M + 1) / 2);
  }
  return words;
}

// byte range [lo, hi) of the PNHWC rows a member reads (input) or writes (output)
static bool ranges_overlap(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t a0 = (uintptr_t)a, b0 = (uintptr_t)b;
  return a0 < b0 + nb && b0 < a0 + na;
}

// Plans every member (conv_plan, as mc_conv_fwd would) and checks that the members form a chain the kernel can run.
static int chain_plan(const mc_conv_desc* descs, int n, ConvPlan* L) {
  MC_CHECK_ARG(descs != nullptr, "mc_conv_chain_fwd: null descriptors");
  MC_CHECK_ARG(n >= 2 && n <= MAX_CHAIN, "mc_conv_chain_fwd: %d members (2..%d)", n, MAX_CHAIN);
  const mc_conv_desc& d0 = descs[0];
  for (int i = 0; i < n; ++i) {
    const mc_conv_desc& di = descs[i];
    MC_CHECK_ARG(di.ksize == 3 && di.epi_mode == MC_EPI_PNHWC,
                 "mc_conv_chain_fwd: member %d must be a 3x3 layer with the PNHWC epilogue", i);
    MC_CHECK_ARG(di.d_stat_sum == nullptr && di.d_stat_sumsq == nullptr,
                 "mc_conv_chain_fwd: member %d asks for batch statistics", i);
    MC_CHECK_ARG(di.B == d0.B && di.H == d0.H && di.W == d0.W, "mc_conv_chain_fwd: member %d has another B, H or W", i);
    mc_conv_desc one = di;
    one.d_ws = nullptr;  // whole units only: the chain schedules the last waves itself
    one.ws_bytes = 0;
    const int rc = conv_plan(&one, &L[i]);
    if (rc) return rc;
    MC_CHECK_ARG(L[i].use_pair, "mc_conv_chain_fwd: member %d does not take the CTA-pair kernel", i);
    MC_CHECK_ARG(L[i].p.tma_bufs > 0, "mc_conv_chain_fwd: member %d does not take the TMA-store epilogue", i);
    MC_CHECK_ARG(L[i].p.block_n == L[0].p.block_n && L[i].p.stages == L[0].p.stages && L[i].p.leaky == L[0].p.leaky &&
                     L[i].smem_bytes == L[0].smem_bytes,
                 "mc_conv_chain_fwd: member %d has another tile width, ring or activation", i);
    if (i > 0) {
      MC_CHECK_ARG(di.d_in == descs[i - 1].d_out && di.Cin_ld == descs[i - 1].ldc,
                   "mc_conv_chain_fwd: member %d does not read member %d's output allocation", i, i - 1);
    }
  }
  // the only dependency the kernel tracks is member i -> i+1: no other member may read or rewrite what one writes
  const size_t rows = (size_t)d0.B * (d0.H + 1) * (d0.W + 1);
  for (int j = 0; j < n; ++j) {
    const size_t out_bytes = rows * descs[j].ldc * 2;
    for (int i = 0; i < n; ++i) {
      if (i != j + 1)
        MC_CHECK_ARG(!ranges_overlap(descs[i].d_in, rows * descs[i].Cin_ld * 2, descs[j].d_out, out_bytes),
                     "mc_conv_chain_fwd: member %d reads member %d's output", i, j);
      if (i != j)
        MC_CHECK_ARG(!ranges_overlap(descs[i].d_out, rows * descs[i].ldc * 2, descs[j].d_out, out_bytes),
                     "mc_conv_chain_fwd: members %d and %d write the same memory", i, j);
    }
  }
  return 0;
}

extern "C" size_t mc_workspace_bytes_conv_chain(const mc_conv_desc* descs, int n) {
  static thread_local ConvPlan L[MAX_CHAIN];  // (CUtensorMap-heavy: kept off the stack)
  if (chain_plan(descs, n, L) != 0) return 0;
  return chain_ws_words(descs, n) * sizeof(unsigned int);
}

extern "C" int mc_conv_chain_fwd(const mc_conv_desc* descs, int n, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  static thread_local ConvPlan L[MAX_CHAIN];
  int rc = chain_plan(descs, n, L);
  if (rc) return rc;
  const mc_conv_desc& d0 = descs[0];
  const size_t need = chain_ws_words(descs, n) * sizeof(unsigned int);
  MC_CHECK_ARG(d0.d_ws != nullptr && d0.ws_bytes >= need && ((uintptr_t)d0.d_ws & 15) == 0,
               "mc_conv_chain_fwd: descs[0] needs a 16-byte aligned workspace of %zu bytes", need);

  static thread_local PairParams P;
  memset(&P, 0, sizeof(P));
  int units = 0, cnt = 0;
  for (int i = 0; i < n; ++i) {
    pair_layer(L[i], &P.layer[i]);
    units += L[i].units;
    P.layer[i].unit_end = units;
    P.layer[i].cnt_off = cnt;
    cnt += (L[i].p.m_tiles + 1) / 2;
  }
  P.n_layers = n;
  P.chain_ws = reinterpret_cast<unsigned int*>(d0.d_ws);
  int max_clusters = 0;
  rc = pair_max_clusters(&max_clusters);
  if (rc) return rc;
  const int clusters = units < max_clusters ? units : max_clusters;
  g_last_plan[0] = 1; g_last_plan[1] = L[0].p.block_n; g_last_plan[2] = 1; g_last_plan[3] = 0; g_last_plan[4] = 1;
  g_last_plan[5] = L[0].p.stages; g_last_plan[6] = 2 * clusters; g_last_plan[7] = 64;
  conv_gemm_tcgen05_pair_kernel<<<2 * clusters, NUM_THREADS, L[0].smem_bytes, stream>>>(P);
  MC_LAUNCH_CHECK("conv_gemm_tcgen05_pair_kernel");
  return 0;
}

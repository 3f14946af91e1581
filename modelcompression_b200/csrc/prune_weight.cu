// prune_weight.cu — global magnitude pruner on the GPU.
//
// Replaces weight_prune (src/pruning/weightPruning/methods.py:9-26): np.percentile over |w| of every
// parameter with dim != 1, then mask = (|w| > thr).float(); and the weight.data *= mask half of
// MaskedConv2d.set_mask (src/pruning/weightPruning/layers.py:41-47); plus the full-tensor scans of
// prune_rate / are_masks_consistent (src/pruning/weightPruning/utils.py:59-93,122-133).
//
// Selection is exact: |w| >= 0, so its fp32 bit pattern is monotone as uint32 and order statistics can be found by
// integer radix/histogram selection on the bit patterns (weight_prune_kernel below: one cooperative launch).
#include <stdlib.h>
#include <cooperative_groups.h>
#include "common.cuh"

namespace {

constexpr int THREADS = 256;
constexpr int ITERS = 4;                  // float4 loads per thread and block-iteration (all issued before use)
constexpr int CHUNK = THREADS * 4 * ITERS;  // elements per block-iteration
constexpr int BINS0 = 4096;         // bits [30:19]

struct Chunks {
  long long cstart[MC_MAX_SEGMENTS + 1];  // prefix of per-segment chunk counts
};

__device__ __forceinline__ unsigned int absbits(float v) { return __float_as_uint(v) & 0x7fffffffu; }

// locate segment of a global chunk id (nseg <= 64: linear scan over a kernel-parameter table)
__device__ __forceinline__ int find_seg(const Chunks& ch, int nseg, long long cid) {
  int s = 0;
  while (s + 1 < nseg && cid >= ch.cstart[s + 1]) ++s;
  return s;
}

// Visit every element of every segment: f(value, seg, index).  Vectorised when the segment base is 16B aligned.
template <typename F>
__device__ __forceinline__ void for_each_element(const SegTable& st, const Chunks& ch, F f) {
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    const float* p = st.ptr[s];
    const bool aligned = (reinterpret_cast<uintptr_t>(p) & 15) == 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      if (aligned && i + 4 <= size) {
        const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(p + i));
        f(v.x, s, i);
        f(v.y, s, i + 1);
        f(v.z, s, i + 2);
        f(v.w, s, i + 3);
      } else {
        for (int j = 0; j < 4; ++j)
          if (i + j < size) f(p[i + j], s, i + j);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// ONE cooperative kernel does the whole of weight_prune (select + masks), with grid-wide barriers between phases:
//
//   S  a stratified sample of SAMPLE keys is ranked by counting (whole grid) to get three pivots
//      lo <= mid <= hi: [lo, hi] brackets the rank-k key with high probability (+-4.5 sigma of the sample rank), mid
//      is the sample's estimate of it.
//   P  ONE pass over W: count keys < lo, append (key, element index) of the keys in [lo, hi] (~5 % of n) to the
//      candidate list (and bin them for the first histogram level), and write the PROVISIONAL mask |w| > mid —
//      final for everything outside the bracket.
//   R  exact rank inside the candidates: 10-bit histogram levels on (key - lo), all from L2.
//   F  fix-up: the candidates on which (|w| > mid) and (|w| > thr) disagree (~0.5 % of n) are rewritten.
//
// HBM traffic on this path: read W once + write the masks once = 8n bytes (SURVEY.md §8d charges 12n).
// If the bracket missed (k outside, non-finite values present, candidate list overflow) the same kernel falls through
// to the EXACT path: 12-bit histogram of all keys -> compact the selected bin -> 10-bit levels -> full mask pass.  The
// result is always the exact order statistic; only the time differs.
constexpr int SAMPLE = 4096;
constexpr int SAMPLE_LOG2 = 12;
constexpr int LVL_BITS = 10;
constexpr int LVL_BINS = 1 << LVL_BITS;
constexpr int MAX_LVLS = 4;     // keys are < 2^31: 10+10+10+1
constexpr int NWARPS = THREADS / 32;
constexpr int STG = 256;        // staged candidates per warp in the fast pass
constexpr int STG_X = 640;      // ... in the exact-path compaction (a warp-iteration appends at most 32*4*ITERS = 512)
constexpr int SMEM_WORDS = 2 * NWARPS * STG_X;  // 40 KB, carved differently per phase
constexpr int MAXB = 2048;      // max blocks of the cooperative grid (148 SMs x <= 8 resident blocks, with headroom)

// Global atomics are avoided on purpose: atomics to one 128-byte line serialise in L2 at ~5 ns each (measured: 600 K
// histogram flushes to 32 lines cost 110 us).  Every block therefore owns a private slice of the candidate list and
// publishes its counts / first-level histogram with plain stores; sums are taken after the grid barrier.
struct SelState {
  unsigned int lvl_hist[2][MAX_LVLS][LVL_BINS];  // [0] fast attempt, [1] exact attempt
  unsigned int hist0[BINS0];                     // exact path: top 12 bits of every key
  unsigned int sample[SAMPLE];
  unsigned int rank_lt[SAMPLE], rank_le[SAMPLE];  // #sample keys < / <= sample[i]
  unsigned int blk_cnt[2][MAXB];       // candidates held by each block ([0] fast, [1] exact)
  unsigned long long blk_below[MAXB];  // fast: #keys < lo seen by each block
  unsigned long long cnt_le[2];  // #keys <= key_a (fast: among candidates; exact: all)
  unsigned int min_gt[2];        // ~(min key > key_a), 0 = none (atomicMax)
  unsigned int lo_key, mid_key, hi_key;
  unsigned int overflow;         // a block's candidate slice overflowed (fast path gives up)
  unsigned int has_nan;          // a NaN/Inf was seen (fast pass: maybe; exact pass: NaN for sure)
  unsigned int used_fast;        // diagnostics: 1 when the fast path produced the result
  unsigned long long tstamp[12]; // diagnostics: globaltimer of block 0 at the phase boundaries
};

__device__ __forceinline__ void stamp(SelState* st, int i) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    st->tstamp[i] = t;
  }
}

namespace cg = cooperative_groups;

// Block-wide: bin of hist[NBINS] holding rank `rank`, and the rank inside it.  hist was produced by atomics of other
// SMs before a grid barrier: read through L2 (__ldcg).  Every block computes this redundantly.
template <int NBINS>
__device__ void find_bin(const unsigned int* hist, unsigned long long rank, unsigned int* bin_out,
                         unsigned long long* rem_out) {
  __shared__ unsigned long long s_w[NWARPS];
  __shared__ unsigned int s_bin;
  __shared__ unsigned long long s_rem;
  constexpr int PER = NBINS / THREADS;
  static_assert(NBINS % THREADS == 0, "bins per thread");
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned int c[PER];
  unsigned long long tot = 0;
#pragma unroll
  for (int j = 0; j < PER; ++j) { c[j] = __ldcg(hist + threadIdx.x * PER + j); tot += c[j]; }
  unsigned long long incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_w[wid] = incl;
  if (threadIdx.x == 0) { s_bin = NBINS - 1; s_rem = 0; }  // rank beyond the total: clamp
  __syncthreads();
  unsigned long long off = 0;
  for (int w = 0; w < wid; ++w) off += s_w[w];
  unsigned long long cum = off + incl - tot;
  if (rank >= cum && rank < cum + tot) {
    int j = 0;
    for (; j < PER - 1; ++j) {
      if (cum + c[j] > rank) break;
      cum += c[j];
    }
    s_bin = threadIdx.x * PER + j;
    s_rem = rank - cum;
  }
  __syncthreads();
  *bin_out = s_bin;
  *rem_out = s_rem;
  __syncthreads();
}

// segment holding global element index g (last segment with start <= g)
__device__ __forceinline__ int seg_of(const SegTable& st, long long g) {
  int lo = 0, hi = st.nseg - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (st.start[mid] <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// ---- S: pivots by rank counting ------------------------------------------------------------------------------
// stratified sample: element i is taken from the i-th of SAMPLE equal slices of the data, position hashed
__device__ __forceinline__ unsigned int sample_key(const SegTable& st, long long n, int i) {
  const long long a = ((long long)i * n) >> SAMPLE_LOG2, b = ((long long)(i + 1) * n) >> SAMPLE_LOG2;
  unsigned int h = (unsigned int)i * 2654435761u;
  h ^= h >> 15;
  const long long g = a + (long long)(h % (unsigned int)((b - a) > 0 ? (b - a) : 1));
  const int s = seg_of(st, g);
  return absbits(st.ptr[s][g - st.start[s]]);
}

// The whole grid ranks the sample by counting (S^2 = 16.7 M compares, ~100 per thread): block b compares its 256 keys
// (key group b % 16) against slice b / 16 of the sample and adds the counts with global atomics.  A radix select in
// one block (8 warps, dependent shuffle/atomic chains) costs 30-50 us; this costs ~5.
__device__ void sample_rank_count(const SegTable& st, long long n, SelState* state, unsigned int* s_slice) {
  constexpr int GROUPS = SAMPLE / THREADS;  // 16
  const int nslices = (int)gridDim.x / GROUPS;
  if (nslices == 0) {  // tiny grid: every block handles whole key groups against the full sample
    for (int grp = blockIdx.x; grp < GROUPS; grp += gridDim.x) {
      const int i = grp * THREADS + threadIdx.x;
      const unsigned int ki = sample_key(st, n, i);
      state->sample[i] = ki;
      unsigned int lt = 0, le = 0;
      for (int j0 = 0; j0 < SAMPLE; j0 += THREADS) {
        __syncthreads();
        s_slice[threadIdx.x] = sample_key(st, n, j0 + threadIdx.x);
        __syncthreads();
        for (int j = 0; j < THREADS; ++j) {
          const unsigned int kj = s_slice[j];
          lt += kj < ki;
          le += kj <= ki;
        }
      }
      state->rank_lt[i] = lt;
      state->rank_le[i] = le;
    }
    return;
  }
  const int grp = blockIdx.x % GROUPS, slice = blockIdx.x / GROUPS;
  if (slice >= nslices) return;
  const int len = (SAMPLE + nslices - 1) / nslices;  // <= THREADS because nslices >= 1 ... guarded below
  const int j0 = slice * len;
  const int jn = (j0 + len < SAMPLE ? j0 + len : SAMPLE) - j0;
  const int i = grp * THREADS + threadIdx.x;
  const unsigned int ki = sample_key(st, n, i);
  for (int j = threadIdx.x; j < jn; j += THREADS) s_slice[j] = sample_key(st, n, j0 + j);
  if (slice == 0) state->sample[i] = ki;
  __syncthreads();
  unsigned int lt = 0, le = 0;
  int j = 0;
  for (; j + 4 <= jn; j += 4) {
    const uint4 kq = *reinterpret_cast<const uint4*>(s_slice + j);
    lt += (kq.x < ki) + (kq.y < ki) + (kq.z < ki) + (kq.w < ki);
    le += (kq.x <= ki) + (kq.y <= ki) + (kq.z <= ki) + (kq.w <= ki);
  }
  for (; j < jn; ++j) {
    const unsigned int kj = s_slice[j];
    lt += kj < ki;
    le += kj <= ki;
  }
  if (lt) atomicAdd(&state->rank_lt[i], lt);
  if (le) atomicAdd(&state->rank_le[i], le);
}

// after the grid barrier: every block finds the sample keys holding three ranks (rank_lt <= r < rank_le)
__device__ void sample_pick(const SelState* state, const unsigned int (&ranks)[3], unsigned int (&piv)[3]) {
  __shared__ unsigned int s_piv[3];
  if (threadIdx.x < 3) s_piv[threadIdx.x] = 0;
  __syncthreads();
  for (int i0 = threadIdx.x * 4; i0 < SAMPLE; i0 += THREADS * 4) {
    const uint4 lt = __ldcg(reinterpret_cast<const uint4*>(state->rank_lt + i0));
    const uint4 le = __ldcg(reinterpret_cast<const uint4*>(state->rank_le + i0));
    const unsigned int l[4] = {lt.x, lt.y, lt.z, lt.w}, e[4] = {le.x, le.y, le.z, le.w};
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int q = 0; q < 3; ++q)
        if (l[u] <= ranks[q] && ranks[q] < e[u]) s_piv[q] = __ldcg(state->sample + i0 + u);  // equal keys: same value
  }
  __syncthreads();
  piv[0] = s_piv[0];
  piv[1] = s_piv[1];
  piv[2] = s_piv[2];
  __syncthreads();
}

// visit the block's own candidate slice, 8 independent loads in flight per thread
template <typename F>
__device__ __forceinline__ void for_each_own(const unsigned int* __restrict__ seg, unsigned int cnt, F f) {
  unsigned int i = threadIdx.x;
  for (; i + 7u * THREADS < cnt; i += 8 * THREADS) {
    unsigned int k[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) k[u] = __ldcg(seg + i + u * THREADS);
#pragma unroll
    for (int u = 0; u < 8; ++u) f(k[u], i + u * THREADS);
  }
  for (; i < cnt; i += THREADS) f(__ldcg(seg + i), i);
}

// first-level geometry of the candidate histogram: keys rel = key - lo in [0, width]
__device__ __forceinline__ int level0_shift(unsigned int width) {
  const int nb = 32 - __clz((int)width);
  return nb - (nb < LVL_BITS ? nb : LVL_BITS);
}

// sum over the blocks of a per-block value published before the last grid barrier
template <typename T>
__device__ unsigned long long grid_total(const T* per_block) {
  __shared__ unsigned long long s_part[NWARPS];
  __shared__ unsigned long long s_tot;
  unsigned long long v = 0;
  for (unsigned int b = threadIdx.x; b < gridDim.x; b += THREADS) v += (unsigned long long)__ldcg(per_block + b);
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < NWARPS; ++w) t += s_part[w];
    s_tot = t;
  }
  __syncthreads();
  const unsigned long long r = s_tot;
  __syncthreads();
  return r;
}

// Exact rank `rank` among the candidate keys held in the blocks' private slices (this block: seg[0..cnt)), all known
// to lie in [lo, lo+width]: 10-bit histogram levels on rel = key - lo, most significant first.  Collective over the
// grid (one barrier per level); returns the key.  Per-block histograms are merged with global atomics on the non-zero
// bins (measured on B200: 740 blocks x 1024 atomics to the same 4 KB complete in ~6 us).
// lvl0_ready: ghist level 0 was already accumulated before the last grid barrier (binned during the fast pass).
__device__ unsigned int resolve_rank(cg::grid_group& grid, unsigned int* ghist /*[MAX_LVLS][LVL_BINS], zeroed*/,
                                     const unsigned int* seg, unsigned int cnt, unsigned int lo, unsigned int width,
                                     unsigned long long rank, unsigned int* s_hist /*[LVL_BINS]*/, bool lvl0_ready) {
  int shift = 32 - __clz((int)width);  // width < 2^31; width == 0 -> no level needed
  unsigned int prefix = 0;
  for (int lvl = 0; shift > 0; ++lvl) {
    const int bits = shift < LVL_BITS ? shift : LVL_BITS;
    const int hi_shift = shift;  // rel >> hi_shift must equal the bits chosen so far
    shift -= bits;
    if (!(lvl == 0 && lvl0_ready)) {
      for (int i = threadIdx.x; i < LVL_BINS; i += THREADS) s_hist[i] = 0;
      __syncthreads();
      const unsigned int bmask = (1u << bits) - 1u;
      for_each_own(seg, cnt, [&](unsigned int key, unsigned int) {
        const unsigned int rel = key - lo;
        if ((rel >> hi_shift) == prefix) atomicAdd(&s_hist[(rel >> shift) & bmask], 1u);
      });
      __syncthreads();
      for (int i = threadIdx.x; i < LVL_BINS; i += THREADS)
        if (s_hist[i]) atomicAdd(&ghist[lvl * LVL_BINS + i], s_hist[i]);
      grid.sync();
    }
    unsigned int bin;
    unsigned long long rem;
    find_bin<LVL_BINS>(ghist + lvl * LVL_BINS, rank, &bin, &rem);
    prefix = (prefix << bits) | bin;
    rank = rem;
  }
  return lo + prefix;
}

// ---- P: the one pass of the fast path.  ~12 instructions per element: the per-element work is three float compares
// (|w| against the pivots), the mask select and two predicated bit-sets; candidate keys are recovered afterwards
// from a per-lane copy of the 16 values in shared memory, only for the ~5 % that are candidates.
template <bool WRITE_MASK>
__device__ __forceinline__ void fast_pass(const SegTable& st, const Chunks& ch, SelState* state, unsigned int lo,
                                          unsigned int mid, unsigned int hi, unsigned int* __restrict__ cand_key,
                                          unsigned int* __restrict__ cand_idx, unsigned int cap, unsigned int* s_mem) {
  __shared__ unsigned int s_cnt;         // candidates appended by this block
  __shared__ unsigned int s_below[NWARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  // smem: [NWARPS][ITERS][32] float4 value copies | [NWARPS][STG] keys | [NWARPS][STG] indices | [LVL_BINS] level-0 bins
  float4* vals = reinterpret_cast<float4*>(s_mem) + wid * (ITERS * 32);
  unsigned int* wkeys = s_mem + NWARPS * ITERS * 32 * 4 + wid * STG;
  unsigned int* widx = wkeys + NWARPS * STG;
  unsigned int* s_lvl = s_mem + NWARPS * ITERS * 32 * 4 + 2 * NWARPS * STG;
  static_assert(NWARPS * ITERS * 32 * 4 + 2 * NWARPS * STG + LVL_BINS <= SMEM_WORDS, "fast_pass smem carve-up");
  const float lo_f = __uint_as_float(lo), mid_f = __uint_as_float(mid), hi_f = __uint_as_float(hi);
  const int shiftA = level0_shift(hi - lo);
  for (int i = threadIdx.x; i < LVL_BINS; i += THREADS) s_lvl[i] = 0;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  unsigned int wcnt = 0;  // warp-uniform
  unsigned int below = 0;
  float nanacc = 0.f;  // becomes NaN iff a NaN or Inf was seen (x*0)
  auto flush = [&]() {  // warp-wide
    unsigned int base = 0;
    if (lane == 0 && wcnt) base = atomicAdd(&s_cnt, wcnt);
    base = __shfl_sync(0xffffffffu, base, 0);
    __syncwarp();
    for (unsigned int i = lane; i < wcnt; i += 32)
      if (base + i < cap) {
        cand_key[base + i] = wkeys[i];
        cand_idx[base + i] = widx[i];
      }
    __syncwarp();
    wcnt = 0;
  };
  const long long nchunks = ch.cstart[st.nseg];
  // software pipeline: the loads of chunk i+1 are issued before chunk i is processed, so every warp keeps 2 KB in
  // flight while it computes (without this the pass is latency-bound at ~40 % of the HBM rate)
  struct Where {
    const float* p;
    float* mk;
    long long base, size, gstart;
    bool full;
  };
  auto locate = [&](long long cid) {
    Where w;
    const int s = find_seg(ch, st.nseg, cid);
    w.size = st.start[s + 1] - st.start[s];
    w.gstart = st.start[s];
    w.base = (cid - ch.cstart[s]) * CHUNK;
    w.p = st.ptr[s];
    w.mk = st.out[s];
    const bool aligned = ((reinterpret_cast<uintptr_t>(w.p) | (WRITE_MASK ? reinterpret_cast<uintptr_t>(w.mk) : 0)) & 15) == 0;
    w.full = aligned && w.base + CHUNK <= w.size;
    return w;
  };
  float4 qn[ITERS];
  Where nxt;
  long long cid = blockIdx.x;
  if (cid < nchunks) {
    nxt = locate(cid);
    if (nxt.full) {
#pragma unroll
      for (int it = 0; it < ITERS; ++it)
        qn[it] = ld_stream_f4(reinterpret_cast<const float4*>(nxt.p + nxt.base + ((long long)it * THREADS + threadIdx.x) * 4));
    }
  }
  for (; cid < nchunks; cid += gridDim.x) {
    const Where cur = nxt;
    float4 q[ITERS];
#pragma unroll
    for (int it = 0; it < ITERS; ++it) q[it] = qn[it];
    if (cid + gridDim.x < nchunks) {
      nxt = locate(cid + gridDim.x);
      if (nxt.full) {
#pragma unroll
        for (int it = 0; it < ITERS; ++it)
          qn[it] = ld_stream_f4(reinterpret_cast<const float4*>(nxt.p + nxt.base + ((long long)it * THREADS + threadIdx.x) * 4));
      }
    }
    const long long size = cur.size, base = cur.base;
    const float* p = cur.p;
    float* mk = cur.mk;
    if (!cur.full) {
      // ragged chunk (segment tail / unaligned tensor): scalar, candidates appended one by one
      for (long long i = base + threadIdx.x; i < size && i < base + CHUNK; i += THREADS) {
        const float v = p[i];
        const float a = fabsf(v);
        nanacc = fmaf(v, 0.f, nanacc);
        if (WRITE_MASK) mk[i] = a > mid_f ? 1.f : 0.f;
        if (a < lo_f) ++below;
        else if (a <= hi_f) {
          const unsigned int key = __float_as_uint(a);
          const unsigned int pos = atomicAdd(&s_cnt, 1u);
          if (pos < cap) {
            cand_key[pos] = key;
            cand_idx[pos] = (unsigned int)(cur.gstart + i);
          }
          atomicAdd(&s_lvl[(key - lo) >> shiftA], 1u);
        }
      }
      continue;
    }
    unsigned int hits = 0, ge = 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const float v[4] = {q[it].x, q[it].y, q[it].z, q[it].w};
      float m4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float a = fabsf(v[j]);
        nanacc = fmaf(v[j], 0.f, nanacc);
        m4[j] = a > mid_f ? 1.f : 0.f;
        const bool p1 = a >= lo_f;
        if (p1) ge |= 1u << (it * 4 + j);
        if (p1 && a <= hi_f) hits |= 1u << (it * 4 + j);
      }
      if (WRITE_MASK)
        st_stream_f4(reinterpret_cast<float4*>(mk + base + ((long long)it * THREADS + threadIdx.x) * 4),
                     make_float4(m4[0], m4[1], m4[2], m4[3]));
      vals[it * 32 + lane] = q[it];
    }
    below += 4 * ITERS - __popc(ge);
    const unsigned int cnt = __popc(hits);
    unsigned int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const unsigned int tot = __shfl_sync(0xffffffffu, incl, 31);
    if (tot == 0) continue;  // warp-uniform
    if (wcnt + tot > STG) flush();
    const bool direct = tot > STG;  // burst (e.g. thousands of equal keys): straight to the global list
    unsigned int gbase = 0;
    if (direct) {
      if (lane == 0) gbase = atomicAdd(&s_cnt, tot);
      gbase = __shfl_sync(0xffffffffu, gbase, 0);
    }
    unsigned int pos = (direct ? gbase : wcnt) + (incl - cnt);
    const unsigned int idx0 = (unsigned int)(cur.gstart + base) + threadIdx.x * 4;
    const float* myvals = reinterpret_cast<const float*>(vals);
    while (hits) {
      const int j = __ffs(hits) - 1;
      hits &= hits - 1;
      const unsigned int key = absbits(myvals[((j >> 2) * 32 + lane) * 4 + (j & 3)]);
      const unsigned int idx = idx0 + (unsigned int)(j >> 2) * (THREADS * 4) + (unsigned int)(j & 3);
      if (direct) {
        if (pos < cap) {
          cand_key[pos] = key;
          cand_idx[pos] = idx;
        }
      } else {
        wkeys[pos] = key;
        widx[pos] = idx;
      }
      ++pos;
      atomicAdd(&s_lvl[(key - lo) >> shiftA], 1u);
    }
    if (!direct) wcnt += tot;
  }
  flush();
  for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
  if (lane == 0) s_below[wid] = below;
  if (nanacc != nanacc) state->has_nan = 1u;  // rare; every writer stores the same value
  __syncthreads();
  // publish this block's results (read by everyone after the grid barrier)
  for (int i = threadIdx.x; i < LVL_BINS; i += THREADS)
    if (s_lvl[i]) atomicAdd(&state->lvl_hist[0][0][i], s_lvl[i]);
  if (threadIdx.x == 0) {
    unsigned long long tot = 0;
    for (int w = 0; w < NWARPS; ++w) tot += s_below[w];
    state->blk_below[blockIdx.x] = tot;
    const unsigned int c = s_cnt;
    state->blk_cnt[0][blockIdx.x] = c < cap ? c : cap;
    if (c > cap) state->overflow = 1u;
  }
}

// Streaming passes of the exact path.
//   MODE 1: stage the keys in [lo, hi] (one 12-bit bin) and append them to the candidate list
//   MODE 2: 4096-bin histogram of key >> 19 into s_mem (flushed by the caller); records NaNs
template <int MODE>
__device__ __forceinline__ void exact_pass(const SegTable& st, const Chunks& ch, SelState* state, unsigned int lo,
                                           unsigned int hi, unsigned int* __restrict__ cand_key, unsigned int cand_cap,
                                           unsigned int* s_mem) {
  __shared__ unsigned int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned int* wkeys = s_mem + wid * STG_X;
  unsigned int wcnt = 0;  // warp-uniform
  bool saw_nan = false;
  auto flush = [&]() {  // warp-wide
    unsigned int base = 0;
    if (lane == 0 && wcnt) base = atomicAdd(&s_cnt, wcnt);
    base = __shfl_sync(0xffffffffu, base, 0);
    __syncwarp();
    for (unsigned int i = lane; i < wcnt; i += 32)
      if (base + i < cand_cap) cand_key[base + i] = wkeys[i];
    __syncwarp();
    wcnt = 0;
  };
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    const float* p = st.ptr[s];
    const bool aligned = (reinterpret_cast<uintptr_t>(p) & 15) == 0;
    float4 q[ITERS];
    int nvalid[ITERS];
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {  // all loads in flight before the first use
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      q[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      nvalid[it] = 0;
      if (aligned && i + 4 <= size) {
        q[it] = ld_stream_f4(reinterpret_cast<const float4*>(p + i));
        nvalid[it] = 4;
      } else if (i < size) {
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < 4; ++j)
          if (i + j < size) { v[j] = p[i + j]; nvalid[it] = j + 1; }
        q[it] = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
    unsigned int keys[4 * ITERS];
    unsigned int hits = 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const float v[4] = {q[it].x, q[it].y, q[it].z, q[it].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned int key = absbits(v[j]);
        keys[it * 4 + j] = key;
        if (j < nvalid[it]) {
          if (MODE == 2) {
            saw_nan |= key > 0x7f800000u;
            atomicAdd(&s_mem[key >> 19], 1u);
          } else if (key >= lo && key <= hi) {
            hits |= 1u << (it * 4 + j);
          }
        }
      }
    }
    if (MODE == 2) continue;
    if (wcnt > STG_X - 32 * 4 * ITERS) flush();
    const unsigned int cnt = __popc(hits);
    unsigned int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    unsigned int pos = wcnt + (incl - cnt);
#pragma unroll
    for (int j = 0; j < 4 * ITERS; ++j)
      if (hits & (1u << j)) wkeys[pos++] = keys[j];
    wcnt += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (MODE == 1) {
    flush();
    __syncthreads();
    if (threadIdx.x == 0) state->blk_cnt[1][blockIdx.x] = s_cnt < cand_cap ? s_cnt : cand_cap;  // cannot overflow
  }
  if (MODE == 2) {
    // has_nan may hold a "maybe" from the fast pass (Inf also trips it): the exact pass decides
    if (saw_nan) atomicOr(&state->has_nan, 2u);
  }
}

// NumPy's _lerp (numpy/lib/_function_base_impl.py) in float32, no FMA contraction:
//   lerp = a + (b-a)*t ; where t >= 0.5: lerp = b - (b-a)*(1-t)
__device__ __forceinline__ float np_lerp_f32(float a, float b, float gamma) {
  const float diff = __fsub_rn(b, a);
  float r = __fadd_rn(a, __fmul_rn(diff, gamma));
  if (gamma >= 0.5f) r = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, gamma)));
  return r;
}

// count(key <= key_a) and max(~key) over keys > key_a, warp-reduced and accumulated into the state
__device__ __forceinline__ void succ_accumulate(SelState* state, int slot, unsigned long long cnt, unsigned int mx) {
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const unsigned int other = __shfl_xor_sync(0xffffffffu, mx, o);
    mx = other > mx ? other : mx;
  }
  if ((threadIdx.x & 31) == 0) {
    if (cnt) atomicAdd(&state->cnt_le[slot], cnt);
    if (mx) atomicMax(&state->min_gt[slot], mx);
  }
}

template <bool WRITE_MASK>
__global__ void __launch_bounds__(THREADS, 4) weight_prune_kernel(const SegTable st, const Chunks ch, SelState* state,
                                                               unsigned int* cand, unsigned long long region_words,
                                                               unsigned long long k, float gamma, int use_fast,
                                                               float* out3) {
  __shared__ __align__(16) unsigned int s_mem[SMEM_WORDS];  // 40 KB: staging | sample keys | histograms
  static_assert(SMEM_WORDS >= SAMPLE && SMEM_WORDS >= BINS0, "shared scratch too small");
  cg::grid_group grid = cg::this_grid();
  const long long n = st.start[st.nseg];
  // this block's private slice of the candidate area: region_words >= the number of elements the block visits
  unsigned int* region = cand + (size_t)blockIdx.x * region_words;
  unsigned int* my_keys = region;
  const unsigned int fast_cap = (unsigned int)(region_words / 2);
  unsigned int* my_idx = region + fast_cap;
  const int need_b = (gamma != 0.f && (long long)k + 1 < n) ? 1 : 0;
  unsigned int key_a = 0, key_b = 0;
  stamp(state, 0);

  if (use_fast) {
    // ---- S ----
    sample_rank_count(st, n, state, s_mem);
    grid.sync();
    stamp(state, 1);
    unsigned int lo, mid, hi;
    {
      // sample ranks: m = k*S/n estimates the pivot, +- (4.5 sigma + 8) brackets it, sigma = sqrt(S q (1-q))
      const double q = (double)k / (double)n;
      const double m = q * SAMPLE;
      const double sig = sqrt((double)SAMPLE * q * (1.0 - q));
      const double d = 4.5 * sig + 8.0;
      long long rlo = (long long)floor(m - d), rhi = (long long)ceil(m + d) + need_b, rmid = (long long)floor(m);
      const bool open_lo = rlo <= 0, open_hi = rhi >= SAMPLE - 1;
      if (rlo < 0) rlo = 0;
      if (rhi > SAMPLE - 1) rhi = SAMPLE - 1;
      if (rmid < rlo) rmid = rlo;
      if (rmid > rhi) rmid = rhi;
      const unsigned int ranks[3] = {(unsigned int)rlo, (unsigned int)rmid, (unsigned int)rhi};
      unsigned int piv[3];
      sample_pick(state, ranks, piv);
      lo = open_lo ? 0u : piv[0];
      mid = piv[1];
      hi = open_hi ? 0x7fffffffu : piv[2];
      if (blockIdx.x == 0 && threadIdx.x == 0) {
        state->lo_key = lo;
        state->mid_key = mid;
        state->hi_key = hi;
      }
    }
    stamp(state, 2);
    // ---- P ----
    fast_pass<WRITE_MASK>(st, ch, state, lo, mid, hi, my_keys, my_idx, fast_cap, s_mem);
    stamp(state, 3);
    grid.sync();
    stamp(state, 4);
    const unsigned long long below = grid_total(state->blk_below);
    const unsigned long long m = grid_total(state->blk_cnt[0]);
    const unsigned int my_cnt = __ldcg(&state->blk_cnt[0][blockIdx.x]);
    const bool ok = !__ldcg(&state->has_nan) && !__ldcg(&state->overflow) && k >= below &&
                    (k + (unsigned long long)need_b - below) < m;
    if (ok) {  // grid-uniform
      // ---- R: exact rank among the candidates (level 0 was binned during the pass) ----
      key_a = resolve_rank(grid, &state->lvl_hist[0][0][0], my_keys, my_cnt, lo, hi - lo, k - below, s_mem, true);
      stamp(state, 5);
      key_b = key_a;
      if (need_b) {
        unsigned long long cnt = 0;
        unsigned int mx = 0;  // max of ~key over keys > key_a  ==  ~(min key > key_a)
        for_each_own(my_keys, my_cnt, [&](unsigned int key, unsigned int) {
          if (key <= key_a) ++cnt;
          else if (~key > mx) mx = ~key;
        });
        succ_accumulate(state, 0, cnt, mx);
        grid.sync();
        const unsigned long long cnt_le = below + __ldcg(&state->cnt_le[0]);
        const unsigned int mg = __ldcg(&state->min_gt[0]);
        if (cnt_le <= k + 1ull && mg) key_b = ~mg;
      }
      const float thr = np_lerp_f32(__uint_as_float(key_a), __uint_as_float(key_b), gamma);
      // ---- F: candidates whose provisional mask (|w| > mid) differs from the final one (|w| > thr) ----
      if (WRITE_MASK) {
        const float mid_f = __uint_as_float(mid);
        for_each_own(my_keys, my_cnt, [&](unsigned int key, unsigned int i) {
          const float a = __uint_as_float(key);
          const bool fin = a > thr;
          if (fin != (a > mid_f)) {
            const long long g = (long long)__ldcg(my_idx + i);
            const int s = seg_of(st, g);
            st.out[s][g - st.start[s]] = fin ? 1.f : 0.f;
          }
        });
      }
      if (blockIdx.x == 0 && threadIdx.x == 0) {
        out3[0] = thr;
        out3[1] = __uint_as_float(key_a);
        out3[2] = __uint_as_float(key_b);
        state->used_fast = 1;
      }
      stamp(state, 6);
      return;
    }
  }

  // ---- exact path ----
  for (int i = threadIdx.x; i < BINS0; i += THREADS) s_mem[i] = 0;
  __syncthreads();
  exact_pass<2>(st, ch, state, 0u, 0u, nullptr, 0u, s_mem);
  __syncthreads();
  for (int i = threadIdx.x; i < BINS0; i += THREADS)
    if (s_mem[i]) atomicAdd(&state->hist0[i], s_mem[i]);
  grid.sync();
  unsigned int bin0;
  unsigned long long rem1;
  find_bin<BINS0>(state->hist0, k, &bin0, &rem1);
  const unsigned int lo = bin0 << 19, hi = lo + ((1u << 19) - 1u);
  exact_pass<1>(st, ch, state, lo, hi, my_keys, (unsigned int)region_words, s_mem);
  grid.sync();
  const unsigned int my_cnt = __ldcg(&state->blk_cnt[1][blockIdx.x]);
  key_a = resolve_rank(grid, &state->lvl_hist[1][0][0], my_keys, my_cnt, lo, hi - lo, rem1, s_mem, false);
  key_b = key_a;
  if (need_b) {
    // count(key <= key_a) and min(key > key_a) over the ORIGINAL data decide sorted[k+1]
    unsigned long long cnt = 0;
    unsigned int mx = 0;
    for_each_element(st, ch, [&](float v, int, long long) {
      const unsigned int key = absbits(v);
      if (key <= key_a) ++cnt;
      else if (~key > mx) mx = ~key;
    });
    succ_accumulate(state, 1, cnt, mx);
    grid.sync();
    const unsigned long long cnt_le = __ldcg(&state->cnt_le[1]);
    const unsigned int mg = __ldcg(&state->min_gt[1]);
    if (cnt_le <= k + 1ull && mg) key_b = ~mg;
  }
  float thr = np_lerp_f32(__uint_as_float(key_a), __uint_as_float(key_b), gamma);
  float fa = __uint_as_float(key_a), fb = __uint_as_float(key_b);
  if (__ldcg(&state->has_nan) & 2u) thr = fa = fb = __uint_as_float(0x7fc00000u);  // np.percentile of data with NaN
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    out3[0] = thr;
    out3[1] = fa;
    out3[2] = fb;
  }
  if (WRITE_MASK) {
    for_each_element(st, ch, [&](float v, int s, long long i) { st.out[s][i] = fabsf(v) > thr ? 1.f : 0.f; });
  }
}

// ---- mask / apply ----------------------------------------------------------------------------------------
template <bool WRITE_MASK, bool APPLY>
__global__ void __launch_bounds__(THREADS) mask_kernel(const SegTable st, const Chunks ch, const float* __restrict__ thr_p) {
  const float thr = *thr_p;
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    float* w = const_cast<float*>(st.ptr[s]);
    float* m = st.out[s];
    const bool aligned = ((reinterpret_cast<uintptr_t>(w) | (WRITE_MASK ? reinterpret_cast<uintptr_t>(m) : 0)) & 15) == 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      if (aligned && i + 4 <= size) {
        const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(w + i));
        float4 mk;
        mk.x = fabsf(v.x) > thr ? 1.f : 0.f;
        mk.y = fabsf(v.y) > thr ? 1.f : 0.f;
        mk.z = fabsf(v.z) > thr ? 1.f : 0.f;
        mk.w = fabsf(v.w) > thr ? 1.f : 0.f;
        if (WRITE_MASK) st_stream_f4(reinterpret_cast<float4*>(m + i), mk);
        if (APPLY) {
          float4 o;
          o.x = __fmul_rn(v.x, mk.x);
          o.y = __fmul_rn(v.y, mk.y);
          o.z = __fmul_rn(v.z, mk.z);
          o.w = __fmul_rn(v.w, mk.w);
          st_stream_f4(reinterpret_cast<float4*>(w + i), o);
        }
      } else {
        for (int j = 0; j < 4; ++j)
          if (i + j < size) {
            const float v = w[i + j];
            const float mk = fabsf(v) > thr ? 1.f : 0.f;
            if (WRITE_MASK) m[i + j] = mk;
            if (APPLY) w[i + j] = __fmul_rn(v, mk);
          }
      }
    }
  }
}

// w *= mask (out[] of the table holds the mask pointers)
__global__ void __launch_bounds__(THREADS) apply_masks_kernel(const SegTable st, const Chunks ch) {
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    float* w = const_cast<float*>(st.ptr[s]);
    const float* m = st.out[s];
    const bool aligned = ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(m)) & 15) == 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      if (aligned && i + 4 <= size) {
        const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(w + i));
        const float4 k = ld_stream_f4(reinterpret_cast<const float4*>(m + i));
        float4 o;
        o.x = __fmul_rn(v.x, k.x);
        o.y = __fmul_rn(v.y, k.y);
        o.z = __fmul_rn(v.z, k.z);
        o.w = __fmul_rn(v.w, k.w);
        st_stream_f4(reinterpret_cast<float4*>(w + i), o);
      } else {
        for (int j = 0; j < 4; ++j)
          if (i + j < size) w[i + j] = __fmul_rn(w[i + j], m[i + j]);
      }
    }
  }
}

__global__ void __launch_bounds__(THREADS) count_zeros_kernel(const SegTable st, const Chunks ch,
                                                              unsigned long long* __restrict__ counts) {
  __shared__ unsigned int s_cnt[MC_MAX_SEGMENTS];
  if (threadIdx.x < MC_MAX_SEGMENTS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    const float* p = st.ptr[s];
    const bool aligned = (reinterpret_cast<uintptr_t>(p) & 15) == 0;
    unsigned int c = 0;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      if (aligned && i + 4 <= size) {
        const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(p + i));
        c += (v.x == 0.f) + (v.y == 0.f) + (v.z == 0.f) + (v.w == 0.f);
      } else {
        for (int j = 0; j < 4; ++j)
          if (i + j < size) c += (p[i + j] == 0.f);
      }
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt[s], c);
  }
  __syncthreads();
  if (threadIdx.x < st.nseg && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

__global__ void __launch_bounds__(THREADS) masked_residual_kernel(const SegTable st, const Chunks ch,
                                                                  double* __restrict__ out) {
  const long long nchunks = ch.cstart[st.nseg];
  for (long long cid = blockIdx.x; cid < nchunks; cid += gridDim.x) {
    const int s = find_seg(ch, st.nseg, cid);
    const long long size = st.start[s + 1] - st.start[s];
    const long long base = (cid - ch.cstart[s]) * CHUNK;
    const float* w = st.ptr[s];
    const float* m = st.out[s];
    double acc = 0.0;
    for (int it = 0; it < ITERS; ++it) {
      const long long i = base + ((long long)it * THREADS + threadIdx.x) * 4;
      for (int j = 0; j < 4; ++j)
        if (i + j < size) acc += (double)(w[i + j] * fabsf(m[i + j] - 1.f));
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc != 0.0) atomicAdd(&out[s], acc);
  }
}

int build_tables(SegTable* st, Chunks* ch, const float* const* ptrs, float* const* outs, const int64_t* sizes,
                 int nseg, const char* who) {
  if (nseg <= 0 || nseg > MC_MAX_SEGMENTS) return mc_set_error(MC_ERR_ARG, "%s: nseg %d out of range 1..%d", who, nseg, MC_MAX_SEGMENTS);
  if (!ptrs || !sizes) return mc_set_error(MC_ERR_ARG, "%s: null table", who);
  st->nseg = nseg;
  st->start[0] = 0;
  ch->cstart[0] = 0;
  for (int s = 0; s < nseg; ++s) {
    if (sizes[s] < 0 || (sizes[s] > 0 && !ptrs[s])) return mc_set_error(MC_ERR_ARG, "%s: segment %d invalid", who, s);
    st->ptr[s] = ptrs[s];
    st->out[s] = outs ? outs[s] : nullptr;
    st->start[s + 1] = st->start[s] + sizes[s];
    ch->cstart[s + 1] = ch->cstart[s] + (sizes[s] + CHUNK - 1) / CHUNK;
  }
  for (int s = nseg; s < MC_MAX_SEGMENTS; ++s) {
    st->ptr[s] = nullptr;
    st->out[s] = nullptr;
    st->start[s + 1] = st->start[nseg];
    ch->cstart[s + 1] = ch->cstart[nseg];
  }
  return 0;
}

int stream_grid(long long nchunks) {
  long long g = (long long)mc_num_sms() * 8;
  if (g > nchunks) g = nchunks;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" size_t mc_workspace_bytes_kth_abs_select(int64_t n_total) {
  if (n_total < 0) n_total = 0;
  // state + per-block candidate slices (worst case of the exact path: every element a candidate, e.g. an
  // already-pruned model; each block's slice is rounded up to whole chunks)
  return ((sizeof(SelState) + 255) / 256) * 256 +
         ((size_t)n_total + (size_t)MAXB * CHUNK) * sizeof(unsigned int) + 256;
}

namespace {

int launch_weight_prune(const float* const* h_w_ptrs, float* const* h_mask_ptrs, const int64_t* h_seg_sizes, int nseg,
                        int64_t k, float gamma, float* d_out3, void* d_ws, size_t ws_bytes, cudaStream_t stream,
                        const char* who) {
  SegTable st;
  Chunks ch;
  int rc = build_tables(&st, &ch, h_w_ptrs, h_mask_ptrs, h_seg_sizes, nseg, who);
  if (rc) return rc;
  const long long n = st.start[nseg];
  MC_CHECK_ARG(n > 0, "%s: empty input", who);
  MC_CHECK_ARG(k >= 0 && k < n, "%s: rank %lld out of range [0,%lld)", who, (long long)k, n);
  MC_CHECK_ARG(d_out3 && d_ws, "%s: null output/workspace", who);
  MC_CHECK_ARG(gamma >= 0.f && gamma < 1.f, "%s: gamma must be in [0,1)", who);
  if (h_mask_ptrs)
    for (int s = 0; s < nseg; ++s) MC_CHECK_ARG(h_mask_ptrs[s] || h_seg_sizes[s] == 0, "%s: null mask %d", who, s);
  if (ws_bytes < mc_workspace_bytes_kth_abs_select(n))
    return mc_set_error(MC_ERR_WS, "%s: workspace %zu < required %zu", who, ws_bytes, mc_workspace_bytes_kth_abs_select(n));
  const size_t state_bytes = ((sizeof(SelState) + 255) / 256) * 256;
  SelState* state = reinterpret_cast<SelState*>(d_ws);
  unsigned int* cand = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(d_ws) + state_bytes);

  // the fast path indexes elements with 32 bits and needs a sample much smaller than the data
  int use_fast = (n >= 8 * SAMPLE && n < (1ll << 32)) ? 1 : 0;

  static int blocks_per_sm[2] = {0, 0};
  const int which = h_mask_ptrs ? 1 : 0;
  if (blocks_per_sm[which] == 0) {
    int nb = 0;
    if (which) MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, weight_prune_kernel<true>, THREADS, 0));
    else MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, weight_prune_kernel<false>, THREADS, 0));
    if (nb < 1) return mc_set_error(MC_ERR_SHAPE, "%s: kernel does not fit an SM", who);
    blocks_per_sm[which] = nb;
  }
  long long grid = (long long)mc_num_sms() * blocks_per_sm[which];
  if (grid > ch.cstart[nseg]) grid = ch.cstart[nseg];
  if (grid > MAXB) grid = MAXB;
  if (grid < 1) grid = 1;
  // a block visits at most ceil(nchunks / grid) chunks: its candidate slice holds that many elements
  unsigned long long region_words = (unsigned long long)((ch.cstart[nseg] + grid - 1) / grid) * CHUNK;

  MC_CUDA(cudaMemsetAsync(d_ws, 0, state_bytes, stream));
  unsigned long long kk = (unsigned long long)k;
  void* args[] = {&st, &ch, &state, &cand, &region_words, &kk, &gamma, &use_fast, &d_out3};
  const void* fn = which ? (const void*)weight_prune_kernel<true> : (const void*)weight_prune_kernel<false>;
  MC_CUDA(cudaLaunchCooperativeKernel(fn, dim3((unsigned)grid), dim3(THREADS), args, 0, stream));
  return 0;
}

}  // namespace

extern "C" int mc_kth_abs_select(const float* const* h_seg_ptrs, const int64_t* h_seg_sizes, int nseg, int64_t k,
                                 float gamma, float* d_out3, void* d_ws, size_t ws_bytes, void* stream_) {
  return launch_weight_prune(h_seg_ptrs, nullptr, h_seg_sizes, nseg, k, gamma, d_out3, d_ws, ws_bytes,
                             reinterpret_cast<cudaStream_t>(stream_), "mc_kth_abs_select");
}

extern "C" int mc_weight_prune_masks(const float* const* h_w_ptrs, float* const* h_mask_ptrs, const int64_t* h_seg_sizes,
                                     int nseg, int64_t k, float gamma, float* d_out3, void* d_ws, size_t ws_bytes,
                                     void* stream_) {
  MC_CHECK_ARG(h_mask_ptrs != nullptr, "mc_weight_prune_masks: null mask table");
  return launch_weight_prune(h_w_ptrs, h_mask_ptrs, h_seg_sizes, nseg, k, gamma, d_out3, d_ws, ws_bytes,
                             reinterpret_cast<cudaStream_t>(stream_), "mc_weight_prune_masks");
}

extern "C" int mc_debug_select_tstamps(const void* d_ws, unsigned long long* h_out12, void* stream_) {
  const SelState* state = reinterpret_cast<const SelState*>(d_ws);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CUDA(cudaMemcpyAsync(h_out12, state->tstamp, sizeof(state->tstamp), cudaMemcpyDeviceToHost, stream));
  MC_CUDA(cudaStreamSynchronize(stream));
  return 0;
}

extern "C" int mc_debug_select_used_fast(const void* d_ws, void* stream_) {
  unsigned int v = 0;
  const SelState* state = reinterpret_cast<const SelState*>(d_ws);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CUDA(cudaMemcpyAsync(&v, &state->used_fast, sizeof(v), cudaMemcpyDeviceToHost, stream));
  MC_CUDA(cudaStreamSynchronize(stream));
  return (int)v;
}

extern "C" int mc_mask_apply_gt(float* const* h_w_ptrs, float* const* h_mask_ptrs, const int64_t* h_seg_sizes,
                                int nseg, const float* d_thr, int apply, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_thr != nullptr, "mc_mask_apply_gt: null threshold pointer");
  MC_CHECK_ARG(h_mask_ptrs != nullptr || apply, "mc_mask_apply_gt: nothing to do (no masks, no apply)");
  SegTable st;
  Chunks ch;
  int rc = build_tables(&st, &ch, const_cast<const float* const*>(h_w_ptrs), h_mask_ptrs, h_seg_sizes, nseg,
                        "mc_mask_apply_gt");
  if (rc) return rc;
  if (h_mask_ptrs)
    for (int s = 0; s < nseg; ++s) MC_CHECK_ARG(h_mask_ptrs[s] || h_seg_sizes[s] == 0, "mc_mask_apply_gt: null mask %d", s);
  if (ch.cstart[nseg] == 0) return 0;
  const int grid = stream_grid(ch.cstart[nseg]);
  if (h_mask_ptrs && apply) mask_kernel<true, true><<<grid, THREADS, 0, stream>>>(st, ch, d_thr);
  else if (h_mask_ptrs) mask_kernel<true, false><<<grid, THREADS, 0, stream>>>(st, ch, d_thr);
  else mask_kernel<false, true><<<grid, THREADS, 0, stream>>>(st, ch, d_thr);
  MC_LAUNCH_CHECK("mask_kernel");
  return 0;
}

extern "C" int mc_apply_masks(float* const* h_w_ptrs, const float* const* h_mask_ptrs, const int64_t* h_seg_sizes,
                              int nseg, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(h_mask_ptrs != nullptr, "mc_apply_masks: null mask table");
  SegTable st;
  Chunks ch;
  int rc = build_tables(&st, &ch, const_cast<const float* const*>(h_w_ptrs),
                        const_cast<float* const*>(reinterpret_cast<const float* const*>(h_mask_ptrs)), h_seg_sizes,
                        nseg, "mc_apply_masks");
  if (rc) return rc;
  for (int s = 0; s < nseg; ++s) MC_CHECK_ARG(h_mask_ptrs[s] || h_seg_sizes[s] == 0, "mc_apply_masks: null mask %d", s);
  if (ch.cstart[nseg] == 0) return 0;
  apply_masks_kernel<<<stream_grid(ch.cstart[nseg]), THREADS, 0, stream>>>(st, ch);
  MC_LAUNCH_CHECK("apply_masks_kernel");
  return 0;
}

extern "C" int mc_count_zeros(const float* const* h_w_ptrs, const int64_t* h_seg_sizes, int nseg, int64_t* d_counts,
                              void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_counts != nullptr, "mc_count_zeros: null output");
  SegTable st;
  Chunks ch;
  int rc = build_tables(&st, &ch, h_w_ptrs, nullptr, h_seg_sizes, nseg, "mc_count_zeros");
  if (rc) return rc;
  MC_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(int64_t) * nseg, stream));
  if (ch.cstart[nseg] == 0) return 0;
  count_zeros_kernel<<<stream_grid(ch.cstart[nseg]), THREADS, 0, stream>>>(st, ch,
                                                                           reinterpret_cast<unsigned long long*>(d_counts));
  MC_LAUNCH_CHECK("count_zeros_kernel");
  return 0;
}

extern "C" int mc_masked_residual(const float* const* h_w_ptrs, const float* const* h_mask_ptrs,
                                  const int64_t* h_seg_sizes, int nseg, double* d_out, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_out != nullptr && h_mask_ptrs != nullptr, "mc_masked_residual: null pointer");
  SegTable st;
  Chunks ch;
  int rc = build_tables(&st, &ch, h_w_ptrs, const_cast<float* const*>(reinterpret_cast<const float* const*>(h_mask_ptrs)),
                        h_seg_sizes, nseg, "mc_masked_residual");
  if (rc) return rc;
  MC_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * nseg, stream));
  if (ch.cstart[nseg] == 0) return 0;
  masked_residual_kernel<<<stream_grid(ch.cstart[nseg]), THREADS, 0, stream>>>(st, ch, d_out);
  MC_LAUNCH_CHECK("masked_residual_kernel");
  return 0;
}

// prune_filter.cu — global filter pruner ("scaled L2 norm" of each filter) on the GPU.
//
// Replaces quick_filter_prune (src/pruning/weightPruning/methods.py:28-78).  The reference computes, per conv
// weight p[O,C,kh,kw] (float32, NumPy):
//     v = np.square(p).sum(axis=1).sum(axis=1).sum(axis=1) / (C*kh*kw)          methods.py:43-44
//     v = v / np.sqrt(np.square(v).sum());  v /= np.max(v)                      methods.py:46-51
//     thr = np.percentile(concat(v of all layers) as float64, perc)             methods.py:53-55
//     mask[o] = 0 where v[o] < thr                                              methods.py:75
// Bit-exactness needs NumPy's float32 summation ORDER (SURVEY.md §8a-6):
//   kh*kw > 1 : s[h,w] = sum over c, sequential in c; then sequential over h; then sequential over w.
//   kh*kw == 1: NumPy pairwise summation over the contiguous C axis (numpy/_core/src/umath/loops_utils.h.src:
//               n<8 sequential; n<=128: 8 strided accumulators, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), tail;
//               else split at n/2 rounded down to a multiple of 8).  sum(v^2) over O uses the same rule.
// All products/sums use *_rn intrinsics so nvcc cannot contract them into FMAs.
#include <limits.h>
#include <stdlib.h>
#include "common.cuh"

namespace {

constexpr int MAX_LAYERS = MC_MAX_SEGMENTS;

struct LayerTable {
  const float* w[MAX_LAYERS];
  float* mask[MAX_LAYERS];
  int O[MAX_LAYERS], C[MAX_LAYERS], taps[MAX_LAYERS];
  int voff[MAX_LAYERS + 1];        // prefix of O
  long long woff[MAX_LAYERS + 1];  // prefix of O*C*taps
  int toff[MAX_LAYERS + 1];        // prefix of threads used by the generic sumsq path (tiled layers take none)
  int nlayers;
  // tiled path (3x3, C % 32 == 0, O % 32 == 0): work items = groups of 32 filters, layers ordered by descending C
  int torder[MAX_LAYERS];          // layer index of the i-th tiled layer
  int tblk[MAX_LAYERS + 1];        // prefix of work items over torder
  int ntiled;
};

// ---- NumPy's pairwise sum of x^2, without recursion ---------------------------------------------------------------
// NumPy's recursion over [0, n), walked in order with an explicit stack: a node longer than 128 is its left half
// [0, n2) plus its right half, n2 = n/2 rounded down to a multiple of 8; a leaf is the current [st, st + ln).
// next(s) adds the current leaf's sum s in the recursion's order and moves to the next leaf; it returns false after the
// last leaf, and total then holds the sum.  Every leaf of an n > 128 walk is at least 64 long.
struct NpWalk {
  static constexpr int DEPTH = 25;  // levels of the recursion for any int n
  int rln[DEPTH];                   // per open level: length of the right half, 0 once the walk is inside it
  float lsum[DEPTH];                // ... and the sum of its left half
  int sp = 0, st = 0, ln;
  float total = 0.f;
  __device__ explicit NpWalk(int n) : ln(n) { descend(); }
  __device__ void descend() {
    while (ln > 128) {
      int n2 = ln / 2;
      n2 -= n2 % 8;
      rln[sp++] = ln - n2;
      ln = n2;
    }
  }
  __device__ bool next(float s) {
    while (sp > 0 && rln[sp - 1] == 0) s = __fadd_rn(lsum[--sp], s);  // right halves complete: (left + right)
    if (sp == 0) {
      total = s;
      return false;
    }
    lsum[sp - 1] = s;  // a left half is complete: its right half starts where the leaf ends
    st += ln;
    ln = rln[sp - 1];
    rln[sp - 1] = 0;
    descend();
    return true;
  }
};

// Leaf sums ls[0, ...) of a pairwise sum over n elements, combined in the recursion's order.
__device__ float np_combine_leaves(const float* ls, int n) {
  NpWalk w(n);
  for (int i = 0; w.next(ls[i]); ++i) {}
  return w.total;
}

// NumPy's pairwise sum of a[i]^2 over one leaf (n <= 128) by an 8-lane group: lane j = lane & 7 runs accumulator j, the
// xor-1/2/4 butterfly performs ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) (fp add is commutative), then the sequential tail.
// All 32 lanes call it, each group with its own leaf (n = 0: none); the result is valid in every lane of the group.
__device__ __forceinline__ float group_leaf_sumsq(const float* a, int n) {
  const int j = threadIdx.x & 7;
  const int body = n - (n % 8);
  float r = 0.f;
  if (n >= 8) {
    float x = a[j];
    r = __fmul_rn(x, x);
    for (int i = 8; i < body; i += 8) {
      x = a[i + j];
      r = __fadd_rn(r, __fmul_rn(x, x));
    }
  }
  float t = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));
  t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 2));
  t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 4));
  float sum = n >= 8 ? t : 0.f;
  for (int i = n >= 8 ? body : 0; i < n; ++i) sum = __fadd_rn(sum, __fmul_rn(a[i], a[i]));
  return sum;
}

// NumPy's pairwise sum of a[i]^2 over [0, n) by one warp, bit-exact: one walk hands out the leaves four at a time
// (group q of 8 lanes sums the q-th), a second walk combines their sums in the recursion's order.  Result in every lane.
// n = 128 * L with L = 2^k <= 128 (and n <= 128) skips the walks: the recursion halves exactly, so the leaves are
// [128 i, 128 i + 128) and their sums combine as a balanced tree, within a group of four by shuffles and across the
// groups by lane (group b sits in lane b).
__device__ float warp_pairwise_sumsq(const float* a, int n) {
  const int lane = threadIdx.x & 31, lq = lane >> 3;
  const int L = n <= 128 ? 1 : n / 128;
  if (n <= 128 || (n % 128 == 0 && (L & (L - 1)) == 0 && L <= 128)) {
    float mine = 0.f;
    for (int b = 0; 4 * b < L; ++b) {
      const int leaf = 4 * b + lq;
      float t = group_leaf_sumsq(a + 128 * leaf, leaf < L ? (n < 128 ? n : 128) : 0);
      if (L >= 2) t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 8));
      if (L >= 4) t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 16));
      if (lane == b) mine = t;
    }
    for (int o = 1; o < L / 4; o <<= 1) mine = __fadd_rn(mine, __shfl_xor_sync(0xffffffffu, mine, o));
    __syncwarp();
    return __shfl_sync(0xffffffffu, mine, 0);
  }
  NpWalk leaves(n), sums(n);
  for (bool more = true; more;) {  // every lane walks the same leaves: the loop is warp-uniform
    int st = 0, ln = 0, cnt = 0;
    for (; cnt < 4 && more; ++cnt) {
      if (cnt == lq) { st = leaves.st; ln = leaves.ln; }
      more = leaves.next(0.f);
    }
    const float s = group_leaf_sumsq(a + st, ln);
    for (int q = 0; q < cnt; ++q) sums.next(__shfl_sync(0xffffffffu, s, 8 * q));
  }
  __syncwarp();  // every lane's reads of a are done before the caller overwrites it
  return sums.total;
}

constexpr int ROW_MAX = 2048;     // 1x1 rows up to this many channels are staged in shared memory (warp path)

// Raw per-filter sums.  taps>1: one thread per (filter, tap) runs the sequential-in-c chain (loads are issued 32 deep
// so the chain is not exposed to memory latency); the taps of a filter sit in adjacent lanes and are combined in
// NumPy's (h then w) order through shared memory.  taps==1: one WARP per filter runs the lane-parallel pairwise sum.
constexpr int SS_THREADS = 288;  // multiple of 9 and of 32

template <int NT>
__device__ void sumsq_generic_block(const LayerTable& lt, int gblk, float* __restrict__ values, float* s_tap,
                                    float* s_rows /*[NT / 32][ROW_MAX]*/) {
  const int gt = gblk * NT + threadIdx.x;  // global thread slot (blocks never straddle layers)
  int l = 0;
  while (l + 1 < lt.nlayers && gt >= lt.toff[l + 1]) ++l;
  const int local = gt - lt.toff[l];
  const int taps = lt.taps[l], C = lt.C[l], O = lt.O[l];
  const float* __restrict__ w = lt.w[l];
  if (taps == 1) {
    // one WARP per filter.  A row (C floats, contiguous) of up to ROW_MAX channels is first staged in shared memory
    // with ONE round of coalesced loads; a wider row is summed straight from global memory.
    const int o = local >> 5, lane = threadIdx.x & 31;
    if (o >= O) return;  // whole warp
    const float* a = w + (long long)o * C;
    if (C <= ROW_MAX) {
      float* srow = s_rows + (threadIdx.x >> 5) * ROW_MAX;
      if ((C & 3) == 0) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        for (int i = lane; i < C / 4; i += 32) reinterpret_cast<float4*>(srow)[i] = ld_stream_f4(a4 + i);
      } else {
        for (int i = lane; i < C; i += 32) srow[i] = a[i];
      }
      __syncwarp();
      a = srow;
    }
    const float s = warp_pairwise_sumsq(a, C);
    if (lane == 0) values[lt.voff[l] + o] = __fdiv_rn(s, (float)C);
    return;
  }
  // blocks hold whole filters: fpb filters x taps threads, the remaining threads of the block idle
  const int fpb = NT / taps;
  const int blk = local / NT, tl = local - blk * NT;
  const int fl = tl / taps, j = tl - fl * taps;
  const int o = (fl < fpb) ? blk * fpb + fl : O;  // O = out of range -> idle
  float acc = 0.f;
  if (o < O) {
    const float* p = w + (long long)o * C * taps + j;
    int c = 0;
    for (; c + 32 <= C; c += 32) {
      float x[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) x[u] = p[(long long)(c + u) * taps];
#pragma unroll
      for (int u = 0; u < 32; ++u) acc = __fadd_rn(acc, __fmul_rn(x[u], x[u]));
    }
    for (; c < C; ++c) {
      const float x = p[(long long)c * taps];
      acc = __fadd_rn(acc, __fmul_rn(x, x));
    }
  }
  s_tap[threadIdx.x] = acc;
  __syncthreads();
  if (o < O && j == 0) {
    // taps = kh*kw with kh == kw (square kernels): s[h][w] at s_tap[base + h*k + w]
    int k = 1;
    while (k * k < taps) ++k;
    const float* s = &s_tap[threadIdx.x];
    float tot = 0.f;
    for (int ww = 0; ww < k; ++ww) {
      float col = 0.f;
      for (int hh = 0; hh < k; ++hh) col = __fadd_rn(col, s[hh * k + ww]);  // .sum(axis=1) over h, sequential
      tot = __fadd_rn(tot, col);                                            // final .sum(axis=1) over w (n<8)
    }
    values[lt.voff[l] + o] = __fdiv_rn(tot, (float)(C * taps));
  }
}

// ---- tiled path for the 3x3 layers (97 % of the weights) ------------------------------------------------------
// A block owns 32 filters and walks their C axis in chunks of 32 channels: the 32 x 288 floats of a chunk are
// contiguous per filter (1152 B) and are copied with 16-byte cp.async into a 3-stage shared-memory ring (two chunks
// = 72 KB in flight per block, no registers involved); thread (f, tap) runs its 32 sequential square-adds on the
// oldest stage meanwhile.  The summation order per (filter, tap) is the same sequential-in-c chain as above.  What
// bounds a block is the LENGTH of that chain (C/32 ring steps), so a step must cost the compute, not a DRAM latency.
constexpr int TL_F = 32;               // filters per block
constexpr int TL_C = 32;               // channels per chunk
constexpr int TL_ROW4 = 74;            // float4 per tile row: 72 data + 2 pad (bank = 8f + tap: 2-way conflicts at most)
constexpr int TL_TILE4 = TL_F * TL_ROW4;
constexpr int TL_STAGES = 3;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const unsigned int d = (unsigned int)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// F filters per block (F * 9 threads run the chains and issue the copies; further threads of the block only take part
// in the barriers), STAGES ring slots of F x 32 channels.
template <int F, int STAGES>
__device__ void sumsq_tiled_block(const LayerTable& lt, int item, float* __restrict__ values,
                                  float4* s_tile /*[STAGES][F * TL_ROW4]*/, float* s_tap /*[blockDim.x]*/) {
  constexpr int WORK = F * 9;          // threads with a (filter, tap) chain
  constexpr int TILE4 = F * TL_ROW4;
  int ti = 0;
  while (ti + 1 < lt.ntiled && item >= lt.tblk[ti + 1]) ++ti;
  const int l = lt.torder[ti];
  const int C = lt.C[l];
  const int o0 = (item - lt.tblk[ti]) * F;
  const int t = threadIdx.x;
  const bool worker = t < WORK;
  const int f = worker ? t / 9 : 0, j = worker ? t - f * 9 : 0;
  const int nchunks = C / TL_C;
  // o0*C*9*4 bytes is a multiple of 16 because C % 32 == 0
  const float4* __restrict__ w4 = reinterpret_cast<const float4*>(lt.w[l] + (long long)o0 * C * 9);
  // this thread's 8 float4 of a chunk: q = u*288 + t -> (row = q / 72, col4 = q % 72)
  int grow[8], scol[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int q = u * WORK + (worker ? t : 0);
    const int row = q / 72, col4 = q - row * 72;
    grow[u] = row * (C * 9 / 4) + col4;  // float4 index inside the block's filters
    scol[u] = row * TL_ROW4 + col4;
  }
  auto issue = [&](int cc) {
    if (cc < nchunks && worker) {
      float4* tile = s_tile + (cc % STAGES) * TILE4;
      const float4* src = w4 + (long long)cc * (TL_C * 9 / 4);
#pragma unroll
      for (int u = 0; u < 8; ++u) cp_async16(tile + scol[u], src + grow[u]);
    }
    cp_async_commit();  // an empty group keeps the wait_group arithmetic uniform at the tail
  };
#pragma unroll
  for (int p = 0; p < STAGES - 1; ++p) issue(p);
  float acc = 0.f;
  for (int cc = 0; cc < nchunks; ++cc) {
    cp_async_wait<STAGES - 2>();  // this thread's copies of chunk cc have landed
    __syncthreads();              // ... and everyone's; all threads are also done with the stage refilled next
    issue(cc + STAGES - 1);
    const float* row = reinterpret_cast<const float*>(s_tile + (cc % STAGES) * TILE4 + f * TL_ROW4) + j;
#pragma unroll
    for (int c = 0; c < TL_C; ++c) {
      const float x = row[c * 9];
      acc = __fadd_rn(acc, __fmul_rn(x, x));
    }
  }
  cp_async_wait<0>();
  s_tap[t] = acc;
  __syncthreads();
  if (worker && j == 0) {
    const float* s = &s_tap[t];
    float tot = 0.f;
    for (int ww = 0; ww < 3; ++ww) {
      float col = 0.f;
      for (int hh = 0; hh < 3; ++hh) col = __fadd_rn(col, s[hh * 3 + ww]);  // .sum(axis=1) over h, sequential
      tot = __fadd_rn(tot, col);                                            // final .sum(axis=1) over w (n<8)
    }
    values[lt.voff[l] + o0 + f] = __fdiv_rn(tot, (float)(C * 9));
  }
}

// blocks [0, n_tiled): tiled work items; the first `first_wave` items (largest C first) land one per SM, the remaining
// items are taken smallest-first so that an SM's second block complements its first.  Blocks beyond: generic path.
__global__ void __launch_bounds__(SS_THREADS) filter_sumsq_kernel(const LayerTable lt, float* __restrict__ values,
                                                                  int n_tiled, int first_wave) {
  extern __shared__ __align__(16) unsigned char dsm[];
  __shared__ float s_tap[SS_THREADS];
  if ((int)blockIdx.x < n_tiled) {
    int item = blockIdx.x;
    if (item >= first_wave) item = first_wave + (n_tiled - 1 - item);
    sumsq_tiled_block<TL_F, TL_STAGES>(lt, item, values, reinterpret_cast<float4*>(dsm), s_tap);
  } else {
    sumsq_generic_block<SS_THREADS>(lt, (int)blockIdx.x - n_tiled, values, s_tap, reinterpret_cast<float*>(dsm));
  }
}
constexpr size_t SUMSQ_SMEM = TL_STAGES * TL_TILE4 * sizeof(float4);  // 113,664 B
static_assert((size_t)(SS_THREADS / 32) * ROW_MAX * sizeof(float) <= SUMSQ_SMEM, "1x1 rows must fit the ring");

// ---- normalise, select, keep, fill: the steps after the sums, shared by the one-launch and three-launch paths ----------
// methods.py:46-51 for one layer's values v[0, O) by NT threads: a warp (NT = 32) or the whole block.  v /= sqrt(sum of
// v^2 in NumPy's pairwise order, run by the first warp), then v /= max(v).  The max of values >= 0 is the max of their
// bit patterns, and a NaN's pattern (sign cleared) beats every number's, so a NaN wins as in np.max.  s_red: NT / 32 + 1
// words (block only).  Returns whether the layer holds a NaN, uniform over the NT threads.
template <int NT>
__device__ bool normalise_layer(float* v, int O, unsigned int* s_red) {
  constexpr int WARPS = NT / 32;
  const int t = threadIdx.x % NT, lane = threadIdx.x & 31;
  float nrm;
  if constexpr (WARPS == 1) {
    nrm = __fsqrt_rn(warp_pairwise_sumsq(v, O));
  } else {
    if (t < 32) {
      const float s = warp_pairwise_sumsq(v, O);
      if (t == 0) s_red[WARPS] = __float_as_uint(__fsqrt_rn(s));
    }
    __syncthreads();
    nrm = __uint_as_float(s_red[WARPS]);
  }
  unsigned int mb = 0u;
  for (int i = t; i < O; i += NT) {
    const float x = __fdiv_rn(v[i], nrm);
    v[i] = x;
    mb = max(mb, __float_as_uint(x) & 0x7fffffffu);
  }
  mb = __reduce_max_sync(0xffffffffu, mb);
  if constexpr (WARPS > 1) {
    if (lane == 0) s_red[t >> 5] = mb;
    __syncthreads();
    mb = __reduce_max_sync(0xffffffffu, lane < WARPS ? s_red[lane] : 0u);
  }
  const float mx = __uint_as_float(mb);
  int nan = 0;
  for (int i = t; i < O; i += NT) {
    const float x = __fdiv_rn(v[i], mx);
    v[i] = x;
    nan |= x != x;
  }
  if constexpr (WARPS == 1) return __any_sync(0xffffffffu, nan) != 0;
  else return __syncthreads_or(nan) != 0;
}

__device__ __forceinline__ void warp_find_bin(const unsigned int* hist, unsigned int rank, unsigned int* out_bin,
                                              unsigned int* out_rem) {
  const int lane = threadIdx.x & 31;
  unsigned int c[8], tot = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) { c[j] = hist[lane * 8 + j]; tot += c[j]; }
  unsigned int incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const unsigned int excl = incl - tot;
  const bool mine = (rank >= excl) && (rank < incl);
  const unsigned int who = __ballot_sync(0xffffffffu, mine);
  const int src = who ? (__ffs(who) - 1) : 31;  // rank beyond the total: clamp (caller validates)
  if (lane == src) {
    unsigned int cum = excl, b = 0;
    for (; b < 7; ++b) {
      if (cum + c[b] > rank) break;
      cum += c[b];
    }
    *out_bin = lane * 8 + b;
    *out_rem = rank - cum;
  }
}


// np.percentile over the n normalised values in shared memory, by the NT threads of the block: the order statistics k and k+1 (both at once), then
// NumPy's float64 _lerp.  The values of a layer crowd into a handful of exponents, so the top byte of the bit patterns
// is resolved by 7 rounds of counting "keys below prefix|bit" (a shared-memory histogram would serialise 32-way on
// those few bins: measured 10 us for that pass alone); the three lower bytes, which are well spread, by 8-bit radix
// passes with shared-memory atomics (one histogram per rank).  Every thread returns the threshold.
template <int NT>
__device__ double select_percentile(const float* s_val, int n, long long k, double gamma, unsigned int* s_hist /*[2][256]*/,
                               unsigned int* s_bin /*[4]*/) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  constexpr int WARPS = NT / 32;
  const long long k1 = (k + 1 < n) ? k + 1 : (long long)n - 1;
  unsigned int rank[2] = {(unsigned int)k, (unsigned int)k1};
  unsigned int prefix[2] = {0, 0};
  unsigned int* s_part = s_hist;  // [2 parities][2 ranks][WARPS] partial counts of the counting rounds
  for (int bit = 30, r = 0; bit >= 24; --bit, ++r) {  // keys < 2^31
    const unsigned int c0 = prefix[0] | (1u << bit), c1 = prefix[1] | (1u << bit);
    unsigned int n0 = 0, n1 = 0;
    for (int i = tid; i < n; i += NT) {
      const unsigned int key = __float_as_uint(s_val[i]);
      n0 += key < c0;
      n1 += key < c1;
    }
    n0 = __reduce_add_sync(0xffffffffu, n0);
    n1 = __reduce_add_sync(0xffffffffu, n1);
    unsigned int* part = s_part + (r & 1) * 2 * WARPS;
    if (lane == 0) {
      part[wid] = n0;
      part[WARPS + wid] = n1;
    }
    __syncthreads();  // (slots alternate by round parity: one barrier per round)
    const unsigned int t0 = __reduce_add_sync(0xffffffffu, lane < WARPS ? part[lane] : 0u);
    const unsigned int t1 = __reduce_add_sync(0xffffffffu, lane < WARPS ? part[WARPS + lane] : 0u);
    if (t0 <= (unsigned int)k) prefix[0] = c0;   // at most k keys below the candidate: the k-th smallest is >= candidate
    if (t1 <= (unsigned int)k1) prefix[1] = c1;
  }
  {  // ranks relative to the keys that share the top byte: subtract the keys below the prefix
    unsigned int n0 = 0, n1 = 0;
    for (int i = tid; i < n; i += NT) {
      const unsigned int key = __float_as_uint(s_val[i]);
      n0 += key < prefix[0];
      n1 += key < prefix[1];
    }
    n0 = __reduce_add_sync(0xffffffffu, n0);
    n1 = __reduce_add_sync(0xffffffffu, n1);
    __syncthreads();
    if (lane == 0) {
      s_part[wid] = n0;
      s_part[WARPS + wid] = n1;
    }
    __syncthreads();
    rank[0] -= __reduce_add_sync(0xffffffffu, lane < WARPS ? s_part[lane] : 0u);
    rank[1] -= __reduce_add_sync(0xffffffffu, lane < WARPS ? s_part[WARPS + lane] : 0u);
    __syncthreads();
  }
  unsigned int mask = 0xff000000u;
  for (int shift = 16; shift >= 0; shift -= 8) {
    for (int i = tid; i < 512; i += NT) s_hist[i] = 0;
    __syncthreads();
    const bool same = prefix[0] == prefix[1];  // block-uniform: one histogram serves both ranks while they agree
    for (int i = tid; i < n; i += NT) {
      const unsigned int key = __float_as_uint(s_val[i]);
      const unsigned int d = (key >> shift) & 255u;
      if ((key & mask) == prefix[0]) atomicAdd(&s_hist[d], 1u);
      else if (!same && (key & mask) == prefix[1]) atomicAdd(&s_hist[256 + d], 1u);
    }
    __syncthreads();
    if (wid == 0) warp_find_bin(s_hist, rank[0], &s_bin[0], &s_bin[2]);
    if (wid == 1) warp_find_bin(same ? s_hist : s_hist + 256, rank[1], &s_bin[1], &s_bin[3]);
    __syncthreads();
    prefix[0] |= s_bin[0] << shift;
    prefix[1] |= s_bin[1] << shift;
    rank[0] = s_bin[2];
    rank[1] = s_bin[3];
    mask |= 255u << shift;
    __syncthreads();
  }
  const double a = (double)__uint_as_float(prefix[0]);
  const double b = (double)__uint_as_float(prefix[1]);
  const double diff = __dsub_rn(b, a);
  double r = __dadd_rn(a, __dmul_rn(diff, gamma));
  if (gamma >= 0.5) r = __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, gamma)));
  return r;
}

// methods.py:75: a filter is pruned when its value is below the float64 threshold (nothing is below a NaN threshold).
__device__ __forceinline__ bool kept(float v, double thr) { return !((double)v < thr); }

// One filter's mask (per floats at m) set to val by the NT threads of a block: scalar head up to 16-byte alignment,
// 128-bit streaming stores, scalar tail.
template <int NT>
__device__ void fill_filter(float* m, int per, float val) {
  const int tid = threadIdx.x;
  int head = (int)(((16 - (reinterpret_cast<uintptr_t>(m) & 15)) & 15) >> 2);
  if (head > per) head = per;
  if (tid < head) m[tid] = val;
  const int body4 = (per - head) >> 2;
  float4* m4 = reinterpret_cast<float4*>(m + head);
  const float4 v4 = make_float4(val, val, val, val);
  for (int i = tid; i < body4; i += NT) st_stream_f4(m4 + i, v4);
  const int tail0 = head + body4 * 4;
  if (tid < per - tail0) m[tail0 + tid] = val;
}

// ---- three launches (sums, finish, mask fill): more filters than the fused kernel holds, and the values alone -------
// One block per layer normalises it.  With k >= 0 the last block to finish then selects the float64 percentile over all
// n values and writes the threshold and the keep flags; with k < 0 it stops at the values (mc_filter_values).
constexpr int FIN_THREADS = 1024;
constexpr size_t FIN_MAX_SMEM = 200 * 1024;  // max(O_l, n) floats: up to 51,200 filters

__global__ void __launch_bounds__(FIN_THREADS) filter_finish_kernel(const LayerTable lt, float* __restrict__ values,
                                                                    long long k, double gamma, double* __restrict__ thr,
                                                                    uint8_t* __restrict__ keep,
                                                                    unsigned int* __restrict__ ticket) {
  extern __shared__ __align__(16) unsigned char dsm[];
  float* s_v = reinterpret_cast<float*>(dsm);  // max(O_l, n) floats
  __shared__ unsigned int s_red[FIN_THREADS / 32 + 1];
  __shared__ unsigned int s_hist[512], s_bin[4];
  __shared__ unsigned int s_last;
  const int O = lt.O[blockIdx.x];
  float* v = values + lt.voff[blockIdx.x];
  for (int o = threadIdx.x; o < O; o += FIN_THREADS) s_v[o] = v[o];
  __syncthreads();
  normalise_layer<FIN_THREADS>(s_v, O, s_red);
  for (int o = threadIdx.x; o < O; o += FIN_THREADS) v[o] = s_v[o];
  if (k < 0) return;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int n = lt.voff[lt.nlayers];
  int nan = 0;
  for (int i = threadIdx.x; i < n; i += FIN_THREADS) {
    const float x = __ldcg(values + i);
    s_v[i] = x;
    nan |= x != x;
  }
  // np.percentile returns nan if any value is nan (an all-zero layer gives 0/0): nothing is < nan
  const double t = __syncthreads_or(nan) ? __longlong_as_double(0x7ff8000000000000LL)
                                         : select_percentile<FIN_THREADS>(s_v, n, k, gamma, s_hist, s_bin);
  if (threadIdx.x == 0) *thr = t;
  if (keep)
    for (int i = threadIdx.x; i < n; i += FIN_THREADS) keep[i] = kept(s_v[i], t) ? 1 : 0;
}

// one block per filter (grid-stride)
__global__ void __launch_bounds__(256) filter_mask_fill_kernel(const LayerTable lt, const float* __restrict__ v,
                                                               const double* __restrict__ thr) {
  const double t = *thr;
  const int nfilters = lt.voff[lt.nlayers];
  for (int f = blockIdx.x; f < nfilters; f += gridDim.x) {
    int l = 0;
    while (l + 1 < lt.nlayers && f >= lt.voff[l + 1]) ++l;
    const int per = lt.C[l] * lt.taps[l];
    fill_filter<256>(lt.mask[l] + (long long)(f - lt.voff[l]) * per, per, kept(v[f], t) ? 1.f : 0.f);
  }
}

// ---- the whole of quick_filter_prune in ONE cooperative launch ------------------------------------------------------
// Persistent blocks (2 per SM, all co-resident) take work items from an atomic queue: groups of FU_F filters of the 3x3
// layers through a 6-stage cp.async ring, and the blocks of the generic path (1x1 layers) slotted in behind the long
// items so that their latency-bound work does not form the tail.  Raw per-filter sums go to a scratch array.  The block
// that completes the last item (the finisher) pulls all raw sums (42 KB for Darknet-19) from L2 into shared memory, runs
// the serial part alone — per-layer normalisation in NumPy's pairwise order, then the two-rank select for
// np.percentile — writes the values and keep flags and publishes the threshold through a flag.  The other blocks fill
// their masks with the provisional value meanwhile and rewrite the filters that differ once the flag is up.  Against
// three launches this removes two full drains + ramps of the grid (~30 us of pure latency between the two bandwidth
// passes).
constexpr int FU_THREADS = 160;  // 16 filters x 9 taps = 144 chain threads, rounded up to whole warps
constexpr int FU_F = 16;
constexpr int FU_STAGES = 6;
constexpr size_t FU_SMEM = (size_t)FU_STAGES * FU_F * TL_ROW4 * sizeof(float4);  // 113,664 B: two blocks per SM
constexpr int FU_AUX_BYTES = 8192;                                                // behind the values: histograms
constexpr int FU_MAX_N = (int)((FU_SMEM - FU_AUX_BYTES) / sizeof(float));         // 26,368 filters
static_assert((size_t)(FU_THREADS / 32) * ROW_MAX * sizeof(float) <= FU_SMEM, "1x1 rows must fit the ring");

struct FusedState {
  unsigned int next_item;  // work queue
  unsigned int pad0[31];
  unsigned int items_done;
  unsigned int pad1[31];
  unsigned int flag;  // polled by idle blocks: its own 128-byte line
  unsigned int pad2[31];
  unsigned long long stamp[8];  // diagnostics (globaltimer ns): block 0 start, last block out of work, last block past the
                                // wait, last block with thr, last block done
};
__device__ __forceinline__ void fused_stamp(FusedState* st, int i, bool max_over_blocks) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  if (max_over_blocks) atomicMax(&st->stamp[i], t);
  else st->stamp[i] = t;
}

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// All raw sums -> normalised values s_val [n] in shared memory (methods.py:43-51 for every layer), by one block: one
// warp per layer.  Returns true (block-uniform) if any value is NaN.
template <int NT>
__device__ bool fused_normalise_all(const LayerTable& lt, const float* __restrict__ raw, float* s_val) {
  const int n = lt.voff[lt.nlayers];
  const int tid = threadIdx.x;
  for (int i0 = 0; i0 < n; i0 += 16 * NT) {  // 16 independent L2 loads in flight per thread
    float x[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int i = i0 + u * NT + tid;
      x[u] = i < n ? __ldcg(raw + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int i = i0 + u * NT + tid;
      if (i < n) s_val[i] = x[u];
    }
  }
  __syncthreads();
  int nan = 0;
  for (int l = tid >> 5; l < lt.nlayers; l += NT / 32) nan |= normalise_layer<32>(s_val + lt.voff[l], lt.O[l], nullptr);
  return __syncthreads_or(nan) != 0;
}

__global__ void __launch_bounds__(FU_THREADS, 2)
filter_prune_fused_kernel(const LayerTable lt, float* __restrict__ raw, float* __restrict__ values, int n_tiled, int n_big,
                          int n_items, long long k, double gamma, double* __restrict__ thr, uint8_t* __restrict__ keep,
                          FusedState* st, int fill) {
  extern __shared__ __align__(16) unsigned char dsm[];
  __shared__ float s_tap[FU_THREADS];
  __shared__ unsigned int s_bin[4];
  __shared__ int s_item;
  __shared__ unsigned int s_last;
  const int tid = threadIdx.x;
  const int n = lt.voff[lt.nlayers];
  if (tid == 0 && blockIdx.x == 0) fused_stamp(st, 0, false);
  if (tid == 0) s_last = 0u;  // (a block that never gets an item is not the finisher)
  __syncthreads();
  // ---- phase 1: raw per-filter sums
  for (;;) {
    if (tid == 0) s_item = (int)atomicAdd(&st->next_item, 1u);
    __syncthreads();
    const int qpos = s_item;
    __syncthreads();
    if (qpos >= n_items) break;
    // queue order: the long tiled items (C >= 1024, one per block: the bandwidth-bound bulk), then the short generic
    // blocks (1x1 layers: latency-bound, hidden behind the bulk instead of forming the tail), then the short tiled items
    const int n_generic = n_items - n_tiled;
    const int item = qpos < n_big ? qpos : (qpos < n_big + n_generic ? n_tiled + (qpos - n_big) : qpos - n_generic);
    if (item < n_tiled)
      sumsq_tiled_block<FU_F, FU_STAGES>(lt, item, raw, reinterpret_cast<float4*>(dsm), s_tap);
    else
      sumsq_generic_block<FU_THREADS>(lt, item - n_tiled, raw, s_tap, reinterpret_cast<float*>(dsm));
    __threadfence();  // this block's sums are visible device-wide before it counts the item in
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(&st->items_done, 1u) == (unsigned int)n_items - 1u) ? 1u : 0u;
    __syncthreads();
    const bool finisher = s_last != 0u;  // block-uniform: this block completed the LAST item
    __syncthreads();
    if (!finisher) continue;
    // ---- phase 2 (the finisher alone; every other block is out of work or about to be): all sums -> normalised values
    //      -> threshold, published for everyone
    __threadfence();
    if (tid == 0) fused_stamp(st, 2, false);
    float* s_val = reinterpret_cast<float*>(dsm);
    const bool any_nan = fused_normalise_all<FU_THREADS>(lt, raw, s_val);
    if (tid == 0) fused_stamp(st, 5, false);
    double t;
    if (any_nan) t = __longlong_as_double(0x7ff8000000000000LL);  // np.percentile returns nan: nothing is < nan
    else t = select_percentile<FU_THREADS>(s_val, n, k, gamma,
                                           reinterpret_cast<unsigned int*>(dsm + (FU_SMEM - FU_AUX_BYTES)), s_bin);
    for (int i = tid; i < n; i += FU_THREADS) {
      values[i] = s_val[i];
      if (keep) keep[i] = kept(s_val[i], t) ? 1 : 0;
    }
    if (tid == 0) *thr = t;
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      fused_stamp(st, 3, false);
      atomicExch(&st->flag, 1u);
    }
    __syncthreads();
  }
  if (tid == 0) fused_stamp(st, 1, true);
  if (!fill) return;
  // ---- phase 3: masks.  A block owns the filters blockIdx.x, blockIdx.x + gridDim.x, ... in both passes below.
  // While the finisher runs the serial part (normalise + percentile: ~38 us during which HBM would sit idle), every other
  // block already fills ITS filters with the PROVISIONAL value — the majority outcome, known from the rank alone: 1 when
  // fewer than half of the filters will be pruned, else 0 — and once the threshold is published only the filters whose
  // flag differs are rewritten (same thread, same addresses: ordered).  The finisher itself writes its filters once.
  const float prov = (2 * k < (long long)n) ? 1.f : 0.f;
  const bool i_finished = (s_last != 0u);  // block-uniform (s_last is only rewritten inside the queue loop)
  auto fill_filters = [&](int pass) {
    const double t = pass ? __ldcg(thr) : 0.0;
    int l = 0;
    for (int f = blockIdx.x; f < n; f += gridDim.x) {
      while (l + 1 < lt.nlayers && f >= lt.voff[l + 1]) ++l;
      float val = prov;
      if (pass) {
        val = kept(__ldcg(values + f), t) ? 1.f : 0.f;
        if (!i_finished && val == prov) continue;  // already written by the provisional pass
      }
      const int per = lt.C[l] * lt.taps[l];
      fill_filter<FU_THREADS>(lt.mask[l] + (long long)(f - lt.voff[l]) * per, per, val);
    }
  };
  if (!i_finished) fill_filters(0);
  if (tid == 0) {
    unsigned int spins = 0;
    while (ld_acquire_u32(&st->flag) == 0u) {
      __nanosleep(128);
      if (++spins > (1u << 26)) __trap();  // (a broken schedule must not hang the GPU)
    }
  }
  __syncthreads();
  fill_filters(1);
  if (tid == 0) fused_stamp(st, 4, true);
}

int build_layers(LayerTable* lt, const float* const* w, float* const* masks, const int* O, const int* C,
                 const int* taps, int nlayers, const char* who, int nt = SS_THREADS, int tl_f = TL_F) {
  if (nlayers <= 0 || nlayers > MAX_LAYERS) return mc_set_error(MC_ERR_ARG, "%s: nlayers %d out of range", who, nlayers);
  lt->nlayers = nlayers;
  lt->voff[0] = 0;
  lt->woff[0] = 0;
  lt->toff[0] = 0;
  for (int l = 0; l < nlayers; ++l) {
    if (O[l] <= 0 || C[l] <= 0 || taps[l] <= 0) return mc_set_error(MC_ERR_ARG, "%s: layer %d has bad dims", who, l);
    lt->w[l] = w[l];
    lt->mask[l] = masks ? masks[l] : nullptr;
    lt->O[l] = O[l];
    lt->C[l] = C[l];
    lt->taps[l] = taps[l];
    lt->voff[l + 1] = lt->voff[l] + O[l];
    // element offsets are rounded up to 4 so the vectorised mask fill never straddles two layers
    const long long sz = (long long)O[l] * C[l] * taps[l];
    lt->woff[l + 1] = lt->woff[l] + ((sz + 3) / 4) * 4;
    const long long thr = (taps[l] == 1) ? O[l] : (long long)O[l] * taps[l];
    // per-layer thread slots rounded up to whole blocks; for taps>1 a block must hold whole filters
    long long slots;
    if (taps[l] == 9 && (C[l] % TL_C) == 0 && (O[l] % tl_f) == 0) slots = 0;  // tiled path
    else if (taps[l] == 1) slots = ((thr * 32 + nt - 1) / nt) * nt;  // one warp per filter
    else {
      const int fpb = nt / taps[l];  // filters per block
      slots = (long long)((O[l] + fpb - 1) / fpb) * nt;
    }
    lt->toff[l + 1] = lt->toff[l] + (int)slots;
  }
  // tiled layers, largest C first (insertion sort; nlayers <= 64)
  lt->ntiled = 0;
  for (int l = 0; l < nlayers; ++l) {
    if (!(taps[l] == 9 && (C[l] % TL_C) == 0 && (O[l] % tl_f) == 0)) continue;
    int pos = lt->ntiled++;
    while (pos > 0 && C[lt->torder[pos - 1]] < C[l]) {
      lt->torder[pos] = lt->torder[pos - 1];
      --pos;
    }
    lt->torder[pos] = l;
  }
  lt->tblk[0] = 0;
  for (int i = 0; i < lt->ntiled; ++i) lt->tblk[i + 1] = lt->tblk[i] + O[lt->torder[i]] / tl_f;
  for (int i = lt->ntiled; i < MAX_LAYERS; ++i) {
    lt->torder[i] = 0;
    lt->tblk[i + 1] = lt->tblk[lt->ntiled];
  }
  for (int l = nlayers; l < MAX_LAYERS; ++l) {
    lt->w[l] = nullptr;
    lt->mask[l] = nullptr;
    lt->O[l] = lt->C[l] = lt->taps[l] = 0;
    lt->voff[l + 1] = lt->voff[nlayers];
    lt->woff[l + 1] = lt->woff[nlayers];
    lt->toff[l + 1] = lt->toff[nlayers];
  }
  return 0;
}

int launch_sumsq(const LayerTable& lt, float* d_values, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    MC_CUDA(cudaFuncSetAttribute(filter_sumsq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SUMSQ_SMEM));
    attr_set = true;
  }
  const int n_tiled = lt.tblk[lt.ntiled];
  const int n_generic = lt.toff[lt.nlayers] / SS_THREADS;
  const int first_wave = n_tiled < mc_num_sms() ? n_tiled : mc_num_sms();
  if (n_tiled + n_generic == 0) return 0;
  filter_sumsq_kernel<<<n_tiled + n_generic, SS_THREADS, SUMSQ_SMEM, stream>>>(lt, d_values, n_tiled, first_wave);
  MC_LAUNCH_CHECK("filter_sumsq_kernel");
  return 0;
}

// filter_finish_kernel over the n values of lt: k < 0 normalises them only, k >= 0 also selects (d_ticket zeroed).
int launch_finish(const LayerTable& lt, float* d_values, long long k, double gamma, double* d_thr, uint8_t* d_keep,
                  unsigned int* d_ticket, cudaStream_t stream, const char* who) {
  const int n = lt.voff[lt.nlayers];
  int staged = k >= 0 ? n : 0;
  for (int l = 0; l < lt.nlayers; ++l) staged = lt.O[l] > staged ? lt.O[l] : staged;
  const size_t smem = (size_t)staged * sizeof(float);
  if (smem > FIN_MAX_SMEM) return mc_set_error(MC_ERR_SHAPE, "%s: %d filters exceed the single-block finish", who, staged);
  static size_t attr = 0;
  if (smem > attr) {
    MC_CUDA(cudaFuncSetAttribute(filter_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  filter_finish_kernel<<<lt.nlayers, FIN_THREADS, smem, stream>>>(lt, d_values, k, gamma, d_thr, d_keep, d_ticket);
  MC_LAUNCH_CHECK("filter_finish_kernel");
  return 0;
}

int launch_mask_fill(const LayerTable& lt, const float* d_v, const double* d_thr, cudaStream_t stream) {
  int blocks = lt.voff[lt.nlayers];
  const int cap = mc_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  filter_mask_fill_kernel<<<blocks, 256, 0, stream>>>(lt, d_v, d_thr);
  MC_LAUNCH_CHECK("filter_mask_fill_kernel");
  return 0;
}
}  // namespace

extern "C" int mc_filter_values(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh,
                                const int* h_kw, int nlayers, float* d_values, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(h_w_ptrs && h_O && h_C && h_kh && h_kw && d_values, "mc_filter_values: null pointer");
  MC_CHECK_ARG(nlayers > 0 && nlayers <= MAX_LAYERS, "mc_filter_values: nlayers out of range");
  int taps[MAX_LAYERS];
  for (int l = 0; l < nlayers; ++l) {
    MC_CHECK_ARG(h_kh[l] == h_kw[l] && h_kh[l] >= 1 && h_kh[l] * h_kw[l] <= 49,
                 "mc_filter_values: layer %d kernel %dx%d unsupported (square, <=7x7)", l, h_kh[l], h_kw[l]);
    MC_CHECK_ARG(h_w_ptrs[l] != nullptr, "mc_filter_values: layer %d null weight", l);
    taps[l] = h_kh[l] * h_kw[l];
  }
  LayerTable lt;
  int rc = build_layers(&lt, h_w_ptrs, nullptr, h_O, h_C, taps, nlayers, "mc_filter_values");
  if (rc) return rc;
  rc = launch_sumsq(lt, d_values, stream);
  if (rc) return rc;
  return launch_finish(lt, d_values, -1, 0.0, nullptr, nullptr, nullptr, stream, "mc_filter_values");
}

/* The whole of quick_filter_prune in one call: ONE cooperative launch (filter_prune_fused_kernel); models with more
 * filters than its finisher block holds take the three-launch path.  See include/mcb200.h. */
extern "C" size_t mc_workspace_bytes_filter_prune(void) { return 2048 + (size_t)FU_MAX_N * sizeof(float); }
static_assert(sizeof(FusedState) <= 2048, "FusedState must fit the head of the filter-prune workspace");

extern "C" int mc_filter_prune(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh,
                               const int* h_kw, int nlayers, int64_t k, double gamma, float* d_values, double* d_thr,
                               float* const* h_mask_ptrs, uint8_t* d_keep, void* d_ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(h_w_ptrs && h_O && h_C && h_kh && h_kw && d_values && d_thr && d_ws, "mc_filter_prune: null pointer");
  MC_CHECK_ARG(nlayers > 0 && nlayers <= MAX_LAYERS, "mc_filter_prune: nlayers out of range");
  if (ws_bytes < mc_workspace_bytes_filter_prune()) return mc_set_error(MC_ERR_WS, "mc_filter_prune: workspace too small");
  int taps[MAX_LAYERS];
  long long n_all = 0;
  for (int l = 0; l < nlayers; ++l) {
    MC_CHECK_ARG(h_kh[l] == h_kw[l] && h_kh[l] >= 1 && h_kh[l] * h_kw[l] <= 49,
                 "mc_filter_prune: layer %d kernel %dx%d unsupported (square, <=7x7)", l, h_kh[l], h_kw[l]);
    MC_CHECK_ARG(h_w_ptrs[l] != nullptr, "mc_filter_prune: layer %d null weight", l);
    MC_CHECK_ARG(!h_mask_ptrs || h_mask_ptrs[l] != nullptr, "mc_filter_prune: null mask %d", l);
    taps[l] = h_kh[l] * h_kw[l];
    n_all += h_O[l];
  }
  // the fused kernel's work items are smaller than the three-launch path's: the table is built for the path taken
  const bool fused = n_all <= FU_MAX_N;
  LayerTable lt;
  int rc = build_layers(&lt, h_w_ptrs, h_mask_ptrs, h_O, h_C, taps, nlayers, "mc_filter_prune",
                        fused ? FU_THREADS : SS_THREADS, fused ? FU_F : TL_F);
  if (rc) return rc;
  const int n = lt.voff[nlayers];
  MC_CHECK_ARG(k >= 0 && k < n, "mc_filter_prune: rank out of range");
  MC_CHECK_ARG(gamma >= 0.0 && gamma < 1.0, "mc_filter_prune: gamma must be in [0,1)");
  if (fused) {
    static int max_blocks = -1;
    if (max_blocks < 0) {
      MC_CUDA(cudaFuncSetAttribute(filter_prune_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FU_SMEM));
      int per_sm = 0;
      MC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, filter_prune_fused_kernel, FU_THREADS, FU_SMEM));
      if (per_sm < 1) return mc_set_error(MC_ERR_SHAPE, "mc_filter_prune: fused kernel does not fit an SM");
      max_blocks = per_sm * mc_num_sms();
    }
    int n_tiled = lt.tblk[lt.ntiled];
    int n_items = n_tiled + lt.toff[lt.nlayers] / FU_THREADS;
    int n_big = 0;  // tiled items of the layers with >= 1024 input channels (torder is sorted by descending C)
    for (int i2 = 0; i2 < lt.ntiled && h_C[lt.torder[i2]] >= 1024; ++i2) n_big = lt.tblk[i2 + 1];
    int grid = n_items < max_blocks ? n_items : max_blocks;
    if (grid < 1) grid = 1;
    MC_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(FusedState), stream));
    long long kk = (long long)k;
    FusedState* stp = reinterpret_cast<FusedState*>(d_ws);
    float* d_raw = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(d_ws) + 2048);  // raw sums [n]
    int fill = h_mask_ptrs ? 1 : 0;
    void* args[] = {&lt, &d_raw, &d_values, &n_tiled, &n_big, &n_items, &kk, &gamma, &d_thr, &d_keep, &stp, &fill};
    MC_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(filter_prune_fused_kernel), dim3((unsigned)grid),
                                        dim3(FU_THREADS), args, FU_SMEM, stream));
    return 0;
  }
  MC_CUDA(cudaMemsetAsync(d_ws, 0, sizeof(unsigned int), stream));
  rc = launch_sumsq(lt, d_values, stream);
  if (!rc) rc = launch_finish(lt, d_values, (long long)k, gamma, d_thr, d_keep, reinterpret_cast<unsigned int*>(d_ws),
                              stream, "mc_filter_prune");
  if (!rc && h_mask_ptrs) rc = launch_mask_fill(lt, d_values, d_thr, stream);
  return rc;
}

// ---- greedy filter pruning: prune_one_filter / filter_prune (methods.py:81-142, arXiv:1611.06440) ----------------------
// The reference re-reads every weight for every filter it removes.  Surviving filters are only ever multiplied by 1.0,
// so a filter's raw value (mean of squares, step 1 of quick_filter_prune) and its count of nonzero weights are computed
// once (pass 1).  A pick sets one raw value to 0, which changes one leaf of its layer's pairwise sum of squares and
// therefore only that layer's norm and candidate: the greedy walk (pass 2) re-sums that leaf, replays the combine and
// rescans the one layer, in one warp with everything in shared memory.  Pass 3 fills the masks from the keep flags.
namespace {


// Nonzero weights per filter (-0.0 counts as zero, as `== 0` does in NumPy): one warp per filter.
__global__ void __launch_bounds__(256) filter_nonzero_kernel(const LayerTable lt, int* __restrict__ nz) {
  const int n = lt.voff[lt.nlayers];
  const int lane = threadIdx.x & 31;
  const int f = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (f >= n) return;
  int l = 0;
  while (l + 1 < lt.nlayers && f >= lt.voff[l + 1]) ++l;
  const int per = lt.C[l] * lt.taps[l];
  const float* w = lt.w[l] + (long long)(f - lt.voff[l]) * per;
  int head = (int)(((16 - (reinterpret_cast<uintptr_t>(w) & 15)) & 15) >> 2);  // scalar head up to 16-byte alignment
  if (head > per) head = per;
  int c = (lane < head && w[lane] != 0.f) ? 1 : 0;
  const int body4 = (per - head) >> 2;
  const float4* w4 = reinterpret_cast<const float4*>(w + head);
#pragma unroll 4
  for (int i = lane; i < body4; i += 32) {
    const float4 v = ld_stream_f4(w4 + i);
    c += (v.x != 0.f) + (v.y != 0.f) + (v.z != 0.f) + (v.w != 0.f);
  }
  for (int i = head + body4 * 4 + lane; i < per; i += 32) c += (w[i] != 0.f) ? 1 : 0;
  c = __reduce_add_sync(0xffffffffu, c);
  if (lane == 0) nz[f] = c;
}

constexpr int GR_THREADS = 256;
constexpr int GR_MAX_N = 20480;  // filters staged in shared memory: raw value, nonzero count, keep flag (9 bytes each)
// Leaves of the pairwise recursion: one per layer of <= 128 filters, otherwise every leaf is at least 57 long.
constexpr int GR_MAX_LEAVES = GR_MAX_N / 56 + 2 * MAX_LAYERS;
constexpr size_t GR_SMEM = (size_t)GR_MAX_N * 9;

enum { GR_DONE = 0, GR_BUDGET = 1, GR_NAN_PICK = 2, GR_NO_CANDIDATE = 3, GR_NONFINITE = 4 };

struct GreedyShared {
  int lst[GR_MAX_LEAVES], lln[GR_MAX_LEAVES];  // leaf (start, length) inside its layer
  float lsum[GR_MAX_LEAVES];                   // leaf sums of raw^2
  int loff[MAX_LAYERS + 1];                    // first leaf of each layer
  float cval[MAX_LAYERS];                      // per-layer arg_nonzero_min: value (inf when it reports (inf, inf))
  int cidx[MAX_LAYERS];                        // ... and index (-1 for (inf, inf))
};

// Layer l's norm from its leaf sums, v = raw / norm, and arg_nonzero_min(list(v)) (utils.py:96-120) by one warp:
// the start is the LAST entry with v != 0 (NaN != 0 too) and only a strict `<` replaces it, so that entry wins a tie
// for the minimum and otherwise the first index of the minimum wins; a NaN start is never replaced; no nonzero entry,
// or index 0 as the last one, reports (inf, inf).
__device__ void greedy_refresh_layer(const LayerTable& lt, int l, const float* s_raw, GreedyShared& g) {
  const int lane = threadIdx.x & 31, O = lt.O[l];
  const float nrm = __fsqrt_rn(np_combine_leaves(g.lsum + g.loff[l], O));
  const float* r = s_raw + lt.voff[l];
  int last = -1, im = INT_MAX;
  float m = INFINITY;
  for (int i = lane; i < O; i += 32) {
    const float v = __fdiv_rn(r[i], nrm);
    if (v != 0.f) {
      last = i;
      if (v == v && (im == INT_MAX || v < m)) { m = v; im = i; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, im, o);
    if (i2 != INT_MAX && (im == INT_MAX || m2 < m || (m2 == m && i2 < im))) { m = m2; im = i2; }
  }
  if (lane == 0) {
    float cv = INFINITY;
    int ci = -1;
    if (last > 0) {
      const float vl = __fdiv_rn(r[last], nrm);
      if (vl == vl && m < vl) { cv = m; ci = im; }
      else { cv = vl; ci = last; }
    }
    g.cval[l] = cv;
    g.cidx[l] = ci;
  }
  __syncwarp();
}

// Pass 2 in one block.  Per pick (warp 0): np.argmin over the per-layer values (the first NaN, else the first minimum),
// record (filter, nonzero count), count the zeros, then the stop test exactly as filter_prune evaluates it (float64
// 100. * zeros / total < perc), after the pick: the reference starts from a rate of 0 and always prunes once.
__global__ void __launch_bounds__(GR_THREADS) filter_greedy_kernel(const LayerTable lt, const float* __restrict__ raw,
                                                                   const int* __restrict__ nz, long long zeros0,
                                                                   long long total, double perc, int max_picks,
                                                                   int2* __restrict__ picks, long long* __restrict__ result,
                                                                   float* __restrict__ keepf, double* __restrict__ half) {
  extern __shared__ __align__(16) unsigned char dsm[];
  __shared__ GreedyShared g;
  const int n = lt.voff[lt.nlayers], nl = lt.nlayers;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  float* s_raw = reinterpret_cast<float*>(dsm);
  int* s_nz = reinterpret_cast<int*>(s_raw + n);
  uint8_t* s_keep = reinterpret_cast<uint8_t*>(s_nz + n);
  int bad = 0;
  for (int i = tid; i < n; i += GR_THREADS) {
    const float x = raw[i];
    s_raw[i] = x;
    s_nz[i] = nz[i];
    s_keep[i] = 1;
    bad |= !isfinite(x);
  }
  if (tid == 0) {
    g.loff[0] = 0;
    for (int l = 0; l < nl; ++l) {
      int leaves = 1;
      for (NpWalk w(lt.O[l]); w.next(0.f);) ++leaves;
      g.loff[l + 1] = g.loff[l] + leaves;
    }
  }
  if (__syncthreads_or(bad)) {
    if (tid == 0) {
      result[0] = 0;
      result[1] = zeros0;
      result[2] = GR_NONFINITE;
    }
    return;
  }
  // leaf tables and sums, norms and candidates of every layer: one warp per layer
  for (int l = wid; l < nl; l += GR_THREADS / 32) {
    const int base = g.loff[l];
    if (lane == 0) {
      NpWalk w(lt.O[l]);
      for (int k = base;; ++k) {
        g.lst[k] = w.st;
        g.lln[k] = w.ln;
        if (!w.next(0.f)) break;
      }
    }
    __syncwarp();
    const float* r = s_raw + lt.voff[l];
    for (int k0 = base; k0 < g.loff[l + 1]; k0 += 4) {  // four leaves at a time
      const int k = k0 + (lane >> 3);
      const bool have = k < g.loff[l + 1];
      const float s = group_leaf_sumsq(r + (have ? g.lst[k] : 0), have ? g.lln[k] : 0);
      if (have && (lane & 7) == 0) g.lsum[k] = s;
    }
    __syncwarp();
    greedy_refresh_layer(lt, l, s_raw, g);
  }
  __syncthreads();
  if (wid == 0) {
    long long zeros = zeros0;
    int npick = 0, status = GR_BUDGET;
    for (;;) {
      float bv = INFINITY;
      int bl = INT_MAX;
      for (int l = lane; l < nl; l += 32) {  // ascending l: a later layer only wins with a NaN or a smaller value
        const float v = g.cval[l];
        if (bl == INT_MAX || (v != v && bv == bv) || (bv == bv && v < bv)) { bv = v; bl = l; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
        const int l2 = __shfl_xor_sync(0xffffffffu, bl, o);
        bool take;
        if (l2 == INT_MAX) take = false;
        else if (bl == INT_MAX) take = true;
        else if ((v2 != v2) != (bv != bv)) take = v2 != v2;
        else if (v2 != v2) take = l2 < bl;
        else take = v2 < bv || (v2 == bv && l2 < bl);
        if (take) { bv = v2; bl = l2; }
      }
      const int ci = g.cidx[bl];
      if (ci < 0) {  // every layer reports (inf, inf): int(inf) raises in the reference
        status = GR_NO_CANDIDATE;
        break;
      }
      const int f = lt.voff[bl] + ci;
      const int c = s_nz[f];
      zeros += c;
      __syncwarp();
      if (lane == 0) {
        picks[npick] = make_int2(f, c);
        s_nz[f] = 0;
        s_keep[f] = 0;
      }
      ++npick;
      if (!(__ddiv_rn(__dmul_rn(100.0, (double)zeros), (double)total) < perc)) {
        status = GR_DONE;
        break;
      }
      if (npick >= max_picks) break;
      if (bv != bv) {  // a NaN pick leaves every value as it was: the reference repeats it forever
        status = GR_NAN_PICK;
        break;
      }
      if (lane == 0) s_raw[f] = 0.f;
      __syncwarp();
      int leaf = -1;
      for (int k0 = g.loff[bl]; k0 < g.loff[bl + 1] && leaf < 0; k0 += 32) {
        const int k = k0 + lane;
        const unsigned int hit = __ballot_sync(0xffffffffu, k < g.loff[bl + 1] && g.lst[k] <= ci &&
                                                                ci < g.lst[k] + g.lln[k]);
        if (hit) leaf = k0 + __ffs(hit) - 1;
      }
      const float s = group_leaf_sumsq(s_raw + lt.voff[bl] + g.lst[leaf], g.lln[leaf]);
      if (lane == 0) g.lsum[leaf] = s;
      __syncwarp();
      greedy_refresh_layer(lt, bl, s_raw, g);
    }
    if (lane == 0) {
      result[0] = npick;
      result[1] = zeros;
      result[2] = status;
    }
  }
  __syncthreads();
  // keep flags as the 0 / 1 values the mask fill kernel compares against 0.5
  for (int i = tid; i < n; i += GR_THREADS) keepf[i] = s_keep[i] ? 1.f : 0.f;
  if (tid == 0) *half = 0.5;
}

}  // namespace

static size_t greedy_ws_offset(int n, int part) {  // workspace: raw f32 [n] | nonzero counts i32 [n] | keep f32 [n] | 0.5
  return (size_t)part * (((size_t)n * 4 + 15) / 16 * 16);
}

extern "C" size_t mc_workspace_bytes_filter_prune_greedy(int n_filters) {
  return n_filters > 0 ? greedy_ws_offset(n_filters, 3) + 16 : 0;
}

extern "C" int mc_filter_prune_greedy(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh,
                                      const int* h_kw, int nlayers, int64_t zeros0, int64_t total_params, double perc,
                                      int max_picks, int32_t* d_picks, int64_t* d_result, float* const* h_mask_ptrs,
                                      void* d_ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(h_w_ptrs && h_O && h_C && h_kh && h_kw && d_picks && d_result && d_ws,
               "mc_filter_prune_greedy: null pointer");
  MC_CHECK_ARG(nlayers > 0 && nlayers <= MAX_LAYERS, "mc_filter_prune_greedy: nlayers %d out of range", nlayers);
  int taps[MAX_LAYERS];
  for (int l = 0; l < nlayers; ++l) {
    MC_CHECK_ARG(h_kh[l] == h_kw[l] && h_kh[l] >= 1 && h_kh[l] * h_kw[l] <= 49,
                 "mc_filter_prune_greedy: layer %d kernel %dx%d unsupported (square, <=7x7)", l, h_kh[l], h_kw[l]);
    MC_CHECK_ARG(h_w_ptrs[l] != nullptr, "mc_filter_prune_greedy: layer %d null weight", l);
    MC_CHECK_ARG(!h_mask_ptrs || h_mask_ptrs[l] != nullptr, "mc_filter_prune_greedy: null mask %d", l);
    taps[l] = h_kh[l] * h_kw[l];
  }
  LayerTable lt;
  int rc = build_layers(&lt, h_w_ptrs, h_mask_ptrs, h_O, h_C, taps, nlayers, "mc_filter_prune_greedy");
  if (rc) return rc;
  const int n = lt.voff[nlayers];
  if (n > GR_MAX_N)
    return mc_set_error(MC_ERR_SHAPE, "mc_filter_prune_greedy: %d filters exceed the %d the greedy walk holds", n, GR_MAX_N);
  MC_CHECK_ARG(max_picks >= 1 && max_picks <= n, "mc_filter_prune_greedy: max_picks %d out of range [1, %d]", max_picks, n);
  MC_CHECK_ARG(total_params > 0 && zeros0 >= 0 && zeros0 <= total_params,
               "mc_filter_prune_greedy: zeros0 / total_params out of range");
  if (ws_bytes < mc_workspace_bytes_filter_prune_greedy(n))
    return mc_set_error(MC_ERR_WS, "mc_filter_prune_greedy: workspace too small");
  unsigned char* ws = reinterpret_cast<unsigned char*>(d_ws);
  float* d_raw = reinterpret_cast<float*>(ws);
  int* d_nz = reinterpret_cast<int*>(ws + greedy_ws_offset(n, 1));
  float* d_keepf = reinterpret_cast<float*>(ws + greedy_ws_offset(n, 2));
  double* d_half = reinterpret_cast<double*>(ws + greedy_ws_offset(n, 3));
  static bool attr_set = false;
  if (!attr_set) {
    MC_CUDA(cudaFuncSetAttribute(filter_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GR_SMEM));
    attr_set = true;
  }
  rc = launch_sumsq(lt, d_raw, stream);
  if (rc) return rc;
  filter_nonzero_kernel<<<(n + 7) / 8, 256, 0, stream>>>(lt, d_nz);
  MC_LAUNCH_CHECK("filter_nonzero_kernel");
  filter_greedy_kernel<<<1, GR_THREADS, (size_t)n * 9, stream>>>(
      lt, d_raw, d_nz, (long long)zeros0, (long long)total_params, perc, max_picks, reinterpret_cast<int2*>(d_picks),
      reinterpret_cast<long long*>(d_result), d_keepf, d_half);
  MC_LAUNCH_CHECK("filter_greedy_kernel");
  return h_mask_ptrs ? launch_mask_fill(lt, d_keepf, d_half, stream) : 0;
}

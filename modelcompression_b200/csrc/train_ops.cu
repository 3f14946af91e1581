// train_ops.cu — batch-statistics BatchNorm, leaky-ReLU and max-pool pieces of the masked retrain step.
//
// Replaces, for the training-mode forward/backward of src/train.py:221-235 on the Darknet of src/nets.py:779-822:
// nn.BatchNorm2d in training mode (batch mean / biased variance, eps 1e-5, running stats momentum 0.1),
// nn.LeakyReLU(0.1), nn.MaxPool2d(2,2) and their autograd backward.  Convolutions (forward, dgrad, wgrad) are the
// tensor-core kernels in conv_tcgen05.cu / conv_wgrad.cu; these kernels are the HBM-bound glue between them.
//
// All activations/gradients are PNHWC bf16 ([rows, ld]; pad rows/columns hold zeros), per-channel statistics fp32.
#include "common.cuh"

namespace {

constexpr int TB = 256;
constexpr int MAX_C = 8 * TB;  // one channel octet per thread of a block

// ---- BN finalize: batch mean / biased var -> (scale, shift, mean, invstd); running stats update --------------------
__global__ void bn_finalize_kernel(const float* __restrict__ sum, const float* __restrict__ sumsq, int C, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                                   float* __restrict__ invstd_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double m = (double)sum[c] / count;
  double var = (double)sumsq[c] / count - m * m;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - (float)m * sc;
  mean_out[c] = (float)m;
  invstd_out[c] = invstd;
  if (running_mean) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

// ---- 8 channels ("an octet") = one 16-byte access per thread ----------------------------------------------------
// Octet mapping of every pass below: a block has O8 * floor(TB / O8) threads (O8 = ceil(C / 8) octets per row; TB for
// every power of two), and thread t keeps octet t % O8 for the whole launch while it walks rows (pooled pixels for the
// pool passes) row0, row0 + stride, ...  Its per-channel constants and accumulators live in registers, consecutive
// threads touch consecutive 16-byte pieces of a row, and the threads that share an octet sit O8 apart in the block.
struct OctetWalk {
  int c0;                         // first channel of the thread's octet
  unsigned int row0, stride;
};
__device__ __forceinline__ OctetWalk octet_walk(int O8) {
  const unsigned int rows_per_block = blockDim.x / O8, q = threadIdx.x / O8;
  return {(int)(threadIdx.x - q * O8) * 8, blockIdx.x * rows_per_block + q, gridDim.x * rows_per_block};
}
inline int octet_threads(int O8) { return O8 * (TB / O8); }

// A ragged last octet (C % 8 != 0, the WHOLE = false instantiations): per-channel vectors read as 0 past C, stores
// only below C (the columns past C may belong to a neighbouring concat slice), and accesses that are not 16-byte
// aligned (Reorg quadrants q*C) go element by element.  n = C - c0 channels are left in the octet.
template <bool WHOLE>
__device__ __forceinline__ void load_ch(const float* __restrict__ p, int c0, int C, float (&v)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = (WHOLE || c0 + j < C) ? p[c0 + j] : 0.f;
}
template <bool WHOLE>
__device__ __forceinline__ uint4 load8(const __nv_bfloat16* p, bool aligned, int n) {
  if constexpr (!WHOLE) {
    if (!aligned) {
      unsigned int h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = j < n ? __bfloat16_as_ushort(p[j]) : 0u;
      return make_uint4(h[0] | h[1] << 16, h[2] | h[3] << 16, h[4] | h[5] << 16, h[6] | h[7] << 16);
    }
  }
  return *reinterpret_cast<const uint4*>(p);
}
__device__ __forceinline__ void unpack8(const uint4& q, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 v = __bfloat1622float2(h[j]);
    f[2 * j] = v.x;
    f[2 * j + 1] = v.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 q;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
  return q;
}
template <bool WHOLE>
__device__ __forceinline__ void store8(__nv_bfloat16* p, bool aligned, int n, const float (&f)[8]) {
  if constexpr (!WHOLE) {
    if (!aligned || n < 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < n) p[j] = __float2bfloat16_rn(f[j]);
      return;
    }
  }
  *reinterpret_cast<uint4*>(p) = pack8(f);
}

// sum[c] += the block's partials a[c] (sumsq[c] += b[c] unless sumsq is NULL): one atomic per channel and block, the
// threads of a channel added in thread order.  Channels >= C (a ragged last octet) are dropped.
__device__ __forceinline__ void block_col_sums(const float (&a)[8], const float (&b)[8], int O8, int C,
                                               float* __restrict__ sum, float* __restrict__ sumsq) {
  __shared__ float s_a[TB][9], s_b[TB][9];  // padded rows: conflict-free column sums
#pragma unroll
  for (int j = 0; j < 8; ++j) { s_a[threadIdx.x][j] = a[j]; s_b[threadIdx.x][j] = b[j]; }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int o = c >> 3, j = c & 7;
    float ta = 0.f, tb = 0.f;
    for (int t = o; t < (int)blockDim.x; t += O8) { ta += s_a[t][j]; tb += s_b[t][j]; }
    atomicAdd(&sum[c], ta);
    if (sumsq) atomicAdd(&sumsq[c], tb);
  }
}

// Division by a run-time constant without the ~30-instruction integer divide (these kernels issue three per 16 bytes
// and were instruction-bound): q = umulhi(n, mul) >> shr, exact for n < 2^31 and d >= 2 (mul = ceil(2^(31+ceil_log2 d) / d)).
struct FastDiv {
  unsigned int d, mul, shr;
};
inline FastDiv make_fastdiv(unsigned int d) {
  FastDiv f;
  f.d = d;
  unsigned int l = 0;
  while ((1u << l) < d) ++l;
  const unsigned long long p = 31ull + l;
  f.mul = (unsigned int)((((unsigned long long)1 << p) + d - 1) / d);
  f.shr = (unsigned int)(p - 32);
  return f;
}
__device__ __forceinline__ unsigned int fdiv(unsigned int n, const FastDiv& f) { return __umulhi(n, f.mul) >> f.shr; }

// row -> (b, y, x) with 32-bit arithmetic; returns interior flag
__device__ __forceinline__ bool row_coords(unsigned int row, const FastDiv& Wp, const FastDiv& Hp, int H, int W, int* b,
                                           int* y, int* x) {
  const unsigned int t = fdiv(row, Wp);
  const unsigned int xx = row - t * Wp.d;
  const unsigned int bb = fdiv(t, Hp);
  const unsigned int yy = t - bb * Hp.d;
  *b = (int)bb;
  *y = (int)yy;
  *x = (int)xx;
  return (int)xx < W && (int)yy < H;
}

// Element offset of row (b, y, x) of an activation in a buffer addressed through (ld, ch_off), or through the Reorg(2)
// shuffle into a (H/2, W/2) buffer at channel ch_off + ((y&1)*2 + (x&1))*C (interior rows only), so that a concat slice
// or a reorg'd tensor is written / read in place.
__device__ __forceinline__ long long act_offset(unsigned int row, int b, int y, int x, int H, int W, int C, int ld,
                                                int ch_off, int reorg) {
  if (!reorg) return (long long)row * ld + ch_off;
  const int Wo = W / 2 + 1, Ho = H / 2 + 1;
  const long long orow = ((long long)b * Ho + (y >> 1)) * Wo + (x >> 1);
  return orow * ld + ch_off + ((y & 1) * 2 + (x & 1)) * C;
}

// ---- column sums: sum[c] += z[row, ch_off+c], sumsq[c] += z[row, ch_off+c]^2 over all rows (pad rows are zero) -----
__global__ void __launch_bounds__(TB) col_stats_vec_kernel(const __nv_bfloat16* __restrict__ z, unsigned int rows, int C,
                                                           int O8, int ld, int ch_off, float* __restrict__ sum,
                                                           float* __restrict__ sumsq) {
  const OctetWalk w = octet_walk(O8);
  const __nv_bfloat16* zc = z + ch_off + w.c0;
  float a[8], b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = b[j] = 0.f;
  unsigned int r = w.row0;
  // 4 independent 16-byte loads in flight per thread
  for (; r + 3 * w.stride < rows; r += 4 * w.stride) {
    uint4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) q[u] = *reinterpret_cast<const uint4*>(zc + (long long)(r + u * w.stride) * ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float f[8];
      unpack8(q[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { a[j] += f[j]; b[j] = fmaf(f[j], f[j], b[j]); }
    }
  }
  for (; r < rows; r += w.stride) {
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(zc + (long long)r * ld), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { a[j] += f[j]; b[j] = fmaf(f[j], f[j], b[j]); }
  }
  block_col_sums(a, b, O8, C, sum, sumsq);
}

// ---- BN apply (+leaky): out = act(z*scale+shift), pads zero; optional reorg / channel-slice store ------------------
template <bool WHOLE>
__global__ void __launch_bounds__(TB) bn_apply_vec_kernel(const __nv_bfloat16* __restrict__ z, int ld_z, int B, int H, int W,
                                                          int C, int O8, const float* __restrict__ scale,
                                                          const float* __restrict__ shift, int leaky,
                                                          __nv_bfloat16* __restrict__ out, int ld_out, int ch_off, int reorg,
                                                          FastDiv fWp, FastDiv fHp) {
  const OctetWalk w = octet_walk(O8);
  const unsigned int rows = (unsigned int)B * (H + 1) * (W + 1);
  float sc[8], sh[8];
  load_ch<WHOLE>(scale, w.c0, C, sc);
  load_ch<WHOLE>(shift, w.c0, C, sh);
  for (unsigned int row = w.row0; row < rows; row += w.stride) {
    int b, y, x;
    const bool in = row_coords(row, fWp, fHp, H, W, &b, &y, &x);
    float o[8];
    if (in) {
      float f[8];
      unpack8(*reinterpret_cast<const uint4*>(z + (long long)row * ld_z + w.c0), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = fmaf(f[j], sc[j], sh[j]);
        o[j] = leaky ? fmaxf(v, 0.1f * v) : v;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = 0.f;
    }
    if (!reorg || in) store8<WHOLE>(out + act_offset(row, b, y, x, H, W, C, ld_out, ch_off, reorg) + w.c0, !reorg, C - w.c0, o);
  }
}

// ---- BN + leaky backward -----------------------------------------------------------------------------------------
// APPLY = false: dbeta += sum g, dgamma += sum g*xhat.  APPLY = true: dz = gamma*invstd*(g - dbeta/N - xhat*dgamma/N)
// at interior pixels, 0 at pads.  g = da * leaky'(gamma*xhat + beta), xhat = (z-mean)*invstd; da is read through
// (ld_da, ch_off, reorg) so a concat slice / reorg'd gradient needs no un-shuffling copy.
template <bool APPLY, bool WHOLE>
__global__ void __launch_bounds__(TB, 3) bn_bwd_vec_kernel(const __nv_bfloat16* __restrict__ z, int ld_z,
                                                           const __nv_bfloat16* __restrict__ da, int ld_da, int ch_off,
                                                           int reorg, int B, int H, int W, int C, int O8,
                                                           const float* __restrict__ mean, const float* __restrict__ invstd,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           int leaky, float* __restrict__ dbeta, float* __restrict__ dgamma,
                                                           float inv_count, __nv_bfloat16* __restrict__ dz, int ld_dz,
                                                           FastDiv fWp, FastDiv fHp) {
  OctetWalk w = octet_walk(O8);
  asm("" : "+r"(w.c0));  // keep c0 in a register: rebuilt from threadIdx.x / O8 in the loop it cost a spill (ptxas -v)
  const unsigned int rows = (unsigned int)B * (H + 1) * (W + 1);
  const int n = C - w.c0;
  float m[8], is[8], g0[8], b0[8], k1[8], kb[8], kg[8], sa[8], sb[8];
  load_ch<WHOLE>(mean, w.c0, C, m);
  load_ch<WHOLE>(invstd, w.c0, C, is);
  load_ch<WHOLE>(gamma, w.c0, C, g0);
  load_ch<WHOLE>(beta, w.c0, C, b0);
  if (APPLY) {
    load_ch<WHOLE>(dbeta, w.c0, C, kb);
    load_ch<WHOLE>(dgamma, w.c0, C, kg);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    k1[j] = g0[j] * is[j];
    kb[j] = APPLY ? kb[j] * inv_count : 0.f;
    kg[j] = APPLY ? kg[j] * inv_count : 0.f;
    sa[j] = sb[j] = 0.f;
  }
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  for (unsigned int row = w.row0; row < rows; row += 2 * w.stride) {  // two rows per step: four 16-byte loads in flight
    uint4 qz[2], qa[2];
    bool ok[2], in[2];
    unsigned int r[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      r[u] = row + u * w.stride;
      ok[u] = r[u] < rows;
      in[u] = false;
      qz[u] = qa[u] = zero4;
      if (ok[u]) {
        int b, y, x;
        in[u] = row_coords(r[u], fWp, fHp, H, W, &b, &y, &x);
        if (in[u]) {
          qz[u] = *reinterpret_cast<const uint4*>(z + (long long)r[u] * ld_z + w.c0);
          qa[u] = load8<WHOLE>(da + act_offset(r[u], b, y, x, H, W, C, ld_da, ch_off, reorg) + w.c0, !reorg, n);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (!(APPLY ? ok[u] : in[u])) continue;
      float out[8];
      if (in[u]) {
        float fz[8], fa[8];
        unpack8(qz[u], fz);
        unpack8(qa[u], fa);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (fz[j] - m[j]) * is[j];
          float g = fa[j];
          if (leaky && (g0[j] * xh + b0[j]) <= 0.f) g *= 0.1f;
          if (APPLY) {
            out[j] = k1[j] * (g - kb[j] - xh * kg[j]);
          } else {
            sa[j] += g;
            sb[j] += g * xh;
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) out[j] = 0.f;
      }
      if (APPLY) store8<WHOLE>(dz + (long long)r[u] * ld_dz + w.c0, true, n, out);
    }
  }
  if (!APPLY) block_col_sums(sa, sb, O8, C, dbeta, dgamma);
}

// ---- max-pool 2x2/2 backward: gradient goes to the first maximum of each window (PyTorch scan order) ---------------
// one thread = one pooled pixel x 8 channels: the 2x2 window is read once, the four gradients written once.  Pad
// rows/columns of d_full are not touched (they are zero and stay zero).
template <bool WHOLE>
__global__ void __launch_bounds__(TB) maxpool_bwd_vec_kernel(const __nv_bfloat16* __restrict__ a_full, int ld_a,
                                                             const __nv_bfloat16* __restrict__ d_pooled, int ld_dp, int B,
                                                             int H, int W, int C, int O8, __nv_bfloat16* __restrict__ d_full,
                                                             int ld_df, int accumulate) {
  const OctetWalk w = octet_walk(O8);
  const int Ho = H / 2, Wo = W / 2, c0 = w.c0;
  const unsigned int pixels = (unsigned int)B * Ho * Wo;
  for (unsigned int pix = w.row0; pix < pixels; pix += w.stride) {
    const unsigned int t = pix / (unsigned int)Wo;
    const int wx = (int)(pix - t * (unsigned int)Wo);
    const int b = (int)(t / (unsigned int)Ho), wy = (int)(t - (t / (unsigned int)Ho) * (unsigned int)Ho);
    const long long r00 = ((long long)b * (H + 1) + 2 * wy) * (W + 1) + 2 * wx;
    const long long roff[4] = {r00, r00 + 1, r00 + W + 1, r00 + W + 2};
    float v[4][8], g[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) unpack8(*reinterpret_cast<const uint4*>(a_full + roff[q] * ld_a + c0), v[q]);
    const long long prow = ((long long)b * (Ho + 1) + wy) * (Wo + 1) + wx;
    unpack8(*reinterpret_cast<const uint4*>(d_pooled + prow * ld_dp + c0), g);
    float o[4][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int arg = 0;
      float best = v[0][j];
      if (v[1][j] > best) { best = v[1][j]; arg = 1; }
      if (v[2][j] > best) { best = v[2][j]; arg = 2; }
      if (v[3][j] > best) { best = v[3][j]; arg = 3; }
#pragma unroll
      for (int q = 0; q < 4; ++q) o[q][j] = (q == arg) ? g[j] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      __nv_bfloat16* dst = d_full + roff[q] * ld_df + c0;
      if (accumulate) {
        float old[8];
        unpack8(*reinterpret_cast<const uint4*>(dst), old);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[q][j] += old[j];
      }
      store8<WHOLE>(dst, true, C - c0, o[q]);
    }
  }
}

// ---- BatchNorm + leaky + 2x2 max-pool as ONE pass each way (layers whose un-pooled activation only feeds the pool) ----
// The un-pooled activation a = leaky(z*scale + shift) is never stored: the forward writes the pooled tensor straight
// from z, and the backward recomputes the four window values from z (same fp32 arithmetic, same bf16 rounding as the
// stored tensor would have had), routes the pooled gradient to the first maximum — nn.MaxPool2d's rule — and feeds the
// BatchNorm reductions / dz directly.  Per pooled layer this moves 1.25 S (forward) + 3.5 S (backward) bytes instead
// of 2 S + 1.25 S and 7.25 S (S = bytes of z): the four pooled layers of Darknet-19 hold 63 % of all activation bytes.
// A thread keeps its octet over the pooled pixels like the kernels above; C is a whole number of octets.
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__device__ __forceinline__ void pool_item(unsigned int pix, const FastDiv& fWo, const FastDiv& fHo, int H, int W,
                                          long long* r00, long long* prow) {
  const unsigned int t = fdiv(pix, fWo);
  const unsigned int wx = pix - t * fWo.d;
  const unsigned int b = fdiv(t, fHo);
  const unsigned int wy = t - b * fHo.d;
  *r00 = ((long long)b * (H + 1) + 2 * wy) * (W + 1) + 2 * wx;
  *prow = ((long long)b * (fHo.d + 1) + wy) * (fWo.d + 1) + wx;
}

__global__ void __launch_bounds__(TB) bn_apply_pool_vec_kernel(const __nv_bfloat16* __restrict__ z, int ld_z, int B, int H,
                                                               int W, int O8, const float* __restrict__ scale,
                                                               const float* __restrict__ shift, int leaky,
                                                               __nv_bfloat16* __restrict__ pooled, int ld_p, FastDiv fWo,
                                                               FastDiv fHo) {
  const OctetWalk w = octet_walk(O8);
  const int c0 = w.c0;
  const unsigned int pixels = (unsigned int)B * fHo.d * fWo.d;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c0 + j]; sh[j] = shift[c0 + j]; }
  for (unsigned int pix = w.row0; pix < pixels; pix += w.stride) {
    long long r00, prow;
    pool_item(pix, fWo, fHo, H, W, &r00, &prow);
    const long long roff[4] = {r00, r00 + 1, r00 + W + 1, r00 + W + 2};
    uint4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) q[u] = *reinterpret_cast<const uint4*>(z + roff[u] * ld_z + c0);
    float best[8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float f[8];
      unpack8(q[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float v = fmaf(f[j], sc[j], sh[j]);
        if (leaky) v = fmaxf(v, 0.1f * v);
        v = bf16_round(v);
        best[j] = (u == 0) ? v : fmaxf(best[j], v);
      }
    }
    *reinterpret_cast<uint4*>(pooled + prow * ld_p + c0) = pack8(best);
  }
}

// APPLY = false: dbeta += sum g, dgamma += sum g * xhat.  APPLY = true: dz = gamma*invstd * (g - dbeta/N - xhat*dgamma/N).
// g = d_pooled at the window's first maximum (0 elsewhere), times the leaky slope where the forward pre-activation
// z*scale + shift is <= 0 (what autograd's LeakyReLU backward tests).  gamma*invstd == scale.
template <bool APPLY>
__global__ void __launch_bounds__(TB, 2) bn_pool_bwd_vec_kernel(const __nv_bfloat16* __restrict__ z, int ld_z,
                                                                const __nv_bfloat16* __restrict__ dp, int ld_dp, int B, int H,
                                                                int W, int O8, const float* __restrict__ scale,
                                                                const float* __restrict__ shift, const float* __restrict__ mean,
                                                                const float* __restrict__ invstd, int leaky,
                                                                float* __restrict__ dbeta, float* __restrict__ dgamma,
                                                                float inv_count, __nv_bfloat16* __restrict__ dz, int ld_dz,
                                                                FastDiv fWo, FastDiv fHo) {
  const OctetWalk w = octet_walk(O8);
  const int c0 = w.c0;
  const unsigned int pixels = (unsigned int)B * fHo.d * fWo.d;
  float sc[8], sh[8], m[8], is[8], kb[8], kg[8], sa[8], sb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = scale[c0 + j]; sh[j] = shift[c0 + j];
    m[j] = mean[c0 + j]; is[j] = invstd[c0 + j];
    sa[j] = sb[j] = 0.f;
    kb[j] = APPLY ? dbeta[c0 + j] * inv_count : 0.f;
    kg[j] = APPLY ? dgamma[c0 + j] * inv_count : 0.f;
  }
  const float slope = leaky ? 0.1f : 1.0f;
  for (unsigned int pix = w.row0; pix < pixels; pix += w.stride) {
    long long r00, prow;
    pool_item(pix, fWo, fHo, H, W, &r00, &prow);
    const long long roff[4] = {r00, r00 + 1, r00 + W + 1, r00 + W + 2};
    uint4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) q[u] = *reinterpret_cast<const uint4*>(z + roff[u] * ld_z + c0);
    const uint4 qg = *reinterpret_cast<const uint4*>(dp + prow * ld_dp + c0);
    float fz[4][8], g[8];
#pragma unroll
    for (int u = 0; u < 4; ++u) unpack8(q[u], fz[u]);
    unpack8(qg, g);
    unsigned int args = 0;  // 2 bits per channel: window position of the first maximum
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int arg = 0;
      float best = 0.f, zbest = 0.f, pre_best = 0.f;
#pragma unroll
      for (int u = 0; u < 4; ++u) {  // the forward's values, the pool's first-maximum rule
        const float pre = fmaf(fz[u][j], sc[j], sh[j]);
        const float v = bf16_round(leaky ? fmaxf(pre, 0.1f * pre) : pre);
        if (u == 0 || v > best) { best = v; arg = u; zbest = fz[u][j]; pre_best = pre; }
      }
      if (!APPLY) {
        const float xh = (zbest - m[j]) * is[j];
        const float gg = pre_best <= 0.f ? g[j] * slope : g[j];
        sa[j] += gg;
        sb[j] += gg * xh;
      } else {
        args |= (unsigned int)arg << (2 * j);
        if (pre_best <= 0.f) g[j] *= slope;  // (only the maximum's gradient is non-zero)
      }
    }
    if (APPLY) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float out[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (fz[u][j] - m[j]) * is[j];
          const float gg = (((args >> (2 * j)) & 3u) == (unsigned int)u) ? g[j] : 0.f;
          out[j] = sc[j] * (gg - kb[j] - xh * kg[j]);
        }
        *reinterpret_cast<uint4*>(dz + roff[u] * ld_dz + c0) = pack8(out);
      }
    }
  }
  if (!APPLY) block_col_sums(sa, sb, O8, O8 * 8, dbeta, dgamma);
}

// Blocks of octet_threads(O8) threads for `rows` rows (pooled pixels).  items_per_thread > 1: kernels that end in
// per-block atomics (one per channel and block) want fewer, longer blocks on the small layers — at 13x13x1024 the cap
// of 8 blocks per SM gave every thread 5 items and the grid 2.4 M atomics
inline int vec_blocks(long long rows, int O8, int items_per_thread = 1) {
  const long long rows_per_block = TB / O8;
  long long blocks = (rows + rows_per_block * items_per_thread - 1) / (rows_per_block * items_per_thread);
  const long long cap = (long long)mc_num_sms() * 8;
  if (items_per_thread > 1 && blocks < 2ll * mc_num_sms()) {
    blocks = (rows + rows_per_block - 1) / rows_per_block;
    if (blocks > 2ll * mc_num_sms()) blocks = 2ll * mc_num_sms();
  }
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

// What the octet passes need (mcb200.h): at most MAX_C channels, pitches and channel offsets (or-ed together) multiples
// of 8 and buffers (or-ed) 16-byte aligned so that an octet is one 16-byte access, row indices below 2^31.
inline bool octets_ok(int C, long long rows, int pitches, uintptr_t ptrs) {
  return C <= MAX_C && (pitches & 7) == 0 && (ptrs & 15) == 0 && rows < (1ll << 31);
}

inline int grid_for(long long total, int threads) {
  long long blocks = (total + threads - 1) / threads;
  const long long cap = (long long)mc_num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace

extern "C" int mc_col_stats(const void* d_z, int64_t rows, int C, int ld, int ch_off, float* d_sum, float* d_sumsq,
                            void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_z && d_sum && rows > 0 && C > 0, "mc_col_stats: bad argument");
  MC_CHECK_ARG((ld % 8) == 0 && (ch_off % 8) == 0 && ch_off + ((C + 7) / 8) * 8 <= ld,
               "mc_col_stats: ld/ch_off must be multiples of 8 and cover round_up(C,8) channels");
  MC_CHECK_ARG(octets_ok(C, rows, ld | ch_off, (uintptr_t)d_z),
               "mc_col_stats: needs C <= 2048, a 16-byte aligned d_z and rows < 2^31");
  MC_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(float) * C, stream));
  if (d_sumsq) MC_CUDA(cudaMemsetAsync(d_sumsq, 0, sizeof(float) * C, stream));
  const int O8 = (C + 7) / 8;
  col_stats_vec_kernel<<<vec_blocks(rows, O8), octet_threads(O8), 0, stream>>>((const __nv_bfloat16*)d_z, (unsigned int)rows,
                                                                              C, O8, ld, ch_off, d_sum, d_sumsq);
  MC_LAUNCH_CHECK("col_stats_vec_kernel");
  return 0;
}

extern "C" int mc_bn_finalize(const float* d_sum, const float* d_sumsq, int C, double count, const float* d_gamma,
                              const float* d_beta, float eps, float momentum, float* d_running_mean,
                              float* d_running_var, float* d_scale, float* d_shift, float* d_mean, float* d_invstd,
                              void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_sum && d_sumsq && d_gamma && d_beta && d_scale && d_shift && d_mean && d_invstd && C > 0 && count > 0,
               "mc_bn_finalize: bad argument");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(d_sum, d_sumsq, C, count, d_gamma, d_beta, eps, momentum,
                                                          d_running_mean, d_running_var, d_scale, d_shift, d_mean,
                                                          d_invstd);
  MC_LAUNCH_CHECK("bn_finalize_kernel");
  return 0;
}

extern "C" int mc_bn_apply(const void* d_z, int ld_z, int B, int H, int W, int C, const float* d_scale,
                           const float* d_shift, int leaky, void* d_out, int ld_out, int ch_off, int reorg,
                           void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_z && d_scale && d_shift && d_out && B > 0 && H > 0 && W > 0 && C > 0, "mc_bn_apply: bad argument");
  MC_CHECK_ARG((ld_z % 8) == 0 && ld_z >= ((C + 7) / 8) * 8, "mc_bn_apply: ld_z must be a multiple of 8 covering C");
  if (reorg) MC_CHECK_ARG((H % 2) == 0 && (W % 2) == 0, "mc_bn_apply: reorg needs even H,W");
  const long long rows = (long long)B * (H + 1) * (W + 1);
  MC_CHECK_ARG(octets_ok(C, rows, ld_out | ch_off, (uintptr_t)d_z | (uintptr_t)d_out),
               "mc_bn_apply: needs C <= 2048, ld_out and ch_off multiples of 8, 16-byte aligned buffers and "
               "B*(H+1)*(W+1) < 2^31");
  const int O8 = (C + 7) / 8;
  auto* kernel = (C % 8) == 0 ? bn_apply_vec_kernel<true> : bn_apply_vec_kernel<false>;
  kernel<<<vec_blocks(rows, O8), octet_threads(O8), 0, stream>>>((const __nv_bfloat16*)d_z, ld_z, B, H, W, C, O8, d_scale,
                                                                d_shift, leaky, (__nv_bfloat16*)d_out, ld_out, ch_off,
                                                                reorg, make_fastdiv(W + 1), make_fastdiv(H + 1));
  MC_LAUNCH_CHECK("bn_apply_vec_kernel");
  return 0;
}

extern "C" int mc_bn_backward(const void* d_z, int ld_z, const void* d_da, int ld_da, int ch_off, int reorg, int B, int H,
                              int W, int C, const float* d_mean, const float* d_invstd, const float* d_gamma,
                              const float* d_beta, int leaky, float* d_dbeta, float* d_dgamma, void* d_dz, int ld_dz,
                              void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_z && d_da && d_mean && d_invstd && d_gamma && d_beta && d_dbeta && d_dgamma && d_dz,
               "mc_bn_backward: null pointer");
  MC_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0, "mc_bn_backward: bad dims");
  const long long rows = (long long)B * (H + 1) * (W + 1);
  MC_CHECK_ARG(octets_ok(C, rows, ld_z | ld_da | ld_dz | ch_off, (uintptr_t)d_z | (uintptr_t)d_da | (uintptr_t)d_dz),
               "mc_bn_backward: needs C <= 2048, pitches and ch_off multiples of 8, 16-byte aligned buffers and "
               "B*(H+1)*(W+1) < 2^31");
  MC_CUDA(cudaMemsetAsync(d_dbeta, 0, sizeof(float) * C, stream));
  MC_CUDA(cudaMemsetAsync(d_dgamma, 0, sizeof(float) * C, stream));
  const float inv_count = 1.0f / (float)((double)B * H * W);
  const int O8 = (C + 7) / 8;
  const bool whole = (C % 8) == 0;
  auto* reduce = whole ? bn_bwd_vec_kernel<false, true> : bn_bwd_vec_kernel<false, false>;
  auto* apply = whole ? bn_bwd_vec_kernel<true, true> : bn_bwd_vec_kernel<true, false>;
  const FastDiv fWp = make_fastdiv(W + 1), fHp = make_fastdiv(H + 1);
  reduce<<<vec_blocks(rows, O8, 16), octet_threads(O8), 0, stream>>>(
      (const __nv_bfloat16*)d_z, ld_z, (const __nv_bfloat16*)d_da, ld_da, ch_off, reorg, B, H, W, C, O8, d_mean, d_invstd,
      d_gamma, d_beta, leaky, d_dbeta, d_dgamma, inv_count, nullptr, ld_dz, fWp, fHp);
  MC_LAUNCH_CHECK("bn_bwd_vec_kernel<reduce>");
  apply<<<vec_blocks(rows, O8), octet_threads(O8), 0, stream>>>(
      (const __nv_bfloat16*)d_z, ld_z, (const __nv_bfloat16*)d_da, ld_da, ch_off, reorg, B, H, W, C, O8, d_mean, d_invstd,
      d_gamma, d_beta, leaky, d_dbeta, d_dgamma, inv_count, (__nv_bfloat16*)d_dz, ld_dz, fWp, fHp);
  MC_LAUNCH_CHECK("bn_bwd_vec_kernel<apply>");
  return 0;
}

extern "C" int mc_maxpool2x2_backward(const void* d_a_full, int ld_a, const void* d_dpooled, int ld_dp, int B, int H,
                                      int W, int C, void* d_dfull, int ld_df, int accumulate, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_a_full && d_dpooled && d_dfull && B > 0 && H > 0 && W > 0 && C > 0, "mc_maxpool2x2_backward: bad argument");
  MC_CHECK_ARG((H % 2) == 0 && (W % 2) == 0, "mc_maxpool2x2_backward: H, W must be even");
  MC_CHECK_ARG(octets_ok(C, (long long)B * (H + 1) * (W + 1), ld_a | ld_dp | ld_df,
                         (uintptr_t)d_a_full | (uintptr_t)d_dpooled | (uintptr_t)d_dfull),
               "mc_maxpool2x2_backward: needs C <= 2048, pitches multiples of 8, 16-byte aligned buffers and "
               "B*(H+1)*(W+1) < 2^31");
  const int O8 = (C + 7) / 8;
  const long long pixels = (long long)B * (H / 2) * (W / 2);
  auto* kernel = (C % 8) == 0 ? maxpool_bwd_vec_kernel<true> : maxpool_bwd_vec_kernel<false>;
  kernel<<<grid_for(pixels * O8, octet_threads(O8)), octet_threads(O8), 0, stream>>>(
      (const __nv_bfloat16*)d_a_full, ld_a, (const __nv_bfloat16*)d_dpooled, ld_dp, B, H, W, C, O8,
      (__nv_bfloat16*)d_dfull, ld_df, accumulate);
  MC_LAUNCH_CHECK("maxpool_bwd_vec_kernel");
  return 0;
}

extern "C" int mc_bn_pool_supported(int C) {
  const int O8 = C / 8;
  return ((C % 8) == 0 && O8 > 0 && (O8 & (O8 - 1)) == 0 && (TB % O8) == 0) ? 1 : 0;
}

extern "C" int mc_bn_apply_pool(const void* d_z, int ld_z, int B, int H, int W, int C, const float* d_scale,
                                const float* d_shift, int leaky, void* d_pooled, int ld_p, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_z && d_scale && d_shift && d_pooled && B > 0 && H > 0 && W > 0 && C > 0, "mc_bn_apply_pool: bad argument");
  MC_CHECK_ARG((H % 2) == 0 && (W % 2) == 0, "mc_bn_apply_pool: H, W must be even");
  MC_CHECK_ARG(mc_bn_pool_supported(C) == 1 && ld_z >= C && ld_p >= C &&
                   octets_ok(C, (long long)B * (H + 1) * (W + 1), ld_z | ld_p, (uintptr_t)d_z | (uintptr_t)d_pooled),
               "mc_bn_apply_pool: needs C = 8 * 2^k <= 2048, pitches multiples of 8, 16-byte aligned buffers and "
               "B*(H+1)*(W+1) < 2^31");
  const int O8 = C / 8;
  bn_apply_pool_vec_kernel<<<vec_blocks((long long)B * (H / 2) * (W / 2), O8), octet_threads(O8), 0, stream>>>(
      (const __nv_bfloat16*)d_z, ld_z, B, H, W, O8, d_scale, d_shift, leaky, (__nv_bfloat16*)d_pooled, ld_p,
      make_fastdiv(W / 2), make_fastdiv(H / 2));
  MC_LAUNCH_CHECK("bn_apply_pool_vec_kernel");
  return 0;
}

extern "C" int mc_bn_pool_backward(const void* d_z, int ld_z, const void* d_dpooled, int ld_dp, int B, int H, int W, int C,
                                   const float* d_scale, const float* d_shift, const float* d_mean, const float* d_invstd,
                                   const float* d_gamma, const float* d_beta, int leaky, float* d_dbeta, float* d_dgamma,
                                   void* d_dz, int ld_dz, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_z && d_dpooled && d_scale && d_shift && d_mean && d_invstd && d_gamma && d_beta && d_dbeta && d_dgamma && d_dz,
               "mc_bn_pool_backward: null pointer");
  MC_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && (H % 2) == 0 && (W % 2) == 0, "mc_bn_pool_backward: bad dims");
  MC_CHECK_ARG(mc_bn_pool_supported(C) == 1 &&
                   octets_ok(C, (long long)B * (H + 1) * (W + 1), ld_z | ld_dp | ld_dz,
                             (uintptr_t)d_z | (uintptr_t)d_dpooled | (uintptr_t)d_dz),
               "mc_bn_pool_backward: needs C = 8 * 2^k <= 2048, pitches multiples of 8, 16-byte aligned buffers and "
               "B*(H+1)*(W+1) < 2^31");
  MC_CUDA(cudaMemsetAsync(d_dbeta, 0, sizeof(float) * C, stream));
  MC_CUDA(cudaMemsetAsync(d_dgamma, 0, sizeof(float) * C, stream));
  const int O8 = C / 8;
  const int vb = vec_blocks((long long)B * (H / 2) * (W / 2), O8);
  const float inv_count = 1.0f / (float)((double)B * H * W);
  const FastDiv fWo = make_fastdiv(W / 2), fHo = make_fastdiv(H / 2);
  bn_pool_bwd_vec_kernel<false><<<vb, octet_threads(O8), 0, stream>>>((const __nv_bfloat16*)d_z, ld_z,
                                                                      (const __nv_bfloat16*)d_dpooled, ld_dp, B, H, W, O8,
                                                                      d_scale, d_shift, d_mean, d_invstd, leaky, d_dbeta,
                                                                      d_dgamma, inv_count, nullptr, ld_dz, fWo, fHo);
  MC_LAUNCH_CHECK("bn_pool_bwd_vec_kernel<reduce>");
  bn_pool_bwd_vec_kernel<true><<<vb, octet_threads(O8), 0, stream>>>((const __nv_bfloat16*)d_z, ld_z,
                                                                     (const __nv_bfloat16*)d_dpooled, ld_dp, B, H, W, O8,
                                                                     d_scale, d_shift, d_mean, d_invstd, leaky, d_dbeta,
                                                                     d_dgamma, inv_count, (__nv_bfloat16*)d_dz, ld_dz, fWo,
                                                                     fHo);
  MC_LAUNCH_CHECK("bn_pool_bwd_vec_kernel<apply>");
  return 0;
}

// ---- dgrad weights: the data gradient of a 'same' 3x3 / 1x1 convolution is itself a 'same' convolution of dZ with the
// spatially flipped, channel-transposed filter:  dA[p, c] = sum_{tap', o} dZ[p + off(tap'), o] * W[o, c, taps-1-tap'].
// So dgrad reuses the forward tcgen05 kernel (mc_conv_fwd) on this packing: bf16 [Cpad, taps*Ko] K-major, row c,
// column tap'*Ko + o  (Ko = round_up(O, 64)), masked like the forward weights (layers.py:59).
namespace {
// Large filter banks: a block transposes a tile of 32 output x 32 input channels through shared memory.  Reading, a warp
// walks the 32*taps contiguous floats that one output channel holds for the tile's input channels (coalesced 128-byte
// requests; the direct kernel below reads 36-byte runs 36 KB apart); writing, two input channels x 16 output-channel
// pairs per warp store 64-byte runs of the K-major dgrad matrix.  All loads of a thread (4 output channels x taps) are
// issued before the one barrier.  (A first tiled version that looped 32 dependent load steps around two barriers was
// slower than the direct kernel: DESIGN.md §9.)
template <int TAPS>
__global__ void __launch_bounds__(256) pack_dgrad_weights_tiled_kernel(const float* __restrict__ w,
                                                                       const float* __restrict__ mask, int O, int C,
                                                                       __nv_bfloat16* __restrict__ out, int Ko) {
  __shared__ float tile[32][32 * TAPS + 1];  // [o][c*TAPS + t]
  const int o0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cw = min(32, C - c0);  // input channels of this tile
  const int run = cw * TAPS;       // contiguous floats per output channel
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int ol = warp * 4 + q;
    const int o = o0 + ol;
    if (o < O) {
      const size_t src = ((size_t)o * C + c0) * TAPS;
#pragma unroll
      for (int j = 0; j < TAPS; ++j) {
        const int e = j * 32 + lane;
        if (e < run) {
          float v = w[src + e];
          if (mask) v *= mask[src + e];
          tile[ol][e] = v;
        }
      }
    }
  }
  __syncthreads();
  // warp: 2 input channels per pass (half-warps), lane & 15 = pair of output channels
  const int half = lane >> 4, op = (lane & 15) * 2;
  for (int cl = warp * 2 + half; cl < cw; cl += 16) {
    const int c = c0 + cl;
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
      const int o = o0 + op;
      if (o < O) {
        const float a = tile[op][cl * TAPS + t];
        const float b = (o + 1 < O) ? tile[op + 1][cl * TAPS + t] : 0.f;
        __nv_bfloat16* dst = out + ((size_t)c * TAPS + (TAPS - 1 - t)) * Ko + o;
        if (o + 1 < O) {
          *reinterpret_cast<__nv_bfloat162*>(dst) = __floats2bfloat162_rn(a, b);
        } else {
          *dst = __float2bfloat16_rn(a);
        }
      }
    }
  }
}

// one thread = one (input channel c, output channel o), o fastest: the taps are read as one contiguous run, each write
// is coalesced over o.  Padding is zeroed by a memset before the launch.
__global__ void pack_dgrad_weights_kernel(const float* __restrict__ w, const float* __restrict__ mask, int O, int C,
                                          int taps, __nv_bfloat16* __restrict__ out, int Cpad, int Ko) {
  const unsigned int total = (unsigned int)O * (unsigned int)C;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const unsigned int c = i / (unsigned int)O, o = i - c * (unsigned int)O;
    const size_t src = ((size_t)o * C + c) * taps;
    __nv_bfloat16* dst = out + (size_t)c * taps * Ko + o;
    for (int t = 0; t < taps; ++t) {
      float v = w[src + t];
      if (mask) v *= mask[src + t];
      dst[(size_t)(taps - 1 - t) * Ko] = __float2bfloat16_rn(v);
    }
  }
}

// ---- weight gradient of the FIRST layer (3-channel fp32 NCHW image): too thin for a tensor-core tile (N = 3), so
// CUDA cores: thread = (4 output channels, input channel, pixel slice) keeps 4 x 9 accumulators in registers over a
// grid-stride sweep of the image lines; one shared-memory reduction and 9*C*O atomics per block at the end.
constexpr int WF_THREADS = 256;
__global__ void __launch_bounds__(WF_THREADS) wgrad_first_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dz,
                                                                 int ld_dz, int B, int H, int W, int C, int O,
                                                                 float* __restrict__ dw) {
  __shared__ float s_acc[32 * 4 * 9];  // [o][c][tap] partial of this block (O <= 32, C <= 4)
  for (int i = threadIdx.x; i < 32 * 4 * 9; i += WF_THREADS) s_acc[i] = 0.f;
  __syncthreads();
  const int og = threadIdx.x & 7, c = (threadIdx.x >> 3) & 3, slice = threadIdx.x >> 5;
  float acc[4][9];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[a][t] = 0.f;
  const bool active = c < C && og * 4 < O;
  const long long lines = (long long)B * H;
  // each of the 8 pixel slices of a block walks a CONTIGUOUS run of the line, so the 3x3 window slides through
  // registers: per pixel 3 new image values + one 8-byte dZ load feed 36 FMAs
  const int run = (W + WF_THREADS / 32 - 1) / (WF_THREADS / 32);
  const int px0 = slice * run, px1 = (px0 + run < W) ? px0 + run : W;
  for (long long ln = blockIdx.x; ln < lines; ln += gridDim.x) {
    const int b = (int)(ln / H), y = (int)(ln - (long long)b * H);
    if (!active || px0 >= px1) continue;
    const __nv_bfloat16* dzl = dz + (((long long)b * (H + 1) + y) * (W + 1)) * ld_dz + og * 4;
    const float* xc = x + ((long long)b * C + c) * H * W;
    const float* xr[3];
    bool rok[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int yy = y + r - 1;
      rok[r] = yy >= 0 && yy < H;
      xr[r] = xc + (long long)(rok[r] ? yy : 0) * W;
    }
    float xw[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      xw[r][1] = (rok[r] && px0 - 1 >= 0) ? __ldg(xr[r] + px0 - 1) : 0.f;
      xw[r][2] = rok[r] ? __ldg(xr[r] + px0) : 0.f;
    }
    // groups of 4 pixels: the 4 dZ loads (DRAM latency) and the 12 image loads are issued before the 144 FMAs
    for (int pg = px0; pg < px1; pg += 4) {
      uint2 q[4];
      float xn[4][3];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int px = pg + u;
        q[u] = (px < px1) ? *reinterpret_cast<const uint2*>(dzl + (long long)px * ld_dz) : make_uint2(0u, 0u);
#pragma unroll
        for (int r = 0; r < 3; ++r) xn[u][r] = (rok[r] && px + 1 < W && px < px1) ? __ldg(xr[r] + px + 1) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          xw[r][0] = xw[r][1];
          xw[r][1] = xw[r][2];
          xw[r][2] = xn[u][r];
        }
        const __nv_bfloat162 h0 = *reinterpret_cast<const __nv_bfloat162*>(&q[u].x);
        const __nv_bfloat162 h1 = *reinterpret_cast<const __nv_bfloat162*>(&q[u].y);
        const float g[4] = {__low2float(h0), __high2float(h0), __low2float(h1), __high2float(h1)};
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int t = 0; t < 9; ++t) acc[a][t] = fmaf(g[a], xw[t / 3][t % 3], acc[a][t]);
      }
    }
  }
  if (active) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int t = 0; t < 9; ++t) atomicAdd(&s_acc[((og * 4 + a) * 4 + c) * 9 + t], acc[a][t]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 32 * 4 * 9; i += WF_THREADS) {
    const int t = i % 9, cc = (i / 9) % 4, o = i / 36;
    if (o < O && cc < C && s_acc[i] != 0.f) atomicAdd(&dw[((long long)o * C + cc) * 9 + t], s_acc[i]);
  }
}

// First-layer im2col for the tensor-core weight gradient: row = PNHWC pixel row (pad rows are zero), column c*9 + tap
// = x[b, c, y+dy-1, x+dx-1] rounded to bf16 (zero outside the image), columns >= C*9 zero.  One thread per row writes
// its 64 bytes with four 16-byte stores; the 9*C image reads of neighbouring pixels overlap in L1.
__global__ void __launch_bounds__(256) im2col_first_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                           int B, int H, int W, int C) {
  const long long rows = (long long)B * (H + 1) * (W + 1);
  for (long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x; row < rows;
       row += (long long)gridDim.x * blockDim.x) {
    const int xx = (int)(row % (W + 1));
    const long long t = row / (W + 1);
    const int yy = (int)(t % (H + 1));
    const int b = (int)(t / (H + 1));
    __align__(16) __nv_bfloat16 v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __float2bfloat16_rn(0.f);
    if (xx < W && yy < H) {
      for (int c = 0; c < C; ++c) {
        const float* xc = x + ((long long)b * C + c) * H * W;
#pragma unroll
        for (int tp = 0; tp < 9; ++tp) {
          const int y2 = yy + tp / 3 - 1, x2 = xx + tp % 3 - 1;
          const bool ok = y2 >= 0 && y2 < H && x2 >= 0 && x2 < W;
          v[c * 9 + tp] = __float2bfloat16_rn(ok ? __ldg(xc + (long long)y2 * W + x2) : 0.f);
        }
      }
    }
    uint4* dst = reinterpret_cast<uint4*>(out + row * 32);
#pragma unroll
    for (int q = 0; q < 4; ++q) dst[q] = reinterpret_cast<const uint4*>(v)[q];
  }
}

// dW[o][j] = mask * (t[o][j] + t[32 + o][32 + j]): the two diagonal blocks of the doubled-row product (see
// mc_conv_wgrad_first)
__global__ void wgrad_fold2_kernel(const float* __restrict__ t, const float* __restrict__ mask, float* __restrict__ dw,
                                   int O, int J) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= O * J) return;
  const int o = i / J, j = i - o * J;
  float v = t[o * 64 + j] + t[(32 + o) * 64 + 32 + j];
  if (mask) v *= mask[i];
  dw[i] = v;
}

// Same rows for C == 3, built for instruction count: 32-bit indexing, one row per thread, interior pixels (all but the
// image border) without bounds logic — the generic kernel above spends ~250 instructions per row on 27 checked loads with
// 64-bit address arithmetic and ran at 1.5 TB/s of its 842 MB.
__global__ void __launch_bounds__(256) im2col_first3_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                            unsigned int rows, int H, int W, FastDiv fWp, FastDiv fHp) {
  const unsigned int row = blockIdx.x * 256u + threadIdx.x;
  if (row >= rows) return;
  int b, yy, xx;
  const bool in = row_coords(row, fWp, fHp, H, W, &b, &yy, &xx);
  uint32_t w[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) w[j] = 0u;
  if (in) {
    const int plane = H * W;
    const float* p0 = x + (b * 3) * plane + yy * W + xx;
    float v[28];
    v[27] = 0.f;
    if (yy >= 1 && yy < H - 1 && xx >= 1 && xx < W - 1) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
          const float* p = p0 + c * plane + (dy - 1) * W;
          v[c * 9 + dy * 3 + 0] = __ldg(p - 1);
          v[c * 9 + dy * 3 + 1] = __ldg(p);
          v[c * 9 + dy * 3 + 2] = __ldg(p + 1);
        }
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int tp = 0; tp < 9; ++tp) {
          const int y2 = yy + tp / 3 - 1, x2 = xx + tp % 3 - 1;
          const bool ok = y2 >= 0 && y2 < H && x2 >= 0 && x2 < W;
          v[c * 9 + tp] = ok ? __ldg(p0 + c * plane + (tp / 3 - 1) * W + (tp % 3 - 1)) : 0.f;
        }
    }
#pragma unroll
    for (int j = 0; j < 14; ++j) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      w[j] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * 32);
#pragma unroll
  for (int q = 0; q < 4; ++q) dst[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}

__global__ void mul_inplace_kernel(float* __restrict__ a, const float* __restrict__ m, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    a[i] *= m[i];
}
}  // namespace

extern "C" int mc_pack_conv_weights_dgrad(const float* d_w, const float* d_mask, int O, int C, int ksize, void* d_wpack,
                                          int Cpad, int Ko, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_w && d_wpack && O > 0 && C > 0 && (ksize == 1 || ksize == 3), "mc_pack_conv_weights_dgrad: bad argument");
  MC_CHECK_ARG(Cpad >= C && (Cpad % 16) == 0 && Ko >= O && (Ko % 32) == 0, "mc_pack_conv_weights_dgrad: bad packed dims");
  const int taps = ksize * ksize;
  MC_CHECK_ARG((long long)O * C < (1ll << 32), "mc_pack_conv_weights_dgrad: tensor too large");
  MC_CUDA(cudaMemsetAsync(d_wpack, 0, (size_t)Cpad * taps * Ko * sizeof(__nv_bfloat16), stream));
  if ((long long)O * C >= 65536 && (Ko % 2) == 0) {
    const dim3 grid((O + 31) / 32, (C + 31) / 32);
    if (taps == 9)
      pack_dgrad_weights_tiled_kernel<9><<<grid, 256, 0, stream>>>(d_w, d_mask, O, C, (__nv_bfloat16*)d_wpack, Ko);
    else
      pack_dgrad_weights_tiled_kernel<1><<<grid, 256, 0, stream>>>(d_w, d_mask, O, C, (__nv_bfloat16*)d_wpack, Ko);
    MC_LAUNCH_CHECK("pack_dgrad_weights_tiled_kernel");
    return 0;
  }
  pack_dgrad_weights_kernel<<<grid_for((long long)O * C, 256), 256, 0, stream>>>(d_w, d_mask, O, C, taps,
                                                                                (__nv_bfloat16*)d_wpack, Cpad, Ko);
  MC_LAUNCH_CHECK("pack_dgrad_weights_kernel");
  return 0;
}

// im2col rows (bf16, 32 columns) + the split-K workspace of the 1x1 tensor-core weight gradient over them
extern "C" size_t mc_workspace_bytes_conv_wgrad_first(int B, int H, int W, int C, int O) {
  if (B <= 0 || H <= 0 || W <= 0 || C < 1 || O < 1 || C * 9 > 32) return 0;
  const size_t rows = (size_t)B * (H + 1) * (W + 1);
  const size_t im2col = (rows * 32 * sizeof(__nv_bfloat16) + 255) & ~(size_t)255;
  size_t w1 = mc_workspace_bytes_conv_wgrad(B, H, W, C * 9, O, 1);
  if ((B % 2) == 0 && O == 32) {  // doubled-row view (see mc_conv_wgrad_first) + its 64x64 product
    const size_t w2 = mc_workspace_bytes_conv_wgrad(B / 2, H, W, 64, 64, 1) + 64 * 64 * sizeof(float) + 256;
    if (w2 > w1) w1 = w2;
  }
  return im2col + w1;
}

extern "C" int mc_conv_wgrad_first(const float* d_x, const void* d_dz, int ld_dz, int B, int H, int W, int C, int O,
                                   const float* d_mask, float* d_dw, void* d_ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(d_x && d_dz && d_dw && B > 0 && H > 0 && W > 0, "mc_conv_wgrad_first: bad argument");
  // Tensor-core path (needs the workspace): dW[o, c*9+tap] = sum_rows dZ[row, o] * im2col[row, c*9+tap] is the 1x1
  // weight gradient over the materialised im2col rows — [O, C*9] is exactly dW[O,C,3,3] in memory.  The im2col
  // costs one pass over the image + a 64 B/pixel write (712 MB at batch 64), far below the ~1.5 ms the CUDA-core
  // kernel below needs for the same 9.6 GMAC.
  const size_t need = mc_workspace_bytes_conv_wgrad_first(B, H, W, C, O);
  if (d_ws != nullptr && need != 0 && ws_bytes >= need && (ld_dz % 8) == 0 && ((uintptr_t)d_ws & 255) == 0) {
    const size_t rows = (size_t)B * (H + 1) * (W + 1);
    const size_t im2col = (rows * 32 * sizeof(__nv_bfloat16) + 255) & ~(size_t)255;
    __nv_bfloat16* cols = reinterpret_cast<__nv_bfloat16*>(d_ws);
    long long g = ((long long)rows + 255) / 256;
    if (g > (long long)mc_num_sms() * 32) g = (long long)mc_num_sms() * 32;
    if (C == 3 && (long long)B * 3 * H * W < (1ll << 31) && rows < (1ull << 31)) {
      im2col_first3_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, stream>>>(d_x, cols, (unsigned)rows, H, W,
                                                                                make_fastdiv(W + 1), make_fastdiv(H + 1));
      MC_LAUNCH_CHECK("im2col_first3_kernel");
    } else {
      im2col_first_kernel<<<(int)g, 256, 0, stream>>>(d_x, cols, B, H, W, C);
      MC_LAUNCH_CHECK("im2col_first_kernel");
    }
    if ((B % 2) == 0 && O == 32 && ld_dz == 32) {
      // Both operands are 32 columns wide, i.e. half of the 64-column (128-byte) rows the MN-major TMA boxes move: every
      // box would be half zero fill, and the kernel is bound by TMA bytes per k-block.  View both matrices as
      // [rows/2, 64] instead — row r holds pixel rows 2r and 2r+1 side by side.  The product of the doubled operands is
      // 64x64 with  D[p*32+o][q*32+j] = sum_r dZ[2r+p][o] * cols[2r+q][j];  the wanted gradient is the sum of its two
      // diagonal blocks (p == q), the off-diagonal blocks are discarded.  Half the k-blocks, no zero fill
      // (B even <=> the row count is even; the batch split B/2 only tells the callee the row count).
      uint8_t* w2 = reinterpret_cast<uint8_t*>(d_ws) + im2col;
      float* prod = reinterpret_cast<float*>(w2);
      uint8_t* ws2 = w2 + ((64 * 64 * sizeof(float) + 255) & ~(size_t)255);
      const size_t ws2_bytes = ws_bytes - im2col - ((64 * 64 * sizeof(float) + 255) & ~(size_t)255);
      int rc = mc_conv_wgrad(cols, 64, 64, d_dz, 64, 64, B / 2, H, W, 1, nullptr, prod, 0, ws2, ws2_bytes, stream_);
      if (rc) return rc;
      const int J = C * 9;
      wgrad_fold2_kernel<<<(O * J + 255) / 256, 256, 0, stream>>>(prod, d_mask, d_dw, O, J);
      MC_LAUNCH_CHECK("wgrad_fold2_kernel");
      return 0;
    }
    return mc_conv_wgrad(cols, 32, C * 9, d_dz, ld_dz, O, B, H, W, 1, d_mask, d_dw, 0,
                         reinterpret_cast<uint8_t*>(d_ws) + im2col, ws_bytes - im2col, stream_);
  }
  MC_CHECK_ARG(C >= 1 && C <= 4 && O >= 1 && O <= 32 && (O % 4) == 0 && (ld_dz % 4) == 0 && ld_dz >= O,
               "mc_conv_wgrad_first: needs C <= 4, O <= 32 (multiple of 4), 3x3 (got C=%d O=%d)", C, O);
  MC_CUDA(cudaMemsetAsync(d_dw, 0, sizeof(float) * (size_t)O * C * 9, stream));
  long long lines = (long long)B * H;
  int grid = mc_num_sms() * 4;
  if (grid > lines) grid = (int)lines;
  wgrad_first_kernel<<<grid, WF_THREADS, 0, stream>>>(d_x, (const __nv_bfloat16*)d_dz, ld_dz, B, H, W, C, O, d_dw);
  MC_LAUNCH_CHECK("wgrad_first_kernel");
  if (d_mask) {
    mul_inplace_kernel<<<4, 256, 0, stream>>>(d_dw, d_mask, (long long)O * C * 9);
    MC_LAUNCH_CHECK("mul_inplace_kernel");
  }
  return 0;
}


// ------------------------------------------------------------------------------------------------------------
// Fused momentum SGD over all parameters in ONE launch — replaces torch.optim.SGD.step() as configured by the
// reference (src/train.py:144-147: lr 1e-5, momentum 0.9, weight_decay 5e-4*batch, dampening 0, no nesterov;
// stepped at src/train.py:233-235), i.e. per element
//     d = g + wd * p;   buf = first_step ? d : momentum * buf + d;   p = p - lr * buf
// with the same fp32 operation order (fma(wd, p, g); mul then add; fma(-lr, buf, p)).  Pruned weights carry exactly
// zero gradients (the weight gradient kernels multiply by the mask), so they stay exactly zero: d = 0 + wd*0.
// ------------------------------------------------------------------------------------------------------------
namespace {
constexpr int SGD_MAX_SEG = 96;
struct SgdTable {
  float* p[SGD_MAX_SEG];
  const float* g[SGD_MAX_SEG];
  float* buf[SGD_MAX_SEG];
  unsigned int start4[SGD_MAX_SEG + 1];  // prefix sums of ceil(size / 4)
  unsigned int size[SGD_MAX_SEG];
  int nseg;
};

__global__ void __launch_bounds__(256) sgd_momentum_kernel(const __grid_constant__ SgdTable t, float lr, float momentum,
                                                           float wd, int first_step) {
  const unsigned int total4 = t.start4[t.nseg];
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += gridDim.x * blockDim.x) {
    int lo = 0, hi = t.nseg - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (t.start4[mid] <= i) lo = mid; else hi = mid - 1;
    }
    const unsigned int e0 = (i - t.start4[lo]) * 4u, n = t.size[lo];
    float* p = t.p[lo] + e0;
    const float* g = t.g[lo] + e0;
    float* b = t.buf[lo] + e0;
    if (e0 + 4u <= n && ((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)b)) & 15) == 0) {
      float4 pv = *reinterpret_cast<float4*>(p);
      const float4 gv = ld_stream_f4(reinterpret_cast<const float4*>(g));
      float4 bv = first_step ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<float4*>(b);
      float pe[4] = {pv.x, pv.y, pv.z, pv.w}, ge[4] = {gv.x, gv.y, gv.z, gv.w}, be[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float d = __fmaf_rn(wd, pe[j], ge[j]);
        be[j] = first_step ? d : __fadd_rn(__fmul_rn(be[j], momentum), d);
        pe[j] = __fmaf_rn(-lr, be[j], pe[j]);
      }
      *reinterpret_cast<float4*>(p) = make_float4(pe[0], pe[1], pe[2], pe[3]);
      *reinterpret_cast<float4*>(b) = make_float4(be[0], be[1], be[2], be[3]);
    } else {
      for (unsigned int j = 0; j < 4u && e0 + j < n; ++j) {
        const float d = __fmaf_rn(wd, p[j], g[j]);
        const float nb = first_step ? d : __fadd_rn(__fmul_rn(b[j], momentum), d);
        b[j] = nb;
        p[j] = __fmaf_rn(-lr, nb, p[j]);
      }
    }
  }
}
}  // namespace

extern "C" int mc_sgd_momentum_step(float* const* h_param_ptrs, const float* const* h_grad_ptrs, float* const* h_buf_ptrs,
                                    const int64_t* h_sizes, int nseg, float lr, float momentum, float weight_decay,
                                    int first_step, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MC_CHECK_ARG(h_param_ptrs && h_grad_ptrs && h_buf_ptrs && h_sizes && nseg > 0, "mc_sgd_momentum_step: bad argument");
  for (int s0 = 0; s0 < nseg; s0 += SGD_MAX_SEG) {
    SgdTable t;
    t.nseg = nseg - s0 < SGD_MAX_SEG ? nseg - s0 : SGD_MAX_SEG;
    unsigned long long acc = 0;
    for (int i = 0; i < t.nseg; ++i) {
      MC_CHECK_ARG(h_param_ptrs[s0 + i] && h_grad_ptrs[s0 + i] && h_buf_ptrs[s0 + i] && h_sizes[s0 + i] > 0 &&
                       h_sizes[s0 + i] < (1ll << 32),
                   "mc_sgd_momentum_step: bad segment %d", s0 + i);
      t.p[i] = h_param_ptrs[s0 + i];
      t.g[i] = h_grad_ptrs[s0 + i];
      t.buf[i] = h_buf_ptrs[s0 + i];
      t.size[i] = (unsigned int)h_sizes[s0 + i];
      t.start4[i] = (unsigned int)acc;
      acc += ((unsigned long long)h_sizes[s0 + i] + 3) / 4;
    }
    MC_CHECK_ARG(acc < (1ull << 32), "mc_sgd_momentum_step: too many elements in one launch");
    t.start4[t.nseg] = (unsigned int)acc;
    long long blocks = ((long long)acc + 255) / 256;
    const long long cap = (long long)mc_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    sgd_momentum_kernel<<<(int)blocks, 256, 0, stream>>>(t, lr, momentum, weight_decay, first_step);
    MC_LAUNCH_CHECK("sgd_momentum_kernel");
  }
  return 0;
}

// train_shrink.cu — the glue of the filter-shrunk retrain step (include/mcb200.h, "Filter-shrunk retrain step").
//
// The convolutions, BatchNorm and pool passes of a shrunk step are the ordinary retrain kernels run over compact shapes;
// these four kernels move parameters and gradients between the full [O, C, k, k] tensors the optimizer sees and the
// compact ones, and add what a dead filter still contributes in training mode (its constant activation leaky(beta),
// carried by one "ones" input column per consumer).  Each is one launch over every layer: blockIdx.y is the segment
// (layer), blockIdx.x strides over that layer's work.
#include "common.cuh"

namespace {

constexpr int SH_THREADS = 256;
constexpr int SH_BLOCKS_X = 256;  // per segment: blocks of a small layer exit at once, the large ones keep every SM busy

__device__ __forceinline__ float act_of(float b, int leaky) { return (leaky && !(b > 0.f)) ? b * 0.1f : b; }
// nn.LeakyReLU's backward: slope 0.1 where the input is not > 0 (so also at exactly 0)
__device__ __forceinline__ float act_slope(float b, int leaky) { return (leaky && !(b > 0.f)) ? 0.1f : 1.f; }

__device__ __forceinline__ float wm(const mc_shrink_seg& s, size_t e) {
  const float v = s.w[e];
  return s.mask ? v * s.mask[e] : v;
}

__global__ void __launch_bounds__(SH_THREADS)
shrink_prepare_kernel(const mc_shrink_seg* __restrict__ segs, const int* __restrict__ idx, float* __restrict__ cbn,
                      float* __restrict__ lk) {
  const mc_shrink_seg s = segs[blockIdx.y];
  if (!s.gamma) return;
  const int* oidx = idx + s.oidx;
  const unsigned int stride = gridDim.x * blockDim.x;
  // rounded to bf16: the value a dead channel's stored activation holds in the dense step
  for (unsigned int f = blockIdx.x * blockDim.x + threadIdx.x; f < (unsigned int)s.O; f += stride)
    lk[s.lk_off + f] = __bfloat162float(__float2bfloat16_rn(act_of(s.beta[f], s.leaky)));
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < (unsigned int)s.n_o; i += stride) {
    const int f = oidx[i];
    float* c = cbn + s.cbn_off + i;
    c[0] = s.gamma[f];
    c[s.cbn_ld] = s.beta[f];
    if (s.rmean) {
      c[2 * s.cbn_ld] = s.rmean[f];
      c[3 * s.cbn_ld] = s.rvar[f];
    }
  }
}

__global__ void __launch_bounds__(SH_THREADS)
shrink_pack_kernel(const mc_shrink_seg* __restrict__ segs, const int* __restrict__ idx, const float* __restrict__ lk,
                   __nv_bfloat16* __restrict__ wp, __nv_bfloat16* __restrict__ wpd) {
  const mc_shrink_seg s = segs[blockIdx.y];
  if (s.kc == 0) return;
  const int* oidx = idx + s.oidx;
  const int* colmap = idx + s.colmap;
  const int* clk = idx + s.clk;
  const int* dead = idx + s.dead_in;
  const unsigned int stride = gridDim.x * blockDim.x;
  // forward pack, element i = (n, tap, j) in the output's own order (consecutive threads store consecutive columns)
  const unsigned int tk = (unsigned int)s.taps * s.kc, nf = (unsigned int)s.npad * tk;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < nf; i += stride) {
    const unsigned int n = i / tk, r = i - n * tk, t = r / s.kc, j = r - t * s.kc;
    float v = 0.f;
    if (n < (unsigned int)s.n_o && s.ones_col >= 0 && ((int)j == s.ones_col || (int)j == s.ones_col + 1))
      continue;  // written by the warps below
    if (n < (unsigned int)s.n_o && j < (unsigned int)s.n_col) {
      const int m = colmap[j];
      if (m >= 0) v = wm(s, ((size_t)oidx[n] * s.C + m) * s.taps + t);
    }
    wp[s.wp_off + i] = __float2bfloat16_rn(v);
  }
  // the ones columns: one warp per (filter, tap) sums bf16(W*mask) * lk over the dead inputs in fp32 (the products of
  // the dense step's operands, exact in fp32), in a fixed order; the sum is stored as a high and a low bf16 half
  if (s.ones_col >= 0) {
    const unsigned int lane = threadIdx.x & 31, nw = (unsigned int)s.n_o * s.taps;
    for (unsigned int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < nw; u += stride >> 5) {
      const unsigned int n = u / s.taps, t = u - n * s.taps;
      const size_t row = (size_t)oidx[n] * s.C;
      float v = 0.f;
      for (int d = lane; d < s.n_dead; d += 32) {
        const int c = dead[d];
        v = __fmaf_rn(__bfloat162float(__float2bfloat16_rn(wm(s, (row + c) * s.taps + t))), lk[clk[c]], v);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) {
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        __nv_bfloat16* dst = wp + s.wp_off + (size_t)n * tk + t * s.kc + s.ones_col;
        dst[0] = hi;
        dst[1] = __float2bfloat16_rn(v - __bfloat162float(hi));
      }
    }
  }
  if (!wpd) return;
  // data-gradient pack [cpad, taps*ko]: row = physical column c, column tap'*ko + n.  A transpose of the forward
  // layout, so it goes through a 32 x 32 shared-memory tile per (tap, filter block, column block): the source is read
  // with consecutive threads on consecutive input columns, the destination written with them on consecutive filters.
  __shared__ float tile[32][33];
  const unsigned int nb = ((unsigned int)s.ko + 31) / 32, cb = ((unsigned int)s.cpad + 31) / 32;
  const unsigned int ntiles = (unsigned int)s.taps * nb * cb, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const unsigned int tko = (unsigned int)s.taps * s.ko;
  for (unsigned int u = blockIdx.x; u < ntiles; u += gridDim.x) {
    const unsigned int t = u / (nb * cb), r = u - t * nb * cb, n0 = (r / cb) * 32, c0 = (r % cb) * 32;
    for (unsigned int k = ty; k < 32; k += SH_THREADS / 32) {
      const unsigned int n = n0 + k, c = c0 + tx;
      float v = 0.f;
      const int m = c < (unsigned int)s.n_col ? colmap[c] : -1;
      if (m >= 0 && n < (unsigned int)s.n_o) v = wm(s, ((size_t)oidx[n] * s.C + m) * s.taps + (s.taps - 1 - t));
      tile[k][tx] = v;
    }
    __syncthreads();
    for (unsigned int k = ty; k < 32; k += SH_THREADS / 32) {
      const unsigned int c = c0 + k, n = n0 + tx;
      if (c < (unsigned int)s.cpad && n < (unsigned int)s.ko)
        wpd[s.wpd_off + (size_t)c * tko + t * s.ko + n] = __float2bfloat16_rn(tile[tx][k]);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(SH_THREADS)
shrink_stats_kernel(const mc_shrink_seg* __restrict__ segs, const int* __restrict__ idx, const float* __restrict__ cbn) {
  const mc_shrink_seg s = segs[blockIdx.y];
  if (!s.rmean) return;
  const int* orow = idx + s.orow;
  const float mom = s.momentum;
  for (unsigned int f = blockIdx.x * blockDim.x + threadIdx.x; f < (unsigned int)s.O; f += gridDim.x * blockDim.x) {
    const int r = orow[f];
    if (r >= 0) {
      s.rmean[f] = cbn[s.cbn_off + 2 * s.cbn_ld + r];
      s.rvar[f] = cbn[s.cbn_off + 3 * s.cbn_ld + r];
    } else {
      // mc_bn_finalize with batch mean = 0 and unbiased variance = 0 (a dead filter's z is exactly 0)
      const float zero = 0.f;
      s.rmean[f] = (1.f - mom) * s.rmean[f] + mom * zero;
      s.rvar[f] = (1.f - mom) * s.rvar[f] + mom * zero;
    }
  }
}

__global__ void __launch_bounds__(SH_THREADS)
shrink_finish_kernel(const mc_shrink_seg* __restrict__ segs, const int* __restrict__ idx, const float* __restrict__ lk,
                     const float* __restrict__ dwc, float* __restrict__ grad) {
  const mc_shrink_seg s = segs[blockIdx.y];
  const int* orow = idx + s.orow;
  const int* cphys = idx + s.cphys;
  const int* clk = idx + s.clk;
  const unsigned int stride = gridDim.x * blockDim.x;
  // full dW
  const unsigned int ct = (unsigned int)s.C * s.taps, nw = (unsigned int)s.O * ct;
  const float* gc = dwc + s.dwc_off;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += stride) {
    const unsigned int o = i / ct, r = i - o * ct, c = r / s.taps, t = r - c * s.taps;
    const int row = orow[o];
    float v = 0.f;
    if (row >= 0) {
      const size_t base = (size_t)row * s.n_col * s.taps + t;
      const int p = cphys[c];
      if (p >= 0)
        v = gc[base + (size_t)p * s.taps];
      else if (s.ones_col >= 0 && clk[c] >= 0)
        v = lk[clk[c]] * gc[base + (size_t)s.ones_col * s.taps];
      if (s.mask) v *= s.mask[i];
    }
    grad[s.dw_off + i] = v;
  }
  if (!s.gamma) return;
  // alive dgamma / dbeta: scatter; dead: dgamma = 0, dbeta = act'(beta) * sum over the consumer inputs (below)
  const float* cdb = dwc + s.cdgb_off;
  for (unsigned int f = blockIdx.x * blockDim.x + threadIdx.x; f < (unsigned int)s.O; f += stride) {
    const int row = orow[f];
    if (row >= 0) grad[s.dbn_off + f] = cdb[row];
    grad[s.dbn_off + s.O + f] = row >= 0 ? cdb[s.n_o + row] : 0.f;
  }
  // dead dbeta: one block per dead filter, a fixed-order block reduction over its consumer inputs' (filter, tap) pairs
  const int* cptr = idx + s.cons_ptr;
  const int* cons = idx + s.cons;
  __shared__ float red[SH_THREADS / 32];
  for (unsigned int f = blockIdx.x; f < (unsigned int)s.O; f += gridDim.x) {
    if (orow[f] >= 0 || cptr[f] == cptr[f + 1]) {
      if (orow[f] < 0 && threadIdx.x == 0) grad[s.dbn_off + f] = 0.f;
      continue;
    }
    float acc = 0.f;
    for (int e = cptr[f]; e < cptr[f + 1]; ++e) {
      const mc_shrink_seg& q = segs[cons[2 * e]];
      const int cin = cons[2 * e + 1], qtaps = q.taps, qC = q.C, qn = q.n_col, qones = q.ones_col;
      if (qones < 0) continue;
      const int* qo = idx + q.oidx;
      const float* g1 = dwc + q.dwc_off + (size_t)qones * qtaps;
      const int n = q.n_o * qtaps;
      for (int k = threadIdx.x; k < n; k += SH_THREADS) {
        const int r = k / qtaps, t = k - r * qtaps;
        acc = __fmaf_rn(wm(q, ((size_t)qo[r] * qC + cin) * qtaps + t), g1[(size_t)r * qn * qtaps + t], acc);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
      for (int w = 0; w < SH_THREADS / 32; ++w) tot += red[w];
      grad[s.dbn_off + f] = act_slope(s.beta[f], s.leaky) * tot;
    }
    __syncthreads();
  }
}

inline dim3 seg_grid(int nseg) { return dim3(SH_BLOCKS_X, nseg); }

}  // namespace

#define SH_ARGS(name)                                                                                          \
  MC_CHECK_ARG(d_segs && d_idx && nseg > 0 && nseg <= MC_MAX_SEGMENTS, name ": bad argument (nseg %d)", nseg)

extern "C" int mc_shrink_prepare(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, float* d_cbn, float* d_lk,
                                 void* stream) {
  SH_ARGS("mc_shrink_prepare");
  MC_CHECK_ARG(d_cbn && d_lk, "mc_shrink_prepare: null buffer");
  shrink_prepare_kernel<<<seg_grid(nseg), SH_THREADS, 0, (cudaStream_t)stream>>>(d_segs, d_idx, d_cbn, d_lk);
  MC_LAUNCH_CHECK("shrink_prepare_kernel");
  return 0;
}

extern "C" int mc_shrink_pack(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_lk, void* d_wp,
                              void* d_wpd, void* stream) {
  SH_ARGS("mc_shrink_pack");
  MC_CHECK_ARG(d_lk && d_wp, "mc_shrink_pack: null buffer");
  shrink_pack_kernel<<<seg_grid(nseg), SH_THREADS, 0, (cudaStream_t)stream>>>(
      d_segs, d_idx, d_lk, (__nv_bfloat16*)d_wp, (__nv_bfloat16*)d_wpd);
  MC_LAUNCH_CHECK("shrink_pack_kernel");
  return 0;
}

extern "C" int mc_shrink_stats(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_cbn,
                               void* stream) {
  SH_ARGS("mc_shrink_stats");
  MC_CHECK_ARG(d_cbn, "mc_shrink_stats: null buffer");
  shrink_stats_kernel<<<seg_grid(nseg), SH_THREADS, 0, (cudaStream_t)stream>>>(d_segs, d_idx, d_cbn);
  MC_LAUNCH_CHECK("shrink_stats_kernel");
  return 0;
}

extern "C" int mc_shrink_finish(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_lk,
                                const float* d_dwc, float* d_grad, void* stream) {
  SH_ARGS("mc_shrink_finish");
  MC_CHECK_ARG(d_lk && d_dwc && d_grad, "mc_shrink_finish: null buffer");
  shrink_finish_kernel<<<seg_grid(nseg), SH_THREADS, 0, (cudaStream_t)stream>>>(d_segs, d_idx, d_lk, d_dwc, d_grad);
  MC_LAUNCH_CHECK("shrink_finish_kernel");
  return 0;
}

"""Bit-exact tests of the forward convolution kernels: every store path, epilogue mode and CTA configuration of
mc_conv_fwd (single CTA with 1, 2 or 3 CTAs per SM, CTA pair with and without the stream-K tail), its batch statistics,
the data gradient through mc_pack_conv_weights_dgrad, and the thin-layer kernels (mc_conv_im2col_fwd,
mc_conv_window_fwd, mc_conv_thin_fwd, mc_conv_direct_fwd).

Method (see test_gpu_split_exact.py for the premise that tcgen05 accumulates integer-valued bf16 products exactly).
Operands are small integers (uint8 images: bf16(x/255), multiples of 2^-15), and each test asserts on its own data that
the sum of |terms| of an output stays below 2^24 quanta, so every fp32 partial sum is exact in any order.  The reference
then reproduces the epilogue's arithmetic instead of a tolerance: acc from a float64 convolution, v = fp32(acc * scale +
shift) (exact in float64, rounded once: what fmaf gives; asserted per element), leaky as max(v, v * 0.1f) in fp32, the
2x2 max for pooled kernels, and round-to-nearest-even to bf16.  Two data regimes: outputs that bf16 holds exactly
(layouts, canaries, statistics) and outputs of 2^8 .. 2^15 with dyadic scales and odd shifts, whose many fp32 values
exactly halfway between two bf16 values tell round-to-nearest-even from truncation or rounding half away from zero.

Every output allocation is filled with NaN before the launch and is larger than the output (rows after the last row,
channels before ch_off and after the written ones), and every byte of it is compared, so a store to a neighbouring
concat slice or past the tensor fails like a wrong value.  Inputs get NaN in the rows after the tensor and in the
columns the tensor map does not cover, and 2^20 in columns [Cin, in_cols) that meet zero weights.
"""
import ctypes
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from modelcompression_b200 import _lib
from modelcompression_b200.engine import _c_floats, _pool_window_weights, _thin_host_weights
from test_gpu_split_exact import BOUND, _gen, _ints, _pack

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
PNHWC, REORG2, NCHW = _lib.MC_EPI_PNHWC, _lib.MC_EPI_REORG2, _lib.MC_EPI_NCHW_F32
FIELDS = ('pair', 'ctas', 'block_n', 'block_k', 'stages', 'a_stages', 'share', 'grid', 'm_tiles', 'n_tiles', 'sk_units',
          'store', 'tma_bufs', 'wide_ld', 'vec_ok', 'last_ksteps')
STORE = {0: 'direct', 1: 'staged', 2: 'tma'}
EXTRA_ROWS = 160        # canary rows after every PNHWC tensor
NAN16 = 0x7FC1          # bf16 canary (a NaN)
TIES = 1000             # exact bf16 ties the rounding-regime data must contain
F32_01 = torch.tensor(0.1, dtype=torch.float32)


def _r(x, m):
    return (x + m - 1) // m * m


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _canary(shape, dtype=torch.bfloat16):
    if dtype == torch.bfloat16:
        return torch.full(shape, NAN16, dtype=torch.int16, device=DEV).view(torch.bfloat16)
    return torch.full(shape, float('nan'), dtype=dtype, device=DEV)


def _assert_bits(got, want, what):
    """Bitwise equality (NaN canaries included); the first differing element is reported with its index."""
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (g.shape, w.shape)
    bad = (g != w).nonzero()
    if bad.shape[0]:
        i = tuple(bad[0].tolist())
        raise AssertionError("%s: %d of %d elements differ; first at %s: got %r, want %r" % (
            what, bad.shape[0], g.numel(), i, got[i].item(), want[i].item()))


def _data(shape, regime, K, g):
    """Integer operands.  exact: |v| <= 2, sparse enough that an output's std is ~8 (|y| well below 256);
    round: dense |v| <= vmax with vmax chosen so that the accumulators reach ~2^10 (K terms each)."""
    if regime == 'round':
        vmax = max(2, min(127, int(round(math.sqrt(3 * 1024 / math.sqrt(K))))))
        return _ints(shape, 1.0, g, vmax)
    return _ints(shape, min(1.0, 8.0 / (2.5 * math.sqrt(K))), g)


def _scale_shift(N, Npad, regime, g):
    """Per-channel scale / shift (zero beyond N, as the engine pads them).  round: dyadic scales, odd shifts."""
    sc, sh = torch.zeros(Npad, device=DEV), torch.zeros(Npad, device=DEV)
    if regime == 'round':
        sc[:N] = torch.tensor([1.0, 0.5, 0.25, 0.125, -0.5, 2.0], device=DEV).repeat(N // 6 + 1)[:N]
        sh[:N] = (torch.randint(-32, 32, (N,), device=DEV, generator=g) * 2 + 1).float()
    else:
        sc[:N] = torch.tensor([1.0, -1.0, 1.0], device=DEV).repeat(N // 3 + 1)[:N]
        sh[:N] = torch.randint(-3, 4, (N,), device=DEV, generator=g).float()
    return sc, sh


def _assert_exact_sum(K, x, w, q=1.0):
    """Every term of an output is a multiple of q and K of them are summed: the sum of |terms| < 2^24 q."""
    s = K * float(x.abs().max()) * float(w.abs().max())
    assert s < BOUND * q, "test data leaves the exact range: %g >= 2^24 * %g" % (s, q)


def _epilogue(acc, sc, sh, leaky):
    """fp32(acc * scale + shift) per channel (dim 1), as fmaf computes it, then leaky in fp32.  acc and scale hold at most
    24 significant bits each, so the float64 product is exact; the sum is checked exact (two-sum error zero) and then
    rounded once."""
    p = acc * sc.double().view(1, -1, 1, 1)
    c = sh.double().view(1, -1, 1, 1).expand_as(p)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    assert bool((err == 0).all()), "float64 reference of the epilogue is not exact"
    v = s.float()
    if leaky:
        v = torch.maximum(v, v * F32_01.to(v.device))
    return v


def _ties(v):
    """fp32 values exactly halfway between two bf16 values"""
    return int(((v.view(torch.int32) & 0xFFFF) == 0x8000).sum())


# ----------------------------------------------------------------------------------------------- mc_conv_fwd cases
def C(name, B, H, W, Cin, N, k, **kw):
    c = dict(name=name, B=B, H=H, W=W, Cin=Cin, N=N, k=k, mode=PNHWC, leaky=1, regime='exact', ch_off=0, ldc=None,
             block_n=0, stages=0, block_k=0, in_extra=0, in_off=0, ws=False, stats=False, want={}, cell=None)
    c.update(kw)
    return c


PAIR = dict(pair=1)
CASES = [
    # single CTA, TMA-store epilogue: 2 slabs + 64-column loads with one CTA per SM, 1 slab with several
    C("k1 tma wide_ld round", 2, 26, 26, 256, 256, 3, block_n=128, regime='round',
      want=dict(pair=0, ctas=1, store=2, tma_bufs=2, wide_ld=1, share=1, last_ksteps=4), cell=('k1', 'tma')),
    C("k2 tma 1 slab round", 16, 52, 52, 64, 64, 1, block_n=64, leaky=0, regime='round',
      want=dict(ctas=2, store=2, tma_bufs=1, wide_ld=0), cell=('k2', 'tma')),
    C("k3 tma 1 slab", 32, 52, 52, 32, 64, 1, block_n=64, block_k=32, want=dict(ctas=3, store=2, tma_bufs=1), cell=('k3', 'tma')),
    C("k3 narrow 1x1 direct", 16, 104, 104, 24, 8, 1, block_k=32, want=dict(ctas=3, block_n=16, store=0), cell=('k3', 'direct')),
    C("bn80 concat ch_off", 2, 20, 20, 72, 80, 3, block_n=80, stages=2, ch_off=16, ldc=112,
      want=dict(ctas=1, stages=2, share=1, block_n=80, store=2, last_ksteps=1), cell=('k1', 'tma')),
    C("bn208 ch_off 64 round", 2, 26, 26, 48, 200, 3, block_n=208, ch_off=64, ldc=320, regime='round',
      want=dict(pair=0, block_n=208, store=2, last_ksteps=3)),
    C("bn256 two n-tiles ragged", 2, 13, 13, 32, 500, 1, block_n=256, block_k=32, regime='round',
      want=dict(block_n=256, n_tiles=2, block_k=32, last_ksteps=2, store=2)),
    # staged store (32 / 48 wide), explicit one-stage ring without the shared box
    C("staged 48 bk32", 4, 104, 104, 16, 40, 3, block_n=48, block_k=32, regime='round',
      want=dict(store=1, block_k=32, share=0, last_ksteps=1), cell=('k2', 'staged')),
    C("staged 32 stages 1", 2, 40, 24, 40, 32, 1, block_n=32, stages=1,
      want=dict(ctas=1, stages=1, share=0, store=1), cell=('k1', 'staged')),
    C("staged one partial tile", 1, 8, 8, 64, 30, 3, block_n=32, want=dict(m_tiles=1, store=1, share=1, last_ksteps=4)),
    C("staged bk32 unshared", 2, 26, 26, 32, 48, 3, block_n=48, block_k=32, want=dict(share=0, block_k=32, store=1)),
    # direct stores: 16-wide tiles, misaligned ch_off / ldc, 32-wide k-blocks with the shared box (>= 2048 m-tiles)
    C("direct bn16 odd image round", 8, 13, 21, 24, 12, 3, block_n=16, block_k=32, regime='round',
      want=dict(store=0, block_n=16, last_ksteps=2)),
    C("direct bk32 shared box wrap", 8, 208, 208, 32, 16, 3, block_k=32, block_n=16,
      want=dict(share=1, block_k=32, store=0)),
    C("direct wrap stages 4", 8, 104, 104, 16, 32, 1, block_n=16, stages=4, block_k=32,
      want=dict(ctas=1, stages=4, n_tiles=2, store=0), cell=('k1', 'direct')),
    C("direct misaligned ch_off", 2, 26, 26, 64, 100, 3, block_n=128, ch_off=4, ldc=112,
      want=dict(store=0, vec_ok=0), cell=('k1', 'direct')),
    C("direct misaligned ldc", 2, 17, 15, 136, 70, 1, block_n=80, ldc=75, regime='round',
      want=dict(store=0, vec_ok=0, last_ksteps=1)),
    # REORG2 and NCHW fp32
    C("reorg N%8==0", 2, 26, 26, 64, 64, 1, mode=REORG2, ch_off=32, ldc=296, want=dict(vec_ok=1), cell=('k1', 'reorg')),
    C("reorg N%8!=0", 2, 14, 22, 40, 36, 3, mode=REORG2, ldc=152, regime='round', want=dict(vec_ok=0)),
    C("nchw leaky 0 round", 2, 13, 13, 200, 125, 1, mode=NCHW, leaky=0, regime='round', cell=('k1', 'nchw')),
    C("nchw leaky 1", 3, 9, 11, 20, 40, 3, mode=NCHW),
    # CTA pair, with and without the stream-K tail
    C("pair tma sk", 24, 13, 13, 512, 1024, 3, ws=True, want=dict(PAIR, store=2), cell=('pair sk', 'tma')),
    C("pair tma round", 24, 13, 13, 512, 1024, 3, regime='round', want=dict(PAIR, sk_units=0, store=2),
      cell=('pair', 'tma')),
    C("pair misaligned sk", 16, 26, 26, 512, 1024, 3, ws=True, ch_off=4, ldc=1032, want=dict(PAIR, store=0, vec_ok=0),
      cell=('pair sk', 'direct')),
    C("pair misaligned", 24, 13, 13, 512, 1024, 3, ch_off=4, ldc=1036, want=dict(PAIR, sk_units=0, vec_ok=0),
      cell=('pair', 'direct')),
    C("pair reorg sk", 16, 26, 26, 512, 1024, 3, mode=REORG2, ws=True, ldc=4096, want=dict(PAIR, vec_ok=1),
      cell=('pair sk', 'reorg')),
    C("pair reorg ragged sk", 16, 26, 26, 1006, 1018, 3, mode=REORG2, ws=True, ldc=4072, want=dict(PAIR, vec_ok=0)),
    C("pair reorg", 24, 14, 14, 512, 1024, 3, mode=REORG2, ldc=4096, block_n=256, want=dict(PAIR, sk_units=0), cell=('pair', 'reorg')),
    C("pair nchw sk", 24, 13, 13, 512, 1024, 3, mode=NCHW, ws=True, want=dict(PAIR), cell=('pair sk', 'nchw')),
    C("pair nchw leaky 0", 24, 13, 13, 512, 1024, 3, mode=NCHW, leaky=0, want=dict(PAIR, sk_units=0),
      cell=('pair', 'nchw')),
    # input slices: in_cols > Cin, the input pointer 2 * in_off bytes into the row
    C("input slice in_cols", 2, 26, 26, 40, 64, 3, in_off=8, in_extra=16, want=dict(last_ksteps=3)),
    C("input slice 1x1 bk32", 2, 13, 13, 24, 48, 1, in_off=24, in_extra=8, block_k=32),
]
STAT_CASES = [
    C("stats k1", 2, 26, 26, 64, 128, 3, want=dict(ctas=1, store=2)),
    C("stats k2", 16, 52, 52, 32, 64, 1, block_k=32, want=dict(ctas=2)),
    C("stats k3", 32, 52, 52, 32, 64, 1, block_k=32, want=dict(ctas=3)),
    C("stats five n-tiles", 2, 26, 26, 48, 300, 3, block_n=64, want=dict(n_tiles=5)),
    C("stats N=33", 2, 20, 20, 16, 33, 3),
    C("stats ragged ch_off", 2, 26, 26, 40, 100, 1, ch_off=64, ldc=176),
    C("stats pair", 24, 13, 13, 512, 1024, 3, want=dict(PAIR, sk_units=0)),
    # the retrain's 26x26 256 -> 512 layer at batch 16: 256-wide tiles give 46 m-pairs x 2 = 92 units over 74 clusters
    # (the planner's own 192-wide tiles give 138 units: no tail)
    C("stats pair sk", 16, 26, 26, 256, 512, 3, block_n=256, ws=True, want=dict(PAIR, block_n=256)),
]
for _c in STAT_CASES:
    _c.update(stats=True, leaky=0)
for _c in CASES + STAT_CASES:
    if _c['ws'] and _c['want'].get('pair'):
        _c['want'] = dict(_c['want'], sk_pos=1)


def _desc(c, bufs):
    d = _lib.mc_conv_desc()
    d.d_in, d.d_wpack = bufs['in_ptr'], bufs['wpack'].data_ptr()
    d.d_scale, d.d_shift, d.d_out = bufs['sc'].data_ptr(), bufs['sh'].data_ptr(), bufs['out'].data_ptr()
    d.B, d.H, d.W, d.Cin, d.Cin_ld = c['B'], c['H'], c['W'], c['Cin'], bufs['Cin_ld']
    d.N, d.Npad, d.ksize, d.leaky, d.epi_mode = c['N'], _r(c['N'], 16), c['k'], c['leaky'], c['mode']
    d.ldc, d.ch_off = bufs['ldc'], c['ch_off'] if c['mode'] != NCHW else 0
    d.block_n, d.stages, d.block_k = c['block_n'], c['stages'], c['block_k']
    d.in_cols = c['Cin'] + c['in_extra'] if c['in_extra'] else 0
    if c['stats']:
        d.d_stat_sum, d.d_stat_sumsq = bufs['ssum'].data_ptr(), bufs['ssq'].data_ptr()
    if c['ws']:
        n = int(_lib.load().mc_workspace_bytes_conv_fwd(ctypes.byref(d)))
        assert n > 0
        bufs['ws'] = torch.zeros(n, dtype=torch.uint8, device=DEV)
        d.d_ws, d.ws_bytes = bufs['ws'].data_ptr(), n
    return d


def _plan(d):
    info = (ctypes.c_int * 16)()
    _lib.check(_lib.load().mc_conv_fwd_plan(ctypes.byref(d), info), "mc_conv_fwd_plan")
    return dict(zip(FIELDS, info))


def _show(p):
    return " ".join("%s=%d" % (f, p[f]) for f in FIELDS)


def _cell(p, mode):
    kern = ('pair sk' if p['sk_units'] else 'pair') if p['pair'] else 'k%d' % p['ctas']
    return kern, {PNHWC: STORE[p['store']], REORG2: 'reorg', NCHW: 'nchw'}[mode]


def _check_want(c, p):
    for key, val in c['want'].items():
        if key == 'sk_pos':
            assert p['sk_units'] > 0, "%s: no stream-K tail: %s" % (c['name'], _show(p))
        else:
            assert p[key] == val, "%s: %s = %d, want %d (%s)" % (c['name'], key, p[key], val, _show(p))
    if c['cell'] is not None:
        assert _cell(p, c['mode']) == c['cell'], (c['name'], _cell(p, c['mode']), _show(p))


def _buffers(c):
    """Operands, canaried input / output allocations and the descriptor of a case."""
    B, H, W, Cin, N, k = c['B'], c['H'], c['W'], c['Cin'], c['N'], c['k']
    g = _gen(zlib.crc32(c['name'].encode()) & 0xFFFF)
    K = Cin * k * k
    x = _data((B, Cin, H, W), c['regime'], K, g)
    w = _data((N, Cin, k, k), c['regime'], K, g)
    Npad = _r(N, 16)
    sc, sh = _scale_shift(N, Npad, 'exact' if c['stats'] else c['regime'], g)
    rows = B * (H + 1) * (W + 1)
    in_off, extra = c['in_off'], c['in_extra']
    Cin_ld = _r(in_off + Cin + extra, 8) + 8 if (in_off or extra) else _r(Cin, 8)
    xin = _canary((rows + EXTRA_ROWS, Cin_ld))
    packed, _ = _pack(x)
    xin[:rows, in_off:in_off + Cin] = packed[:, :Cin]
    if extra:
        xin[:rows, in_off + Cin:in_off + Cin + extra] = 2.0 ** 20
    bk = c['block_k'] or 64
    Kc = _r(Cin, bk)
    wpack = torch.empty(Npad, k * k * Kc, dtype=torch.bfloat16, device=DEV)
    lib = _lib.load()
    _lib.check(lib.mc_pack_conv_weights(w.data_ptr(), None, N, Cin, k, None, N, None, Cin, wpack.data_ptr(), Npad, Kc,
                                        _lib.stream_ptr()), "mc_pack_conv_weights")
    mode, ch_off = c['mode'], c['ch_off']
    if mode == PNHWC:
        ldc = c['ldc'] or _r(ch_off + N, 8) + 8
        out = _canary((rows + EXTRA_ROWS, ldc))
    elif mode == REORG2:
        ldc = c['ldc']
        out = _canary((B * (H // 2 + 1) * (W // 2 + 1) + EXTRA_ROWS, ldc))
    else:
        ldc = N
        out = _canary((B * N * H * W + 4096,), torch.float32)
    bufs = dict(x=x, w=w, sc=sc, sh=sh, xin=xin, in_ptr=xin.data_ptr() + 2 * in_off, Cin_ld=Cin_ld, wpack=wpack,
                out=out, ldc=ldc, K=K)
    if c['stats']:
        bufs['ssum'] = torch.cat([torch.zeros(N, device=DEV), _canary((16,), torch.float32)])
        bufs['ssq'] = bufs['ssum'].clone()
    bufs['d'] = _desc(c, bufs)
    return bufs


def _expected(c, bufs, p, yb):
    """The whole output allocation as the kernel must leave it."""
    B, H, W, N, ch_off, ldc, mode = c['B'], c['H'], c['W'], c['N'], c['ch_off'], bufs['ldc'], c['mode']
    exp = bufs['out'].clone()
    if mode == NCHW:
        exp[:B * N * H * W] = yb.flatten()
        return exp
    if mode == PNHWC:
        rows = B * (H + 1) * (W + 1)
        v = exp[:rows].view(B, H + 1, W + 1, ldc)
        # pad rows are written (zeros); with 16-byte stores so are channels [N, round8(N)) of every row
        v[..., ch_off:ch_off + (_r(N, 8) if p['vec_ok'] else N)] = 0
        v[:, :H, :W, ch_off:ch_off + N] = yb.permute(0, 2, 3, 1)
        return exp
    Ho, Wo = H // 2, W // 2
    v = exp[:B * (Ho + 1) * (Wo + 1)].view(B, Ho + 1, Wo + 1, ldc)
    for i in range(2):
        for j in range(2):
            q = ch_off + (i * 2 + j) * N
            v[:, :Ho, :Wo, q:q + N] = yb[:, :, i::2, j::2].permute(0, 2, 3, 1)
    return exp



def _reference(c, bufs):
    x, w, K = bufs['x'], bufs['w'], bufs['K']
    _assert_exact_sum(K, x, w)
    acc = F.conv2d(x.double(), w.double(), None, 1, c['k'] // 2)
    return _epilogue(acc, bufs['sc'][:c['N']], bufs['sh'][:c['N']], c['leaky'])


def _run(c):
    bufs = _buffers(c)
    d = bufs['d']
    p = _plan(d)
    print(c['name'], _show(p))
    _check_want(c, p)
    v = _reference(c, bufs)
    if c['regime'] == 'round' and c['mode'] != NCHW:
        assert _ties(v) >= TIES, "%s: only %d bf16 ties in the data" % (c['name'], _ties(v))
    yb = v if c['mode'] == NCHW else v.bfloat16()
    if c['mode'] != NCHW and c['regime'] == 'exact' and c['stats']:
        assert float(v.abs().max()) <= 256 and torch.equal(yb.float(), v), "outputs must be exact in bf16"
    with torch.cuda.device(0):
        _lib.check(_lib.load().mc_conv_fwd(ctypes.byref(d), _lib.stream_ptr()), "mc_conv_fwd")
    torch.cuda.synchronize()
    _assert_bits(bufs['out'], _expected(c, bufs, p, yb), "%s [%s]" % (c['name'], _show(p)))
    if c['ws']:
        assert int(bufs['ws'][:2048].count_nonzero()) == 0, "stream-K counters not left zero"
    return bufs, yb, p


@pytest.mark.parametrize("c", CASES, ids=[c['name'].replace(" ", "_") for c in CASES])
def test_conv_fwd_bit_exact(c):
    _run(c)


def test_conv_fwd_plans_reach_every_cell():
    """No launch: the cases above still reach every (kernel x store path x mode) cell, and the staged store only ever
    takes 32- or 48-wide tiles (the planner sends every wider aligned PNHWC tile to the TMA stores)."""
    need = {('k1', 'tma'), ('k2', 'tma'), ('k3', 'tma'), ('k1', 'staged'), ('k2', 'staged'), ('k1', 'direct'),
            ('k3', 'direct'), ('k1', 'reorg'), ('k1', 'nchw'), ('pair', 'tma'), ('pair sk', 'tma'), ('pair', 'direct'),
            ('pair sk', 'direct'), ('pair', 'reorg'), ('pair sk', 'reorg'), ('pair', 'nchw'), ('pair sk', 'nchw')}
    seen, plans = set(), []
    for c in CASES + STAT_CASES:
        bufs = _buffers(c)
        p = _plan(bufs['d'])
        del bufs
        print("%-32s %-20s %s" % (c['name'], _cell(p, c['mode']), _show(p)))
        _check_want(c, p)
        seen.add(_cell(p, c['mode']))
        plans.append((c, p))
    assert need <= seen, "cells not reached: %s" % sorted(need - seen)
    assert {p['block_n'] for _, p in plans if p['store'] == 1} <= {32, 48}
    assert {p['tma_bufs'] for _, p in plans if p['store'] == 2} == {1, 2}
    assert {p['wide_ld'] for _, p in plans if p['store'] == 2 and not p['pair']} == {0, 1}
    assert {p['last_ksteps'] for _, p in plans} >= {1, 2, 3, 4}
    assert {p['block_k'] for _, p in plans} == {32, 64}
    assert any(p['share'] and p['block_k'] == 32 and p['m_tiles'] >= 2048 for _, p in plans)
    assert any(p['stages'] == 1 and not p['share'] for _, p in plans) and any(
        c['stages'] == 2 and p['share'] for c, p in plans)
    assert {p['block_n'] for _, p in plans} >= {16, 32, 48, 64, 80, 128, 208, 256}
    assert any(p['m_tiles'] == 1 for _, p in plans)
    assert any(p['m_tiles'] * p['n_tiles'] >= 8 * p['grid'] for _, p in plans if not p['pair'])
    assert any(c['mode'] == REORG2 and p['vec_ok'] for c, p in plans) and any(
        c['mode'] == REORG2 and not p['vec_ok'] for c, p in plans)
    assert any(p['pair'] and p['sk_units'] for c, p in plans if c['stats'])


@pytest.mark.parametrize("c", STAT_CASES, ids=[c['name'].replace(" ", "_") for c in STAT_CASES])
def test_conv_fwd_batch_statistics_bit_exact(c):
    """d_stat_sum / d_stat_sumsq equal the float64 sums of the stored bf16 outputs, and the outputs equal the reference.
    (Every partial sum is an integer below 2^24, so the order of the kernel's adds and atomics does not matter.)"""
    bufs, yb, p = _run(c)
    y = yb.double()
    s, q = y.sum(dim=(0, 2, 3)), (y * y).sum(dim=(0, 2, 3))
    assert float(y.abs().sum(dim=(0, 2, 3)).max()) < BOUND and float(q.max()) < BOUND
    N = c['N']
    _assert_bits(bufs['ssum'][:N], s.float(), "sum [%s]" % _show(p))
    _assert_bits(bufs['ssq'][:N], q.float(), "sum of squares [%s]" % _show(p))
    assert bool(bufs['ssum'][N:].isnan().all() and bufs['ssq'][N:].isnan().all()), "statistics written past N"


# ------------------------------------------------------------------------------------------------ data gradient
DARKNET = [("conv2", 32, 64, 208, 3), ("conv3", 64, 128, 104, 3), ("conv4", 128, 64, 104, 1), ("conv5", 64, 128, 104, 3),
           ("conv6", 128, 256, 52, 3), ("conv7", 256, 128, 52, 1), ("conv8", 128, 256, 52, 3),
           ("conv9/13", 256, 512, 26, 3), ("conv10", 512, 256, 26, 1), ("conv14", 512, 1024, 13, 3),
           ("conv15", 1024, 512, 13, 1), ("conv18", 1024, 1024, 13, 3), ("conv21", 512, 64, 26, 1),
           ("conv22", 1280, 1024, 13, 3), ("head", 1024, 125, 13, 1)]
DGRAD_CASES = [(n, 16, C_, O, H, k, 0) for n, C_, O, H, k in DARKNET]
DGRAD_CASES += [("conv14 batch 64", 64, 512, 1024, 13, 3, 0), ("conv21 into a concat slice", 16, 512, 64, 26, 1, 256)]


@pytest.mark.parametrize("name,B,C_,O,H,k,ch_off", DGRAD_CASES, ids=[c[0].replace(" ", "_").replace("/", "_")
                                                                     for c in DGRAD_CASES])
def test_dgrad_bit_exact(name, B, C_, O, H, k, ch_off):
    """da = conv2d_input(dz, W * mask): mc_pack_conv_weights_dgrad + mc_conv_fwd as the retrain backward runs them (k-block
    32 for <= 32 gradient channels) equal the float64 reference rounded to bf16, written at ch_off into a canaried
    buffer."""
    lib = _lib.load()
    g = _gen(B * 1000 + C_ + O)
    K = O * k * k
    dz = _data((B, O, H, H), 'exact', K, g)
    w = _data((O, C_, k, k), 'exact', K, g)
    mask = (torch.rand(O, C_, k, k, device=DEV, generator=g) > 0.3).float()
    _assert_exact_sum(K, dz, w)
    ref = torch.nn.grad.conv2d_input((B, C_, H, H), (w * mask).double(), dz.double(), padding=k // 2)
    yb = ref.float().bfloat16()
    assert torch.equal(yb.double(), ref)
    kb = 32 if O <= 32 else 64
    Cpad, Ko = _r(C_, 16), _r(O, kb)
    s = _lib.stream_ptr()
    wpack = torch.empty(Cpad, k * k * Ko, dtype=torch.bfloat16, device=DEV)
    _lib.check(lib.mc_pack_conv_weights_dgrad(w.data_ptr(), mask.data_ptr(), O, C_, k, wpack.data_ptr(), Cpad, Ko, s),
               "mc_pack_conv_weights_dgrad")
    rows = B * (H + 1) * (H + 1)
    dzp, ldz = _pack(dz)
    ldc = ch_off + _r(C_, 8) + (64 if ch_off else 0)
    out = _canary((rows + EXTRA_ROWS, ldc))
    ones, zeros = torch.ones(Cpad, device=DEV), torch.zeros(Cpad, device=DEV)
    d = _lib.mc_conv_desc()
    d.d_in, d.d_wpack, d.d_scale, d.d_shift, d.d_out = dzp.data_ptr(), wpack.data_ptr(), ones.data_ptr(), zeros.data_ptr(), out.data_ptr()
    d.B, d.H, d.W, d.Cin, d.Cin_ld, d.N, d.Npad = B, H, H, O, ldz, C_, Cpad
    d.ksize, d.leaky, d.epi_mode, d.ldc, d.ch_off, d.block_k = k, 0, PNHWC, ldc, ch_off, kb
    p = _plan(d)
    print(name, _show(p))
    with torch.cuda.device(0):
        _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "mc_conv_fwd (dgrad)")
    torch.cuda.synchronize()
    c = dict(B=B, H=H, W=H, N=C_, ch_off=ch_off, mode=PNHWC)
    _assert_bits(out, _expected(c, dict(out=_canary((rows + EXTRA_ROWS, ldc)), ldc=ldc), p, yb), "%s [%s]" % (name, _show(p)))


# ------------------------------------------------------------------------------------------------ thin-layer kernels
# fp32(u / 255) as IEEE division (torch's CUDA division by a scalar multiplies by the rounded reciprocal instead)
_U8_DIV_255 = torch.from_numpy(np.arange(256, dtype=np.float32) / np.float32(255))


def _image(B, C_, H, W, kind, g):
    """kind 0: integer activations; 1: fp32 image u/255; 2: uint8 image u.  Returns (kernel input, exact operand as the
    kernel sees it in fp32, quantum of its values)."""
    if kind == 0:
        x = _ints((B, C_, H, W), 0.7, g)
        return x, x, 1.0
    u = torch.randint(0, 256, (B, C_, H, W), device=DEV, generator=g, dtype=torch.uint8)
    xf = _U8_DIV_255.to(DEV)[u.long()]
    return (xf if kind == 1 else u), xf.bfloat16().float(), 2.0 ** -15


def _thin_expected(y, B, Ho, Wo, N, ld, out, zero_to):
    exp = out.clone()
    v = exp[:B * (Ho + 1) * (Wo + 1)].view(B, Ho + 1, Wo + 1, ld)
    v[:, :Ho, :Wo, :zero_to] = 0
    v[:, :Ho, :Wo, :N] = y.permute(0, 2, 3, 1)
    return exp


def _thin_ref(xe, w, sc, sh, leaky, pool, q):
    K = w.shape[1] * w.shape[2] * w.shape[3]
    _assert_exact_sum(K, xe, w, q)
    v = _epilogue(F.conv2d(xe.double(), w.double(), None, 1, w.shape[2] // 2), sc, sh, leaky)
    return F.max_pool2d(v, 2, 2) if pool else v


IM2COL_CASES = [  # (B, Cin, H, W, N, kind, pool, leaky)
    (2, 5, 24, 40, 24, 0, 0, 1),      # PNHWC, CL 8
    (2, 12, 32, 16, 40, 0, 0, 1),     # PNHWC, CL 16
    (2, 8, 18, 22, 8, 0, 1, 0),       # npos 8, ragged tiles
    (1, 3, 416, 416, 32, 1, 0, 0),    # the retrain's first layer (fp32 image, linear, scale 1, shift 0)
    (2, 3, 64, 48, 16, 1, 1, 1),      # fp32 image, pooled
    (2, 3, 64, 48, 16, 2, 1, 1),      # uint8 RGB pooled: the inline x/255 of the fast path
    (2, 3, 32, 48, 32, 2, 0, 1),      # uint8, pool 0: the shared-memory x/255 table
    (2, 1, 32, 32, 4, 2, 1, 1),       # uint8, 1 channel: the table
    (2, 4, 32, 32, 12, 2, 1, 0),      # uint8, 4 channels: the table
]


@pytest.mark.parametrize("B,Cin,H,W,N,kind,pool,leaky", IM2COL_CASES)
def test_im2col_bit_exact(B, Cin, H, W, N, kind, pool, leaky):
    lib = _lib.load()
    g = _gen(B * 7 + Cin * 31 + N + 100 * kind + pool)
    x, xe, q = _image(B, Cin, H, W, kind, g)
    w = _ints((N, Cin, 3, 3), 0.8, g)
    first = (kind, Cin, N, pool) == (1, 3, 32, 0)
    sc = torch.ones(N, device=DEV) if first else torch.tensor([0.75, -1.25, 2.0, 0.5], device=DEV).repeat(N)[:N]
    sh = torch.zeros(N, device=DEV) if first else torch.randint(-3, 4, (N,), device=DEV, generator=g).float() / 4
    cl, npos, nb, kpad = (ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int())
    _lib.check(lib.mc_conv_im2col_geometry(Cin, kind, N, pool, ctypes.byref(cl), ctypes.byref(npos), ctypes.byref(nb),
                                           ctypes.byref(kpad)), "mc_conv_im2col_geometry")
    cl, npos, nb, kpad = cl.value, npos.value, nb.value, kpad.value
    wd = w.permute(0, 2, 3, 1)
    nb_pad = _r(nb, 16)
    wfull = torch.zeros(nb_pad, kpad, device=DEV)
    if pool:
        wfull[:, :16 * cl] = _pool_window_weights(wd, nb_pad, npos, cl)
    else:
        wfull[:N, :9 * cl] = torch.nn.functional.pad(wd, (0, cl - Cin)).reshape(N, 9 * cl)
    wfull = wfull.bfloat16().contiguous()
    nsc = max(_r(npos, 16), 16)
    scp, shp = torch.zeros(nsc, device=DEV), torch.zeros(nsc, device=DEV)
    scp[:N], shp[:N] = sc, sh
    s = _lib.stream_ptr()
    if kind == 0:
        xin = torch.zeros(B * (H + 1) * (W + 1) + EXTRA_ROWS, cl, dtype=torch.bfloat16, device=DEV)
        xin[B * (H + 1) * (W + 1):] = float('nan')
        xin[:B * (H + 1) * (W + 1)] = _pack(x, cl)[0]
    else:
        xin = x.contiguous()
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    ld = _r(N, 8) + 8
    out = _canary((B * (Ho + 1) * (Wo + 1) + EXTRA_ROWS, ld))
    _lib.check(lib.mc_conv_im2col_fwd(xin.data_ptr(), kind, wfull.data_ptr(), scp.data_ptr(), shp.data_ptr(),
                                      out.data_ptr(), B, H, W, Cin, cl if kind == 0 else Cin, N, ld, leaky, pool, s),
               "mc_conv_im2col_fwd")
    torch.cuda.synchronize()
    y = _thin_ref(xe, w, sc, sh, leaky, pool, q).bfloat16()
    _assert_bits(out, _thin_expected(y, B, Ho, Wo, N, ld, out, _r(N, 8)), "im2col")


WINDOW_CASES = [  # (B, Cin, H, W, N, kind, pool)
    (2, 4, 32, 32, 1, 0, 1), (3, 1, 24, 40, 17, 0, 0), (1, 8, 16, 8, 16, 0, 0), (2, 7, 52, 52, 80, 0, 0),
    (5, 3, 18, 22, 5, 0, 1),
    (2, 3, 64, 64, 4, 1, 1), (3, 3, 36, 48, 13, 1, 1), (2, 3, 96, 160, 32, 1, 1),
    (2, 3, 64, 64, 4, 2, 1), (1, 3, 32, 16, 8, 2, 1), (3, 3, 36, 48, 13, 2, 1), (2, 3, 96, 160, 32, 2, 1),
]


def _uint8_scales(n):
    """fp32 scales s for which fp32(s / 255) (the window kernel's folded scale) differs from fp32(s * fp32(1/255))"""
    cand = (np.arange(1, 4000, dtype=np.float32) / np.float32(997)) + np.float32(0.25)
    diff = cand[(cand / np.float32(255)) != cand * (np.float32(1) / np.float32(255))]
    assert diff.size >= n, "no scales where s/255 and s*(1/255) differ"
    return torch.from_numpy(diff[:n].copy()).to(DEV)


@pytest.mark.parametrize("B,Cin,H,W,N,kind,pool", WINDOW_CASES)
def test_window_bit_exact(B, Cin, H, W, N, kind, pool):
    """mc_conv_window_fwd.  uint8 images: the integers 0..255 enter the GEMM and the epilogue scale is fp32(s/255); the
    data puts most accumulators near -shift/scale, where the cancellation exposes a one-ulp change of that scale."""
    lib = _lib.load()
    g = _gen(B * 11 + Cin * 13 + N + 1000 * kind)
    if kind == 2:
        u = torch.randint(248, 256, (B, Cin, H, W), device=DEV, generator=g, dtype=torch.uint8)
        x, xe, q = u, u.float(), 1.0
        w = torch.ones(N, Cin, 3, 3, device=DEV)
        w[:, :, 1, 1] = 2.0
        sc = _uint8_scales(N)
        sc_eff = torch.from_numpy(sc.cpu().numpy() / np.float32(255)).to(DEV)  # IEEE division, as __fdiv_rn
        sh = -(float(252 * 30) * sc_eff).float()   # y ~ (acc - 7560) * s/255: small, next to the interior's acc
    else:
        x, xe, q = _image(B, Cin, H, W, kind, g)
        w = _ints((N, Cin, 3, 3), 0.8, g)
        sc = torch.tensor([0.75, -1.25, 2.0, 0.5], device=DEV).repeat(N)[:N]
        sh = torch.randint(-3, 4, (N,), device=DEV, generator=g).float() / 4
        sc_eff = sc
    npos, nb, kcols = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    assert lib.mc_conv_window_supported(Cin, kind, N, pool) == 1
    _lib.check(lib.mc_conv_window_geometry(Cin, kind, N, pool, ctypes.byref(npos), ctypes.byref(nb), ctypes.byref(kcols)),
               "mc_conv_window_geometry")
    npos, nb, kcols = npos.value, nb.value, kcols.value
    wd = w.permute(0, 2, 3, 1)
    if kind == 0:
        wk = torch.zeros(nb, 10, 8, device=DEV)
        wk[:N, :9, :Cin] = wd.reshape(N, 9, Cin)
    else:
        wk = _pool_window_weights(wd, nb, npos, 4)
    wk = wk.reshape(nb, kcols).bfloat16().contiguous()
    nsc = max(_r(npos, 16), 16)
    scp, shp = torch.zeros(nsc, device=DEV), torch.zeros(nsc, device=DEV)
    scp[:N], shp[:N] = sc, sh
    s = _lib.stream_ptr()
    if kind == 0:
        rows = B * (H + 1) * (W + 1)
        xin = torch.full((rows + EXTRA_ROWS, 8), float('nan'), dtype=torch.bfloat16, device=DEV)
        xin[:rows] = _pack(x, 8)[0]
    else:
        xin = x.contiguous()
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    ld = _r(N, 8) + 8
    out = _canary((B * (Ho + 1) * (Wo + 1) + EXTRA_ROWS, ld))
    _lib.check(lib.mc_conv_window_fwd(xin.data_ptr(), kind, wk.data_ptr(), scp.data_ptr(), shp.data_ptr(), out.data_ptr(),
                                      B, H, W, Cin, N, ld, 1, pool, s), "mc_conv_window_fwd")
    torch.cuda.synchronize()
    y = _thin_ref(xe, w, sc_eff, sh, 1, pool, q).bfloat16()
    _assert_bits(out, _thin_expected(y, B, Ho, Wo, N, ld, out, _r(N, 8)), "window")


THIN_CASES = [  # test_thin_conv_kernel's shapes; fused pairs with leaky and leaky2 set independently
    (3, 4, 1, 1, 0, 20, 24, 1, 1), (3, 1, 17, 0, 0, 12, 20, 1, 1), (1, 17, 4, 0, 0, 12, 20, 0, 1),
    (3, 4, 11, 1, 0, 16, 16, 1, 1), (3, 1, 17, 0, 4, 12, 20, 1, 0), (3, 8, 8, 0, 8, 10, 14, 0, 1),
    (3, 2, 3, 0, 0, 9, 7, 1, 1), (1, 32, 8, 0, 0, 6, 10, 1, 1), (3, 5, 4, 1, 0, 8, 12, 1, 1), (3, 2, 24, 0, 0, 8, 8, 1, 1),
    (3, 1, 17, 0, 4, 12, 20, 0, 0), (3, 8, 8, 0, 8, 10, 14, 1, 1),
]


@pytest.mark.parametrize("k,Cin,N,pool,N2,H,W,leaky,leaky2", THIN_CASES)
def test_thin_bit_exact(k, Cin, N, pool, N2, H, W, leaky, leaky2):
    """mc_conv_thin_fwd; the fused pair rounds its first stage to bf16 before the 1x1, and so does the reference."""
    lib = _lib.load()
    g = _gen(100 * Cin + N + 7 * N2)
    B = 3
    ct, nt, n2t = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    assert lib.mc_conv_thin_geometry(k, Cin, N, pool, N2, ctypes.byref(ct), ctypes.byref(nt), ctypes.byref(n2t)) == 1
    ct, nt, n2t = ct.value, nt.value, n2t.value
    x = _ints((B, Cin, H, W), 0.8, g)
    w = _ints((N, Cin, k, k), 0.8, g)
    sc = torch.tensor([0.75, -1.25, 2.0, 0.5], device=DEV).repeat(N)[:N]
    sh = torch.randint(-3, 4, (N,), device=DEV, generator=g).float() / 4
    ld_in = max(_r(Cin, 8), ct)
    rows = B * (H + 1) * (W + 1)
    xin = torch.full((rows + EXTRA_ROWS, ld_in), float('nan'), dtype=torch.bfloat16, device=DEV)
    xin[:rows] = _pack(x, ld_in)[0]
    hw, hsc, hsh = _thin_host_weights(w, sc, sh, ct, nt)
    y = _thin_ref(x, w, sc, sh, leaky, pool, 1.0)
    Ho, Wo = y.shape[2:]
    hw2 = hsc2 = hsh2 = None
    n_out = N
    if N2:
        w2 = _ints((N2, N), 0.8, g)
        sc2 = torch.tensor([0.5, -1.0, 1.5], device=DEV).repeat(N2)[:N2]
        sh2 = torch.randint(-3, 4, (N2,), device=DEV, generator=g).float() / 2
        w2p = torch.zeros(nt, n2t)
        w2p[:N, :N2] = w2.t().cpu()
        s2p, h2p = torch.zeros(n2t), torch.zeros(n2t)
        s2p[:N2], h2p[:N2] = sc2.cpu(), sh2.cpu()
        hw2, hsc2, hsh2 = _c_floats(w2p), _c_floats(s2p), _c_floats(h2p)
        y1 = y.bfloat16().float()
        nz = y1[y1 != 0].abs()
        q2 = 2.0 ** (math.floor(math.log2(float(nz.min()))) - 7) if nz.numel() else 1.0  # smallest bf16 quantum in y1
        y = _thin_ref(y1, w2.view(N2, N, 1, 1), sc2, sh2, leaky2, 0, q2)
        n_out = N2
    ld_out = _r(n_out, 8) + 8
    out = _canary((B * (Ho + 1) * (Wo + 1) + EXTRA_ROWS, ld_out))
    _lib.check(lib.mc_conv_thin_fwd(xin.data_ptr(), hw, hsc, hsh, hw2, hsc2, hsh2, out.data_ptr(), B, H, W, Cin, ld_in, N,
                                    ld_out, k, leaky, pool, N2, leaky2, _lib.stream_ptr()), "mc_conv_thin_fwd")
    torch.cuda.synchronize()
    _assert_bits(out, _thin_expected(y.bfloat16(), B, Ho, Wo, n_out, ld_out, out, _r(n_out, 8)), "thin")


DIRECT_CASES = [  # (B, Cin, H, W, N, k, nchw, pool)
    (2, 3, 32, 48, 32, 3, 1, 1), (2, 3, 30, 22, 16, 3, 1, 0), (2, 4, 16, 16, 5, 1, 1, 0),
    (2, 20, 24, 20, 12, 3, 0, 1), (2, 32, 14, 18, 8, 3, 0, 0), (3, 7, 17, 13, 32, 1, 0, 0), (2, 16, 20, 20, 3, 1, 0, 1),
]


@pytest.mark.parametrize("B,Cin,H,W,N,k,nchw,pool", DIRECT_CASES)
def test_direct_bit_exact(B, Cin, H, W, N, k, nchw, pool):
    """mc_conv_direct_fwd (CUDA cores) at the limits mc_conv_direct_supported accepts.  Dyadic scales keep acc * scale
    exact in fp32, so a contracted or separate multiply-add give the same result."""
    lib = _lib.load()
    assert lib.mc_conv_direct_supported(Cin, N, k) == 1
    g = _gen(B + Cin * 3 + N * 5 + k)
    x = _ints((B, Cin, H, W), 0.8, g)
    w = _ints((N, Cin, k, k), 0.8, g)
    sc = torch.tensor([0.5, -2.0, 1.0, 0.25], device=DEV).repeat(N)[:N]
    sh = torch.randint(-3, 4, (N,), device=DEV, generator=g).float() / 4
    s = _lib.stream_ptr()
    if nchw:
        xin, ld_in = x.contiguous(), Cin
    else:
        ld_in = _r(Cin, 8) + 8
        rows = B * (H + 1) * (W + 1)
        xin = torch.full((rows + EXTRA_ROWS, ld_in), float('nan'), dtype=torch.bfloat16, device=DEV)
        xin[:rows] = _pack(x, ld_in)[0]
    Ho, Wo = (H // 2, W // 2) if pool else (H, W)
    ld = _r(N, 8) + 8
    out = _canary((B * (Ho + 1) * (Wo + 1) + EXTRA_ROWS, ld))
    _lib.check(lib.mc_conv_direct_fwd(xin.data_ptr(), nchw, w.contiguous().data_ptr(), sc.data_ptr(), sh.data_ptr(),
                                      out.data_ptr(), B, H, W, Cin, ld_in, N, ld, k, 1, pool, s), "mc_conv_direct_fwd")
    torch.cuda.synchronize()
    y = _thin_ref(x, w, sc, sh, 1, pool, 1.0).bfloat16()
    _assert_bits(out, _thin_expected(y, B, Ho, Wo, N, ld, out, N), "direct")

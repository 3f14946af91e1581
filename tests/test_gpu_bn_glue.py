"""Bit-exact tests of the retrain step's BatchNorm / leaky / max-pool passes (train_ops.cu) at every channel count the
entry points take, through mc_col_stats, mc_bn_apply, mc_bn_backward, mc_maxpool2x2_backward, mc_bn_apply_pool and
mc_bn_pool_backward.

Method (that of test_gpu_split_exact.py).  Activations and gradients are small integers, means are integers, invstd,
gamma and the affine scale are small dyadic numbers and B*H*W is a power of two.  Then every product and every fp32
partial sum is exact whatever the order or the block a term lands in, so the outputs must EQUAL a float64 reference
(rounded to bf16 where the kernel stores bf16): a dropped, doubled or misplaced row, channel or octet is a hard failure.
Where leaky's 0.1f makes the sums inexact the reductions get a tolerance.

Layouts.  Every buffer has columns outside the channels a call owns (a concat slice at ch_off > 0, the pitch past C,
the rest of a ragged last octet) filled with a canary value: reads of them would show in the sums, writes to them are
checked.  Reorg addressing is tested with C % 8 == 0 and C % 8 != 0.
"""
import ctypes

import pytest
import torch

from modelcompression_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
CHANNELS = [1, 3, 8, 12, 24, 40, 64, 125, 256, 1024, 1280, 2048]
B, H, W = 4, 16, 16       # B*H*W = 1024 pixels; 1,156 PNHWC rows: several blocks for every channel count
CANARY = -77.0            # exact in bf16; a read of it shows in the sums
SLOPE = torch.tensor(0.1, dtype=torch.float32)
SUM_RTOL = 400 * 2.0 ** -24
# (ch_off, reorg, extra pitch columns) of the activation / gradient buffer that mc_bn_apply writes and mc_bn_backward reads
LAYOUTS = {'plain': (0, 0, 0), 'slice': (16, 0, 5), 'reorg': (0, 1, 0), 'reorg_slice': (8, 1, 3)}


def _r8(n):
    return (n + 7) // 8 * 8


def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


def _ints(shape, lo, hi, g):
    return torch.randint(lo, hi + 1, shape, device=DEV, generator=g).double()


def _pick(values, n, g):
    v = torch.tensor(values, dtype=torch.float64, device=DEV)
    return v[torch.randint(0, len(values), (n,), device=DEV, generator=g)]


def _pnhwc(data, ld, ch_off=0, h=H, w=W):
    """bf16 [B*(h+1)*(w+1), ld] holding data [B, h, w, C] at columns [ch_off, ch_off+C) of the interior pixels, zero at
    the pad rows of those columns, CANARY everywhere else."""
    C = data.shape[-1]
    t = torch.full((B, h + 1, w + 1, ld), CANARY, dtype=torch.bfloat16, device=DEV)
    t[..., ch_off:ch_off + C] = 0
    t[:, :h, :w, ch_off:ch_off + C] = data.to(torch.bfloat16)
    return t.view(-1, ld)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _vec(v, extra=8):
    """fp32 per-channel vector with `extra` CANARY elements behind it (a store past C shows)."""
    return torch.cat([v.float(), torch.full((extra,), CANARY, device=DEV)])


def _act(v):
    """bf16(leaky(v)) with the kernels' fp32 arithmetic (v exact in fp32)."""
    v = v.float()
    return torch.maximum(v, v * SLOPE)


def _assert_equal(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not torch.equal(got, want):
        bad = (got != want).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError("%s: %d of %d entries differ; first at %s: got %r, want %r" % (
            what, bad.shape[0], got.numel(), i, got[i].item(), want[i].item()))


def _assert_close(got, want, rtol, what):
    err = (got.double() - want.double()).abs()
    lim = rtol * want.double().abs() + rtol * want.double().abs().max() * 1e-3
    assert bool((err <= lim).all()), "%s: max err %.3g" % (what, (err - lim).max().item())


def _bn_data(C, seed):
    """z [B,H,W,C] integers, per-channel mean (integer), invstd / gamma (dyadic), beta, and the affine scale / shift."""
    g = _gen(seed)
    z = _ints((B, H, W, C), -3, 3, g)
    mean = _ints((C,), -1, 1, g)
    invstd = _pick([0.5, 1.0, 2.0], C, g)
    gamma = _pick([0.5, 1.0, 1.5, 2.0], C, g)
    beta = _pick([-1.0, -0.5, 0.0, 0.25, 1.0], C, g)
    scale = gamma * invstd
    shift = beta - mean * scale
    return g, z, mean, invstd, gamma, beta, scale, shift


def _windows(t):
    """[B, H, W, C] -> [B, H/2, W/2, 4, C], window positions in PyTorch scan order (0,0), (0,1), (1,0), (1,1)."""
    Bq, Hq, Wq, C = t.shape
    return t.view(Bq, Hq // 2, 2, Wq // 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(Bq, Hq // 2, Wq // 2, 4, C)


def _unwindows(t):
    Bq, Ho, Wo, _, C = t.shape
    return t.view(Bq, Ho, Wo, 2, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(Bq, 2 * Ho, 2 * Wo, C)


def _first_max(v):
    """one-hot [.., 4, C] of the first maximum of each window (nn.MaxPool2d's rule)."""
    best = v.max(dim=-2, keepdim=True).values
    hit = (v == best).int()
    first = (hit.cumsum(dim=-2) == 1) & (hit == 1)
    return first


# --------------------------------------------------------------------------------------------------- mc_col_stats
@pytest.mark.parametrize("C", CHANNELS)
def test_col_stats_exact(C):
    g = _gen(C)
    z = _ints((B, H, W, C), -4, 4, g)
    ch_off = 8
    ld = _r8(ch_off + C) + 8
    zp = _pnhwc(z, ld, ch_off)
    s, sq = _vec(torch.zeros(C, device=DEV)), _vec(torch.zeros(C, device=DEV))
    lib = _lib.load()
    with torch.cuda.device(0):
        _lib.check(lib.mc_col_stats(zp.data_ptr(), zp.shape[0], C, ld, ch_off, s.data_ptr(), sq.data_ptr(),
                                    _lib.stream_ptr()), "mc_col_stats")
    torch.cuda.synchronize()
    want = torch.cat([z.sum(dim=(0, 1, 2)), torch.full((8,), CANARY, dtype=torch.float64, device=DEV)])
    _assert_equal(s.double(), want, "sum")
    want[:C] = (z * z).sum(dim=(0, 1, 2))
    _assert_equal(sq.double(), want, "sumsq")


# ---------------------------------------------------------------------------------------------------- mc_bn_apply
def _out_buffer(C, layout):
    """The buffer mc_bn_apply writes / mc_bn_backward reads: (ld, ch_off, reorg, its pixel grid h, w)."""
    ch_off, reorg, extra = LAYOUTS[layout]
    h, w = (H // 2, W // 2) if reorg else (H, W)
    ld = _r8(ch_off + (4 if reorg else 1) * C + extra)
    return ld, ch_off, reorg, h, w


def _to_layout(a, reorg):
    """[B, H, W, C] -> what the buffer holds: itself, or the Reorg(2) shuffle [B, H/2, W/2, 4C] (channel q*C + c)."""
    if not reorg:
        return a
    return _windows(a).reshape(B, H // 2, W // 2, 4 * a.shape[-1])


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("leaky", [0, 1])
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_apply_exact(C, leaky, layout):
    _, z, _, _, _, _, scale, shift = _bn_data(C, 100 + C)
    ldz = _r8(C) + 8
    zp = _pnhwc(z, ldz)
    ld, ch_off, reorg, h, w = _out_buffer(C, layout)
    out = torch.full((B * (h + 1) * (w + 1), ld), CANARY, dtype=torch.bfloat16, device=DEV)
    sc, sh = _vec(scale), _vec(shift)
    lib = _lib.load()
    with torch.cuda.device(0):
        _lib.check(lib.mc_bn_apply(zp.data_ptr(), ldz, B, H, W, C, _ptr(sc), _ptr(sh), leaky,
                                   out.data_ptr(), ld, ch_off, reorg, _lib.stream_ptr()), "mc_bn_apply")
    torch.cuda.synchronize()
    v = z * scale + shift                      # exact in fp32
    a = (_act(v) if leaky else v.float()).to(torch.bfloat16)
    want = torch.full((B, h + 1, w + 1, ld), CANARY, dtype=torch.bfloat16, device=DEV)
    n = (4 if reorg else 1) * C
    if not reorg:
        want[..., ch_off:ch_off + n] = 0       # pad rows of the slice are written as zeros
    want[:, :h, :w, ch_off:ch_off + n] = _to_layout(a, reorg)
    _assert_equal(out.view(B, h + 1, w + 1, ld), want, "out")


# ------------------------------------------------------------------------------------------------- mc_bn_backward
def _bn_backward_ref(z, g, mean, invstd, gamma, beta, leaky):
    """float64 dbeta, dgamma, dz of BatchNorm (training) + leaky with g = da before the leaky slope, fp32 slope; and
    the per-channel sums of |terms| of dbeta and dgamma (what bounds the fp32 rounding error of the reductions)."""
    xh = (z - mean) * invstd
    if leaky:
        g = torch.where(gamma * xh + beta <= 0, (g.float() * SLOPE).double(), g)
    dbeta, dgamma = g.sum(dim=(0, 1, 2)), (g * xh).sum(dim=(0, 1, 2))
    n = z.shape[0] * z.shape[1] * z.shape[2]
    dz = gamma * invstd * (g - dbeta / n - xh * (dgamma / n))
    return dbeta, dgamma, dz, (g.abs().sum(dim=(0, 1, 2)), (g * xh).abs().sum(dim=(0, 1, 2)))


def _assert_sum_close(got, want, abs_sum, what):
    """An fp32 sum whose terms are inexact: off by at most SUM_RTOL * sum of |terms| (a chain of ~400 additions per
    channel: per-thread rows, the block's threads, one atomic per block)."""
    err = (got.double() - want).abs()
    assert bool((err <= SUM_RTOL * abs_sum).all()), "%s: max err / sum|terms| %.3g" % (what, (err / abs_sum).max().item())


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("leaky", [0, 1])
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_backward_exact(C, leaky, layout):
    g, z, mean, invstd, gamma, beta, _, _ = _bn_data(C, 200 + C)
    da = _ints((B, H, W, C), -2, 2, g)
    ldz = _r8(C) + 8
    zp = _pnhwc(z, ldz)
    ld, ch_off, reorg, h, w = _out_buffer(C, layout)
    dap = _pnhwc(_to_layout(da, reorg), ld, ch_off, h, w)
    ld_dz = _r8(C) + 8
    dz = torch.full((B * (H + 1) * (W + 1), ld_dz), CANARY, dtype=torch.bfloat16, device=DEV)
    db, dg = _vec(torch.zeros(C, device=DEV)), _vec(torch.zeros(C, device=DEV))
    vecs = [_vec(t) for t in (mean, invstd, gamma, beta)]
    lib = _lib.load()
    with torch.cuda.device(0):
        _lib.check(lib.mc_bn_backward(zp.data_ptr(), ldz, dap.data_ptr(), ld, ch_off, reorg, B, H, W, C,
                                      *[_ptr(t) for t in vecs], leaky,
                                      db.data_ptr(), dg.data_ptr(), dz.data_ptr(), ld_dz, _lib.stream_ptr()),
                   "mc_bn_backward")
    torch.cuda.synchronize()
    dbeta, dgamma, dz_ref, (sb, sg) = _bn_backward_ref(z, da, mean, invstd, gamma, beta, leaky)
    canary8 = torch.full((8,), CANARY, dtype=torch.float64, device=DEV)
    want = torch.full((B, H + 1, W + 1, ld_dz), CANARY, dtype=torch.bfloat16, device=DEV)
    want[..., :C] = 0
    want[:, :H, :W, :C] = dz_ref.float().to(torch.bfloat16)
    got = dz.view(B, H + 1, W + 1, ld_dz)
    _assert_equal(db.double()[C:], canary8, "dbeta past C")
    _assert_equal(dg.double()[C:], canary8, "dgamma past C")
    if not leaky:
        _assert_equal(db.double()[:C], dbeta, "dbeta")
        _assert_equal(dg.double()[:C], dgamma, "dgamma")
        _assert_equal(got, want, "dz")
    else:
        _assert_sum_close(db[:C], dbeta, sb, "dbeta")
        _assert_sum_close(dg[:C], dgamma, sg, "dgamma")
        _assert_equal(got[..., C:], want[..., C:], "dz past C")
        _assert_equal(got[:, H, :, :C], want[:, H, :, :C], "dz pad rows")
        _assert_equal(got[:, :, W, :C], want[:, :, W, :C], "dz pad columns")
        _assert_close(got[:, :H, :W, :C].float(), dz_ref, 2 ** -7, "dz")


# ----------------------------------------------------------------------------------------- mc_maxpool2x2_backward
@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("C", CHANNELS)
def test_maxpool_backward_exact(C, accumulate):
    g = _gen(300 + C)
    a = _ints((B, H, W, C), -2, 2, g)           # few values: many ties inside the windows
    dp = _ints((B, H // 2, W // 2, C), -4, 4, g)
    old = _ints((B, H, W, C), -4, 4, g)
    ld_a, ld_dp, ld_df = _r8(C), _r8(C) + 8, _r8(C) + 16
    ap = _pnhwc(a, ld_a)
    dpp = _pnhwc(dp, ld_dp, 0, H // 2, W // 2)
    df = _pnhwc(old, ld_df)
    lib = _lib.load()
    with torch.cuda.device(0):
        _lib.check(lib.mc_maxpool2x2_backward(ap.data_ptr(), ld_a, dpp.data_ptr(), ld_dp, B, H, W, C, df.data_ptr(),
                                              ld_df, accumulate, _lib.stream_ptr()), "mc_maxpool2x2_backward")
    torch.cuda.synchronize()
    routed = _unwindows(_first_max(_windows(a)) * dp.unsqueeze(3))
    want = _pnhwc(routed + old if accumulate else routed, ld_df).view(B, H + 1, W + 1, ld_df)
    _assert_equal(df.view(B, H + 1, W + 1, ld_df), want, "d_full")


# -------------------------------------------------------------------------- mc_bn_apply_pool / mc_bn_pool_backward
def _pool_supported(C):
    return C % 8 == 0 and (C // 8) & (C // 8 - 1) == 0 and C <= 2048


@pytest.mark.parametrize("leaky", [0, 1])
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_apply_pool_exact(C, leaky):
    lib = _lib.load()
    assert lib.mc_bn_pool_supported(C) == int(_pool_supported(C))
    _, z, _, _, _, _, scale, shift = _bn_data(C, 400 + C)
    ldz, ldp = _r8(C) + 8, _r8(C) + 16
    zp = _pnhwc(z, ldz)
    sc, sh = _vec(scale), _vec(shift)
    out = torch.full((B * (H // 2 + 1) * (W // 2 + 1), ldp), CANARY, dtype=torch.bfloat16, device=DEV)
    with torch.cuda.device(0):
        rc = lib.mc_bn_apply_pool(zp.data_ptr(), ldz, B, H, W, C, _ptr(sc), _ptr(sh), leaky,
                                  out.data_ptr(), ldp, _lib.stream_ptr())
    torch.cuda.synchronize()
    if not _pool_supported(C):
        assert rc != 0
        return
    _lib.check(rc, "mc_bn_apply_pool")
    v = z * scale + shift
    a = (_act(v) if leaky else v.float()).to(torch.bfloat16).float()
    pooled = _windows(a).max(dim=3).values
    want = torch.full((B, H // 2 + 1, W // 2 + 1, ldp), CANARY, dtype=torch.bfloat16, device=DEV)
    want[:, :H // 2, :W // 2, :C] = pooled.to(torch.bfloat16)
    _assert_equal(out.view(B, H // 2 + 1, W // 2 + 1, ldp), want, "pooled")


@pytest.mark.parametrize("leaky", [0, 1])
@pytest.mark.parametrize("C", CHANNELS)
def test_bn_pool_backward_exact(C, leaky):
    lib = _lib.load()
    g, z, mean, invstd, gamma, beta, scale, shift = _bn_data(C, 500 + C)
    dp = _ints((B, H // 2, W // 2, C), -2, 2, g)
    ldz, ldp, ld_dz = _r8(C) + 8, _r8(C) + 16, _r8(C) + 8
    zp = _pnhwc(z, ldz)
    dpp = _pnhwc(dp, ldp, 0, H // 2, W // 2)
    dz = _pnhwc(torch.zeros(B, H, W, C, device=DEV), ld_dz)
    db, dg = _vec(torch.zeros(C, device=DEV)), _vec(torch.zeros(C, device=DEV))
    vecs = [_vec(t) for t in (scale, shift, mean, invstd, gamma, beta)]
    with torch.cuda.device(0):
        rc = lib.mc_bn_pool_backward(zp.data_ptr(), ldz, dpp.data_ptr(), ldp, B, H, W, C, *[_ptr(t) for t in vecs],
                                     leaky, db.data_ptr(), dg.data_ptr(), dz.data_ptr(), ld_dz, _lib.stream_ptr())
    torch.cuda.synchronize()
    if not _pool_supported(C):
        assert rc != 0
        return
    _lib.check(rc, "mc_bn_pool_backward")
    # the forward's window values (fp32 pre-activation, bf16 activation) pick the first maximum; da is d_pooled there
    v = z * scale + shift
    a = (_act(v) if leaky else v.float()).to(torch.bfloat16).float()
    da = _unwindows(_first_max(_windows(a)) * dp.unsqueeze(3))
    dbeta, dgamma, dz_ref, (sb, sg) = _bn_backward_ref(z, da, mean, invstd, gamma, beta, leaky)
    want = _pnhwc(dz_ref.float(), ld_dz).view(B, H + 1, W + 1, ld_dz)
    got = dz.view(B, H + 1, W + 1, ld_dz)
    canary8 = torch.full((8,), CANARY, dtype=torch.float64, device=DEV)
    _assert_equal(db.double()[C:], canary8, "dbeta past C")
    _assert_equal(dg.double()[C:], canary8, "dgamma past C")
    if not leaky:
        _assert_equal(db.double()[:C], dbeta, "dbeta")
        _assert_equal(dg.double()[:C], dgamma, "dgamma")
        _assert_equal(got, want, "dz")
    else:
        _assert_sum_close(db[:C], dbeta, sb, "dbeta")
        _assert_sum_close(dg[:C], dgamma, sg, "dgamma")
        _assert_equal(got[..., C:], want[..., C:], "dz past C")
        _assert_close(got[:, :H, :W, :C].float(), dz_ref, 2 ** -7, "dz")

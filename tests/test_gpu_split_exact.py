"""Bit-exact tests of the split-K reductions: mc_conv_wgrad at training batch sizes (every split-reduction kernel the
planner can pick), mc_conv_wgrad_first at the image layer's training shape, and the stream-K tail of the CTA-pair
forward convolution.

Method.  The operands are small integers (bf16 holds them exactly), so every product and every partial sum is an
integer.  While the sum of |products| of an output stays below BOUND, every fp32 partial sum is exact whatever the
order, the split or the tile a term lands in: the kernel's fp32 dW must then EQUAL the float64 reference, and a bf16
output must equal the float64 reference rounded to bf16.  A dropped, doubled or misplaced row, tap, channel or split is
a hard failure at any size, where a float tolerance would hide it.  Every test checks that bound first (as
S = conv(|a|, |b|) in float64), so data that leaves the exact regime fails as a test bug, not as a kernel bug.  The
references are float64 convolutions on the GPU (an fp32 reference may use TF32, FFT or Winograd, which are not exact).

Premise.  That tcgen05.mma.kind::f16 adds integer-valued bf16 products into its fp32 accumulator without alignment
truncation is measured, not assumed, by test_premise_accumulation_is_exact: an accumulator that starts at 2^L (one
power-of-two product at the first pixel row) takes thousands of small products afterwards, for L = 12, 16, 20 and 23.
Measured on a B200 (1,000 W power limit): exact at every level up to 2^23 (S.max() = 8,389,921), so BOUND = 2^24 (the
fp32 integer range) and the other tests keep S near 2^20.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import modelcompression_b200 as mc
from modelcompression_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
BOUND = 2 ** 24          # sums of |products| below this are exact in fp32 (see the premise test)
TARGET = 2 ** 20         # what the data of the other tests aims S.max() at
REDUCE = {1: 'rows<9>', 2: 'rows<1>', 3: 'small<1>', 4: 'small<4>', 5: 'small<8>'}


# ----------------------------------------------------------------------------------------------------- helpers
def _plan(B, H, W, C, O, k):
    """What mc_conv_wgrad does for this shape (no launch)."""
    info = (ctypes.c_int * 8)()
    _lib.check(_lib.load().mc_conv_wgrad_plan(B, H, W, C, O, k, info), "mc_conv_wgrad_plan")
    p = dict(nsplit=info[0], m_tiles=info[1], n_tiles=info[2], block_n=info[3], share3=info[4], merge3=info[5],
             reduce=info[6], num_kb=info[7])
    p['uneven'] = p['num_kb'] % p['nsplit'] != 0
    return p


def _show(p):
    return "nsplit=%d (%s) m_tiles=%d n_tiles=%d block_n=%d share3=%d merge3=%d num_kb=%d%s" % (
        p['nsplit'], REDUCE[p['reduce']], p['m_tiles'], p['n_tiles'], p['block_n'], p['share3'], p['merge3'],
        p['num_kb'], " uneven" if p['uneven'] else "")


def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


def _ints(shape, density, gen, vmax=2, signed=True):
    """fp32 integers: a fraction `density` of the entries uniform in {1..vmax} (random sign if signed), the rest 0."""
    v = torch.randint(1, vmax + 1, shape, device=DEV, generator=gen)
    if signed:
        v = v * (torch.randint(0, 2, shape, device=DEV, generator=gen) * 2 - 1)
    keep = torch.rand(shape, device=DEV, generator=gen) < density
    return (v * keep).float()


def _density(terms, mean_abs=1.5, target=TARGET):
    """Density of both operands such that terms * (density * mean_abs)^2 ~ target."""
    return min(1.0, (target / terms) ** 0.5 / mean_abs)


def _pack(x, ld=None):
    """fp32 NCHW -> PNHWC bf16 through the library (pad rows and channels >= C zero)."""
    B, C, H, W = x.shape
    ld = ld or (C + 7) // 8 * 8
    out = torch.empty(B * (H + 1) * (W + 1), ld, dtype=torch.bfloat16, device=DEV)
    _lib.check(_lib.load().mc_pack_pnhwc(x.contiguous().data_ptr(), out.data_ptr(), B, H, W, C, ld, _lib.stream_ptr()),
               "mc_pack_pnhwc")
    return out, ld


def _interior_rows(B, H, W):
    r = torch.arange(B * (H + 1) * (W + 1), device=DEV)
    return ((r % (W + 1)) < W) & (((r // (W + 1)) % (H + 1)) < H)


def _wgrad_ref(a, dz, k):
    """float64 dW of F.conv2d(a, w, padding=(k-1)/2), after checking that it is in the exact regime."""
    O, C = dz.shape[1], a.shape[1]
    pad = (k - 1) // 2
    S = torch.nn.grad.conv2d_weight(a.double().abs(), (O, C, k, k), dz.double().abs(), padding=pad)
    smax = S.max().item()
    del S
    assert smax < BOUND, "test data leaves the exact range: S.max() = %d >= %d" % (smax, BOUND)
    return torch.nn.grad.conv2d_weight(a.double(), (O, C, k, k), dz.double(), padding=pad), smax


def _run_wgrad(ap, lda, C, dzp, ldz, O, B, H, W, k, mask, dw=None, accumulate=0):
    """mc_conv_wgrad with a workspace full of NaN bytes (a partial tile the reduction reads but no CTA wrote shows)."""
    lib = _lib.load()
    if dw is None:
        dw = torch.full((O, C, k, k), float('nan'), device=DEV)
    nbytes = lib.mc_workspace_bytes_conv_wgrad(B, H, W, C, O, k)
    assert nbytes > 0
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=DEV)
    with torch.cuda.device(0):
        _lib.check(lib.mc_conv_wgrad(ap.data_ptr(), lda, C, dzp.data_ptr(), ldz, O, B, H, W, k,
                                     None if mask is None else mask.data_ptr(), dw.data_ptr(), accumulate,
                                     ws.data_ptr(), nbytes, _lib.stream_ptr()), "mc_conv_wgrad")
    torch.cuda.synchronize()
    return dw


def _wgrad_data(B, C, O, H, W, k, seed):
    g = _gen(seed)
    d = _density(B * H * W)
    a = _ints((B, C, H, W), d, g)
    dz = _ints((B, O, H, W), d, g)
    mask = (torch.rand(O, C, k, k, device=DEV, generator=g) > 0.3).float()
    return a, dz, mask


def _first_diff(got, want):
    bad = (got != want).nonzero()
    i = tuple(bad[0].tolist())
    return "%d of %d entries differ; first at %s: got %r, want %r" % (
        bad.shape[0], got.numel(), i, got[i].item(), want[i].item())


def _assert_equal(got, want, what):
    assert got.shape == want.shape, (got.shape, want.shape)
    if not torch.equal(got, want):
        raise AssertionError("%s: %s" % (what, _first_diff(got, want)))


# ------------------------------------------------------------------------------------------------ the premise
@pytest.mark.parametrize("level", [12, 16, 20, 23])
def test_premise_accumulation_is_exact(level):
    """One accumulator starts at 2^level and then takes every other product of a long reduction: the wgrad kernel
    without splits (nsplit = 1, 183 k-blocks in one CTA) and the forward conv (K = 9 * 1024, whole tiles)."""
    # ---- wgrad: pixel 0 of image 0 (the first row of the reduction) holds a power of two in every channel of both
    # operands, so the centre tap of every dW entry is 2^level + (small integers added after it)
    B, C, O, H, W, k = 16, 1280, 2048, 26, 26, 3
    plan = _plan(B, H, W, C, O, k)
    print("wgrad", (B, C, O, H, W, k), _show(plan))
    assert plan['nsplit'] == 1
    g = _gen(level)
    d = _density(B * H * W, target=2 ** 10)
    a = _ints((B, C, H, W), d, g)
    dz = _ints((B, O, H, W), d, g)
    pa = level // 2
    a[0, :, 0, 0] = 2.0 ** pa
    dz[0, :, 0, 0] = 2.0 ** (level - pa)
    ref, smax = _wgrad_ref(a, dz, k)
    print("wgrad S.max() = %d (2^%.2f)" % (smax, torch.tensor(float(smax)).log2().item()))
    assert smax >= 2 ** level
    ap, lda = _pack(a)
    dzp, ldz = _pack(dz)
    del a, dz
    dw = _run_wgrad(ap, lda, C, dzp, ldz, O, B, H, W, k, None)
    _assert_equal(dw, ref.float(), "wgrad at 2^%d" % level)
    del ref, dw, ap, dzp

    # ---- forward: input channel 0 is 2^pa everywhere, its centre-tap weight 2^(level - pa), the bias -2^level: the
    # accumulator holds 2^level + r and the epilogue's bias brings it back to the small integer r, exact in bf16
    B, C, O, H, W = 2, 1024, 256, 26, 26
    conv = mc.MaskedConv2d(C, O, 3, 1, 1, bias=True).to(DEV)
    conv.b200_no_workspace = True
    x = _ints((B, C, H, W), 0.1, g)
    w = _ints((O, C, 3, 3), 0.1, g)
    x[:, 0] = 2.0 ** pa
    w[:, 0] = 0.0
    w[:, 0, 1, 1] = 2.0 ** (level - pa)
    conv.weight.data.copy_(w)
    conv.bias.data.fill_(-2.0 ** level)
    smax = F.conv2d(x.double().abs(), w.double().abs(), None, 1, 1).max().item()
    assert 2 ** level <= smax < BOUND, smax
    y = conv(x)
    ref = F.conv2d(x.double(), w.double(), conv.bias.data.double(), 1, 1)
    _assert_equal(y, ref.float().bfloat16().float(), "forward at 2^%d" % level)
    assert float(ref.abs().max()) <= 256  # the outputs are exact in bf16, so any lost unit of the accumulator shows


# ------------------------------------------------------------------------------- mc_conv_wgrad at training shapes
# (name, B, C, O, H, W, k): the Darknet-19 layers at the retrain batch, the ones with the most splits at batch 64 too
DARKNET = [("conv2", 32, 64, 208, 3), ("conv3", 64, 128, 104, 3), ("conv4", 128, 64, 104, 1), ("conv5", 64, 128, 104, 3),
           ("conv6", 128, 256, 52, 3), ("conv7", 256, 128, 52, 1), ("conv8", 128, 256, 52, 3),
           ("conv9/13", 256, 512, 26, 3), ("conv10", 512, 256, 26, 1), ("conv14", 512, 1024, 13, 3),
           ("conv15", 1024, 512, 13, 1), ("conv18", 1024, 1024, 13, 3), ("conv21", 512, 64, 26, 1),
           ("conv22", 1280, 1024, 13, 3), ("head", 1024, 125, 13, 1)]
WGRAD_CASES = [(n, 16, C, O, H, H, k) for n, C, O, H, k in DARKNET]
WGRAD_CASES += [(n, 64, C, O, H, H, k) for n, C, O, H, k in DARKNET if n in ("conv2", "conv4", "conv10", "head")]
WGRAD_CASES += [
    ("C1 merge3", 4, 1, 16, 224, 224, 3),           # >= 200 k rows, block_n 16, the three dx taps as one MMA
    ("C8 merge3", 4, 8, 32, 224, 224, 3),
    ("ragged C300 O200", 4, 300, 200, 26, 26, 3),  # share3 with 3 N tiles of 112; a partial second M tile
    ("O64 half dZ box", 8, 128, 64, 52, 52, 3),    # <= 64 filters: the second dZ box is not loaded
    ("O65", 8, 128, 65, 52, 52, 3),                # one filter more: it is
    ("ragged 1x1", 3, 72, 200, 37, 29, 1),         # non-square image, ragged C and O, 1x1
    ("C64 small<4>", 3, 64, 64, 37, 37, 3),        # 8 splits (the smallest count of small<4>) over 68 k-blocks
    ("two splits", 2, 8, 16, 30, 22, 3),           # small<1>
    ("conv9 batch 2", 2, 256, 512, 26, 26, 3),     # rows<9> with 2 splits
    ("conv10 batch 2", 2, 512, 256, 26, 26, 1),    # rows<1> with 2 splits
]
_IDS = ["%s-b%d" % (c[0].replace(" ", "_").replace("/", "_"), c[1]) for c in WGRAD_CASES]


@pytest.mark.parametrize("name,B,C,O,H,W,k", WGRAD_CASES, ids=_IDS)
def test_wgrad_bit_exact(name, B, C, O, H, W, k):
    plan = _plan(B, H, W, C, O, k)
    print(name, (B, C, O, H, W, k), _show(plan))
    a, dz, mask = _wgrad_data(B, C, O, H, W, k, seed=B * 7919 + C * 31 + O)
    ref, smax = _wgrad_ref(a, dz, k)
    ap, lda = _pack(a)
    dzp, ldz = _pack(dz)
    del a, dz
    dw = _run_wgrad(ap, lda, C, dzp, ldz, O, B, H, W, k, mask)
    want = (ref * mask).float()
    assert float(want.abs().max()) > 0
    _assert_equal(dw, want, "%s (S.max() = %d)" % (name, smax))


def test_wgrad_plans_reach_every_branch():
    """No launch: the shapes above still reach every split reduction and tile layout (a change of the planner's
    constants or of the SM count that moves a shape off its branch is reported here instead of losing coverage)."""
    plans = [(c, _plan(c[1], c[4], c[5], c[2], c[3], c[6])) for c in WGRAD_CASES]
    for c, p in plans:
        print(c, _show(p))
    assert {p['reduce'] for _, p in plans} == set(REDUCE), "split reductions not reached: %s" % sorted(
        set(REDUCE) - {p['reduce'] for _, p in plans})
    for r in (1, 2):  # the row-wise reductions with more than one split, not only the nsplit = 1 copy
        assert any(p['reduce'] == r and p['nsplit'] > 1 for _, p in plans), REDUCE[r]
    assert any(p['nsplit'] == 1 for _, p in plans)
    assert any(p['nsplit'] >= 100 for _, p in plans)
    assert any(p['merge3'] for _, p in plans)
    assert any(p['share3'] and p['n_tiles'] > 1 for _, p in plans)
    assert any(p['m_tiles'] > 1 and c[3] % 128 != 0 for c, p in plans)
    assert any(p['uneven'] and p['nsplit'] > 1 for _, p in plans)
    assert any(c[3] <= 64 for c, _ in plans) and any(64 < c[3] <= 128 for c, _ in plans)


# one shape per split reduction (batch 2 and smaller: cheap), with the kernel each must reach
REDUCE_CASES = [(5, 2, 128, 64, 104, 104, 1), (4, 2, 128, 256, 52, 52, 3), (3, 2, 8, 16, 30, 22, 3),
                (2, 2, 512, 256, 26, 26, 1), (1, 2, 256, 512, 26, 26, 3)]


@pytest.mark.parametrize("reduce,B,C,O,H,W,k", REDUCE_CASES, ids=[REDUCE[c[0]] for c in REDUCE_CASES])
def test_wgrad_accumulate(reduce, B, C, O, H, W, k):
    """accumulate = 1 adds the masked gradient to dW: dW = dW_old + mask * grad; masked entries keep dW_old."""
    plan = _plan(B, H, W, C, O, k)
    print((B, C, O, H, W, k), _show(plan))
    assert plan['reduce'] == reduce
    a, dz, mask = _wgrad_data(B, C, O, H, W, k, seed=reduce)
    ref, _ = _wgrad_ref(a, dz, k)
    old = torch.randint(-1000, 1001, (O, C, k, k), device=DEV, generator=_gen(99)).float()
    ap, lda = _pack(a)
    dzp, ldz = _pack(dz)
    dw = _run_wgrad(ap, lda, C, dzp, ldz, O, B, H, W, k, mask, dw=old.clone(), accumulate=1)
    _assert_equal(dw, (old.double() + ref * mask).float(), "accumulate")
    assert torch.equal(dw[mask == 0], old[mask == 0])


@pytest.mark.parametrize("B,C,O,H,W,k,lda,ldz", [(2, 128, 64, 104, 104, 1, 136, 72),     # small<8>
                                                 (4, 300, 200, 26, 26, 3, 320, 216),     # share3, 3 N tiles
                                                 (2, 512, 256, 26, 26, 1, 520, 264)])    # rows<1>
def test_wgrad_pitch_columns_are_ignored(B, C, O, H, W, k, lda, ldz):
    """lda > C and ld_dz > O with nonzero values in the columns beyond C and O of the interior rows (the pad rows stay
    zero, as the layout requires): dW is bit-identical to the run on clean, tightly pitched buffers."""
    print((B, C, O, H, W, k), _show(_plan(B, H, W, C, O, k)))
    a, dz, mask = _wgrad_data(B, C, O, H, W, k, seed=lda)
    ref, _ = _wgrad_ref(a, dz, k)
    ap, lda0 = _pack(a)
    dzp, ldz0 = _pack(dz)
    clean = _run_wgrad(ap, lda0, C, dzp, ldz0, O, B, H, W, k, mask)
    _assert_equal(clean, (ref * mask).float(), "clean buffers")
    g = _gen(lda + ldz)
    inner = _interior_rows(B, H, W)
    ap2, _ = _pack(a, lda)
    dzp2, _ = _pack(dz, ldz)
    ap2[inner, C:] = torch.randint(1, 8, (int(inner.sum()), lda - C), device=DEV, generator=g).to(torch.bfloat16)
    dzp2[inner, O:] = torch.randint(1, 8, (int(inner.sum()), ldz - O), device=DEV, generator=g).to(torch.bfloat16)
    dirty = _run_wgrad(ap2, lda, C, dzp2, ldz, O, B, H, W, k, mask)
    _assert_equal(dirty, clean, "pitch columns")


# ------------------------------------------------------------------------------- mc_conv_wgrad_first (image layer)
@pytest.mark.parametrize("B,C,O,H,W", [(16, 3, 32, 416, 416),   # doubled-row view over im2col_first3_kernel rows
                                       (3, 3, 32, 416, 416),    # odd batch: the plain 1x1 wgrad over the rows
                                       (2, 1, 16, 64, 64)])     # C = 1: the generic im2col_first_kernel
@pytest.mark.parametrize("workspace", [True, False], ids=["tensor_core", "cuda_core"])
def test_wgrad_first_bit_exact(B, C, O, H, W, workspace):
    """Integer images 0..3 and integer dZ: the tensor-core path (bf16 im2col rows + tcgen05) and the CUDA-core path
    (fp32 FMA, no workspace) both equal the float64 reference."""
    lib = _lib.load()
    g = _gen(B * 100 + C)
    x = torch.randint(0, 4, (B, C, H, W), device=DEV, generator=g).float()
    dz = _ints((B, O, H, W), min(1.0, TARGET / (B * H * W * 1.5 * 1.5)), g)
    mask = (torch.rand(O, C, 3, 3, device=DEV, generator=g) > 0.3).float()
    ref, smax = _wgrad_ref(x, dz, 3)
    dzp, ldz = _pack(dz)
    nbytes = lib.mc_workspace_bytes_conv_wgrad_first(B, H, W, C, O) if workspace else 0
    assert (nbytes > 0) == workspace
    if workspace:
        rows_ld = 64 if (B % 2 == 0 and O == 32) else C * 9
        print("1x1 wgrad over the im2col rows:", _show(_plan(B // 2 if rows_ld == 64 else B, H, W, rows_ld,
                                                              64 if rows_ld == 64 else O, 1)))
    ws = torch.full((max(nbytes, 256),), 0xFF, dtype=torch.uint8, device=DEV)
    dw = torch.full((O, C, 3, 3), float('nan'), device=DEV)
    with torch.cuda.device(0):
        _lib.check(lib.mc_conv_wgrad_first(x.data_ptr(), dzp.data_ptr(), ldz, B, H, W, C, O, mask.data_ptr(),
                                           dw.data_ptr(), ws.data_ptr() if workspace else None, nbytes,
                                           _lib.stream_ptr()), "mc_conv_wgrad_first")
    torch.cuda.synchronize()
    _assert_equal(dw, (ref * mask).float(), "mc_conv_wgrad_first (S.max() = %d)" % smax)


# ------------------------------------------------------------------------------- stream-K tail of the CTA pair
def _last_plan():
    info = (ctypes.c_int * 8)()
    _lib.check(_lib.load().mc_conv_last_plan(info), "mc_conv_last_plan")
    return dict(pair=info[0], block_n=info[1], sk_units=info[3])


@pytest.mark.parametrize("B,C,H,W,O,sk", [
    (64, 512, 13, 13, 1024, False),   # 196 pair-units over 74 clusters: whole tiles
    (24, 512, 13, 13, 1024, True),    # 2 units in the tail, each cut into 3 spans
    (16, 512, 26, 26, 1024, True),    # 36 units in the tail
    (16, 1006, 26, 26, 1018, True),   # ragged channel-block tail inside the K spans
    (64, 1006, 15, 15, 1018, True),   # the same at batch 64: 64 m-pairs x 4 = 256 units, 34 in the tail
])
def test_conv_stream_k_tail_bit_exact(B, C, H, W, O, sk):
    """Integer x, W and bias: the stream-K launch, the whole-tile launch and the float64 reference rounded to bf16 are
    the same tensor."""
    g = _gen(C + O + B)
    conv = mc.MaskedConv2d(C, O, 3, 1, 1, bias=True).to(DEV)
    d = _density(9 * C, target=2 ** 8)  # outputs mostly within the integers bf16 holds exactly
    x = _ints((B, C, H, W), d, g)
    w = _ints((O, C, 3, 3), d, g)
    conv.weight.data.copy_(w)
    conv.bias.data.copy_(torch.randint(-4, 5, (O,), device=DEV, generator=g).float())
    smax = F.conv2d(x.double().abs(), w.double().abs(), None, 1, 1).max().item()
    assert smax < BOUND
    y_sk = conv(x)
    plan = _last_plan()
    conv.b200_no_workspace = True
    y_dp = conv(x)
    print((B, C, H, W, O), plan, "S.max() = %d" % smax)
    assert plan['pair'] == 1 and (plan['sk_units'] > 0) == sk
    assert _last_plan()['pair'] == 1 and _last_plan()['sk_units'] == 0
    ref = F.conv2d(x.double(), w.double(), conv.bias.data.double(), 1, 1).float().bfloat16().float()
    _assert_equal(y_dp, ref, "whole tiles")
    _assert_equal(y_sk, ref, "stream-K")

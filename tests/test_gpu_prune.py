"""GPU parity: pruning masks, surviving-filter indices and mask bookkeeping — bit-exact vs the oracle and vs the golden
vectors of the reference (tests/golden/, oracle/make_golden.py)."""
import hashlib

import numpy as np
import pytest
import torch

import modelcompression_b200 as mc
from conftest import SmallNet, load_golden, make_darknet
from oracle import prune_oracle

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _bits(m):
    return np.packbits(np.asarray(m).astype(bool).ravel())


@pytest.fixture(scope='module')
def darknet(cfg_path):
    return make_darknet(cfg_path, seed=0, device=DEV)


def test_weight_prune_small_net_interpolated_threshold():
    # n = 1,664 < 2^24: np.percentile interpolates between two order statistics in float32 (gamma != 0)
    g = load_golden('weight_prune_small.npz')
    net = SmallNet.build().to(DEV)
    for i, perc in enumerate(g['percs']):
        masks = mc.weight_prune(net, float(perc))
        assert len(masks) == 4 and all(m.is_cuda and m.dtype == torch.float32 for m in masks)
        got = np.concatenate([_bits(m.cpu().numpy()) for m in masks])
        assert np.array_equal(got, g['bits_%d' % i]), "perc %s" % perc


def test_weight_threshold_values_small_net():
    from modelcompression_b200.pruning.weightPruning.methods import weight_threshold
    g = load_golden('weight_prune_small.npz')
    net = SmallNet.build().to(DEV)
    params = [p.data for p in net.parameters() if p.dim() != 1]
    allw = np.sort(np.concatenate([p.abs().cpu().numpy().ravel() for p in params]))
    for i, perc in enumerate(g['percs']):
        out3 = weight_threshold(params, float(perc)).cpu().numpy()
        assert out3[0] == g['thr_%d' % i], "perc %s" % perc
        assert out3[1] in allw


@pytest.mark.parametrize("idx", [0, 1, 2, 3])
def test_weight_prune_darknet_bit_exact(darknet, idx):
    g = load_golden('weight_prune_darknet.npz')
    perc = float(g['percs'][idx])
    masks = mc.weight_prune(darknet, perc)
    assert len(masks) == 23
    zeros = [int(m.numel() - m.sum().item()) for m in masks]
    assert zeros == g['zeros_%d' % idx].tolist()
    assert [_sha(_bits(m.cpu().numpy())) for m in masks] == g['sha_%d' % idx].tolist()
    for m, p in zip(masks, [p for p in darknet.parameters() if p.dim() != 1]):
        assert m.shape == p.shape and m.device == p.device


def _used_fast():
    """1 when the last weight_prune on cuda:0 took the sample-pivot fast path, 0 when it fell back to the exact radix
    select."""
    from modelcompression_b200 import _lib
    from modelcompression_b200.pruning.weightPruning import methods
    ws = methods._WS[('cuda', 0)]
    with torch.cuda.device(0):
        return _lib.load().mc_debug_select_used_fast(ws.data_ptr(), _lib.stream_ptr())


def test_weight_prune_uses_fast_path(darknet):
    # on the 50.6 M-weight model the sample-pivot bracket holds: one pass over W (the exact path is the fallback)
    mc.weight_prune(darknet, 70.)
    assert _used_fast() == 1


class _ParamBag(torch.nn.Module):
    def __init__(self, tensors):
        super().__init__()
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(t) for t in tensors])


@pytest.mark.parametrize("sizes", [(70001,), (300000, 17, 700003), (1 << 20, 5)])
def test_weight_prune_midsize_interpolated(sizes):
    # n < 2^24 so float32 np.percentile interpolates (gamma != 0) and n >= 8*SAMPLE so the fast path runs: the
    # (k+1)-th order statistic is resolved among the bracketed candidates
    from modelcompression_b200 import _lib
    from modelcompression_b200.pruning.weightPruning import methods
    gen = torch.Generator().manual_seed(5)
    ts = [torch.randn(sz, 3, generator=gen) for sz in sizes]
    bag = _ParamBag(ts).to(DEV)
    ws = [t.numpy() for t in ts]
    for perc in (0.0, 0.01, 12.5, 33.3, 70.0, 99.99, 100.0):
        thr_o, masks_o = prune_oracle.weight_prune_np(ws, perc)
        masks = mc.weight_prune(bag, perc)
        for a, b in zip(masks, masks_o):
            assert np.array_equal(a.cpu().numpy(), b), "perc %s" % perc
        out3 = methods.weight_threshold([p.data for p in bag.parameters()], perc).cpu().numpy()
        assert out3[0] == np.float32(thr_o), "perc %s" % perc
    # heavy ties: quantised weights (the k-th value is shared by thousands of elements)
    tq = [torch.round(t * 4) / 4 for t in ts]
    bagq = _ParamBag(tq).to(DEV)
    for perc in (20.0, 61.7):
        _, masks_o = prune_oracle.weight_prune_np([t.numpy() for t in tq], perc)
        for a, b in zip(mc.weight_prune(bagq, perc), masks_o):
            assert np.array_equal(a.cpu().numpy(), b), "perc %s" % perc


def test_weight_prune_unaligned_and_degenerate_inputs():
    """Ragged edge cases of the one-pass pruner: parameters whose storage is only 4-byte aligned (every chunk takes the
    scalar path), a tensor of all-equal values (every element is a candidate: the candidate slices overflow and the
    exact path takes over), NaN / Inf weights (np.percentile semantics), and 1- and 2-element tensors."""
    gen = torch.Generator().manual_seed(8)
    base = torch.randn(400003, generator=gen)
    views = [base[1:150002].view(-1, 1), base[150003:150004].view(1, 1), base[150005:400003].view(-1, 2)]
    bag = _ParamBag([v.clone() for v in views]).to(DEV)
    # re-point the parameters at 4-byte-aligned views of one device buffer
    dbase = base.to(DEV)
    dviews = [dbase[1:150002].view(-1, 1), dbase[150003:150004].view(1, 1), dbase[150005:400003].view(-1, 2)]
    for p, v in zip(bag.parameters(), dviews):
        p.data = v
        assert p.data_ptr() % 16 != 0 or p.numel() == 1
    ws = [v.numpy() for v in views]
    for perc in (5.0, 50.0, 93.7):
        _, masks_o = prune_oracle.weight_prune_np(ws, perc)
        for a, b in zip(mc.weight_prune(bag, perc), masks_o):
            assert np.array_equal(a.cpu().numpy(), b), "perc %s" % perc
    const = _ParamBag([torch.full((300000, 2), 0.25), torch.full((7, 3), -0.25)]).to(DEV)
    for perc in (10.0, 99.0):
        _, masks_o = prune_oracle.weight_prune_np([p.detach().cpu().numpy() for p in const.parameters()], perc)
        for a, b in zip(mc.weight_prune(const, perc), masks_o):
            assert np.array_equal(a.cpu().numpy(), b)
    bad = torch.randn(200000, 2, generator=gen)
    bad[17, 1] = float('inf')
    bagi = _ParamBag([bad.clone()]).to(DEV)
    _, masks_o = prune_oracle.weight_prune_np([bad.numpy()], 60.0)
    assert np.array_equal(mc.weight_prune(bagi, 60.0)[0].cpu().numpy(), masks_o[0])
    assert _used_fast() == 0  # 400,000 elements would take the fast path; a non-finite value forces the exact one
    bad[5, 0] = float('nan')
    bagn = _ParamBag([bad.clone()]).to(DEV)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, masks_o = prune_oracle.weight_prune_np([bad.numpy()], 60.0)
    assert np.array_equal(mc.weight_prune(bagn, 60.0)[0].cpu().numpy(), masks_o[0])  # threshold NaN: nothing survives
    assert _used_fast() == 0
    tiny = _ParamBag([torch.tensor([[3.0]]), torch.tensor([[1.0, -2.0]])]).to(DEV)
    for perc in (0.0, 50.0, 100.0):
        _, masks_o = prune_oracle.weight_prune_np([p.detach().cpu().numpy() for p in tiny.parameters()], perc)
        for a, b in zip(mc.weight_prune(tiny, perc), masks_o):
            assert np.array_equal(a.cpu().numpy(), b)


def test_weight_prune_vs_oracle_other_percentiles(darknet):
    ws = [p.detach().cpu().numpy() for p in darknet.parameters() if p.dim() != 1]
    for perc in (1.0, 50.0, 99.9):
        masks = mc.weight_prune(darknet, perc)
        _, masks_o = prune_oracle.weight_prune_np(ws, perc)
        for a, b in zip(masks, masks_o):
            assert np.array_equal(a.cpu().numpy(), b)


def test_set_masks_prune_rate_consistency(cfg_path):
    g = load_golden('prune_rate.npz')
    model = make_darknet(cfg_path, seed=0, device=DEV)
    masks = mc.weight_prune(model, 90.)
    before = [p.detach().clone() for p in model.parameters() if p.dim() == 4]
    model.set_masks(masks)
    for w0, p, m in zip(before, [p for p in model.parameters() if p.dim() == 4], masks):
        assert torch.equal(p.data, w0 * m)
    sd = model.state_dict()
    assert sum(1 for k in sd if k.endswith('.mask')) == 23 and 'models.0.conv1.mask' in sd
    assert all(c.mask_flag for c in model.masked_convs())
    rate = mc.prune_rate(model, verbose=False)
    assert rate == float(g['rate90'])  # 89.963056: the denominator includes BN/bias parameters
    assert mc.are_masks_consistent(model, masks) is True
    # break one masked weight -> inconsistent
    w = model.models[0][0].weight.data
    pos = (masks[0] == 0).nonzero()[0]
    w[tuple(pos.tolist())] = 0.5
    assert mc.are_masks_consistent(model, masks) is False
    # pruning an already-pruned model: >= 90 % of |w| are exactly 0 -> threshold 0, the zero bin holds the rank
    masks2 = mc.weight_prune(model, 50.)
    assert _used_fast() == 0  # the zero keys overflow the fast path's candidate slices: the exact radix select runs
    ws = [p.detach().cpu().numpy() for p in model.parameters() if p.dim() != 1]
    _, masks_o = prune_oracle.weight_prune_np(ws, 50.)
    for a, b in zip(masks2, masks_o):
        assert np.array_equal(a.cpu().numpy(), b)


@pytest.mark.parametrize("idx", range(7))
def test_quick_filter_prune_darknet_bit_exact(darknet, idx):
    g = load_golden('filter_prune_darknet.npz')
    perc = float(g['percs'][idx])
    masks, keep = mc.quick_filter_prune(darknet, perc, return_keep=True)
    per_layer = g['filters_per_layer'].tolist()
    want = np.unpackbits(g['keep_%d' % idx])[:sum(per_layer)].astype(bool)
    off = 0
    for m, kp, n, p in zip(masks, keep, per_layer, [p for p in darknet.parameters() if p.dim() == 4]):
        w = want[off:off + n]
        assert kp.cpu().tolist() == np.nonzero(w)[0].tolist()
        assert m.shape == p.shape
        flat = m.reshape(n, -1)
        assert torch.equal(flat.min(dim=1).values, flat.max(dim=1).values)  # whole filters
        assert torch.equal(flat[:, 0].cpu(), torch.from_numpy(w.astype(np.float32)))
        off += n


def test_filter_values_bit_exact(darknet):
    from modelcompression_b200.pruning.weightPruning.methods import filter_values
    g = load_golden('filter_prune_darknet.npz')
    params = [p.data for p in darknet.parameters() if p.dim() == 4]
    v = filter_values(params).cpu().numpy()
    assert np.array_equal(v.astype(np.float64), g['values'])


def test_filter_prune_odd_shapes():
    # pairwise-sum corner cases (C < 8, C % 8 != 0, C > 128 with odd halves), a 5x5 kernel, a 1x1 row wider than the
    # 2,048 channels staged in shared memory, and a layer of 3,000 filters (not 128 * 2^k: an uneven recursion)
    from modelcompression_b200.pruning.weightPruning.methods import filter_values
    torch.manual_seed(3)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.a = torch.nn.Conv2d(5, 7, 1)
            self.b = torch.nn.Conv2d(17, 9, 1)
            self.c = torch.nn.Conv2d(130, 33, 1)
            self.d = torch.nn.Conv2d(1001, 4, 1)
            self.e = torch.nn.Conv2d(6, 10, 5)
            self.f = torch.nn.Conv2d(300, 40, 3)
            self.g = torch.nn.Conv2d(2500, 6, 1)
            self.h = torch.nn.Conv2d(8, 3000, 1)

    net = Net().to(DEV)
    cw = [p.detach().cpu().numpy() for p in net.parameters() if p.dim() == 4]
    v = filter_values([p.data for p in net.parameters() if p.dim() == 4]).cpu().numpy()
    assert np.array_equal(v, np.concatenate([prune_oracle.filter_values_np(w) for w in cw]))
    for perc in (10., 47.3, 90.):
        masks, keep = mc.quick_filter_prune(net, perc, return_keep=True)
        _, _, keep_o, masks_o = prune_oracle.quick_filter_prune_np(cw, perc)
        for a, b in zip(masks, masks_o):
            assert np.array_equal(a.cpu().numpy(), b)
        for a, b in zip(keep, keep_o):
            assert a.cpu().tolist() == np.nonzero(b)[0].tolist()


def test_filter_prune_tiled_and_generic_mix():
    # 3x3 layers with C % 32 == 0 and O % 32 == 0 take the tiled shared-memory path, the others the generic one; an
    # all-zero layer gives 0/0 -> NaN values -> NaN percentile -> nothing is pruned (NumPy semantics)
    torch.manual_seed(9)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.a = torch.nn.Conv2d(32, 32, 3)      # tiled, one chunk
            self.b = torch.nn.Conv2d(96, 160, 3)     # tiled, 3 chunks, 5 groups
            self.c = torch.nn.Conv2d(64, 48, 3)      # generic (O % 32 != 0)
            self.d = torch.nn.Conv2d(40, 64, 3)      # generic (C % 32 != 0)
            self.e = torch.nn.Conv2d(320, 32, 3)     # tiled, 10 chunks
            self.f = torch.nn.Conv2d(64, 37, 1)      # 1x1

    net = Net().to(DEV)
    cw = [p.detach().cpu().numpy() for p in net.parameters() if p.dim() == 4]
    for perc in (0., 25., 61.8, 100.):
        masks, keep = mc.quick_filter_prune(net, perc, return_keep=True)
        _, _, keep_o, masks_o = prune_oracle.quick_filter_prune_np(cw, perc)
        for a, b in zip(masks, masks_o):
            assert np.array_equal(a.cpu().numpy(), b), "perc %s" % perc
        for a, b in zip(keep, keep_o):
            assert a.cpu().tolist() == np.nonzero(b)[0].tolist()
    with torch.no_grad():
        net.c.weight.zero_()
    cw = [p.detach().cpu().numpy() for p in net.parameters() if p.dim() == 4]
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, thr_o, keep_o, _ = prune_oracle.quick_filter_prune_np(cw, 50.)
    assert np.isnan(thr_o)
    _, keep = mc.quick_filter_prune(net, 50., return_keep=True)
    for a, b in zip(keep, keep_o):
        assert a.cpu().tolist() == np.nonzero(b)[0].tolist()


def test_filter_prune_more_filters_than_the_fused_kernel_holds():
    # 27,064 filters > 26,368 (the single cooperative launch's limit): the three-launch path (sums, select, mask fill)
    torch.manual_seed(11)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.a = torch.nn.Conv2d(32, 64, 3)
            self.b = torch.nn.Conv2d(4, 27000, 1)

    net = Net().to(DEV)
    cw = [p.detach().cpu().numpy() for p in net.parameters() if p.dim() == 4]
    for perc in (10., 47.3, 90.):
        masks, keep = mc.quick_filter_prune(net, perc, return_keep=True)
        _, _, keep_o, masks_o = prune_oracle.quick_filter_prune_np(cw, perc)
        for a, b in zip(masks, masks_o):
            assert np.array_equal(a.cpu().numpy(), b), "perc %s" % perc
        for a, b in zip(keep, keep_o):
            assert a.cpu().tolist() == np.nonzero(b)[0].tolist(), "perc %s" % perc


def test_count_zeros_and_unaligned_segments():
    from modelcompression_b200.pruning.weightPruning.utils import count_zeros
    torch.manual_seed(0)
    base = torch.randn(10007, device=DEV)
    base[::3] = 0
    views = [base[1:5000], base[5001:5003], base[5003:]]  # 4-byte aligned only, ragged sizes
    views = [v.clone() if False else v for v in views]
    got = count_zeros([v.contiguous() for v in views])
    assert got == [int((v == 0).sum()) for v in views]

"""GPU: greedy filter pruning (prune_one_filter / filter_prune) against the incremental NumPy restatement, pick for pick,
with bit-exact masks; the cases where the reference never returns raise; the physically shrunk forward of a greedily
pruned network stays within the whole-net gates of test_gpu_conv.py."""
import re

import pytest
import torch

import filter_prune_oracle as fpo
import modelcompression_b200 as mc
from conftest import make_darknet

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'

_PICK = re.compile(r'^Prune filter #(\d+) in layer #(\d+)$')


def _printed(out):
    """(picks, printed rate lines) from the captured output."""
    lines = out.splitlines()
    picks = [(int(m.group(2)), int(m.group(1))) for m in map(_PICK.match, lines) if m]
    rates = [ln for ln in lines if ln.endswith(' pruned')]
    return picks, rates


def _params_np(model):
    return [p.detach().cpu().numpy() for p in model.parameters()]


def _check_against_oracle(model, perc, capsys, n_picks=None):
    params0 = _params_np(model)
    conv0 = [p.detach().clone() for p in model.parameters() if p.dim() == 4]
    keep_o, picks_o, rates_o, status_o = fpo.filter_prune_incremental_np(params0, perc, want_masks=False)
    assert status_o == 'done'
    capsys.readouterr()
    masks = mc.filter_prune(model, perc)
    picks, rate_lines = _printed(capsys.readouterr().out)
    assert picks == picks_o
    assert rate_lines == ['{:.2f} pruned'.format(r) for r in rates_o]
    if n_picks is not None:
        assert len(picks) == n_picks
    assert mc.prune_rate(model, verbose=False) == rates_o[-1]
    assert mc.are_masks_consistent(model, masks)
    conv = [p.data for p in model.parameters() if p.dim() == 4]
    assert len(masks) == len(conv) == len(keep_o)
    for m, w, w0, kp in zip(masks, conv, conv0, keep_o):
        assert m.dtype == torch.float32 and m.device == w.device and m.shape == w.shape
        k = torch.from_numpy(kp).to(DEV)
        want = k.float().view(-1, 1, 1, 1).expand_as(m)
        assert torch.equal(m, want)  # bit-exact: 1.0 / 0.0 everywhere
        assert torch.equal(w[k].view(torch.int32), w0[k].view(torch.int32))  # kept filters bitwise unchanged
        assert bool((w[~k] == 0).all())
    return picks


@pytest.fixture(scope='module')
def darknet_state(cfg_path):
    model = make_darknet(cfg_path, seed=0, device=DEV)
    return model, [p.detach().clone() for p in model.parameters()]


def _restored(darknet_state):
    model, state = darknet_state
    with torch.no_grad():
        for p, s in zip(model.parameters(), state):
            p.copy_(s)
    return model


@pytest.mark.parametrize('perc,n_picks', [(5., 362), (20., 1398), (40., 2803), (60., 4775), (90., 8654)])
def test_darknet_matches_oracle(darknet_state, capsys, perc, n_picks):
    model = _restored(darknet_state)
    _check_against_oracle(model, perc, capsys, n_picks)
    if perc == 40.:
        kept = [int(c.mask.flatten(1)[:, 0].sum()) for c in model.masked_convs()]
        assert kept == [32, 64, 128, 64, 128, 256, 128, 256, 511, 256, 511, 256, 511, 558, 503, 559, 501, 558, 562, 563,
                        64, 564, 125]


def test_darknet_weight_pruned_first(darknet_state, capsys):
    # per-filter zero counts: half of the weights are already zero
    model = _restored(darknet_state)
    model.set_masks(mc.weight_prune(model, 50.))
    rate0 = mc.prune_rate(model, verbose=False)
    assert 49. < rate0 < 50.
    state = [p.detach().clone() for p in model.parameters()]
    for perc in (60., 75.):
        with torch.no_grad():
            for p, s in zip(model.parameters(), state):
                p.copy_(s)
        _check_against_oracle(model, perc, capsys)
    with torch.no_grad():
        for p, s in zip(model.parameters(), state):
            p.copy_(s)
    picks = _check_against_oracle(model, 10., capsys)  # below the starting rate: exactly one pick
    assert len(picks) == 1


def test_zero_target_leaves_the_model_alone(darknet_state, capsys):
    model = _restored(darknet_state)
    before = [p.detach().clone() for p in model.parameters()]
    assert mc.filter_prune(model, 0.) == []
    assert mc.filter_prune(model, -5.) == []
    assert capsys.readouterr().out == ''
    assert all(torch.equal(p, b) for p, b in zip(model.parameters(), before))


def test_prune_one_filter(darknet_state, capsys):
    model = _restored(darknet_state)
    params0 = _params_np(model)
    before = [p.detach().clone() for p in model.parameters()]
    oracle_masks, layer, filt = fpo.prune_one_filter_np(params0, [])
    want_line = 'Prune filter #{} in layer #{}\n'.format(filt, layer)
    capsys.readouterr()
    empty = []
    masks = mc.prune_one_filter(model, empty)
    assert capsys.readouterr().out == want_line
    assert empty == [] and len(masks) == len(oracle_masks)  # an empty argument is replaced, as `masks = []` does there
    for m, o in zip(masks, oracle_masks):
        assert m.dtype == torch.float32 and m.device.type == 'cuda'
        assert torch.equal(m, torch.from_numpy(o).to(DEV))
    # an existing list: mutated in place (its contents are not read), weights untouched
    existing = [torch.ones_like(p) for p in model.parameters() if p.dim() == 4]
    existing[3][5] = 0.
    got = mc.prune_one_filter(model, existing)
    assert got is existing
    assert capsys.readouterr().out == want_line
    for i, m in enumerate(existing):
        want = torch.ones_like(m)
        if i == 3:
            want[5] = 0.
        if i == layer:
            want[filt] = 0.
        assert torch.equal(m, want)
    assert all(torch.equal(p, b) for p, b in zip(model.parameters(), before))
    with pytest.raises(AssertionError):
        mc.prune_one_filter(model, existing[:-1])


@pytest.mark.parametrize('name', sorted(set(fpo.small_nets()) - {'no_candidate'}))
@pytest.mark.parametrize('perc', [1., 10., 33.3, 60., 85.])
def test_small_nets(name, perc, capsys):
    params = fpo.small_nets()[name]
    masks_o, picks_o, rates_o, status_o = fpo.filter_prune_literal_np(params, perc)
    net = fpo.torch_small_net(params, DEV)
    capsys.readouterr()
    if status_o != 'done':
        with pytest.raises(RuntimeError):
            mc.filter_prune(net, perc)
        assert _printed(capsys.readouterr().out)[0] == picks_o
        return
    masks = mc.filter_prune(net, perc)
    picks, rate_lines = _printed(capsys.readouterr().out)
    assert picks == picks_o
    assert rate_lines == ['{:.2f} pruned'.format(r) for r in rates_o]
    for m, o in zip(masks, masks_o):
        assert torch.equal(m, torch.from_numpy(o).to(DEV))
    assert mc.prune_rate(net, verbose=False) == rates_o[-1]


def test_never_returning_cases_raise(darknet_state, capsys):
    # a target above the reachable rate: every layer ends with filter 0 alone
    model = _restored(darknet_state)
    before = [p.detach().clone() for p in model.parameters()]
    with pytest.raises((OverflowError, RuntimeError), match='rate'):
        mc.filter_prune(model, 100.)
    assert all(torch.equal(p, b) for p, b in zip(model.parameters(), before))
    # a layer pruned empty: 0 / 0 = NaN is picked forever by the reference
    params = fpo.small_nets()['pairwise_inf']
    assert fpo.filter_prune_incremental_np(params, 100.)[3] == 'nan_pick'
    with pytest.raises(RuntimeError, match='loop forever'):
        mc.filter_prune(fpo.torch_small_net(params, DEV), 100.)
    # NaN / inf weights
    for bad in (float('nan'), float('inf')):
        p = [a.copy() for a in fpo.small_nets()['ties']]
        p[1][3, 2, 1, 1] = bad
        net = fpo.torch_small_net(p, DEV)
        with pytest.raises(ValueError, match='non-finite'):
            mc.filter_prune(net, 10.)
        with pytest.raises(ValueError, match='non-finite'):
            mc.prune_one_filter(net, [])
    # every layer reports (inf, inf): the reference raises OverflowError at int(inf)
    net = fpo.torch_small_net(fpo.small_nets()['no_candidate'], DEV)
    with pytest.raises(OverflowError):
        mc.filter_prune(net, 10.)
    with pytest.raises(OverflowError):
        mc.prune_one_filter(net, [])
    capsys.readouterr()


def test_greedy_pruned_network_physically_shrunk(cfg_path):
    from test_gpu_conv import _check_blocks
    model = make_darknet(cfg_path, seed=0, kn=True, randbn=True, device=DEV)
    mc.filter_prune(model, 40.)
    torch.manual_seed(1)
    x1 = torch.rand(1, 3, 416, 416).to(DEV)
    model.b200_shrink = True
    y_s, _ = _check_blocks(model, x1, 'greedy40-shrunk')
    model.b200_shrink = False
    with torch.no_grad():
        y_d = model(x1)
    assert ((y_s - y_d).norm() / y_d.norm()).item() <= 2e-2

"""CPU restatements of the reference's greedy filter pruner, prune_one_filter / filter_prune
(src/pruning/weightPruning/methods.py:81-142), and the small networks the tests run them on.

filter_prune_literal_np     the reference loop on NumPy arrays: every step recomputes every layer's values from the
                            masked weights and recounts the pruning rate.
filter_prune_incremental_np raw filter values and nonzero counts computed once; a pick re-normalises its own layer only
                            (the algorithm libmcb200's mc_filter_prune_greedy runs).

Both return (masks, picks, rates, status): picks = [(layer, filter)] in order, rates = the rate printed after each
pick, status = 'done', 'nan_pick' (a pick that changes nothing: the reference repeats it forever), 'no_candidate'
(every layer reports (inf, inf): the reference's int(inf) raises), 'nonfinite' (incremental only: inf / NaN raw
values are rejected before the first pick) or 'budget'.
"""
import numpy as np

from modelcompression_b200.pruning.weightPruning.utils import arg_nonzero_min
from oracle.prune_oracle import prune_rate_np


def raw_values_np(p):
    """methods.py:93-94 before the normalisation (float32, NumPy's order)."""
    return np.square(p).sum(axis=1).sum(axis=1).sum(axis=1) / (p.shape[1] * p.shape[2] * p.shape[3])


def prune_one_filter_np(params, masks):
    """methods.py:81-126 on the arrays ``params`` (model.parameters() order).  Returns (masks, layer, filter); raises
    OverflowError where the reference does."""
    no_masks = not masks
    if no_masks:
        masks = []
    values = []
    for p in params:
        if p.ndim == 4:
            if no_masks:
                masks.append(np.ones(p.shape).astype('float32'))
            v = raw_values_np(p)
            v = v / np.sqrt(np.square(v).sum())
            min_value, min_ind = arg_nonzero_min(list(v))
            values.append([min_value, min_ind])
    assert len(masks) == len(values), "something wrong here"
    values = np.array(values)
    layer = int(np.argmin(values[:, 0]))
    filt = int(values[layer, 1])
    masks[layer][filt] = 0.
    return masks, layer, filt


def filter_prune_literal_np(params, pruning_perc):
    params = [np.array(p, dtype=np.float32) for p in params]
    masks, picks, rates = [], [], []
    current = 0.
    while current < pruning_perc:
        try:
            masks, layer, filt = prune_one_filter_np(params, masks)
        except OverflowError:
            return masks, picks, rates, 'no_candidate'
        conv = [i for i, p in enumerate(params) if p.ndim == 4]
        for i, m in zip(conv, masks):  # model.set_masks(masks): weight.data *= mask
            params[i] = params[i] * m
        rate = prune_rate_np(params)
        if picks and picks[-1] == (layer, filt) and rates[-1] == rate:
            return masks, picks, rates, 'nan_pick'  # same state, same pick: the loop never ends
        picks.append((layer, filt))
        rates.append(rate)
        current = rate
    return masks, picks, rates, 'done'


def _arg_nonzero_min_vec(v):
    """arg_nonzero_min(list(v)) vectorised: (value, index), index None for the reference's (inf, inf)."""
    nz = np.flatnonzero(v != 0)  # NaN != 0
    if nz.size == 0 or nz[-1] == 0:
        return np.inf, None
    last = int(nz[-1])
    if np.isnan(v[last]):
        return v[last], last
    ok = nz[~np.isnan(v[nz])]
    m = v[ok].min()
    if m < v[last]:
        return m, int(ok[np.argmax(v[ok] == m)])
    return v[last], last


def _candidate(raw):
    with np.errstate(invalid='ignore', divide='ignore'):  # 0 / 0 of a layer pruned empty is NaN, as in the reference
        return _arg_nonzero_min_vec(raw / np.sqrt(np.square(raw).sum()))


def filter_prune_incremental_np(params, pruning_perc, want_masks=True):
    """With want_masks=False the first element is the per-layer keep flags instead of full-shape masks."""
    if not (0. < pruning_perc):
        return [], [], [], 'done'
    conv = [np.asarray(p, dtype=np.float32) for p in params if p.ndim == 4]
    total = sum(p.size for p in params)
    zeros = sum(int(np.count_nonzero(p == 0)) for p in params if p.ndim != 1)
    raw = [raw_values_np(p) for p in conv]
    nzc = [np.count_nonzero(p.reshape(p.shape[0], -1), axis=1).astype(np.int64) for p in conv]
    keep = [np.ones(p.shape[0], bool) for p in conv]
    picks, rates = [], []
    status = 'budget'
    if all(np.isfinite(r).all() for r in raw):
        cand = [_candidate(r) for r in raw]
        while len(picks) < sum(p.shape[0] for p in conv):
            layer = int(np.argmin(np.array([c[0] for c in cand], dtype=np.float64)))
            v, filt = cand[layer]
            if filt is None:
                status = 'no_candidate'
                break
            zeros += int(nzc[layer][filt])
            nzc[layer][filt] = 0
            keep[layer][filt] = False
            picks.append((layer, filt))
            rates.append(100. * zeros / total)
            if not rates[-1] < pruning_perc:
                status = 'done'
                break
            if np.isnan(v):
                status = 'nan_pick'
                break
            raw[layer][filt] = 0
            cand[layer] = _candidate(raw[layer])
    else:
        status = 'nonfinite'
    if not want_masks:
        return keep, picks, rates, status
    masks = []
    for p, kp in zip(conv, keep):
        m = np.ones(p.shape, np.float32)
        m[~kp] = 0.
        masks.append(m)
    return masks, picks, rates, status


# ---- small networks ----------------------------------------------------------------------------------------------
def _conv(rs, o, c, k, scales=None):
    w = rs.standard_normal((o, c, k, k)).astype(np.float32)
    s = rs.uniform(0.2, 3.0, o).astype(np.float32) if scales is None else np.asarray(scales, np.float32)
    return (w * s[:, None, None, None]).astype(np.float32)


def small_nets():
    """name -> list of parameter arrays (4-D conv weights, 1-D biases / BN, 2-D Linear weights)."""
    nets = {}
    rs = np.random.RandomState(5)
    # pre-existing zero weights and all-zero filters, a Linear weight counted in the rate
    a = _conv(rs, 8, 3, 3)
    a[1] = 0.                      # all-zero filter
    a[4, 0] = 0.                   # zero weights inside a filter
    a[:, :, 0, 0][rs.rand(8, 3) < 0.3] = 0.
    b = _conv(rs, 16, 8, 3)
    b[np.abs(b) < 0.1] = 0.
    nets['zeros_linear'] = [a, rs.standard_normal(8).astype(np.float32), b, np.ones(16, np.float32),
                            np.zeros(16, np.float32), rs.standard_normal((10, 16)).astype(np.float32) * 0.1,
                            rs.standard_normal(10).astype(np.float32)]
    # duplicate filters, one of them a tie with the layer's last nonzero filter, and two identical layers
    c = _conv(rs, 12, 6, 3)
    c[3] = c[7]                    # duplicates in the middle
    c[11] = c[2] * np.float32(0.05)  # the layer minimum, last filter ...
    c[5] = c[11]                   # ... tied by an earlier filter: the last nonzero entry wins the tie
    d = _conv(rs, 12, 6, 3)
    d[10] *= np.float32(0.01)
    d[0] = d[9] = d[10]            # a minimum shared by three filters, not the last one: the first index wins
    nets['ties'] = [c, d, d.copy(), rs.standard_normal(12).astype(np.float32)]
    # a layer with only filter 0 nonzero (it reports (inf, inf)), a 1x1 layer over 300 channels (pairwise sums), a
    # layer with more than 128 filters (its norm is a pairwise sum over several leaves), a 5x5 layer, filter 0 zero
    e = _conv(rs, 5, 4, 3)
    e[1:] = 0.
    f = _conv(rs, 20, 300, 1)
    g = _conv(rs, 300, 4, 1)
    h = _conv(rs, 6, 3, 5)
    h[0] = 0.
    nets['pairwise_inf'] = [e, f, rs.standard_normal(20).astype(np.float32), g, h]
    # every layer reports (inf, inf) from the start: the reference raises at int(inf)
    nets['no_candidate'] = [e.copy(), e * np.float32(2), rs.standard_normal(5).astype(np.float32)]
    return nets


def torch_small_net(params, device):
    """A module whose parameters() are ``params`` (in order), with MaskedConv2d for the 4-D weights and set_masks."""
    import torch
    from modelcompression_b200.pruning.weightPruning.layers import MaskedConv2d

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.layers = torch.nn.ModuleList()
            for p in params:
                if p.ndim == 4:
                    m = MaskedConv2d(p.shape[1], p.shape[0], p.shape[2], bias=False)
                    m.weight.data = torch.from_numpy(p.copy())
                elif p.ndim == 2:
                    m = torch.nn.Linear(p.shape[1], p.shape[0], bias=False)
                    m.weight.data = torch.from_numpy(p.copy())
                else:
                    m = torch.nn.Module()
                    m.vec = torch.nn.Parameter(torch.from_numpy(p.copy()))
                self.layers.append(m)

        def set_masks(self, masks):
            convs = [m for m in self.layers if isinstance(m, MaskedConv2d)]
            assert len(convs) == len(masks)
            for m, mask in zip(convs, masks):
                m.set_mask(mask)

    return Net().to(device)

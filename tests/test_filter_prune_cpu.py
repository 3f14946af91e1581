"""CPU: the incremental restatement of greedy filter pruning (raw values computed once, one layer re-normalised per
pick) makes the same picks as the reference's literal loop, and the C-ABI entry point validates its arguments before
touching a device."""
import ctypes

import numpy as np
import pytest

import filter_prune_oracle as fpo
from modelcompression_b200 import _lib

NETS = fpo.small_nets()


@pytest.mark.parametrize('name', sorted(NETS))
@pytest.mark.parametrize('perc', [1., 10., 33.3, 60., 85.])
def test_incremental_matches_literal(name, perc):
    params = NETS[name]
    m_l, p_l, r_l, s_l = fpo.filter_prune_literal_np(params, perc)
    m_i, p_i, r_i, s_i = fpo.filter_prune_incremental_np(params, perc)
    assert (s_i, p_i, r_i) == (s_l, p_l, r_l)
    assert p_i or s_i == 'no_candidate'
    if s_i == 'done':
        assert len(m_i) == len(m_l)
        for a, b in zip(m_i, m_l):
            assert a.dtype == b.dtype == np.float32 and np.array_equal(a, b)


def test_small_nets_exercise_the_quirks():
    # the last nonzero filter wins a tie for the minimum; otherwise the first index of the minimum wins
    c, d = NETS['ties'][0], NETS['ties'][1]
    vc = fpo.raw_values_np(c) / np.sqrt(np.square(fpo.raw_values_np(c)).sum())
    vd = fpo.raw_values_np(d) / np.sqrt(np.square(fpo.raw_values_np(d)).sum())
    assert vc[5] == vc[11] == vc.min() and fpo._arg_nonzero_min_vec(vc)[1] == 11
    assert vd[0] == vd[9] == vd[10] == vd.min() and fpo._arg_nonzero_min_vec(vd)[1] == 0
    # two identical layers: the first one takes the cross-layer tie
    _, picks, _, _ = fpo.filter_prune_literal_np(NETS['ties'], 40.)
    assert picks[:4] == [(1, 0), (1, 9), (1, 10), (2, 0)]
    assert picks.index((0, 11)) < picks.index((0, 5))
    # a layer whose only nonzero filter is filter 0 is never picked
    _, picks, _, _ = fpo.filter_prune_incremental_np(NETS['pairwise_inf'], 85.)
    assert all(layer != 0 for layer, _ in picks)


def test_zero_and_already_met_targets():
    params = NETS['zeros_linear']
    assert fpo.filter_prune_literal_np(params, 0.) == ([], [], [], 'done')
    assert fpo.filter_prune_incremental_np(params, 0.) == ([], [], [], 'done')
    assert fpo.filter_prune_incremental_np(params, -3.)[1] == []
    rate0 = fpo.prune_rate_np(params)
    assert rate0 > 1.
    for fn in (fpo.filter_prune_literal_np, fpo.filter_prune_incremental_np):
        _, picks, rates, status = fn(params, 1.)  # below the initial rate: exactly one pick
        assert len(picks) == 1 and status == 'done' and rates[0] >= rate0


def test_unreachable_targets_stop():
    for name, params in NETS.items():
        _, p_l, _, s_l = fpo.filter_prune_literal_np(params, 100.)
        _, p_i, _, s_i = fpo.filter_prune_incremental_np(params, 100.)
        assert s_l == s_i and s_i in ('nan_pick', 'no_candidate') and p_l == p_i
    assert fpo.filter_prune_incremental_np(NETS['no_candidate'], 10.)[1:] == ([], [], 'no_candidate')
    with pytest.raises(OverflowError):
        fpo.prune_one_filter_np(NETS['no_candidate'], [])
    bad = [p.copy() for p in NETS['ties']]
    bad[1][3, 0, 0, 0] = np.nan
    assert fpo.filter_prune_incremental_np(bad, 10.)[3] == 'nonfinite'


def test_greedy_entry_point_validates_arguments():
    lib = _lib.load()
    O, C, K = _lib.int_array([8, 16]), _lib.int_array([3, 8]), _lib.int_array([3, 3])
    w = (ctypes.c_void_p * 2)(16, 16)
    ws = lib.mc_workspace_bytes_filter_prune_greedy(24)
    assert ws >= 24 * 12

    def call(wp=w, nlayers=2, max_picks=4, picks=16, result=16, d_ws=16, zeros0=0, total=1000):
        return lib.mc_filter_prune_greedy(wp, O, C, K, K, nlayers, zeros0, total, 10., max_picks, picks, result,
                                          None, d_ws, ws, None)

    for kw in (dict(wp=None), dict(picks=None), dict(result=None), dict(d_ws=None)):
        assert call(**kw) == -1 and b'null pointer' in lib.mc_last_error_string()
    for nl in (0, -1, 65):
        assert call(nlayers=nl) == -1 and b'nlayers' in lib.mc_last_error_string()
    for mp in (0, -2, 25):
        assert call(max_picks=mp) == -1 and b'max_picks' in lib.mc_last_error_string()
    assert call(zeros0=1001) == -1 and b'zeros0' in lib.mc_last_error_string()
    assert call(wp=(ctypes.c_void_p * 2)(16, None)) == -1 and b'null weight' in lib.mc_last_error_string()
    big = _lib.int_array([20481, 1])
    rc = lib.mc_filter_prune_greedy(w, big, C, K, K, 2, 0, 1000, 10., 1, 16, 16, None, 16, ws, None)
    assert rc == -2 and b'exceed' in lib.mc_last_error_string()

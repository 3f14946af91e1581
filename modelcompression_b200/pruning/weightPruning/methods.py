"""Drop-in for src/pruning/weightPruning/methods.py of the reference: weight_prune (:9-26), quick_filter_prune
(:28-78), prune_one_filter (:81-126) and filter_prune (:129-142), computed on the GPU by libmcb200 (no device->host copy
of the weights).

Host-side logic kept here is the data-independent part of ``np.percentile``: the rank ``k`` and interpolation
weight ``gamma`` of the 'linear' method, evaluated in the SAME dtype NumPy 2.x uses (float32 for the float32
magnitude array of weight_prune, float64 for the float64 value array of quick_filter_prune; SURVEY.md §8a-5/6).
"""
from itertools import chain as _chain

import numpy as np
import torch

from ... import _lib
from .utils import count_zeros


def percentile_rank(n, pruning_perc, dtype):
    """(k, gamma) such that np.percentile(a, pruning_perc) == _lerp(sorted(a)[k], sorted(a)[k+1], gamma) for an
    array ``a`` of ``n`` elements of ``dtype`` (NumPy >= 2.0, method='linear').

    Follows numpy/lib/_function_base_impl.py: percentile() divides by ``a.dtype.type(100)`` so a Python-float
    percentage takes the data dtype; _quantile(): virtual_index = (n-1)*q in that dtype; _get_indexes():
    previous = floor(virtual_index), clipped when virtual_index >= n-1; _get_gamma(): fractional part."""
    dtype = np.dtype(dtype)
    q = np.true_divide(pruning_perc, dtype.type(100) if dtype.kind == "f" else 100)
    if not (0 <= q <= 1):
        raise ValueError("Percentiles must be in the range [0, 100]")
    virtual_index = np.asanyarray((n - 1) * q)
    if virtual_index >= n - 1:
        return n - 1, 0.0
    if virtual_index < 0:
        return 0, 0.0
    previous = np.floor(virtual_index).astype(np.intp)
    gamma = np.asanyarray(virtual_index - previous).astype(virtual_index.dtype)
    return int(previous), float(gamma)


_WS = {}


def _workspace(dev, nbytes):
    """Scratch buffer kept between calls (the select needs up to 4n bytes; allocating 200 MB per call costs more
    than the kernels)."""
    key = (dev.type, dev.index)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = _WS[key] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    return ws


def _flat_like_all(params):
    """One allocation for all masks (23 allocator calls -> 1).  Returns (flat, element offsets); every offset is a
    multiple of 4 so each mask starts 16-byte aligned."""
    offs, off = [], 0
    for p in params:
        offs.append(off)
        off += ((p.numel() + 3) // 4) * 4
    return torch.empty(off, dtype=torch.float32, device=params[0].device), offs


def _views(flat, offs, params):
    return [flat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, params)]


def _empty_like_all(params):
    flat, offs = _flat_like_all(params)
    return _views(flat, offs, params)


class _ParamIndex(object):
    """model.parameters() without walking the module tree on every call (the nn.Module generator walk costs ~200 us on
    the 75-module Darknet, twice the pruning kernel).  The tree is walked once.  Afterwards a call (1) checks at C speed
    that the tree is the one that was walked — every module's ``_modules`` values by identity, every module's number
    of parameters — and (2) re-reads the parameter objects from their ``_parameters`` dicts, so a replaced Parameter is
    picked up, and a replaced / added / removed sub-module or a new parameter invalidates the index."""

    def __init__(self, model):
        mods, seen = [], set()

        def walk(m):
            if id(m) in seen:
                return
            seen.add(id(m))
            mods.append(m)
            for c in m._modules.values():
                if c is not None:
                    walk(c)
        walk(model)
        self.pdicts = [m._parameters for m in mods]
        self.mdicts = [m._modules for m in mods]
        self.mids = tuple(map(id, _chain.from_iterable(map(dict.values, self.mdicts))))
        self.plens = list(map(len, self.pdicts))
        slots, seen_p = [], set()
        for d in self.pdicts:  # parameters() order: first occurrence of every non-None parameter
            for name, p in d.items():
                if p is not None and id(p) not in seen_p:
                    seen_p.add(id(p))
                    slots.append((d, name))
        self.slots = slots
        self.shared = len(seen_p) != sum(1 for d in self.pdicts for p in d.values() if p is not None)
        self.plans = {}  # conv_only -> _PrunePlan

    def valid(self):
        return tuple(map(id, _chain.from_iterable(map(dict.values, self.mdicts)))) == self.mids and \
            list(map(len, self.pdicts)) == self.plens

    def parameters(self):
        """Current parameter objects in parameters() order (None slots / re-shared parameters force a re-walk)."""
        out = [d[name] for d, name in self.slots]
        if any(p is None for p in out) or (len(set(map(id, out))) != len(out)):
            return None
        return out


def _index(model):
    """(index, current parameter list) for the model, rebuilding the index when the module tree changed."""
    idx = model.__dict__.get('_b200_param_index')
    params = idx.parameters() if (idx is not None and idx.valid() and not idx.shared) else None
    if params is None:
        idx = model.__dict__['_b200_param_index'] = _ParamIndex(model)
        params = idx.parameters()
        if params is None:  # cannot happen right after a walk
            raise RuntimeError("internal: parameter index inconsistent")
    return idx, params


def _all_parameters(model):
    return _index(model)[1]


class _PrunePlan(object):
    """Everything about the prunable tensors that only depends on their shapes: which parameter slots, the ctypes size
    tables for the C-ABI, the layout of the flat mask buffer."""

    def __init__(self, params, conv_only):
        self.slots, self.shapes = [], []
        for i, p in enumerate(params):
            nd = p.dim()
            if (nd == 4) if conv_only else (nd != 1):
                self.slots.append(i)
                self.shapes.append(p.shape)
        self.numels = [int(np.prod(sh)) if len(sh) else 1 for sh in self.shapes]
        self.n = sum(self.numels)
        self.sizes64 = _lib.int64_array(self.numels)
        self.offs, off = [], 0
        for ne in self.numels:  # every mask starts 16-byte aligned inside the flat buffer
            self.offs.append(off)
            off += (ne + 3) // 4 * 4
        self.flat_len = off
        self.padded = [(ne + 3) // 4 * 4 for ne in self.numels]
        if conv_only:
            self.O = [sh[0] for sh in self.shapes]
            self.tables = tuple(_lib.int_array([sh[d] for sh in self.shapes]) for d in range(4))
        self.ok_ptrs = None   # data pointers of the last call that passed the device/dtype/contiguity checks
        self.ptr_array = None  # ... and their ctypes array
        self.ws_bytes = None


def _plan_and_tensors(model, conv_only):
    """(plan, tensors, ctypes pointer array): the prunable parameter tensors in parameters() order, validated (CUDA,
    float32, contiguous).  The per-tensor checks are skipped when the storage pointers are the ones already checked."""
    idx, params = _index(model)
    plan = idx.plans.get(conv_only)
    if plan is not None:
        if len(plan.slots) and plan.slots[-1] >= len(params):
            plan = None
        else:
            for i, sh in zip(plan.slots, plan.shapes):
                if params[i].shape != sh:  # replaced parameter / .data re-assigned with another shape
                    plan = None
                    break
    if plan is None:
        plan = idx.plans[conv_only] = _PrunePlan(params, conv_only)
    tensors = [params[i] for i in plan.slots]
    ptrs = [t.data_ptr() for t in tensors]
    if ptrs != plan.ok_ptrs:
        checked = []
        all_contig = True
        for t in tensors:
            if not t.is_cuda:
                _lib.require_cuda(t, "weight_prune / quick_filter_prune")
            if t.dtype != torch.float32:
                raise TypeError("pruners expect float32 parameters, got %s" % t.dtype)
            if not t.is_contiguous():
                all_contig = False
                t = t.data.contiguous()
            checked.append(t)
        tensors = checked
        arr = _lib.ptr_array(tensors)
        if all_contig:
            plan.ok_ptrs, plan.ptr_array = ptrs, arr
        else:
            plan.ok_ptrs = plan.ptr_array = None
        return plan, tensors, arr
    return plan, tensors, plan.ptr_array


def _prunable(model, conv_only):
    return [t.data for t in _plan_and_tensors(model, conv_only)[1]]


def _mask_views(flat, plan):
    """Per-parameter views of the flat mask buffer: one split + one view per tensor (created while the kernel runs)."""
    chunks = flat[:plan.flat_len].split(plan.padded)
    return [(c if c.numel() == ne else c[:ne]).view(sh) for c, ne, sh in zip(chunks, plan.numels, plan.shapes)]


def _on_device(dev):
    """Context that makes ``dev`` current; free when it already is (torch.cuda.device costs ~8 us per call)."""
    if torch.cuda.current_device() == (dev.index if dev.index is not None else torch.cuda.current_device()):
        return _NULLCTX
    return torch.cuda.device(dev)


class _NullCtx(object):
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NULLCTX = _NullCtx()


def weight_threshold(params, pruning_perc):
    """Device tensor [3] = (thr, sorted|w|[k], sorted|w|[k+1]) for the global magnitude percentile."""
    lib = _lib.load()
    n = sum(p.numel() for p in params)
    k, gamma = _rank_cached(n, pruning_perc, np.float32)
    dev = params[0].device
    segs = params
    if len(segs) > _lib.MC_MAX_SEGMENTS:  # rare: more tensors than one launch takes -> select on a flat copy
        segs = [torch.cat([p.reshape(-1) for p in params])]
    ws_bytes = lib.mc_workspace_bytes_kth_abs_select(n)
    ws = _workspace(dev, ws_bytes)
    out3 = torch.empty(3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.mc_kth_abs_select(_lib.ptr_array(segs), _lib.int64_array([t.numel() for t in segs]), len(segs),
                                         k, gamma, out3.data_ptr(), ws.data_ptr(), ws_bytes, _lib.stream_ptr()),
                   "mc_kth_abs_select")
    return out3


_RANK_CACHE = {}


def _rank_cached(n, pruning_perc, dtype):
    key = (n, float(pruning_perc), dtype)
    got = _RANK_CACHE.get(key)
    if got is None:
        if len(_RANK_CACHE) > 256:
            _RANK_CACHE.clear()
        got = _RANK_CACHE[key] = percentile_rank(n, pruning_perc, dtype)
    return got


def weight_prune(model, pruning_perc):
    '''
    Prune pruning_perc% weights globally (not layer-wise)
    arXiv: 1606.09274

    methods.py:9-26.  Returns one float32 {0,1} mask per parameter with dim != 1, in model.parameters() order, on
    the parameter's device: mask = |w| > np.percentile(|all w|, pruning_perc) (strict; ties are pruned).
    One cooperative kernel launch (mc_weight_prune_masks): W is read once and the masks are written once.
    '''
    lib = _lib.load()
    plan, params, parr = _plan_and_tensors(model, conv_only=False)
    if not params:
        return []
    if len(params) > _lib.MC_MAX_SEGMENTS:  # more tensors than one launch takes: threshold first, then mask in groups
        return _weight_prune_grouped(lib, [t.data for t in params], pruning_perc)
    n = plan.n
    k, gamma = _rank_cached(n, pruning_perc, np.float32)
    dev = params[0].device
    if plan.ws_bytes is None:
        plan.ws_bytes = lib.mc_workspace_bytes_kth_abs_select(n)
    ws_bytes = plan.ws_bytes
    # one allocation: the masks (flat, every mask 16-byte aligned) followed by the 3 result floats
    flat = torch.empty(plan.flat_len + 4, dtype=torch.float32, device=dev)
    base = flat.data_ptr()
    mask_ptrs = (_lib.c_void_p * len(params))(*[base + 4 * o for o in plan.offs])
    ws = _workspace(dev, ws_bytes)
    with _on_device(dev):
        _lib.check(lib.mc_weight_prune_masks(parr, mask_ptrs, plan.sizes64, len(params), k, gamma,
                                             base + 4 * plan.flat_len, ws.data_ptr(), ws_bytes, _lib.stream_ptr()),
                   "mc_weight_prune_masks")
    return _mask_views(flat, plan)


def _weight_prune_grouped(lib, params, pruning_perc):
    out3 = weight_threshold(params, pruning_perc)
    masks = _empty_like_all(params)
    dev = params[0].device
    with torch.cuda.device(dev):
        for lo in range(0, len(params), _lib.MC_MAX_SEGMENTS):
            grp, mgrp = params[lo:lo + _lib.MC_MAX_SEGMENTS], masks[lo:lo + _lib.MC_MAX_SEGMENTS]
            _lib.check(lib.mc_mask_apply_gt(_lib.ptr_array(grp), _lib.ptr_array(mgrp),
                                            _lib.int64_array([t.numel() for t in grp]), len(grp), out3.data_ptr(), 0,
                                            _lib.stream_ptr()), "mc_mask_apply_gt")
    return masks


def filter_values(params):
    """Normalised per-filter values of every conv weight, concatenated (device float32 [sum O])."""
    lib = _lib.load()
    if len(params) > _lib.MC_MAX_SEGMENTS:
        raise NotImplementedError("quick_filter_prune: more than %d conv layers" % _lib.MC_MAX_SEGMENTS)
    dev = params[0].device
    O = [p.shape[0] for p in params]
    values = torch.empty(sum(O), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.mc_filter_values(_lib.ptr_array(params), _lib.int_array(O),
                                        _lib.int_array([p.shape[1] for p in params]),
                                        _lib.int_array([p.shape[2] for p in params]),
                                        _lib.int_array([p.shape[3] for p in params]), len(params),
                                        values.data_ptr(), _lib.stream_ptr()), "mc_filter_values")
    return values


def quick_filter_prune(model, pruning_perc, return_keep=False):
    '''
    Prune pruning_perc% filters globally

    methods.py:28-78.  Per conv weight: v = mean(w^2) per filter (float32, NumPy summation order), v /= ||v||_2,
    v /= max(v); thr = float64 np.percentile over all layers; mask[o] = 0 where v[o] < thr.  Returns full-shape
    float32 masks in parameter order.  (The reference returns CPU tensors built from NumPy, methods.py:77, and
    set_mask moves them to the GPU; here they are created on the parameters' device.)
    With return_keep=True also returns the per-layer surviving-filter index tensors (int64, ascending).
    '''
    lib = _lib.load()
    plan, params, parr = _plan_and_tensors(model, conv_only=True)
    if not params:
        return ([], []) if return_keep else []
    if len(params) > _lib.MC_MAX_SEGMENTS:
        raise NotImplementedError("quick_filter_prune: more than %d conv layers" % _lib.MC_MAX_SEGMENTS)
    dev = params[0].device
    O = plan.O
    n = sum(O)
    k, gamma = _rank_cached(n, pruning_perc, np.float64)
    # one allocation: masks (flat, 16-byte aligned each) | values [n] f32 | thr f64 | kernel workspace | keep [n] u8
    n4 = (n + 1) // 2 * 2
    wsf = (int(lib.mc_workspace_bytes_filter_prune()) + 15) // 16 * 4  # workspace in floats
    flat = torch.empty(plan.flat_len + n4 + 2 + wsf + (n + 3) // 4, dtype=torch.float32, device=dev)
    mbase = flat.data_ptr()
    vbase = mbase + 4 * plan.flat_len
    mask_ptrs = (_lib.c_void_p * len(params))(*[mbase + 4 * o for o in plan.offs])
    with _on_device(dev):
        _lib.check(lib.mc_filter_prune(parr, plan.tables[0], plan.tables[1], plan.tables[2],
                                       plan.tables[3], len(params), k, gamma, vbase, vbase + 4 * n4, mask_ptrs,
                                       vbase + 4 * n4 + 8 + 4 * wsf, vbase + 4 * n4 + 8, 4 * wsf, _lib.stream_ptr()),
                   "mc_filter_prune")
    masks = _mask_views(flat, plan)
    if not return_keep:
        return masks
    keep = flat[plan.flat_len + n4 + 2 + wsf:].view(torch.uint8)[:n]
    keep_idx = [torch.nonzero(kp, as_tuple=False).flatten() for kp in torch.split(keep, O)]
    return masks, keep_idx


_GREEDY_DONE, _GREEDY_BUDGET, _GREEDY_NAN_PICK, _GREEDY_NO_CANDIDATE, _GREEDY_NONFINITE = range(5)


def _greedy_prune(model, perc, max_picks, zeros0, total, want_masks):
    """One mc_filter_prune_greedy call over the conv (4-D) weights.  Returns (masks or None, [(layer, filter, nonzero
    weights)] in pick order, final zero count, status).  The picks come back in one device->host copy."""
    lib = _lib.load()
    plan, params, parr = _plan_and_tensors(model, conv_only=True)
    if not params:
        raise ValueError("filter pruning: the model has no 4-D (conv) parameters")
    if len(params) > _lib.MC_MAX_SEGMENTS:
        raise NotImplementedError("filter pruning: more than %d conv layers" % _lib.MC_MAX_SEGMENTS)
    dev = params[0].device
    n = sum(plan.O)
    ws_bytes = lib.mc_workspace_bytes_filter_prune_greedy(n)
    ws = _workspace(dev, ws_bytes)
    out = torch.empty(6 + 2 * max_picks, dtype=torch.int32, device=dev)  # result int64 [3] | picks int32 [max_picks][2]
    flat = mask_ptrs = None
    if want_masks:
        flat = torch.empty(plan.flat_len, dtype=torch.float32, device=dev)
        mask_ptrs = (_lib.c_void_p * len(params))(*[flat.data_ptr() + 4 * o for o in plan.offs])
    with _on_device(dev):
        _lib.check(lib.mc_filter_prune_greedy(parr, plan.tables[0], plan.tables[1], plan.tables[2], plan.tables[3],
                                              len(params), zeros0, total, float(perc), max_picks, out.data_ptr() + 24,
                                              out.data_ptr(), mask_ptrs, ws.data_ptr(), ws_bytes, _lib.stream_ptr()),
                   "mc_filter_prune_greedy")
    host = out.cpu().numpy()
    npick, zeros, status = (int(x) for x in host[:6].view(np.int64))
    fc = host[6:6 + 2 * npick].reshape(-1, 2).astype(np.int64)
    layer_of = np.searchsorted(np.cumsum(plan.O), fc[:, 0], side='right')
    first = np.concatenate(([0], np.cumsum(plan.O)))[layer_of]
    picks = list(zip(layer_of.tolist(), (fc[:, 0] - first).tolist(), fc[:, 1].tolist()))
    masks = _mask_views(flat, plan) if want_masks else None
    return masks, picks, zeros, status


def _raise_for_status(status, what):
    if status == _GREEDY_NONFINITE:
        raise ValueError("%s: a conv weight gives a non-finite filter value (inf or NaN weights); nothing was pruned"
                         % what)
    if status == _GREEDY_NO_CANDIDATE:  # the reference raises OverflowError from int(inf) here
        raise OverflowError("%s: no conv layer has a nonzero filter value left to prune" % what)


def prune_one_filter(model, masks):
    '''
    methods.py:81-126.  Picks the filter with the smallest nonzero value v = mean(w^2) / ||mean(w^2) of its layer||_2
    over all conv (4-D) parameters, read from the CURRENT weights (``masks`` is not consulted), and zeroes
    ``masks[layer][filter]`` in place.  An empty ``masks`` is first filled with all-ones float32 masks on the parameters'
    device.  Does not call set_masks.  Prints the reference's "Prune filter #f in layer #l" line and returns ``masks``.
    Non-finite weights raise ValueError; when no layer has a nonzero filter left it raises OverflowError, as the
    reference's int(inf) does.
    '''
    no_masks = not masks
    if no_masks:
        masks = []
    else:
        assert len(masks) == len(_prunable(model, conv_only=True)), "something wrong here"
    built, picks, _, status = _greedy_prune(model, float('inf'), 1, 0, 1, want_masks=no_masks)
    _raise_for_status(status, "prune_one_filter")
    layer, filt, _ = picks[0]
    if no_masks:
        masks.extend(built)  # the picked filter is already zero in these
    else:
        masks[layer][filt] = 0.
    print('Prune filter #{} in layer #{}'.format(filt, layer))
    return masks


def filter_prune(model, pruning_perc):
    '''
    Greedy filter pruning, one filter at a time (arXiv:1611.06440).  methods.py:129-142.

    Repeats prune_one_filter until prune_rate(model) >= pruning_perc, starting from a rate of 0 (so at least one filter
    is pruned whenever pruning_perc > 0; pruning_perc <= 0 returns [] and leaves the model alone).  A pruned filter's
    surviving neighbours are only ever multiplied by 1.0, so the whole walk is one GPU call: each filter's value is
    computed once and a pick re-normalises its own layer only.  Returns all-ones float32 masks with the picked filters
    zeroed and applies them with model.set_masks (replacing earlier masks; weights zeroed earlier stay zero).  Prints
    the reference's two lines per pick.  Where the reference never returns (a layer pruned empty, NaN weights, a target
    above the reachable rate) or raises, this raises and leaves the model unchanged.
    '''
    if not (0. < pruning_perc):
        return []
    params = list(model.parameters())
    total = sum(p.numel() for p in params)
    prunable = [p.data for p in params if p.dim() != 1]
    zeros0 = sum(count_zeros(prunable)) if prunable else 0
    n = sum(_plan_and_tensors(model, conv_only=True)[0].O)
    masks, picks, zeros, status = _greedy_prune(model, pruning_perc, n, zeros0, total, want_masks=True)
    z = zeros0
    for layer, filt, nz in picks:
        z += nz
        print('Prune filter #{} in layer #{}'.format(filt, layer))
        print('{:.2f} pruned'.format(100. * z / total))
    rate = 100. * zeros / total
    _raise_for_status(status, "filter_prune (pruning rate %.4f%% after %d picks)" % (rate, len(picks)))
    if status == _GREEDY_NAN_PICK:
        raise RuntimeError("filter_prune: stopped at a pruning rate of %.4f%% < %s: a conv layer has no filter with a "
                           "nonzero value left (all pruned or all-zero weights), the reference would loop forever"
                           % (rate, pruning_perc))
    if status == _GREEDY_BUDGET:
        raise RuntimeError("filter_prune: every filter was pruned and the rate reached is only %.4f%% < %s"
                           % (rate, pruning_perc))
    model.set_masks(masks)
    return masks

"""B200 training-mode engine behind ``Darknet.forward`` when ``model.training`` is set: the masked retrain step of the
reference (src/train.py:214-235 — forward with batch-statistics BatchNorm, ``loss.backward()``, ``optimizer.step()``).

The reference builds an autograd graph over nn.Modules (MaskedConv2d -> BatchNorm2d -> LeakyReLU -> MaxPool2d ...,
src/nets.py:720-822).  Here the whole network is ONE autograd node: its forward launches the libmcb200 kernels and keeps
the per-layer tensors the backward needs; its backward launches the gradient kernels and hands autograd the gradients
of every parameter, so ``loss.backward()`` / ``optimizer.step()`` work unchanged on the reference's parameters.

Per conv layer (all activations PNHWC bf16, include/mcb200.h):
  forward   z = conv(a_prev, W*mask)            mc_conv_fwd (tcgen05; the 3-channel first layer: mc_conv_im2col_fwd)
            batch mean/var of z                 mc_col_stats + mc_bn_finalize (also updates the running statistics)
            a = leaky(z*scale + shift)          mc_bn_apply (writes concat slices / the Reorg shuffle directly)
            p = maxpool2x2(a)                   mc_maxpool2x2
  backward  da = unpool(dp)                     mc_maxpool2x2_backward (accumulates when `a` has two consumers)
            dz, dgamma, dbeta                   mc_bn_backward
            dW = mask * (a_prev^T dz)           mc_conv_wgrad (tcgen05, MN-major operands; first layer: CUDA cores)
            da_prev = conv(dz, flip(W*mask)^T)  mc_conv_fwd on mc_pack_conv_weights_dgrad weights
Masked weights get exactly zero gradient (dW is multiplied by the mask, layers.py:59), so with the reference's SGD
(weight decay of a zero weight is zero) they stay zero: ``are_masks_consistent`` holds after the step.

No CPU / PyTorch fallback: a CPU tensor or an unsupported cfg raises.
"""
import ctypes
import weakref

import torch

from . import _lib


def _round_up(x, m):
    return (x + m - 1) // m * m


class _Act(object):
    """An activation tensor in PNHWC: buffer name + geometry."""

    def __init__(self, name, H, W, C, ld, ch_off=0):
        self.name, self.H, self.W, self.C, self.ld, self.ch_off = name, H, W, C, ld, ch_off


class _Layer(object):
    pass


class TrainPlan(object):
    """Static description of the cfg graph for training: layers, which buffer each reads/writes."""

    def __init__(self, model):
        self.lib = _lib.load()
        blocks = model.blocks
        H, W = model.height, model.width
        if H % 32 or W % 32:
            raise NotImplementedError("input size must be a multiple of 32 (cfg has %dx%d)" % (W, H))
        self.in_hw = (H, W)
        self.layers = []
        self.buf_specs = {}   # name -> (H, W, ld)
        self.grad_specs = {}  # name -> (H, W, ld) gradient buffers (same geometry as the activation they belong to)
        cat_of = {}
        ind = -2
        for block in blocks:
            ind += 1
            if block['type'] == 'route':
                ls = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                if len(ls) == 2:
                    cat_of[ls[0]] = (ind, 0)
                    cat_of[ls[1]] = (ind, 1)
                elif len(ls) != 1:
                    raise NotImplementedError("route with %d inputs" % len(ls))
        last_conv = max(i for i, b in enumerate(blocks[1:]) if b['type'] == 'convolutional')
        out_of = {}      # block index -> _Act
        cur = None       # None = the fp32 NCHW image
        cur_hw = (H, W)
        in_ch = int(blocks[0]['channels'])
        cat_parts = {}   # route index -> {slot: (C, producer layer)}
        pending = None   # the convolution a following maxpool / reorg block belongs to
        ind = -2
        skip = False
        for bi, block in enumerate(blocks):
            ind += 1
            t = block['type']
            if t == 'net':
                continue
            if t == 'convolutional':
                seq = model.models[ind]
                conv = seq[0]
                k = conv.kernel_size[0]
                if conv.kernel_size != (k, k) or k not in (1, 3) or conv.stride != (1, 1) or \
                        conv.padding != ((k - 1) // 2, (k - 1) // 2) or conv.groups != 1 or conv.dilation != (1, 1):
                    raise NotImplementedError("conv %s is outside the B200 path" % (conv,))
                act = block['activation']
                if act not in ('leaky', 'linear'):
                    raise NotImplementedError("activation '%s'" % act)
                L = _Layer()
                L.ind, L.conv, L.k = ind, conv, k
                L.bn = seq[1] if int(block['batch_normalize']) else None
                L.leaky = int(act == 'leaky')
                L.src = cur
                L.H, L.W = cur_hw
                L.C = in_ch if cur is None else cur.C
                L.O = conv.out_channels
                if conv.in_channels != L.C:
                    raise RuntimeError("conv at block %d expects %d input channels, graph provides %d" % (ind, conv.in_channels, L.C))
                L.is_head = ind == last_conv
                nxt = blocks[bi + 1] if bi + 1 < len(blocks) else None
                L.pool = bool(nxt is not None and nxt['type'] == 'maxpool' and int(nxt['size']) == 2 and int(nxt['stride']) == 2)
                L.reorg = bool(nxt is not None and nxt['type'] == 'reorg' and int(nxt['stride']) == 2)
                if L.is_head:
                    if L.bn is not None or L.leaky or L.pool or L.reorg:
                        raise NotImplementedError("head convolution must be linear without BatchNorm")
                    if conv.bias is None:
                        raise NotImplementedError("head convolution without bias")
                    L.z = L.act = L.pooled = None
                    cur = None
                else:
                    if L.bn is None:
                        raise NotImplementedError("training path needs BatchNorm on every hidden convolution")
                    ldz = _round_up(L.O, 8)
                    L.z = _Act('z%d' % ind, L.H, L.W, L.O, ldz)
                    self.buf_specs[L.z.name] = (L.H, L.W, ldz)
                    self.grad_specs['dz%d' % ind] = (L.H, L.W, ldz)
                    if L.reorg:
                        if (ind + 1) not in cat_of:
                            raise NotImplementedError("reorg must feed a concat")
                        route, slot = cat_of[ind + 1]
                        cat_parts.setdefault(route, {})[slot] = (4 * L.O, L)
                        L.act = None  # resolved when the concat is complete
                        skip = True
                        cur_hw = (L.H // 2, L.W // 2)
                    elif ind in cat_of:
                        route, slot = cat_of[ind]
                        cat_parts.setdefault(route, {})[slot] = (L.O, L)
                        L.act = None
                    else:
                        L.act = _Act('a%d' % ind, L.H, L.W, L.O, ldz)
                        self.buf_specs[L.act.name] = (L.H, L.W, ldz)
                        self.grad_specs['d' + L.act.name] = (L.H, L.W, ldz)
                    L.pooled = None
                    if L.pool:
                        if L.act is None:
                            raise NotImplementedError("maxpool after a concat producer")
                        Ho, Wo = L.H // 2, L.W // 2
                        L.pooled = _Act('p%d' % ind, Ho, Wo, L.O, ldz)
                        self.buf_specs[L.pooled.name] = (Ho, Wo, ldz)
                        self.grad_specs['d' + L.pooled.name] = (Ho, Wo, ldz)
                        skip = True
                    cur = L.act  # the conv block's own output is the full-resolution activation
                    pending = L
                self.layers.append(L)
                out_of[ind] = cur
                # a concat becomes addressable once both producers are known
                for route, parts in cat_parts.items():
                    if len(parts) == 2 and ('cat%d' % route) not in self.buf_specs:
                        (c0, l0), (c1, l1) = parts[0], parts[1]
                        h0, w0 = (l0.H // 2, l0.W // 2) if l0.reorg else (l0.H, l0.W)
                        h1, w1 = (l1.H // 2, l1.W // 2) if l1.reorg else (l1.H, l1.W)
                        if (h0, w0) != (h1, w1):
                            raise NotImplementedError("concat of different resolutions")
                        off1 = _round_up(c0, 8)
                        ld = _round_up(off1 + c1, 8)
                        if off1 != c0:
                            raise NotImplementedError("concat parts must be multiples of 8 channels")
                        name = 'cat%d' % route
                        self.buf_specs[name] = (h0, w0, ld)
                        self.grad_specs['d' + name] = (h0, w0, ld)
                        l0.act = _Act(name, h0, w0, c0, ld, 0)
                        l1.act = _Act(name, h1, w1, c1, ld, off1)
                        out_of['cat%d' % route] = _Act(name, h0, w0, c0 + c1, ld, 0)
            elif t == 'maxpool':
                if not skip or pending is None or not pending.pool:
                    raise NotImplementedError("maxpool (2x2/2 only) must directly follow a convolution")
                skip = False
                cur = pending.pooled
                cur_hw = (cur.H, cur.W)
                out_of[ind] = cur
            elif t == 'reorg':
                if not skip or pending is None or not pending.reorg:
                    raise NotImplementedError("reorg that does not directly follow a convolution")
                skip = False
                cur = None  # only reachable through the concat it feeds
                out_of[ind] = None
            elif t == 'route':
                ls = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                if len(ls) == 1:
                    cur = out_of[ls[0]]
                    if cur is None:
                        raise NotImplementedError("route to a concat producer")
                else:
                    cur = out_of.get('cat%d' % ind)
                    if cur is None:
                        raise NotImplementedError("concat inputs must both be produced by convolutions")
                cur_hw = (cur.H, cur.W)
                out_of[ind] = cur
            elif t == 'region':
                continue
            else:
                raise NotImplementedError("cfg block type '%s'" % t)
        if not self.layers or not self.layers[-1].is_head:
            raise NotImplementedError("the network must end in the linear head convolution")
        for L in self.layers:
            if not L.is_head and L.act is None:
                raise NotImplementedError("unresolved concat producer at block %d" % L.ind)
        # Pooled layers whose full-resolution activation feeds nothing but the pool: BatchNorm + leaky + pool run as one
        # pass each way (mc_bn_apply_pool / mc_bn_pool_backward) and the activation / its gradient are never stored
        for L in self.layers:
            L.fused_pool = False
            if not (L.pool and not L.is_head and L.act is not None and L.act.name == 'a%d' % L.ind):
                continue
            if self.lib.mc_bn_pool_supported(L.O) != 1 or any(o.src is L.act for o in self.layers):
                continue
            L.fused_pool = True
            del self.buf_specs[L.act.name]
            del self.grad_specs['d' + L.act.name]
            L.act = None
        self._bufs = {}  # (B, device) -> dict name -> tensor
        self._consts = {}  # (device, kind, n) -> constant vectors / reusable staging tensors (no fill kernels per step)
        self.dp_group = None   # set by train_dp.enable(): gradients are all-reduced inside the backward
        self.dp_world = 1

    def const(self, dev, val, n):
        """A cached float32 vector of n copies of val (scale = 1 / shift = 0 operands of the conv epilogues): allocating
        them per layer and step cost ~100 fill launches (0.58 ms of a 15.9 ms step)."""
        key = (str(dev), float(val), int(n))
        t = self._consts.get(key)
        if t is None:
            t = self._consts[key] = torch.full((int(n),), float(val), device=dev)
        return t

    def scratch(self, dev, name, shape, dtype=torch.float32, zero=False):
        """A cached staging tensor (rewritten in place every step by stream-ordered kernels)."""
        key = (str(dev), name, tuple(shape), dtype)
        t = self._consts.get(key)
        if t is None:
            t = self._consts[key] = (torch.zeros if zero else torch.empty)(tuple(shape), dtype=dtype, device=dev)
        return t

    # ------------------------------------------------------------------------------------------------ parameters
    def parameters(self):
        """The tensors autograd must see, in the order the backward returns their gradients."""
        ps = []
        for L in self.layers:
            ps.append(L.conv.weight)
            if L.bn is not None:
                ps += [L.bn.weight, L.bn.bias]
            if L.is_head:
                ps.append(L.conv.bias)
        return ps

    def buffers(self, B, dev, owner=None):
        """A buffer set (activations saved for backward + gradient buffers) for batch B.  Sets are cached per (B, device).
        A set whose forward still has a backward pending (its `owner`, the _Saved object autograd holds through ctx, is
        alive and not yet consumed) is never handed out again: a second training-mode forward before the backward —
        gradient accumulation over two micro-batches, loss(model(x1)) + loss(model(x2)), or a train-mode forward under
        no_grad — gets another set instead of overwriting the saved tensors of the pending graph (the reference's
        autograd graph keeps every forward's tensors alive in the same way).  owner=None: the caller promises no
        backward (no_grad / tests); the set is free again immediately."""
        key = (B, str(dev))
        sets = self._bufs.setdefault(key, [])
        for st in sets:
            ref = st['owner']
            if ref is None or ref() is None or ref().consumed:
                break
        else:
            st = {'owner': None, 't': {}}
            for name, (H, W, ld) in list(self.buf_specs.items()) + list(self.grad_specs.items()):
                st['t'][name] = torch.zeros(B * (H + 1) * (W + 1), ld, dtype=torch.bfloat16, device=dev)
            sets.append(st)
        st['owner'] = weakref.ref(owner) if owner is not None else None
        return st['t']


def _kblk(C, k=1):
    """k-block of the tcgen05 conv: 32 (64-byte swizzle) where it halves the K work, i.e. for <= 32 channels (TMA cost
    follows the box area: measured faster than a half-empty 64-wide box, see engine.py)."""
    return 32 if C <= 32 else 64


def _conv_desc(in_ptr, wpack, scale, shift, out_ptr, B, H, W, Cin, Cin_ld, N, Npad, k, leaky, epi, ldc, ch_off, block_k=0,
               plan=None, dev=None):
    d = _lib.mc_conv_desc()
    d.block_k = block_k
    d.d_in, d.d_wpack, d.d_scale, d.d_shift, d.d_out = in_ptr, wpack, scale, shift, out_ptr
    d.B, d.H, d.W, d.Cin, d.Cin_ld, d.N, d.Npad = B, H, W, Cin, Cin_ld, N, Npad
    d.ksize, d.leaky, d.epi_mode, d.ldc, d.ch_off, d.block_n, d.stages = k, leaky, epi, ldc, ch_off, 0, 0
    if plan is not None:
        need = int(plan.lib.mc_workspace_bytes_conv_fwd(ctypes.byref(d)))
        if need:
            ws = plan.scratch(dev, 'conv_ws', (need,), torch.uint8, zero=True)
            d.d_ws, d.ws_bytes = ws.data_ptr(), need
    return d


def _masked(conv):
    return conv.mask.data_ptr() if getattr(conv, 'mask_flag', False) else None


class _Saved(object):
    consumed = False  # set once the backward has run (or the caller declared that none will)


def _forward(plan, x, training_stats=True, after_layer=None, needs_backward=True):
    """Launch the training-mode forward; returns (y, saved).  after_layer(L, bufs) is a test hook called once a hidden
    layer's activation (and pooled activation) is in its buffer."""
    lib = plan.lib
    dev = x.device
    B, _, H, W = x.shape
    if (H, W) != plan.in_hw:
        raise NotImplementedError("the plan was built for %dx%d inputs (cfg width/height); got %dx%d" %
                                  (plan.in_hw[1], plan.in_hw[0], W, H))
    sv = _Saved()
    bufs = plan.buffers(B, dev, sv if needs_backward else None)
    sv.x, sv.B, sv.bufs, sv.stats = x, B, bufs, {}
    s = _lib.stream_ptr()
    y = None
    fuse_stats = bool(getattr(plan, 'fuse_stats', True))
    for L in plan.layers:
        stats_done = False
        st = None
        conv = L.conv
        w = conv.weight.data
        mask_ptr = _masked(conv)
        O, C, k = L.O, L.C, L.k
        Npad = _round_up(O, 16)
        ones = plan.const(dev, 1.0, max(Npad, 16))
        zeros = plan.const(dev, 0.0, max(Npad, 16))
        if L.src is None:
            # first layer: im2col tensor-core kernel straight from the fp32 NCHW image (weights expanded on the host:
            # row n, column (r*3+s)*CL + c; include/mcb200.h)
            if k != 3 or lib.mc_conv_im2col_supported(C, 1, O, 0) != 1:
                raise NotImplementedError("first layer must be a 3x3 convolution on <= 4 channels with <= 256 filters")
            cl, npos, nb, kpad = (ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int())
            _lib.check(lib.mc_conv_im2col_geometry(C, 1, O, 0, ctypes.byref(cl), ctypes.byref(npos), ctypes.byref(nb),
                                                   ctypes.byref(kpad)), "mc_conv_im2col_geometry")
            weff = w if mask_ptr is None else w * conv.mask
            nb_pad = _round_up(nb.value, 16)
            # expanded weights: the zero padding is written once, the 27 real columns are refreshed in place
            wexp = plan.scratch(dev, 'wexp1', (nb_pad, kpad.value // cl.value, cl.value), zero=True)
            wexp[:O, :9, :C] = weff.permute(0, 2, 3, 1).reshape(O, 9, C)
            wfull = plan.scratch(dev, 'wfull1', (nb_pad, kpad.value), torch.bfloat16)
            wfull.copy_(wexp.view(nb_pad, kpad.value))
            n_sc = max(_round_up(npos.value, 16), 16)
            sc1, sh0 = plan.const(dev, 1.0, n_sc), plan.const(dev, 0.0, n_sc)
            z = bufs[L.z.name]
            _lib.check(lib.mc_conv_im2col_fwd(x.data_ptr(), 1, wfull.data_ptr(), sc1.data_ptr(), sh0.data_ptr(),
                                              z.data_ptr(), B, L.H, L.W, C, C, O, L.z.ld, 0, 0, s), "conv1 forward")
            sv.keep_alive = (wfull, sc1, sh0)
        else:
            kb = _kblk(C, k)
            Kc = _round_up(C, kb)
            wpack = torch.empty(Npad, k * k * Kc, dtype=torch.bfloat16, device=dev)
            _lib.check(lib.mc_pack_conv_weights(w.data_ptr(), mask_ptr, O, C, k, None, O, None, C, wpack.data_ptr(), Npad,
                                                Kc, s), "mc_pack_conv_weights")
            src = L.src
            in_ptr = bufs[src.name].data_ptr() + 2 * src.ch_off
            if L.is_head:
                y = torch.empty(B, O, L.H, L.W, dtype=torch.float32, device=dev)
                shift = plan.scratch(dev, 'head_shift', (Npad,), zero=True)
                shift[:O].copy_(conv.bias.data)
                d = _conv_desc(in_ptr, wpack.data_ptr(), ones.data_ptr(), shift.data_ptr(), y.data_ptr(), B, L.H, L.W, C,
                               src.ld, O, Npad, k, 0, _lib.MC_EPI_NCHW_F32, 0, 0, kb, plan, dev)
                _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "head forward")
                continue
            z = bufs[L.z.name]
            d = _conv_desc(in_ptr, wpack.data_ptr(), ones.data_ptr(), zeros.data_ptr(), z.data_ptr(), B, L.H, L.W, C,
                           src.ld, O, Npad, k, 0, _lib.MC_EPI_PNHWC, L.z.ld, 0, kb, plan, dev)
            if fuse_stats and O > 32 and (L.z.ld % 8) == 0:
                # batch statistics straight from the conv epilogue (sums of the stored bf16 z): no mc_col_stats pass
                st = torch.zeros(6, O, device=dev)
                d.d_stat_sum, d.d_stat_sumsq = st[0].data_ptr(), st[1].data_ptr()
                stats_done = True
            _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "conv forward (block %d)" % L.ind)
        # ---- batch statistics + affine + leaky
        bn = L.bn
        rows = B * (L.H + 1) * (L.W + 1)
        if not stats_done:
            st = torch.empty(6, O, device=dev)  # sum, sumsq, scale, shift, mean, invstd
            _lib.check(lib.mc_col_stats(z.data_ptr(), rows, O, L.z.ld, 0, st[0].data_ptr(), st[1].data_ptr(), s),
                       "mc_col_stats")
        upd = training_stats and bn.track_running_stats and bn.running_mean is not None
        mom = bn.momentum if bn.momentum is not None else 0.1
        _lib.check(lib.mc_bn_finalize(st[0].data_ptr(), st[1].data_ptr(), O, float(B * L.H * L.W), bn.weight.data_ptr(),
                                      bn.bias.data_ptr(), bn.eps, mom,
                                      bn.running_mean.data_ptr() if upd else None,
                                      bn.running_var.data_ptr() if upd else None,
                                      st[2].data_ptr(), st[3].data_ptr(), st[4].data_ptr(), st[5].data_ptr(), s),
                   "mc_bn_finalize")
        if upd and bn.num_batches_tracked is not None:
            bn.num_batches_tracked += 1
        sv.stats[L.ind] = st
        if L.fused_pool:
            _lib.check(lib.mc_bn_apply_pool(z.data_ptr(), L.z.ld, B, L.H, L.W, O, st[2].data_ptr(), st[3].data_ptr(),
                                            L.leaky, bufs[L.pooled.name].data_ptr(), L.pooled.ld, s), "mc_bn_apply_pool")
            if after_layer is not None:
                after_layer(L, bufs)
            continue
        a = L.act
        _lib.check(lib.mc_bn_apply(z.data_ptr(), L.z.ld, B, L.H, L.W, O, st[2].data_ptr(), st[3].data_ptr(), L.leaky,
                                   bufs[a.name].data_ptr(), a.ld, a.ch_off, int(L.reorg), s), "mc_bn_apply")
        if L.pool:
            _lib.check(lib.mc_maxpool2x2(bufs[a.name].data_ptr(), bufs[L.pooled.name].data_ptr(), B, L.H, L.W, O, a.ld,
                                         L.pooled.ld, s), "mc_maxpool2x2")
        if after_layer is not None:
            after_layer(L, bufs)
    return y, sv


_WS = {}


def _workspace(dev, nbytes):
    key = str(dev)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = _WS[key] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=dev)
    return ws


def _backward(plan, sv, dy, before_bn=None):
    """Launch the backward; returns the gradients in plan.parameters() order.  before_bn(L, bufs) is a test hook called
    when the gradient of a hidden layer's activation is complete (just before its BatchNorm backward)."""
    lib = plan.lib
    dev = dy.device
    B, bufs = sv.B, sv.bufs
    s = _lib.stream_ptr()
    grads = {}
    written = set()  # gradient buffers that already hold a contribution in this backward
    pending = []     # data-parallel: (work handle, tensor) of the gradient all-reduces in flight

    def reduce_async(t):
        # SURVEY.md §8f N4: the all-reduce of a layer's gradient is issued as soon as the layer's wgrad is queued, so NCCL
        # (its own stream, NVLink/NVSwitch) overlaps the backward of the layers below
        if plan.dp_world > 1:
            import torch.distributed as dist
            pending.append((dist.all_reduce(t, group=plan.dp_group, async_op=True), t))
        return t
    head = plan.layers[-1]
    Hh, Wh = head.H, head.W
    ld_h = _round_up(head.O, 8)
    dzh = torch.empty(B * (Hh + 1) * (Wh + 1), ld_h, dtype=torch.bfloat16, device=dev)
    _lib.check(lib.mc_pack_pnhwc(dy.data_ptr(), dzh.data_ptr(), B, Hh, Wh, head.O, ld_h, s), "mc_pack_pnhwc(dy)")

    for L in reversed(plan.layers):
        conv = L.conv
        O, C, k = L.O, L.C, L.k
        mask_ptr = _masked(conv)
        if L.is_head:
            dz_ptr, ld_dz = dzh.data_ptr(), ld_h
            # bias gradient = column sums of dY; computed in fp32 from dy itself (tiny)
            grads[id(conv.bias)] = reduce_async(dy.sum(dim=(0, 2, 3)))
        elif L.fused_pool:
            st = sv.stats[L.ind]
            dp_name = 'd' + L.pooled.name
            if dp_name not in written:
                raise RuntimeError("internal: pooled gradient of block %d was never produced" % L.ind)
            if before_bn is not None:
                before_bn(L, bufs)
            dz = bufs['dz%d' % L.ind]
            dgb = torch.empty(2, O, device=dev)
            bn = L.bn
            _lib.check(lib.mc_bn_pool_backward(bufs[L.z.name].data_ptr(), L.z.ld, bufs[dp_name].data_ptr(), L.pooled.ld, B,
                                               L.H, L.W, O, st[2].data_ptr(), st[3].data_ptr(), st[4].data_ptr(),
                                               st[5].data_ptr(), bn.weight.data_ptr(), bn.bias.data_ptr(), L.leaky,
                                               dgb[0].data_ptr(), dgb[1].data_ptr(), dz.data_ptr(), L.z.ld, s),
                       "mc_bn_pool_backward")
            reduce_async(dgb)
            grads[id(bn.bias)] = dgb[0]
            grads[id(bn.weight)] = dgb[1]
            dz_ptr, ld_dz = dz.data_ptr(), L.z.ld
        else:
            st = sv.stats[L.ind]
            a = L.act
            da_name = 'd' + a.name
            if L.pool:
                dp = bufs['d' + L.pooled.name]
                if ('d' + L.pooled.name) not in written:
                    raise RuntimeError("internal: pooled gradient of block %d was never produced" % L.ind)
                _lib.check(lib.mc_maxpool2x2_backward(bufs[a.name].data_ptr(), a.ld, dp.data_ptr(), L.pooled.ld, B, L.H,
                                                      L.W, O, bufs[da_name].data_ptr(), a.ld,
                                                      1 if da_name in written else 0, s), "mc_maxpool2x2_backward")
                written.add(da_name)
            if da_name not in written:
                raise RuntimeError("internal: gradient of block %d was never produced" % L.ind)
            if before_bn is not None:
                before_bn(L, bufs)
            dz = bufs['dz%d' % L.ind]
            dgb = torch.empty(2, O, device=dev)
            bn = L.bn
            _lib.check(lib.mc_bn_backward(bufs[L.z.name].data_ptr(), L.z.ld, bufs[da_name].data_ptr(), a.ld, a.ch_off,
                                          int(L.reorg), B, L.H, L.W, O, st[4].data_ptr(), st[5].data_ptr(),
                                          bn.weight.data_ptr(), bn.bias.data_ptr(), L.leaky, dgb[0].data_ptr(),
                                          dgb[1].data_ptr(), dz.data_ptr(), L.z.ld, s), "mc_bn_backward")
            reduce_async(dgb)
            grads[id(bn.bias)] = dgb[0]
            grads[id(bn.weight)] = dgb[1]
            dz_ptr, ld_dz = dz.data_ptr(), L.z.ld
        # ---- weight gradient
        dw = torch.empty_like(conv.weight.data)
        if L.src is None:
            # image layer: bf16 im2col rows in the workspace + the 1x1 tcgen05 weight gradient over them
            nbytes = lib.mc_workspace_bytes_conv_wgrad_first(B, L.H, L.W, C, O)
            ws = _workspace(dev, nbytes) if nbytes else None
            _lib.check(lib.mc_conv_wgrad_first(sv.x.data_ptr(), dz_ptr, ld_dz, B, L.H, L.W, C, O, mask_ptr, dw.data_ptr(),
                                               ws.data_ptr() if ws is not None else None, nbytes, s),
                       "mc_conv_wgrad_first")
        else:
            src = L.src
            nbytes = lib.mc_workspace_bytes_conv_wgrad(B, L.H, L.W, C, O, k)
            ws = _workspace(dev, nbytes)
            _lib.check(lib.mc_conv_wgrad(bufs[src.name].data_ptr() + 2 * src.ch_off, src.ld, C, dz_ptr, ld_dz, O, B, L.H,
                                         L.W, k, mask_ptr, dw.data_ptr(), 0, ws.data_ptr(), nbytes, s), "mc_conv_wgrad")
        grads[id(conv.weight)] = reduce_async(dw)
        # ---- data gradient: the same tcgen05 conv kernel on the flipped / transposed filter
        if L.src is not None:
            src = L.src
            dname = 'd' + src.name
            if dname in written:
                raise NotImplementedError("two convolutions consume the same activation slice (block %d)" % L.ind)
            kb = _kblk(O, k)
            Cpad, Ko = _round_up(C, 16), _round_up(O, kb)
            wpack = torch.empty(Cpad, k * k * Ko, dtype=torch.bfloat16, device=dev)
            _lib.check(lib.mc_pack_conv_weights_dgrad(conv.weight.data_ptr(), mask_ptr, O, C, k, wpack.data_ptr(), Cpad, Ko,
                                                      s), "mc_pack_conv_weights_dgrad")
            ones = plan.const(dev, 1.0, Cpad)
            zeros = plan.const(dev, 0.0, Cpad)
            d = _conv_desc(dz_ptr, wpack.data_ptr(), ones.data_ptr(), zeros.data_ptr(), bufs[dname].data_ptr(), B, L.H, L.W,
                           O, ld_dz, C, Cpad, k, 0, _lib.MC_EPI_PNHWC, src.ld, src.ch_off, kb, plan, dev)
            _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "dgrad (block %d)" % L.ind)
            written.add(dname)
    for work, t in pending:  # the current stream waits for NCCL; gradients become the mean over the replicas
        work.wait()
        t.div_(plan.dp_world)
    sv.consumed = True  # the buffer set may serve the next forward
    return [grads[id(p)] for p in plan.parameters()]


class _DarknetTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, plan, needs_backward, *params):
        y, sv = _forward(plan, x, needs_backward=needs_backward)
        ctx.plan, ctx.sv = plan, sv
        return y

    @staticmethod
    def backward(ctx, dy):
        plan, sv = ctx.plan, ctx.sv
        if sv.consumed:
            raise RuntimeError("Darknet (training): backward called twice on the same forward (retain_graph is not "
                               "supported: the saved activations are recycled after the first backward)")
        with torch.cuda.device(dy.device):
            g = _backward(plan, sv, dy.contiguous().float())
        return (None, None, None) + tuple(g)


def darknet_train_forward(model, x):
    """``Darknet.forward`` in training mode (src/nets.py:720-774 with model.train(); src/train.py:221-224)."""
    _lib.require_cuda(x, "Darknet.forward (training)")
    if x.dim() != 4:
        raise ValueError("expected [B,3,H,W] input")
    plan = model.__dict__.get('_b200_train_plan')
    if plan is None:
        plan = model.__dict__['_b200_train_plan'] = TrainPlan(model)
    params = plan.parameters()
    for p in params:
        _lib.require_cuda(p, "Darknet.forward (training)")
        if p.dtype != torch.float32 or not p.is_contiguous():
            raise TypeError("training path expects contiguous float32 parameters")
    x = x.detach().float().contiguous()
    # under no_grad (or with every parameter frozen) autograd records nothing: the forward must not claim a buffer set
    needs_backward = torch.is_grad_enabled() and any(p.requires_grad for p in params)
    with torch.cuda.device(x.device):
        return _DarknetTrainFn.apply(x, plan, needs_backward, *params)

"""B200 forward engine behind ``Darknet.forward`` (reference: src/nets.py:720-774 walks nn.Modules; here the graph is
compiled once into a list of libmcb200 kernel launches).

Compile step (host, once per weight/mask version):
  * BatchNorm (eval) is folded into a per-channel fp32 (scale, shift) applied in the conv epilogue
    (nn.BatchNorm2d eps=1e-5, src/nets.py:802); leaky-ReLU(0.1) (:809) is fused in the same epilogue.
  * conv weights (already multiplied by their mask — MaskedConv2d.forward, layers.py:59) are packed to bf16
    [Npad, taps*Kc] K-major for the TMA/tcgen05 implicit GEMM.
  * route/concat (:735-746) and Reorg (:648-667) become store addressing: conv20 and conv21 write disjoint channel
    slices of one buffer; conv21's epilogue performs the space-to-depth shuffle.
  * "physical shrink": a filter whose masked weights are all zero is removed from its layer and from every consumer's
    input channels.  Its output is the constant leaky(shift[o]); when that constant is non-zero it is folded into the
    consumers through ONE extra "ones" channel (value 1 inside the image, 0 in the padding, so border taps are
    handled exactly).  With the reference's default BN statistics the constant is 0 and nothing is added.

Activation layout between layers is PNHWC bf16 (include/mcb200.h).  There is no PyTorch/CPU fallback: a missing
library, a CPU tensor or an unsupported cfg raises.
"""
import ctypes
import weakref

import torch
import torch.nn as nn

from . import _lib


def _round_up(x, m):
    return (x + m - 1) // m * m


def _pitch(n):
    """Row pitch (channels) of a PNHWC activation with n physical channels.  TMA takes its fast path only for boxes that
    lie wholly inside the tensor, and a consumer's k-block is 32 (<= 32 channels) or 64 wide — so the pitch is rounded up
    to that width where it costs little (<= 32 channels, or <= 25 % growth) and the whole pitch is exposed to the
    consumer's tensor map (mc_conv_desc.in_cols).  The extra columns are never written: they stay the zeros the buffer was
    created with.  <= 16 channels keep the 8/16 pitch the im2col kernel expects."""
    ld = _round_up(n, 8)
    if n <= 16:
        return ld
    if n <= 32:
        return 32
    full = _round_up(n, 64)
    return full if full * 4 <= ld * 5 else ld


def _c_floats(t):
    """host float array handed to libmcb200 by pointer (kernel-parameter weights of csrc/conv_thin.cu)."""
    vals = t.flatten().tolist()
    return (ctypes.c_float * len(vals))(*vals)


def _thin_host_weights(wd, sc, sh, ct, nt):
    """mc_conv_thin_fwd's weight layout [(tap*ct + c)*nt + n] from the gathered fp32 [n, c, k, k] weights, rounded to bf16
    (the operand precision of the tensor-core layers), zero padded; scale/shift padded to nt."""
    n, c, k, _ = wd.shape
    wt = torch.zeros(k * k, ct, nt)
    wt[:, :c, :n] = wd.to(torch.bfloat16).float().permute(2, 3, 1, 0).reshape(k * k, c, n).cpu()
    sct = torch.zeros(nt)
    sht = torch.zeros(nt)
    sct[:n] = sc.float().cpu()
    sht[:n] = sh.float().cpu()
    return _c_floats(wt), _c_floats(sct), _c_floats(sht)


class _TensorRef(object):
    """A logical activation: where it lives and how its physical channels map to the original channel space."""

    def __init__(self, buf_id, H, W, c_orig, colsrc, const, ch_off=0):
        self.buf_id = buf_id      # index into the buffer table
        self.H, self.W = H, W
        self.c_orig = c_orig      # channel count of the un-shrunk tensor
        self.colsrc = colsrc      # list[int], len = physical channels: orig channel, -1 unused, -2 the ones channel
        self.const = const        # float32 cpu tensor [c_orig]: value of removed channels (0 where kept)
        self.ch_off = ch_off      # channel offset inside the buffer

    @property
    def c_phys(self):
        return len(self.colsrc)


class _Buf(object):
    def __init__(self, H, W, ld, zero_init=False, fp32_nchw_channels=0):
        self.H, self.W, self.ld = H, W, ld
        self.zero_init = zero_init
        self.dead = False  # True: its producer was fused into the consumer (never allocated)
        self.fp32_nchw_channels = fp32_nchw_channels  # >0: this is the fp32 NCHW network output


class CompiledDarknet(object):
    def __init__(self, model, shrink=True):
        self.lib = _lib.load()
        params = list(model.parameters())
        if not params:
            raise RuntimeError("Darknet has no parameters")
        self.device = params[0].device
        _lib.require_cuda(params[0], "Darknet.forward")
        with torch.cuda.device(self.device):
            if self.lib.mc_device_ok() != 1:
                raise RuntimeError("Darknet.forward: " + self.lib.mc_last_error_string().decode())
        self.shrink = bool(shrink)
        # CUDA-core kernel for the degenerate layers of a shrunk net (csrc/conv_thin.cu): 0 off, 1 on, 2 on + the 1x1 layer
        # behind a thin 3x3 layer applied in the same kernel
        self.use_thin = int(getattr(model, 'b200_thin', 2))
        self.bufs = []       # list[_Buf] (shapes depend on input H, W: compiled for the cfg's width/height lazily)
        self.ops = []        # list of dict
        self.block_out = {}  # models index -> _TensorRef
        self.flops_per_image = 0  # algorithmic (unpadded) conv FLOPs of the compiled (possibly shrunk) network
        self._alloc = {}     # (B, H, W) -> list of tensors
        self._graphs = {}    # (shape, input address, stream) -> (CUDAGraph, static output, input)
        self._graph_seen = {}
        self.use_graph = True
        self.in_hw = None
        self._compile(model)
        self._chain_runs = self._chain_runs_of(self.ops)
        self._items = {}     # (B, H, W) -> launch list (ops, and one entry per chained run)
        self._last_items = None

    # ------------------------------------------------------------------------------------------------ compile
    def _new_buf(self, H, W, ld, **kw):
        self.bufs.append(_Buf(H, W, ld, **kw))
        return len(self.bufs) - 1

    def _compile(self, model):
        blocks = model.blocks
        H, W = model.height, model.width
        if H % 32 or W % 32:
            raise NotImplementedError("input size must be a multiple of 32 (cfg has %dx%d)" % (W, H))
        self.in_hw = (H, W)
        # which block outputs feed a 2-input route (concat)?  producer index -> (route index, slot)
        cat_of = {}
        ind = -2
        for block in blocks:
            ind += 1
            if block['type'] == 'route':
                layers = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                if len(layers) == 2:
                    cat_of[layers[0]] = (ind, 0)
                    cat_of[layers[1]] = (ind, 1)
                elif len(layers) != 1:
                    raise NotImplementedError("route with %d inputs" % len(layers))
        n_models = len(model.models)
        last_conv = max(i for i, b in enumerate(blocks[1:]) if b['type'] == 'convolutional')

        cur = None  # _TensorRef of the running activation; None = the fp32 NCHW input image
        cur_hw = (H, W)
        cat_state = {}  # route index -> dict(buf_id, parts)
        ind = -2
        skip_next_pool = False
        for bi, block in enumerate(blocks):
            ind += 1
            btype = block['type']
            if btype == 'net':
                in_ch = int(block['channels'])
                continue
            if btype == 'convolutional':
                seq = model.models[ind]
                conv = seq[0]
                bn = seq[1] if int(block['batch_normalize']) else None
                act = block['activation']
                if act not in ('leaky', 'linear'):
                    raise NotImplementedError("activation '%s'" % act)
                k = conv.kernel_size[0]
                if conv.kernel_size != (k, k) or k not in (1, 3) or conv.stride != (1, 1) or \
                        conv.padding != ((k - 1) // 2, (k - 1) // 2) or conv.groups != 1 or conv.dilation != (1, 1):
                    raise NotImplementedError("conv %s is outside the B200 path (need k in {1,3}, stride 1, 'same' "
                                              "padding)" % (conv,))
                is_head = (ind == last_conv)
                nxt = blocks[bi + 1] if bi + 1 < len(blocks) else None
                nxt_is_pool = nxt is not None and nxt['type'] == 'maxpool' and int(nxt['size']) == 2 and \
                    int(nxt['stride']) == 2
                nxt_is_reorg = nxt is not None and nxt['type'] == 'reorg' and int(nxt['stride']) == 2
                cur, fused = self._compile_conv(conv, bn, act == 'leaky', cur, cur_hw, in_ch, is_head, ind, cat_of,
                                                cat_state, nxt_is_pool, nxt_is_reorg)
                self.block_out[ind] = cur
                if fused == 'pool':
                    skip_next_pool = True
                    cur_hw = (cur.H, cur.W)
                elif fused == 'reorg':
                    skip_next_pool = True  # the reorg block is already applied
                    cur_hw = (cur.H, cur.W)
            elif btype == 'maxpool':
                if skip_next_pool:
                    skip_next_pool = False
                    self.block_out[ind] = cur
                    continue
                if int(block['size']) != 2 or int(block['stride']) != 2:
                    raise NotImplementedError("maxpool size=%s stride=%s" % (block['size'], block['stride']))
                src = cur
                Ho, Wo = src.H // 2, src.W // 2
                ld = _pitch(src.c_phys)
                bid = self._new_buf(Ho, Wo, ld, zero_init=True)
                self.ops.append(dict(kind='pool', src=src, dst_buf=bid, C=src.c_phys, name='pool@%d' % ind))
                cur = _TensorRef(bid, Ho, Wo, src.c_orig, list(src.colsrc), src.const)
                cur_hw = (Ho, Wo)
                self.block_out[ind] = cur
            elif btype == 'reorg':
                if skip_next_pool:
                    skip_next_pool = False
                    self.block_out[ind] = cur
                    continue
                raise NotImplementedError("reorg that does not directly follow a convolution")
            elif btype == 'route':
                layers = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                if len(layers) == 1:
                    cur = self.block_out[layers[0]]
                else:
                    st = cat_state.get(ind)
                    if st is None or len(st['parts']) != 2:
                        raise NotImplementedError("concat inputs must both be produced by convolutions (cfg block %d)" % bi)
                    p0, p1 = st['parts'][0], st['parts'][1]
                    colsrc = list(p0.colsrc) + [-1] * (p1.ch_off - p0.c_phys)  # alignment gap: zero, never written
                    have_ones = -2 in colsrc
                    for c in p1.colsrc:
                        if c >= 0:
                            colsrc.append(c + p0.c_orig)
                        elif c == -2 and not have_ones:
                            colsrc.append(-2)
                            have_ones = True
                        else:
                            colsrc.append(-1)
                    cur = _TensorRef(st['buf_id'], p0.H, p0.W, p0.c_orig + p1.c_orig, colsrc,
                                     torch.cat([p0.const, p1.const]))
                cur_hw = (cur.H, cur.W)
                self.block_out[ind] = cur
            elif btype == 'region':
                continue
            else:
                raise NotImplementedError("cfg block type '%s'" % btype)
        self.out_ref = cur
        del n_models
        if self.use_thin >= 2:
            routed = set()
            ind = -2
            for block in blocks:
                ind += 1
                if block['type'] == 'route':
                    routed.update(int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(','))
            self._fuse_thin_pairs(routed)

    def _chain_runs_of(self, ops):
        """Runs of 3x3 conv ops in which each reads the previous one's output (mc_conv_chain_fwd runs them as one launch;
        which parts it takes depends on the batch size and is asked at run time, _launch_items).  An op between two
        members may sit in a run when its input is produced before the run and no earlier member reads its output: it is
        launched in front of the run (YOLOv2's reorg branch conv21 writes its slice of the concat buffer that the run's
        last member reads).  self.ops keeps one entry per layer, in layer order."""
        def chainable(op):
            return op['kind'] == 'conv' and op['ksize'] == 3 and op['epi'] == _lib.MC_EPI_PNHWC

        runs, i = [], 0
        while i < len(ops):
            if not chainable(ops[i]):
                i += 1
                continue
            run, j, last = [ops[i]], i + 1, i
            while j < len(ops) and len(run) < 4:
                nxt = ops[j]
                if chainable(nxt) and nxt['src'].buf_id == run[-1]['dst_buf'] and nxt['src'].ch_off == 0:
                    run.append(nxt)
                    last = j
                elif nxt.get('src') is None or 'dst_buf' not in nxt or \
                        nxt['src'].buf_id in {m['dst_buf'] for m in run} or \
                        nxt['dst_buf'] in {m['src'].buf_id for m in run}:
                    break
                j += 1
            if len(run) >= 2:
                runs.append(run)
            i = last + 1
        return runs

    def _fuse_thin_pairs(self, routed):
        """thin 3x3 layer -> 1x1 layer with <= 8 outputs: the second layer is applied by the same thread to the bf16-rounded
        activations (csrc/conv_thin.cu, N2T > 0); the intermediate tensor is never stored and its block output is no
        longer available to block_activation()."""
        i = 0
        while i + 1 < len(self.ops):
            a, b = self.ops[i], self.ops[i + 1]
            i += 1
            if a['kind'] != 'thin' or a['pool'] or a['ksize'] != 3 or a['N2'] or a['ind'] in routed:
                continue
            if b['kind'] == 'conv':
                if b['ksize'] != 1 or not b.get('plain') or b['epi'] != _lib.MC_EPI_PNHWC or b['ch_off'] != 0:
                    continue
                b_ld = b['ldc']
            elif b['kind'] == 'thin':
                if b['ksize'] != 1 or b['N2']:
                    continue
                b_ld = b['ld']
            else:
                continue
            if b['src'].buf_id != a['dst_buf'] or b['src'].ch_off != 0 or b['Cin'] != a['N']:
                continue
            ct, nt, n2t = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
            if self.lib.mc_conv_thin_geometry(3, a['Cin'], a['N'], 0, b['N'], ctypes.byref(ct), ctypes.byref(nt),
                                              ctypes.byref(n2t)) != 1:
                continue
            ct, nt, n2t = ct.value, nt.value, n2t.value
            if self.bufs[a['src'].buf_id].ld < ct or b_ld < _round_up(n2t, 8):
                continue
            # first layer's weights re-padded to the fused instance's NT; second layer's from its packed bf16 matrix
            taps, ct0, nt0 = 9, a['hw_shape'][1], a['hw_shape'][2]
            w1 = torch.tensor(list(a['hw'])).view(taps, ct0, nt0)
            w1p = torch.zeros(taps, ct, nt)
            w1p[:, :min(ct, ct0), :min(nt, nt0)] = w1[:, :min(ct, ct0), :min(nt, nt0)]
            sc1 = torch.zeros(nt)
            sh1 = torch.zeros(nt)
            sc1[:a['N']] = torch.tensor(list(a['hsc']))[:a['N']]
            sh1[:a['N']] = torch.tensor(list(a['hsh']))[:a['N']]
            w2 = torch.zeros(nt, n2t)
            sc2 = torch.zeros(n2t)
            sh2 = torch.zeros(n2t)
            if b['kind'] == 'conv':
                w2[:a['N'], :b['N']] = b['wpack'][:b['N'], :a['N']].float().t().cpu()
                sc2[:b['N']] = b['scale'][:b['N']].cpu()
                sh2[:b['N']] = b['shift'][:b['N']].cpu()
            else:
                wb = torch.tensor(list(b['hw'])).view(b['hw_shape'])[0]  # [ct_b, nt_b] = w2[o, c] at [c, o]
                w2[:a['N'], :b['N']] = wb[:a['N'], :b['N']]
                sc2[:b['N']] = torch.tensor(list(b['hsc']))[:b['N']]
                sh2[:b['N']] = torch.tensor(list(b['hsh']))[:b['N']]
            fused = dict(a)
            fused.update(hw=_c_floats(w1p), hsc=_c_floats(sc1), hsh=_c_floats(sh1), hw_shape=(taps, ct, nt),
                         hw2=_c_floats(w2), hsc2=_c_floats(sc2), hsh2=_c_floats(sh2), N2=b['N'], leaky2=b['leaky'],
                         dst_buf=b['dst_buf'], ld=b_ld, name='thin@%d+%d' % (a['ind'], b['ind']),
                         flops_per_image=a['flops_per_image'] + b['flops_per_image'], fused_n1=a['N'])
            self.bufs[a['dst_buf']].dead = True  # the intermediate activation no longer exists
            self.block_out.pop(a['ind'], None)
            self.ops[i - 1:i + 1] = [fused]

    def _compile_conv(self, conv, bn, leaky, src, src_hw, in_ch, is_head, ind, cat_of, cat_state, nxt_is_pool,
                      nxt_is_reorg):
        dev = self.device
        H, W = src_hw
        w = conv.weight.data.float()
        if getattr(conv, 'mask_flag', False):
            w = w * conv.mask.to(dev)
        O, Corig = w.shape[0], w.shape[1]
        k = w.shape[2]
        taps = k * k
        # folded BN / bias
        if bn is not None:
            scale = bn.weight.data.float() / torch.sqrt(bn.running_var.float() + bn.eps)
            shift = bn.bias.data.float() - bn.running_mean.float() * scale
        else:
            scale = torch.ones(O, device=dev)
            shift = conv.bias.data.float() if conv.bias is not None else torch.zeros(O, device=dev)
        # ---- input channel map
        if src is None:
            in_colsrc, in_const, c_in_orig = list(range(in_ch)), torch.zeros(in_ch), in_ch
        else:
            in_colsrc, in_const, c_in_orig = src.colsrc, src.const, src.c_orig
        if c_in_orig != Corig:
            raise RuntimeError("conv at block %d expects %d input channels, graph provides %d" % (ind, Corig, c_in_orig))
        # ---- output channel set
        if self.shrink and not is_head:
            alive = (w.abs().amax(dim=(1, 2, 3)) > 0)
            if not bool(alive.any()):
                alive[0] = True  # keep the layer non-empty
            keep = torch.nonzero(alive).flatten()
        else:
            keep = torch.arange(O, device=dev)
        n_keep = int(keep.numel())
        const_out = torch.zeros(O)
        need_ones_out = False
        if n_keep < O:
            dead = torch.ones(O, dtype=torch.bool, device=dev)
            dead[keep] = False
            cval = shift.clone()
            if leaky:
                cval = torch.where(cval > 0, cval, 0.1 * cval)
            cval = torch.where(dead, cval, torch.zeros_like(cval))
            const_out = cval.cpu()
            need_ones_out = bool((const_out != 0).any())
        # a ones channel is also forwarded when the input has one and downstream may need it? No: each producer
        # decides from its own removed filters only.
        out_colsrc = [int(i) for i in keep.tolist()] + ([-2] if need_ones_out else [])
        n_phys = len(out_colsrc)
        # ---- packed weights in the PHYSICAL input-channel order
        in_has_const = bool((in_const != 0).any())
        w_aug = w
        if in_has_const:
            if -2 not in in_colsrc:
                raise RuntimeError("internal: constant input channels without a ones channel")
            w1 = torch.einsum('ocrs,c->ors', w, in_const.to(dev))  # combined weight of all removed channels
            w_aug = torch.cat([w, w1[:, None]], dim=1)
        cidx = [(c if c >= 0 else (Corig if (c == -2 and in_has_const) else -1)) for c in in_colsrc]
        c_phys_in = len(cidx)
        op_flops = 2 * H * W * n_keep * sum(1 for c in in_colsrc if c >= 0) * taps  # algorithmic, unpadded
        self.flops_per_image += op_flops
        o_list = [int(i) for i in keep.tolist()] + ([-1] if need_ones_out else [])
        sc = torch.cat([scale[keep], torch.zeros(1, device=dev)]) if need_ones_out else scale[keep]
        sh = torch.cat([shift[keep], torch.ones(1, device=dev)]) if need_ones_out else shift[keep]
        Npad = _round_up(n_phys, 16)
        scale_p = torch.zeros(Npad, device=dev)
        shift_p = torch.zeros(Npad, device=dev)
        scale_p[:n_phys] = sc
        shift_p[:n_phys] = sh

        # ---- thin layers.  3x3 with <= 16 input channels (or the fp32 image): tensor cores with the im2col tile built
        #      in shared memory, pool fused (csrc/conv_im2col_tc.cu).  Other first layers: direct CUDA-core kernel.
        plain_dst = (ind not in cat_of) and not (nxt_is_reorg and (ind + 1) in cat_of) and not is_head
        first = src is None
        pool = 1 if nxt_is_pool else 0

        def gathered_fp32():
            rows = torch.tensor([o if o >= 0 else 0 for o in o_list], dtype=torch.long, device=dev)
            cols = torch.tensor([c if c >= 0 else 0 for c in cidx], dtype=torch.long, device=dev)
            wd = w_aug[rows][:, cols].clone()  # [n_phys, c_phys_in, k, k]
            wd[torch.tensor([o < 0 for o in o_list], device=dev)] = 0
            wd[:, torch.tensor([c < 0 for c in cidx], device=dev)] = 0
            return wd

        # ---- degenerate layers (a few hundred multiply-adds per pixel): CUDA-core kernel with the weights as kernel
        #      parameters (csrc/conv_thin.cu).  Measured on B200 at batch 64 (tools/bench_layers.py): 4 -> 1 + pool at 208^2,
        #      1 -> 17 at 104^2, 17 -> 4 (1x1) and 4 -> 11 + pool at 104^2 took 37 / 28 / 31 / 25 us on the tensor-core thin
        #      kernels (per-tile latency chain), bound by reading the input once here.
        if self.use_thin and plain_dst and not first and src.ch_off == 0 and (not pool or (H % 2 == 0 and W % 2 == 0)):
            ct, nt = ctypes.c_int(), ctypes.c_int()
            src_ld = self.bufs[src.buf_id].ld
            if self.lib.mc_conv_thin_geometry(k, c_phys_in, n_phys, pool, 0, ctypes.byref(ct), ctypes.byref(nt), None) == 1 \
                    and src_ld >= ct.value and _pitch(n_phys) >= _round_up(nt.value, 8):
                ct, nt = ct.value, nt.value
                Ho, Wo = (H // 2, W // 2) if pool else (H, W)
                ld = _pitch(n_phys)
                bid = self._new_buf(Ho, Wo, ld, zero_init=True)  # pad line/column stay zero: the kernel never writes them
                hw, hsc, hsh = _thin_host_weights(gathered_fp32(), sc, sh, ct, nt)
                self.ops.append(dict(kind='thin', src=src, hw=hw, hsc=hsc, hsh=hsh, hw_shape=(taps, ct, nt), dst_buf=bid, N=n_phys, Cin=c_phys_in,
                                     H=H, W=W, ld=ld, pool=pool, ksize=k, leaky=int(leaky), N2=0, leaky2=0, ind=ind,
                                     name='thin%s@%d' % ('+pool' if pool else '', ind), flops_per_image=op_flops))
                return _TensorRef(bid, Ho, Wo, O, out_colsrc, const_out), ('pool' if pool else None)

        # ---- no-build window kernel (csrc/conv_window.cu): the image layer with its pool, and <= 8-channel PNHWC inputs
        win_kind = None
        if plain_dst and k == 3 and (not pool or (H % 2 == 0 and W % 2 == 0)):
            # Measured on B200 (batch 64): the window kernel wins for the narrow image layer
            # (3 -> <= 8 filters: 92 -> 68 us) and for un-pooled <= 8-channel layers (37 -> 31 us); with 32 filters its
            # epilogue (128 accumulator columns per pool window) costs what the im2col build saved (194 vs 192 us), and
            # pooled pitch-8 layers lose to the pool-window GEMM of conv_im2col_tc.cu (49 vs 39 us).
            if first and pool and c_phys_in <= 3 and n_phys <= 8:
                win_kind = 1  # (2 when the caller hands in uint8 pixels: decided per call)
            elif not first and not pool and src.ch_off == 0 and self.bufs[src.buf_id].ld == 8 and c_phys_in <= 8:
                win_kind = 0
        if win_kind is not None and self.lib.mc_conv_window_supported(c_phys_in, win_kind, n_phys, pool) == 1:
            npos, nb, kcols = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
            _lib.check(self.lib.mc_conv_window_geometry(c_phys_in, win_kind, n_phys, pool, ctypes.byref(npos),
                                                        ctypes.byref(nb), ctypes.byref(kcols)), "mc_conv_window_geometry")
            npos, nb, kcols = npos.value, nb.value, kcols.value
            wd = gathered_fp32().permute(0, 2, 3, 1)  # [n, r, s, c]
            if win_kind == 0:
                wk = torch.zeros(nb, 10, 8, device=dev)
                wk[:n_phys, :9, :c_phys_in] = wd.reshape(n_phys, 9, c_phys_in)
            else:
                wk = torch.zeros(nb, 4, 4, 4, device=dev)
                for dy in range(2):
                    for dx in range(2):
                        r0 = (dy * 2 + dx) * npos
                        wk[r0:r0 + n_phys, dy:dy + 3, dx:dx + 3, :c_phys_in] = wd
            wk = wk.reshape(nb, kcols).to(torch.bfloat16).contiguous()
            Ho, Wo = (H // 2, W // 2) if pool else (H, W)
            ld = _pitch(n_phys)
            bid = self._new_buf(Ho, Wo, ld, zero_init=True)  # pad line/column stay zero: the kernel never writes them
            n_sc = max(_round_up(npos, 16), 16)
            sc2 = torch.zeros(n_sc, device=dev)
            sh2 = torch.zeros(n_sc, device=dev)
            sc2[:n_phys] = sc
            sh2[:n_phys] = sh
            self.ops.append(dict(kind='window', src=src, w=wk, scale=sc2, shift=sh2, dst_buf=bid, N=n_phys, Cin=c_phys_in,
                                 H=H, W=W, ld=ld, pool=pool, leaky=int(leaky), in_kind=win_kind,
                                 name='window%s@%d' % ('+pool' if pool else '', ind), flops_per_image=op_flops))
            return _TensorRef(bid, Ho, Wo, O, out_colsrc, const_out), ('pool' if pool else None)

        src_ok = first or (src.ch_off == 0 and self.bufs[src.buf_id].ld == (8 if c_phys_in <= 8 else 16))
        if plain_dst and k == 3 and src_ok and (H % 2 == 0 and W % 2 == 0 or not pool) and \
                self.lib.mc_conv_im2col_supported(c_phys_in, 1 if first else 0, n_phys, pool) == 1:
            cl, npos, nb, kpad = (ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int())
            _lib.check(self.lib.mc_conv_im2col_geometry(c_phys_in, 1 if first else 0, n_phys, pool, ctypes.byref(cl),
                                                        ctypes.byref(npos), ctypes.byref(nb), ctypes.byref(kpad)),
                       "mc_conv_im2col_geometry")
            cl, npos, nb, kpad = cl.value, npos.value, nb.value, kpad.value
            wd = gathered_fp32().permute(0, 2, 3, 1)  # [n, r, s, c]
            nb_pad = _round_up(nb, 16)
            if pool:
                wexp = torch.zeros(nb_pad, 4, 4, cl, device=dev)
                for dy in range(2):
                    for dx in range(2):
                        r0 = (dy * 2 + dx) * npos
                        wexp[r0:r0 + n_phys, dy:dy + 3, dx:dx + 3, :c_phys_in] = wd
                wexp = wexp.reshape(nb_pad, 16 * cl)
            else:
                wexp = torch.zeros(nb_pad, 3, 3, cl, device=dev)
                wexp[:n_phys, :, :, :c_phys_in] = wd
                wexp = wexp.reshape(nb_pad, 9 * cl)
            wfull = torch.zeros(nb_pad, kpad, device=dev)
            wfull[:, :wexp.shape[1]] = wexp
            Ho, Wo = (H // 2, W // 2) if pool else (H, W)
            ld = _pitch(n_phys)
            bid = self._new_buf(Ho, Wo, ld, zero_init=True)  # pad line/column stay zero: the kernel never writes them
            n_sc = max(_round_up(npos, 16), 16)
            sc2 = torch.zeros(n_sc, device=dev)
            sh2 = torch.zeros(n_sc, device=dev)
            sc2[:n_phys] = sc
            sh2[:n_phys] = sh
            self.ops.append(dict(kind='im2col', src=src, w=wfull.to(torch.bfloat16).contiguous(), scale=sc2, shift=sh2,
                                 dst_buf=bid, N=n_phys, Cin=c_phys_in, H=H, W=W, ld=ld, pool=pool, leaky=int(leaky),
                                 name='im2col%s@%d' % ('+pool' if pool else '', ind), flops_per_image=op_flops))
            return _TensorRef(bid, Ho, Wo, O, out_colsrc, const_out), ('pool' if pool else None)
        if first and plain_dst and self.lib.mc_conv_direct_supported(c_phys_in, n_phys, k) == 1:
            wd = gathered_fp32().reshape(n_phys, c_phys_in, taps)
            Ho, Wo = (H // 2, W // 2) if pool else (H, W)
            ld = _pitch(n_phys)
            bid = self._new_buf(Ho, Wo, ld, zero_init=True)
            self.ops.append(dict(kind='direct', src=src, w=wd.contiguous(), scale=scale_p, shift=shift_p, dst_buf=bid,
                                 N=n_phys, Cin=c_phys_in, H=H, W=W, ld=ld, pool=pool, ksize=k, leaky=int(leaky),
                                 name='direct%s@%d' % ('+pool' if pool else '', ind), flops_per_image=op_flops))
            return _TensorRef(bid, Ho, Wo, O, out_colsrc, const_out), ('pool' if pool else None)
        if src is None:
            # generic first layer: pack the image to PNHWC (C=3 -> pitch 8) and run the tensor-core kernel
            bid_in = self._new_buf(H, W, 8)
            self.ops.append(dict(kind='pack_input', dst_buf=bid_in, C=in_ch, H=H, W=W, name='pack_input'))
            src = _TensorRef(bid_in, H, W, in_ch, list(range(in_ch)), torch.zeros(in_ch))

        # k-block of 32 (64-byte swizzle) where it halves K (<= 32 input channels).  Measured on B200: TMA cost follows the
        # box AREA, not the valid channels, so a 64-wide box (shared activation box) is slower than
        # 32-wide boxes for <= 32 channels (dense conv2: 402 us vs 524 us; shrunk conv8: 33 us vs 39 us); and for
        # 69 -> 96 instead of 128 columns the extra pipeline steps cost more than the zero padding they remove.
        kblk = 32 if c_phys_in <= 32 else 64
        Kc = _round_up(c_phys_in, kblk)
        wpack = torch.empty(Npad, taps * Kc, dtype=torch.bfloat16, device=dev)
        oidx_t = torch.tensor(o_list, dtype=torch.int32, device=dev)
        cidx_t = torch.tensor(cidx, dtype=torch.int32, device=dev)
        w_src = w_aug.contiguous()
        with torch.cuda.device(dev):
            _lib.check(self.lib.mc_pack_conv_weights(w_src.data_ptr(), None, w_src.shape[0], w_src.shape[1], k,
                                                     oidx_t.data_ptr(), n_phys, cidx_t.data_ptr(), c_phys_in,
                                                     wpack.data_ptr(), Npad, Kc, _lib.stream_ptr()),
                       "mc_pack_conv_weights")
        op = dict(kind='conv', src=src, wpack=wpack, scale=scale_p, shift=shift_p, N=n_phys, Npad=Npad, ksize=k,
                  leaky=int(leaky), Cin=c_phys_in, name='conv@%d' % ind, H=H, W=W, flops_per_image=op_flops, block_k=kblk,
                  ind=ind, plain=bool(plain_dst))
        fused = None
        if is_head:
            bid = self._new_buf(H, W, 0, fp32_nchw_channels=n_phys)
            op.update(epi=_lib.MC_EPI_NCHW_F32, dst_buf=bid, ldc=0, ch_off=0)
            out = _TensorRef(bid, H, W, O, out_colsrc, const_out)
        elif nxt_is_reorg and (ind + 1) in cat_of:
            route, slot = cat_of[ind + 1]
            Ho, Wo = H // 2, W // 2
            st = cat_state.setdefault(route, dict(buf_id=None, parts={}, pending=[]))
            colsrc4 = []
            for q in range(4):
                for c in out_colsrc:
                    colsrc4.append(c + q * O if c >= 0 else (c if (c == -2 and q == 0) else -1))
            out = _TensorRef(None, Ho, Wo, 4 * O, colsrc4, const_out.repeat(4))
            op.update(epi=_lib.MC_EPI_REORG2)
            st['parts'][slot] = out
            st['pending'].append((op, slot))
            fused = 'reorg'
        elif ind in cat_of:
            route, slot = cat_of[ind]
            st = cat_state.setdefault(route, dict(buf_id=None, parts={}, pending=[]))
            out = _TensorRef(None, H, W, O, out_colsrc, const_out)
            op.update(epi=_lib.MC_EPI_PNHWC)
            st['parts'][slot] = out
            st['pending'].append((op, slot))
        else:
            ld = _pitch(n_phys)
            bid = self._new_buf(H, W, ld)
            op.update(epi=_lib.MC_EPI_PNHWC, dst_buf=bid, ldc=ld, ch_off=0)
            out = _TensorRef(bid, H, W, O, out_colsrc, const_out)
        self.ops.append(op)
        # resolve a concat once both producers are known
        for route, st in cat_state.items():
            if st['buf_id'] is None and len(st['parts']) == 2:
                p0, p1 = st['parts'][0], st['parts'][1]
                if (p0.H, p0.W) != (p1.H, p1.W):
                    raise NotImplementedError("concat of different resolutions")
                off1 = _round_up(p0.c_phys, 8)  # 16-byte aligned slice start -> vector stores in the epilogue
                ld = _pitch(off1 + p1.c_phys)
                st['buf_id'] = self._new_buf(p0.H, p0.W, ld, zero_init=True)
                for pop, slot in st['pending']:
                    pop.update(dst_buf=st['buf_id'], ldc=ld, ch_off=0 if slot == 0 else off1)
                p0.buf_id = p1.buf_id = st['buf_id']
                p1.ch_off = off1
        return out, fused

    # ------------------------------------------------------------------------------------------------ run
    def _buffers(self, B, H, W):
        key = (B, H, W)
        got = self._alloc.get(key)
        if got is not None:
            return got
        if (H, W) != self.in_hw:
            raise NotImplementedError("this plan was compiled for %dx%d inputs (cfg width/height); got %dx%d" %
                                      (self.in_hw[1], self.in_hw[0], W, H))
        tensors = []
        for b in self.bufs:
            if b.fp32_nchw_channels or b.dead:
                tensors.append(None)  # allocated per call (returned to the caller) / fused away
            else:
                # zero-initialised: pad rows/columns that no kernel writes, and the channels between a layer's physical
                # channel count and the 8-aligned pitch, must be finite zeros (0-weight x NaN garbage would poison
                # consumers that read whole 16-byte pixels)
                rows = B * (b.H + 1) * (b.W + 1)
                tensors.append(torch.zeros(rows, b.ld, dtype=torch.bfloat16, device=self.device))
        self._alloc[key] = tensors
        return tensors

    def run(self, x, events=None, detect=None, repeat=1):
        """Forward.  The launch sequence is captured into a CUDA graph the second time an input buffer (same
        device address and shape) is seen and replayed afterwards: ~25 launches per step otherwise cost more host time
        than the GPU needs for the small layers.  events: optional list; when given the eager path is used and
        (op, start_event, end_event) is appended per op (bench/profiling); with repeat > 1 every op is launched that many
        times between its two events (same inputs, same outputs), so the events' own cost — a few microseconds per pair,
        comparable to the short kernels — is amortised: interval / repeat is the kernel's device time.
        detect=(conf_thresh, only_objectness, want_cls): the head convolution runs with the region decode fused into
        its epilogue (MC_EPI_DECODE) and the call returns (boxes [B,P,8] dense slot table, cls [B,P,nc] or None)
        instead of the raw head."""
        if events is not None or not self.use_graph or not x.is_cuda or x.dtype not in (torch.float32, torch.uint8) or \
                not x.is_contiguous() or x.requires_grad:
            return self._run_eager(x, events, detect, repeat)
        # Graphs are keyed by the input ADDRESS (they read it in place).  A tensor OBJECT seen a third time gets its own
        # graph (zero-copy: a serving loop rotating over a few device buffers it keeps); any other input is copied into a
        # plan-owned static input buffer and replays that buffer's graph (33 MB for a uint8 batch of 64: ~10 us), so
        # callers that hand in a fresh tensor every step never trigger a capture or an eager step.
        base = (tuple(x.shape), torch.cuda.current_stream(x.device).cuda_stream, x.dtype, detect)
        key = base + (x.data_ptr(),)
        entry = self._graphs.get(key)
        if entry is not None and entry[2] is not x:
            # same address, another tensor object: the allocator recycled the block of a dead tensor.  Not a pinned buffer.
            entry = None
            key = None
        if entry is None:
            seen = 0
            if key is not None:
                ref = self._graph_seen.get(key)
                # only sightings of the SAME live tensor object count (a serving loop that keeps its input buffers);
                # a recycled allocation shows up as a new object at an old address and starts over
                seen = (ref[1] if ref is not None and ref[0]() is x else 0) + 1
                if len(self._graph_seen) > 4096:
                    self._graph_seen.clear()
                self._graph_seen[key] = (weakref.ref(x), seen)
            if seen >= 3 and sum(1 for k in self._graphs if k[:4] == base and k[4] != 'static') < 8:
                entry = self._capture(key, x, detect)
            else:
                skey = base + ('static',)
                entry = self._graphs.get(skey)
                if entry is None:
                    cnt = self._graph_seen.get(skey, 0) + 1
                    self._graph_seen[skey] = cnt
                    if cnt < 2:
                        return self._run_eager(x, None, detect)  # first call of this shape: eager (warms the kernels)
                    entry = self._capture(skey, torch.empty_like(x), detect)
                entry[2].copy_(x)
        entry[0].replay()
        if detect is None:
            return entry[1].clone()
        return tuple(None if t is None else t.clone() for t in entry[1])

    def _capture(self, key, x, detect):
        if len(self._graphs) >= 24:
            self._graphs.pop(next(iter(self._graphs)))
        with torch.cuda.device(self.device):
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self._run_eager(x, None, detect)
        entry = (graph, out, x)  # keep the input tensor alive: the graph reads its address
        self._graphs[key] = entry
        return entry

    def _conv_workspace(self, nbytes):
        """One scratch buffer for every conv launch of the plan (stream-K partial tiles of the CTA-pair kernel, and behind
        them the tickets and counters of chained launches; launches on a stream are ordered, and a captured graph keeps
        reading the same address).  64 KB more than asked: the chain's counters grow with the batch size, and a batch
        size first seen after a graph capture must not need a larger buffer."""
        ws = getattr(self, '_ws', None)
        if ws is None or ws.numel() < nbytes:
            if ws is not None and self._graphs:
                raise RuntimeError("internal: conv workspace grew after a CUDA graph captured its address")
            ws = self._ws = torch.zeros(nbytes + 65536, dtype=torch.uint8, device=self.device)  # (counters start at zero)
        return ws

    def supports_detect(self, model):
        """The fused decode epilogue needs the head to be the last op, all A*(5+nc) channels in one tile."""
        if not self.ops or self.ops[-1].get('epi') != _lib.MC_EPI_NCHW_F32:
            return False
        n = self.ops[-1]['N']
        return n == model.num_anchors * (5 + model.num_classes) and self.ops[-1]['Npad'] <= 256 and \
            len(model.anchors) == 2 * model.num_anchors and model.num_anchors <= 16

    def _conv_desc(self, op, bufs, B):
        """mc_conv_desc of a conv op on this call's buffers (the head's output and decode are set by the caller)"""
        s = op['src']
        sb = self.bufs[s.buf_id]
        d = _lib.mc_conv_desc()
        d.d_in = bufs[s.buf_id].data_ptr() + 2 * s.ch_off
        d.d_wpack = op['wpack'].data_ptr()
        d.d_scale = op['scale'].data_ptr()
        d.d_shift = op['shift'].data_ptr()
        if op['epi'] != _lib.MC_EPI_NCHW_F32:
            d.d_out = bufs[op['dst_buf']].data_ptr()
        d.B, d.H, d.W = B, op['H'], op['W']
        d.Cin, d.Cin_ld = op['Cin'], sb.ld
        d.in_cols = sb.ld - s.ch_off  # the rest of the row: pad channels (zero) / a neighbouring slice (finite)
        d.N, d.Npad = op['N'], op['Npad']
        d.ksize, d.leaky, d.epi_mode = op['ksize'], op['leaky'], op['epi']
        d.ldc, d.ch_off = op['ldc'], op['ch_off']
        d.block_n = op.get('block_n', 0)
        d.stages = op.get('stages', 0)
        d.block_k = op.get('block_k', 0)
        return d

    def _launch_items(self, B, H, W, bufs):
        """The launches of a forward at this input shape: self.ops, except that every maximal part of a run from
        _chain_runs_of that mc_conv_chain_fwd accepts at this batch size (its members take the CTA-pair kernel) is ONE
        entry of kind 'conv' named chain@<members>, launched in place of its first member."""
        key = (B, H, W)
        items = self._items.get(key)
        if items is not None:
            return items
        lib = self.lib
        first, skip = {}, set()
        with torch.cuda.device(self.device):
            for run in self._chain_runs:
                i = 0
                while i < len(run) - 1:
                    for j in range(len(run), i + 1, -1):
                        descs = (_lib.mc_conv_desc * (j - i))(*[self._conv_desc(m, bufs, B) for m in run[i:j]])
                        nbytes = int(lib.mc_workspace_bytes_conv_chain(descs, j - i))
                        if nbytes:
                            break
                    else:
                        i += 1
                        continue
                    members = run[i:j]
                    # the chain's words sit behind the region the stream-K tail of single launches uses
                    ws_off = int(lib.mc_workspace_bytes_conv_fwd(ctypes.byref(descs[0])))
                    ws_off = (ws_off + 255) // 256 * 256
                    k0, k1 = self.ops.index(members[0]), self.ops.index(members[-1])
                    ahead = [o for o in self.ops[k0 + 1:k1] if not any(o is m for m in members)]
                    first[id(members[0])] = ahead + [dict(kind='conv', chain=members, ws_off=ws_off, ws_bytes=nbytes,
                                                          name='chain@' + '+'.join(str(m['ind']) for m in members))]
                    skip.update(id(o) for o in self.ops[k0 + 1:k1 + 1])
                    i = j
        items = []
        for op in self.ops:
            if id(op) not in skip:
                items += first.get(id(op), [op])
        self._items[key] = items
        return items

    def _run_eager(self, x, events=None, detect=None, repeat=1):
        if x.dim() != 4:
            raise ValueError("expected [B,3,H,W] input")
        _lib.require_cuda(x, "Darknet.forward")
        if x.device != self.device:
            raise RuntimeError("input on %s, model on %s" % (x.device, self.device))
        x = x.detach()
        # uint8 images (what PIL / cv2 hand to do_detect, src/nets2_utils.py:346-352) are scaled by 1/255 inside the
        # first-layer kernel: 4x less host->device traffic than shipping the float tensor the reference builds on the CPU
        u8 = x.dtype == torch.uint8 and self.ops and self.ops[0]['kind'] in ('im2col', 'window') and \
            self.ops[0]['src'] is None
        if x.dtype == torch.uint8 and not u8:
            x = x.float().div_(255.0)
        elif x.dtype not in (torch.float32, torch.uint8):
            x = x.float()
        x = x.contiguous()
        B, _, H, W = x.shape
        lib = self.lib
        with torch.cuda.device(self.device):
            bufs = list(self._buffers(B, H, W))
            stream = _lib.stream_ptr()
            out = None
            self._prev_op = None
            items = self._launch_items(B, H, W, bufs)
            self._last_items = items
            for op in (o for o in items for _ in range(repeat if events is not None else 1)):
                kind = op['kind']
                first_rep = op is not getattr(self, '_prev_op', None)
                self._prev_op = op
                if events is not None and first_rep:
                    ev0 = torch.cuda.Event(enable_timing=True)
                    ev0.record()
                    reps_left = repeat
                if kind == 'im2col':
                    s = op['src']
                    if s is None:
                        in_ptr, nchw, cin_ld = x.data_ptr(), (2 if u8 else 1), op['Cin']
                    else:
                        in_ptr, nchw, cin_ld = bufs[s.buf_id].data_ptr(), 0, self.bufs[s.buf_id].ld
                    _lib.check(lib.mc_conv_im2col_fwd(in_ptr, nchw, op['w'].data_ptr(), op['scale'].data_ptr(),
                                                      op['shift'].data_ptr(), bufs[op['dst_buf']].data_ptr(), B,
                                                      op['H'], op['W'], op['Cin'], cin_ld, op['N'], op['ld'],
                                                      op['leaky'], op['pool'], stream), op['name'])
                elif kind == 'window':
                    s = op['src']
                    if s is None:
                        in_ptr, in_kind = x.data_ptr(), (2 if u8 else 1)
                    else:
                        in_ptr, in_kind = bufs[s.buf_id].data_ptr(), 0
                    _lib.check(lib.mc_conv_window_fwd(in_ptr, in_kind, op['w'].data_ptr(), op['scale'].data_ptr(),
                                                      op['shift'].data_ptr(), bufs[op['dst_buf']].data_ptr(), B, op['H'],
                                                      op['W'], op['Cin'], op['N'], op['ld'], op['leaky'], op['pool'],
                                                      stream), op['name'])
                elif kind == 'thin':
                    s = op['src']
                    _lib.check(lib.mc_conv_thin_fwd(bufs[s.buf_id].data_ptr(), op['hw'], op['hsc'], op['hsh'],
                                                    op.get('hw2'), op.get('hsc2'), op.get('hsh2'),
                                                    bufs[op['dst_buf']].data_ptr(), B, op['H'], op['W'], op['Cin'],
                                                    self.bufs[s.buf_id].ld, op['N'], op['ld'], op['ksize'], op['leaky'],
                                                    op['pool'], op['N2'], op['leaky2'], stream), op['name'])
                elif kind == 'direct':
                    s = op['src']
                    if s is None:
                        in_ptr, nchw, cin_ld = x.data_ptr(), 1, op['Cin']
                    else:
                        in_ptr, nchw, cin_ld = bufs[s.buf_id].data_ptr() + 2 * s.ch_off, 0, self.bufs[s.buf_id].ld
                    _lib.check(lib.mc_conv_direct_fwd(in_ptr, nchw, op['w'].data_ptr(), op['scale'].data_ptr(),
                                                      op['shift'].data_ptr(), bufs[op['dst_buf']].data_ptr(), B,
                                                      op['H'], op['W'], op['Cin'], cin_ld, op['N'], op['ld'],
                                                      op['ksize'], op['leaky'], op['pool'], stream), op['name'])
                elif kind == 'pack_input':
                    _lib.check(lib.mc_pack_pnhwc(x.data_ptr(), bufs[op['dst_buf']].data_ptr(), B, op['H'], op['W'],
                                                 op['C'], 8, stream), op['name'])
                elif kind == 'pool':
                    s = op['src']
                    sb = self.bufs[s.buf_id]
                    if s.ch_off != 0:
                        raise NotImplementedError("maxpool on a channel slice")
                    _lib.check(lib.mc_maxpool2x2(bufs[s.buf_id].data_ptr(), bufs[op['dst_buf']].data_ptr(), B, s.H, s.W,
                                                 op['C'], sb.ld, self.bufs[op['dst_buf']].ld, stream), op['name'])
                elif kind == 'conv' and 'chain' in op:
                    members = op['chain']
                    descs = (_lib.mc_conv_desc * len(members))(*[self._conv_desc(m, bufs, B) for m in members])
                    ws = self._conv_workspace(op['ws_off'] + op['ws_bytes'])
                    descs[0].d_ws, descs[0].ws_bytes = ws.data_ptr() + op['ws_off'], op['ws_bytes']
                    _lib.check(lib.mc_conv_chain_fwd(descs, len(members), stream), op['name'])
                elif kind == 'conv':
                    d = self._conv_desc(op, bufs, B)
                    epi = op['epi']
                    if epi == _lib.MC_EPI_NCHW_F32 and detect is not None:
                        # region decode fused into the head's epilogue: dense slot table instead of the raw head
                        thr, only_obj, want_cls = detect
                        A, nc = self.detect_geom
                        P = op['H'] * op['W'] * A
                        boxes = torch.empty(B, P, 8, dtype=torch.float32, device=self.device)
                        cls = torch.empty(B, P, nc, dtype=torch.float32, device=self.device) if want_cls else None
                        dec = _lib.mc_decode_params()
                        dec.d_boxes = boxes.data_ptr()
                        dec.d_cls = cls.data_ptr() if cls is not None else None
                        dec.d_head = None
                        dec.A, dec.nc, dec.conf_thresh, dec.only_objectness = A, nc, float(thr), 1 if only_obj else 0
                        for i, a in enumerate(self.detect_anchors):
                            dec.anchors[i] = float(a)
                        d.epi_mode = _lib.MC_EPI_DECODE
                        out = (boxes, cls)
                        d.decode = ctypes.pointer(dec)
                        d.d_out = None
                    elif epi == _lib.MC_EPI_NCHW_F32:
                        out = torch.empty(B, op['N'], op['H'], op['W'], dtype=torch.float32, device=self.device)
                        bufs[op['dst_buf']] = out
                        d.d_out = out.data_ptr()
                    if op.get('ws_bytes') is None:
                        op['ws_bytes'] = int(lib.mc_workspace_bytes_conv_fwd(ctypes.byref(d)))
                    if op['ws_bytes']:
                        ws = self._conv_workspace(op['ws_bytes'])
                        d.d_ws, d.ws_bytes = ws.data_ptr(), ws.numel()
                    _lib.check(lib.mc_conv_fwd(ctypes.byref(d), stream), op['name'])
                else:
                    raise RuntimeError("unknown op " + kind)
                if events is not None:
                    reps_left -= 1
                    if reps_left == 0:
                        ev1 = torch.cuda.Event(enable_timing=True)
                        ev1.record()
                        events.append((op, ev0, ev1))
            self._prev_op = None
            self._last_bufs = bufs
        return out

    @property
    def num_launches(self):
        """kernel launches per forward (of the last forward's input shape: which layers run chained depends on it)."""
        return len(self._last_items if self._last_items is not None else self.ops)

    def block_activation(self, ind):
        """fp32 NCHW view (in the ORIGINAL channel space) of the output of models[ind] from the last run — for the
        per-block parity tests.  Removed channels are filled with their folded constant."""
        ref = self.block_out[ind]
        bufs = self._last_bufs
        t = bufs[ref.buf_id]
        if t.dtype == torch.float32:
            return t
        B = t.shape[0] // ((ref.H + 1) * (ref.W + 1))
        phys = torch.empty(B, ref.c_phys, ref.H, ref.W, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mc_unpack_pnhwc(t.data_ptr(), phys.data_ptr(), B, ref.H, ref.W, ref.c_phys,
                                                self.bufs[ref.buf_id].ld, ref.ch_off, _lib.stream_ptr()),
                       "mc_unpack_pnhwc")
        full = ref.const.to(self.device).view(1, -1, 1, 1).expand(B, ref.c_orig, ref.H, ref.W).clone()
        for p, c in enumerate(ref.colsrc):
            if c >= 0:
                full[:, c] = phys[:, p]
        return full


def _plan_key(model):
    """Cheap change detector (~20 us): autograd version counters of every parameter/buffer (optimizer steps,
    load_state_dict, in-place edits), storage addresses of the conv weights (.data reassignment, .to()), and the
    set_mask epochs (libmcb200 writes weight.data behind autograd's back)."""
    watch = getattr(model, '_b200_watch', None)
    if watch is None:
        tensors = list(model.parameters()) + list(model.buffers())
        convs = [m for m in model.modules() if getattr(m, 'name', None) == 'MaskedConv2d']
        watch = model._b200_watch = (tensors, convs, len(tensors))
    tensors, convs, _ = watch
    return (bool(getattr(model, 'b200_shrink', True)), tuple(t._version for t in tensors),
            tuple(c.weight.data_ptr() for c in convs),
            tuple((getattr(c, '_mask_epoch', 0), c.mask.data_ptr() if c.mask_flag else 0) for c in convs))


def compile_darknet(model, force=False):
    key = _plan_key(model)
    if force or model._b200_plan is None or model._b200_plan_key != key:
        model._b200_plan = CompiledDarknet(model, shrink=key[0])
        model._b200_plan_key = key
    return model._b200_plan


def darknet_detect_forward(model, x, conf_thresh, only_objectness, want_cls):
    """Eval-mode forward with get_region_boxes' arithmetic (src/nets2_utils.py:158-205) fused into the head
    convolution's epilogue.  Returns (boxes [B,P,8] dense slot table, cls [B,P,nc] or None) for nets2_utils.nms_device
    (counts=None), or None when the compiled plan cannot fuse (the caller then decodes the raw head)."""
    if model.training:
        return None
    plan = compile_darknet(model)
    if not plan.supports_detect(model):
        return None
    plan.detect_geom = (int(model.num_anchors), int(model.num_classes))
    plan.detect_anchors = [float(a) for a in model.anchors]
    return plan.run(x, detect=(float(conf_thresh), 1 if only_objectness else 0, bool(want_cls)))


def darknet_forward(model, x):
    if model.training:
        # batch-statistics BatchNorm + autograd-visible output: the retrain step (src/train.py:221-235)
        from .engine_train import darknet_train_forward
        return darknet_train_forward(model, x)
    return compile_darknet(model).run(x)


def single_conv_forward(conv, x):
    """Stand-alone MaskedConv2d.forward (layers.py:53-64) through the same tcgen05 kernel: fp32 NCHW in/out."""
    lib = _lib.load()
    _lib.require_cuda(x, "MaskedConv2d.forward")
    k = conv.kernel_size[0]
    if conv.kernel_size != (k, k) or k not in (1, 3) or conv.stride != (1, 1) or \
            conv.padding != ((k - 1) // 2, (k - 1) // 2) or conv.groups != 1 or conv.dilation != (1, 1):
        raise NotImplementedError("MaskedConv2d on the B200 path needs k in {1,3}, stride 1, 'same' padding")
    dev = x.device
    x = x.detach().float().contiguous()
    B, C, H, W = x.shape
    w = conv.weight.data.float().contiguous()
    mask = conv.mask.to(dev).contiguous() if getattr(conv, 'mask_flag', False) else None
    O = w.shape[0]
    kblk = 32 if C <= 32 else 64  # the engine's rule (see _compile_conv)
    ld_in, Kc, Npad, ld_out = _round_up(C, 8), _round_up(C, kblk), _round_up(O, 16), _round_up(O, 8)
    xin = torch.empty(B * (H + 1) * (W + 1), ld_in, dtype=torch.bfloat16, device=dev)
    wpack = torch.empty(Npad, k * k * Kc, dtype=torch.bfloat16, device=dev)
    scale = torch.zeros(Npad, device=dev)
    shift = torch.zeros(Npad, device=dev)
    scale[:O] = 1
    if conv.bias is not None:
        shift[:O] = conv.bias.data.float()
    yb = torch.empty(B * (H + 1) * (W + 1), ld_out, dtype=torch.bfloat16, device=dev)
    y = torch.empty(B, O, H, W, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        s = _lib.stream_ptr()
        _lib.check(lib.mc_pack_pnhwc(x.data_ptr(), xin.data_ptr(), B, H, W, C, ld_in, s), "mc_pack_pnhwc")
        _lib.check(lib.mc_pack_conv_weights(w.data_ptr(), None if mask is None else mask.data_ptr(), O, C, k, None, O,
                                            None, C, wpack.data_ptr(), Npad, Kc, s), "mc_pack_conv_weights")
        d = _lib.mc_conv_desc()
        d.d_in, d.d_wpack, d.d_scale, d.d_shift, d.d_out = (xin.data_ptr(), wpack.data_ptr(), scale.data_ptr(),
                                                            shift.data_ptr(), yb.data_ptr())
        d.B, d.H, d.W, d.Cin, d.Cin_ld, d.N, d.Npad = B, H, W, C, ld_in, O, Npad
        d.ksize, d.leaky, d.epi_mode, d.ldc, d.ch_off, d.block_n, d.stages = k, 0, _lib.MC_EPI_PNHWC, ld_out, 0, 0, 0
        d.block_k = kblk
        need = int(lib.mc_workspace_bytes_conv_fwd(ctypes.byref(d)))
        if need and not getattr(conv, 'b200_no_workspace', False):  # (attribute: tests compare with / without stream-K)
            ws = torch.zeros(need, dtype=torch.uint8, device=dev)
            d.d_ws, d.ws_bytes = ws.data_ptr(), need
        _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "mc_conv_fwd")
        _lib.check(lib.mc_unpack_pnhwc(yb.data_ptr(), y.data_ptr(), B, H, W, O, ld_out, 0, s), "mc_unpack_pnhwc")
    return y

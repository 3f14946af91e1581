"""Drop-in for the YOLOv2 part of src/nets.py of the reference: parse_cfg (:39-73), Reorg (:648-667),
MaxPoolStride1 (:640-646), GlobalAvgPool2d (:669-680), EmptyModule (:683-688), Darknet (:692-1061), getYOLOv2
(:1069-1074), and the darknet ``.weights`` reader/writer (:194-279, :897-948, :1007-1051).

Module tree, attribute names and ``state_dict`` keys are the reference's (``models.{i}.conv{n}.weight``,
``models.{i}.bn{n}.*``, ``models.{i}.conv{n}.mask``), so checkpoints interchange.  What differs is the forward:
``Darknet.forward`` hands the whole graph to the B200 engine (engine.py: tcgen05 implicit-GEMM convs with folded
BatchNorm + leaky-ReLU epilogues, fused reorg/concat addressing) instead of walking ``nn.Module``s.
"""
import numpy as np
import torch
import torch.nn as nn

from .pruning.weightPruning.layers import MaskedConv2d
from .pruning.weightPruning.methods import quick_filter_prune, weight_prune  # noqa: F401  (re-exported like nets.py:18)
from .pruning.weightPruning.utils import are_masks_consistent, prune_rate  # noqa: F401


def parse_cfg(cfgfile, verbose=0):
    """nets.py:39-73 — darknet cfg -> list of dict blocks.  ``[convolutional]`` defaults batch_normalize=0; a key
    called ``type`` inside a block is stored as ``_type`` (the section name owns ``type``)."""
    blocks = []
    block = None
    with open(cfgfile, 'r') as fp:
        for raw in fp:
            line = raw.rstrip()
            if line == '' or line[0] == '#':
                continue
            if line[0] == '[':
                if block is not None:
                    if verbose:
                        print(' - block : ', block)
                    blocks.append(block)
                block = {'type': line.lstrip('[').rstrip(']')}
                if block['type'] == 'convolutional':
                    block['batch_normalize'] = 0
            else:
                key, value = line.split('=')
                key = key.strip()
                if key == 'type':
                    key = '_type'
                block[key] = value.strip()
    if block is not None:
        blocks.append(block)
    return blocks


class MaxPoolStride1(nn.Module):
    """nets.py:640-646 (not used by yolov2-voc.cfg; out of the B200 path)."""

    def forward(self, x):
        raise NotImplementedError("MaxPoolStride1 is not used by yolov2-voc.cfg (SURVEY.md §2 #4)")


class Reorg(nn.Module):
    """nets.py:648-667: out[b,(i*s+j)*C+c,y,x] = in[b,c,s*y+i,s*x+j].  Inside ``Darknet`` the engine fuses this into
    the producing conv's store addressing (MC_EPI_REORG2); a direct call of the module runs mc_reorg_nchw."""

    def __init__(self, stride=2):
        super(Reorg, self).__init__()
        self.stride = stride

    def forward(self, x):
        """Stand-alone call (float32 NCHW CUDA tensor in and out, the reference's layout): one libmcb200 kernel."""
        from . import _lib
        lib = _lib.load()
        _lib.require_cuda(x, "Reorg.forward")
        assert x.dim() == 4
        B, C, H, W = x.shape
        s = int(self.stride)
        assert H % s == 0 and W % s == 0
        xin = x.detach().float().contiguous()
        out = torch.empty(B, s * s * C, H // s, W // s, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.mc_reorg_nchw(xin.data_ptr(), out.data_ptr(), B, C, H, W, s, _lib.stream_ptr()), "mc_reorg_nchw")
        return out


class GlobalAvgPool2d(nn.Module):
    def forward(self, x):
        raise NotImplementedError("GlobalAvgPool2d is not used by yolov2-voc.cfg (SURVEY.md §2 #4)")


class EmptyModule(nn.Module):
    """Placeholder for route/shortcut blocks (nets.py:683-688)."""

    def forward(self, x):
        return x


class RegionLoss(nn.Module):
    """nets.py:442-636.  Hyper-parameters as in the reference (filled by create_network :873-889).  ``forward`` is the
    libmcb200 call of region_loss.py (csrc/region_loss.cu; SURVEY.md §8f N3): no copy to the CPU, no Python loop over
    images / boxes / anchors; loss and gradient equal the reference's to float32 round-off (tests/golden/region_loss.npz,
    written by oracle/make_golden_region.py from the unmodified reference)."""

    def __init__(self, num_classes=20, anchor_list=None, anchors_cell=5):
        super(RegionLoss, self).__init__()
        anchor_list = list(anchor_list) if anchor_list is not None else []
        self.num_classes = num_classes
        self.anchors = anchor_list
        self.num_anchors = anchors_cell
        self.anchor_step = int(len(anchor_list) / anchors_cell) if anchors_cell else 0
        self.coord_scale = 1
        self.noobject_scale = 1
        self.object_scale = 1
        self.class_scale = 1
        self.thresh = 0.6
        self.seen = 0

    def forward(self, output, target, verbose=0):
        from .region_loss import region_loss
        return region_loss(output, target, self.anchors, self.num_anchors, self.num_classes, self.coord_scale,
                           self.noobject_scale, self.object_scale, self.class_scale, self.thresh)


class Darknet(nn.Module):
    """nets.py:692-1061."""

    def __init__(self, cfgfile, verbose=0):
        super(Darknet, self).__init__()
        self.blocks = parse_cfg(cfgfile)
        self.models = self.create_network(self.blocks)
        self.loss = self.models[len(self.models) - 1]

        self.width = int(self.blocks[0]['width'])
        self.height = int(self.blocks[0]['height'])

        if self.blocks[(len(self.blocks) - 1)]['type'] == 'region':
            self.anchors = self.loss.anchors
            self.num_anchors = self.loss.num_anchors
            self.anchor_step = self.loss.anchor_step
            self.num_classes = self.loss.num_classes
            if verbose:
                print('  -- [Darknet] anchors', self.anchors, 'num_anchors', self.num_anchors, 'num_classes',
                      self.num_classes)

        self.header = torch.IntTensor([0, 0, 0, 0])
        self.seen = 0
        # B200 engine state (not part of state_dict)
        self._b200_plan = None
        self._b200_plan_key = None
        self._b200_watch = None
        self.b200_shrink = True      # physically drop filters whose (masked) weights are all zero
        # training mode: run the retrain step over the filters the masks keep (engine_train.shrink_layout)
        self.b200_shrink_train = False
        self.b200_keep_blocks = False  # keep every block's activation buffer alive for per-block parity checks

    # ------------------------------------------------------------------ graph construction (nets.py:779-895)
    def create_network(self, blocks):
        models = nn.ModuleList()
        prev_filters = 3
        out_filters = []
        conv_id = 0
        for block in blocks:
            btype = block['type']
            if btype == 'net':
                prev_filters = int(block['channels'])
                continue
            elif btype == 'convolutional':
                conv_id += 1
                batch_normalize = int(block['batch_normalize'])
                filters = int(block['filters'])
                kernel_size = int(block['size'])
                stride = int(block['stride'])
                pad = int((kernel_size - 1) / 2) if int(block['pad']) else 0
                activation = block['activation']
                model = nn.Sequential()
                if batch_normalize:
                    model.add_module('conv{0}'.format(conv_id),
                                     MaskedConv2d(prev_filters, filters, kernel_size, stride, pad, bias=False))
                    model.add_module('bn{0}'.format(conv_id), nn.BatchNorm2d(filters))
                else:
                    model.add_module('conv{0}'.format(conv_id),
                                     MaskedConv2d(prev_filters, filters, kernel_size, stride, pad))
                if activation == 'leaky':
                    model.add_module('leaky{0}'.format(conv_id), nn.LeakyReLU(0.1, inplace=True))
                elif activation == 'relu':
                    model.add_module('relu{0}'.format(conv_id), nn.ReLU(inplace=True))
                prev_filters = filters
                out_filters.append(prev_filters)
                models.append(model)
            elif btype == 'maxpool':
                pool_size = int(block['size'])
                stride = int(block['stride'])
                model = nn.MaxPool2d(pool_size, stride) if stride > 1 else MaxPoolStride1()
                out_filters.append(prev_filters)
                models.append(model)
            elif btype == 'avgpool':
                out_filters.append(prev_filters)
                models.append(GlobalAvgPool2d())
            elif btype == 'reorg':
                stride = int(block['stride'])
                prev_filters = stride * stride * prev_filters
                out_filters.append(prev_filters)
                models.append(Reorg(stride))
            elif btype == 'route':
                layers = block['layers'].split(',')
                ind = len(models)
                layers = [int(i) if int(i) > 0 else int(i) + ind for i in layers]
                if len(layers) == 1:
                    prev_filters = out_filters[layers[0]]
                elif len(layers) == 2:
                    assert (layers[0] == ind - 1)
                    prev_filters = out_filters[layers[0]] + out_filters[layers[1]]
                out_filters.append(prev_filters)
                models.append(EmptyModule())
            elif btype == 'shortcut':
                ind = len(models)
                prev_filters = out_filters[ind - 1]
                out_filters.append(prev_filters)
                models.append(EmptyModule())
            elif btype == 'region':
                loss = RegionLoss()
                loss.anchors = [float(i) for i in block['anchors'].split(',')]
                loss.num_classes = int(block['classes'])
                loss.num_anchors = int(block['num'])
                loss.anchor_step = len(loss.anchors) / loss.num_anchors
                loss.object_scale = float(block['object_scale'])
                loss.noobject_scale = float(block['noobject_scale'])
                loss.class_scale = float(block['class_scale'])
                loss.coord_scale = float(block['coord_scale'])
                out_filters.append(prev_filters)
                models.append(loss)
            else:
                raise NotImplementedError("cfg block type '%s' is not supported by the B200 path" % btype)
        return models

    # ------------------------------------------------------------------ forward (nets.py:720-774)
    def forward(self, x):
        """[B,3,H,W] float32 CUDA -> raw region head [B, A*(5+classes), H/32, W/32] float32 (the region block is
        skipped, nets.py:761-762)."""
        from .engine import darknet_forward
        return darknet_forward(self, x)

    def print_network(self):
        for i, block in enumerate(self.blocks[1:]):
            print('%3d %-14s %s' % (i, block['type'], {k: v for k, v in block.items() if k != 'type'}))

    # ------------------------------------------------------------------ masks (nets.py:1053-1061)
    def masked_convs(self):
        """MaskedConv2d layers in set_masks order (module order == parameter order)."""
        out = []
        for m in self.modules():
            if isinstance(m, nn.Sequential) and len(m) > 0 and getattr(m[0], 'name', None) == 'MaskedConv2d':
                out.append(m[0])
        return out

    def set_masks(self, masks):
        """Assign masks[count] to the count-th MaskedConv2d (module order).  The reference silently ignores every
        error here (bare ``except: pass``, nets.py:1060-1061); a wrong-length list raises instead."""
        convs = self.masked_convs()
        if len(masks) != len(convs):
            raise ValueError("set_masks: got %d masks for %d MaskedConv2d layers" % (len(masks), len(convs)))
        for conv, mask in zip(convs, masks):
            conv.set_mask(mask)
        self._b200_plan = None
        self._b200_watch = None  # new mask buffers: rebuild the change-detector's tensor list

    # ------------------------------------------------------------------ darknet .weights IO
    def _conv_blocks(self, cutoff=None):
        ind = -2
        for bi, block in enumerate(self.blocks):
            ind += 1
            if cutoff is not None and bi > cutoff:
                break
            if block['type'] == 'convolutional':
                yield block, self.models[ind]

    def load_weights(self, weightfile):
        """nets.py:897-948: header int32 x3 (+ seen as int64 when major*10+minor >= 2, else int32), then per conv
        [bn.bias, bn.weight, running_mean, running_var, conv.weight] or [conv.bias, conv.weight], float32."""
        with open(weightfile, 'rb') as f:
            major, minor, revision = np.fromfile(f, dtype=np.int32, count=3)
            if major * 10 + minor >= 2 and major < 1000 and minor < 1000:
                seen = np.fromfile(f, dtype=np.int64, count=1)
            else:
                seen = np.fromfile(f, dtype=np.int32, count=1)
            # The reference reads and DISCARDS the file header (nets.py:899-905): self.header stays [0,0,0,0], so a later
            # save_weights always writes version 0.0.0 with an int32 `seen` — a 16-byte header both loaders read back.
            # Copying a v0.2 file's major/minor here would make save_weights emit "0.2" with a 16-byte header, which every
            # reader then mis-aligns by 4 bytes.  Only the image counter is kept (clamped to what int32 `seen` can hold).
            self.seen = int(seen[0]) & 0x7fffffff

            def read_into(t):
                buf = np.fromfile(f, dtype=np.float32, count=t.numel())
                if buf.size != t.numel():
                    raise IOError("%s: truncated weights file" % weightfile)
                t.data.copy_(torch.from_numpy(buf).view_as(t))

            for block, model in self._conv_blocks():
                conv = model[0]
                if int(block['batch_normalize']):
                    bn = model[1]
                    for t in (bn.bias, bn.weight, bn.running_mean, bn.running_var, conv.weight):
                        read_into(t)
                else:
                    read_into(conv.bias)
                    read_into(conv.weight)
        self._b200_plan = None

    def save_weights(self, outfile, cutoff=0):
        """nets.py:1007-1051: header = IntTensor[4] with header[3] = seen, then the per-conv records."""
        if cutoff <= 0:
            cutoff = len(self.blocks) - 1
        with open(outfile, 'wb') as fp:
            self.header[3] = self.seen
            self.header.numpy().tofile(fp)
            for block, model in self._conv_blocks(cutoff):
                conv = model[0]
                if int(block['batch_normalize']):
                    bn = model[1]
                    tensors = (bn.bias.data, bn.weight.data, bn.running_mean, bn.running_var, conv.weight.data)
                else:
                    tensors = (conv.bias.data, conv.weight.data)
                for t in tensors:
                    t.detach().cpu().numpy().astype(np.float32).tofile(fp)


    # ------------------------------------------------------------------ physically shrunk checkpoints (SURVEY.md §8f N2)
    def channel_map(self):
        """Which original channels survive filter pruning, per convolution: a filter whose (masked) weights are all zero
        is removed from its layer and from the input of every consumer (through maxpool / reorg / route exactly like
        engine.py).  The head convolution keeps all its outputs (the region layer's channel layout is positional).
        Returns a list of dicts (one per conv, cfg order): block, keep_out, keep_in, out_full, in_full, nonzero_out
        (filters with any non-zero weight: equals keep_out except for the head)."""
        alive = {}          # block index -> list of surviving ORIGINAL channel indices of that block's output
        full = {}           # block index -> original channel count
        cur, cur_full = list(range(int(self.blocks[0]['channels']))), int(self.blocks[0]['channels'])
        convs = [i for i, b in enumerate(self.blocks[1:]) if b['type'] == 'convolutional']
        out = []
        ind = -2
        for block in self.blocks:
            ind += 1
            t = block['type']
            if t == 'net':
                continue
            if t == 'convolutional':
                conv = self.models[ind][0]
                w = conv.weight.data
                if getattr(conv, 'mask_flag', False):
                    w = w * conv.mask.to(w.device)
                nonzero = torch.nonzero(w.abs().amax(dim=(1, 2, 3)) > 0).flatten().tolist()
                keep = list(range(w.shape[0])) if ind == convs[-1] else (nonzero or [0])
                out.append(dict(block=ind, keep_out=keep, keep_in=list(cur), out_full=int(w.shape[0]),
                                in_full=int(w.shape[1]), nonzero_out=nonzero))
                cur, cur_full = keep, int(w.shape[0])
            elif t == 'reorg':
                s2 = int(block['stride']) ** 2
                cur = [q * cur_full + c for q in range(s2) for c in cur]
                cur_full = s2 * cur_full
            elif t == 'route':
                ls = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                if len(ls) == 1:
                    cur, cur_full = list(alive[ls[0]]), full[ls[0]]
                else:
                    cur = list(alive[ls[0]]) + [c + full[ls[0]] for c in alive[ls[1]]]
                    cur_full = full[ls[0]] + full[ls[1]]
            alive[ind], full[ind] = list(cur), cur_full
        return out

    def save_shrunk_weights(self, outfile, mapfile=None):
        """Write the PHYSICALLY shrunk network as a darknet ``.weights`` file (same record layout as save_weights:
        [bn.bias, bn.weight, running_mean, running_var, conv.weight] or [conv.bias, conv.weight], only the surviving
        filters and input channels) plus a JSON side-car: the per-layer channel map, the BatchNorm parameters of the
        removed filters and a cfg text with the shrunk filter counts.  A removed filter's output is the constant
        leaky(beta - gamma*mean/sqrt(var+eps)) — zero with default BatchNorm statistics — and the consumers' weights on
        removed input channels are NOT stored: per consumer the side-car keeps `fold` [kept_out, k, k] = sum over removed
        input channels of w * constant (what engine.py feeds through its ones channel), or null when it is all zero.
        Returns the side-car dict.  The reference never shrinks (README "params after pruning" counts zeros)."""
        import json
        cmap = self.channel_map()
        side = dict(format='mcb200-shrunk-1', seen=int(self.seen), layers=[])
        cfg_lines, conv_i = [], 0
        prev_const = torch.zeros(int(self.blocks[0]['channels']))  # constant value of every input channel (0 if kept)
        consts = {}  # block index -> per-channel constants of that block's output
        ind_of = {id(m): i for i, m in enumerate(self.models)}
        with open(outfile, 'wb') as fp:
            np.array([0, 0, 0, int(self.seen) & 0x7fffffff], dtype=np.int32).tofile(fp)
            for block, model in self._conv_blocks():
                m = cmap[conv_i]
                conv_i += 1
                conv = model[0]
                ko = torch.tensor(m['keep_out'], dtype=torch.long)
                ki = torch.tensor(m['keep_in'], dtype=torch.long)
                w = conv.weight.data.detach().cpu()
                if getattr(conv, 'mask_flag', False):
                    w = w * conv.mask.detach().cpu()
                entry = dict(m)
                # constants arriving on this conv's input: follow the graph like channel_map does
                in_const = self._input_constants(m['block'], consts)
                gone_in = torch.tensor(sorted(set(range(m['in_full'])) - set(m['keep_in'])), dtype=torch.long)
                fold = torch.einsum('ocrs,c->ors', w[ko][:, gone_in], in_const[gone_in]) if gone_in.numel() else None
                entry['fold'] = fold.tolist() if fold is not None and bool((fold != 0).any()) else None
                out_const = torch.zeros(m['out_full'])
                if int(block['batch_normalize']):
                    bn = model[1]
                    ps = [bn.bias.data, bn.weight.data, bn.running_mean, bn.running_var]
                    ps = [t.detach().cpu() for t in ps]
                    gone = torch.tensor(sorted(set(range(m['out_full'])) - set(m['keep_out'])), dtype=torch.long)
                    entry['removed'] = gone.tolist()
                    entry['removed_bn'] = [t[gone].tolist() for t in ps]
                    shift = ps[0] - ps[2] * ps[1] / torch.sqrt(ps[3] + bn.eps)
                    cval = torch.where(shift > 0, shift, 0.1 * shift) if block['activation'] == 'leaky' else shift
                    out_const[gone] = cval[gone]
                    for t in ps:
                        t[ko].numpy().astype(np.float32).tofile(fp)
                else:
                    conv.bias.data.detach().cpu()[ko].numpy().astype(np.float32).tofile(fp)
                w[ko][:, ki].contiguous().numpy().astype(np.float32).tofile(fp)
                consts[m['block']] = out_const
                side['layers'].append(entry)
        conv_i = 0
        for block in self.blocks:
            cfg_lines.append('[%s]' % block['type'])
            for k, v in block.items():
                if k == 'type':
                    continue
                if block['type'] == 'convolutional' and k == 'filters':
                    v = len(cmap[conv_i]['keep_out'])
                cfg_lines.append('%s=%s' % ('type' if k == '_type' else k, v))
            if block['type'] == 'convolutional':
                conv_i += 1
            cfg_lines.append('')
        side['cfg'] = '\n'.join(cfg_lines)
        if mapfile is not None:
            with open(mapfile, 'w') as f:
                json.dump(side, f)
        return side

    def _input_constants(self, conv_block, consts):
        """Per-channel constants (values of removed channels) on the input of the conv at models[conv_block], given
        the constants of every earlier conv's output; walks maxpool / reorg / route like channel_map."""
        vals = {}
        cur = torch.zeros(int(self.blocks[0]['channels']))
        ind = -2
        for block in self.blocks:
            ind += 1
            t = block['type']
            if t == 'net':
                continue
            if ind == conv_block:
                return cur
            if t == 'convolutional':
                cur = consts[ind]
            elif t == 'reorg':
                cur = cur.repeat(int(block['stride']) ** 2)
            elif t == 'route':
                ls = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
                cur = vals[ls[0]] if len(ls) == 1 else torch.cat([vals[ls[0]], vals[ls[1]]])
            vals[ind] = cur
        return cur

    def load_shrunk_weights(self, weightfile, side):
        """Inverse of save_shrunk_weights on a FULL-size model built from the original cfg: surviving weights go back to
        their original positions, removed filters get zero weights, a zero mask and their recorded BatchNorm parameters.
        The restored model equals the masked model the file was written from except for the (dropped) weights on removed
        input channels, which only matter when a removed filter's constant is non-zero (side-car `fold`).  Returns the
        masks (quick_filter_prune form: whole filters)."""
        import json
        if isinstance(side, str):
            with open(side) as f:
                side = json.load(f)
        if side.get('format') != 'mcb200-shrunk-1':
            raise ValueError("not a shrunk-weights side-car")
        masks = []
        with open(weightfile, 'rb') as f:
            np.fromfile(f, dtype=np.int32, count=4)
            self.seen = int(side.get('seen', 0))
            for (block, model), m in zip(self._conv_blocks(), side['layers']):
                conv = model[0]
                ko = torch.tensor(m['keep_out'], dtype=torch.long)
                ki = torch.tensor(m['keep_in'], dtype=torch.long)

                def read(n):
                    buf = np.fromfile(f, dtype=np.float32, count=n)
                    if buf.size != n:
                        raise IOError("%s: truncated shrunk weights file" % weightfile)
                    return torch.from_numpy(buf)
                if int(block['batch_normalize']):
                    bn = model[1]
                    gone = torch.tensor(m['removed'], dtype=torch.long)
                    for t, rem in zip((bn.bias.data, bn.weight.data, bn.running_mean, bn.running_var), m['removed_bn']):
                        v = torch.empty(m['out_full'])
                        v[ko] = read(len(m['keep_out']))
                        v[gone] = torch.tensor(rem, dtype=torch.float32)
                        t.copy_(v.to(t.device))
                else:
                    v = torch.zeros(m['out_full'])
                    v[ko] = read(len(m['keep_out']))
                    conv.bias.data.copy_(v.to(conv.bias.device))
                k = conv.kernel_size[0]
                ws = read(len(m['keep_out']) * len(m['keep_in']) * k * k).view(len(m['keep_out']), len(m['keep_in']), k, k)
                w = torch.zeros(m['out_full'], m['in_full'], k, k)
                w[ko.view(-1, 1), ki.view(1, -1)] = ws
                conv.weight.data.copy_(w.to(conv.weight.device))
                mask = torch.zeros(m['out_full'], m['in_full'], k, k)
                mask[torch.tensor(m['nonzero_out'], dtype=torch.long)] = 1.0  # whole filters (methods.py:75)
                masks.append(mask)
        self._b200_plan = None
        return masks


def getYOLOv2(cfgfile, weightfile):
    """nets.py:1069-1074."""
    model = Darknet(cfgfile)
    model.load_weights(weightfile)
    if torch.cuda.is_available():
        model.cuda()
    return model

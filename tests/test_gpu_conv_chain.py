"""Chained CTA-pair launches (mc_conv_chain_fwd): 2..4 wide 3x3 layers, member i+1 reading member i's output, as one
persistent launch.  The arithmetic of every unit is that of the member's own mc_conv_fwd launch, so outputs must be
bit-identical to the per-layer path; only the schedule (and with it the cross-layer readiness protocol) is new."""
import ctypes

import pytest
import torch

import modelcompression_b200 as mc
from modelcompression_b200 import _lib
from modelcompression_b200.engine import compile_darknet

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
H = W = 13


def _pitch(c):
    return (c + 7) // 8 * 8


class Layer(object):
    """one 3x3 layer, weights packed the way tools/trace_conv.py packs them; reads rows of `src` (pitch src_ld) and
    writes channels [ch_off, ch_off + N) of rows of pitch ldc"""

    def __init__(self, lib, gen, Cin, N, src_ld, ldc, ch_off=0):
        self.Cin, self.N, self.src_ld, self.ldc, self.ch_off = Cin, N, src_ld, ldc, ch_off
        Kc, self.Npad = (Cin + 63) // 64 * 64, (N + 15) // 16 * 16
        w = (torch.randn(N, Cin, 3, 3, generator=gen) / (9 * Cin) ** 0.5).to(DEV)
        self.wpack = torch.empty(self.Npad, 9 * Kc, dtype=torch.bfloat16, device=DEV)
        _lib.check(lib.mc_pack_conv_weights(w.data_ptr(), None, N, Cin, 3, None, N, None, Cin, self.wpack.data_ptr(),
                                            self.Npad, Kc, _lib.stream_ptr()), "pack")
        self.scale = (1 + 0.1 * torch.randn(self.Npad, generator=gen)).to(DEV)
        self.shift = (0.1 * torch.randn(self.Npad, generator=gen)).to(DEV)

    def desc(self, B, d_in, d_out, block_n=256):
        d = _lib.mc_conv_desc()
        d.d_in, d.d_wpack, d.d_scale, d.d_shift, d.d_out = d_in, self.wpack.data_ptr(), self.scale.data_ptr(), \
            self.shift.data_ptr(), d_out
        d.B, d.H, d.W, d.Cin, d.Cin_ld, d.N, d.Npad = B, H, W, self.Cin, self.src_ld, self.N, self.Npad
        d.ksize, d.leaky, d.epi_mode, d.ldc, d.ch_off = 3, 1, _lib.MC_EPI_PNHWC, self.ldc, self.ch_off
        d.block_n, d.stages, d.block_k = block_n, 0, 64
        return d


def _rows(B):
    return B * (H + 1) * (W + 1)


def _ragged(lib, gen):
    # 818 -> 1006 -> (36-channel slice + 1018 at channel 40) -> 1022: the middle layer writes a slice of a concat buffer
    c_ld = _pitch(40 + 1018)
    return [Layer(lib, gen, 818, 1006, _pitch(818), _pitch(1006)),
            Layer(lib, gen, 1006, 1018, _pitch(1006), c_ld, ch_off=40),
            Layer(lib, gen, 40 + 1018, 1022, c_ld, _pitch(1022))], 36


def _dense(lib, gen, n):
    return [Layer(lib, gen, 1024, 1024, 1024, 1024) for _ in range(n)], 0


class Chain(object):
    """input, per-member output buffers and workspace of one chain at batch B"""

    def __init__(self, lib, layers, pre, B, gen):
        self.lib, self.layers, self.B = lib, layers, B
        rows = _rows(B)
        self.x = torch.randn(rows, layers[0].src_ld, generator=gen).to(torch.bfloat16).to(DEV)
        self.outs = [torch.zeros(rows, L.ldc, dtype=torch.bfloat16, device=DEV) for L in layers]
        # channels before a member's slice were written by another layer before the chain (conv21's reorg slice)
        for o, L in zip(self.outs, layers):
            if L.ch_off:
                o[:, :pre] = torch.randn(rows, pre, generator=gen).to(torch.bfloat16).to(DEV)
        self.descs = (_lib.mc_conv_desc * len(layers))(
            *[L.desc(B, (self.x if i == 0 else self.outs[i - 1]).data_ptr(), self.outs[i].data_ptr())
              for i, L in enumerate(layers)])
        self.ws_bytes = int(lib.mc_workspace_bytes_conv_chain(self.descs, len(layers)))
        assert self.ws_bytes > 0, _lib.load().mc_last_error_string().decode()
        self.ws = torch.zeros(self.ws_bytes, dtype=torch.uint8, device=DEV)
        self.descs[0].d_ws, self.descs[0].ws_bytes = self.ws.data_ptr(), self.ws_bytes

    def run_chain(self):
        _lib.check(self.lib.mc_conv_chain_fwd(self.descs, len(self.layers), _lib.stream_ptr()), "mc_conv_chain_fwd")

    def run_per_layer(self):
        """the same members through mc_conv_fwd, into copies of the output buffers (the reference)"""
        ref = [o.clone() for o in self.outs]
        for i, L in enumerate(self.layers):
            d = L.desc(self.B, (self.x if i == 0 else ref[i - 1]).data_ptr(), ref[i].data_ptr())
            _lib.check(self.lib.mc_conv_fwd(ctypes.byref(d), _lib.stream_ptr()), "mc_conv_fwd")
        return ref

    def words(self):
        return self.ws.view(torch.int32).cpu()


@pytest.fixture(scope='module')
def lib():
    return _lib.load()


@pytest.mark.parametrize("B", [1, 3, 24, 64])
@pytest.mark.parametrize("kind", ["ragged3", "dense2", "dense3", "dense4"])
def test_chain_bit_exact_vs_per_layer(lib, kind, B):
    gen = torch.Generator().manual_seed(7)
    layers, pre = _ragged(lib, gen) if kind == 'ragged3' else _dense(lib, gen, int(kind[-1]))
    ch = Chain(lib, layers, pre, B, gen)
    ref = ch.run_per_layer()
    for _ in range(2):  # a second launch starts from the workspace the first one left
        ch.run_chain()
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(ch.outs, ref)):
        assert torch.equal(a, b), "member %d differs from its mc_conv_fwd launch" % i
    assert int(ch.words().abs().sum()) == 0, "tickets / counters / status not zero after the launches"


@pytest.mark.parametrize("kind", ["ragged3", "dense3"])
def test_chain_graph_replay_alternating_inputs(lib, kind):
    """a dependency or fence bug shows up as the PREVIOUS replay's values in a later member's output"""
    gen = torch.Generator().manual_seed(11)
    layers, pre = _ragged(lib, gen) if kind == 'ragged3' else _dense(lib, gen, 3)
    ch = Chain(lib, layers, pre, 64, gen)
    inputs = [torch.randn(ch.x.shape, generator=gen).to(torch.bfloat16).to(DEV) for _ in range(2)]
    refs = []
    for x in inputs:
        ch.x.copy_(x)
        refs.append(ch.run_per_layer())
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ch.run_chain()  # warm (module load, attributes) outside the capture
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ch.run_chain()
    for r in range(10):
        ch.x.copy_(inputs[r % 2])
        g.replay()
        torch.cuda.synchronize()
        for i, (a, b) in enumerate(zip(ch.outs, refs[r % 2])):
            assert torch.equal(a, b), "replay %d: member %d differs" % (r, i)
    assert int(ch.words().abs().sum()) == 0


def test_chain_rejections_launch_nothing(lib):
    gen = torch.Generator().manual_seed(3)
    layers, _ = _dense(lib, gen, 3)
    ch = Chain(lib, layers, 0, 64, gen)
    sentinel = [o.clone() for o in ch.outs]
    s = _lib.stream_ptr()

    def bad(descs, n=3):
        arr = (_lib.mc_conv_desc * len(descs))(*descs)
        return lib.mc_conv_chain_fwd(arr, n, s), lib.mc_workspace_bytes_conv_chain(arr, n)

    base = list(ch.descs)

    def mod(i, **kw):
        ds = [_lib.mc_conv_desc.from_buffer_copy(d) for d in base]
        for k, v in kw.items():
            setattr(ds[i], k, v)
        return ds

    cases = {
        'one member': (base[:1], 1),
        'five members': (base + base[:2], 5),
        'not the pair kernel': (mod(1, block_n=64), 3),
        'other batch': (mod(2, B=32), 3),
        'ksize 1': (mod(1, ksize=1), 3),
        'statistics': (mod(1, d_stat_sum=ch.ws.data_ptr(), d_stat_sumsq=ch.ws.data_ptr()), 3),
        'reads another allocation': (mod(1, d_in=ch.x.data_ptr()), 3),
        'pitch differs': (mod(1, Cin_ld=1016), 3),
        'no workspace': (mod(0, d_ws=None, ws_bytes=0), 3),
        'NCHW epilogue': (mod(2, epi_mode=_lib.MC_EPI_NCHW_F32), 3),
    }
    for name, (descs, n) in cases.items():
        rc, nbytes = bad(descs, n)
        assert rc != 0, name
        if name != 'no workspace':
            assert nbytes == 0, name
    # member 2 also reading member 0's output (a dependency the kernel does not track)
    ds = mod(2, d_in=ch.outs[0].data_ptr())
    ds[1] = _lib.mc_conv_desc.from_buffer_copy(base[1])
    assert bad(ds)[0] != 0
    torch.cuda.synchronize()
    for a, b in zip(ch.outs, sentinel):
        assert torch.equal(a, b), "a rejected chain launched"


def _plan_model(shrink):
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(DEV).eval()
    if shrink:
        masks = mc.quick_filter_prune(model, 40.0)
        model.set_masks(masks)
    model.b200_shrink = shrink
    return model


@pytest.mark.parametrize("shrink,want", [(True, [23, 24, 29]), (False, [22, 23, 24, 29])])
def test_plan_chains_the_wide_layers(shrink, want):
    model = _plan_model(shrink)
    plan = compile_darknet(model)
    gen = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randint(0, 256, (64, 3, 416, 416), dtype=torch.uint8, device=DEV, generator=gen)
    with torch.no_grad():
        y = plan.run(x, events=[])
        items = plan._last_items
        chains = [o for o in items if 'chain' in o]
        assert [[m['ind'] for m in c['chain']] for c in chains] == [want]
        assert chains[0]['name'] == 'chain@' + '+'.join(map(str, want))
        names = [o['name'] for o in items]
        assert names.index('conv@26') < names.index(chains[0]['name'])  # the reorg branch runs ahead of the chain
        if shrink:
            assert plan.num_launches == 22 and len(plan.ops) == 24
        acts = {m['ind']: plan.block_activation(m['ind']).clone() for m in chains[0]['chain']}
        # reference: the same plan and buffers, every layer through mc_conv_fwd
        key = next(k for k in plan._items if k[0] == 64)
        plan._items[key] = list(plan.ops)
        y_ref = plan.run(x, events=[])
        for ind, a in acts.items():
            assert torch.equal(a, plan.block_activation(ind)), "block %d" % ind
        assert torch.equal(y, y_ref)

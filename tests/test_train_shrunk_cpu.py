"""Host-side checks of the filter-shrunk retrain step (model.b200_shrink_train): the training plan's physical channel
layout (engine_train.shrink_layout, no device needed) and the exactness of the construction itself, proved on the fp32
oracle: the shrunk restatement (compact convolutions + one ones channel + the expansion rules) equals the dense masked
step to fp32 round-off."""
import numpy as np
import pytest
import torch

import modelcompression_b200 as mc
from modelcompression_b200 import engine_train
from oracle import prune_oracle, train_oracle, train_shrunk_oracle
from oracle.forward_oracle import kaiming_normal_init_, randomize_bn_

# a small Darknet with every structure of YOLOv2's: pools, a 1x1 layer, an activation with two consumers (block 4: the
# pool and the route), a Reorg producer, a concat of the Reorg and a 3x3 layer, and the linear head
SMALL_CFG = """[net]
height=64
width=64
channels=3

[convolutional]
batch_normalize=1
filters=8
size=3
stride=1
pad=1
activation=leaky

[maxpool]
size=2
stride=2

[convolutional]
batch_normalize=1
filters=16
size=3
stride=1
pad=1
activation=leaky

[maxpool]
size=2
stride=2

[convolutional]
batch_normalize=1
filters=16
size=3
stride=1
pad=1
activation=leaky

[maxpool]
size=2
stride=2

[convolutional]
batch_normalize=1
filters=24
size=1
stride=1
pad=1
activation=leaky

[convolutional]
batch_normalize=1
filters=32
size=3
stride=1
pad=1
activation=leaky

[route]
layers=-4

[convolutional]
batch_normalize=1
filters=8
size=1
stride=1
pad=1
activation=leaky

[reorg]
stride=2

[route]
layers=-1,-4

[convolutional]
batch_normalize=1
filters=32
size=3
stride=1
pad=1
activation=leaky

[convolutional]
filters=10
size=1
stride=1
pad=1
activation=linear

[region]
anchors = 1.0, 1.0
bias_match=1
classes=5
coords=4
num=1
softmax=1
jitter=.3
rescore=1
object_scale=5
noobject_scale=1
class_scale=1
coord_scale=1
absolute=1
thresh = .6
random=1
"""


def _set_masks_host(model, masks):
    for conv, m in zip(model.masked_convs(), masks):
        conv.register_buffer('mask', torch.as_tensor(np.asarray(m, np.float32)))
        conv.weight.data *= conv.mask
        conv.mask_flag = True


@pytest.fixture(scope='module')
def yolo_40(tmp_path_factory):
    """seed-0 default-init YOLOv2-VOC, 40 % quick_filter_prune masks (computed by the NumPy oracle)."""
    cfg = mc.write_yolov2_voc_cfg(str(tmp_path_factory.mktemp('cfg') / 'yolov2-voc.cfg'))
    torch.manual_seed(0)
    model = mc.Darknet(cfg)
    ws = [c.weight.detach().numpy() for c in model.masked_convs()]
    _, _, keep, masks = prune_oracle.quick_filter_prune_np(ws, 40.)
    _set_masks_host(model, masks)
    return model, keep


def test_channel_maps_of_the_filter_pruned_net(yolo_40):
    model, keep = yolo_40
    # a kept filter whose weights are all zero still trains: dead is decided by the mask
    conv5 = model.masked_convs()[4]
    f = int(np.nonzero(keep[4])[0][0])
    saved = conv5.weight.data[f].clone()
    conv5.weight.data[f] = 0
    try:
        plan = engine_train.TrainPlan(model, shrink=True)
    finally:
        conv5.weight.data[f] = saved
    assert plan.shrunk
    layers = plan.layers
    for L, k in zip(layers, keep):
        if L.is_head:
            assert L.keep == list(range(L.O_full))
        else:
            assert L.keep == list(np.nonzero(k)[0])
    assert [L.O for L in layers[:5]] == [4, 1, 17, 4, 11]
    for name, (H, W, ld) in list(plan.buf_specs.items()) + list(plan.grad_specs.items()):
        assert ld % 8 == 0, name
    for L in layers:
        for a in (L.z, L.act, L.pooled, L.src):
            if a is not None:
                assert a.ld % 8 == 0 and a.ch_off % 8 == 0
        if L.src is not None:
            assert L.C == L.src.ld and L.C % 8 == 0  # contraction over the whole pitch, pads meet zero weights
    # producer columns: alive filters in order, then the two ones columns (high and low half of the fold)
    for L in layers:
        if L.act is not None and L.act.name in plan.colmap and not L.reorg and L.act.name not in plan.cat_parts:
            cols = plan.colmap[L.act.name]
            assert cols[:L.O] == L.keep and cols[L.O:L.O + 2] == [-2, -2] and set(cols[L.O + 2:]) <= {-1}
    # the concat: Reorg part (4 x alive, quadrant-major), padded to 8, then conv20's part, then the two ones columns
    (name, (l0, l1)), = plan.cat_parts.items()
    cols = plan.colmap[name]
    n0 = 4 * l0.O
    assert cols[:n0] == [q * l0.O_full + f for q in range(4) for f in l0.keep]
    off1 = -(-n0 // 8) * 8
    assert set(cols[n0:off1]) <= {-1} and l1.act.ch_off == off1 and l0.act.ch_off == 0
    assert cols[off1:off1 + l1.O] == [4 * l0.O_full + f for f in l1.keep]
    assert cols[off1 + l1.O:off1 + l1.O + 2] == [-2, -2] and cols.count(-2) == 2
    assert plan.ones_cols[name] == off1 + l1.O
    # every dead input of a consumer is served by its ones column
    for L in layers:
        if L.dead_in:
            assert L.ones_col >= 0 and all(L.cphys[c] < 0 for c, _ in L.dead_in)


def test_no_dead_filter_is_the_dense_plan(yolo_40):
    model, _ = yolo_40
    masks = [c.mask.clone() for c in model.masked_convs()]
    try:
        for c in model.masked_convs():
            c.mask = torch.ones_like(c.mask)
        dense, shrunk = engine_train.TrainPlan(model), engine_train.TrainPlan(model, shrink=True)
    finally:
        for c, m in zip(model.masked_convs(), masks):
            c.mask = m
    assert not shrunk.shrunk and not shrunk.ones_cols
    assert shrunk.buf_specs == dense.buf_specs and shrunk.grad_specs == dense.grad_specs
    for a, b in zip(dense.layers, shrunk.layers):
        assert (a.O, a.C, a.fused_pool) == (b.O, b.C, b.fused_pool)
        for x, y in ((a.z, b.z), (a.act, b.act), (a.pooled, b.pooled), (a.src, b.src)):
            assert (x is None) == (y is None)
            if x is not None:
                assert (x.name, x.C, x.ld, x.ch_off) == (y.name, y.C, y.ld, y.ch_off)


def _small_model(tmp_path, randbn):
    cfg = tmp_path / 'small.cfg'
    cfg.write_text(SMALL_CFG)
    torch.manual_seed(0)
    model = mc.Darknet(str(cfg))
    kaiming_normal_init_(model, 7)
    if randbn:
        randomize_bn_(model, 1)
    gen = torch.Generator().manual_seed(5)
    masks, alive = [], []
    convs = model.masked_convs()
    for i, conv in enumerate(convs):
        O = conv.weight.shape[0]
        m = (torch.rand(conv.weight.shape, generator=gen) > 0.2).float()  # scattered zeros inside alive filters
        if i < len(convs) - 1:
            dead = torch.randperm(O, generator=gen)[:max(1, O // 3)]
            if i == 5:
                dead = torch.arange(O)[torch.arange(O) % 8 != 3]  # the Reorg producer: 1 alive filter (odd)
            m[dead] = 0
        else:
            m[:3] = 0  # head rows: still computed (they produce the bias)
        masks.append(m)
        alive.append(list(range(O)) if i == len(convs) - 1 else
                      torch.nonzero(m.reshape(O, -1).any(1)).flatten().tolist())
    _set_masks_host(model, masks)
    return model.train(), alive


@pytest.mark.parametrize("randbn", [True, False])
def test_shrunk_construction_equals_dense_step(tmp_path, randbn):
    """On rand-BN (beta != 0: non-zero constants) and default BN (beta = 0: the constants start at 0 but dbeta does
    not), the shrunk restatement matches the dense masked train_step_fp32: logits, every parameter gradient (dead
    input columns' dW and dead dbeta included; dead dgamma exactly 0) and the running statistics."""
    model, alive = _small_model(tmp_path, randbn)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    torch.manual_seed(1)
    x = torch.rand(3, 3, 64, 64)
    g = torch.randn(3, 10, 8, 8)
    y, grads, bufs = train_oracle.train_step_fp32(model.blocks, state, x, g)
    ys, grads_s, bufs_s = train_shrunk_oracle.train_step_shrunk_fp32(model.blocks, state, x, g, alive)

    def rel(a, b):
        return float((a - b).norm() / b.norm().clamp_min(1e-30))
    assert rel(ys, y) <= 1e-5
    dead_db = 0
    for name, ref in grads.items():
        assert rel(grads_s[name], ref) <= 1e-5, (name, rel(grads_s[name], ref))
    for i, conv in enumerate(model.masked_convs()[:-1]):
        O = conv.weight.shape[0]
        dead = torch.ones(O, dtype=torch.bool)
        dead[alive[i]] = False
        key = [k for k in grads if k.endswith('bn%d.weight' % (i + 1))][0]
        assert torch.equal(grads_s[key][dead], torch.zeros(int(dead.sum())))
        # a dead channel's dbeta only comes from the borders of 3x3 consumers and from a consumer without BatchNorm (a
        # BatchNorm consumer cancels a constant input shift), so it is small: bound it against the layer's whole dbeta
        bkey = key[:-len('weight')] + 'bias'
        err = float((grads_s[bkey][dead] - grads[bkey][dead]).abs().max())
        assert err <= 1e-5 * float(grads[bkey].norm()), bkey
        dead_db += float(grads[bkey][dead].abs().sum())
    assert dead_db > 0
    for k, v in bufs.items():
        if 'running' in k:
            assert rel(bufs_s[k], v) <= 1e-5, k

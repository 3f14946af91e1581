"""fp32 restatement of the filter-shrunk retrain step (TEST INFRASTRUCTURE — see oracle/__init__.py).

The same step as train_oracle.train_step_fp32, computed the way model.b200_shrink_train computes it: each convolution
runs over its alive filters only, on a physical input made of the alive channels of its producers plus one ones channel
whose weight is sum over dead inputs c of (W*mask)[o,c] * act(beta_c); the compact gradients are expanded with
    dW[o, c_dead] = mask * act(beta_c) * G1[o]          (G1: weight gradient of the ones channel)
    dbeta_c (dead) = act'(beta_c) * sum over consumer inputs c_in carrying c of sum_{o,tap} (W*mask)[o, c_in] * G1[o]
    dgamma_c (dead) = 0,  running statistics of a dead channel decay with batch mean = var = 0.
If the construction is exact, this equals the dense masked step to fp32 round-off (tests/test_train_shrunk_cpu.py).
"""
import torch
import torch.nn.functional as F

from .forward_oracle import reorg


def _act(b, leaky):
    return F.leaky_relu(b, 0.1) if leaky else b


def _slope(b, leaky):
    return torch.where(b > 0, torch.ones_like(b), torch.full_like(b, 0.1)) if leaky else torch.ones_like(b)


def train_step_shrunk_fp32(blocks, state, x, g, alive):
    """alive: per convolution (cfg order) the sorted list of filters it keeps (every filter for the head).
    Returns (y, grads dict name -> full-shape tensor, updated running-stat dict) like train_step_fp32."""
    sd = {k: v.detach().clone().float() for k, v in state.items() if v.is_floating_point()}
    convs = []     # per conv: dict(pre, keep, Wc leaf, cols, dead list [(c, producer conv, filter)], ...)
    outputs = {}   # block index -> (tensor, cols, prov)  prov(c) -> (conv record, filter)
    cur = (x, [0, 1, 2], None)
    ind, conv_id = -2, 0
    for block in blocks:
        ind += 1
        t = block['type']
        if t == 'net':
            continue
        if t == 'convolutional':
            conv_id += 1
            pre = 'models.%d.' % ind
            w = sd[pre + 'conv%d.weight' % conv_id]
            mk = sd.get(pre + 'conv%d.mask' % conv_id)
            wm = w * mk if mk is not None else w
            keep = alive[conv_id - 1]
            bnorm = int(block['batch_normalize'])
            leaky = block['activation'] == 'leaky'
            X, cols, prov = cur
            dead = [] if prov is None else [(c,) + prov(c) for c in range(wm.shape[1]) if c not in cols]
            Wc = torch.zeros(len(keep), len(cols), wm.shape[2], wm.shape[3])
            for j, c in enumerate(cols):
                if c >= 0:
                    Wc[:, j] = wm[keep, c]
                elif c == -2:
                    for cd, P, f in dead:
                        Wc[:, j] += wm[keep, cd] * _act(P['beta'][f], P['leaky'])
            Wc.requires_grad_(True)
            rec = dict(pre=pre, cid=conv_id, keep=keep, Wc=Wc, cols=cols, dead=dead, wm=wm, mask=mk, leaky=leaky,
                       O=wm.shape[0], C=wm.shape[1], bn=bnorm)
            k = int(block['size'])
            bias = sd.get(pre + 'conv%d.bias' % conv_id)
            if bias is not None:
                rec['bias'] = bias.clone().requires_grad_(True)
            z = F.conv2d(X, Wc, rec.get('bias'), 1, (k - 1) // 2 if int(block['pad']) else 0)
            if bnorm:
                bn = pre + 'bn%d.' % conv_id
                rec['beta'] = sd[bn + 'bias']
                rec['gc'] = sd[bn + 'weight'][keep].clone().requires_grad_(True)
                rec['bc'] = sd[bn + 'bias'][keep].clone().requires_grad_(True)
                rm, rv = sd[bn + 'running_mean'][keep].clone(), sd[bn + 'running_var'][keep].clone()
                z = F.batch_norm(z, rm, rv, rec['gc'], rec['bc'], True, 0.1, 1e-5)
                orow = torch.zeros(rec['O'], dtype=torch.bool)
                orow[keep] = True
                for key, comp in (('running_mean', rm), ('running_var', rv)):
                    full = sd[bn + key]
                    full[~orow] = (1.0 - 0.1) * full[~orow] + 0.1 * 0.0
                    full[keep] = comp
            if leaky:
                z = F.leaky_relu(z, 0.1)
            convs.append(rec)
            has_dead = len(keep) < rec['O']
            if has_dead:
                z = torch.cat((z, torch.ones_like(z[:, :1])), 1)
            cur = (z, list(keep) + ([-2] if has_dead else []), (lambda R: (lambda c: (R, c)))(rec))
        elif t == 'maxpool':
            X, cols, prov = cur
            cur = (F.max_pool2d(X, int(block['size']), int(block['stride'])), cols, prov)
        elif t == 'reorg':
            X, cols, prov = cur
            R = prov(0)[0]
            n = len(R['keep'])
            s = int(block['stride'])
            cur = (reorg(X[:, :n], s), [q * R['O'] + f for q in range(s * s) for f in R['keep']],
                   (lambda R, s: (lambda c: (R, c % R['O'])))(R, s), R, s)
        elif t == 'route':
            layers = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
            if len(layers) == 1:
                cur = outputs[layers[0]][:3]
            else:
                a, b = outputs[layers[0]], outputs[layers[1]]
                Ra, Rb = a[2](0)[0], b[2](0)[0]
                na = len(a[1]) - (1 if -2 in a[1] else 0)
                nb = len(b[1]) - (1 if -2 in b[1] else 0)
                base = Ra['O'] * (a[4] ** 2 if len(a) > 3 else 1)
                Xc = torch.cat((a[0][:, :na], b[0][:, :nb]), 1)
                cols = a[1][:na] + [base + c for c in b[1][:nb]]
                if len(Ra['keep']) < Ra['O'] or len(Rb['keep']) < Rb['O']:
                    Xc = torch.cat((Xc, torch.ones_like(Xc[:, :1])), 1)
                    cols.append(-2)

                def pv(c, a=a, b=b, base=base):
                    return a[2](c) if c < base else b[2](c - base)
                cur = (Xc, cols, pv)
        elif t == 'region':
            continue
        else:
            raise NotImplementedError(t)
        outputs[ind] = cur
    y = cur[0]
    (y * g).sum().backward()
    grads = {}
    for R in convs:
        G = R['Wc'].grad
        dW = torch.zeros_like(R['wm'])
        ones = R['cols'].index(-2) if -2 in R['cols'] else -1
        lk = {cd: _act(P['beta'][f], P['leaky']) for cd, P, f in R['dead']}
        for j, c in enumerate(R['cols']):
            if c >= 0:
                dW[R['keep'], c] = G[:, j]
        for cd in lk:
            dW[R['keep'], cd] = lk[cd] * G[:, ones]
        if R['mask'] is not None:
            dW = dW * R['mask']
        grads[R['pre'] + 'conv%d.weight' % R['cid']] = dW
        if 'bias' in R:
            grads[R['pre'] + 'conv%d.bias' % R['cid']] = R['bias'].grad
        if R['bn']:
            bn = R['pre'] + 'bn%d.' % R['cid']
            dg, db = torch.zeros(R['O']), torch.zeros(R['O'])
            dg[R['keep']], db[R['keep']] = R['gc'].grad, R['bc'].grad
            grads[bn + 'weight'], grads[bn + 'bias'] = dg, db
    # dead dbeta: every consumer input that carries the dead channel
    for Q in convs:
        if -2 not in Q['cols']:
            continue
        G1 = Q['Wc'].grad[:, Q['cols'].index(-2)]
        for cd, P, f in Q['dead']:
            s = (Q['wm'][Q['keep'], cd] * G1).sum()
            key = P['pre'] + 'bn%d.bias' % P['cid']
            grads[key][f] += _slope(P['beta'][f], P['leaky']) * s
    bufs = {k: v for k, v in sd.items() if 'running' in k}
    return y.detach(), grads, bufs

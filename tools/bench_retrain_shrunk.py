"""Retrain step of a filter-pruned network, dense (model.b200_shrink_train = False) against shrunk (True), in one process.

Workloads (batch 64, MaskedSGD): the seed-0 default-init YOLOv2-VOC with 40 % quick_filter_prune, and bench.py's own
retrain workload (seed-0 default init, 90 % weight_prune: conv19, conv20 and conv22 lose every filter).  One JSON line per
(workload, arm): forward / backward / SGD ms (medians of device-event timings), the algorithmic GFLOP/img of the arm
(2 x MACs of the convolutions it runs: forward, data gradient except the first layer's, weight gradient), TFLOP/s and
the kernel launches of one step (torch.profiler, in a separate step).

    python tools/bench_retrain_shrunk.py [--steps 20] [--warmup 5] [--batch 64]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import modelcompression_b200 as mc  # noqa: E402


def gflop_per_img(plan):
    total = 0
    for i, L in enumerate(plan.layers):
        # real input channels only: a shrunk plan's pad and ones columns are not counted
        cin = L.C if getattr(L, 'colmap', None) is None else sum(1 for c in L.colmap if c >= 0)
        total += L.H * L.W * L.O * cin * L.k * L.k * (2 if i == 0 else 3)
    return 2.0 * total / 1e9


def run_arm(model, x, g, shrink, steps, warmup):
    model.b200_shrink_train = shrink
    opt = mc.MaskedSGD(model.parameters(), lr=1e-5, momentum=0.9, weight_decay=5e-4 * x.shape[0])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    fwd, bwd, sgd = [], [], []
    for it in range(warmup + steps):
        opt.zero_grad(set_to_none=False)
        ev[0].record()
        y = model(x)
        ev[1].record()
        (y * g).sum().backward()
        ev[2].record()
        opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        if it >= warmup:
            fwd.append(ev[0].elapsed_time(ev[1]))
            bwd.append(ev[1].elapsed_time(ev[2]))
            sgd.append(ev[2].elapsed_time(ev[3]))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        opt.zero_grad(set_to_none=False)
        (model(x) * g).sum().backward()
        opt.step()
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    plan = model._b200_train_plan
    gf = gflop_per_img(plan)
    step = med(fwd) + med(bwd) + med(sgd)
    return dict(shrink=shrink, forward_ms=med(fwd), backward_ms=med(bwd), sgd_ms=med(sgd), step_ms=step,
                gflop_per_img=gf, tflops=gf * x.shape[0] / step, launches_per_step=len(kernels),
                top_kernels=[(e.name[:60], round(e.device_time_total / 1e3, 4)) for e in
                             sorted(kernels, key=lambda e: -e.device_time_total)[:12]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--batch', type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_retrain_shrunk needs a CUDA device")
    dev = torch.device('cuda:0')
    props = torch.cuda.get_device_properties(dev)
    import subprocess
    power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits', '-i', '0'],
                           capture_output=True, text=True).stdout.strip()
    torch.manual_seed(1)
    x = torch.rand(args.batch, 3, 416, 416, device=dev)
    g = torch.randn(args.batch, 125, 13, 13, device=dev) * 1e-3
    cfg = mc.write_yolov2_voc_cfg()
    for name, prune in (("quick_filter_prune 40%", lambda m: mc.quick_filter_prune(m, 40.)),
                        ("weight_prune 90% (bench.py retrain)", lambda m: mc.weight_prune(m, 90.))):
        torch.manual_seed(0)
        model = mc.Darknet(cfg).to(dev)
        model.set_masks(prune(model))
        model.train()
        state = {k: v.clone() for k, v in model.state_dict().items()}
        res = {}
        for shrink in (False, True):
            model.load_state_dict(state)
            res[shrink] = run_arm(model, x, g, shrink, args.steps, args.warmup)
        for shrink in (False, True):
            line = dict(workload=name, batch=args.batch, gpu=props.name, power_limit_w=power, **res[shrink])
            line['speedup_vs_dense'] = res[False]['step_ms'] / res[shrink]['step_ms']
            print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()

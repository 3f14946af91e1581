"""Greedy filter pruning (filter_prune) on the 50.6 M-weight YOLOv2-VOC Darknet (seed 0): device time of the
mc_filter_prune_greedy call (CUDA events, launch queue primed by a spin kernel as bench.py does), its picks, us per
pick, and a per-kernel breakdown (torch.profiler, a separate run) giving the share of pass 1 (filter sums + nonzero
counts).  Prints one JSON line per target with the card name and power limit read in the same run.
Usage: bench_filter_prune.py [reps] [out_dir]"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import modelcompression_b200 as mc  # noqa: E402
from modelcompression_b200 import _lib  # noqa: E402
from modelcompression_b200.pruning.weightPruning import methods  # noqa: E402

PASS1 = ('filter_sumsq_kernel', 'filter_nonzero_kernel')
KERNELS = PASS1 + ('filter_greedy_kernel', 'filter_mask_fill_kernel')


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = 'unknown'
    return name, q


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 9
    out_dir = sys.argv[2] if len(sys.argv) > 2 else None
    dev = torch.device('cuda:0')
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(dev).eval()
    lib = _lib.load()
    plan, params, parr = methods._plan_and_tensors(model, conv_only=True)
    n = sum(plan.O)
    all_params = list(model.parameters())
    total = sum(p.numel() for p in all_params)
    zeros0 = sum(mc.pruning.weightPruning.utils.count_zeros([p.data for p in all_params if p.dim() != 1]))
    ws_bytes = lib.mc_workspace_bytes_filter_prune_greedy(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    out = torch.empty(6 + 2 * n, dtype=torch.int32, device=dev)
    flat = torch.empty(plan.flat_len, dtype=torch.float32, device=dev)
    mask_ptrs = (_lib.c_void_p * len(params))(*[flat.data_ptr() + 4 * o for o in plan.offs])
    name, power = card()

    def call(perc):
        _lib.check(lib.mc_filter_prune_greedy(parr, plan.tables[0], plan.tables[1], plan.tables[2], plan.tables[3],
                                              len(params), zeros0, total, perc, n, out.data_ptr() + 24,
                                              out.data_ptr(), mask_ptrs, ws.data_ptr(), ws_bytes, _lib.stream_ptr()),
                   "mc_filter_prune_greedy")

    for perc in (40., 90.):
        for _ in range(2):
            call(perc)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(3000000)
            e0.record()
            call(perc)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        res = out[:6].cpu().view(torch.int64).tolist()
        picks = res[0]
        # per-kernel device time from the profiler (separate run)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                call(perc)
            torch.cuda.synchronize()
        ktime = {k: 0.0 for k in KERNELS}
        for ev in prof.events():
            for k in KERNELS:
                if k in ev.name:
                    ktime[k] += ev.device_time / 3.0
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            prof.export_chrome_trace(os.path.join(out_dir, 'filter_prune_%d.json' % int(perc)))
        # the public call end to end (host clock: includes count_zeros, the D2H of the picks, printing, set_masks)
        saved = [p.detach().clone() for p in all_params]
        devnull = open(os.devnull, 'w')
        old, sys.stdout = sys.stdout, devnull
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mc.filter_prune(model, perc)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
        finally:
            sys.stdout = old
            devnull.close()
        with torch.no_grad():
            for p, s in zip(all_params, saved):
                p.copy_(s)
        med = statistics.median(ts)
        pass1 = ktime[PASS1[0]] + ktime[PASS1[1]]
        print(json.dumps({
            "workload": "filter_prune(darknet seed 0, %g%%)" % perc, "filters": n, "picks": picks,
            "status": res[2], "device_us_median": round(med, 1), "device_us_min": round(min(ts), 1),
            "us_per_pick_walk": round(ktime['filter_greedy_kernel'] / picks, 3),
            "kernel_us": {k: round(v, 1) for k, v in ktime.items()},
            "pass1_share": round(pass1 / med, 4), "public_call_ms_host": round(wall, 2),
            "timing": "CUDA events around mc_filter_prune_greedy, launch queue primed; kernels by torch.profiler",
            "gpu": name, "power_limit_and_max_sm_clock": power}))


if __name__ == '__main__':
    main()

"""Per-launch timing of the bench workload's forward (shrunk by default, `dense` for the un-pruned net), for comparing
builds inside one GPU lease.  Usage: bench_layers.py [dense] [tag]
Prints one JSON line: {"tag":…, "ms_per_step": graph-replayed step, "per_op_us": {...}}"""
import json
import os
import statistics
import sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import modelcompression_b200 as mc
from modelcompression_b200.engine import compile_darknet

dense = 'dense' in sys.argv
tag = sys.argv[-1] if len(sys.argv) > 1 else ''
B = int(os.environ.get("BENCH_B", "64"))
dev = torch.device('cuda:0')
torch.manual_seed(0)
model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(dev).eval()
if os.environ.get("BENCH_THIN"):
    model.b200_thin = int(os.environ["BENCH_THIN"])
if not dense:
    model.set_masks(mc.quick_filter_prune(model, 40.))
    model.b200_shrink = True
plan = compile_darknet(model)
gen = torch.Generator(device=dev).manual_seed(1)
xs = [torch.rand(B, 3, 416, 416, device=dev, generator=gen) for _ in range(3)]
with torch.no_grad():
    for i in range(9):
        y = model(xs[i % 3])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(60):
        y = model(xs[i % 3])
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 60
    per = {}
    for i in range(15):
        evs = []
        plan.run(xs[i % 3], events=evs)
        torch.cuda.synchronize()
        for op, e0, e1 in evs:
            per.setdefault(op['name'], []).append(e0.elapsed_time(e1) * 1e3)
print(json.dumps({"tag": tag, "dense": dense, "ms_per_step": round(ms, 4), "img_per_s": round(B / ms * 1e3),
                  "checksum": float(y.double().abs().sum()),
                  "per_op_us": {k: round(statistics.median(v), 1) for k, v in per.items()}}))

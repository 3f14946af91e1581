"""Timelines of the CTA-pair conv launches of the shrunk bench step (seed 0, 40 % filter pruning, batch 64): what running
the wide 13x13 layers back to back in one launch could recover, and what the chained launch (mc_conv_chain_fwd) does.

The plan runs eagerly with the launch queue primed (a spin kernel holds the stream while the host enqueues), so gaps
between launches are device time.  Every conv launch gets its own mc_debug_conv_trace buffer (slots as in
tools/trace_conv.py: 0 entry, 4 first operands landed (leader CTA), 13+2i epilogue of unit i done (first 8 units),
30 exit).  A cluster ends with the last epilogue stamp of its two CTAs.  Reported per pair launch:
  tail   = sum over clusters of (layer's last epilogue - cluster's last epilogue) / clusters: the idle cluster time of
           the partial last wave, in us per cluster;
and per pair of consecutive pair launches:
  gap    = next launch's first opnd0 stamp - this launch's last epilogue stamp (launches between them included);
  between = device span of the launches between them (entry of the first to exit of the last), part of `gap`;
and per chained launch: the spread of the clusters' exits (a cluster's exit is the later exit of its two CTAs).
usage: python tools/trace_chain.py [runs]"""
import ctypes, os, statistics, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import modelcompression_b200 as mc
from modelcompression_b200 import _lib
from modelcompression_b200.engine import compile_darknet

dev = torch.device('cuda', 0)
runs = int(sys.argv[1]) if len(sys.argv) > 1 else 5
SLOTS, MAX_CTAS = 32, 600

torch.manual_seed(0)
model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(dev).eval()
masks = mc.quick_filter_prune(model, 40.0)
model.set_masks(masks)
model.b200_shrink = True
plan = compile_darknet(model)
gen = torch.Generator(device=dev).manual_seed(1)
x = torch.randint(0, 256, (64, 3, 416, 416), dtype=torch.uint8, device=dev, generator=gen)
conv_ops = [op for op in plan.ops if op['kind'] == 'conv']  # (at most this many conv launches)


class TracingLib:
    """the engine's library handle with every mc_conv_fwd traced into its own buffer"""

    def __init__(self, lib, bufs):
        self._lib, self._bufs, self.launches = lib, bufs, []

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def mc_conv_fwd(self, d, stream):
        buf = self._bufs[len(self.launches)]
        self._lib.mc_debug_conv_trace(buf.data_ptr())
        rc = self._lib.mc_conv_fwd(d, stream)
        self._lib.mc_debug_conv_trace(None)
        info = (ctypes.c_int * 8)()
        self._lib.mc_conv_last_plan(info)
        self.launches.append((buf, list(info)))
        return rc

    def mc_conv_chain_fwd(self, descs, n, stream):
        buf = self._bufs[len(self.launches)]
        self._lib.mc_debug_conv_trace(buf.data_ptr())
        rc = self._lib.mc_conv_chain_fwd(descs, n, stream)
        self._lib.mc_debug_conv_trace(None)
        info = (ctypes.c_int * 8)()
        self._lib.mc_conv_last_plan(info)
        self.launches.append((buf, list(info)))
        return rc


def stamps(buf, grid):
    t = buf.view(MAX_CTAS, SLOTS)[:grid].cpu().double()
    t[t == 0] = float('nan')
    return t


lib = plan.lib
with torch.no_grad():
    for _ in range(3):
        plan._run_eager(x)
    torch.cuda.synchronize()
    results = []
    for r in range(runs):
        bufs = [torch.zeros(SLOTS * MAX_CTAS, dtype=torch.int64, device=dev) for _ in conv_ops]
        tl = TracingLib(lib, bufs)
        plan.lib = tl
        torch.cuda.synchronize()
        torch.cuda._sleep(8000000)
        plan._run_eager(x)
        torch.cuda.synchronize()
        plan.lib = lib
        launched = [op for op in plan._last_items if op['kind'] == 'conv']
        assert len(tl.launches) == len(launched)
        spans = []  # per conv launch: (entry min, end max) in ns
        pair = []   # per pair launch: dict
        chains = []  # per chained launch: dict
        for k, (op, (buf, info)) in enumerate(zip(launched, tl.launches)):
            t = stamps(buf, info[6])
            epi = t[:, [13 + 2 * i for i in range(8)]]
            cta_end = torch.nan_to_num(epi, nan=-1).max(dim=1).values
            entry = float(torch.nan_to_num(t[:, 0], nan=float('inf')).min())
            if 'chain' in op:
                cl_exit = torch.nan_to_num(t[:, 30], nan=-1).view(-1, 2).max(dim=1).values
                chains.append(dict(name=op['name'], clusters=cl_exit.numel(), span=float(cl_exit.max()) - entry,
                                   exit_first=float(cl_exit.min()) - entry, exit_med=float(cl_exit.median()) - entry))
                spans.append((entry, float(cl_exit.max())))
            elif info[0] == 1:
                cl_end = cta_end.view(-1, 2).max(dim=1).values
                end = float(cl_end.max())
                opnd0 = float(torch.nan_to_num(t[:, 4], nan=float('inf')).min())
                pair.append(dict(k=k, name=op['name'], clusters=cl_end.numel(), entry=entry, opnd0=opnd0, end=end,
                                 first_end=float(cl_end.min()), med_end=float(cl_end.median()),
                                 tail=float((end - cl_end).sum()) / cl_end.numel(), units=info[6] // 2))
                spans.append((entry, end))
            else:
                ex = float(torch.nan_to_num(t[:, 30], nan=-1).max())
                spans.append((entry, ex))
        bounds = []
        for a, b in zip(pair, pair[1:]):
            mid = spans[a['k'] + 1:b['k']]
            between = (max(e for _, e in mid) - min(s for s, _ in mid)) if mid else 0.0
            bounds.append(dict(name=a['name'] + '->' + b['name'], gap=b['opnd0'] - a['end'], between=between,
                               mid=[launched[i]['name'] for i in range(a['k'] + 1, b['k'])]))
        results.append((pair, bounds, chains))

    for r in results:
        for c in r[2]:
            print("  %s: %d clusters, entry -> exit first / median / last %.1f / %.1f / %.1f us" % (
                c['name'], c['clusters'], c['exit_first'] / 1e3, c['exit_med'] / 1e3, c['span'] / 1e3))
    if not results[0][0]:
        sys.exit(0)
    for pair, bounds, _ in results[-1:]:
        t0 = pair[0]['entry']
        print("last run, us from the first pair launch's entry:")
        for p in pair:
            print("  %-10s clusters %2d  entry %7.1f  opnd0 %7.1f  cluster end first/median/last %7.1f / %7.1f / %7.1f"
                  "  tail %5.1f" % (p['name'], p['clusters'], (p['entry'] - t0) / 1e3, (p['opnd0'] - t0) / 1e3,
                                    (p['first_end'] - t0) / 1e3, (p['med_end'] - t0) / 1e3, (p['end'] - t0) / 1e3,
                                    p['tail'] / 1e3))
        for b in bounds:
            print("  %-22s gap %6.1f  between %6.1f  (%s)" % (b['name'], b['gap'] / 1e3, b['between'] / 1e3,
                                                             ' '.join(b['mid']) or '-'))
    print("median over %d runs (us):" % runs)
    names = [p['name'] for p in results[0][0]]
    for i, n in enumerate(names):
        print("  %-10s tail %5.1f  span entry->last epilogue %6.1f" % (
            n, statistics.median(r[0][i]['tail'] for r in results) / 1e3,
            statistics.median(r[0][i]['end'] - r[0][i]['entry'] for r in results) / 1e3))
    for i, b in enumerate(results[0][1]):
        g = statistics.median(r[1][i]['gap'] for r in results) / 1e3
        w = statistics.median(r[1][i]['between'] for r in results) / 1e3
        print("  %-22s gap %6.1f  between %6.1f  gap - between %6.1f" % (b['name'], g, w, g - w))
    tails = [statistics.median(r[0][i]['tail'] for r in results) / 1e3 for i in range(len(names))]
    gaps = [statistics.median(r[1][i]['gap'] - r[1][i]['between'] for r in results) / 1e3 for i in range(len(results[0][1]))]
    print("recoverable by a chain: tails of all but the last member %.1f + boundary gaps without the launches between %.1f"
          " = %.1f us" % (sum(tails[:-1]), sum(gaps), sum(tails[:-1]) + sum(gaps)))

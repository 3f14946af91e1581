#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: "YOLOv2-416 pruned-fwd images/sec ...; prune-mask ms vs
HBM roofline").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): YOLOv2-VOC, seed-0 default init, 40 % global filter pruning
(quick_filter_prune) with the pruned filters PHYSICALLY removed, bf16 forward, batch 64 per GPU, 416x416 synthetic
images (uint8 NCHW, the type do_detect hands to the network; x/255 happens in the first-layer kernel).  One step = one
forward over one batch.  Under torchrun each rank runs the same per-GPU batch on its own images (weak scaling, weights
replicated, no data-path collective); the timed region is bracketed by barrier + synchronize, measured with CUDA
events on the launching stream, and the elapsed time is the max over ranks.

`--impl reference` times the CPU path (oracle port of the reference's PyTorch forward: same F.conv2d / batch_norm /
leaky_relu / max_pool2d calls, same masked weights) on the host cores, on a bounded sample per step.

`--dump-outputs DIR` writes the head the last timed step returned (rank 0's) as DIR/head.npy, float32 [B, 125, 13, 13].
Weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.

Extras in the same JSON line (rank 0): roofline against the BURST bf16 peak (the timed region is milliseconds long) with
the sustained fraction beside it, whole-net fractions, per-op times, decode / NMS microseconds per image, the mask
kernels against the HBM roofline, the dense (un-pruned) network, the retrain step (configs[2]), the 4952-image
evaluation pipeline (configs[4]) with its multi-GPU parity assertion, the data-parallel retrain step at N > 1, a GPU
library baseline (the reference's own model.cuda() path: ATen/cuDNN) and the CPU legs of BASELINE.md §3.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 64
IMG = 416
PRUNE_PERC = 40.0
METRIC = "yolov2_416_pruned_fwd_images_per_sec"
CPU_SAMPLE_BATCH = 4
PER_OP_REPS = 6  # launches per event pair in the per-kernel timing (amortises the events' own cost)
N_INPUT_BUFFERS = 6  # 6 x 33 MB uint8 batches = 199 MB > 126 MB L2
DENSE_GFLOP_PER_IMAGE = 29.360
DUMP_MAX_BYTES = 64 * 1000 * 1000


def profiled_traffic():
    """dram__bytes_read+write per launch of the dominant kernel from the committed ncu --set full capture of this same
    workload (newest profiles/r*_ncu_full_conv_gemm.json; tools/run_ncu_full.sh); (None, None) when there is none."""
    best = None
    pdir = os.path.join(ROOT, 'profiles')
    try:
        for name in sorted(os.listdir(pdir)):
            if name.endswith('_ncu_full_conv_gemm.json'):
                best = name
        if best is None:
            return None, None
        with open(os.path.join(pdir, best)) as f:
            return float(json.load(f)['dram_bytes_per_launch']), 'profiles/' + best
    except Exception:
        return None, None


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p.get('hbm_gbs', 6650.0), bf16=p.get('bf16_tflops', 1590.0),
                    bf16_sustained=p.get('bf16_tflops_sustained', 1400.0), source='measured')
    return dict(hbm_gbs=6650.0, bf16=1590.0, bf16_sustained=1400.0, source='fallback')


def nvml_handle(pynvml, index):
    """NVML handle of CUDA device `index` of this process (NVML numbers physical GPUs, CUDA_VISIBLE_DEVICES renumbers
    CUDA's): matched by UUID, falling back to the index."""
    try:
        import torch
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        if not uuid.startswith('GPU-'):
            uuid = 'GPU-' + uuid
        return pynvml.nvmlDeviceGetHandleByUUID(uuid)
    except Exception:
        return pynvml.nvmlDeviceGetHandleByIndex(index)


class ClockProbe(object):
    """SM clock and throttle reasons through NVML.  Built BEFORE the warm-up (nvmlInit takes tens of ms); no thread:
    sample() is called by the main thread while the GPU works through the already-enqueued timed steps, so the samples
    are taken under load and nothing competes with the launch loop for the interpreter."""

    NAMES = {'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20,
             'hw_power_brake': 0x80, 'sync_boost': 0x10}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = nvml_handle(pynvml, index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for k, bit in self.NAMES.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "how": "NVML polled by the main thread while the GPU ran the enqueued timed steps"}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs NVML reports as local to the GPU (same NUMA node / PCIe root) BEFORE the pinned
    host buffers are allocated, so they land in memory next to the GPU: on a two-socket host a pinned buffer on the far
    socket halves the host->device rate of the end-to-end loop.  Returns the number of CPUs bound to (None if NVML or
    the affinity call is unavailable — the run then proceeds unbound)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = nvml_handle(pynvml, index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return None


def build_pruned_model(device):
    """seed-0 default-init Darknet, 40 % filter pruning applied with set_masks (reference flow: src/train.py:167-174)."""
    import torch
    import modelcompression_b200 as mc
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(device).eval()
    masks, keep = mc.quick_filter_prune(model, PRUNE_PERC, return_keep=True)
    model.set_masks(masks)
    model.b200_shrink = True
    return model, masks, keep


def dump_head(out_dir, head):
    """Write one step's head as out_dir/head.npy (float32).  A head larger than DUMP_MAX_BYTES keeps a seeded sample of
    whole images in batch order (the same images for the same --batch), so that the file stays comparable across runs."""
    import numpy as np
    import torch
    head = head.detach().float().cpu()
    per_image = head[0].numel() * 4
    n = max(1, (DUMP_MAX_BYTES - 128) // per_image)  # 128: the .npy header
    if n < head.shape[0]:
        idx = torch.randperm(head.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
        head = head[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'head.npy'), head.numpy())


# ----------------------------------------------------------------------------------------------------- CPU legs
def cpu_forward_sample(state, blocks, batch, steps, warmup=1):
    """Oracle port of the reference forward on the host cores.  Returns (images/s, seconds per step, head of the last
    step)."""
    import torch
    from oracle import forward_oracle
    torch.manual_seed(1)
    x = torch.rand(batch, 3, IMG, IMG)
    with torch.no_grad():
        for _ in range(warmup):
            forward_oracle.darknet_forward_fp32(blocks, state, x)
        t0 = time.perf_counter()
        for _ in range(steps):
            y, _ = forward_oracle.darknet_forward_fp32(blocks, state, x)
        dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, y


def cpu_stage_legs(dense_state, blocks, anchors):
    """The non-forward stages of BASELINE.md §3 on the host cores, oracle ports (kind "port"): NumPy/PyTorch restatements
    of the reference functions with the same library calls.  Each leg is a bounded sample."""
    import numpy as np
    import torch
    from oracle import detect_oracle, prune_oracle, train_oracle
    legs = {}
    cw = [v.numpy() for k, v in dense_state.items() if v.dim() == 4 and k.endswith('.weight')]
    n = sum(w.size for w in cw)
    t0 = time.perf_counter()
    prune_oracle.weight_prune_np(cw, 70.)
    legs["weight_prune_70"] = {"seconds": time.perf_counter() - t0, "sample": "1 call, all %d weights" % n,
                               "note": "np.percentile on the concatenated |w| (methods.py:18); the reference's own call "
                                       "also builds a 50.6 M-element Python list first (13.4 s in the survey container)"}
    t0 = time.perf_counter()
    prune_oracle.quick_filter_prune_np(cw, 40.)
    legs["quick_filter_prune_40"] = {"seconds": time.perf_counter() - t0, "sample": "1 call, 23 layers, full masks"}
    # decode + NMS on N(0, 2^2) head logits (SURVEY.md §8d: realistic candidate counts), 8 images
    torch.manual_seed(2)
    head = torch.randn(8, 125, 13, 13) * 2
    t0 = time.perf_counter()
    dec = detect_oracle.decode_np(head, 0.005, 20, anchors, 5, 0)
    t_dec = time.perf_counter() - t0
    t0 = time.perf_counter()
    ncand = 0
    for d in dec:
        ncand += d['box'].shape[0]
        detect_oracle.nms_np(d['box'][:, :5], 0.45)
    t_nms = time.perf_counter() - t0
    legs["decode_0.005"] = {"us_per_image": t_dec / 8 * 1e6, "sample": "8 images of N(0,4) logits, vectorised port "
                            "(the reference's per-box Python loop takes 0.06-0.42 s per image)"}
    legs["nms_0.45"] = {"us_per_image": t_nms / 8 * 1e6, "candidates_per_image": ncand / 8,
                        "sample": "8 images, NumPy port with the reference's fp32 op order (the reference's Python "
                                  "O(n^2) loop takes 17-20 s per image at 845 candidates)"}
    # masked train step, batch 2 (BASELINE.md §3)
    torch.manual_seed(1)
    x = torch.rand(2, 3, IMG, IMG)
    torch.manual_seed(3)
    g = torch.randn(2, 125, 13, 13)
    t0 = time.perf_counter()
    train_oracle.train_step_fp32(blocks, dense_state, x, g)
    legs["train_step_b2"] = {"seconds": time.perf_counter() - t0, "sample": "1 forward+backward at batch 2 (no optimizer)"}
    return legs


def run_reference_arm(args, rank):
    """CPU implementation of the path (oracle port; the reference itself is Python and cannot travel to the box)."""
    if rank != 0:
        return
    import torch
    import modelcompression_b200 as mc
    from oracle import prune_oracle
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 for its workers)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        pass
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).eval()
    cw = [p.data.numpy() for p in model.parameters() if p.dim() == 4]
    _, _, _, masks = prune_oracle.quick_filter_prune_np(cw, PRUNE_PERC)
    state = dict(model.state_dict())
    for (name, p), m in zip([(n, p) for n, p in model.named_parameters() if p.dim() == 4], masks):
        state[name] = p.data * torch.from_numpy(m)  # set_mask: weight.data *= mask (layers.py:46)
    cores = torch.get_num_threads()
    ips, sps, head = cpu_forward_sample(state, model.blocks, CPU_SAMPLE_BATCH, args.steps, args.warmup)
    if args.dump_outputs:
        dump_head(args.dump_outputs, head)
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "yolov2-voc-416 40% filter-pruned (masked) forward, CPU oracle port of the reference "
                               "PyTorch path", "batch_per_step": CPU_SAMPLE_BATCH, "prune": "quick_filter_prune 40%"},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "%d steps of batch %d (each step is a bounded sample of the batch-64 workload)" %
                                   (args.steps, CPU_SAMPLE_BATCH)},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------- GPU extras
def time_masks(model_dense, peaks):
    """prune-mask ms vs the HBM roofline (SURVEY.md §8d): weight_prune = 12n bytes, quick_filter_prune = 8n bytes."""
    import torch
    import modelcompression_b200 as mc
    n = sum(p.numel() for p in model_dense.parameters() if p.dim() != 1)
    out = {}
    for name, fn, nbytes in (("weight_prune_70", lambda: mc.weight_prune(model_dense, 70.), 12 * n),
                             ("quick_filter_prune_40", lambda: mc.quick_filter_prune(model_dense, 40.), 8 * n)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        # (1) call on an IDLE GPU: event -> host prelude of the Python call -> launches -> event.  Includes the launch
        #     latency of the first kernel.
        # (2) launch queue primed: a ~1.5 ms spin kernel runs first, so the call's launches are already queued when the
        #     start event fires and the interval is the device time of the call's kernels alone (what a pruning call
        #     costs inside a busy stream, and the kernel duration the HBM roofline is quoted against).
        idle, ts = [], []
        for primed in (False, True):
            for _ in range(7):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                if primed:
                    torch.cuda._sleep(3000000)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                (ts if primed else idle).append(e0.elapsed_time(e1))
        ms = statistics.median(ts)
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "ms_call_on_idle_gpu": statistics.median(idle), "algorithmic_bytes": nbytes,
                     "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks['hbm_gbs'],
                     "timing": "CUDA events around the public call with the launch queue primed (device time of the "
                               "call's kernels); ms_call_on_idle_gpu adds the first launch's host latency"}
    return out


def kn_model(device):
    """KN-init + rand-BN weights (SURVEY.md §8d): realistic logit ranges for decode / NMS / mAP."""
    import torch
    import modelcompression_b200 as mc
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg())
    g = torch.Generator().manual_seed(7)
    for p in model.parameters():
        if p.dim() == 4:
            fan_in = p.shape[1] * p.shape[2] * p.shape[3]
            p.data.copy_(torch.randn(p.shape, generator=g) * (2.0 / (1.01 * fan_in)) ** 0.5)
    return model.to(device).eval()


def time_detect_stages(model, device, B):
    """decode and NMS as microseconds per image and GB/s (SURVEY.md §8d: latency-bound, reported, not a roofline claim).
    Two inputs: N(0, 2^2) logits (realistic candidate counts) and the default-init head (every box a candidate)."""
    import torch
    from modelcompression_b200.nets2_utils import decode_device, nms_device
    out = {}
    torch.manual_seed(2)
    heads = {"randn2_logits": torch.randn(B, 125, 13, 13, device=device) * 2,
             "all_845_candidates": torch.zeros(B, 125, 13, 13, device=device)}
    for tag, head in heads.items():
        for thr, oo, val in ((0.005, 0, True), (0.25, 1, False)):
            td, tn = [], []
            for it in range(8):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                torch.cuda._sleep(1000000)
                e[0].record()
                boxes, counts, cls = decode_device(head, thr, 20, model.anchors, model.num_anchors, oo, val)
                e[1].record()
                keep, kc = nms_device(boxes, counts, 0.45)
                e[2].record()
                torch.cuda.synchronize()
                if it >= 2:
                    td.append(e[0].elapsed_time(e[1]))
                    tn.append(e[1].elapsed_time(e[2]))
            d_ms, n_ms = statistics.median(td), statistics.median(tn)
            ncand = float(counts.float().mean())
            dec_bytes = B * 125 * 169 * 4 + ncand * B * (32 + (80 if val else 0))
            nms_bytes = ncand * B * (32 + 4)
            out["%s_conf%g" % (tag, thr)] = {
                "candidates_per_image": ncand, "kept_per_image": float(kc.float().mean()),
                "decode_us_per_img": d_ms * 1e3 / B, "decode_gbs": dec_bytes / (d_ms * 1e-3) / 1e9,
                "nms_us_per_img": n_ms * 1e3 / B, "nms_gbs": nms_bytes / (n_ms * 1e-3) / 1e9}
    out["note"] = "one CTA per image; both stages are latency-bound (84.5 KB of logits and <= 27 KB of boxes per image)"
    return out


def eval_image_source(device, B):
    """Deterministic synthetic image set for the evaluation pipeline: image i is pool[i % P] with every byte XOR-ed by
    (i // P) & 0xFF — a function of the GLOBAL image index only, so any sharding sees the same images."""
    import torch
    P = 2 * B
    g = torch.Generator(device=device).manual_seed(7)
    pool = torch.randint(0, 256, (P, 3, IMG, IMG), dtype=torch.uint8, device=device, generator=g)

    def get_batch(lo, hi):
        idx = torch.arange(lo, hi, device=device)
        return pool[idx % P] ^ ((idx // P) & 0xFF).to(torch.uint8).view(-1, 1, 1, 1)

    return get_batch


def time_eval_pipeline(model, device, B, rank, world, tag, conf=0.005, n_images=4952):
    """BASELINE.json configs[4]: batch-sharded evaluation of 4952 synthetic VOC2007-test-shaped images — forward,
    region decode (conf 0.005, validation mode: multi-class rows), per-image NMS (0.45), compaction, one gather of the
    detections to rank 0 at the end (src/predict.py:116-179 restated in eval.evaluate_sharded).  Images are generated
    on the device per batch (uint8), so the number is the device pipeline; returns images/s over all ranks.
    At world > 1 rank 0 also re-runs a prefix of the set alone and asserts the gathered rows are torch.equal."""
    import torch
    import torch.distributed as dist
    from modelcompression_b200.eval import evaluate_sharded

    get_batch = eval_image_source(device, B)
    # warm-up at FULL size: the first pass also pays the caching allocator's cudaMalloc of the ~1 GB detection tensors
    # (0.1-0.2 s, once per process), which is not the pipeline
    evaluate_sharded(model, get_batch, n_images, B, conf, 0.45, 0, rank, world, validation=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # two timed passes, the faster one is reported and both are listed: this is wall clock around ~80 batches with
    # ~1 GB of detection tensors, and a pass now and then pays a cudaFree/cudaMalloc round of the caching allocator
    # (0.8 s instead of 0.2 s was seen once) that is not the pipeline
    runs = []
    for _ in range(2):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        dets = evaluate_sharded(model, get_batch, n_images, B, conf, 0.45, 0, rank, world, validation=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        runs.append(dt)
    dt = min(runs)
    res = {"workload": "%d synthetic 416x416 images (%s weights), batch %d per GPU: forward + decode (%g, validation) + "
                       "NMS (0.45) + detection gather to rank 0" % (n_images, tag, B, conf),
           "images_per_s": n_images / dt, "seconds": dt, "seconds_runs": [round(r, 5) for r in runs],
           "detection_rows": int(dets.shape[0]) if rank == 0 else None,
           "includes": "images produced on the device per batch (uint8); no host->device copies"}
    ph = {}
    evaluate_sharded(model, get_batch, n_images, B, conf, 0.45, 0, rank, world, validation=True, phases=ph)
    res["phases_rank%d" % rank] = {k: round(v, 5) for k, v in ph.items()}
    if world > 1:
        allp = [None] * world
        dist.all_gather_object(allp, {k: round(v, 5) for k, v in ph.items()})
        res["phases_max_over_ranks"] = {k: max(p[k] for p in allp) for k in ph}
        # parity of the multi-GPU path on hardware: gathered detections == the 1-GPU result for the same images
        n_chk = min(n_images, 3 * B * world + 7)
        got = evaluate_sharded(model, get_batch, n_chk, B, conf, 0.45, 0, rank, world, validation=True)
        ok = None
        if rank == 0:
            alone = evaluate_sharded(model, get_batch, n_chk, B, conf, 0.45, 0, 0, 1, validation=True, gather=False)
            ok = bool(got.shape == alone.shape and torch.equal(got, alone))
            res["gather_equals_1gpu"] = ok
            res["gather_check"] = "%d images, %d rows: NCCL-gathered rows of %d ranks torch.equal to rank 0 alone" % (
                n_chk, int(alone.shape[0]), world)
            assert ok, "gathered detections differ from the 1-GPU result"
        dist.barrier()
    return res


def time_scorer_and_loss(model, device, B):
    """SURVEY.md §8f N1 / N3, timed: the VOC07 scorer (voc_eval.mean_ap, src/predict.py:216-437; csrc/voc_eval.cu) on the
    detections of 512 KN-init images against synthetic labels, and RegionLoss forward + backward (src/nets.py:442-636;
    csrc/region_loss.cu) on a batch-B head."""
    import numpy as np
    import torch
    from modelcompression_b200 import voc_eval
    from modelcompression_b200.eval import evaluate_sharded
    n = 512
    get_batch = eval_image_source(device, B)
    dets = evaluate_sharded(model, get_batch, n, B, 0.005, 0.45, 0, validation=True)
    rng = np.random.RandomState(4)
    rows = []
    for i in range(n):  # SURVEY.md §8d: 1-5 boxes per image, class U{0..19}, centre U[0.1,0.9], size U[0.05,0.5]
        for _ in range(rng.randint(1, 6)):
            c = int(rng.randint(0, 20))
            cx, cy = rng.uniform(0.1, 0.9, 2)
            w, h = rng.uniform(0.05, 0.5, 2)
            rows.append([i, c, max(int((cx - w / 2) * IMG), 1), max(int((cy - h / 2) * IMG), 1),
                         min(int((cx + w / 2) * IMG), IMG), min(int((cy + h / 2) * IMG), IMG), 0])
    gts = torch.tensor(rows, device=device)
    voc_eval.mean_ap(dets, gts, 20, None, 0.5, True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    aps, m = voc_eval.mean_ap(dets, gts, 20, None, 0.5, True)
    torch.cuda.synchronize()
    t_map = time.perf_counter() - t0
    torch.manual_seed(5)
    head = torch.randn(B, 125, 13, 13, device=device, requires_grad=True)
    target = torch.zeros(B, 250, device=device)
    for b in range(B):
        for j in range(3):
            target[b, 5 * j:5 * j + 5] = torch.tensor([float((b + j) % 20), 0.2 + 0.2 * j, 0.3 + 0.1 * j, 0.2, 0.3])
    ts = []
    for it in range(5):
        head.grad = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = model.loss(head, target)
        loss.backward()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return {"voc_map_scorer": {"seconds": t_map, "images": n, "detection_rows": int(dets.shape[0]), "gt_boxes": len(rows),
                               "mAP": m, "note": "wall clock of voc_eval.mean_ap (libmcb200 mc_voc_table + mc_voc_match over all classes, torch.sort / cumsum, vectorised 11-point AP)"},
            "region_loss": {"ms_forward_backward": statistics.median(ts) * 1e3, "batch": B,
                            "note": "wall clock of RegionLoss forward + backward (libmcb200 mc_region_loss: two kernels)"}}


def time_retrain(device, peaks, B, steps=5):
    """BASELINE.json configs[2]: 90 % weight pruning, masked forward + backward + SGD step at batch B on one B200
    (src/train.py:214-235 with the synthetic loss of SURVEY.md §8d: loss = (y*g).sum())."""
    import torch
    import modelcompression_b200 as mc
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(device)
    model.set_masks(mc.weight_prune(model, 90.))
    model.train()
    opt = make_sgd(model, B)
    gen = torch.Generator(device=device).manual_seed(1)
    xs = [torch.rand(B, 3, IMG, IMG, device=device, generator=gen) for _ in range(2)]
    g = torch.randn(B, 125, 13, 13, device=device, generator=gen)
    tf, tb, ts = [], [], []
    for it in range(steps + 2):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        opt.zero_grad(set_to_none=True)
        ev[0].record()
        loss = (model(xs[it % 2]) * g).sum()
        ev[1].record()
        loss.backward()
        ev[2].record()
        opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        if it >= 2:
            tf.append(ev[0].elapsed_time(ev[1]))
            tb.append(ev[1].elapsed_time(ev[2]))
            ts.append(ev[2].elapsed_time(ev[3]))
    f, b, s = statistics.median(tf), statistics.median(tb), statistics.median(ts)
    gflop_img = 3 * DENSE_GFLOP_PER_IMAGE - 0.299  # fwd + dgrad + wgrad, no dgrad for conv1 (SURVEY.md §8d)
    ok = bool(mc.are_masks_consistent(model, [c.mask for c in model.masked_convs()]))
    tfl = gflop_img * B / (f + b + s)
    return {"workload": "yolov2-voc-416 90%% weight-pruned, masked forward+backward+SGD step, batch %d" % B,
            "forward_ms": f, "backward_ms": b, "sgd_ms": s, "ms_per_step": f + b + s,
            "images_per_s": B / (f + b + s) * 1e3, "algorithmic_gflop_per_image": gflop_img, "tflops": tfl,
            "frac_of_bf16_burst": tfl / peaks['bf16'], "frac_of_bf16_sustained": tfl / peaks['bf16_sustained'],
            "masks_consistent_after_steps": ok, "optimizer": type(opt).__module__ + "." + type(opt).__name__ +
            "(lr 1e-5, momentum 0.9, wd 5e-4*B) as src/train.py:144-147"}


def make_sgd(model, B, world=1):
    """The reference's optimizer (src/train.py:144-147): SGD lr 1e-5, momentum 0.9, weight decay 5e-4 * batch — as one
    fused libmcb200 kernel when the package provides it, else torch.optim.SGD."""
    import torch
    import modelcompression_b200 as mc
    kw = dict(lr=1e-5, momentum=0.9, weight_decay=5e-4 * B * world)
    fused = getattr(mc, 'MaskedSGD', None)
    if fused is not None:
        return fused(model.parameters(), **kw)
    return torch.optim.SGD(model.parameters(), **kw)


def time_dp_retrain(device, B, rank, world, steps=5):
    """SURVEY.md §8f N4 on hardware: the masked retrain step with the per-layer NCCL gradient all-reduce issued inside
    the backward vs the same step without the exchange; the averaged gradients must equal the mean of the ranks' local
    gradients and be identical on every rank."""
    import torch
    import torch.distributed as dist
    import modelcompression_b200 as mc
    from modelcompression_b200 import train_dp
    torch.manual_seed(0)
    model = mc.Darknet(mc.write_yolov2_voc_cfg()).to(device)
    model.set_masks(mc.weight_prune(model, 90.))
    train_dp.broadcast_parameters(model)
    model.train()
    gen = torch.Generator(device=device).manual_seed(10 + rank)
    x = torch.rand(B, 3, IMG, IMG, device=device, generator=gen)
    g = torch.randn(B, 125, 13, 13, device=device, generator=gen)
    model.zero_grad()
    (model(x) * g).sum().backward()
    mean_g = []
    for p in model.parameters():
        m = p.grad.clone()
        dist.all_reduce(m)
        mean_g.append(m / world)
    train_dp.enable(model)
    model.zero_grad()
    (model(x) * g).sum().backward()
    worst, same = 0.0, True
    for p, m in zip(model.parameters(), mean_g):
        worst = max(worst, float((p.grad - m).abs().max() / m.abs().max().clamp_min(1e-30)))
        chk = p.grad.clone()
        dist.broadcast(chk, src=0)
        same = same and bool(torch.equal(chk, p.grad))
    opt = make_sgd(model, B, world)

    def step():
        opt.zero_grad(set_to_none=True)
        (model(x) * g).sum().backward()
        opt.step()

    def timed():
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms_dp = timed()
    train_dp.disable(model)
    ms_local = timed()
    flags = torch.tensor([1.0 if same else 0.0, worst], device=device)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok = bool(mc.are_masks_consistent(model, [c.mask for c in model.masked_convs()]))
    del model, opt
    torch.cuda.empty_cache()
    return {"workload": "masked retrain step, batch %d per GPU, %d GPUs, gradients averaged by per-layer NCCL all-reduce "
                        "inside the backward" % (B, world), "ms_per_step_with_allreduce": ms_dp,
            "ms_per_step_without": ms_local, "images_per_s": B * world / (ms_dp * 1e-3),
            "averaged_equals_mean_of_local_max_rel": worst, "identical_on_all_ranks": bool(flags[0].item() == 1.0),
            "masks_consistent_after_steps": ok, "gradient_bytes_per_step": 4 * sum(p.numel() for p in mean_g)}


def library_forward(blocks, state, x):
    """The reference's own GPU path (model.cuda() -> ATen/cuDNN; src/predict.py:126-129): the same module calls
    Darknet.forward makes (src/nets.py:720-774), written with torch.nn.functional on a state_dict."""
    import torch
    import torch.nn.functional as F
    outputs = {}
    ind, conv_id = -2, 0
    for block in blocks:
        ind += 1
        t = block['type']
        if t in ('net', 'region'):
            continue
        if t == 'convolutional':
            conv_id += 1
            pre = 'models.%d.' % ind
            k = int(block['size'])
            x = F.conv2d(x, state[pre + 'conv%d.weight' % conv_id], state.get(pre + 'conv%d.bias' % conv_id), 1,
                         (k - 1) // 2 if int(block['pad']) else 0)
            if int(block['batch_normalize']):
                x = F.batch_norm(x, state[pre + 'bn%d.running_mean' % conv_id], state[pre + 'bn%d.running_var' % conv_id],
                                 state[pre + 'bn%d.weight' % conv_id], state[pre + 'bn%d.bias' % conv_id], False, 0.1, 1e-5)
            if block['activation'] == 'leaky':
                x = F.leaky_relu(x, 0.1)
        elif t == 'maxpool':
            x = F.max_pool2d(x, int(block['size']), int(block['stride']))
        elif t == 'reorg':
            B, C, H, W = x.shape
            x = x.reshape(B, C, H // 2, 2, W // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(B, 4 * C, H // 2, W // 2)
        elif t == 'route':
            ls = [int(i) if int(i) > 0 else int(i) + ind for i in block['layers'].split(',')]
            x = outputs[ls[0]] if len(ls) == 1 else torch.cat((outputs[ls[0]], outputs[ls[1]]), 1)
        outputs[ind] = x
    return x


def time_library_baseline(model, device, B, x_f32):
    """`gpu_library_baseline`: the masked-dense network (the reference never shrinks) through ATen/cuDNN on this GPU, in
    the reference's fp32 (TF32 off and on) and in bf16 channels_last (the strongest stock-PyTorch configuration).  This
    is library code timed beside the product, not part of it."""
    import torch
    out = {}
    blocks = model.blocks
    base = {k: v.detach() for k, v in model.state_dict().items() if not k.endswith('.mask')}

    def run(tag, state, x, tf32):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.benchmark = True
        with torch.no_grad():
            for _ in range(3):
                library_forward(blocks, state, x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(2000000)
            e0.record()
            for _ in range(5):
                library_forward(blocks, state, x)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        out[tag] = {"ms_per_step": ms, "images_per_s": B / (ms * 1e-3),
                    "tflops_dense_equivalent": DENSE_GFLOP_PER_IMAGE * B / ms}

    try:
        run("fp32_cudnn", base, x_f32, False)
        run("tf32_cudnn", base, x_f32, True)
        st16 = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v) for k, v in base.items()}
        st16 = {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in st16.items()}
        run("bf16_channels_last_cudnn", st16, x_f32.to(torch.bfloat16).contiguous(memory_format=torch.channels_last), True)
    except Exception as exc:  # the library baseline must never take the product's bench line down
        out["error"] = repr(exc)[:200]
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = False
    out["note"] = ("masked-dense YOLOv2 (40 %% of the filters zeroed, not removed: the reference's own formulation) through "
                   "torch.nn.functional on this GPU; eager launches, no CUDA graph, batch %d" % B)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=BATCH)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-dense', action='store_true', help='skip the extra un-pruned dense-network timing')
    ap.add_argument('--no-retrain', action='store_true', help='skip the extra retrain-step timings (configs[2], N4)')
    ap.add_argument('--no-eval', action='store_true', help='skip the extra evaluation-pipeline timing (configs[4])')
    ap.add_argument('--no-library', action='store_true', help='skip the ATen/cuDNN library baseline')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the head of the last timed step as DIR/head.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else max(args.warmup, 1)

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    import modelcompression_b200 as mc
    from modelcompression_b200.engine import compile_darknet

    assert torch.cuda.is_available(), "bench.py (b200 arm) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    bound_cpus = bind_to_gpu_numa(local_rank)
    probe = ClockProbe(local_rank)  # NVML initialised here, long before the timed region
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    peaks = measured_peaks()
    B = args.batch
    K = args.steps

    model, masks, keep = build_pruned_model(device)
    plan = compile_darknet(model)
    flops_img = plan.flops_per_image

    # inputs resident in HBM: rotating uint8 batches, together larger than L2
    gen = torch.Generator(device=device).manual_seed(1 + rank)
    xs = [torch.randint(0, 256, (B, 3, IMG, IMG), dtype=torch.uint8, device=device, generator=gen)
          for _ in range(N_INPUT_BUFFERS)]
    input_mb = B * 3 * IMG * IMG / 1e6

    def step(i):
        return model(xs[i % len(xs)])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # warm-up: at least W steps and at least four passes over every input buffer (the engine captures a CUDA graph
        # for an input address the third time it sees it; captures must not land in the timed region)
        for i in range(max(args.warmup, 4 * len(xs))):
            step(i)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        barrier()
        # The launch queue is primed: a ~1.5 ms spin kernel holds the stream while the host enqueues the timed steps, so
        # the interval between the first and the last event is device time of exactly K steps (no idle gap before the
        # first launch, no host jitter inside a window that is only milliseconds long).
        # The spin covers the host's enqueue time of all K steps (~60 us each: plan check, graph replay, output clone), and
        # the garbage collector is off meanwhile: a host stall inside the loop (one 45 ms pause was seen in a 100-step
        # run) would otherwise be billed to the device.
        import gc

        def timed_region():
            gc.collect()
            gc.disable()
            torch.cuda._sleep(max(3000000, 130000 * K))
            ev[0].record()
            for i in range(K):
                out = step(i)
                ev[i + 1].record()
            gc.enable()
            # NVML queries perturb the GPU: polling every 0.5 ms cost 1.2 % of the step (79.9 k vs 80.95 k img/s, same
            # lease, five runs); ~10 samples per timed region are enough to see a clock drop or a throttle reason
            poll_s = min(5e-3, max(1e-3, K * 0.8e-3 / 10))
            while not ev[K].query():  # clocks / throttle reasons sampled DURING the timed region, off the launch path
                probe.sample()
                time.sleep(poll_s)
            probe.sample()
            barrier()
            return [ev[i].elapsed_time(ev[i + 1]) for i in range(K)], out

        # A timed region in which ONE step is many times the median (seen once: a 70 ms step among 99 of 0.79 ms, i.e. the
        # host stalled longer than the spin kernel covers and the GPU sat idle waiting for launches) is not a measurement
        # of the device: like a throttled run it is rejected and re-measured (at most twice), and the rejected attempts
        # stay in the JSON line ("rejected_attempts").  All ranks decide together.
        rejected_attempts = []
        for attempt in range(3):
            step_ms, last_head = timed_region()
            med = statistics.median(step_ms)
            stalled = 1.0 if (K >= 4 and max(step_ms) > 5.0 * med) else 0.0
            if world > 1:
                t = torch.tensor([stalled], device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                stalled = float(t.item())
            if not stalled or attempt == 2:
                break
            rejected_attempts.append({"rank": rank, "total_ms": ev[0].elapsed_time(ev[K]), "median_step_ms": med,
                                      "max_step_ms": max(step_ms), "why": "a step > 5x the median: host stall"})
        if args.dump_outputs and rank == 0:
            dump_head(args.dump_outputs, last_head)
        y = step(0)
        clocks = probe.result()
        elapsed_ms = ev[0].elapsed_time(ev[K])
        step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
        my_ms_per_step = elapsed_ms / K
        per_rank = None
        if world > 1:
            # every rank's own step time and clocks (diagnostic: which rank sets the max, and whether it was clocked down)
            mine = {"rank": rank, "ms_per_step": my_ms_per_step, "median_step_ms": statistics.median(step_ms),
                    "max_step_ms": max(step_ms), "sm_mhz": clocks.get("sm_mhz"), "reasons": clocks.get("reasons")}
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            per_rank = gathered
            t = torch.tensor([elapsed_ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            elapsed_ms = float(t.item())
        value = B * K * world / (elapsed_ms * 1e-3)

        # ---- per-kernel timing (CUDA events around every launch, same stream), up to 20 steps
        conv_ms, other_ms = 0.0, 0.0
        per_layer = {}
        ksteps = min(K, 20)
        for i in range(ksteps):
            events = []
            # queue primed: the eager launches (ctypes calls, ~20 us of host time each) are enqueued while the GPU spins, so
            # an event interval is the kernel's duration on the device, not the host's latency between record and launch
            torch.cuda._sleep(8000000)
            plan.run(xs[i % len(xs)], events=events, repeat=PER_OP_REPS)
            torch.cuda.synchronize()
            for op, a, b in events:
                ms = a.elapsed_time(b) / PER_OP_REPS
                if op['kind'] == 'conv':
                    conv_ms += ms
                else:
                    other_ms += ms
                per_layer.setdefault(op['name'], []).append(ms)
        conv_flops_step, all_flops_step, conv_launches = 0.0, 0.0, 0
        for op in plan.ops:
            f = float(op.get('flops_per_image', 0)) * B
            all_flops_step += f
            if op['kind'] == 'conv':
                conv_launches += 1
                conv_flops_step += f
        conv_ms_per_launch = conv_ms / (ksteps * max(conv_launches, 1))
        achieved_tflops = conv_flops_step * ksteps / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0

        # ---- fp32-input variant of the same step (the reference's ToTensor type; 133 MB per batch instead of 33 MB)
        xf = [x.float().div_(255.0) for x in xs[:3]]
        for i in range(12):
            model(xf[i % 3])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(3000000)
        a.record()
        for i in range(20):
            model(xf[i % 3])
        b.record()
        torch.cuda.synchronize()
        fp32_in_ms = a.elapsed_time(b) / 20

        # ---- end to end through the public API with HOST buffers (H2D of the batch + D2H of the head every step),
        #      double-buffered on a copy stream so the transfer of step i+1 overlaps the forward of step i
        # host images are uint8 NCHW, what the reference's do_detect receives from PIL/cv2 before its CPU-side
        # float().div(255) (src/nets2_utils.py:346-352); Darknet.forward scales them inside the first-layer kernel
        host_in = [torch.randint(0, 256, (B, 3, IMG, IMG), dtype=torch.uint8).pin_memory() for _ in range(2)]
        host_out = [torch.empty(B, y.shape[1], y.shape[2], y.shape[3]).pin_memory() for _ in range(2)]
        dev_in = [torch.empty(B, 3, IMG, IMG, dtype=torch.uint8, device=device) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=device)
        out_stream = torch.cuda.Stream(device=device)
        main_stream = torch.cuda.current_stream()
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        produced = [torch.cuda.Event() for _ in range(2)]
        in_flight = [None, None]
        d2h_done = [torch.cuda.Event() for _ in range(2)]

        def e2e_loop(nsteps):
            with torch.cuda.stream(copy_stream):
                dev_in[0].copy_(host_in[0], non_blocking=True)
                ready[0].record(copy_stream)
            for i in range(nsteps):
                cur, nxt = i % 2, (i + 1) % 2
                if i + 1 < nsteps:
                    with torch.cuda.stream(copy_stream):
                        if i >= 1:
                            copy_stream.wait_event(consumed[nxt])
                        dev_in[nxt].copy_(host_in[nxt], non_blocking=True)
                        ready[nxt].record(copy_stream)
                main_stream.wait_event(ready[cur])
                if in_flight[cur] is not None:
                    d2h_done[cur].synchronize()  # the copy of two steps ago (finished long since): its block may be reused
                    in_flight[cur] = None
                out = model(dev_in[cur])
                consumed[cur].record(main_stream)
                produced[cur].record(main_stream)
                with torch.cuda.stream(out_stream):  # device->host read of the head, off the compute stream
                    out_stream.wait_event(produced[cur])
                    host_out[cur].copy_(out, non_blocking=True)
                    d2h_done[cur].record(out_stream)
                # keep the head alive until the slot is reused two steps later (its copy has long finished by then)
                # instead of Tensor.record_stream: the allocator's per-malloc event bookkeeping for stream-recorded
                # blocks cost 0.2-0.9 ms of HOST time per step on some hosts (tools/e2e_probe.py)
                in_flight[cur] = out
            torch.cuda.synchronize()

        # raw host->device rate of this host for the same pinned buffer (the end-to-end loop is bound by it whenever
        # 33 MB / rate exceeds the forward time): reported next to the end-to-end value
        with torch.cuda.stream(copy_stream):
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dev_in[0].copy_(host_in[0], non_blocking=True)
            h0.record(copy_stream)
            for _ in range(5):
                dev_in[0].copy_(host_in[0], non_blocking=True)
            h1.record(copy_stream)
        torch.cuda.synchronize()
        h2d_gbs = 5 * host_in[0].numel() / (h0.elapsed_time(h1) * 1e-3) / 1e9

        e2e_loop(8)
        barrier()
        t0 = time.perf_counter()
        e2e_loop(K)
        e2e_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e_s], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        e2e_value = B * K * world / e2e_s

    # The timed region is K steps of < 1 ms at full boost clocks (burst conditions), so the roofline denominator is the
    # BURST bf16 peak; the fraction of the sustained peak is printed beside it.
    traffic, traffic_src = profiled_traffic()
    whole_tflops = flops_img * value / world / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
        "warmup": args.warmup, "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "yolov2-voc-416 (seed-0 default init) 40% filter-pruned, filters physically removed, "
                               "forward", "batch_per_gpu": B, "global_batch": B * world, "parallelism": "dp%d" % world,
                   "prune": "quick_filter_prune 40%% -> %d/%d filters kept" % (sum(int(k.numel()) for k in keep),
                                                                            sum(m.shape[0] for m in masks)),
                   "algorithmic_gflop_per_image": flops_img / 1e9,
                   "input": "uint8 NCHW images resident in HBM (x/255 in the first-layer kernel)",
                   "l2": "inputs larger than L2: %d rotating %.0f MB batches" % (len(xs), input_mb),
                   "timing": "CUDA events on the launching stream, launch queue primed by a 1.5 ms spin kernel"},
        "clocks": clocks,
        "step_ms": {"median": statistics.median(step_ms), "min": min(step_ms), "max": max(step_ms),
                    "median_x_steps_ms": statistics.median(step_ms) * K, "total_ms": my_ms_per_step * K},
        "rejected_attempts": rejected_attempts,
        "value_fp32_input": {"images_per_s": B / (fp32_in_ms * 1e-3), "ms_per_step": fp32_in_ms,
                             "note": "same step fed the reference's float32 [0,1] tensor (133 MB per batch)"},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 3 * IMG * IMG,
                "d2h_bytes_per_step": int(y.numel() * 4),
                "input": "uint8 NCHW images in pinned host memory (do_detect's input type), x/255 on the device",
                "host_cpus_bound_to_gpu_numa_node": bound_cpus, "h2d_gbs_measured": h2d_gbs,
                "h2d_bound_images_per_s": h2d_gbs * 1e9 / (3 * IMG * IMG),
                "note": "double-buffered: step time = max(H2D of the next batch, forward, D2H); on this host the H2D "
                        "of the 33 MB batch is the longest of the three when h2d_bound_images_per_s < value"},
        "gpu_launches": plan.num_launches * K,
        "roofline": {"bound": "tensor", "kernel": "conv_gemm_tcgen05_kernel + conv_gemm_tcgen05_pair_kernel (the conv GEMM "
                     "launches of a forward)", "achieved": achieved_tflops, "peak": peaks['bf16'], "unit": "TFLOP/s",
                     "frac": achieved_tflops / peaks['bf16'] if peaks['bf16'] else None,
                     "frac_of_sustained": achieved_tflops / peaks['bf16_sustained'] if peaks['bf16_sustained'] else None,
                     "peak_source": "%s bf16_tflops (burst: the timed region is %.0f ms at boost clocks)" % (
                         peaks['source'], elapsed_ms),
                     "traffic": traffic, "traffic_unit": "bytes of DRAM traffic per launch (ncu --set full, %s)" % traffic_src,
                     "avg_launch_ms": conv_ms_per_launch, "launches_per_step": conv_launches,
                     "how": "eager forwards on the launching stream with the launch queue primed by a spin kernel; every "
                            "launch is issued %d times back to back between its two CUDA events and the interval divided "
                            "by %d (an event pair costs a few microseconds, comparable to the short kernels); the timed "
                            "steps themselves replay a CUDA graph" % (PER_OP_REPS, PER_OP_REPS),
                     "algorithmic_gflop_per_step": conv_flops_step / 1e9,
                     "kernel_share_of_step": conv_ms / max(conv_ms + other_ms, 1e-9),
                     "whole_net_tflops": whole_tflops, "whole_net_frac": whole_tflops / peaks['bf16'],
                     "whole_net_frac_of_sustained": whole_tflops / peaks['bf16_sustained'],
                     "whole_net_algorithmic_gflop_per_step": all_flops_step / 1e9},
        "whole_net_tflops": whole_tflops,
    }
    if per_rank is not None:
        line["per_rank"] = per_rank
    if not args.no_eval:
        with torch.no_grad():
            line["eval_pipeline"] = time_eval_pipeline(model, device, B, rank, world, "default-init worst case")
            kn = kn_model(device)
            line["eval_pipeline_kn"] = time_eval_pipeline(kn, device, B, rank, world, "KN-init, dense un-pruned network")
            if world == 1 and rank == 0:
                with torch.enable_grad():
                    line["next_rows"] = time_scorer_and_loss(kn, device, B)
            del kn
    if world > 1 and not args.no_retrain:
        torch.cuda.empty_cache()
        line["dp_retrain"] = time_dp_retrain(device, B, rank, world)
    if rank == 0:
        line["per_op_ms"] = {k: round(statistics.median(v), 4) for k, v in per_layer.items()}
        if world == 1:
            with torch.no_grad():
                line["detect_stages"] = time_detect_stages(model, device, B)
            torch.manual_seed(0)
            dense = mc.Darknet(mc.write_yolov2_voc_cfg()).to(device).eval()
            line["mask"] = time_masks(dense, peaks)
            if not args.no_dense:
                with torch.no_grad():
                    for i in range(4 * len(xs)):
                        dense(xs[i % len(xs)])
                    torch.cuda.synchronize()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda._sleep(3000000)
                    a.record()
                    for i in range(20):
                        dense(xs[i % len(xs)])
                    b.record()
                    torch.cuda.synchronize()
                    ms = a.elapsed_time(b) / 20
                    dplan = compile_darknet(dense)
                    dper = {}
                    for i in range(5):
                        evs = []
                        torch.cuda._sleep(8000000)
                        dplan.run(xs[i % len(xs)], events=evs, repeat=PER_OP_REPS)
                        torch.cuda.synchronize()
                        for op, e0_, e1_ in evs:
                            dper.setdefault(op['name'], []).append(e0_.elapsed_time(e1_) / PER_OP_REPS)
                tfl = DENSE_GFLOP_PER_IMAGE * B / ms
                line["dense"] = {"images_per_s": B / (ms * 1e-3), "tflops": tfl, "frac_of_bf16_burst": tfl / peaks['bf16'],
                                 "frac_of_bf16_sustained": tfl / peaks['bf16_sustained'], "ms_per_step": ms,
                                 "per_op_ms": {k: round(statistics.median(v), 4) for k, v in dper.items()}}
            dense_state = {k: v.detach().cpu() for k, v in dense.state_dict().items()}
            del dense
            if not args.no_library:
                line["gpu_library_baseline"] = time_library_baseline(model, device, B, xf[0])
            if not args.no_retrain:
                del xf
                torch.cuda.empty_cache()
                line["retrain"] = time_retrain(device, peaks, B)
            if not args.no_cpu_baseline:
                state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
                ips, sps, _ = cpu_forward_sample(state, model.blocks, CPU_SAMPLE_BATCH, 6, 1)
                line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": torch.get_num_threads(),
                                        "kind": "port", "sample": "6 forwards of batch %d of the same pruned network "
                                        "(oracle port of the reference PyTorch CPU path)" % CPU_SAMPLE_BATCH,
                                        "legs": cpu_stage_legs(dense_state, model.blocks, model.anchors)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

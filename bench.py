#!/usr/bin/env python
"""bench.py -- RGB+IR pairs/s of the yolov5l-CFTx3 two-stream forward on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 32] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one forward of the hot path over one batch of synthetic 640x640 RGB+IR pairs
(config 2 of BASELINE.json: yolov5l_fusion_transformerx3 FLIR cfg, bf16, batch 32 per GPU).
Prints ONE JSON line on rank 0:
  value      whole-job pairs/s, inputs resident in HBM, K steps timed with CUDA events between
             barrier+synchronize on both sides, max over ranks (weak scaling: batch 32 per GPU)
  e2e        the same metric through the public API from HOST buffers: every step copies the loader's
             uint8 [B,6,H,W] wire-format batch from pinned host memory to the device and reads the decoded
             detections z back to the host, all inside the timed region
  roofline   the dominant kernel (tcgen05 implicit-GEMM conv/linear): the algorithmic FLOPs that kernel executes per
             step / time it is resident per step -- the union of the in-kernel %globaltimer spans of its launches
             inside a CUDA-graph replay (the timed mode), measured live -- against the measured sustained bf16 peak
  cpu_baseline  the reference's forward on the host cores on a bounded sample (batch-1 forwards of the same graph / size):
             the UNMODIFIED reference's own modules when its tree -- or the copy staged into oracle/_ref by
             oracle/stage_reference.py, which travels with the built tree -- is importable (kind "reference"), else the
             oracle's restatement of it (kind "port")
--impl reference: the same CPU forward as a whole arm (fastest of 8/16/32/all host threads, measured first) -- rank 0 only.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "RGB+IR pairs/sec yolov5l-CFTx3 fwd @640"
CFG_NAME = "yolov5l_fusion_transformerx3_FLIR_aligned"
H = W = 640


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons, power, rows = [], [], set(), [], []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                rows.append((float(f[1]), float(f[2]), float(f[3])))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # the sampler runs from the first warm-up step to the end of the timed loop; "under load" = power well
        # above idle (the timed loop alone can be shorter than one 200 ms sampling period)
        pmax = max((r[2] for r in rows), default=0.0)
        load = [r for r in rows if r[2] >= 0.6 * pmax] or rows
        sm, smax, power = [r[0] for r in load], [r[1] for r in load], [r[2] for r in load]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(rows), "samples_under_load": len(load),
                "reasons": sorted(reasons)}


def host_threads():
    """Threads the process may actually use (cgroup/affinity aware; os.cpu_count() over-subscribes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def fused_state(sd, eps):
    """Model.fuse() (models/yolo_test.py:296-304, utils/torch_utils.py:181-201) applied to a state dict: the reference's
    inference entry points run the fused model (attempt_load -> fuse, models/experimental.py:113-134)."""
    import torch
    out = {}
    for k, v in sd.items():
        if ".bn." in k:
            continue
        if k.endswith("conv.weight") and k.replace("conv.weight", "bn.weight") in sd:
            p = k[:-len("conv.weight")]
            scale = sd[p + "bn.weight"] / torch.sqrt(sd[p + "bn.running_var"] + eps)
            out[k] = v * scale.view(-1, 1, 1, 1)
            out[p + "conv.bias"] = sd[p + "bn.bias"] - sd[p + "bn.running_mean"] * scale
        else:
            out[k] = v
    return out


def best_thread_count(fwd, candidates=None):
    """The reference arm may use every host thread, but PyTorch's CPU kernels do not always scale to all of them
    (a batch-1 forward on 64 threads can be slower than on 16): time one forward per candidate thread count and keep the
    fastest, so that the CPU baseline is the best the host can do, not the most threads it can occupy."""
    import torch
    top = host_threads()
    cands = candidates or sorted({t for t in (8, 16, 32, top) if t <= top} | {top})
    best_t, best_dt = top, None
    for t in cands:
        torch.set_num_threads(t)
        fwd()                                        # warm-up at this thread count
        t0 = time.perf_counter()
        fwd()
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best_t, best_dt = t, dt
    torch.set_num_threads(best_t)
    return best_t


def cpu_forward(batch, force_port=False):
    """The reference's CPU forward of the headline graph on a seeded batch: (callable, kind, description).  `kind` is
    "reference" when the UNMODIFIED reference's own modules run it (the tree, or its staged copy oracle/_ref --
    oracle/stage_reference.py; fused and eval as test.py:66-68 / detect_twostream.py:40-41 run them, fp32 on the CPU),
    else "port": the oracle's restatement of the same forward (oracle/cft_oracle.py)."""
    import torch
    from oracle import cft_oracle as O
    from oracle import ref_shim
    pkg = importlib.import_module("multispectral-object-detection_b200")
    cfg = pkg.named_config(CFG_NAME)
    x, x2 = O.make_inputs(batch, H, W, seed=1)
    if ref_shim.available() and not force_port:
        try:
            yt = ref_shim.import_reference()
            rm = yt.Model(ref_shim.reference_yaml(CFG_NAME), ch=3)
            rm.load_state_dict(O.init_state(cfg, seed=0), strict=True)
            rm = rm.float().fuse().eval()

            def fwd_ref():
                with torch.no_grad():
                    return rm(x, x2)
            fwd_ref()
            return fwd_ref, "reference", "the reference's own modules (models/yolo_test.py Model, fused, eval), fp32, PyTorch CPU"
        except Exception as e:       # an unimportable reference tree must not take the baseline down with it
            sys.stderr.write(f"bench: reference modules unavailable ({type(e).__name__}: {e}); timing the oracle port\n")
    sd = fused_state(O.init_state(cfg, seed=0), O.BN_EPS)       # BN folded, as the reference's inference path runs
    return (lambda: O.forward(sd, cfg, x, x2)), "port", "fp32 oracle port of the reference forward, PyTorch CPU"


def cpu_baseline(seconds_budget=20.0, batch=1, force_port=False):
    """The reference forward on the host cores (see cpu_forward): batch-1 forwards of the headline graph."""
    import torch
    fwd, kind, what = cpu_forward(batch, force_port)
    best_thread_count(fwd)                                     # also the warm-up
    times, t_start = [], time.perf_counter()
    while len(times) < 3 or (time.perf_counter() - t_start < seconds_budget and len(times) < 50):
        t0 = time.perf_counter()
        fwd()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": batch / med, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{len(times)} forwards of batch {batch} @ {H}x{W} ({what}, median {med * 1e3:.0f} ms; "
                      f"fastest of 8/16/32/{host_threads()} threads)"}


def dump_outputs(out_dir, arrays, budget=64 << 20):
    """Write each tensor of `arrays` as <out_dir>/<name>.npy in float32.  When they exceed `budget` bytes together, every
    array keeps the same seeded subset of its rows (dim 1), so that two runs with the same arguments stay comparable."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * 4 for t in arrays.values())
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        if total > budget:
            keep = max(1, t.shape[1] * budget // total)
            idx = torch.randperm(t.shape[1], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[:, idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def run_reference(args, rank):
    if rank != 0:
        return
    import torch
    b = 1                                             # bounded sample per step
    fwd, kind, what = cpu_forward(b)
    best_thread_count(fwd)                            # fastest of 8/16/32/all host threads; doubles as warm-up
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        fwd()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        z, _ = fwd()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"z": z})
    v = b * steps / dt
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{CFG_NAME} forward, {H}x{W}, {what}, bounded sample: batch {b} per step"},
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": kind,
                             "sample": f"{steps} forwards of batch {b} @ {H}x{W}"},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def extra_rooflines(pkg, model, B, peaks, dev):
    """The two kernel classes BASELINE.json's north_star quotes targets for, measured in isolation on this GPU with an
    L2 flush (256 MiB memset) between timed iterations, median of 5:
      c3_1x1_hbm   the 1x1 convolutions of the P2/P3 C3 stacks (AI 32-128 flop/B: HBM-bound) -- algorithmic bytes
                   (input + output + weights, bf16) / time, against the measured HBM peak
      cft_block_*  one whole CFT block (tokeniser, 8 x [LN, QKV GEMM, attention, out-proj, LN, MLP], ln_f) per scale --
                   algorithmic FLOPs (24576 d^2 + 524288 d per pair, SURVEY.md section 8d) / time, against the
                   measured sustained bf16 peak; `attention_core_hbm` is the attention kernel alone, which is HBM-bound
                   (AI = 64 flop/B): Q, K, V read + O written once per (image, head)."""
    import math
    import torch
    ops = pkg.ops
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n=5):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            flush.zero_()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    out = {}
    tot_b = tot_ms = 0.0
    shapes = []
    for cin, cout, hw, count in ((128, 128, 160, 2), (64, 64, 160, 3), (256, 256, 80, 2), (128, 128, 80, 9)):
        x = torch.randn(B, cin, hw, hw, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        wp, bp = ops.pack_conv_weight(torch.randn(cout, cin, 1, 1) / math.sqrt(cin), torch.zeros(cout), None, device=dev)
        y = ops.conv2d(x, wp, bp, 1, 1, 1, cout=cout)
        ms = timed(lambda: ops.conv2d(x, wp, bp, 1, 1, 1, out=y, cout=cout))
        byts = 2.0 * (B * hw * hw * (cin + cout) + cin * cout)
        shapes.append({"shape": f"{cin}->{cout} 1x1 @{hw}x{hw}", "us": round(ms * 1e3, 1), "gbs": round(byts / ms / 1e6, 1),
                       "per_c3_stack_stream": count})
        tot_b += byts * count
        tot_ms += ms * count
        del x, y
    ach = tot_b / tot_ms / 1e6
    out["c3_1x1_hbm"] = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": ach / peaks["hbm_gbs"], "shapes": shapes,
                         "note": "launch-count-weighted over the 1x1 convs of the P2 (n=3) and P3 (n=9) C3 stacks"}
    gpts = []
    for i, m in enumerate(model.model):
        if not isinstance(m, pkg.GPT):
            continue
        d = m.n_embd
        hw = {256: 80, 512: 40, 1024: 20}.get(d, 40)
        rgb = torch.randn(B, d, hw, hw, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        ir = torch.randn(B, d, hw, hw, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        gpts.append((m, rgb, ir))
        with torch.no_grad():                       # graph replay, like the forward itself (eager launches are host-bound)
            m.tokens(rgb, ir)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                m.tokens(rgb, ir)
            ms = timed(gr.replay, n=5)
        flops = (24576.0 * d * d + 524288.0 * d) * B
        ach = flops / ms / 1e9
        out[f"cft_block_d{d}"] = {"bound": "tensor", "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                                  "frac": ach / peaks["tflops_sustained"], "ms": round(ms, 4), "layer": i}
    pkg._lib.prof_enable(True)              # per-launch CUDA events: a separate pass, they would perturb the timing above
    with torch.no_grad():
        for m, rgb, ir in gpts:
            m.tokens(rgb, ir)
    torch.cuda.synchronize()
    prof = pkg._lib.prof_get()
    pkg._lib.prof_enable(False)
    a_ms, a_n = prof["attention"]
    if a_n:
        # 8 attention launches per block and scale; bytes per launch: Q, K, V read + O written = 4 * (B*128) * d * 2 B
        byts = sum(4.0 * B * 128 * d * 2 for d in (256, 512, 1024)) / 3.0
        per_launch_ms = a_ms / a_n
        ach = byts / per_launch_ms / 1e6
        out["attention_core_hbm"] = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                     "frac": ach / peaks["hbm_gbs"], "us_per_launch": round(per_launch_ms * 1e3, 2),
                                     "note": "mean over the three scales; per-launch CUDA events (includes launch gaps)"}
    try:        # the step after the forward: batched NMS of a batch-B z (synthetic boxes, reference defaults 0.25 / 0.45)
        g = torch.Generator().manual_seed(3)
        pr = torch.rand(B, 25200, 8, generator=g)
        pr[..., :2] *= float(H)
        pr[..., 2:4] = 20.0 + 100.0 * pr[..., 2:4]
        pr = pr.to(dev)
        det = torch.zeros(B, 300, 6, device=dev)
        cnt = torch.zeros(B, dtype=torch.int32, device=dev)
        ws = torch.empty(B * 25200, dtype=torch.int64, device=dev)
        ms = timed(lambda: pkg.nms_batched(pr, out=det, counts=cnt, workspace=ws))
        out["nms_batch"] = {"us": round(ms * 1e3, 1), "rows_per_image": 25200, "kept_mean": float(cnt.float().mean()),
                            "note": "cft_nms, one launch for the batch; uniform random boxes"}
    except Exception as e:
        out["nms_batch"] = {"error": repr(e)[:200]}
    return out


def conv_kernel_busy_ms(pkg, model, x_rgb, x_ir, dev, reps=5):
    """Time the dominant kernel occupies the GPU inside ONE step of the TIMED mode (CUDA-graph replay, RGB / IR branches on
    two streams, programmatic dependent launch): every cft_conv2d launch of a freshly captured graph reports
    {first CTA start, last CTA end} in %globaltimer ns (cft_debug_conv_spans); the union of those intervals is the time at
    least one launch of the kernel is resident, <= the step time by construction.  Returns (union ms, sum of spans ms,
    launches, graph replay ms), medians over `reps` replays."""
    import ctypes
    import torch
    lib = pkg._lib.lib()
    MAXL = 1024
    buf = torch.zeros(2 * MAXL, dtype=torch.int64, device=dev)
    init = torch.zeros(2 * MAXL, dtype=torch.int64)
    init[0::2] = torch.iinfo(torch.int64).max
    init = init.to(dev)
    stream = torch.cuda.Stream(dev)
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    pkg._lib.check(lib.cft_debug_conv_spans(ctypes.c_void_p(buf.data_ptr()), MAXL), "cft_debug_conv_spans")
    try:
        with torch.no_grad(), torch.cuda.graph(g, stream=stream):
            model(x_rgb, x_ir)
    finally:
        pkg._lib.check(lib.cft_debug_conv_spans(ctypes.c_void_p(0), 0), "cft_debug_conv_spans")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    unions, sums, replays, n = [], [], [], 0
    for _ in range(reps + 1):
        buf.copy_(init)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            e0.record(stream)
            g.replay()
            e1.record(stream)
        torch.cuda.synchronize()
        t = buf.cpu().view(-1, 2)
        t = t[t[:, 1] > 0]
        n = int(t.shape[0])
        iv = sorted(zip(t[:, 0].tolist(), t[:, 1].tolist()))
        busy, cs, ce = 0, iv[0][0], iv[0][1]
        for a, b in iv[1:]:
            if a > ce:
                busy += ce - cs
                cs, ce = a, b
            else:
                ce = max(ce, b)
        busy += ce - cs
        unions.append(busy / 1e6)
        sums.append(float((t[:, 1] - t[:, 0]).sum()) / 1e6)
        replays.append(e0.elapsed_time(e1))
    med = lambda v: sorted(v[1:])[len(v[1:]) // 2]          # the first replay of a fresh graph is a warm-up
    del g
    return med(unions), med(sums), n, med(replays)


def gpu_eager_baseline(pkg, cfg, B, dev, steps=5):
    """The existing GPU path on the same device, a reported baseline beside cpu_baseline (never on the product path):
    the UNMODIFIED reference's own modules in PyTorch eager (cuDNN / cuBLAS), `attempt_load`-style fused and `.half()` as
    test.py:66-68,107 / detect_twostream.py:40-41,72 run them -- when the reference tree (or its staged copy
    oracle/_ref, oracle/stage_reference.py) is present; else the oracle's restatement of the same op sequence with its
    tensors on the GPU (bf16, channels_last)."""
    import torch
    from oracle import cft_oracle as O
    from oracle import ref_shim
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, 3, H, W, generator=g)
    x2 = torch.rand(B, 3, H, W, generator=g)
    if ref_shim.available():
        yt = ref_shim.import_reference()
        rm = yt.Model(ref_shim.reference_yaml(CFG_NAME), ch=3)
        rm.load_state_dict(O.init_state(cfg, seed=0), strict=True)
        rm = rm.float().fuse().eval().to(dev).half()
        x, x2 = x.to(dev).half(), x2.to(dev).half()
        fwd = lambda: rm(x, x2)
        kind = "the reference's own modules, PyTorch eager (cuDNN/cuBLAS), fused, .half() as test.py:66-68, same GPU"
    else:
        sd = {}
        for k, v in fused_state(O.init_state(cfg, seed=0), O.BN_EPS).items():
            if v.is_floating_point():
                v = v.to(dev, torch.bfloat16)
                if v.dim() == 4:
                    v = v.contiguous(memory_format=torch.channels_last)
            else:
                v = v.to(dev)
            sd[k] = v
        x = x.to(dev, torch.bfloat16).contiguous(memory_format=torch.channels_last)
        x2 = x2.to(dev, torch.bfloat16).contiguous(memory_format=torch.channels_last)
        fwd = lambda: O.forward(sd, cfg, x, x2)
        kind = "pytorch eager (cuDNN/cuBLAS) restatement of the reference op sequence, BN fused, bf16 channels_last, same GPU"
    with torch.no_grad():
        for _ in range(2):
            fwd()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fwd()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del fwd, x, x2
    torch.cuda.empty_cache()
    return {"value": B / (ms / 1e3), "unit": "pairs/s", "ms_per_step": ms, "kind": kind,
            "sample": f"{steps} forwards of batch {B} @ {H}x{W}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=32, help="pairs per GPU per step (weak scaling)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cfg", default=CFG_NAME, help="graph (config name); the default is BASELINE.json's headline config 2; "
                    "yolov5x_fusion_transformerx3_FLIR_aligned = config 5")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--slots", type=int, default=2, help="engine slots (double-buffered copy pipeline)")
    ap.add_argument("--concurrent", action="store_true",
                    help="experiment: one compute stream per slot (batches overlap on the GPU); measured: no gain")
    ap.add_argument("--no-eager-baseline", action="store_true",
                    help="skip the PyTorch-eager (cuDNN/cuBLAS) forward of the same graph on this GPU")
    ap.add_argument("--no-extras", action="store_true", help="skip the isolated C3-1x1 / CFT-block roofline measurements")
    ap.add_argument("--ncu-range", action="store_true",
                    help="after the measurements, run ONE eager step between cudaProfilerStart/Stop (for ncu "
                         "--profile-from-start off launch lists; numbers printed under ncu are never bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (z, float32) to DIR/z.npy; the inputs and weights are "
                         "seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("multispectral-object-detection_b200")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W_ = max(args.warmup, 3)
    K = args.steps
    B = args.batch

    cfg = pkg.named_config(args.cfg)
    torch.manual_seed(0)
    model = pkg.Model(cfg).eval()
    # random-init weights of the architecture with non-degenerate BN statistics / pos_emb (SURVEY.md §8d config 2)
    g = torch.Generator().manual_seed(2)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
            if isinstance(m, pkg.GPT):
                m.pos_emb.copy_(torch.randn(m.pos_emb.shape, generator=g) * 0.02)
    model = model.to(dev)

    gi = torch.Generator().manual_seed(1 + rank)
    x6_host = torch.randint(0, 256, (B, 6, H, W), dtype=torch.uint8, generator=gi).pin_memory()
    x6 = x6_host.to(dev)                       # inputs resident in HBM for the `value` measurement
    x_rgb, x_ir = x6[:, :3], x6[:, 3:]

    def step():
        return model(x_rgb, x_ir)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- warm-up (also builds packed weights) ----------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    with torch.no_grad():
        for _ in range(W_):
            z, _ = step()
    torch.cuda.synchronize()

    # ---------------- the serving executor: CUDA-graph replay + double-buffered copy pipeline ----------------
    engine = pkg.ForwardEngine(model, B, H, W, device=dev, slots=args.slots, use_graph=not args.no_graph,
                               concurrent=args.concurrent)
    launches_per_step = engine.launches_per_forward
    for s_ in range(engine.slots):
        engine.x_dev[s_].copy_(x6)
    for _ in range(2):
        for s_ in range(engine.slots):
            engine.run_resident(s_)
    torch.cuda.synchronize()

    # ---------------- timed region: K steps, device-resident inputs ----------------
    # Step i replays slot (i mod slots)'s graph; all slots share one compute stream unless --concurrent (an experiment:
    # batches overlapping on the GPU bought nothing measurable and cost 2-3 % end to end, profiles/r01_timeline.md).
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cur = torch.cuda.current_stream()
    barrier()
    e0.record(cur)
    for st in engine.computes:
        st.wait_event(e0)
    for i in range(K):
        z_last = engine.run_resident(i % engine.slots)
    for st in engine.computes:
        cur.wait_stream(st)
    e1.record(cur)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"z": z_last})       # before later replays of the slot overwrite it
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * K / (ms_max / 1e3)

    # ---------------- end-to-end: host uint8 batch -> device -> forward -> z back to host ----------------
    # Public API call = ForwardEngine.submit()/collect(): every step copies the loader's uint8 [B,6,H,W] batch from
    # pinned host memory and reads the decoded detections back; copies of neighbouring steps overlap the compute.
    def e2e_loop(n):
        for _ in range(n):
            if len(engine._pending) == engine.slots:
                engine.collect()
            engine.submit(x6_host)
        engine.drain()

    e2e_loop(3)
    barrier()
    e0.record(engine.compute)
    e2e_loop(K)                                   # drain() inside: every z is on the host when this returns
    for s_ in range(engine.slots):
        engine.compute.wait_event(engine.ev_free[s_])
    e1.record(engine.compute)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (float(t.item()) / 1e3)
    h2d = x6_host.numel() * x6_host.element_size()
    d2h = engine.z_host[0].numel() * engine.z_host[0].element_size()
    graph = engine.graphs[0]

    # ---------------- roofline of the dominant kernel (profiled eager pass, rank 0) ----------------
    roofline, kernel_ms = None, None
    if rank == 0:
        from oracle import cft_oracle as O       # FLOP model only (SURVEY.md §8d) -- nothing is executed
        peaks = load_peaks()
        flops_pair = O.conv_linear_flops(cfg, H, W)
        attn_core = sum(len(m_.trans_blocks) * 4.0 * 128 * 128 * m_.n_embd for m_ in model.model if isinstance(m_, pkg.GPT))
        # (1) per-kernel totals of one step: per-launch CUDA events only add up when launches are serialised, so this pass
        # walks the graph eagerly on ONE stream -- it feeds `kernel_ms_per_step` (shares), not the roofline
        two = model.two_streams
        model.two_streams = False
        pkg._lib.prof_enable(True)
        nprof = 3
        with torch.no_grad():
            for _ in range(nprof):
                step()
        torch.cuda.synchronize()
        prof = pkg._lib.prof_get()
        pkg._lib.prof_enable(False)
        model.two_streams = two
        kernel_ms = {k: round(v[0] / nprof, 4) for k, v in prof.items() if v[1]}
        # (2) the roofline of the dominant kernel, measured in the TIMED mode: in-kernel %globaltimer spans of every conv /
        # linear launch inside a CUDA-graph replay (two streams, PDL) -> time the kernel is resident per step
        busy_ms, span_sum_ms, conv_n, replay_ms = conv_kernel_busy_ms(pkg, model, x_rgb, x_ir, dev)
        # FLOPs that kernel executes: conv + linear FLOPs of the graph (SURVEY.md section 8d) minus what other kernels run:
        # the attention cores, the fused uint8 Focus layers (cft_focus_tcgen05_kernel) and the Linear layers of the CFT
        # blocks that run inside the one-launch cft_gpt_block kernel
        c0 = model.model[0].conv.conv.out_channels
        focus_flops = 2 * 2.0 * (H // 2) * (W // 2) * c0 * 12 * 9
        blk_flops = 0.0
        for m_ in model.model:
            if isinstance(m_, pkg.GPT) and m_.fused_block and m_.n_embd <= m_.fused_block_max_d \
                    and pkg.ops.gpt_block_supported(B, m_.n_embd, m_.h, 2 * m_.vert_anchors * m_.horz_anchors):
                blk_flops += 24576.0 * m_.n_embd * m_.n_embd
        conv_flops_step = (flops_pair - attn_core - focus_flops - blk_flops) * B
        achieved = conv_flops_step / (busy_ms / 1e3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r01_conv_dram_traffic.json")
        if os.path.isfile(tpath):          # summed dram__bytes_{read,write} of the kernel's launches in one step (ncu)
            traffic = json.load(open(tpath)).get("dram_bytes_per_step")
        roofline = {"kernel": "cft_conv_tcgen05_kernel", "bound": "tensor", "achieved": achieved,
                    "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops_sustained"],
                    "peak_source": peaks["source"] + " sustained bf16", "traffic": traffic,
                    "traffic_note": "sum over the kernel's launches of one step (profiles/r01_conv_dram_traffic.json, ncu)",
                    "launches_per_step": conv_n, "ms_per_step_in_kernel": busy_ms,
                    "how": "union of the [first CTA start, last CTA end] %globaltimer spans of the kernel's launches inside "
                           "one CUDA-graph replay of the step (the timed mode: two streams, PDL); "
                           f"sum of spans {span_sum_ms:.3f} ms, replay {replay_ms:.3f} ms",
                    "algorithmic_gflop_per_step": conv_flops_step / 1e9,
                    "gflop_per_step_in_other_kernels": {"attention_core": attn_core * B / 1e9, "focus_fused": focus_flops * B / 1e9,
                                                        "cft_gpt_block": blk_flops * B / 1e9},
                    "whole_forward_tensor_frac": (flops_pair * value / world) / (peaks["tflops_sustained"] * 1e12)}

    extras = None
    if rank == 0 and not args.no_extras and args.cfg == CFG_NAME:
        try:
            extras = extra_rooflines(pkg, model, B, load_peaks(), dev)
        except Exception as e:          # never lose the headline line over a side measurement
            extras = {"error": repr(e)[:300]}

    eager = None
    if rank == 0 and world == 1 and not args.no_eager_baseline and args.cfg == CFG_NAME:
        try:
            eager = gpu_eager_baseline(pkg, cfg, B, dev)
        except Exception as e:          # a side measurement must never cost the headline line
            eager = {"error": repr(e)[:300]}

    if args.ncu_range and rank == 0:
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        with torch.no_grad():
            step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    if world > 1:
        dist.barrier()
    if rank == 0:
        cpu = None
        if not (args.no_cpu_baseline or world > 1 or args.cfg != CFG_NAME):      # rank 0 at N = 1 only
            try:
                cpu = cpu_baseline()
            except Exception as e:      # a reported baseline must never cost the measured line
                sys.stderr.write(f"bench: cpu_baseline with the reference modules failed ({type(e).__name__}: {e}); oracle port\n")
                cpu = cpu_baseline(force_port=True)
        if cpu is not None and eager is not None:
            cpu["gpu_eager_same_box"] = eager      # the existing GPU path (PyTorch eager, cuDNN / cuBLAS) beside the CPU number
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.cfg} forward (eval, BN folded), batch {B} per GPU @ {H}x{W}, nc={cfg['nc']}",
                       "global_batch": B * world, "parallelism": f"dp{world} (pairs sharded, no data-path collective)",
                       "l2": "working set (inputs 79 MB + weights 412 MB + activations > 5 GB per step) >> 126 MB L2",
                       "launch": "cuda-graph replay" if graph is not None else "eager",
                       "batches_in_flight": len(engine.computes)},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches_per_step * K,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "kernel_ms_per_step": kernel_ms,
            "rooflines_extra": extras, "gpu_eager_baseline": eager,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- PartialConv U-Net (ImageFillOrigin) 512x512 images/sec, forward + backward (+ SGD update).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # B200 path: also save what the last timed step computed

Prints ONE JSON line (rank 0).  Workload = BASELINE.json configs[2] ("image_inpainting.py PartialConv UNet
@512x512 batch=8, 1xB200 fwd+bwd bf16"), the configuration the headline metric is quoted on; weak scaling
(batch 8 per GPU, gradients all-reduced over NCCL).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The driver reads ONE JSON line from stdout.  Libraries print there too (NCCL's version banner under torchrun, the reference's
# constructors): keep a handle on the real stdout for that line and point fd 1 at stderr for everything else.
_REAL_STDOUT = sys.stdout


def _isolate_stdout():
    """(script entry only) keep a handle on the real stdout for the JSON line; fd 1 -> stderr for every library underneath"""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "PartialConv UNet 512x512 images/sec (fwd+bwd)"
PER_GPU_BATCH = 8
HW = 512
FWD_GFLOP_PER_IMAGE = 75.94        # feature convs only, SURVEY 8d (mask convs are a box sum: 0 FLOPs)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="unet", choices=["unet", "textseg", "xception"],
                    help="unet = BASELINE configs[2]/[4] (the headline metric); textseg = configs[1]; xception = configs[3]")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-layers", action="store_true", help="print a per-layer CUDA-event table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="B200 path only: after the timed steps, write what the last one computed to DIR/<name>.npy "
                         "(see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs saves the outputs of the b200 path")
    return args


# --------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in a side process during the timed region)
# --------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # "under load" = upper half of the samples (the sampler also sees the idle edges)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU baseline: the reference's algorithm on the host cores (oracle port of models/image_inpainting.py)
# --------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may actually use: CPU affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    n = min(n, max(1, q // int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())))
        except Exception:  # noqa: BLE001
            pass
    return max(1, n)


def pick_threads():
    """oneDNN convolutions stop scaling (and can collapse) when the pool is far wider than the machine can feed:
    time one representative layer at a few pool sizes and keep the fastest."""
    import torch
    import torch.nn.functional as F
    cores = usable_cores()
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | {min(cores, 8)})
    x = torch.randn(1, 192, 256, 256); w = torch.randn(64, 192, 3, 3)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        F.conv2d(x, w, padding=1)
        t0 = time.perf_counter()
        for _ in range(2):
            F.conv2d(x, w, padding=1)
        t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best, cores


def cpu_reference_steps(steps, warmup, batch=1, seed=0, workload="unet"):
    """fwd + bwd + SGD of the workload's network on the host cores, computed by the oracle's functional restatement of the
    reference (same ATen ops in the same order; pinned bit-exactly by tests/golden).  Returns (images_per_sec, ms_per_step,
    cores, kind)."""
    import torch

    from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks

    cores, avail = pick_threads()
    torch.manual_seed(seed)
    x = torch.randn(batch, 3, HW, HW)
    mask = torch.from_numpy(random_hole_masks(batch, HW, HW, seed=seed))
    xin = x * mask
    kind = "port"
    if workload != "unet":
        import contextlib
        import io
        cls = {"textseg": "TextSegament", "xception": "XceptionTextSegment"}[workload]
        with contextlib.redirect_stdout(io.StringIO()):
            from oracle import seg_torch as OS                         # cpu_baseline leg: allowed importer of oracle/
            from oracle.pconv_torch import clone_state_dict
            from text_segmentation_image_inpainting_b200.models import text_segmentation as MT
            sd = clone_state_dict(getattr(MT, cls)().state_dict(), requires_grad=True)
            params = [v for v in sd.values() if v.requires_grad]
            fwd = lambda: OS.NETWORKS[cls](sd, x)                          # noqa: E731
    else:
        from oracle import pconv_torch as O                       # cpu_baseline leg: allowed importer of oracle/
        from text_segmentation_image_inpainting_b200.models.image_inpainting import ImageFillOrigin
        skeleton = ImageFillOrigin()                               # parameter names / shapes / default init only
        sd = O.clone_state_dict(skeleton.state_dict(), requires_grad=True)
        params = [v for v in sd.values() if v.requires_grad]
        fwd = lambda: O.image_fill_origin(sd, xin, mask, training=True)   # noqa: E731
    opt = torch.optim.SGD(params, lr=2e-4, momentum=0.9, weight_decay=1e-4, nesterov=True)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = fwd().abs().mean()
        loss.backward()
        opt.step()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return batch * len(times) / total, 1e3 * total / len(times), f"{cores} of {avail} usable", kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                               # other ranks exit 0 without work
    ips, ms, cores, kind = cpu_reference_steps(args.steps, args.warmup, batch=1, workload=args.workload)
    cores_n = int(str(cores).split()[0])
    W = WORKLOADS[args.workload]
    line = {
        "impl": "reference", "metric": W["metric"], "value": ips, "unit": "images/sec", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": W["label"] + " 512x512 fwd+bwd+SGD, CPU (reference algorithm via the oracle port)",
                   "batch_per_step": 1, "note": f"each step is a bounded sample (1 image) of the batch-{W['batch']} workload"},
        "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": cores_n, "cores_note": cores, "kind": kind,
                         "sample": f"{args.steps} steps x 1 image @512x512 after {args.warmup} warm-up"},
        "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
WORKLOADS = {
    # BASELINE.json configs[2] (and [4] under torchrun): the headline
    "unet": {"metric": METRIC, "net": ("image_inpainting", "ImageFillOrigin"), "batch": 8, "fwd_gf": 75.94, "no_dgrad_gf": 1.23,
             "masks": True, "label": "ImageFillOrigin (PartialConv U-Net)"},
    # BASELINE.json configs[1]: text_segmentation.py MobileNetV2 encoder-decoder @512x512 batch 8
    "textseg": {"metric": "TextSegament (MobileNetV2+RFB) 512x512 images/sec (fwd+bwd)", "net": ("text_segmentation", "TextSegament"),
                "batch": 8, "fwd_gf": 90.67, "no_dgrad_gf": 0.0, "masks": False, "label": "TextSegament (DilatedMobileNetV2 x2 + RFB)"},
    # BASELINE.json configs[3]: Xception + atrous / ASP segmentation @512x512 batch 16 bf16
    "xception": {"metric": "XceptionTextSegment 512x512 images/sec (fwd+bwd)", "net": ("text_segmentation", "XceptionTextSegment"),
                 "batch": 16, "fwd_gf": 148.70, "no_dgrad_gf": 0.0, "masks": False, "label": "XceptionTextSegment (Xception + ASP)"},
}
KERNEL_OF = {"tc_fwd": "pconv_tc_tma_kernel<MODE=0> (+ conv_k2r 1x1 GEMM + k2r_combine for the RGB tail, s2d_kernel + the same kernel for the space-to-depth stem)",
             "tc_dgrad": "pconv_tc_tma_kernel<MODE=1> / pconv_tc_sp_kernel<MODE=1> (+ k2r_dbuild + 1x1 dgrad for the tail)",
             "tc_wgrad": "pconv_tc_wgrad_tma_kernel (+ k2r_dbuild + 1x1 wgrad for the tail, s2d_kernel + <64,4,true> for the stem)",
             "dw_fwd": "dw4_s1_kernel<FLIP=0> (dwconv.cu)", "dw_dgrad": "dw4_s1_kernel<FLIP=1> (dwconv.cu)", "dw_wgrad": "dw4_s1_wgrad_kernel (dwconv.cu)"}


def conv_flops(g):
    return 2.0 * g.n * g.ho * g.wo * g.cout * (g.cin // g.groups) * g.kh * g.kw


def conv_bytes(kind, g):
    """ALGORITHMIC HBM bytes of a depthwise launch (SURVEY 8d): one read of each input + one write of each output at the
    storage dtype; weights / the fp32 weight gradient are negligible."""
    xin, yout = g.n * g.cin * g.h * g.w * g.esz, g.n * g.cout * g.ho * g.wo * g.esz
    return float(xin + yout)          # fwd: read x, write y | dgrad: read dc, write dx | wgrad: read x, read dc


def layer_profile(ts, x, mask, peaks, verbose):
    """One instrumented EAGER step: CUDA events around every conv launch on the launching stream.
    Returns (roofline dict of the dominant family, per-family [work, ms, launches], per-family rooflines)."""
    import torch
    from text_segmentation_image_inpainting_b200 import _lib, ops

    rec = []
    ops.set_profile(rec)
    ts._fwd_bwd(x, mask)              # forward + backward only: no collective (rank 0 runs this alone)
    torch.cuda.synchronize()
    ops.set_profile(None)
    fam = {}
    rows = []
    for kind, g, s, e in rec:
        ms = s.elapsed_time(e)
        c = g.struct(None)
        dw = g.groups > 1 and g.groups == g.cin and g.cout == g.cin
        tc = bool(_lib.load().pcb_conv_uses_tensor_cores(_lib.ctypes.byref(c)))
        key = ("dw_" if dw else ("tc_" if tc else "generic_")) + kind
        work = conv_bytes(kind, g) if dw else conv_flops(g)
        f = fam.setdefault(key, [0.0, 0.0, 0])
        f[0] += work; f[1] += ms; f[2] += 1
        rows.append((key, f"{g.cin}->{g.cout} k{g.kh} s{g.stride} d{g.dil} g{g.groups} @{g.h}x{g.w}", work / 1e9, ms))
    if verbose:
        for r in rows:
            unit = "GB" if r[0].startswith("dw_") else "GF"
            print(f"  {r[0]:14s} {r[1]:36s} {r[2]:8.2f} {unit} {r[3]:8.3f} ms {r[2] / max(r[3], 1e-9):8.1f} T{unit[1]}/s", file=sys.stderr)
        for k, (fl, ms, n) in sorted(fam.items(), key=lambda kv: -kv[1][1]):
            print(f"  == {k:14s} launches={n:3d} {fl / 1e9:9.1f} G {ms:8.3f} ms {fl / 1e9 / max(ms, 1e-9):8.1f} T/s", file=sys.stderr)
    peak_t = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_b = peaks.get("hbm_gbs") or 6500.0
    roofs = {}
    for k, (work, ms, n) in fam.items():
        if k.startswith("tc_"):
            ach = work / (ms * 1e-3) / 1e12
            roofs[k] = {"bound": "tensor", "kernel": KERNEL_OF.get(k, k), "achieved": ach, "peak": peak_t, "unit": "TFLOP/s", "frac": ach / peak_t,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if "bf16_tflops_sustained" in peaks else "fallback",
                        "launches_per_step": n, "flops_per_step": work, "ms_per_step_in_kernel": ms}
        elif k.startswith("dw_"):
            ach = work / (ms * 1e-3) / 1e9
            roofs[k] = {"bound": "hbm", "kernel": KERNEL_OF.get(k, k), "achieved": ach, "peak": peak_b, "unit": "GB/s", "frac": ach / peak_b,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback",
                        "launches_per_step": n, "bytes_per_step": work, "ms_per_step_in_kernel": ms}
    if not roofs:
        return None, fam, roofs
    dom = max(roofs.items(), key=lambda kv: kv[1]["ms_per_step_in_kernel"])
    roof = dict(dom[1])
    # DRAM bytes per launch of that family from the committed `ncu --set full` capture of one step (profiles/README.md)
    roof["traffic"] = None
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic_final.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))[dom[0]]
            roof["traffic"] = t["dram_bytes"] / max(roof["launches_per_step"], 1)
            roof["traffic_note"] = (f"dram__bytes_read+write of all kernels of the family in one step (ncu --set full, profiles/{name}) / "
                                    "launches_per_step: per layer call, like flops_per_step / launches_per_step")
            break
        except Exception:  # noqa: BLE001
            pass
    return roof, fam, roofs


DUMP_MAX_ELEMS = 1 << 22          # per array (16 MB of float32): the four arrays of a dump stay under 64 MB together


def dump_outputs(out_dir, loss, net):
    """Save what the last timed step handed back, so that two builds can be compared output for output on identical inputs:
    loss.npy (float64, the step's loss), and the model the step left behind as float32 vectors -- params.npy (parameters after
    the SGD update), grads.npy (the step's gradients) and bn_stats.npy (floating-point buffers: BatchNorm running statistics).
    Each vector concatenates its tensors in named_parameters() / named_buffers() order, every tensor flattened in logical NCHW
    order.  A vector longer than DUMP_MAX_ELEMS is replaced by a fixed sample: the elements at DUMP_MAX_ELEMS sorted indices
    drawn without replacement by numpy's default_rng(0), which depend only on the vector's length."""
    import numpy as np
    import torch

    def flat(tensors):
        return torch.cat([t.detach().float().reshape(-1).cpu() for t in tensors]).numpy()

    params = [p for p in net.parameters() if p.requires_grad]
    arrays = {"loss": np.array([float(loss)], dtype=np.float64), "params": flat(params), "grads": flat(p.grad for p in params),
              "bn_stats": flat(b for b in net.buffers() if b.is_floating_point())}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.size > DUMP_MAX_ELEMS:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args):
    import importlib

    import torch
    import torch.distributed as dist

    from text_segmentation_image_inpainting_b200 import _lib
    from text_segmentation_image_inpainting_b200.engine import SegTrainStep, TrainStep
    from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks

    W = WORKLOADS[args.workload]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    _lib.load()

    def note(msg):
        if world > 1 or os.environ.get("PCB_BENCH_VERBOSE"):
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    torch.manual_seed(0)                                        # identical initial weights on every rank
    mod = importlib.import_module("text_segmentation_image_inpainting_b200.models." + W["net"][0])
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):             # the reference's constructors print ("No check point ...")
        net = getattr(mod, W["net"][1])().to(dev)
    Step = TrainStep if W["masks"] else SegTrainStep
    ts = Step(net, compute_dtype=torch.bfloat16, process_group=pg, use_graph=not args.no_graph)

    # synthetic inputs (SURVEY 8d): x ~ N(0,1); inpainting: free-form line/ellipse holes, one plane per image x3 channels
    B = W["batch"]
    g = torch.Generator().manual_seed(1234 + rank)
    NBUF = 2
    host_x = [torch.randn(B, 3, HW, HW, generator=g).pin_memory() for _ in range(NBUF)]
    host_m = [torch.from_numpy(random_hole_masks(B, HW, HW, seed=100 * rank + i)).pin_memory() for i in range(NBUF)] if W["masks"] else None
    dev_x = [t.to(dev) for t in host_x]
    dev_m = [t.to(dev) for t in host_m] if host_m else [None] * NBUF
    h2d_bytes = host_x[0].numel() * 4 + (host_m[0].numel() * 4 if host_m else 0)

    note("inputs ready; eager warm-up + graph capture")
    ts.warmup_and_capture(dev_x[0], dev_m[0], eager_warmup=2)
    note("captured; device-resident timing")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident timing: inputs already in HBM (two input sets alternate; the step's working set
    # (GBs of activations) is far larger than L2, so no explicit flush is needed)
    for i in range(args.warmup):
        ts.step(dev_x[i % NBUF], dev_m[i % NBUF])
    clocks = Clocks(local)
    barrier()
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        ts.step(dev_x[i % NBUF], dev_m[i % NBUF])
    e1.record()
    barrier()
    ms_total = maxreduce(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_total * 1e-3)
    note(f"device-resident done: {ms_total / args.steps:.2f} ms/step; end-to-end timing")

    # ---------------- end to end: host (pinned) buffers -> H2D on a copy stream, double buffered against
    # compute -> step -> D2H of the loss, every step inside the timed region
    copy_stream = torch.cuda.Stream()
    stage_x = [torch.empty_like(dev_x[0]) for _ in range(2)]
    stage_m = [torch.empty_like(dev_m[0]) if host_m else None for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def upload(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            stage_x[b].copy_(host_x[i % NBUF], non_blocking=True)
            if host_m:
                stage_m[b].copy_(host_m[i % NBUF], non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_run(nsteps):
        for b in range(2):
            consumed[b].record()
        upload(0)
        for i in range(nsteps):
            if i + 1 < nsteps:
                upload(i + 1)
            b = i % 2
            torch.cuda.current_stream().wait_event(ready[b])
            loss = ts.step(stage_x[b], stage_m[b])
            consumed[b].record()
            loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return loss

    e2e_run(max(2, min(args.warmup, 3)))
    barrier()
    e0.record()
    last_loss = e2e_run(args.steps)
    e1.record()
    barrier()
    e2e_ms = maxreduce(e0.elapsed_time(e1))
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)
    note("end-to-end done")
    if args.dump_outputs and rank == 0:
        # before the instrumented eager step below, which recomputes the gradients
        dump_outputs(args.dump_outputs, last_loss, net)

    # ---------------- per-kernel roofline (rank 0): eager instrumented step, events on the launching stream
    roof, fam, roofs = (None, {}, {})
    if rank == 0:
        roof, fam, roofs = layer_profile(ts, dev_x[0], dev_m[0], peaks, args.profile_layers)
    barrier()

    # ---------------- CPU baseline beside it (rank 0, N == 1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ips, ms, cores, kind = cpu_reference_steps(steps=3, warmup=1, batch=1, workload=args.workload)
        cpu = {"value": ips, "unit": "images/sec", "cores": int(str(cores).split()[0]), "cores_note": cores, "kind": kind,
               "sample": "3 steps x 1 image @512x512 (fwd+bwd+SGD) after 1 warm-up, all host threads"}

    if rank == 0:
        step_flop = (3 * W["fwd_gf"] - W["no_dgrad_gf"]) * 1e9 * B          # SURVEY 8d: fwd+bwd (minus the stem dgrad)
        line = {
            "metric": W["metric"], "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{W['label']} 512x512, batch {B} per GPU, fwd+bwd+SGD(nesterov), train-mode BN",
                       "global_batch": B * world, "parallelism": f"dp{world}", "cuda_graph": ts.graph is not None,
                       "allreduce": ("overlapped with backward (captured)" if ts.overlap_active else "after backward") if world > 1 else "none",
                       "l2": "inputs+activations per step (GBs) exceed the 126 MB L2; no explicit flush",
                       "loss": "out.abs().mean()", "algorithmic_tflop_per_step_per_gpu": step_flop / 1e12},
            "step_tflops_per_gpu": step_flop / 1e12 / (ms_total / args.steps * 1e-3),
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": ts.launches_per_step * args.steps,
            "roofline": roof,
            # every conv family of the step (the dominant one above flips between tc_fwd and tc_wgrad run to run: report all)
            "rooflines": {k: {kk: v[kk] for kk in ("bound", "achieved", "peak", "unit", "frac", "launches_per_step", "ms_per_step_in_kernel")}
                          for k, v in sorted(roofs.items())},
            "kernel_families_ms": {k: round(v[1], 4) for k, v in fam.items()},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        # graphs that captured NCCL collectives must die before the communicator (engine.TrainStep.close); the timer only
        # guards the teardown itself -- the measurement is complete and printed at this point
        import threading
        threading.Timer(60.0, lambda: os._exit(0)).start()
        ts.close()
        barrier()
        dist.destroy_process_group()
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    _isolate_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)

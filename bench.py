#!/usr/bin/env python
"""Headline benchmark: VNet3d(1,2) 96^3, batch 2 per GPU, bf16 storage, forward + loss + backward
(+ gradient all-reduce for N > 1) in voxels/second (BASELINE.json `metric`, config[1] / config[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-graph] [--dump-outputs DIR]

N > 1 is launched by the driver as ``python -m torch.distributed.run --nproc-per-node N bench.py --gpus N``
(one rank per GPU, NCCL).  Rank 0 prints ONE JSON line.  A "step" = one pass of the hot path
(forward in train mode with dropout masks drawn, MutilDiceLoss, backward of all 128 parameter
tensors; no optimizer -- the metric is "fwd+bwd", SURVEY.md section 8d) over one synthetic batch.

Timing: CUDA events on the launching stream, one event pair per step, L2 flushed (256 MiB write)
before every timed step outside the event pair, max over ranks; W >= 3 warm-up steps.  The clock sampler
(nvidia-smi) runs on EVERY rank and is started before the warm-up, i.e. well before the barrier that aligns the
timed region (round 1 started it on rank 0 between the barrier and the first step: the other ranks waited in
their first all-reduce and the N=8 line was wrong).
  value : inputs resident in HBM, CUDA-graph replay of the step (GraphedStep); mean of the K timed steps
          (median / min / max reported beside it; sum of the event times is checked against the wall clock).
  e2e   : same, but every step copies x (fp32) and labels (int64) from pinned host memory and reads
          the loss back to the host inside the timed region.
  roofline     : the kernel with the largest share of the step, from ONE serialised, instrumented eager step
                 (weight gradients on the main stream, device synchronised between ops, so an event pair times a
                 kernel and not a queue): algorithmic bytes/flops (DESIGN.md section 5) / its mean duration vs
                 MEASURED_PEAKS.json; per network block (10 VNet3d blocks) in `roofline_blocks`.
  variants (N=1 only): forward-only, optimizer-inclusive (fused AdamW inside the graph) and the fp32 parity mode.
  cpu_baseline : the CPU oracle (oracle/, a restatement of the reference's PyTorch path: "port")
                 timed on this box's host cores, same shapes/seeds, fwd+loss+bwd, rank 0, N=1.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SPATIAL = (96, 96, 96)
BATCH_PER_GPU = 2
NUMCLASS = 2
# SURVEY.md section 8d: algorithmic work of one fwd+bwd step of VNet3d(1,2) 96^3 B=2 (bf16 storage)
STEP_GFLOP = 433.11
STEP_MB = 3239.9
ARCH = "vnet3d"
LOSS = "MutilDiceLoss"

# --workload: the headline metric is vnet3d96 (BASELINE.json configs[1]/[3]); the others are the remaining
# GPU configs of BASELINE.json, timed with the same harness for DESIGN.md (not the graded bench line)
WORKLOADS = {
    "vnet3d96": dict(arch="vnet3d", spatial=(96, 96, 96), batch=2, ncls=2, loss="MutilDiceLoss", gflop=433.11,
                     mb=3239.9, desc="VNet3d(1,2) 96x96x96, batch 2 per GPU"),
    "unet3d128": dict(arch="unet3d", spatial=(128, 128, 128), batch=1, ncls=4, loss="MutilCrossEntropyDiceLoss",
                      gflop=715.01, mb=3393.9, desc="UNet3d(1,4) 128x128x128, batch 1 per GPU"),
    "unet2d512": dict(arch="unet2d", spatial=(512, 512), batch=8, ncls=1, loss="BinaryDiceFocalLoss", gflop=578.01,
                      mb=4841.1, desc="UNet2d(1,1) 512x512, batch 8 per GPU"),
}


def select_workload(name):
    global SPATIAL, BATCH_PER_GPU, NUMCLASS, STEP_GFLOP, STEP_MB, ARCH, LOSS, WL_DESC
    w = WORKLOADS[name]
    SPATIAL, BATCH_PER_GPU, NUMCLASS = w["spatial"], w["batch"], w["ncls"]
    STEP_GFLOP, STEP_MB, ARCH, LOSS, WL_DESC = w["gflop"], w["mb"], w["arch"], w["loss"], w["desc"]


WL_DESC = WORKLOADS["vnet3d96"]["desc"]


def voxels_per_sample():
    v = 1
    for s_ in SPATIAL:
        v *= s_
    return v


def oracle_step_fn():
    """(state_dict with grads, step()) for the CPU arm of the selected workload."""
    import oracle
    from oracle import nets as onets
    if ARCH == "vnet3d":
        spec = onets.vnet3d_state_spec(1, NUMCLASS)
        fwd = lambda sd, x, m: onets.vnet3d_forward(sd, x, m)
        draw = lambda n: onets.draw_dropout_masks_vnet3d(n)
    else:
        dims = 3 if ARCH == "unet3d" else 2
        spec = onets.unet_state_spec(1, NUMCLASS, dims)
        fwd = lambda sd, x, m: onets.unet_forward(sd, x, dims, m)
        draw = lambda n: onets.draw_dropout_masks_unet(n, dims)
    sd = {k: v.requires_grad_(True) for k, v in onets.init_state_dict(spec, seed=0).items()}
    x, y = make_batch(0, 1)
    alpha = torch.ones(NUMCLASS)

    def step():
        for v in sd.values():
            v.grad = None
        logits, _ = fwd(sd, x, draw(x.shape[0]))
        loss = oracle.loss_forward(LOSS, logits, y, alpha)
        loss.backward()
        return float(loss.detach())
    return step


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "bf16_tflops_burst": d["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "bf16_tflops_burst": 1590.0,
            "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# stdout hygiene: libraries (NCCL's version banner, ...) write to file descriptor 1 directly.  While the bench runs,
# fd 1 points at stderr; the one JSON line is emitted through the saved descriptor.
# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# per-kernel timing wrapper (instrumentation around the real CudaBackend)
# ------------------------------------------------------------------------------------------------
class TimedBackend:
    TIMED = ("conv", "conv_bwdstats", "wgrad", "apply", "gn_bwd_reduce", "gn_bwd_apply", "gn_finalize", "gn_bwd_finalize",
             "apply_gn", "gn_bwd_reduce_gn", "gn_bwd_apply_gn", "gn_bwd_fused_gn", "pack_weight", "unpack_wgrad",
             "colsum", "head_probs", "head_fwd", "head_bwd", "loss_partials", "loss_finalize", "loss_bwd", "pool_fwd",
             "pool_bwd", "pack_many", "pack_launch", "unpack_many", "dropout_masks", "metric_finalize", "adam_step")

    def __init__(self, inner):
        self.inner, self.records, self.tag = inner, [], "other"

    def __getattr__(self, name):
        fn = getattr(self.inner, name)
        if name not in self.TIMED:
            return fn

        def wrapped(*a, **k):
            # serialised: nothing else is in flight when the op starts, and it has finished before the next one is
            # issued.  A ~1 ms spin kernel is queued first so that the start event, the op's kernel(s) and the stop
            # event are all enqueued while the GPU is still busy: the event pair then brackets device execution only,
            # not the host's launch path (ctypes call, descriptor tables), which a CUDA-graph replay does not pay
            torch.cuda.synchronize()
            torch.cuda._sleep(2_000_000)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            torch.cuda.synchronize()
            self.records.append((name, self._describe(name, a), e0, e1, self._work(name, a), self.tag))
            return r
        return wrapped

    @staticmethod
    def _describe(name, a):
        if name == "conv":
            kind, dims, x, wpk, bias, y = a[:6]
            path = {2: "/tcgen05", 3: "/tcgen05-halo", 4: "/tcgen05-halo-ws"}.get(getattr(wpk, "code", 0), "/cuda-core")
            if x.shape[-1] == 1 and y.dtype == torch.bfloat16:
                path = "/mma.sync-stem"
            elif (kind in (1, 3) and getattr(wpk, "code", 0) == 2 and max(x.shape[-1], y.shape[-1]) <= 64
                  and y.numel() // y.shape[-1] >= 65536 and x.shape[-1] * y.shape[-1] <= (512 if kind == 3 else 2048)):
                path = "/mma.sync-pointwise"      # pw_mma.cu takes these shapes ahead of the tcgen05 kernel
            return f"conv[k{kind}{path}] {x.shape[-1]}->{y.shape[-1]}@{tuple(y.shape[1:4])}"
        if name == "conv_bwdstats":
            kind, dims, x, wpk, y = a[:5]
            return f"conv+gn_bwd_sums[k{kind}/tcgen05-halo] {x.shape[-1]}->{y.shape[-1]}@{tuple(y.shape[1:4])}"
        if name == "wgrad":
            kind, dims, x, dy = a[:4]
            return f"wgrad[k{kind}] {x.shape[-1]}x{dy.shape[-1]}@{tuple(dy.shape[1:4])}"
        if name == "gn_bwd_fused_gn":
            name = "gn_bwd_fused(reduce+barrier+apply)"
        t = next((v for v in a if isinstance(v, torch.Tensor) and v.dim() == 5), None)
        return f"{name} {t.shape[-1]}@{tuple(t.shape[1:4])}" if t is not None else name

    @staticmethod
    def _work(name, a):
        """(algorithmic bytes, algorithmic flops) of one launch (DESIGN.md section 5)."""
        def nbytes(t):
            return 0 if t is None else t.numel() * t.element_size()
        if name == "conv":
            kind, dims, x, wpk, bias, y, stats, addend = a[:8]
            w = wpk.t if hasattr(wpk, "t") else wpk
            taps_cin = w.numel() // y.shape[-1]
            vox_out = y.numel() // y.shape[-1]
            if kind == 3:  # UP: K = Cin per fine voxel
                flops = 2.0 * vox_out * y.shape[-1] * x.shape[-1]
            else:
                flops = 2.0 * vox_out * y.shape[-1] * taps_cin
            return nbytes(x) + nbytes(y) + nbytes(w) + nbytes(addend), flops
        if name == "conv_bwdstats":
            kind, dims, x, wpk, y, addend, yfwd = a[:7]
            w = wpk.t if hasattr(wpk, "t") else wpk
            vox_out = y.numel() // y.shape[-1]
            return (nbytes(x) + nbytes(y) + nbytes(w) + nbytes(addend) + nbytes(yfwd),
                    2.0 * vox_out * y.shape[-1] * (w.numel() // y.shape[-1]))
        if name == "wgrad":
            kind, dims, x, dy, dwp = a[:5]
            vox = dy.numel() // dy.shape[-1]
            return nbytes(x) + nbytes(dy) + nbytes(dwp), 2.0 * vox * dwp.numel()
        b = sum(nbytes(v) for v in a if isinstance(v, torch.Tensor) and v.dim() == 5)
        return b, 0.0

    def summary(self):
        torch.cuda.synchronize()
        agg, blocks = {}, {}
        for name, desc, e0, e1, (by, fl), tag in self.records:
            ms = e0.elapsed_time(e1)
            d = agg.setdefault(desc, {"ms": 0.0, "n": 0, "bytes": by, "flops": fl})
            d["ms"] += ms
            d["n"] += 1
            b = blocks.setdefault(tag, {"ms": 0.0, "n": 0})
            b["ms"] += ms
            b["n"] += 1
        return agg, blocks


# ------------------------------------------------------------------------------------------------
def make_batch(rank: int, world: int):
    """global batch = 2*world samples drawn from one seeded generator; rank r takes [2r, 2r+2)."""
    import oracle
    x, y = oracle.make_inputs(BATCH_PER_GPU * world, 1, SPATIAL, NUMCLASS, seed=1234)
    sl = slice(BATCH_PER_GPU * rank, BATCH_PER_GPU * (rank + 1))
    return x[sl].contiguous(), y[sl].contiguous()


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(loss, dice, model):
    """What a caller of the timed step receives: the loss, the per-step Dice and the gradient of every parameter,
    copied to the host as float32 arrays {name: array}."""
    import numpy as np
    out = {"loss": loss, "dice": dice}
    out.update({"grad." + n: p.grad for n, p in model.named_parameters()})
    return {k: np.array(v.detach().float().cpu().numpy()) for k, v in out.items()}


def write_outputs(directory, outputs):
    """DIR/<name>.npy for every array; refuses more than DUMP_LIMIT_BYTES in all."""
    import numpy as np
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"[bench] --dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_reference(args):
    """The reference's own CPU path for this metric: the oracle restatement (kind 'port') on all host cores."""
    import oracle
    from oracle import nets as onets
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = pick_cpu_threads()
    torch.set_num_threads(cores)
    step = oracle_step_fn()

    steps, warm = max(1, min(args.steps, 5)), max(1, min(args.warmup, 2))
    for _ in range(warm):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    vox = BATCH_PER_GPU * voxels_per_sample()
    val = vox / t
    line = {"impl": "reference", "metric": "voxels_per_sec_fwd_bwd", "value": val, "unit": "voxels/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WL_DESC + ", fwd+loss(" + LOSS + ")+bwd, train mode, CPU fp32",
                       "global_batch": BATCH_PER_GPU},
            "cpu_baseline": {"value": val, "unit": "voxels/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{steps} full steps ({WL_DESC}) of the oracle restatement on "
                                       f"{torch.get_num_threads()} host threads"},
            "e2e": {"value": val, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


def pick_cpu_threads():
    """Host threads for the CPU arm: all cores the process may use, unless a short probe (one 3x3x3
    conv at the 32-channel level) shows fewer threads are faster on this (shared) host."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    xs = torch.randn(2, 32, 48, 48, 48)
    ws = torch.randn(32, 32, 3, 3, 3)
    best, best_t = avail, None
    cand = sorted({avail, max(1, avail // 2), max(1, avail // 4), min(avail, 32), min(avail, 16)}, reverse=True)
    for th in cand:
        torch.set_num_threads(th)
        torch.nn.functional.conv3d(xs, ws, padding=1)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.conv3d(xs, ws, padding=1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
    return best


def cpu_baseline_sample():
    import oracle
    from oracle import nets as onets
    prev = torch.get_num_threads()
    cores = pick_cpu_threads()
    torch.set_num_threads(cores)
    step = oracle_step_fn()
    ts = []
    for i in range(3):
        t0 = time.perf_counter()
        step()
        if i > 0:
            ts.append(time.perf_counter() - t0)
    torch.set_num_threads(prev)
    t = statistics.median(ts)
    vox = BATCH_PER_GPU * voxels_per_sample()
    return {"value": vox / t, "unit": "voxels/s", "cores": cores, "kind": "port",
            "sample": f"2 timed full steps (+1 warm-up) of {WL_DESC} fwd+loss+bwd, oracle restatement, fp32, "
                      f"{cores} host threads; median {t * 1e3:.0f} ms/step"}


# per-block algorithmic work of VNet3d(1,2) 96^3 B=2 bf16, fwd+bwd (SURVEY.md section 8d): (GFLOP, MB)
VNET96_BLOCKS = {"in_tr": (3.17, 353.9), "down_tr32": (78.8, 481.8), "down_tr64": (57.8, 147.9),
                 "down_tr128": (28.9, 47.4), "down_tr256": (14.4, 53.6), "up_tr256": (28.9, 45.7),
                 "up_tr128": (57.8, 134.2), "up_tr64": (78.8, 425.3), "up_tr32": (84.3, 1302.4),
                 "out_tr": (0.34, 247.7)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the fwd-only / optimizer / fp32 variants (N=1)")
    ap.add_argument("--workload", default="vnet3d96", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, Dice, every parameter gradient) as "
                         "DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _capture_stdout()
    select_workload(args.workload)
    args.warmup = max(3, args.warmup)

    if args.impl == "reference":
        run_reference(args)
        return

    import pytorchdeeplearing_b200 as b200
    from pytorchdeeplearing_b200 import runtime
    from pytorchdeeplearing_b200.graphed import GraphedStep
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the b200 arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    sampler.start()                   # every rank, long before the barrier-aligned timed region
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout = the one JSON line
        dist.init_process_group("nccl", device_id=dev)
        b200.enable_data_parallel()
    b200.set_precision(args.precision)

    def make_model():
        torch.manual_seed(0)
        m = {"vnet3d": b200.VNet3d, "unet3d": b200.UNet3d, "unet2d": b200.UNet2d}[ARCH](1, NUMCLASS)
        m.apply(b200.initialize_weights)
        return m.to(dev).train()

    model = make_model()
    losscls = getattr(b200, LOSS)
    lossfn = losscls(torch.ones(NUMCLASS, device=dev)) if LOSS.startswith("Mutil") else losscls()
    xh, yh = make_batch(rank, world)
    xh, yh = xh.pin_memory(), yh.pin_memory()
    x, y = xh.to(dev), yh.to(dev)
    # the SAME seed on every rank: a rank takes its rows of the global-batch dropout draw (SURVEY.md 8e)
    torch.manual_seed(100)
    be = runtime.cuda_backend()

    def eager_step(xx, yy, mdl=None):
        mdl = mdl or model
        for p in mdl.parameters():
            p.grad = None
        logits, _ = mdl(xx)
        loss = lossfn(logits, yy)
        loss.backward()
        return loss

    use_graph = not args.no_graph
    graphed = None
    if use_graph:
        try:
            graphed = GraphedStep(model, lossfn, x, y, warmup=2)
        except Exception as e:  # pragma: no cover
            print(f"[bench] rank {rank}: CUDA graph capture failed ({type(e).__name__}: {e}); eager launches",
                  file=sys.stderr)
            graphed = GraphedStep(model, lossfn, x, y, warmup=1, use_graph=False)
            torch.cuda.synchronize()
    n_graphs = len(graphed.graphs) if graphed is not None else 0

    # ---- launches per step (counted on the step as it is benchmarked: one eager GraphedStep pass)
    torch.cuda.synchronize()
    c0 = be.launch_count
    if graphed is not None:
        graphed._eager_step()
    else:
        eager_step(x, y)
    torch.cuda.synchronize()
    launches = be.launch_count - c0

    # ---- per-kernel / per-block timing: ONE serialised, instrumented eager step (rank 0 only; no collectives)
    kern, blocks = {}, {}
    if rank == 0:
        dp_prev = runtime.dp_state()
        runtime.disable_data_parallel()
        os.environ["B200SEG_WGRAD_SIDE_STREAM"] = "0"
        os.environ["B200SEG_CHECK_LABELS"] = "0"
        tb = TimedBackend(be)
        runtime._set_backend_for_testing(tb)
        try:
            probe = GraphedStep(model, lossfn, x, y, warmup=1, use_graph=False)
            tb.records.clear()
            probe._eager_step()
            kern, blocks = tb.summary()
        finally:
            runtime._set_backend_for_testing(None)
            del os.environ["B200SEG_WGRAD_SIDE_STREAM"]
            del os.environ["B200SEG_CHECK_LABELS"]
            if dp_prev[0]:
                runtime.enable_data_parallel(dp_prev[1])
        del probe

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, k):
        evs = []
        for _ in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step_fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    last_loss = [None]

    def resident_step():
        if use_graph:
            last_loss[0] = graphed()       # replays on the static (HBM-resident) input buffers
        else:
            last_loss[0] = eager_step(x, y)

    host_losses = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_values = []

    def e2e_loop(k):
        """k steps through the public API with HOST inputs, software-pipelined the way a training loop runs around a
        CUDA graph: the inputs of step i+1 are copied from pinned host memory on a copy stream while step i
        executes, and the loss of step i is copied back asynchronously and READ ON THE HOST while step i+1 executes
        (one step of lag, every loss is read).  One timed region around the whole loop: all k H2D copies and all k
        D2H reads are inside it.  Returns ms per step."""
        torch.cuda.synchronize()
        loss_values.clear()
        done = [torch.cuda.Event(), torch.cuda.Event()]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if use_graph:
            graphed.prefetch(xh, yh)
        for i in range(k):
            if use_graph:
                loss = graphed(prefetched=True)
                if i + 1 < k:
                    graphed.prefetch(xh, yh)
            else:
                loss = eager_step(xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True))
            host_losses[i & 1].copy_(loss.detach(), non_blocking=True)
            done[i & 1].record()
            if i > 0:                                       # the previous step's loss is on the host by now
                done[(i - 1) & 1].synchronize()
                loss_values.append(float(host_losses[(i - 1) & 1]))
        done[(k - 1) & 1].synchronize()
        loss_values.append(float(host_losses[(k - 1) & 1]))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    for _ in range(args.warmup):
        resident_step()
    barrier()
    wall0 = time.perf_counter()
    ms = timed(resident_step, args.steps)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    if sum(ms) * 1e-3 > wall * 1.02 + 1e-3:
        raise SystemExit(f"[bench] rank {rank}: inconsistent timing: event sum {sum(ms):.2f} ms > wall {wall * 1e3:.2f} ms")
    # the e2e loop below reuses the step's static buffers: copy the last timed step's outputs first
    outputs = None
    if args.dump_outputs and rank == 0:
        dice = graphed.dice if use_graph else lossfn.last_dice()
        outputs = step_outputs(last_loss[0], dice, model)
    e2e_loop(2)
    barrier()
    ms_e2e = e2e_loop(args.steps)
    barrier()

    tot = torch.tensor([sum(ms), ms_e2e * args.steps, statistics.median(ms), min(ms), max(ms)], dtype=torch.float64,
                       device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    t_step = tot[0].item() / args.steps * 1e-3
    t_e2e = tot[1].item() / args.steps * 1e-3
    vox_step = world * BATCH_PER_GPU * voxels_per_sample()

    # ---- variants (single GPU): forward only, optimizer inclusive, fp32 parity mode
    variants = {}
    if world == 1 and use_graph and not args.no_variants:
        vox1 = BATCH_PER_GPU * voxels_per_sample()

        def time_fn(fn, k, w=3):
            for _ in range(w):
                fn()
            return statistics.median(timed(fn, k))
        try:
            # forward only (train mode, masks drawn): one graph around model(x) under no_grad
            gfw = torch.cuda.CUDAGraph()
            with torch.no_grad():
                model(x)
                torch.cuda.synchronize()
                with torch.cuda.graph(gfw):
                    model(x)
            t_fwd = time_fn(gfw.replay, 20)
            variants["fwd_only"] = {"ms_per_step": t_fwd, "voxels_per_s": vox1 / (t_fwd * 1e-3)}
            del gfw
            # optimizer inclusive: fused AdamW (one launch on the flat buckets) inside the step graph
            m2 = make_model()
            opt = b200.FusedAdamW(m2.parameters(), lr=1e-3)
            g2 = GraphedStep(m2, lossfn, x, y, warmup=2, optimizer=opt)
            t_opt = time_fn(g2, 20)
            variants["with_fused_adamw"] = {"ms_per_step": t_opt, "voxels_per_s": vox1 / (t_opt * 1e-3)}
            del g2, opt, m2
            # fp32 parity mode (the kernel set that meets north_star's 1e-3 / identical-argmax bar)
            if args.precision == "bf16":
                b200.set_precision("fp32")
                m3 = make_model()
                g3 = GraphedStep(m3, lossfn, x, y, warmup=1)
                t32 = time_fn(g3, 5, w=1)
                variants["fp32_parity_mode"] = {"ms_per_step": t32, "voxels_per_s": vox1 / (t32 * 1e-3)}
                del g3, m3
                b200.set_precision("bf16")
        except Exception as e:  # pragma: no cover
            variants["error"] = f"{type(e).__name__}: {e}"
            b200.set_precision(args.precision)

    if rank == 0:
        peaks = load_peaks()
        total_ms = max(1e-9, sum(v["ms"] for v in kern.values()))
        # dominant kernel of the step = largest share of the serialised step time
        desc, d = max(kern.items(), key=lambda kv: kv[1]["ms"])
        dur = d["ms"] / d["n"] * 1e-3
        gbs = d["bytes"] / dur / 1e9
        tfs = d["flops"] / dur / 1e12
        hbm_frac = gbs / peaks["hbm_gbs"]
        tc_frac = tfs / peaks["bf16_tflops_burst"]
        if tc_frac > hbm_frac:
            roof = {"bound": "tensor", "achieved": tfs, "peak": peaks["bf16_tflops_burst"], "unit": "TFLOP/s",
                    "frac": tc_frac}
        else:
            roof = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_frac}
        traffic = None                # DRAM bytes per launch from the committed ncu --set full capture, if this
        try:                          # kernel/shape was captured (profiles/ncu_traffic.json)
            with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f).get(desc, {}).get("dram_bytes")
        except (OSError, ValueError):
            pass
        roof.update({"kernel": desc, "launches_per_step": d["n"], "avg_us": dur * 1e6, "traffic": traffic,
                     "algorithmic_bytes": d["bytes"], "algorithmic_flops": d["flops"],
                     "peaks": peaks["source"], "share_of_step": d["ms"] / total_ms,
                     "how": "serialised eager step: weight gradients on the main stream, device sync between ops"})
        ranked_all = sorted(kern.items(), key=lambda kv: -kv[1]["ms"])
        ranked = ranked_all[:14]
        if os.environ.get("B200SEG_BENCH_TABLE"):        # development aid: the full per-op table of the eager pass
            with open(os.environ["B200SEG_BENCH_TABLE"], "w") as f:
                for k, v in ranked_all:
                    f.write(f"{v['ms'] * 1e3:9.1f} us  x{v['n']:3d}  {k}\n")
                for k, v in sorted(blocks.items(), key=lambda kv: -kv[1]["ms"]):
                    f.write(f"block {k:12s} {v['ms'] * 1e3:9.1f} us  x{v['n']:3d}\n")
        block_table = None
        if args.workload == "vnet3d96":
            block_table = {}
            for bname, (gf, mb) in VNET96_BLOCKS.items():
                mb_ = mb * (1.0 if args.precision == "bf16" else 2.0)     # fp32 storage doubles the activation bytes
                t_tc = gf / 1e3 / peaks["bf16_tflops_burst"]
                t_hbm = mb_ / 1e3 / peaks["hbm_gbs"]
                t_roof = max(t_tc, t_hbm)
                t_meas = blocks.get(bname, {}).get("ms", 0.0) * 1e-3
                block_table[bname] = {"bound": "tensor" if t_tc > t_hbm else "hbm", "roof_us": t_roof * 1e6,
                                      "measured_us": t_meas * 1e6, "launches": blocks.get(bname, {}).get("n", 0),
                                      "frac": (t_roof / t_meas) if t_meas > 0 else None}
            block_table["other(pack/unpack/masks)"] = {"measured_us": blocks.get("other", {}).get("ms", 0.0) * 1e3,
                                                       "launches": blocks.get("other", {}).get("n", 0)}
        step_roof = {"hbm_GBps": STEP_MB / 1e3 / t_step, "tflops": STEP_GFLOP / 1e3 / t_step,
                     "frac_hbm": STEP_MB / 1e3 / t_step / peaks["hbm_gbs"],
                     "frac_tensor": STEP_GFLOP / 1e3 / t_step / peaks["bf16_tflops"],
                     "algorithmic_GFLOP": STEP_GFLOP, "algorithmic_MB": STEP_MB,
                     "serialised_kernel_sum_ms": total_ms}
        line = {
            "metric": "voxels_per_sec_fwd_bwd", "value": vox_step / t_step, "unit": "voxels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "ms_per_step_median": tot[2].item(), "ms_per_step_min": tot[3].item(), "ms_per_step_max": tot[4].item(),
            "config": {"workload": WL_DESC + ", fwd (train mode, dropout masks drawn) + " + LOSS +
                                   " (+ per-step Dice accuracy from the same pass) + bwd of all parameter tensors"
                                   + (" + NCCL SUM all-reduce of the flat fp32 gradient bucket (two pieces, the first "
                                      "overlapping the rest of backward)" if world > 1 else ""),
                       "global_batch": BATCH_PER_GPU * world, "parallelism": f"dp{world}",
                       "l2": "value: 256 MiB flush before every timed step; e2e: one timed region over all steps, "
                             "no flush (inputs arrive from the host every step; per-step working set > 1 GB >> 126 MB L2)",
                       "e2e_pipeline": "H2D of step i+1 on a copy stream overlaps step i; the loss of every step is "
                                       "copied back and read on the host while the next step runs (one step of lag)",
                       "cuda_graph": bool(use_graph and n_graphs > 0), "graphs_per_step": n_graphs,
                       "nccl_inside_graph": bool(world > 1 and n_graphs == 1),
                       "precision_mode": args.precision},
            "e2e": {"value": vox_step / t_e2e, "unit": "voxels/s", "ms_per_step": t_e2e * 1e3,
                    "h2d_bytes_per_step": xh.numel() * 4 + yh.numel() * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "clocks": clocks, "roofline": roof, "roofline_step": step_roof, "roofline_blocks": block_table,
            "variants": variants,
            "top_kernels": [{"kernel": k, "ms_per_step": v["ms"], "launches": v["n"],
                             "GBps": v["bytes"] / (v["ms"] / v["n"] * 1e-3) / 1e9 if v["ms"] > 0 else None,
                             "TFLOPs": v["flops"] / (v["ms"] / v["n"] * 1e-3) / 1e12 if v["ms"] > 0 else None}
                            for k, v in ranked],
            "wall_s_timed_region": wall, "event_sum_s_timed_region": sum(ms) * 1e-3,
            "final_loss": loss_values[-1] if loss_values else None,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_sample()
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        _emit(line)
    if world > 1:
        del graphed                    # graphs first, then the communicator
        torch.cuda.synchronize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

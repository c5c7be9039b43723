#!/usr/bin/env python
"""Benchmark of the VideoPose3D temporal-convolution hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|bf16x3]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): TemporalModel,
arc 3,3,3,3,3 (243-frame receptive field), C = 1024, 17 joints, eval-mode forward of N = 1024
windows of T = 243 synthetic 2-D keypoint frames per GPU -> 1024 predicted 3-D frames per step.
metric = predicted frames per second over all GPUs (the reference counts batches "in terms of
predicted frames", common/arguments.py:37).  One step = one forward over one batch.

Printed JSON (one line, rank 0): see the task contract.  `value` is measured with inputs resident
in HBM (CUDA events around each step, L2 flushed between steps); `e2e` goes through the public
host-buffer call (pinned host input -> H2D -> kernels -> D2H) every step; `roofline` brackets the
dominant kernel (block-1 3-tap conv GEMM, M = 27648, K = 3072, N = 1024) with CUDA events on its
own stream inside the timed steps; `cpu_baseline` times the oracle's torch.nn.functional port of
the reference (what the reference executes on a host) on a bounded sample.

Beside the headline the line carries `roofline_step` (executed FLOPs of the whole forward / step
time / peak), `modes` (the other precision modes, short runs), and the training path: at N = 1 a
`train` block for BASELINE configs[2] (TemporalModelOptimized1f, device-resident ChunkedGenerator
-> forward + backward -> fused mpjpe -> FusedAdam, N = 1024), at N > 1 a `train_dp` block for
configs[3] (the same step data-parallel: generator rows sharded by rank, one gradient all-reduce per
step through data_parallel.GradientReducer over NCCL).

--impl reference: the reference's own CPU implementation of the same path on the host cores, same
metric / config: the UNMODIFIED reference classes from the archive staged by oracle/stage_ref.py
(`cpu_baseline.kind` = "reference") or, if that is absent, the oracle port ("port").
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARC = [3, 3, 3, 3, 3]
J, F, C, N_PER_GPU, T = 17, 2, 1024, 1024, 243
METRIC = "frames/sec (arc 3,3,3,3,3, T=243, N=1024)"
UNIT = "frames/s"
# Executed (dependency-cone) forward FLOPs per sample, 2 FLOP per MAC (SURVEY.md §8d): eval-mode
# TemporalModel on one receptive field only needs the rows on the output frame's cone.
FLOPS_PER_SAMPLE_CONE = 352.6e6
FLOPS_PER_SAMPLE_DENSE = 5217.8e6     # what the reference executes as written (all positions)
# dominant kernel: block-1 conv, rows = N*27, K = 3*1024, N = 1024
DOMINANT_FLOPS_PER_LAUNCH = 2.0 * (N_PER_GPU * 27) * 3072 * 1024
# its compulsory HBM bytes: A 27648x3072 bf16 + W 1024x3072 bf16 + out 27648x1024 bf16
DOMINANT_ALGORITHMIC_BYTES = 2.0 * (N_PER_GPU * 27 * 3072 + 1024 * 3072 + N_PER_GPU * 27 * 1024)
# DRAM bytes of that launch: read from the summary of an `ncu --set full` capture of THIS build
# (profiles/traffic.json, written by tools/summarize_ncu_full.py --traffic; carries the sha256 of
# the library it was captured from) -- null when no capture of the loaded library is committed.
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "traffic.json")
# training step (configs[2]): fwd 352.6 + dgrad 335.7 + wgrad 352.6 MFLOP/sample (SURVEY §8d)
FLOPS_PER_SAMPLE_TRAIN = 1040.9e6
WORKLOAD = ("TemporalModel arc=3,3,3,3,3 T=243 C=1024 J=17 eval forward, N=1024 windows per GPU "
            "(BASELINE configs[1])")


def lib_sha256():
    import hashlib
    from videopose3d_b200 import _capi
    try:
        with open(_capi.lib_path(), "rb") as f:
            return hashlib.sha256(f.read()).hexdigest()
    except OSError:
        return None


def load_traffic(kernel_key):
    """DRAM bytes per launch of `kernel_key` from the committed capture, with provenance."""
    try:
        with open(TRAFFIC_FILE) as f:
            t = json.load(f)
    except (OSError, ValueError):
        return None, "no profiles/traffic.json"
    ent = t.get("kernels", {}).get(kernel_key)
    if not ent:
        return None, f"{kernel_key} not in profiles/traffic.json"
    same = t.get("lib_sha256") == lib_sha256()
    src = (f"ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of this launch "
           f"({t.get('source', '?')}); captured from library sha256 {str(t.get('lib_sha256'))[:12]} "
           f"({'the library loaded now' if same else 'NOT the library loaded now'})")
    return float(ent["dram_bytes"]), src


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


def load_sustained_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["bf16_tflops_sustained"])
    except Exception:
        return 1400.0


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPU cores NVML reports as local to GPU `index` BEFORE the pinned
    host buffers are allocated (first touch places them on that NUMA node): host->device copies
    from the far socket ran at half the PCIe rate on some boxes.  Returns the previous affinity
    (to restore for the CPU baseline) or None when nothing was changed."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        old = os.sched_getaffinity(0)
        new = cpus & old
        if not new or new == old:
            return None
        os.sched_setaffinity(0, new)
        return old
    except Exception:
        return None


def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, not just the
    machine's logical CPU count (a 128-thread pool on a quota of a few cores crawls)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def reference_model_module():
    """`common.model` of the UNMODIFIED reference (/root/reference, or the archive staged by
    oracle/stage_ref.py that travelled to this box), or None."""
    try:
        from oracle import stage_ref
        return stage_ref.import_reference()
    except Exception:
        return None


def make_cpu_reference(ref_mod):
    """(callable x -> y, kind): the reference's own TemporalModel in eval mode on the CPU
    ("reference"), else the oracle's torch.nn.functional port ("port").  Same seeded parameters."""
    import torch
    from oracle import temporal_model_oracle as orc
    sd = orc.make_state_dict(J, F, J, ARC, C, seed=0)
    if ref_mod is not None:
        m = ref_mod.TemporalModel(J, F, J, filter_widths=ARC, causal=False, dropout=0.25, channels=C)
        m.load_state_dict(sd)
        m.eval()
        return (lambda x: m(x)), "reference"
    return (lambda x: orc.forward_torch(sd, x, ARC)), "port"


def pick_cpu_threads():
    """The reference gets the thread count that serves it best: a short calibration of the same
    forward over {8, 16, 32, 64, all usable cores} threads, fastest wins."""
    import torch
    from oracle import temporal_model_oracle as orc
    cores = usable_cores()
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | {cores})
    fwd, _ = make_cpu_reference(reference_model_module())
    x = orc.make_input(8, T, J, F, seed=1)
    best, best_dt = cands[-1], None
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            fwd(x[:2])
            t0 = time.perf_counter()
            fwd(x)
            dt = time.perf_counter() - t0
            if best_dt is None or dt < best_dt:
                best, best_dt = c, dt
    return best, cores


def cpu_reference_run(n_sample, reps, threads):
    """Time the reference TemporalModel (dense as written, fp32, MKL-DNN) on the host: the real
    reference class when its archive is present, else the oracle port.  -> frames/s, s, kind."""
    import torch
    from oracle import temporal_model_oracle as orc
    torch.set_num_threads(threads)
    fwd, kind = make_cpu_reference(reference_model_module())
    x = orc.make_input(n_sample, T, J, F, seed=1)
    with torch.no_grad():
        fwd(x[: max(1, n_sample // 8)])  # warm-up (thread pool, primitives)
        t0 = time.perf_counter()
        for _ in range(reps):
            y = fwd(x)
        dt = time.perf_counter() - t0
    assert y.shape == (n_sample, 1, J, 3)
    return n_sample * reps / dt, dt, kind


def cudnn_reference_arch(dev, x, our_value):
    """TemporalModel (dense as written, common/model.py:126-138) built from stock torch.nn modules
    and run by PyTorch/cuDNN on the GPU: fp32 with TF32 convolutions (PyTorch's default) and bf16
    autocast.  Random weights; only the time matters."""
    import torch
    import torch.nn as nn

    class Ref(nn.Module):
        def __init__(self):
            super().__init__()
            self.expand = nn.Conv1d(J * F, C, ARC[0], bias=False)
            self.expand_bn = nn.BatchNorm1d(C)
            convs, bns, self.pads, d = [], [], [], ARC[0]
            for w in ARC[1:]:
                self.pads.append((w - 1) * d // 2)
                convs += [nn.Conv1d(C, C, w, dilation=d, bias=False), nn.Conv1d(C, C, 1, bias=False)]
                bns += [nn.BatchNorm1d(C), nn.BatchNorm1d(C)]
                d *= w
            self.convs, self.bns = nn.ModuleList(convs), nn.ModuleList(bns)
            self.shrink = nn.Conv1d(C, J * 3, 1)

        def forward(self, x):
            n = x.shape[0]
            x = x.view(n, x.shape[1], -1).permute(0, 2, 1)
            x = torch.relu(self.expand_bn(self.expand(x)))
            for i, p in enumerate(self.pads):
                res = x[:, :, p: x.shape[2] - p]
                x = torch.relu(self.bns[2 * i](self.convs[2 * i](x)))
                x = res + torch.relu(self.bns[2 * i + 1](self.convs[2 * i + 1](x)))
            return self.shrink(x).permute(0, 2, 1).reshape(n, -1, J, 3)

    torch.backends.cudnn.benchmark = True
    ref_mod = reference_model_module()
    if ref_mod is not None:   # the reference's own class, unmodified
        ref = ref_mod.TemporalModel(J, F, J, filter_widths=ARC, causal=False, dropout=0.25,
                                    channels=C).to(dev).eval()
        impl = "reference common/model.py TemporalModel (staged archive)"
    else:
        ref = Ref().to(dev).eval()
        impl = "re-statement of the reference architecture (no staged reference on this box)"
    out = {"implementation": impl}
    for name, autocast in (("fp32_tf32", False), ("bf16_autocast", True)):
        def run():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                return ref(x)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        out[name] = {"ms_per_step": ms, "frames_per_s": N_PER_GPU / ms * 1e3,
                     "speedup_of_value": our_value / (N_PER_GPU / ms * 1e3)}
    out["target"] = "north_star: >= 20x the reference PyTorch/cuDNN TemporalModel frames/s on this GPU"
    del ref
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    n_sample = 32
    import torch
    from oracle import temporal_model_oracle as orc
    threads, cores = pick_cpu_threads()
    torch.set_num_threads(threads)
    fwd, kind = make_cpu_reference(reference_model_module())
    x = orc.make_input(n_sample, T, J, F, seed=1)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 3))):
            fwd(x)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fwd(x)
        dt = time.perf_counter() - t0
    value = n_sample * args.steps / dt
    what = ("the reference's own common/model.py TemporalModel (unmodified, staged archive)"
            if kind == "reference" else "oracle forward_torch port of the reference TemporalModel")
    sample = (f"{n_sample} windows of T=243 per step (bounded sample of the N=1024 batch; rows are "
              f"independent), {what}, dense-as-written, fp32, torch CPU, {threads} threads "
              f"(best of a calibration over thread counts; {cores} usable cores)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def synthetic_stream(n_seq, seed=0):
    """H36M-shaped synthetic stream of SURVEY §8d cfg4: `n_seq` sequences of 1000-6000 frames,
    17 joints, 2-D keypoints ~U(-1, 1) and 3-D joints ~N(0, 0.5^2) m, float32."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lens = rng.integers(1000, 6001, size=n_seq)
    p2 = [rng.uniform(-1, 1, (int(n), J, F)).astype(np.float32) for n in lens]
    p3 = [rng.normal(0, 0.5, (int(n), J, 3)).astype(np.float32) for n in lens]
    return lens, p2, p3


def measure_train(dev, rank, world, steps, warmup, n_seq, compress=None):
    """BASELINE configs[2] (world = 1) / configs[3] (world > 1): TemporalModelOptimized1f training
    step exactly as run.py:401-420 drives it -- batch from the (device-resident) ChunkedGenerator,
    root joint zeroed, forward, mpjpe, backward, Adam(amsgrad) -- with this repo's fused loss and
    optimiser.  Data parallel: global batch 1024 x world rows, rows sharded by rank, one gradient
    all-reduce per step (GradientReducer, overlapped with the backward).  Returns a dict."""
    import torch
    import torch.distributed as dist
    import videopose3d_b200 as vp
    from videopose3d_b200 import generators as G, loss as vloss
    from videopose3d_b200.data_parallel import GradientReducer
    from videopose3d_b200.optim import FusedAdam

    lens, p2, p3 = synthetic_stream(n_seq, seed=0)
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    gen = G.ChunkedGenerator(N_PER_GPU * world, None, p3, p2, 1, pad=121, causal_shift=0, shuffle=True,
                             random_seed=1234, augment=True, kps_left=left, kps_right=right,
                             joints_left=left, joints_right=right, endless=True, device=dev,
                             rank=rank, world_size=world)
    it = gen.next_epoch()
    torch.manual_seed(0)   # identical initial parameters on every rank
    model = vp.TemporalModelOptimized1f(J, F, J, filter_widths=ARC, causal=False, dropout=0.25,
                                        channels=C).to(dev).train()
    opt = FusedAdam(model.parameters(), lr=1e-3, amsgrad=True)
    overlap = bool(int(os.environ.get("VP3D_BENCH_DP_OVERLAP", "1")))
    reserve = int(os.environ.get("VP3D_BENCH_DP_RESERVE_SMS", "0"))
    reducer = GradientReducer(overlap=overlap, compress=compress, reserve_sms=reserve) if world > 1 else None

    def step():
        _, y3, x2 = next(it)
        y3[:, :, 0] = 0                       # run.py:407
        opt.zero_grad()
        loss = vloss.mpjpe(model(x2), y3)
        loss.backward()
        opt.step()
        return loss

    def timed(n):
        """(device ms/step with the launch queue kept full, wall ms/step when the loss is read back
        every step as run.py:414 does, last loss)."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            loss = step()
        b.record()
        torch.cuda.synchronize()
        gpu_ms = a.elapsed_time(b) / n
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            loss = step()
            last = loss.item()                # run.py:414 reads the loss every step
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        return gpu_ms, wall / n * 1e3, float(last)

    out = {}
    if world > 1:
        # the same step without the collective first (per-rank cost of the local work in THIS run)
        for _ in range(max(3, warmup)):
            step()
        local_ms, local_wall_ms, _ = timed(steps)
        reducer.attach(model)
        out["local_step_ms_no_collective"] = local_ms
    # (NCCL sets its channels up lazily: the first collectives of a process are several times
    # slower, and a 3-step warm-up left them inside the timed window on some boxes)
    for _ in range(max(12 if world > 1 else 3, warmup)):
        step()
    launches_bwd = model.last_launch_count()
    gpu_ms, wall_ms, last_loss = timed(steps)
    if world > 1:
        t = torch.tensor([gpu_ms, wall_ms, out["local_step_ms_no_collective"]], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gpu_ms, wall_ms, local_ms = (float(v) for v in t)
        out["local_step_ms_no_collective"] = local_ms
    peak_tf, _, _ = load_peaks()
    sustained = load_sustained_peak()
    tf = FLOPS_PER_SAMPLE_TRAIN * N_PER_GPU / (gpu_ms * 1e-3) / 1e12
    out.update({
        "workload": ("TemporalModelOptimized1f arc=3,3,3,3,3 C=1024 training step: device ChunkedGenerator "
                     f"batch ({n_seq} sequences of 1000-6000 frames, pad 121, shuffle + flip augmentation) "
                     "-> forward (BatchNorm batch statistics, dropout 0.25) -> fused mpjpe -> backward -> "
                     "FusedAdam(amsgrad), N=1024 windows per GPU"
                     + (" (BASELINE configs[2])" if world == 1 else
                        f", global batch {N_PER_GPU * world} rows sharded over {world} ranks, one gradient "
                        "all-reduce per step (BASELINE configs[3])")),
        "ms_per_step": gpu_ms, "ms_per_step_wall_incl_loss_item": wall_ms,
        "frames_per_s": N_PER_GPU * world / (gpu_ms * 1e-3),
        "frames_per_s_wall": N_PER_GPU * world / (wall_ms * 1e-3),
        "executed_tflops_per_s_per_gpu": tf,
        "frac_of_bf16_peak_burst": tf / peak_tf, "frac_of_bf16_peak_sustained": tf / sustained,
        "dtype": "bf16 operands, fp32 accumulate / statistics / master weights",
        "steps": steps, "last_loss": last_loss, "h2d_bytes_per_step": 0,
        "timing": "ms_per_step: CUDA events around `steps` back-to-back steps (launch queue full, max "
                  "over ranks); ms_per_step_wall_incl_loss_item: host clock with loss.item() after "
                  "every step as run.py does; the step's working set (~1 GB) exceeds L2",
    })
    if world > 1:
        grad_bytes = sum(p.numel() for p in model.parameters()) * (2 if compress == "bf16" else 4)
        out.update({
            "parallelism": f"dp{world}: rows of each global batch sharded by rank, per-GPU BatchNorm "
                           "statistics, ONE gradient all-reduce per step (NCCL, staged slices on a side "
                           "stream overlapping the remaining backward)",
            "allreduce_bytes_per_step": grad_bytes, "allreduce_wire_dtype": compress or "fp32",
            "overlap": overlap, "sm_limit": os.environ.get("VP3D_SM_LIMIT"),
            "allreduce_slices_per_step": reducer.launched // max(1, steps + max(3, warmup)),
            "exposed_collective_ms": gpu_ms - out["local_step_ms_no_collective"],
            "weak_scaling_efficiency_vs_local_step": out["local_step_ms_no_collective"] / gpu_ms,
        })
    del model, opt, gen
    torch.cuda.empty_cache()
    return out


def cudnn_train_step(dev):
    """The reference's TemporalModelOptimized1f training step on stock PyTorch/cuDNN on this GPU
    (TF32 default and bf16 autocast), torch.optim.Adam(amsgrad), same shapes; time only."""
    import torch
    from oracle import temporal_model_oracle as orc
    ref_mod = reference_model_module()
    if ref_mod is None:
        return {"unavailable": "no staged reference on this box"}
    torch.backends.cudnn.benchmark = True
    x = orc.make_input(N_PER_GPU, T, J, F, seed=3).to(dev)
    y = torch.randn(N_PER_GPU, 1, J, 3, device=dev) * 0.3
    out = {"implementation": "reference common/model.py TemporalModelOptimized1f (staged archive)"}
    for name, autocast in (("fp32_tf32", False), ("bf16_autocast", True)):
        m = ref_mod.TemporalModelOptimized1f(J, F, J, filter_widths=ARC, causal=False, dropout=0.25,
                                             channels=C).to(dev).train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, amsgrad=True)

        def step():
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                pred = m(x)
            loss = torch.mean(torch.norm(pred.float() - y, dim=-1))
            loss.backward()
            opt.step()
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        out[name] = {"ms_per_step": ms, "frames_per_s": N_PER_GPU / ms * 1e3}
        del m, opt
        torch.cuda.empty_cache()
    return out


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import videopose3d_b200 as vp
    from videopose3d_b200 import _capi
    from oracle import temporal_model_oracle as orc

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        # NCCL kernels on a high-priority stream: the gradient all-reduce overlaps persistent
        # one-CTA-per-SM GEMM grids; at default priority its CTAs queue behind every pending compute
        # CTA, the two ranks enter the collective far apart and spin on each other for milliseconds
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            dist.init_process_group("nccl", device_id=dev, pg_options=opts)
        except Exception:
            dist.init_process_group("nccl", device_id=dev)

    # random-init weights of the named architecture (no datasets / checkpoints offline)
    sd = orc.make_state_dict(J, F, J, ARC, C, seed=0)
    model = vp.TemporalModel(J, F, J, filter_widths=ARC, causal=False, dropout=0.25, channels=C)
    model.load_state_dict(sd)
    model = model.to(dev).eval().set_precision(args.precision)

    n_buf = 8  # 8 x 33.8 MB distinct inputs
    xs = [orc.make_input(N_PER_GPU, T, J, F, seed=100 + rank * n_buf + i).to(dev) for i in range(n_buf)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    lib = _capi.load()
    with torch.no_grad():
        y = model(xs[0])
        torch.cuda.synchronize()
        launches_per_step = model.last_launch_count()
        for i in range(args.warmup):
            y = model(xs[i % n_buf])
        torch.cuda.synchronize()

        # ---------------- device-resident timing (value) + roofline bracket
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        # the dominant launch is the block-1 k-tap conv: 9th from the end of the forward's launch list
        # (conv, 1x1 for each of the 4 blocks, then shrink), whatever precedes it (input pack fused
        # into the expand GEMM or not)
        dominant_index = launches_per_step - 9
        _capi.check(lib.vp3d_profile_launch(model._plan, dominant_index), "profile_launch")
        sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ
                               else _visible_index(local_rank))
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler.start()
        t_wall0 = time.perf_counter()
        for i in range(args.steps):
            flush.zero_()                      # evict L2 between timed iterations (not timed)
            starts[i].record()
            y = model(xs[i % n_buf])
            stops[i].record()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"pose_3d": y})
        step_ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
        total_ms = float(sum(step_ms))
        ms = _capi.ctypes.c_float()
        cnt = _capi.ctypes.c_int()
        _capi.check(lib.vp3d_profile_read(model._plan, _capi.ctypes.byref(ms), _capi.ctypes.byref(cnt)),
                    "profile_read")
        _capi.check(lib.vp3d_profile_launch(model._plan, -1), "profile_launch")
        dom_ms = ms.value / max(cnt.value, 1)

        # ---------------- end-to-end through the host-buffer API
        old_affinity = bind_to_gpu_numa_node(_visible_index(local_rank))
        xh = [orc.make_input(N_PER_GPU, T, J, F, seed=500 + rank * 2 + i).pin_memory() for i in range(2)]
        yh = torch.empty((N_PER_GPU, 1, J, 3), dtype=torch.float32).pin_memory()
        for i in range(max(3, args.warmup // 4)):
            model.forward_host(xh[i % 2], out=yh)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e2e_steps = args.steps
        # (a) one synchronous call per step: copy-in, kernels, copy-out, sync
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            model.forward_host(xh[i % 2], out=yh)
        torch.cuda.synchronize()
        e2e_sync_s = time.perf_counter() - t0
        # (b) the same per-step work through the two-slot pipelined calls: the PCIe copy of step
        # i+1 overlaps the kernels of step i; every step still moves its own input and output
        yhs = [yh, torch.empty_like(yh).pin_memory()]
        # untimed warm-up of the pipelined path itself: the device-timed loop above moved nothing
        # over PCIe for milliseconds, and the first copies after such a pause ran at half rate on
        # some boxes (link power state) -- 1.2 instead of 0.65 ms/step over a 30-step window
        for i in range(max(32, args.warmup)):
            s = i & 1
            if i >= 2:
                model.forward_host_wait(s)
            model.forward_host_submit(xh[s], yhs[s], s)
        model.forward_host_wait(0)
        model.forward_host_wait(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            s = i & 1
            if i >= 2:
                model.forward_host_wait(s)
            model.forward_host_submit(xh[s], yhs[s], s)
        for i in range(max(0, e2e_steps - 2), e2e_steps):
            model.forward_host_wait(i & 1)
        e2e_s = time.perf_counter() - t0
        if old_affinity is not None:
            os.sched_setaffinity(0, old_affinity)

    # max over ranks
    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])
        dist.barrier()

    # ---------------- the other precision modes (short, rank 0 prints them; not the headline)
    modes = {}
    if world == 1 and not args.no_modes:
        with torch.no_grad():
            for prec in ("fp16", "bf16", "mixed", "bf16x3"):
                if prec == args.precision:
                    continue
                model.set_precision(prec)
                for i in range(3):
                    model(xs[i % n_buf])
                torch.cuda.synchronize()
                evs = []
                for i in range(10):
                    flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    model(xs[i % n_buf])
                    b.record()
                    evs.append((a, b))
                torch.cuda.synchronize()
                m_ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
                modes[prec] = {"ms_per_step": m_ms, "frames_per_s": N_PER_GPU / (m_ms * 1e-3)}
            model.set_precision(args.precision)
    del xs, flush
    torch.cuda.empty_cache()

    # ---------------- training path (configs[2] at N = 1, configs[3] data-parallel at N > 1)
    train = None
    if not args.no_train:
        try:
            train = measure_train(dev, rank, world, args.train_steps, 5, args.sequences,
                                  compress=args.grad_wire)
        except Exception as e:  # the headline must survive a failure of the side measurement
            train = {"error": repr(e)[:300]}

    frames = N_PER_GPU * world * args.steps
    value = frames / (total_ms * 1e-3)
    e2e_value = N_PER_GPU * world * e2e_steps / e2e_s
    peak_tf, peak_gbs, peak_src = load_peaks()
    achieved_tf = DOMINANT_FLOPS_PER_LAUNCH / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0

    line = None
    if rank == 0:
        traffic, traffic_src = load_traffic("dominant_eval_" + args.precision)
        step_tf = FLOPS_PER_SAMPLE_CONE * N_PER_GPU / (total_ms / args.steps * 1e-3) / 1e12
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads, cores = pick_cpu_threads()
            n_sample = 64
            cpu_value, cpu_dt, cpu_kind = cpu_reference_run(n_sample, 2, threads)
            cpu = {"value": cpu_value, "unit": UNIT, "cores": threads, "kind": cpu_kind,
                   "sample": f"2 x {n_sample} windows of T=243 ({cpu_dt:.1f} s), "
                             + ("the reference's own TemporalModel (unmodified, staged archive)"
                                if cpu_kind == "reference" else "oracle forward_torch port")
                             + f", dense-as-written, fp32 torch CPU, {threads} "
                             f"threads = best of a calibration; {cores} usable cores"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp16": "fp16 (IEEE fp16 operands and activations, fp32 accumulate)",
                      "bf16": "bf16", "bf16x3": "bf16x3 (split-bf16 operands, fp32 accumulate)",
                      "mixed": "bf16 (residual blocks plain bf16 on a hi+lo residual stream; expand "
                               "and shrink split-bf16; fp32 accumulate)"}[args.precision],
            "data": "synthetic",
            "config": {"workload": WORKLOAD},
            "config_detail": {
                "batch_per_gpu": N_PER_GPU, "receptive_field": 243,
                "parallelism": f"dp{world} (eval: independent batches per rank, no collective; the "
                               "data-parallel training step with its gradient all-reduce is `train_dp`)",
                "schedule": "eval dependency-cone (strided) schedule: 352.6 MFLOP/sample executed "
                            "vs 5217.8 MFLOP/sample dense-as-written",
                "l2": "256 MiB memset between timed steps + 8 rotating 33.8 MB input buffers",
                "timing": "CUDA events per step, summed; max over ranks",
                "precision_mode": args.precision,
            },
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": N_PER_GPU * T * J * F * 4,
                    "d2h_bytes_per_step": N_PER_GPU * J * 3 * 4,
                    "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "api": "TemporalModel.forward_host_submit/_wait -> vp3d_forward_eval_host_submit/"
                           "_wait (pinned host buffers, two slots: copy-in of step i+1 overlaps the "
                           "kernels of step i)",
                    "host_numa_binding": "process bound to the GPU-local cores (NVML) while the pinned "
                                         "buffers were allocated and the copies issued"
                                         if old_affinity is not None else "none (already local / unavailable)",
                    "sync_call_ms_per_step": e2e_sync_s / e2e_steps * 1e3,
                    "sync_call_value": N_PER_GPU * e2e_steps / e2e_sync_s},
            "gpu_launches": launches_per_step * args.steps,
            "launches_per_step": launches_per_step,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "algorithmic_bytes": DOMINANT_ALGORITHMIC_BYTES, "peak_source": peak_src,
                         "kernel": "conv_gemm_kernel<256> block-1 3-tap conv (M=27648,K=3072,N=1024)",
                         "flops_per_launch": DOMINANT_FLOPS_PER_LAUNCH, "ms_per_launch": dom_ms,
                         "launches_timed": cnt.value},
            "roofline_step": {"bound": "tensor", "achieved": step_tf, "peak": peak_tf, "unit": "TFLOP/s",
                              "frac": step_tf / peak_tf,
                              "frac_of_sustained_peak": step_tf / load_sustained_peak(),
                              "what": "executed FLOPs of the whole forward (352.6 MFLOP/sample x 1024) / "
                                      "ms_per_step, per GPU; all launches of the step incl. input pack, "
                                      "expand and shrink"},
            "executed_tflops_per_s": FLOPS_PER_SAMPLE_CONE * N_PER_GPU * world * args.steps / (total_ms * 1e-3) / 1e12,
            "dense_equivalent_tflops_per_s": FLOPS_PER_SAMPLE_DENSE * N_PER_GPU * world * args.steps / (total_ms * 1e-3) / 1e12,
            "wall_s_timed_region": t_wall,
            "input_frames_per_s": value * T,   # secondary column of SURVEY §8d: N*T / time
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if modes:
            line["modes"] = modes
        if train is not None:
            line["train" if world == 1 else "train_dp"] = train
        if world == 1 and not args.no_cudnn:
            # informational: the reference architecture executed by stock PyTorch/cuDNN on this same
            # GPU and batch (the number north_star asks to beat by >= 20x); not the driver's
            # reference arm, which is the CPU run of --impl reference
            try:
                x_ref = orc.make_input(N_PER_GPU, T, J, F, seed=100).to(dev)
                line["cudnn_same_gpu"] = cudnn_reference_arch(dev, x_ref, value)
                del x_ref
                if isinstance(train, dict) and "ms_per_step" in train:
                    ct = cudnn_train_step(dev)
                    for k in ("fp32_tf32", "bf16_autocast"):
                        if k in ct:
                            ct[k]["speedup_of_train_step"] = ct[k]["ms_per_step"] / train["ms_per_step"]
                    line["train"]["cudnn_same_gpu"] = ct
            except Exception as e:  # never let the side measurement break the bench line
                line.setdefault("cudnn_same_gpu", {})["error"] = repr(e)[:200]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def run_input_pipeline(args):
    """SURVEY §8 row f1: the training input pipeline.  Device-resident generator
    (videopose3d_b200.generators.ChunkedGenerator -> vp3d_gather_windows) against the CPU port of
    the reference's ChunkedGenerator + cast + H2D copy (generators.py:99-160, run.py:401-406), on
    an H36M-shaped synthetic stream (SURVEY §8d cfg4), and the training step fed either way."""
    import numpy as np
    import torch
    import videopose3d_b200 as vp
    from videopose3d_b200 import generators as G
    from oracle import generator_oracle as gorc  # CPU baseline leg only

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rng = np.random.RandomState(0)
    n_seq = args.sequences
    lens = rng.randint(1000, 6001, size=n_seq)
    p2 = [rng.uniform(-1, 1, (n, J, F)).astype(np.float32) for n in lens]
    p3 = [rng.normal(0, 0.5, (n, J, 3)).astype(np.float32) for n in lens]
    left, right = [4, 5, 6, 11, 12, 13], [1, 2, 3, 14, 15, 16]
    kw = dict(pad=121, causal_shift=0, shuffle=True, random_seed=1234, augment=True, kps_left=left,
              kps_right=right, joints_left=left, joints_right=right)
    t0 = time.perf_counter()
    gen = G.ChunkedGenerator(N_PER_GPU, None, p3, p2, 1, device=dev, **kw)
    torch.cuda.synchronize()
    upload_s = time.perf_counter() - t0
    it = gen.next_epoch()
    t0 = time.perf_counter()
    next(it)
    torch.cuda.synchronize()
    epoch_start_s = time.perf_counter() - t0   # permutation draw + table upload + first batch
    for _ in range(max(3, args.warmup)):
        next(it)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    for a, b in ev:
        flush.zero_()
        a.record()
        batch = next(it)
        b.record()
    torch.cuda.synchronize()
    gather_ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    # kernel-only time of the dominant gather (2-D windows): the C-ABI entry point called back to
    # back on 8 rotating 33.8 MB outputs (working set > L2), CUDA events around the burst
    import ctypes
    from videopose3d_b200 import _capi
    lib = _capi.load()
    outs = [torch.empty((N_PER_GPU, T, J, F), dtype=torch.float32, device=dev) for _ in range(8)]
    rows = gen._rows_dev
    descs = []
    for k in range(args.steps):
        d = _capi.GatherDesc()
        d.src, d.seq_first, d.seq_len = gen._p2.data.data_ptr(), gen._p2.seq_first.data_ptr(), gen._p2.seq_len.data_ptr()
        d.rows = rows.data_ptr() + 16 * N_PER_GPU * (k % 64)
        d.src_joint = gen._p2.src_joint.data_ptr()
        d.out = outs[k % 8].data_ptr()
        d.n_windows, d.frames, d.joints, d.features, d.first_offset = N_PER_GPU, T, J, F, -121
        descs.append(d)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for d in descs[:8]:
        _capi.check(lib.vp3d_gather_windows(ctypes.byref(d), stream), "vp3d_gather_windows")
    torch.cuda.synchronize()
    ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ka.record()
    for d in descs:
        lib.vp3d_gather_windows(ctypes.byref(d), stream)
    kb.record()
    torch.cuda.synchronize()
    kernel_ms = ka.elapsed_time(kb) / args.steps
    win_bytes = N_PER_GPU * T * J * F * 4
    algo_bytes = 2 * win_bytes              # every output element is read once and written once
    _, peak_gbs, peak_src = load_peaks()
    # host wall clock per batch of the device generator (Python + 2 launches, GPU idle otherwise)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        batch = next(it)
    torch.cuda.synchronize()
    dev_wall_ms = (time.perf_counter() - t0) / args.steps * 1e3

    # CPU port of the reference path: generator batch -> float32 -> pinned -> H2D
    orc = gorc.ChunkedGeneratorOracle(N_PER_GPU, None, p3, p2, 1, **kw)
    oit = orc.next_epoch()
    next(oit)
    cpu_batches = 4
    t0 = time.perf_counter()
    for _ in range(cpu_batches):
        _, b3, b2 = next(oit)
    cpu_gen_ms = (time.perf_counter() - t0) / cpu_batches * 1e3
    t0 = time.perf_counter()
    for _ in range(cpu_batches):
        _, b3, b2 = next(oit)
        x = torch.from_numpy(b2.astype("float32")).cuda()
        y = torch.from_numpy(b3.astype("float32")).cuda()
    torch.cuda.synchronize()
    cpu_fed_ms = (time.perf_counter() - t0) / cpu_batches * 1e3

    # training step (Optimized1f, fwd + bwd + AMSGrad) fed by either pipeline.  "stock" = the
    # reference's torch.optim.Adam + torch loss expression (run.py:252, 413); "fused" = this
    # repo's single-launch FusedAdam + fused mpjpe (rows f4, f2).
    from videopose3d_b200 import loss as vloss
    from videopose3d_b200.optim import FusedAdam

    def make(kind):
        torch.manual_seed(0)
        m = vp.TemporalModelOptimized1f(J, F, J, filter_widths=ARC, channels=C).to(dev).train()
        if kind == "fused":
            opt = FusedAdam(m.parameters(), lr=1e-3, amsgrad=True)
            crit = vloss.mpjpe
        else:
            opt = torch.optim.Adam(m.parameters(), lr=1e-3, amsgrad=True)
            crit = lambda p, y: torch.mean(torch.norm(p - y, dim=-1))  # noqa: E731

        def step(x, y):
            opt.zero_grad()
            loss = crit(m(x), y)
            loss.backward()
            opt.step()
            return loss
        return step

    def timed_device_fed(step):
        for _ in range(3):
            _, y, x = next(it)
            step(x, y)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(args.steps):
            _, y, x = next(it)
            loss = step(x, y)
        b.record()
        loss.item()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / args.steps * 1e3, a.elapsed_time(b) / args.steps

    step_stock, step_fused = make("stock"), make("fused")
    train_dev_ms, train_dev_gpu_ms = timed_device_fed(step_stock)
    train_fused_ms, train_fused_gpu_ms = timed_device_fed(step_fused)
    host_steps = 4
    t0 = time.perf_counter()
    for _ in range(host_steps):
        _, b3, b2 = next(oit)
        loss = step_stock(torch.from_numpy(b2.astype("float32")).cuda(),
                          torch.from_numpy(b3.astype("float32")).cuda())
    loss.item()
    torch.cuda.synchronize()
    train_host_ms = (time.perf_counter() - t0) / host_steps * 1e3

    line = {
        "what": "train_input_pipeline (SURVEY 8 f1)", "n_gpus": 1, "steps": args.steps,
        "config": {"workload": f"ChunkedGenerator batch 1024 x (243,17,2) + (1,17,3), shuffle + flip "
                               f"augmentation, {n_seq} sequences of 1000-6000 frames "
                               f"({int(lens.sum())} frames, {int(lens.sum()) * J * F * 4 / 1e6:.0f} MB of 2-D input)",
                   "l2": "256 MiB memset between timed gathers"},
        "device_generator": {"gather_ms_per_batch_incl_launch_gaps": gather_ms, "host_wall_ms_per_batch": dev_wall_ms,
                             "dataset_upload_s": upload_s, "epoch_start_s": epoch_start_s,
                             "h2d_bytes_per_step": 0, "gpu_launches_per_batch": 2},
        "roofline": {"bound": "hbm", "achieved": algo_bytes / (kernel_ms * 1e-3) / 1e9, "peak": peak_gbs,
                     "unit": "GB/s", "frac": algo_bytes / (kernel_ms * 1e-3) / 1e9 / peak_gbs,
                     "algorithmic_bytes": algo_bytes, "ms_per_launch": kernel_ms,
                     "traffic": 39.4e6, "traffic_source": "ncu --set full dram read+write of this launch "
                     "(profiles/r1n_ncu_full_gather.csv; most reads and part of the writes stay in L2)",
                     "peak_source": peak_src,
                     "kernel": "gather_windows_kernel, 2-D windows 1024 x (243,17,2) fp32"},
        "cpu_baseline": {"generator_ms_per_batch": cpu_gen_ms, "generator_cast_h2d_ms_per_batch": cpu_fed_ms,
                         "kind": "port", "cores": 1,
                         "sample": f"{cpu_batches} batches, oracle ChunkedGeneratorOracle (NumPy, single "
                                   "thread like the reference's Python loop) + astype(float32) + .cuda()"},
        "train_step_ms": {
            "host_generator+stock_adam (reference pipeline, CPU port)": train_host_ms,
            "device_generator+stock_adam": train_dev_ms,
            "device_generator+fused_adam+fused_mpjpe": train_fused_ms,
            "device_generator+stock_adam (GPU time, events)": train_dev_gpu_ms,
            "device_generator+fused_adam+fused_mpjpe (GPU time, events)": train_fused_gpu_ms},
        "train_frames_per_s": {"host_fed": N_PER_GPU / (train_host_ms * 1e-3),
                               "device_fed_stock": N_PER_GPU / (train_dev_ms * 1e-3),
                               "device_fed_fused": N_PER_GPU / (train_fused_ms * 1e-3)},
    }
    print(json.dumps(line), flush=True)
    return line


def dump_outputs(out_dir, arrays):
    """Write each tensor as `out_dir/<name>.npy` in float32, so that two builds run with the same
    arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def _visible_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    try:
        return int(vis.split(",")[local_rank])
    except Exception:
        return local_rank


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 200, or 50 with --input-pipeline)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "mixed", "bf16", "bf16x3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cudnn", action="store_true",
                    help="skip the informational PyTorch/cuDNN measurement of the reference architecture")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step block")
    ap.add_argument("--no-modes", action="store_true", help="skip the short runs of the other precision modes")
    ap.add_argument("--train-steps", type=int, default=30)
    ap.add_argument("--grad-wire", default=None, choices=[None, "bf16"],
                    help="wire dtype of the gradient all-reduce in the data-parallel training block")
    ap.add_argument("--input-pipeline", action="store_true",
                    help="measure the training input pipeline (device generator vs CPU port) instead")
    ap.add_argument("--sequences", type=int, default=300)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's prediction (N x 1 x 17 x 3, "
                         "float32) as DIR/pose_3d.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 50 if args.input_pipeline else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.input_pipeline or args.impl == "reference"):
        ap.error("--dump-outputs writes the eval forward of --impl ours only")
    if args.input_pipeline:
        run_input_pipeline(args)
        return
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
               f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port", "29531",
               os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--precision", args.precision,
               "--train-steps", str(args.train_steps), "--sequences", str(args.sequences)]
        cmd += ["--no-train"] if args.no_train else []
        cmd += ["--grad-wire", args.grad_wire] if args.grad_wire else []
        cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else []
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()

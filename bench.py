#!/usr/bin/env python
"""Headline benchmark: clips/sec (10 s @ 32 kHz) of the mn10_as training step (mel + forward + backward +
Adam, the body of reference ex_audioset.py:135-199) on N B200s of one node, weak scaling by clip batch.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference algorithm on the host cores (oracle port, CPU)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions of every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CLIP_SAMPLES = 320000            # 10 s @ 32 kHz
N_CLASSES = 527
METRIC = "clips/sec (10s@32kHz) mn10_as fwd+bwd"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"],
                    help="ours: this package; reference: the reference's CPU PyTorch path on the host cores; "
                         "reference-gpu: the reference's own modules (cuFFT/cuDNN/cuBLAS) on the same GPUs")
    ap.add_argument("--amp", default="none", choices=["none", "bf16"], help="reference-gpu only: torch.autocast dtype")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the gpu_baseline leg of the default run")
    ap.add_argument("--batch", type=int, default=256, help="clips per GPU per step")
    ap.add_argument("--precision", default=os.environ.get("EAT_PRECISION", "fp32"), choices=["fp32", "bf16"])
    ap.add_argument("--model", default="mn10", choices=["mn04", "mn10", "mn20", "mn40", "dymn04", "dymn10", "dymn20"])
    ap.add_argument("--mode", default="train", choices=["train", "eval"],
                    help="train: the headline training step; eval: mel + forward only (BASELINE.json configs[1])")
    ap.add_argument("--cpu-baseline-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sync-readback", action="store_true",
                    help="e2e loop: read the loss back with a blocking .cpu() after every step instead of the pipelined LossReader")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0), for comparing two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write {name: device tensor} as DIR/<name>.npy in float32 / float64, at most DUMP_MAX_BYTES in all.  A larger
    tensor is cut to a fixed sample (seeded indices, sorted), the same for every run with the same arguments."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    budget = DUMP_MAX_BYTES // max(len(arrays), 1)
    for name, t in arrays.items():
        t = t.detach().reshape(-1)
        t = t.double() if t.dtype == torch.float64 else t.float()
        cap = budget // t.element_size()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop, self.thread = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def _synth_batch(batch, seed):
    """the synthetic shard both arms train on: waveforms, labels, teacher soft targets, unknown-teacher mask"""
    from efficientat_b200.synth import synth_labels, synth_waveform
    wave = synth_waveform(batch, CLIP_SAMPLES, seed=1000 + seed)
    y = synth_labels(batch, N_CLASSES, seed=2000 + seed)
    teacher = torch.sigmoid(torch.randn(batch, N_CLASSES, generator=torch.Generator().manual_seed(3000 + seed)))
    known = torch.ones(batch, dtype=torch.bool)
    known[4::5] = False                                       # every 5th clip has no teacher entry (ex_audioset.py:166-177)
    return wave, y, teacher, known


def cpu_reference_step_factory(batch, model="mn10"):
    """One training step of the reference on the host: the reference's OWN modules from the oracle/_ref mirror when it
    is present (kind "reference"), else the oracle port of the same algorithm (kind "port").  Same step as the GPU arm:
    mel + mixup + forward + hard/distillation BCE with the unknown-teacher mask + backward + Adam."""
    from baseline import ref_step
    wave, y, teacher, known = _synth_batch(batch, 0)
    dev = torch.device("cpu")
    if ref_step.available():
        return ref_step.make_train_step(model, wave, y, teacher, known, dev), "reference"
    from oracle import mel_oracle, net_oracle
    from efficientat_b200.helpers.utils import mixup
    from efficientat_b200.models.mn.model import get_model
    from efficientat_b200.synth import synth_state_
    if model.startswith("dymn"):
        from efficientat_b200.models.dymn.model import get_model
    width = ref_step.WIDTH[model]
    torch.manual_seed(0)
    net = synth_state_(get_model(width_mult=width, verbose=False), seed=7)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    names = [k for k, _ in net.named_parameters()]
    for k in names:
        sd[k].requires_grad_(True)
    opt = torch.optim.Adam([sd[k] for k in names], lr=8e-4)
    fwd = net_oracle.dymn_forward if model.startswith("dymn") else net_oracle.mn_forward
    kd = 0.1

    def step():
        spec = mel_oracle.mel_forward(wave).unsqueeze(1)
        rn, lam = mixup(batch, 0.3)
        spec = spec * lam.reshape(batch, 1, 1, 1) + spec[rn] * (1. - lam.reshape(batch, 1, 1, 1))
        logits, _ = fwd(sd, spec, width_mult=width, training=True, **({"temperature": 30.0} if model.startswith("dymn") else {}))
        bce = torch.nn.functional.binary_cross_entropy_with_logits
        y_mix = y * lam.reshape(batch, 1) + y[rn] * (1. - lam.reshape(batch, 1))
        soft = bce(logits, teacher, reduction="none").mean(1) * lam + bce(logits, teacher[rn], reduction="none").mean(1) * (1. - lam)
        loss = kd * bce(logits, y_mix) + (1 - kd) * (soft * known.float()).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        return float(loss.detach())
    return step, "port"


def usable_cores():
    """host threads this process may actually use: scheduler affinity, capped by the cgroup CPU quota if there is one"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:                                                    # cgroup v2, then v1
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = max(1, min(n, quota // period))
        except Exception:
            pass
    return n


def time_cpu_reference(batch, steps, warmup, budget_s=150.0, model="mn10"):
    """-> (clips/s, s/step, threads, clips per step, kind).  The per-step sample is bounded: a two-clip calibration step
    (which is also a warm-up) sets the clips per step so that warm-up + timed steps stay within `budget_s`."""
    cores = usable_cores()
    one, kind = cpu_reference_step_factory(2, model)          # 2 clips: training-mode BatchNorm needs > 1 value per channel
    best = None
    for n in ([cores, 16] if cores > 16 else [cores]):      # a shared box may expose more CPUs than it lets us run on:
        torch.set_num_threads(n)                            # keep whichever thread count is actually faster
        one()                                               # first call pays allocator / thread-pool start-up
        t0 = time.perf_counter()
        one()
        dt1 = time.perf_counter() - t0
        if best is None or dt1 < best[0]:
            best = (dt1, n)
    t1, cores = best[0] / 2, best[1]                        # seconds per clip, threads used
    torch.set_num_threads(cores)
    batch = max(2, min(batch, int(budget_s / max(t1 * (steps + max(1, warmup)), 1e-6))))
    step, kind = cpu_reference_step_factory(batch, model)
    for _ in range(max(1, warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, cores, batch, kind


def _workload(args, where):
    return (f"{args.model}_as training step: mel + mixup + fwd + BCE/KD loss (unknown-teacher mask) + bwd + Adam "
            f"(ex_audioset.py:135-199), 10 s @ 32 kHz clips, {where}")


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU PyTorch implementation of the same step on the host cores (rank 0 only).
    Exactly --steps timed and --warmup untimed steps; each step is a bounded sample (clips per step calibrated so the
    whole run stays within ~2.5 minutes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, s_per_step, cores, b, kind = time_cpu_reference(args.cpu_baseline_batch, args.steps, args.warmup, model=args.model)
    what = "the reference's own modules (oracle/_ref mirror)" if kind == "reference" else "oracle port of the reference modules"
    sample = f"{args.steps} steps x {b} clips ({args.warmup} warm-up), same training step as the GPU arm, fp32, {what}"
    line = {"impl": "reference", "metric": METRIC if args.model == "mn10" else f"clips/sec (10s@32kHz) {args.model}_as fwd+bwd",
            "value": value, "unit": "clips/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": _workload(args, f"host cores, {b} clips per step (bounded sample of the batch-{args.batch} workload)"),
                       "model": f"{args.model}_as", "batch_per_step": b},
            "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_reference_gpu(model, mode, B, steps, warmup, dev, amp, world, seed):
    """the reference's own modules on this GPU (baseline/ref_step.py) -> (ms total over `steps`, peak GiB) or raises"""
    from baseline import ref_step
    torch.backends.cudnn.benchmark = True
    wave, y, teacher, known = (t.to(dev) for t in _synth_batch(B, seed))
    dt = {"none": None, "bf16": torch.bfloat16}[amp]
    if mode == "eval":
        step = ref_step.make_eval_step(model, wave, dev, amp=dt)
    else:
        step = ref_step.make_train_step(model, wave, y, teacher, known, dev, amp=dt, ddp=world > 1)
    torch.cuda.reset_peak_memory_stats(dev)
    for _ in range(max(warmup, 3)):
        step()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return ms, torch.cuda.max_memory_allocated(dev) / 2 ** 30


def gpu_baseline_entry(model, mode, B, steps, warmup, dev, amp, world, seed):
    from baseline import ref_step
    if not ref_step.available():
        return {"unavailable": "oracle/_ref (mirror of the reference checkout, made by oracle/make_ref.py) is not present"}
    try:
        ms, gib = time_reference_gpu(model, mode, B, steps, warmup, dev, amp, world, seed)
    except torch.cuda.OutOfMemoryError:
        torch.cuda.empty_cache()
        return {"unavailable": f"reference modules ran out of memory at batch {B}/GPU", "amp": amp}
    return {"value": world * B * steps / (ms * 1e-3), "unit": "clips/s", "ms_per_step": ms / steps, "steps": steps,
            "amp": amp, "batch_per_gpu": B, "peak_mem_gib": round(gib, 1),
            "what": "the reference's own nn.Modules (oracle/_ref mirror) through stock PyTorch: cuFFT + cuDNN + cuBLAS, "
                    "cudnn.benchmark, " + ("fp32 params / TF32 convolutions (PyTorch defaults)" if amp == "none" else "torch.autocast(bfloat16)")
                    + (", DistributedDataParallel" if world > 1 else "") + "; same synthetic batch and loop body "
                    "(ex_audioset.py:135-199 incl. its 3 loss read-backs per step)"}


def run_reference_gpu_arm(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl reference-gpu needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    with ClockSampler(local) as clocks:
        r = gpu_baseline_entry(args.model, args.mode, args.batch, args.steps, args.warmup, dev, args.amp, world, rank)
    if rank == 0:
        if "unavailable" in r:
            print(json.dumps({"impl": "reference-gpu", **r}), flush=True)
        else:
            line = {"impl": "reference-gpu", "metric": METRIC if (args.mode == "train" and args.model == "mn10") else
                    f"clips/sec (10s@32kHz) {args.model}_as {'fwd+bwd' if args.mode == 'train' else 'fwd'}",
                    "value": r["value"], "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                    "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f32" if args.amp == "none" else "bf16", "data": "synthetic",
                    "config": {"workload": _workload(args, f"batch {args.batch}/GPU") if args.mode == "train" else
                               f"{args.model}_as mel + eval forward, batch {args.batch}/GPU", "model": f"{args.model}_as",
                               "global_batch": args.batch * world, "parallelism": f"ddp{world}", "amp": args.amp},
                    "gpu_baseline": r, "clocks": clocks.summary()}
            print(json.dumps(line), flush=True)
    _shutdown(world)


# ----------------------------------------------------------------------------------------------- GPU arm
def algo_bytes(name, a):
    """Algorithmic HBM bytes of one launch from its C-ABI arguments (operands read once + result written once)."""
    sz = lambda code: 2 if code == 1 else 4
    if name == "eat_gemm_simt_fwd" or name == "eat_pw_tc_fwd":
        A, adt, W, wt, C, cdt, M, N, K = a[:9]
        res = a[17]
        return M * K * sz(adt) + M * N * sz(cdt) * (2 if res else 1) + N * K * 4
    if name == "eat_pw_tma_fwd":             # (A, W, w_trans, C, M, N, K, in_scale, in_shift, in_act, gate, rps, scale, shift, act, residual, ...)
        M, N, K, res = a[4], a[5], a[6], a[15]
        return M * K * 4 + M * N * 4 * (2 if res else 1) + N * K * 4
    if name == "eat_pw_tma_dyn_fwd":         # (A, W, att, dyn_k, w_trans, C, M, N, K, rps, scale, shift, act, residual, ...)
        nk, M, N, K, res = a[3], a[6], a[7], a[8], a[13]
        return M * K * 4 + M * N * 4 * (2 if res else 1) + nk * N * K * 4
    if name == "eat_pw_tc_dyn_fwd":          # + the dyn_k weight banks (read once; re-reads per tile hit L2)
        A, dt, W, att, nk, C, M, N, K, rps = a[:10]
        res = a[16]
        return M * K * sz(dt) + M * N * sz(dt) * (2 if res else 1) + nk * N * K * 4
    if name == "eat_pw_tc_wgrad_persample":  # G + A read once, per-sample gradients written once
        G, A, dt, S, M, N, K, rps = a[:8]
        return M * (N + K) * sz(dt) + (M // rps) * N * K * 4
    if name == "eat_dyn_wgrad_mix":          # S [B, n] read once, banks read + bank gradients written
        S, att, W, dW, datt, B, n, k = a[:8]
        return B * n * 4 + 2 * k * n * 4
    if name == "eat_gemm_simt_wgrad" or name == "eat_pw_tc_wgrad":
        G, gdt, A, adt, dW, db, M, N, K = a[:9]
        return M * N * sz(gdt) + M * K * sz(adt) + N * K * 4
    if name == "eat_dw_conv_fwd":
        inp, wt, out, dt, B, F, T, C, k, s = a[:10]
        Fo, To = (F + 2 * ((k - 1) // 2) - k) // s + 1, (T + 2 * ((k - 1) // 2) - k) // s + 1
        return B * C * sz(dt) * (F * T + Fo * To)
    if name in ("eat_bn_bwd_reduce", "eat_bn_bwd_apply"):
        gA = a[0]
        if name == "eat_bn_bwd_reduce":
            dt, B, P, C = a[9:13]
            return B * P * C * sz(dt) * (2 if gA else 1)
        dt, B, P, C = a[12:16]
        return B * P * C * sz(dt) * (3 if gA else 2)
    if name == "eat_se_bn_bwd_reduce":      # (dp, z, scale, shift, mean, act, dgate, part, parts, dtype, B, P, C): dp + z read, 4 partial sums written
        parts, dt, B, P, C = a[8:13]
        return 2 * B * P * C * sz(dt) + parts * 4 * B * C * 4
    if name == "eat_se_bn_bwd_combine":     # (part, parts, gate, dpool, invstd, B, C, s1, s2)
        parts, B, C = a[1], a[5], a[6]
        return (parts * 4 + 2) * B * C * 4
    if name == "eat_se_bwd_reduce":         # (dp, z, scale, shift, act, dgate, dtype, B, P, C)
        dt, B, P, C = a[6:10]
        return 2 * B * P * C * sz(dt)
    if name == "eat_bn_act_pool":           # (z, scale, shift, act, pool, mul, dtype, B, P, C)
        dt, B, P, C = a[6:10]
        return B * P * C * sz(dt)
    if name == "eat_dw_conv_dgrad_bnred":   # (dz, wt, res, din, z, ..., dtype, B, F, T, C, k, stride): dz + z read, din written
        res, dt, B, F, T, C, k, s = a[2], a[12], a[13], a[14], a[15], a[16], a[17], a[18]
        Fo, To = (F + 2 * ((k - 1) // 2) - k) // s + 1, (T + 2 * ((k - 1) // 2) - k) // s + 1
        return B * C * sz(dt) * (F * T * (3 if res else 2) + Fo * To)
    if name == "eat_dw_conv_dgrad":
        dz, wt, wbs, res, din, dt, B, F, T, C, k, s = a[:12]
        Fo, To = (F + 2 * ((k - 1) // 2) - k) // s + 1, (T + 2 * ((k - 1) // 2) - k) // s + 1
        return B * C * sz(dt) * (F * T * (2 if res else 1) + Fo * To)
    if name == "eat_dw_conv_wgrad":
        dz, inp, s0, s1, act, dw, dbs, dt, B, F, T, C, k, s = a[:14]
        Fo, To = (F + 2 * ((k - 1) // 2) - k) // s + 1, (T + 2 * ((k - 1) // 2) - k) // s + 1
        return B * C * sz(dt) * (F * T + Fo * To)
    if name == "eat_mel_fwd":
        B, N = a[1], a[2]
        hop, n_mels = a[5], a[12]
        return B * N * 4 + B * n_mels * (1 + (N - 1) // hop) * 4
    return None


# DRAM traffic of the dominant kernel from one `ncu --set full` capture (profiles/README.md): dram read + write bytes
# relative to the algorithmic bytes of the captured launch.  Used to scale the per-launch `traffic` figure.
NCU_TRAFFIC = {
    # `ncu --set full` capture (profiles/r02_ncu_full_pw_tma_wgrad_tma_mel.csv) of the data-gradient launch M = 2 048 000,
    # K = 16, N = 64 of pw_tma_kernel at B = 64: dram read 131.2 MB + write 467.0 MB against 655.4 MB algorithmic (the tail
    # of the output is still dirty in the 126 MB L2 when the kernel ends: no re-reads)
    "eat_pw_tma_fwd": {"dram_bytes": 131.18336e6 + 466.999552e6, "algorithmic_bytes": 2048000 * (16 + 64) * 4 + 64 * 16 * 4,
                       "capture": "profiles/r02_ncu_full_pw_tma_wgrad_tma_mel.csv"},
}


class KernelTimer:
    """Wraps the ctypes launchers: CUDA events around launches of the selected C-ABI entry points."""

    def __init__(self, lib, only=None):
        self.lib, self.only, self.records, self.orig = lib, only, [], {}

    def __enter__(self):
        for name in self.lib.protos:
            short = name[4:]
            fn = getattr(self.lib, short)
            if self.only is not None and name not in self.only:
                continue
            if self.lib.protos[name][0] is not __import__("ctypes").c_int or name == "eat_abi_version":
                continue
            self.orig[short] = fn
            setattr(self.lib, short, self._wrap(name, fn))
        return self

    def _wrap(self, name, fn):
        def call(*args):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(*args)
            e1.record()
            try:
                nbytes = algo_bytes(name, args)
            except Exception:                     # an accounting slip must never take the measurement down
                nbytes = None
            self.records.append((name, e0, e1, nbytes, args if name in ("eat_pw_tma_fwd", "eat_pw_tc_fwd", "eat_pw_tc_wgrad") else None))
        return call

    def __exit__(self, *a):
        for short, fn in self.orig.items():
            setattr(self.lib, short, fn)

    def table(self):
        agg = {}
        for name, e0, e1, nbytes, _ in self.records:
            ms = e0.elapsed_time(e1)
            t = agg.setdefault(name, [0.0, 0, 0, True])
            t[0] += ms
            t[1] += 1
            if nbytes is None:
                t[3] = False
            else:
                t[2] += nbytes
        return agg


def run_ours(args):
    import torch.distributed as dist
    from efficientat_b200._lib import lib
    from efficientat_b200.models.mn.model import get_model
    from efficientat_b200.models.preprocess import AugmentMelSTFT
    from efficientat_b200.synth import synth_labels, synth_state_, synth_waveform
    from efficientat_b200.train import AudioSetTrainer
    import contextlib, io

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = lib()
    L.device_check(local)

    B = args.batch
    width = {"mn10": 1.0, "mn04": 0.4, "mn20": 2.0, "mn40": 4.0, "dymn04": 0.4, "dymn10": 1.0, "dymn20": 2.0}[args.model]
    if args.model.startswith("dymn"):
        from efficientat_b200.models.dymn.model import get_model
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model = synth_state_(get_model(width_mult=width, precision=args.precision, verbose=False), seed=7).to(dev)
        mel = AugmentMelSTFT(freqm=0, timem=0).to(dev)          # ex_audioset.py defaults: freqm = timem = 0
    trainer = AudioSetTrainer(model, mel, lr=8e-4, kd_lambda=0.1, mixup_alpha=0.3, cuda_graph=not args.no_graph)
    if args.mode == "eval":
        model.eval()
        mel.eval()

        class _Eval:                                             # same .step() shape as the trainer
            def step(self, w, y_, t_, k_=None):
                with torch.no_grad():
                    logits, _ = model(mel(w).unsqueeze(1))
                self.logits = logits
                return logits[:, :2].double().sum(0)             # tiny device result read back in the e2e loop
        trainer = _Eval()
    import numpy as np
    np.random.seed(rank)
    torch.manual_seed(100 + rank)

    # synthetic shard for this rank: waveforms, labels, teacher soft targets (sigmoid of N(0,1) logits)
    wave_h, y_h, t_h, k_h = _synth_batch(B, rank)
    wave_h, y_h, t_h, k_h = wave_h.pin_memory(), y_h.pin_memory(), t_h.pin_memory(), k_h.float().pin_memory()
    wave, y, teacher, known = wave_h.to(dev), y_h.to(dev), t_h.to(dev), k_h.to(dev)
    if args.mode == "train":
        real = trainer

        class _Train:                                            # fixed (wave, y, teacher[, known]) signature for the loops below
            cuda_graph = real.cuda_graph

            def step(self, w, y_, t_, k_=None):
                real.cuda_graph = self.cuda_graph
                return real.step(w, y_, t_, teacher_known=known if k_ is None else k_)
        trainer = _Train()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up, eager: also finds the dominant kernel for the roofline figure and counts launches per step
    use_graph = getattr(trainer, "cuda_graph", False)
    if use_graph:
        trainer.cuda_graph = False
    for _ in range(max(args.warmup - 1, 2)):
        trainer.step(wave, y, teacher)
    torch.cuda.synchronize()
    with KernelTimer(L) as kt:
        trainer.step(wave, y, teacher)
        torch.cuda.synchronize()
    prof = kt.table()
    top = max(prof.items(), key=lambda kv: kv[1][0])[0]
    step_launches_before = L.launches
    trainer.step(wave, y, teacher)
    launches_per_step = L.launches - step_launches_before
    if use_graph:                                   # capture forward + loss + backward once, replay from now on
        trainer.cuda_graph = True
        for _ in range(2):
            trainer.step(wave, y, teacher)
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        h0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            loss = trainer.step(wave, y, teacher)
        e1.record()
        host_ms = (time.perf_counter() - h0) * 1e3 / args.steps      # time the host needs to ENQUEUE one step
        barrier()
    ms = e0.elapsed_time(e1)
    # what the last timed step computed: its [label, distillation] loss and the parameters its Adam update wrote (train),
    # or the logits (eval).  Copied out now: the steps below keep training the same model.  Compare parameters with a
    # tolerance: Adam turns the reduction-order noise of small gradients into differences of a fraction of lr per step
    # (two runs of one build, mn10, 10 timed steps, one B200: up to 8e-3, 99.9 % within 2.4e-3; the loss within 1e-5)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, "params": real.flat_p} if args.mode == "train"
                     else {"logits": trainer.logits})
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * B * args.steps / (ms * 1e-3)

    # ---- per-launch timing of the dominant kernel: the same K steps once more, launched eagerly with CUDA events
    # around every launch of that kernel (inside a replayed graph there is no host call to bracket)
    if use_graph:
        trainer.cuda_graph = False
    with KernelTimer(L, only={top}) as kt2:
        for _ in range(args.steps):
            # park the stream behind a ~60 ms spin kernel so that the host enqueues the whole step ahead of the GPU: the
            # events then sit directly before / after each launch on the device, with no host gap inside an interval
            torch.cuda._sleep(int(0.06 * 1.9e9))
            trainer.step(wave, y, teacher)
        torch.cuda.synchronize()
    if use_graph:
        trainer.cuda_graph = True
    top_ms, top_n, top_bytes, bytes_ok = kt2.table()[top]
    if os.environ.get("EAT_BENCH_KERNELS") == "2" and rank == 0:      # per-launch table of the GEMM entry points (last step)
        per = len(kt2.records) // max(args.steps, 1)
        for name, e0, e1, nbytes, a_ in kt2.records[-per:]:
            if a_ is not None and name == "eat_pw_tma_fwd":
                ms_ = e0.elapsed_time(e1)
                print(f"  pw_fwd M={a_[4]:8d} N={a_[5]:4d} K={a_[6]:4d} wT={a_[2]} xf={int(bool(a_[7]))} gate={int(bool(a_[10]))} "
                      f"res={int(bool(a_[15]))} stats={int(bool(a_[16]))}  {ms_ * 1e3:8.1f} us {nbytes / ms_ / 1e6:7.0f} GB/s", file=sys.stderr)

    # ---- end to end: pinned host buffers -> H2D -> step -> D2H loss, every step.  The copies go through the package's
    # double-buffered HostPrefetcher (batch i+1 is copied on a side stream while step i runs, as a pinned-memory
    # DataLoader would); all K copies and K loss read-backs happen inside the timed region.
    # The loss read-back is pipelined through the package's LossReader: step i's result is copied into pinned host memory
    # behind step i and collected while step i+1 is already queued (--sync-readback restores `loss.cpu()` after every
    # step, which leaves the device idle while the host enqueues the next step: ~0.9 ms per step).
    from efficientat_b200.train import HostPrefetcher, LossReader
    pf = HostPrefetcher(dev)
    rd = LossReader(dev)
    barrier()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    pf.submit(0, (wave_h, y_h, t_h, k_h))
    losses_read = 0
    for i in range(args.steps):
        if i + 1 < args.steps:
            pf.submit((i + 1) % 2, (wave_h, y_h, t_h, k_h))
        w_d, y_d, t_d, k_d = pf.get(i % 2)
        loss = trainer.step(w_d, y_d, t_d, k_d)
        pf.release(i % 2)
        if args.sync_readback:
            loss_host = loss.cpu()                  # device -> host read of the step's result (synchronises)
            losses_read += 1
        else:
            rd.push(loss)                           # asynchronous device -> host copy of step i's result ...
            if i:
                loss_host = rd.pop()                # ... and the host collects step i-1's while step i runs
                losses_read += 1
    if not args.sync_readback:
        loss_host = rd.pop()
        losses_read += 1
    e3.record()
    assert losses_read == args.steps
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
    h2d = wave_h.numel() * 4 + y_h.numel() * 4 + t_h.numel() * 4 + k_h.numel() * 4
    d2h = loss_host.numel() * 8

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
        achieved = (top_bytes / 1e9) / (top_ms * 1e-3) if (bytes_ok and top_ms > 0) else None
        shares = {k: round(v[0] / sum(x[0] for x in prof.values()), 4) for k, v in
                  sorted(prof.items(), key=lambda kv: -kv[1][0])[:8]}
        if os.environ.get("EAT_BENCH_KERNELS"):      # full per-entry-point table of the instrumented eager step, on stderr
            for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0]):
                print(f"  {k:28s} {v[0]:8.3f} ms/step {v[1]:5d} launches"
                      + (f" {v[2] / 1e6 / v[0]:8.0f} GB/s" if v[3] and v[0] > 0 else ""), file=sys.stderr)
        line = {
            "metric": METRIC if (args.mode == "train" and args.model == "mn10") else
            f"clips/sec (10s@32kHz) {args.model}_as {'fwd+bwd' if args.mode == 'train' else 'fwd'}", "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": (f"{args.model}_as training step: mel + mixup + fwd + BCE/KD loss + bwd + Adam "
                                    f"(ex_audioset.py:135-199), batch {B}/GPU, 10 s @ 32 kHz clips") if args.mode == "train"
                       else f"{args.model}_as mel + eval forward (inference.py:51-53), batch {B}/GPU, 10 s @ 32 kHz clips",
                       "model": f"{args.model}_as", "global_batch": B * world, "parallelism": f"dp{world}",
                       "precision_mode": args.precision, "cuda_graph": (not args.no_graph) and args.mode == "train",
                       "l2": "inputs (waveforms %.0f MB/GPU) exceed L2; no explicit flush" % (wave.numel() * 4 / 1e6)},
            "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "readback": "loss.cpu() after every step" if args.sync_readback else
                    "every step's loss, asynchronous copy into pinned memory collected one step behind (LossReader)"},
            "gpu_launches": launches_per_step * args.steps, "host_enqueue_ms_per_step": host_ms,
            "clocks": clocks.summary(),
            "roofline": {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None,
                         "traffic": (top_bytes / max(top_n, 1) * NCU_TRAFFIC[top]["dram_bytes"] / NCU_TRAFFIC[top]["algorithmic_bytes"])
                         if (top in NCU_TRAFFIC and bytes_ok) else None,
                         "traffic_source": NCU_TRAFFIC[top]["capture"] + " (dram/algorithmic ratio of the captured launch x "
                         "this run's algorithmic bytes per launch)" if top in NCU_TRAFFIC else None,
                         "peak_source": peak_src,
                         "timing": "CUDA events directly around every launch of this kernel over the same K steps, launched eagerly "
                                   "right after the graph-replayed timed region with the stream parked behind a spin kernel "
                                   "(the host runs ahead: no host gap inside an interval)" if use_graph
                                   else "CUDA events inside the timed region",
                         "launches_timed": top_n, "avg_launch_ms": top_ms / max(top_n, 1),
                         "algorithmic_bytes_per_launch": top_bytes / max(top_n, 1) if bytes_ok else None},
            "kernel_time_shares": shares,
            "loss": [float(v) for v in loss_host.tolist()],
        }
        if not args.no_cpu_baseline and world == 1:
            v, s_per_step, cores, cb, kind = time_cpu_reference(args.cpu_baseline_batch, 2, 1, budget_s=30.0, model=args.model)
            line["cpu_baseline"] = {"value": v, "unit": "clips/s", "cores": cores, "kind": kind,
                                    "sample": f"2 steps x {cb} clips (1 warm-up), same training step (mixup, hard + "
                                              "distillation loss with the unknown-teacher mask, Adam), fp32, "
                                              + ("the reference's own modules (oracle/_ref mirror)" if kind == "reference"
                                                 else "oracle port of the reference modules") + " on the host cores"}
    # ---- the reference's own GPU path on the same device(s): cuFFT / cuDNN / cuBLAS through the unmodified modules
    gb = None
    import gc
    if args.mode == "train":
        real.close()                 # the captured graph holds NCCL kernels: it must die before the process group does
        del real
    del trainer, pf
    gc.collect()
    if not args.no_gpu_baseline:
        torch.cuda.empty_cache()
        gb = {}
        for amp in ("none", "bf16"):
            gb["fp32" if amp == "none" else "autocast_bf16"] = gpu_baseline_entry(
                args.model, args.mode, B, min(args.steps, 5), 3, dev, amp, world, rank)
    if rank == 0:
        if gb is not None:
            line["gpu_baseline"] = gb
        print(json.dumps(line), flush=True)
    _shutdown(world)


def _shutdown(world):
    """leave a multi-rank run without giving NCCL's communicator teardown a chance to hang the launcher: every rank
    passes a final barrier (the JSON line is out), then exits the process directly"""
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    elif a.impl == "reference-gpu":
        run_reference_gpu_arm(a)
    else:
        run_ours(a)

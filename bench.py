#!/usr/bin/env python
"""bench.py — adversarial images / second, MI-FGSM ResNet-50 224^2 10 iterations (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (N>1: launched by torch.distributed.run)
    python bench.py [...] --dump-outputs DIR                       … and the last timed step's perturbation → DIR/delta.npy
    python bench.py --impl reference [...]                          the reference's CPU path (oracle port) on the host cores
    python bench.py --kernels                                       per-kernel roofline table  (gpurun_out/kernels.json)
    python bench.py --sweep                                         fused-update tuning sweep  (gpurun_out/sweep.json)

A "step" is one complete attack (10 iterations, each = surrogate forward + backward + the per-iteration kernels) on
one batch of B=64 synthetic 3x224x224 images per GPU (configs[1] of BASELINE.json). The batch shards across ranks with
no data-path collective (weak scaling: 64 images per GPU). One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG_ELEMS = 3 * 224 * 224
FUSED_BYTES_PER_ELEM = 28           # reads g, m, delta, x (16) + writes m', delta', x_adv (12)  — DESIGN.md §kernels
METRIC = "adv images/sec, MI-FGSM ResNet-50 224^2 10-iter"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=64, help="images per GPU")
    p.add_argument("--arch", default="resnet50")
    p.add_argument("--attack", default="mifgsm")
    p.add_argument("--epoch", type=int, default=10)
    p.add_argument("--mean-mode", default="torch", choices=["torch", "aten", "exact"])
    p.add_argument("--no-extras", action="store_true", help="skip the time-boxed rows for BASELINE configs 1 / 3 / 4 and the ensemble block")
    p.add_argument("--graph", type=int, default=int(os.environ.get("TA_B200_GRAPH", "1")))
    p.add_argument("--kernels", action="store_true")
    p.add_argument("--sweep", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-worker", default="", help="internal: 'sample_b,steps,warmup' → JSON on stdout")
    p.add_argument("--no-eager-gpu", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="after the timed steps, write the perturbation the last timed step returned to DIR/delta.npy (float32)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.kernels or args.sweep):
        p.error("--dump-outputs applies to the attack timed by `--impl ours` (not --kernels / --sweep)")
    return args


# ------------------------------------------------------------------------------------------------------------------
def peaks():
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        d = json.load(open(f))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = None
        self.p = None

    def __enter__(self):
        if self.gpu is None:
            return self
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        return self

    def __exit__(self, *a):
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.f is None:
            return out
        try:
            self.f.flush()
            rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
            os.unlink(self.f.name)
        except Exception:
            return out
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(n)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def host_cores():
    """threads the CPU legs may really use: scheduler affinity, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def build_attack(pkg, name, net, **kw):
    cls = pkg.load_attack_class(name)
    wrap = pkg.utils.wrap_model
    # load_model is the documented override point (attack.py:40-65); the class supplying the surrogate declares it capturable
    P = type("Bench" + cls.__name__, (cls,), {"load_model": lambda self, _n: wrap(net), "graph_safe": True})
    return P(model_name="synthetic", **kw)


def make_net(arch, device, seed=0):
    import torchvision
    torch.manual_seed(seed)
    kw = {"aux_logits": True, "init_weights": False} if arch == "inception_v3" else {}
    return getattr(torchvision.models, arch)(weights=None, **kw).eval().to(device)


def seed_host(s):
    import random
    torch.manual_seed(s); np.random.seed(s); random.seed(s)


def parity_stats(d, dr, x):
    """north_star's acceptance: perturbation within 1e-5 abs fp32, bit-identical after uint8 quantisation (utils.py:63-66)"""
    from oracle import torch_ref
    d, dr, x = d.float().cpu(), dr.float().cpu(), x.float().cpu()
    diff = (d - dr).abs()
    q, qr = torch_ref.save_images_u8(x, d), torch_ref.save_images_u8(x, dr)
    return {"bit_identical": bool(torch.equal(d, dr)), "n_gt_1e-5": int((diff > 1e-5).sum()), "u8_mismatch": int((q != qr).sum()),
            "max_abs": float(diff.max()), "numel": int(d.numel())}


def parity_block(atk, net, x_dev, y_dev, args, last):
    """the perturbation of the LAST TIMED step against the eager restatement of the reference (oracle/torch_ref.py — the checker,
    outside every timed region) on the same GPU, surrogate and inputs; plus the reference against itself (its own floor)."""
    from oracle import torch_ref
    kw = {"epoch": args.epoch}
    ref = torch_ref.REF_ZOO[args.attack](torch_ref.ref_wrap_model(net), **kw)
    seed_host(7); torch.cuda.manual_seed_all(7)
    dr = ref(x_dev, y_dev)
    seed_host(7); torch.cuda.manual_seed_all(7)
    dr2 = ref(x_dev, y_dev)
    seed_host(7); torch.cuda.manual_seed_all(7)
    d = atk(x_dev, y_dev)
    out = parity_stats(d, dr, x_dev)
    out["timed_output_equals_checked_output"] = bool(last is not None and torch.equal(last, d)) if args.attack in (
        "mifgsm", "ifgsm", "nifgsm", "fgsm", "tim", "sim", "emifgsm") else None      # host-RNG attacks draw per call
    out["reference_vs_itself"] = parity_stats(dr, dr2, x_dev)
    out["against"] = "oracle/torch_ref.py (eager restatement of attack.py:67-153) on the same GPU, surrogate and inputs"
    return out


def synth(B, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 3, 224, 224, generator=g), torch.randint(0, 1000, (B,), generator=g)


# ------------------------------------------------------------------------------------------------------------------
class EagerHooksMIFGSM:
    """The reference's eager-PyTorch hook chain on the GPU (attack.py:88,128,147-153 — 14 ATen launches per iteration),
    written out here as the comparator for the 'x vs the reference's PyTorch-GPU path' figure. Measured, never shipped."""

    def __init__(self, model, epsilon=16 / 255, alpha=1.6 / 255, epoch=10, decay=1.0):
        self.model, self.epsilon, self.alpha, self.epoch, self.decay = model, epsilon, alpha, epoch, decay
        self.loss = torch.nn.CrossEntropyLoss()

    def __call__(self, data, label):
        dev = next(self.model.parameters()).device
        data = data.clone().detach().to(dev); label = label.clone().detach().to(dev)
        delta = torch.zeros_like(data).requires_grad_(True)
        momentum = 0
        for _ in range(self.epoch):
            loss = self.loss(self.model(data + delta), label)
            grad = torch.autograd.grad(loss, delta)[0]
            momentum = momentum * self.decay + grad / (grad.abs().mean(dim=(1, 2, 3), keepdim=True))
            delta = torch.clamp(delta + self.alpha * momentum.sign(), -self.epsilon, self.epsilon)
            delta = torch.min(torch.max(delta, 0 - data), 1.0 - data).detach().requires_grad_(True)
        return delta.detach()


def cpu_reference_run(args, sample_b, steps, warmup):
    """oracle/torch_ref.py (eager restatement of the reference; the Python reference cannot travel to this box) on the
    host cores, all threads."""
    from oracle import torch_ref
    torch.set_num_threads(host_cores())
    net = make_net(args.arch, "cpu")
    atk = torch_ref.REF_ZOO[args.attack](torch_ref.ref_wrap_model(net), epoch=args.epoch)
    x, y = synth(sample_b)
    for _ in range(warmup):
        atk(x, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        atk(x, y)
    dt = time.perf_counter() - t0
    return sample_b * steps / dt, dt / steps


def cpu_worker(args):
    """child process: time `steps` attacks (after `warmup`) on `sample_b` images on the host cores, print JSON"""
    sample_b, steps, warmup = [int(float(v)) for v in args.cpu_worker.split(",")]
    val, per_step = cpu_reference_run(args, sample_b, steps, warmup)
    print(json.dumps({"value": val, "per_step_s": per_step, "sample_b": sample_b, "cores": host_cores()}), flush=True)


def cpu_leg(args, sample_b, steps, warmup, hard_timeout):
    """run the CPU leg in a child with a hard wall-clock bound (killed by PID on overrun)"""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", "%d,%d,%d" % (sample_b, steps, warmup),
           "--arch", args.arch, "--attack", args.attack, "--epoch", str(args.epoch)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=hard_timeout, env=env)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (out.stderr or "no output")[-300:]}
    except subprocess.TimeoutExpired:
        return {"error": "cpu leg exceeded %ds" % hard_timeout}


def run_reference_arm(args, rank):
    """the reference's own CPU path (oracle/torch_ref.py: the port; the Python reference cannot travel to this box) on all host
    threads; every step = one full 10-iteration attack on a bounded sample of CPU_SAMPLE_B of the batch's images."""
    if rank != 0:
        return
    sample_b = min(CPU_SAMPLE_B, args.batch)
    # bound the whole run: ~0.35 s per image and attack on 16 threads → 25 steps of 16 images ≈ 2.5 min
    r = cpu_leg(args, sample_b, args.steps, args.warmup, 900)
    if "error" in r:   # the oracle always exists; report the failure loudly but keep the line parseable
        r = {"value": float("nan"), "per_step_s": float("nan"), "sample_b": 0, "cores": host_cores(), "error": r["error"]}
    val, per_step, sample_b = r["value"], r["per_step_s"], r["sample_b"]
    cores = r["cores"]
    sample = "%d of %d images per step, %d iterations each, oracle/torch_ref.py on %d host threads" % (sample_b, args.batch, args.epoch, cores)
    cfg = workload_config(args, 1)
    cfg.update({"device": "cpu", "parallelism": "host threads x%d" % cores, "sample": sample})
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if "error" in r:
        line["error"] = r["error"]
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def timed_steps(fn, steps, dist, device):
    """barrier + synchronize, CUDA events around exactly `steps` calls on the launching stream, max over ranks."""
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(device)
    ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(ms.item())


def tail_kernel_name(atk, x_dev):
    """which form of the fused tail this attacker launches for inputs like x_dev (also the key into profiles/traffic.json)"""
    from transferattack_b200 import _lib
    kmode = atk._mean_kernel_mode(x_dev)
    fold = atk._fold_plan(x_dev, kmode)
    nf = "" if fold is None else (",nf+adjoint" if fold[4] else ",nf")
    if fold is not None and fold[5]:
        # the Normalize-adjoint kernel at the end of the backward formed ATen's column sums of |g| and its last CTA per sample finished
        # the mean: the tail is the streaming kernel alone
        return "ta_fused_tail[stream,nf] (mean|g| finished inside ta_normalize_bwd_colsum)", 1
    if kmode is None:
        return "ta_fused_tail[stream%s] after ATen abs+mean" % nf, 3
    if kmode == _lib.TA_MEAN_TORCH and x_dev.numel() * 4 <= 64 * 1024 * 1024 and int(os.environ.get("TA_FUSED_STRATEGY", "0")) in (0, 2):
        # csrc/fused_update.cu: a gradient that fits L2 takes the two-launch form (mean kernel, then the flat streaming kernel)
        return "ta_abs_mean_per_sample[torch order%s] + ta_fused_tail[stream%s]" % (", g/std" if (fold is not None and fold[4]) else "", nf), 2
    return "ta_fused_tail[cluster,%s%s]" % ("torch-order mean" if kmode == _lib.TA_MEAN_TORCH else "fp64 mean", nf), 1


def outside_note(atk, x_dev):
    fold = atk._fold_plan(x_dev, atk._mean_kernel_mode(x_dev))
    if fold is None or fold[4]:
        return None
    if fold[5]:
        return ("Normalize's adjoint g/std at the end of autograd.grad: one ta_normalize_bwd_colsum launch (8 B/elem) that also forms "
                "ATen's per-column sums of |g| and whose last CTA per sample finishes torch's mean from them — no separate mean kernel, "
                "the gradient is not read a second time; standalone timings of that kernel and of plain ta_normalize_bwd: bench.py --kernels")
    return "Normalize's adjoint g/std: one ta_normalize_bwd launch (8 B/elem) at the end of autograd.grad"


def graph_status(atk, requested):
    return {"requested": bool(requested), "captured": bool(getattr(atk, "_graphs", None)),
            "failed": bool(atk.__dict__.get("_graph_failed", False)), "error": atk.__dict__.get("_graph_error")}


def time_attack(atk, x_dev, y_dev, steps, warmup, dist, device):
    for _ in range(warmup):
        atk(x_dev, y_dev)
    torch.cuda.synchronize(device)
    return timed_steps(lambda: atk(x_dev, y_dev), steps, dist, device)


def tail_events(atk, x_dev, y_dev, steps, dist, device):
    """CUDA events around the WHOLE tail of every iteration (everything between autograd.grad and the next forward), on its
    stream, live inside a run of the same attack (eager launches of the same kernels: a graph replay cannot host events)"""
    ev = []
    atk._kernel_events = ev
    ms = timed_steps(lambda: atk(x_dev, y_dev), steps, dist, device)
    atk._kernel_events = None
    return [a.elapsed_time(b) for a, b in ev], ms


def run_ours(args, rank, local_rank, world, dist):
    import transferattack_b200 as tab
    from transferattack_b200 import _lib
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    hbm_peak, peak_src = peaks()
    B = args.batch
    net = make_net(args.arch, device)
    atk = build_attack(tab, args.attack, net, epoch=args.epoch)
    atk.mean_mode = args.mean_mode
    atk.use_cuda_graph = bool(args.graph)
    x_host, y_host = synth(B, seed=1 + rank)
    x_pin, y_pin = x_host.pin_memory(), y_host.pin_memory()
    x_dev, y_dev = x_host.to(device), y_host.to(device)
    out_pin = torch.empty_like(x_pin).pin_memory()
    n_elem = B * IMG_ELEMS

    # -- warm-up (also triggers cuDNN heuristics / graph capture / the one-time TA_MEAN_TORCH self-check) ----------
    for _ in range(max(args.warmup, 3)):
        atk(x_dev, y_dev)
    torch.cuda.synchronize(device)

    # -- value: inputs resident in HBM ---------------------------------------------------------------------------
    keep = {}

    def step_resident():
        keep["d"] = atk(x_dev, y_dev)
    # nvidia-smi is started on rank 0 only and BEFORE the timed region (its start-up enumerates every GPU of the box through NVML:
    # measured at N = 2 as +10 ms per step on the rank it overlapped with); one more untimed step runs while it comes up, then the
    # timed region is sampled every 100 ms
    with ClockSampler(local_rank if rank == 0 else None) as clk:
        step_resident()
        torch.cuda.synchronize(device)
        launches0 = _lib.launch_count()
        ms = timed_steps(step_resident, args.steps, dist, device)
        launches = _lib.launch_count() - launches0
    clocks = clk.summary()
    value = world * B * args.steps / (ms / 1e3)
    gstat = graph_status(atk, args.graph)
    if gstat["captured"]:  # kernels replayed from the captured graph are not host launches: add the graph's own count per replay
        sts = list(atk._graphs.values())
        launches += sts[-1].get("kernels_per_replay", 0) * args.epoch * args.steps
    last_timed = keep.get("d")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_timed, rank, world, dist)

    # -- roofline of the tail -----------------------------------------------------------------------------------------
    k_ms, ms_ev = tail_events(atk, x_dev, y_dev, max(2, args.steps // 2), dist, device)
    kname, tail_launches = tail_kernel_name(atk, x_dev)

    # -- e2e: host buffers through the plugin call, H2D of the batch and D2H of the perturbation inside the timed region
    def e2e_step():
        d = atk(x_pin, y_pin)
        out_pin.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    for _ in range(2):
        e2e_step()
    ms_e2e = timed_steps(e2e_step, args.steps, dist, device)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)

    roof = None
    if k_ms:
        avg_ms = float(np.mean(k_ms))
        achieved = FUSED_BYTES_PER_ELEM * n_elem / (avg_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tf = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tf):
            ent = json.load(open(tf)).get("%s B=%d" % (kname, B))       # keyed by the kernel form that was timed: never another variant's
            if isinstance(ent, dict):
                traffic, traffic_src = ent.get("dram_bytes"), ent.get("source")
        roof = {"bound": "hbm", "kernel": kname, "bracket": "the whole tail of an iteration: everything between autograd.grad and the "
                "next forward (%d launch%s)" % (tail_launches, "" if tail_launches == 1 else "es"),
                "outside_the_bracket": outside_note(atk, x_dev),
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "avg_launch_us": avg_ms * 1e3, "launches_timed": len(k_ms),
                "algorithmic_bytes_per_launch": FUSED_BYTES_PER_ELEM * n_elem, "share_of_step": float(np.sum(k_ms)) / ms_ev}

    parity = None
    if rank == 0:
        parity = parity_block(atk, net, x_dev, y_dev, args, last_timed)

    extra = {}
    if rank == 0 and world == 1:
        # the other mean modes, for the record (same timed procedure)
        alts = {}
        for other in [m for m in ("torch", "aten", "exact") if m != args.mean_mode]:
            atk.mean_mode = other
            ms2 = time_attack(atk, x_dev, y_dev, max(3, args.steps // 2), 2, None, device)
            k2, _ = tail_events(atk, x_dev, y_dev, 3, None, device)
            ach2 = FUSED_BYTES_PER_ELEM * n_elem / (float(np.mean(k2)) * 1e-3) / 1e9 if k2 else None
            alts[other] = {"value": B * max(3, args.steps // 2) / (ms2 / 1e3), "kernel": tail_kernel_name(atk, x_dev)[0],
                           "roofline": {"achieved": ach2, "frac": ach2 / hbm_peak if ach2 else None,
                                        "avg_tail_us": float(np.mean(k2)) * 1e3 if k2 else None}}
        atk.mean_mode = args.mean_mode
        # same mean mode with the separate torch-order mean kernel (the adjoint kernel does not leave column sums)
        prev_cs = atk.colsum_adjoint
        atk.colsum_adjoint = False
        ms2 = time_attack(atk, x_dev, y_dev, max(3, args.steps // 2), 2, None, device)
        k2, _ = tail_events(atk, x_dev, y_dev, 3, None, device)
        ach2 = FUSED_BYTES_PER_ELEM * n_elem / (float(np.mean(k2)) * 1e-3) / 1e9 if k2 else None
        alts["%s, separate mean kernel (plain ta_normalize_bwd in the backward)" % args.mean_mode] = {
            "value": B * max(3, args.steps // 2) / (ms2 / 1e3), "kernel": tail_kernel_name(atk, x_dev)[0],
            "roofline": {"achieved": ach2, "frac": ach2 / hbm_peak if ach2 else None, "avg_tail_us": float(np.mean(k2)) * 1e3 if k2 else None}}
        atk.colsum_adjoint = prev_cs
        # same mean mode, Normalize's adjoint folded into the tail kernels (2 launches instead of 3; the division then runs twice)
        prev = atk.fold_adjoint
        atk.fold_adjoint = True
        ms2 = time_attack(atk, x_dev, y_dev, max(3, args.steps // 2), 2, None, device)
        k2, _ = tail_events(atk, x_dev, y_dev, 3, None, device)
        ach2 = FUSED_BYTES_PER_ELEM * n_elem / (float(np.mean(k2)) * 1e-3) / 1e9 if k2 else None
        alts["%s, Normalize's adjoint folded into the tail (no ta_normalize_bwd launch in the backward)" % args.mean_mode] = {
            "value": B * max(3, args.steps // 2) / (ms2 / 1e3), "kernel": tail_kernel_name(atk, x_dev)[0],
            "roofline": {"achieved": ach2, "frac": ach2 / hbm_peak if ach2 else None, "avg_tail_us": float(np.mean(k2)) * 1e3 if k2 else None}}
        atk.fold_adjoint = prev
        extra["alt_mean_modes"] = alts
        if not args.no_eager_gpu:
            # the reference's eager hook chain on this GPU (same surrogate, torchvision normalise incl. its host sync)
            from oracle import torch_ref  # comparator only
            eager = EagerHooksMIFGSM(torch_ref.ref_wrap_model(net), epoch=args.epoch)
            for _ in range(2):
                eager(x_dev, y_dev)
            ms3 = timed_steps(lambda: eager(x_dev, y_dev), args.steps, None, device)

            def eager_e2e():
                d = eager(x_host, y_host)
                d.cpu()
            eager_e2e()
            ms4 = timed_steps(eager_e2e, max(2, args.steps // 2), None, device)
            extra["reference_gpu_eager"] = {"value": B * args.steps / (ms3 / 1e3), "ms_per_step": ms3 / args.steps,
                                            "e2e_value": B * max(2, args.steps // 2) / (ms4 / 1e3),
                                            "note": "eager PyTorch hooks of attack.py on the same GPU/surrogate; informational"}
        if not args.no_extras:
            extra["other_configs"] = other_config_rows(args, device, hbm_peak)
            extra["fast_mode"] = fast_mode_block(args, tab, net, x_dev, y_dev, value, device)

    if world > 1 and not args.no_extras:
        ens = ens_block(args, rank, local_rank, world, dist, device)
        if rank == 0:
            extra["ens"] = ens

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_leg(args, CPU_SAMPLE_B, 2, 1, 300)
        if "error" in r:
            cpu_base = {"value": None, "unit": "images/s", "cores": host_cores(), "kind": "port", "sample": "failed: " + r["error"]}
        else:
            cpu_base = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                        "sample": "%d of %d images per step, %d iterations each, 1 warm-up + 2 timed steps, oracle/torch_ref.py on %d host threads"
                                  % (r["sample_b"], B, args.epoch, r["cores"])}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(args, world, atk, x_dev),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * IMG_ELEMS * 4 + B * 8,
                    "d2h_bytes_per_step": B * IMG_ELEMS * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "roofline": roof,
            "parity": parity,
            "graph": gstat,
            "cpu_baseline": cpu_base,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, delta, rank, world, dist):
    """--dump-outputs: the perturbation the last timed step returned (every rank's shard, in rank order) as DIR/delta.npy in
    float32. The inputs are seeded, so two builds run with the same arguments can be compared element for element. An output
    larger than DUMP_BYTES is written as a fixed sample of its flattened elements (distinct indices drawn with seed 0, in
    increasing order), and those indices go to DIR/delta_index.npy (float64, exact below 2^53)."""
    if dist is not None:
        parts = [torch.empty_like(delta) for _ in range(world)]
        dist.all_gather(parts, delta.contiguous())
        delta = torch.cat(parts)
    if rank != 0:
        return
    d = delta.float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    if d.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(d.size, DUMP_BYTES // 16, replace=False))   # 4 + 8 bytes per sample
        d = d.reshape(-1)[idx]
        np.save(os.path.join(out_dir, "delta_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "delta.npy"), d)


def workload_config(args, world, atk=None, x_dev=None):
    B = args.batch
    cfg = {"workload": ("MI-FGSM, ResNet-50, batch 64, 10 iters, eps=16/255 (BASELINE configs[1])"
                        if (args.attack, args.arch, B, args.epoch) == ("mifgsm", "resnet50", 64, 10)
                        else "%s, %s, batch %d, %d iters, eps=16/255" % (args.attack, args.arch, B, args.epoch)),
           "attack": args.attack, "arch": args.arch, "batch_per_gpu": B, "global_batch": B * world, "epoch": args.epoch,
           "parallelism": "batch-sharded x%d, no collective" % world,
           "surrogate": "torch autograd, fp32 (cuDNN TF32 convs as torch defaults), random-init weights"}
    if atk is not None:
        kmode = atk._mean_kernel_mode(x_dev)
        cfg.update({"normalize_folded": bool(atk._fold_plan(x_dev, kmode) is not None), "mean_mode": args.mean_mode,
                    "l2": "working set per step (activations of %d images) exceeds the 126 MB L2; no explicit flush" % B,
                    "cuda_graph": bool(getattr(atk, "_graphs", None))})
    return cfg


# ------------------------------------------------------------------------------------------------------------------
def kernel_fracs(B, hbm_peak, names):
    """standalone fraction-of-peak of the dominant kernels of a configuration at ITS batch size (clean L2 before every launch)"""
    from transferattack_b200 import ops, _lib
    import transferattack_b200.input_transformation.tim as tim
    be = ops.backend()
    dev = "cuda"
    N = B * IMG_ELEMS
    flush = torch.empty(512 * 1024 * 1024 // 4, device=dev)
    g = torch.randn(B, 3, 224, 224, device=dev) * 1e-4
    m = torch.randn_like(g); x = torch.rand_like(g); d = (torch.rand_like(g) * 2 - 1) * (16 / 255)
    m2, d2, xa, v = torch.empty_like(g), torch.empty_like(g), torch.empty_like(g), torch.randn_like(g) * 1e-5
    so = torch.empty(B, device=dev)
    k2d, kcol, krow = tim.make_kernel("gaussian", 15)
    kc3 = torch.from_numpy(np.stack([kcol] * 3)).to(dev); kr3 = torch.from_numpy(np.stack([krow] * 3)).to(dev)
    hc, hr = kc3.cpu().numpy(), kr3.cpu().numpy()
    a, al = 1.6 / 255, 16 / 255
    table = {
        "dim_fwd": (8, lambda: be.dim(x, 235, 246, 5, 6, True)),
        "dim_bwd": (8, lambda: be.dim(g, 235, 246, 5, 6, False)),
        "tim_dwconv2d_sep_k15": (8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr))),
        "fused_tail_torch_order": (28, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH)),
        "fused_tail_addend_torch_order": (32, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0,
                                                                    mean_mode=_lib.TA_MEAN_TORCH, addend=v)),
        "neighbor_stage_philox": (12, lambda: be.neighbor_stage_philox(x, d, -0.09, 0.09)),
        "accumulate": (12, lambda: be.accumulate(m2, g, False)),
    }
    out = {}
    for nme in names:
        bpe, fn = table[nme]
        med, _ = time_kernel(fn, iters=10, flush=flush)
        gbs = bpe * N / (med * 1e-3) / 1e9
        out[nme] = {"us": med * 1e3, "bytes_per_elem": bpe, "GBps": gbs, "frac": gbs / hbm_peak}
    return out


def fast_mode_block(args, tab, net, x_dev, y_dev, strict_value, device):
    """OPT-IN fast modes (Attack.fast_mode: BatchNorm folded into the convolutions and / or a bf16 channels_last twin of the
    surrogate, fp32 kernels around it) on the headline configuration. NOT the parity path and never the headline: reported under its own key with its own acceptance —
    the white-box loss the perturbation reaches on the fp32 surrogate next to the strict path's (SURVEY §7 H2)."""
    try:
        wrapped = tab.utils.wrap_model(net)
        ce = torch.nn.CrossEntropyLoss()

        def loss_of(d):
            with torch.no_grad():
                return float(ce(wrapped(x_dev + d), y_dev))
        strict = build_attack(tab, args.attack, net, epoch=args.epoch)
        d0 = strict(x_dev, y_dev)
        clean = loss_of(torch.zeros_like(d0))
        out = {"label": "opt-in, not bit-comparable with the reference; never the headline",
               "acceptance_rule": "white-box CE reached on the fp32 surrogate vs the strict path's", "ce_clean": clean, "ce_strict": loss_of(d0),
               "modes": {}}
        steps = max(3, args.steps // 2)
        for mode in ("bnfold", "bf16", "bnfold+bf16"):
            fast = build_attack(tab, args.attack, net, epoch=args.epoch)
            fast.fast_mode = mode
            ms = time_attack(fast, x_dev, y_dev, steps, 3, None, device)
            d1 = fast(x_dev, y_dev)
            v = x_dev.shape[0] * steps / (ms / 1e3)
            out["modes"][mode] = {"value": v, "unit": "images/s", "speedup_vs_strict": v / strict_value,
                                  "cuda_graph": bool(getattr(fast, "_graphs", None)), "ce_fast": loss_of(d1),
                                  "max_abs_delta": float(d1.abs().max()),
                                  "in_box": bool(float((x_dev + d1).min()) >= 0 and float((x_dev + d1).max()) <= 1)}
            del fast
            torch.cuda.empty_cache()
        return out
    except Exception as e:
        return {"error": repr(e)[:300]}


CPU_SAMPLE_B = 16        # images per step of every CPU leg (a bounded sample of the batch-64 workload; stated in the line)


def other_config_rows(args, device, hbm_peak):
    """time-boxed rows for BASELINE configs 1 / 3 / 4 (SURVEY §8d): images/s through the plugin API + the dominant kernels'
    fraction of the measured HBM peak at that configuration's batch size. Informational; the headline stays configs[1]."""
    import transferattack_b200 as tab
    rows = {}
    # configs[0]: I-FGSM / ResNet-18 / B=4 on the host cores (the reference's own CPU-runnable case), oracle port
    import copy
    a1 = copy.copy(args); a1.attack, a1.arch, a1.epoch = "ifgsm", "resnet18", 10
    r = cpu_leg(a1, 4, 5, 1, 120)
    rows["config1_ifgsm_resnet18_b4_cpu"] = ({"error": r["error"]} if "error" in r else
                                              {"images_per_s": r["value"], "s_per_attack": r["per_step_s"], "cores": r["cores"], "device": "cpu",
                                               "impl": "oracle/torch_ref.py (port of the reference), 1 warm-up + 5 timed attacks"})
    for key, attack, arch, B, kw, steps, knames in (
            ("config3_ditimi_resnet50_b32_per_gpu_share", "ditimi", "resnet50", 32, {}, 5, ["dim_fwd", "dim_bwd", "tim_dwconv2d_sep_k15", "fused_tail_torch_order"]),
            ("config4_vmifgsm_n20_vit_b16_b16", "vmifgsm", "vit_b_16", 16, {"num_neighbor": 20}, 1,
             ["neighbor_stage_philox", "accumulate", "fused_tail_addend_torch_order"])):
        try:
            net = make_net(arch, device)
            atk = build_attack(tab, attack, net, epoch=10, **kw)
            x, y = synth(B, seed=3)
            x, y = x.to(device), y.to(device)
            seed_host(11)
            ms = time_attack(atk, x, y, steps, 1, None, device)
            rows[key] = {"images_per_s": B * steps / (ms / 1e3), "ms_per_attack": ms / steps, "batch": B, "steps": steps,
                         "cuda_graph": bool(getattr(atk, "_graphs", None)), "kernels": kernel_fracs(B, hbm_peak, knames)}
            del atk, net
            torch.cuda.empty_cache()
        except Exception as e:       # an informational row must never cost the headline line
            rows[key] = {"error": repr(e)[:300]}
    return rows


ENS_MEMBERS = ["resnet50", "resnet152", "inception_v3", "vit_b_16"]


def ens_block(args, rank, local_rank, K, dist, device):
    """BASELINE configs[4] — ensemble MI-FGSM, ONE surrogate per GPU (K = world size, members cycled) — beside the headline:
      p2p    ta_fused_allreduce_update_linf: gradient reduce-scatter + update + all-gather of the next input in ONE kernel over
             NVLink peer memory (logits by all_gather + the reference's own mean);
      nccl   NCCL all-reduce of logits (forward) and input gradient (backward) + replicated fused update;
      single the reference's layout: all K members sequentially on ONE GPU (rank 0), same kernels.
    Times are CUDA events, max over ranks; the three perturbations are compared (reference semantics: utils.py:82-105,
    ensemble/ens.py:31-36; SURVEY §8e steps 1-5)."""
    import transferattack_b200 as tab
    from transferattack_b200 import multigpu, _lib, ops
    B, steps = args.batch, 2
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, 3, 224, 224, generator=g).to(device)
    y = torch.randint(0, 1000, (B,), generator=g).to(device)
    names = [ENS_MEMBERS[k % len(ENS_MEMBERS)] for k in range(K)]
    member = tab.utils.wrap_model(make_net(names[rank], device, seed=rank))
    ens_cls = tab.load_attack_class("ens")
    out = {"K": K, "batch": B, "epoch": args.epoch, "members": names, "mean_mode": "exact"}

    def timed(fn):
        return timed_steps(fn, steps, dist, device) / steps

    a_nccl = multigpu.make_ens_attack(ens_cls, member, epoch=args.epoch)
    a_nccl.mean_mode = "exact"
    d_nccl = a_nccl(x, y); a_nccl(x, y)
    ms = timed(lambda: a_nccl(x, y))
    out["nccl"] = {"ms_per_attack": ms, "images_per_s": B / ms * 1e3}

    a_p2p = multigpu.make_fused_p2p_ens(ens_cls, member, epoch=args.epoch)
    d_p2p = a_p2p(x, y); a_p2p(x, y)
    ms = timed(lambda: a_p2p(x, y))
    out["p2p"] = {"ms_per_attack": ms, "images_per_s": B / ms * 1e3}
    out["p2p_vs_nccl_mismatch"] = int((d_p2p != d_nccl).sum())

    # the exchange + update step in isolation (same gradient tensor on every rank; median of 20 after 5 warm-ups)
    be = ops.backend(); lib = _lib.load()
    gfull = torch.randn_like(x) * 1e-4
    m = torch.zeros_like(x); d = torch.zeros_like(x); xa = torch.empty_like(x); so = torch.empty(B, device=device)
    st = a_p2p._buffers(x)
    lo, hi = multigpu.shard_bounds(B, rank, K)
    n = x[0].numel()
    stream = torch.cuda.current_stream(device)

    def step_nccl():
        gg = gfull.clone()
        dist.all_reduce(gg)
        be.fused_update_linf(gg, m, m, d, d, x, xa, None, so, 1.0, 1.6 / 255, 16 / 255, 0, 1.0)

    def step_p2p():
        st["G"].copy_(gfull)
        st["hg"].barrier(channel=0)
        _lib.check(lib.ta_fused_allreduce_update_linf(st["g_ptrs"], st["x_ptrs"], K, m.data_ptr(), m.data_ptr(), d.data_ptr(), d.data_ptr(),
                                                      x.data_ptr(), None, so.data_ptr(), 0, 1.0, 1.6 / 255, 16 / 255, 0.0, 1.0, lo, hi - lo, n,
                                                      stream.cuda_stream), "p2p")
        st["hx"].barrier(channel=0)

    for name, fn in (("nccl_allreduce_plus_update_us", step_nccl), ("p2p_fused_exchange_update_us", step_p2p)):
        for _ in range(5):
            fn()
        ts = sorted(timed_steps(fn, 1, dist, device) * 1e3 for _ in range(20))
        out[name] = ts[len(ts) // 2]
    # NVLink volume of the fused step per GPU: (K-1)/K of the gradient in + (K-1)/K of the next input out
    wire = 2 * (K - 1) / K * B * IMG_ELEMS * 4
    out["p2p_nvlink_bytes_per_gpu"] = wire
    out["p2p_nvlink_GBps_per_direction"] = (wire / 2) / (out["p2p_fused_exchange_update_us"] * 1e-6) / 1e9
    out["nvlink_peak_GBps_per_direction"] = 770.0

    # the reference's layout: every member on one device, sequentially (rank 0 measures, the others wait at the barrier)
    single = None
    if rank == 0:
        nets = [tab.utils.wrap_model(make_net(names[k], device, seed=k)) for k in range(K)]
        P = type("SingleENS", (ens_cls,), {"load_model": lambda self, _n: tab.utils.EnsembleModel(nets), "graph_safe": True})
        a_one = P(model_name="all-on-one", epoch=args.epoch)
        a_one.mean_mode = "exact"
        d_one = a_one(x, y); a_one(x, y)
        ms1 = timed_steps(lambda: a_one(x, y), steps, None, device) / steps
        single = {"ms_per_attack": ms1, "images_per_s": B / ms1 * 1e3}
        out["single_gpu_all_members"] = single
        out["p2p_vs_single_mismatch"] = int((d_p2p != d_one).sum())
        out["nccl_vs_single_mismatch"] = int((d_nccl != d_one).sum())
        out["bit_identical"] = out["p2p_vs_single_mismatch"] == 0 and out["nccl_vs_single_mismatch"] == 0 and out["p2p_vs_nccl_mismatch"] == 0
        per_iter_ms = out["p2p"]["ms_per_attack"] / args.epoch
        out["bound"] = ("the slowest member's forward/backward bounds the step: the fused exchange+update is %.0f us of a %.1f ms iteration"
                        % (out["p2p_fused_exchange_update_us"], per_iter_ms))
        del nets, a_one
    dist.barrier()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------------------
def flush_l2(buf):
    # displace L2 with CLEAN lines (a read-only pass over 256 MB): a memset would leave 126 MB of dirty lines whose
    # write-back then competes with the timed kernel for DRAM
    buf.sum()


def time_kernel(fn, iters=20, flush=None):
    """per-launch duration with CUDA events on the launching stream; L2 flushed (256 MB memset) before each launch."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush_l2(flush)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    time_kernel.last = ts
    return float(np.median(ts)), float(np.min(ts))


def run_kernels(args):
    """roofline table of every kernel at BASELINE sizes (B=64): algorithmic bytes / measured time vs measured HBM peak."""
    from transferattack_b200 import ops, _lib
    import transferattack_b200.input_transformation.tim as tim
    be = ops.backend()
    hbm_peak, peak_src = peaks()
    B = args.batch
    N = B * IMG_ELEMS
    dev = "cuda"
    flush = torch.empty(1024 * 1024 * 1024 // 4, device=dev)     # 1 GB read-only pass (~170 us): displaces L2 with clean lines AND
    # keeps the GPU busy long enough that the host-side launch path of the next call is off the measured interval
    g = torch.randn(B, 3, 224, 224, device=dev) * 1e-4
    m = torch.randn_like(g); x = torch.rand_like(g); d = (torch.rand_like(g) * 2 - 1) * (16 / 255)
    m2, d2, xa = torch.empty_like(g), torch.empty_like(g), torch.empty_like(g)
    so = torch.empty(B, device=dev)
    scale = be.abs_mean(g)
    k2d, kcol, krow = tim.make_kernel("gaussian", 15)
    kc3 = torch.from_numpy(np.stack([kcol] * 3)).to(dev); kr3 = torch.from_numpy(np.stack([krow] * 3)).to(dev)
    k3 = torch.from_numpy(k2d.reshape(3, 15, 15)).to(dev)
    g5 = torch.randn(5 * B, 3, 224, 224, device=dev)
    a, al = 1.6 / 255, 16 / 255
    rows = []

    def add(name, bpe, fn, elems=N):
        med, mn = time_kernel(fn, flush=flush)
        gbs = bpe * elems / (med * 1e-3) / 1e9
        # event timestamps on this GPU tick every 2.048 us (all medians fall on that grid): the mean of the 20 launches without
        # the two slowest resolves finer than one tick, since the launches start at arbitrary phases of the tick
        tm = float(np.mean(sorted(time_kernel.last)[:-2]))
        rows.append({"kernel": name, "bytes_per_elem": bpe, "elems": elems, "median_us": med * 1e3, "min_us": mn * 1e3,
                     "trimmed_mean_us": tm * 1e3, "achieved_GBps": gbs, "frac_of_peak": gbs / hbm_peak,
                     "frac_of_peak_by_trimmed_mean": bpe * elems / (tm * 1e-3) / 1e9 / hbm_peak})

    add("ATen reference: torch.add(x, d, out=) (same harness)", 12, lambda: torch.add(x, d, out=xa))
    add("ATen reference: tensor.copy_ (same harness)", 8, lambda: xa.copy_(x))
    MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    vadd = torch.randn_like(g) * 1e-5; gb = torch.empty_like(g)
    _lib.tune_set("fused.strategy", 1)
    add("fused_tail[cluster, fp64 mean]", 28, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_EXACT))
    add("fused_tail[cluster, torch-order mean]", 28, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH))
    add("fused_tail[cluster, torch-order mean, nf]", 28, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH,
                                                                              mean=MEAN, std=STD, emit_normalized=True))
    add("fused_tail[cluster, torch-order mean, nf+adjoint] (the default base loop)", 28,
        lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH, mean=MEAN, std=STD,
                              emit_normalized=True, grad_wrt_xn=True))
    _lib.tune_set("fused.strategy", 1)         # rows above/below labelled "cluster": the one-launch form, whatever the size
    for un in (1, 4):
        _lib.tune_set("fused.unroll", un)
        add("  fused_tail[cluster, torch-order mean, nf+adjoint] unroll=%d" % un, 28,
            lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH, mean=MEAN, std=STD,
                                  emit_normalized=True, grad_wrt_xn=True))
    _lib.tune_set("fused.unroll", 2)
    add("fused_tail[cluster, torch-order mean, addend] (VMI)", 32, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0,
                                                                                        mean_mode=_lib.TA_MEAN_TORCH, addend=vadd))
    add("fused_tail[cluster, torch-order mean, gbar] (EMI)", 32, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0,
                                                                                      mean_mode=_lib.TA_MEAN_TORCH, gbar_out=gb))
    _lib.tune_set("fused.strategy", 2)
    add("fused_tail[split: torch-order mean kernel + stream] (2 launches)", 32, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0,
                                                                                                   mean_mode=_lib.TA_MEAN_TORCH))
    add("fused_tail[split: torch-order mean kernel + stream, nf+adjoint] (2 launches; the default base loop at B=64)", 32,
        lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0, mean_mode=_lib.TA_MEAN_TORCH, mean=MEAN, std=STD,
                              emit_normalized=True, grad_wrt_xn=True))
    add("fused_tail[split, addend] (VMI)", 40, lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, a, al, 0, 1.0,
                                                                    mean_mode=_lib.TA_MEAN_TORCH, addend=vadd))
    _lib.tune_set("fused.strategy", 0)
    add("fused_tail[stream, scale given]", 28, lambda: be.fused_update_linf(g, m, m2, d, d2, x, xa, scale, None, 1.0, a, al, 0, 1.0))
    add("abs_mean_per_sample [torch order]", 4, lambda: be.abs_mean(g, _lib.TA_MEAN_TORCH))
    std_dev = torch.tensor(STD, device=dev)
    cs_n = be.colsum_size(B, g[0].numel(), g.device)
    if cs_n is not None:
        cs = torch.empty(B * cs_n, device=dev)
        add("normalize_bwd (Normalize's adjoint, plain)", 8, lambda: be.normalize(g, None, std_dev, False))
        add("normalize_bwd_colsum (the adjoint + ATen's column sums of |g|)", 8, lambda: be.normalize_bwd_colsum(g, std_dev, cs))
        cnt = torch.zeros(B, dtype=torch.int32, device=dev)
        add("normalize_bwd_colsum, mean finished in-launch (what the attack loop runs)", 8, lambda: be.normalize_bwd_colsum(g, std_dev, cs, so, cnt))
        add("abs_mean_from_colsums (trees over the column sums; %d floats per sample)" % cs_n, 4, lambda: be.abs_mean_from_colsums(cs, so, B, g[0].numel()),
            elems=B * cs_n)
    add("ATen reference: g.abs().mean(dim=(1,2,3)) (2 launches)", 12, lambda: g.abs().mean(dim=(1, 2, 3)))
    for cap in (0, 4, 8, 16):
        for un in (1, 2, 4):
            _lib.tune_set("stream.cap", cap); _lib.tune_set("stream.unroll", un)
            add("  fused stream variant cap=%d unroll=%d" % (cap, un), 28,
                lambda: be.fused_update_linf(g, m, m2, d, d2, x, xa, scale, None, 1.0, a, al, 0, 1.0))
    _lib.tune_set("stream.cap", 0); _lib.tune_set("stream.unroll", 1)
    add("abs_mean_per_sample", 4, lambda: be.abs_mean(g))
    add("momentum", 12, lambda: be.momentum(g, m, scale, 1.0, out=m2))
    add("update_linf", 16, lambda: be.update_linf(d, x, m, a, al, 0, 1.0, out=d2))
    add("stage_add", 12, lambda: be.stage_add(x, d, out=xa))
    add("sim_fwd S=5", 24, lambda: be.sim(x, 5, True))
    add("sim_bwd S=5", 24, lambda: be.sim(g5, 5, False))
    for impl, bwd, fwdtab, tag in ((2, 0, 0, "default: register-carried forward, separable-pass adjoint"), (3, 0, 0, "separable passes in shared memory"),
                                   (1, 0, 0, "direct; fwd tables = kernel parameters; adjoint = gather + scatter, tables in workspace"),
                                   (1, 1, 1, "direct; fwd tables in workspace; adjoint = independent gather"), (0, 0, 0, "4-pass")):
        _lib.tune_set("dim.impl", impl); _lib.tune_set("dim.bwd", bwd); _lib.tune_set("dim.fwdtab", fwdtab)
        add("dim_fwd [%s]" % tag, 8, lambda: be.dim(x, 235, 246, 5, 6, True))
        add("dim_bwd [%s]" % tag, 8, lambda: be.dim(g, 235, 246, 5, 6, False))
    _lib.tune_set("dim.impl", 4)
    for rb, st in ((16, 1), (16, 0), (32, 1), (32, 0)):
        _lib.tune_set("dim.walk_rb", rb); _lib.tune_set("dim.walk_stage", st)
        add("dim_fwd [source-driven walk, %d-row bands, source rows %s]" % (rb, "staged by TMA" if st else "from global memory"), 8,
            lambda: be.dim(x, 235, 246, 5, 6, True))
    _lib.tune_set("dim.walk_rb", 16); _lib.tune_set("dim.walk_stage", 1)
    _lib.tune_set("dim.impl", 3); _lib.tune_set("dim.sepconst", 0)
    add("dim_fwd [separable passes, run-time pitches]", 8, lambda: be.dim(x, 235, 246, 5, 6, True))
    add("dim_bwd [separable passes, run-time pitches]", 8, lambda: be.dim(g, 235, 246, 5, 6, False))
    _lib.tune_set("dim.impl", 2); _lib.tune_set("dim.sepconst", 1); _lib.tune_set("dim.bwd", 0); _lib.tune_set("dim.fwdtab", 0)
    hc, hr = kc3.cpu().numpy(), kr3.cpu().numpy()
    _lib.tune_set("tim.band", 4)
    add("dwconv2d_sep k=15 [unrolled band walk, paired weights, tap-exact column pass (default)]", 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.band", 5)
    add("dwconv2d_sep k=15 [the same walk fed from a warp-private cp.async ring]", 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.band", 4)
    _lib.tune_set("tim.split", 1)
    add("dwconv2d_sep k=15 [unrolled band walk, interior / edge windows in separate CTAs]", 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.split", 0)
    _lib.tune_set("tim.deep", 1)
    add("dwconv2d_sep k=15 [unrolled band walk, loads two rows ahead]", 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.deep", 0)
    for pf in (2, 1, 0):
        _lib.tune_set("tim.prefetch2", pf)
        add("dwconv2d_sep k=15 [unrolled band walk, prefetch mode %d]" % pf, 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.prefetch2", 3)
    for band, f2, tag in ((3, 1, "register-sliding from global memory, FFMA2"), (3, 0, "register-sliding from global memory, FFMA"),
                          (2, 0, "register-sliding from TMA-staged smem")):
        _lib.tune_set("tim.band", band); _lib.tune_set("tim.f2", f2)
        add("dwconv2d_sep k=15 [%s, factors as kernel parameters]" % tag, 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
        _lib.tune_set("tim.bh", 56)
        add("dwconv2d_sep k=15 [%s, parameters, band 56]" % tag, 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
        _lib.tune_set("tim.bh", 32)
        add("dwconv2d_sep k=15 [%s, factors from device arrays]" % tag, 8, lambda: be.dwconv2d_sep(g, kc3, kr3))
    _lib.tune_set("tim.band", 3); _lib.tune_set("tim.f2", 1)
    for pf in (1, 0):
        _lib.tune_set("tim.prefetch", pf)
        add("dwconv2d_sep k=15 [from global memory, FFMA2, parameters, prefetch mode %d]" % pf, 8, lambda: be.dwconv2d_sep(g, kc3, kr3, host=(hc, hr)))
    _lib.tune_set("tim.prefetch", 2)
    _lib.tune_set("tim.band", 1)
    add("dwconv2d_sep k=15 [two-pass band kernel]", 8, lambda: be.dwconv2d_sep(g, kc3, kr3))
    _lib.tune_set("tim.band", 4); _lib.tune_set("tim.f2", 1)
    add("dwconv2d k=15 (direct)", 8, lambda: be.dwconv2d(g, k3))
    add("accumulate", 12, lambda: be.accumulate(m2, g, False))
    add("quantize_u8", 9, lambda: be.quantize_u8(x, d, True))
    # torch eager equivalents of the fused tail, for the same tensors
    def eager_tail():
        mm = m * 1.0 + g / g.abs().mean(dim=(1, 2, 3), keepdim=True)
        dd = torch.clamp(d + a * mm.sign(), -al, al)
        dd = torch.min(torch.max(dd, 0 - x), 1.0 - x)
        return x + dd
    med, mn = time_kernel(eager_tail, flush=flush)
    rows.append({"kernel": "torch eager tail (14 ATen launches, attack.py:88,128,147-153)", "bytes_per_elem": 128, "elems": N,
                 "median_us": med * 1e3, "min_us": mn * 1e3, "achieved_GBps": 128 * N / (med * 1e-3) / 1e9, "frac_of_peak": None})
    out = {"hbm_peak_GBps": hbm_peak, "peak_source": peak_src, "batch": B, "l2": "read-only pass over a 1 GB buffer before every timed launch (clean L2, host launch path hidden)", "rows": rows}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "kernels.json"), "w"), indent=1)
    for r in rows:
        print("%-70s %8.1f us  %8.1f GB/s  %s%s" % (r["kernel"], r["median_us"], r["achieved_GBps"],
                                                     "" if r["frac_of_peak"] is None else "%.2f of peak" % r["frac_of_peak"],
                                                     "  (trimmed mean %.1f us, %.2f)" % (r["trimmed_mean_us"], r["frac_of_peak_by_trimmed_mean"])
                                                     if "trimmed_mean_us" in r else ""))


def run_sweep(args):
    from transferattack_b200 import ops, _lib
    be = ops.backend()
    hbm_peak, _ = peaks()
    dev = "cuda"
    flush = torch.empty(1024 * 1024 * 1024 // 4, device=dev)
    res = []
    for B in (64, 256):
        N = B * IMG_ELEMS
        g = torch.randn(B, 3, 224, 224, device=dev) * 1e-4
        m = torch.randn_like(g); x = torch.rand_like(g); d = (torch.rand_like(g) * 2 - 1) * (16 / 255)
        m2, d2, xa = torch.empty_like(g), torch.empty_like(g), torch.empty_like(g)
        so = torch.empty(B, device=dev)
        for mode_name, mode in (("exact", _lib.TA_MEAN_EXACT), ("torch", _lib.TA_MEAN_TORCH)):
            for cl in (2, 4, 8, 16):
                for unroll in (1, 2, 4):
                    for k, v in (("fused.cluster", cl), ("fused.unroll", unroll)):
                        _lib.tune_set(k, v)
                    ok = be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, 1.6 / 255, 16 / 255, 0, 1.0, mean_mode=mode)
                    if not ok:
                        res.append({"B": B, "mean": mode_name, "cluster": cl, "unroll": unroll, "error": _lib.last_error()[:120]})
                        continue
                    med, mn = time_kernel(lambda: be.fused_tail(g, m, m2, d, d2, x, xa, None, so, 1.0, 1.6 / 255, 16 / 255, 0, 1.0, mean_mode=mode),
                                          iters=10, flush=flush)
                    gbs = 28 * N / (med * 1e-3) / 1e9
                    res.append({"B": B, "mean": mode_name, "cluster": cl, "unroll": unroll,
                                "median_us": med * 1e3, "GBps": gbs, "frac": gbs / hbm_peak})
        del g, m, x, d, m2, d2, xa
    for k, v in (("fused.cluster", 0), ("fused.unroll", 2)):
        _lib.tune_set(k, v)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(res, open(os.path.join(ROOT, "gpurun_out", "sweep.json"), "w"), indent=1)
    ok = [r for r in res if "GBps" in r]
    for B in (64, 256):
        best = sorted([r for r in ok if r["B"] == B], key=lambda r: -r["GBps"])[:5]
        for r in best:
            print(B, r)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.cpu_worker:
        cpu_worker(args)
        return
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.kernels:
        run_kernels(args); return
    if args.sweep:
        run_sweep(args); return
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world, dist)
    finally:
        if dist is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

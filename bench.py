#!/usr/bin/env python
"""Benchmark of the Defense-GAN projection loop (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision fp16|fp32]
                    [--config mnist|fmnist|celeba] [--batch B --rec_rr R --rec_iters L]
                    [--scaling weak|strong] [--no_extra] [--no_profile] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic images: one `gan.reconstruct` call =
R restarts x L momentum-GD steps of generator forward + MSE + backward-to-z, then arg-min select.

Workloads (BASELINE.json `configs`):
  N=1   configs[1]: MNIST 28x28, R=10, L=200, batch=256 on one B200 - the configuration the metric is quoted on.
        The same line carries configs[2] (F-MNIST: the same generator class with a second weight seed, SURVEY 8d)
        and configs[3] (CelebA 64x64x3, batch 128) under `extra_configs`, and the per-GPU share of configs[4]
        (512 images on one GPU) under `weak_scaling_base`.
  N>1   configs[4]: MNIST R=10 L=200, batch 4096 over 8 GPUs = 512 images per GPU, held fixed as N varies
        (`scaling: weak`, the default).  `--scaling strong` runs the whole 4096-image batch at every N.
The image axis is sharded with no data-path collective; ONE NCCL all-gather of the reconstructions ends each step
and is inside both timed regions.

Prints ONE JSON line (rank 0).  `value` = images/s with inputs resident in HBM, CUDA-event timed, max over ranks;
`e2e` = the same through the public Python API with pinned HOST buffers (H2D of the images, the all-gather and the
D2H of the reconstructions inside the timed region); `roofline` = the dominant kernel's algorithmic FLOP/s (CUDA
events around each launch on the launching stream, in a separate pass) against the measured bf16 tensor peak in
MEASURED_PEAKS.json; `cpu_baseline` = the oracle restatement of the reference's TF1 CPU path on this box's host
cores (bounded sample).  `--impl reference` times only that CPU port (the reference itself cannot run: no TF1/py2).

The inputs are drawn on the host from fixed seeds (the generator's forward in float64 by the CPU oracle), so the same
arguments give the same inputs on every run and with every build of the library.  `--dump-outputs DIR` writes what the
last timed step returned to its caller, the reconstructions, as DIR/reconstructions.npy (float32): two builds can then
be compared output for output.  An output over 64 MiB is replaced by a fixed, seeded sample of its images, whose indices
go to DIR/reconstructions_rows.npy.
"""
import argparse
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

import numpy as np
import torch

CONFIGS = {
    # name: (dataset, default batch per GPU, R, L)
    "mnist": ("mnist", 256, 10, 200),     # BASELINE.json configs[1]
    "fmnist": ("f-mnist", 256, 10, 200),  # configs[2]
    "celeba": ("celeba", 128, 10, 200),   # configs[3]
}
C5_GLOBAL_BATCH = 4096                    # configs[4]: MNIST R=10 L=200, batch 4096 sharded across 8 GPUs
C5_PER_GPU = C5_GLOBAL_BATCH // 8
FMNIST_WEIGHT_SEED = 11241991             # synthetic C3 differs from C2 only in the weights (SURVEY 8d)
FALLBACK_PEAKS = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}
DUMP_BYTES = 64 * 2 ** 20 - 4096          # --dump-outputs: all files together, .npy headers included, stay under 64 MiB
DUMP_SAMPLE_SEED = 0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


def dump_output(out_dir, name, t):
    """Write `t` as out_dir/<name>.npy in float32.  Above DUMP_BYTES only a fixed, seeded sample of its leading-axis rows
    is written (the same rows for the same shape), and out_dir/<name>_rows.npy holds their indices (float64)."""
    a = t.detach().float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    if a.nbytes > DUMP_BYTES:
        row_bytes = a.nbytes // a.shape[0]
        n = DUMP_BYTES // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(a.shape[0], n, replace=False))
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        a = a[rows]
    path = os.path.join(out_dir, name + ".npy")
    np.save(path, a)
    return path


class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [c for c, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU port of the reference path (oracle/), data-parallel over images so that a many-core host is used
# ------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def _cpu_worker_init(threads):
    torch.set_num_threads(threads)
    from oracle import defensegan_oracle as O
    _CPU_STATE["O"] = O


def _cpu_worker_run(job):
    dataset, R, L, lo, hi, total = job
    O = _CPU_STATE["O"]
    arch = O.canonical_arch(dataset)
    key = ("w", arch)
    if key not in _CPU_STATE:
        _CPU_STATE[key] = O.init_generator_weights(arch)
    w = _CPU_STATE[key]
    ikey = ("in", arch, total, R)
    if ikey not in _CPU_STATE:
        _CPU_STATE[ikey] = (O.synthetic_images(arch, w, total), O.sample_z0(total * R, 128))
    imgs, z0 = _CPU_STATE[ikey]
    out = O.reconstruct(arch, w, imgs[lo:hi], R, L, z_init_val=z0[lo * R:hi * R])
    return float(out["loss_min"].sum())


class CpuPort:
    """The oracle restatement of the reference's TF1 CPU path (oracle/defensegan_oracle.py, fp32) on the host cores.
    One torch process stops scaling near 16 threads on these small per-step tensors (tens of rows).  Splitting the
    sample's images over several worker processes (DGAN_CPU_PROCS) is supported, but on the pool's GPU boxes it measured
    SLOWER (8 x 16 threads: 1.8 images/s against 3.0-3.6 for 1 x 16; 128 logical CPUs are visible, the container's CPU
    share evidently is not), so the default is one process - cores used = procs x threads is reported next to cores present."""

    def __init__(self, sample_images):
        self.cores_present = os.cpu_count() or 1
        self.threads = int(os.environ.get("DGAN_CPU_THREADS", min(self.cores_present, 16)))
        want = int(os.environ.get("DGAN_CPU_PROCS", 1))
        self.procs = max(1, min(want, sample_images))
        self.pool = None
        if self.procs > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("spawn").Pool(self.procs, initializer=_cpu_worker_init, initargs=(self.threads,))
        else:
            _cpu_worker_init(self.threads)

    @property
    def cores_used(self):
        return self.procs * self.threads

    def run(self, dataset, R, L, sample_images):
        """Seconds for `sample_images` images at the full R and L."""
        bounds = [round(i * sample_images / self.procs) for i in range(self.procs + 1)]
        jobs = [(dataset, R, L, bounds[i], bounds[i + 1], sample_images) for i in range(self.procs) if bounds[i + 1] > bounds[i]]
        t0 = time.perf_counter()
        if self.pool is not None:
            self.pool.map(_cpu_worker_run, jobs)
        else:
            for j in jobs:
                _cpu_worker_run(j)
        return time.perf_counter() - t0

    def describe(self, sample_images, R, L, secs=None):
        s = "%d images%s at full R=%d, L=%d on %d processes x %d threads (%d host cores present); oracle restatement of " \
            "the TF1 CPU path (the Python-2/TF-1.7 reference cannot run offline)" % (
                sample_images, " per step" if secs is None else "", R, L, self.procs, self.threads, self.cores_present)
        if secs is not None:
            s += "; %.1f s" % secs
        return s

    def close(self):
        if self.pool is not None:
            self.pool.terminate()
            self.pool.join()


def run_reference_arm(args, rank, world, out):
    """--impl reference: the reference's own CPU implementation of the path cannot run here (Python 2 +
    TensorFlow 1.7, neither present nor installable offline) => the oracle port is timed on the host cores, rank 0
    only; each step is a bounded sample (`--ref_sample` images) of the arm's workload."""
    if rank != 0:
        return
    dataset, B, R, L = resolve_workload(args, world)
    sample = max(1, args.ref_sample)
    port = CpuPort(sample)
    port.run(dataset, R, L, min(sample, port.procs))           # start-up (imports, weight draw) outside the timed region
    for _ in range(args.warmup):
        port.run(dataset, R, L, sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        port.run(dataset, R, L, sample)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": "reconstructed images/sec at R=%d,L=%d" % (R, L), "value": value,
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": arm_config(dataset, B, R, L, world, args.precision),
        "per_step_sample_images": sample,
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": port.cores_used, "cores_present": port.cores_present,
                         "kind": "port", "sample": port.describe(sample, R, L)},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    port.close()
    out.emit(json.dumps(line))


def resolve_workload(args, world):
    """(dataset, images per GPU, R, L) of this run."""
    dataset, B, R, L = CONFIGS[args.config]
    if world > 1 and args.config == "mnist":
        B = C5_PER_GPU if args.scaling == "weak" else C5_GLOBAL_BATCH // world
    elif args.scaling == "strong" and args.config == "mnist":
        B = C5_GLOBAL_BATCH
    if args.batch:
        B = args.batch
    if args.rec_rr:
        R = args.rec_rr
    if args.rec_iters:
        L = args.rec_iters
    return dataset, B, R, L


def workload_name(dataset, B, R, L, world=1):
    return "%s %s generator projection, batch=%d/GPU x %d GPU, R=%d, L=%d" % (
        dataset, "64x64x3" if dataset == "celeba" else "28x28x1", B, world, R, L)


def arm_config(dataset, B, R, L, world, precision):
    """The `config` object of the JSON line.  Both arms (this repo's and `--impl reference`) print the SAME object for
    the same command line - the contract runs the reference arm "on your arm's config" - so entries that only one arm
    can realise say which arm they describe."""
    b_global = B * world
    if (R, L) != (10, 200):
        base = "custom"
    elif world == 1 and B == 256 and dataset == "mnist":
        base = "configs[1]"
    elif dataset == "mnist" and b_global == C5_GLOBAL_BATCH:
        base = "configs[4]"
    elif dataset == "mnist" and B == C5_PER_GPU:
        base = "configs[4] per-GPU share x %d GPUs" % world
    elif world == 1 and (dataset, B) in (("f-mnist", 256), ("celeba", 128)):
        base = "configs[2]" if dataset == "f-mnist" else "configs[3]"
    else:
        base = "custom"
    return {"workload": workload_name(dataset, B, R, L, world), "dataset": dataset, "global_batch": b_global,
            "per_gpu_batch": B, "rec_rr": R, "rec_iters": L, "rec_lr": 10.0, "baseline_config": base,
            "precision": "GPU arm: %s operands, f32 accumulate and state; CPU reference arm: f32" % precision,
            "parallelism": "GPU arm: image-shard x%d + 1 all-gather (inside value and e2e); CPU reference arm: rank 0's "
                           "host cores on a bounded sample of this workload (cpu_baseline.sample)" % world,
            "l2": "GPU arm: 192 MiB memset between steps (inside the timed bracket); CPU reference arm: not applicable",
            "e2e_bytes": "GPU arm, summed over ranks: each rank copies the full batch in and the full result out"}


class _OnlyJsonOnStdout:
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner to fd 1) must not
    leak into it: while active, fd 1 points at stderr; emit() writes to the real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self._real = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.write(self._real, (text + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._real, 1)
        os.close(self._real)
        return False


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Workload:
    """One (generator, batch, R, L) on this rank's GPU with its synthetic inputs resident in HBM."""

    def __init__(self, dataset, B_local, R, L, precision, dev, rank, world, weight_seed=None):
        from defensegan_b200.models.gan import dataset_gan_dict
        self.dataset, self.B, self.R, self.L, self.dev, self.rank, self.world = dataset, B_local, R, L, dev, rank, world
        kw = {} if weight_seed is None else {"seed": weight_seed}
        self.gan = dataset_gan_dict[dataset](test_mode=True, verbose=False, precision=precision, batch_size=R * 5, **kw)
        self.gan.rec_rr, self.gan.rec_iters, self.gan.rec_lr = R, L, 10.0
        self.hwc = int(np.prod(self.gan.image_dim))
        self.B_global = B_local * world
        # synthetic inputs (SURVEY 8d, S1: on-manifold + noise): G(z*) by the float64 CPU oracle, not by the library under
        # test, so that every build is fed the same images
        from oracle import defensegan_oracle as O
        g = torch.Generator(device="cpu").manual_seed(1990)
        sig = (1.0 / self.gan.latent_dim) ** 0.5
        zstar = torch.randn(self.B_global, self.gan.latent_dim, generator=g) * sig
        eps = torch.randn(self.B_global, *self.gan.image_dim, generator=g)
        lo = -1.0 if dataset == "celeba" else 0.0
        with torch.no_grad():
            on_manifold = O.generator_forward(dataset, O.weights_to_torch(self.gan.weights, torch.float64), zstar.double())
        self.x_full = (on_manifold.float() + 0.1 * eps).clamp_(lo, 1.0).to(dev).contiguous()
        self.z0_full = (torch.randn(self.B_global * R, self.gan.latent_dim, generator=g) * sig).to(dev)
        self.x_host = self.x_full.cpu().pin_memory()
        self.out_host = torch.empty_like(self.x_host).pin_memory()

    def step(self):
        """Device-resident inputs -> full [B_global, H, W, C] result on every rank (all-gather inside)."""
        if self.world > 1:
            from defensegan_b200.parallel import reconstruct_sharded
            return reconstruct_sharded(self.gan, self.x_full, z_init_val=self.z0_full)
        return self.gan.reconstruct(self.x_full, z_init_val=self.z0_full)

    def e2e_step(self):
        """The call a user makes, host to host: pinned images -> device, projection (+ all-gather), result -> pinned host."""
        xd = self.x_host.to(self.dev, non_blocking=True)
        if self.world > 1:
            from defensegan_b200.parallel import reconstruct_sharded
            r = reconstruct_sharded(self.gan, xd, z_init_val=self.z0_full)
        else:
            r = self.gan.reconstruct(xd, z_init_val=self.z0_full)
        self.out_host.copy_(r, non_blocking=True)
        return r

    def close(self):
        self.gan.close()


def timed(fn, steps, warmup, dev, flush, distributed):
    """(ms for `steps` calls of fn, CUDA events, barrier + synchronize on both sides, max over ranks; what the last call
    returned)."""
    import torch.distributed as dist

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        flush.zero_()
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(steps):
        flush.zero_()                      # > L2 capacity written between timed iterations (inside the bracket)
        if i + 1 < steps:
            fn()                           # dropped at once, so the next step can reuse its memory
        else:
            last = fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), last


def kernel_breakdown(wl, peaks, precision):
    """Per-kernel CUDA-event pass (rank 0; not part of `value`): [{kernel, launches, avg_us, share, tflops}], roofline."""
    nat = wl.gan._native
    x_loc = wl.x_full[:wl.B].contiguous()
    z_loc = wl.z0_full[:wl.B * wl.R].contiguous()
    nat.profile_enable(True)
    wl.gan.reconstruct(x_loc, z_init_val=z_loc)
    torch.cuda.synchronize(wl.dev)
    prof = nat.profile_read()
    nat.profile_enable(False)
    tot_ms = sum(k["ms"] for k in prof) or 1.0
    kernels = []
    for k in prof:
        if k["launches"] == 0:
            continue
        avg_ms = k["ms"] / k["launches"]
        tf = k["flops_per_launch"] / (avg_ms * 1e-3) / 1e12 if avg_ms > 0 else 0.0
        kernels.append({"kernel": k["name"], "launches": k["launches"], "avg_us": round(avg_ms * 1e3, 2),
                        "share": round(k["ms"] / tot_ms, 4), "tflops": round(tf, 2)})
    if not kernels:
        return None, None
    dom = max(kernels, key=lambda k: k["share"])
    # a kernel that runs for tens of milliseconds settles at the power-capped clock: the sustained figure is its peak;
    # a sub-millisecond kernel timed alone is compared with the burst figure (B200_PROFILING.md)
    long_running = dom["avg_us"] >= 5000.0
    peak = peaks["bf16_tflops_sustained" if long_running else "bf16_tflops"] if precision == "fp16" else None
    traffic, tsrc = None, None
    tp = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        ent = tj.get("workloads", {}).get("%s/%d/%s" % (wl.dataset, wl.B * wl.R, precision), {}).get(dom["kernel"])
        if ent:
            traffic, tsrc = ent.get("dram_bytes_per_launch"), ent.get("source")
    roofline = {"bound": "tensor", "kernel": dom["kernel"], "achieved": dom["tflops"], "peak": peak, "unit": "TFLOP/s",
                "frac": (dom["tflops"] / peak) if peak else None, "traffic": traffic,
                "traffic_unit": "bytes/launch (dram__bytes_read.sum + dram__bytes_write.sum; %s)" % (tsrc or "no ncu capture for this workload"),
                "peak_source": "%s cuBLAS bf16 %s (MEASURED_PEAKS.json; fp16 and bf16 share the kind::f16 rate)" % (
                    peaks["_source"], "sustained: the kernel runs for %.1f ms" % (dom["avg_us"] / 1e3) if long_running else "burst"),
                "operand_format": precision,
                "flops_per_launch": next(k["flops_per_launch"] for k in prof if k["name"] == dom["kernel"])}
    return kernels, roofline


def pipeline_timeline(wl, roofline):
    """Where an L-step goes inside the real chain (graph replay, PDL): the probe build of the library (same sources,
    -DDGAN_PROBE: per-CTA %globaltimer stamps) runs one short call of this workload in a process of its own and reports, per
    kernel of the last L-step, how long it was busy and what the hand-over from its predecessor cost.  CUDA events around a
    single launch (`kernels`, `roofline.achieved`) also time the launch, set-up and drain that PDL overlaps with the
    neighbouring kernels; this pass does not.  Returns None when the probe library is not built."""
    import subprocess
    from defensegan_b200 import _native
    if not os.path.exists(_native.PROBE_LIB_PATH) or wl.dataset == "celeba":
        return None
    env = dict(os.environ, DGAN_LIB=_native.PROBE_LIB_PATH)
    try:
        res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "probe_step.py"), wl.dataset, str(wl.B), "50", "--json"],
                             env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=300)
        tl = json.loads(res.stdout.strip().splitlines()[-1])
    except Exception as e:      # a measurement aid must not take the bench line down
        return {"error": repr(e)}
    if roofline is not None:
        for k in tl["kernels"]:
            if k["kernel"] == roofline["kernel"] and k["tflops_while_busy"] and roofline.get("peak"):
                roofline["in_pipeline"] = {"busy_us": k["busy_us"], "handover_us": k["handover_us"], "achieved": k["tflops_while_busy"],
                                           "frac": k["tflops_while_busy"] / roofline["peak"],
                                           "how": "probe build, %globaltimer: last CTA entry -> last CTA end of this kernel in the graph-replayed chain"}
    return tl


def main():
    with _OnlyJsonOnStdout() as out:
        _main(out)


def _main(out):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "fp32"])
    ap.add_argument("--config", default="mnist", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (overrides the config)")
    ap.add_argument("--rec_rr", type=int, default=0)
    ap.add_argument("--rec_iters", type=int, default=0)
    ap.add_argument("--ref_sample", type=int, default=16, help="images per step of the CPU reference arm")
    ap.add_argument("--cpu_sample", type=int, default=64, help="images of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--no_profile", action="store_true")
    ap.add_argument("--no_extra", action="store_true", help="skip the configs[2]/[3]/[4]-share and batch-50 sub-measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's reconstructions to DIR (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; the reference arm has no such output")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world, out)
        return
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d does not match WORLD_SIZE %d" % (args.gpus, world))
    if args.warmup < 3:
        print("note: the timing rules ask for >= 3 warm-up steps", file=sys.stderr)

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    dataset, B, R, L = resolve_workload(args, world)
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    wl = Workload(dataset, B, R, L, args.precision, dev, rank, world,
                  weight_seed=FMNIST_WEIGHT_SEED if dataset == "f-mnist" else None)

    # ---- device-timed throughput (`value`) --------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    for _ in range(args.warmup):
        flush.zero_()
        wl.step()
    torch.cuda.synchronize(dev)
    if rank == 0:
        sampler.start()
    ms, last_rec = timed(wl.step, args.steps, 0, dev, flush, distributed)
    clocks = sampler.stop() if rank == 0 else None
    launches_per_step = wl.gan._native.last_launch_count
    enqueues_per_call = wl.gan._native.last_enqueue_count
    value = wl.B_global * args.steps / (ms / 1000.0)
    if args.dump_outputs and rank == 0:
        print("wrote", dump_output(args.dump_outputs, "reconstructions", last_rec), file=sys.stderr)
    del last_rec

    # ---- end-to-end through the public API with HOST buffers (`e2e`) ------------------------------------
    ms_e2e, _ = timed(wl.e2e_step, args.steps, max(1, min(args.warmup, 2)), dev, flush, distributed)
    e2e_value = wl.B_global * args.steps / (ms_e2e / 1000.0)

    peaks = load_peaks()
    kernels, roofline = (None, None)
    timeline = None
    if rank == 0 and not args.no_profile:
        kernels, roofline = kernel_breakdown(wl, peaks, args.precision)
        if world == 1 and args.precision == "fp16":
            timeline = pipeline_timeline(wl, roofline)

    # ---- the other BASELINE configs, measured the same way at reduced step counts (rank 0 / N=1 only) ----
    extra, weak_base, small_batch = None, None, None
    if world == 1 and not args.no_extra and args.config == "mnist" and not args.batch:
        k = max(3, min(args.steps, 5))

        def sub(ds, b, seed=None):
            w2 = Workload(ds, b, R, L, args.precision, dev, 0, 1, weight_seed=seed)
            m, _ = timed(w2.step, k, 3, dev, flush, False)
            me, _ = timed(w2.e2e_step, k, 1, dev, flush, False)
            macs = w2.gan._native.macs_per_row
            r = {"workload": workload_name(ds, b, R, L), "value": b * k / (m / 1e3), "ms_per_step": m / k, "steps": k,
                 "e2e": b * k / (me / 1e3), "gpu_launches_per_step": w2.gan._native.last_launch_count,
                 "tflops_whole_step": b * k / (m / 1e3) * 4.0 * macs * R * L / 1e12}
            w2.close()
            return r

        extra = [dict(sub("f-mnist", CONFIGS["fmnist"][1], FMNIST_WEIGHT_SEED), baseline_config="configs[2]"),
                 dict(sub("celeba", CONFIGS["celeba"][1]), baseline_config="configs[3]")]
        weak_base = dict(sub("mnist", C5_PER_GPU), baseline_config="configs[4] per-GPU share (512 images on one GPU)")
        small_batch = dict(sub("mnist", 50), baseline_config="the reference's own BATCH_SIZE 50 (default.yml:2)")

    # ---- CPU baseline (rank 0, N=1 only, bounded sample) ---------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        port = CpuPort(args.cpu_sample)
        port.run(dataset, R, L, min(args.cpu_sample, port.procs))     # start-up outside the timed sample
        secs = port.run(dataset, R, L, args.cpu_sample)
        cpu_baseline = {"value": args.cpu_sample / secs, "unit": "images/s", "cores": port.cores_used,
                        "cores_present": port.cores_present, "kind": "port",
                        "sample": port.describe(args.cpu_sample, R, L, secs)}
        port.close()

    if rank == 0:
        macs = wl.gan._native.macs_per_row
        gflop_per_image = 4.0 * macs * R * L / 1e9        # 2 FLOP/MAC x (fwd + bwd-to-z)
        step_tflops = value * gflop_per_image / 1e3
        bytes_io = wl.B_global * wl.hwc * 4 * world        # every rank moves the full batch in and the full result out
        line = {
            "metric": "reconstructed images/sec at R=%d,L=%d" % (R, L), "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f16" if args.precision == "fp16" else "f32", "data": "synthetic",
            "config": arm_config(dataset, B, R, L, world, args.precision),
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": bytes_io, "d2h_bytes_per_step": bytes_io},
            "gpu_launches": int(launches_per_step) * args.steps * world,
            "gpu_launches_per_call": int(launches_per_step),
            "host_enqueues_per_call": int(enqueues_per_call),
            "clocks": clocks,
            "algorithmic": {"gflop_per_image": gflop_per_image, "tflops_whole_step": step_tflops,
                            "frac_of_sustained_bf16_peak": step_tflops / (world * peaks["bf16_tflops_sustained"]),
                            "frac_of_burst_bf16_peak": step_tflops / (world * peaks["bf16_tflops"])},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "kernels": kernels, "timeline": timeline,
            "kernel_timing": None if not kernels else {
                "sum_of_kernel_us_per_call": round(sum(k["avg_us"] * k["launches"] for k in kernels), 1),
                "live_us_per_call": round(1e3 * ms / args.steps, 1),
                "note": "per-kernel times are CUDA events around each plain launch (graph replay off, no PDL overlap of "
                        "neighbouring kernels), so their sum exceeds the live call; shares, not sums, carry over"},
            "extra_configs": extra, "weak_scaling_base": weak_base, "reference_batch_size": small_batch,
        }
        out.emit(json.dumps(line))
    if distributed:
        dist.destroy_process_group()
    wl.close()


if __name__ == "__main__":
    main()

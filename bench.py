#!/usr/bin/env python
"""Benchmark of the hot path.  Default workload = BASELINE.json configs[1]:
rCCA.fit(), 2 views, n=100000 rows per GPU, d=[1024,1024], k=64, c=0.1, float32 inputs.

    python bench.py --gpus 1 --steps 10 --warmup 3            # our CUDA path (+ cpu_baseline and parity at N=1)
    python bench.py --impl reference --steps 1 --warmup 0     # the reference algorithm on the host cores, FULL size
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # sample-sharded, one all-reduce
    python bench.py --workload mcca4|ccaloss64|ccaloss512     # the other BASELINE configs (same JSON contract)
    python bench.py ... --dump-outputs DIR   # also write the last timed step's results as DIR/<name>.npy

One "step" = one fit (rcca, mcca4) or one forward+backward of the objective (ccaloss*).  Under N ranks every rank
holds its own row shard (weak scaling): the job is ONE fit over N x rows per step and its throughput is reported in
units of the 1-GPU workload (`value` = N fit-units / s; at N=1 plain fit()/s).  CCALoss is "replicas only"
(per-replica batch statistics, as in the reference): N independent replicas.  Prints ONE JSON line on rank 0.

CPU arms.  The reference is pure Python over LAPACK and /root/reference does not exist on the GPU box, so both CPU legs
run the oracle's line-by-line restatement of the reference algorithm (`kind: "port"`): `--impl reference` and the
`cpu_baseline` object time the FULL workload (no row sampling, no extrapolation); a fit of configs[1] takes about a
minute on the host cores, so the number of timed CPU fits is capped by a wall-clock budget (at least one, reported in
`steps` / `sample`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (model, rows per GPU, dims, k, c, snr, description)
    "rcca": dict(model="rcca", n=100_000, dims=[1024, 1024], k=64, c=0.1, snr=2.0 / 1024, metric="rcca_fit_per_s",
                 unit="fit/s",
                 text="rCCA.fit 2 views n=100000 rows/GPU d=[1024,1024] k=64 c=0.1 float32 (JointData snr=2/1024)"),
    "mcca4": dict(model="mcca", n=125_000, dims=[512] * 4, k=32, c=0.0, snr=2.0 / 512, metric="mcca_fit_per_s",
                  unit="fit/s",
                  text="MCCA.fit 4 views n=125000 rows/GPU d=[512]*4 k=32 c=0 float32 (JointData snr=2/512)"),
    "ccaloss64": dict(model="ccaloss", n=4096, dims=[64, 64], k=16, c=None, snr=None, metric="ccaloss_fwdbwd_per_s",
                      unit="step/s", text="CCALoss forward+backward batch=4096 widths=[64,64] eps=1e-5 float32"),
    "ccaloss512": dict(model="ccaloss", n=4096, dims=[512, 512], k=16, c=None, snr=None,
                       metric="ccaloss_fwdbwd_per_s", unit="step/s",
                       text="CCALoss forward+backward batch=4096 widths=[512,512] eps=1e-5 float32"),
}
W = dict(WORKLOADS["rcca"])
CPU_BUDGET_S = 150.0   # wall-clock budget of a CPU arm (the first fit always completes)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """Write what the timed path handed back in its last step as <out_dir>/<name>.npy (float32 / float64).  The inputs
    are seeded, so two builds run with the same arguments can be compared output for output."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class gpu_local_cpus:
    """Context manager: run the enclosed allocations on the CPUs next to GPU `index` (PCIe root / NUMA node from sysfs),
    so that the pinned staging buffers of the end-to-end leg are first-touched on the GPU's own node -- on a two-socket
    box the H2D rate from the far node is half the near one's.  The affinity is restored on exit (the CPU legs use all
    cores).  Any failure leaves the placement to the OS."""

    def __init__(self, index: int):
        self.index, self.old, self.note = index, None, "os default"

    def __enter__(self):
        try:
            import torch

            pr = torch.cuda.get_device_properties(self.index)     # CUDA ordinal (honours CUDA_VISIBLE_DEVICES)
            if hasattr(pr, "pci_bus_id"):
                path = (f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/"
                        f"local_cpulist")
            else:
                import pynvml

                pynvml.nvmlInit()
                bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(self.index)).busId
                bus = bus.decode() if isinstance(bus, bytes) else bus
                dom, rest = bus.split(":", 1)
                path = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/local_cpulist"
            cpus = set()
            for part in open(path).read().strip().split(","):
                if "-" in part:
                    a, b = part.split("-")
                    cpus.update(range(int(a), int(b) + 1))
                elif part:
                    cpus.add(int(part))
            self.old = os.sched_getaffinity(0)
            cpus &= self.old
            if cpus and cpus != self.old:
                os.sched_setaffinity(0, cpus)
                self.note = f"first touch on the {len(cpus)} CPUs local to GPU {self.index}"
        except Exception as e:                                    # noqa: BLE001
            self.note = f"os default ({type(e).__name__})"
        return self

    def __exit__(self, *exc):
        if self.old is not None:
            try:
                os.sched_setaffinity(0, self.old)
            except Exception:                                     # noqa: BLE001
                pass
        return False


def make_views(seed: int, n_rows: int | None = None):
    """Rows of ONE JointData-style population (cca_zoo/datasets/_simulated.py:113-125): the loading matrices
    W_i come from a fixed stream shared by every rank, the latent draws and the noise from `seed`, so that
    the row shards of different ranks are samples of the same model (a sharded data set, not N unrelated ones)."""
    n_rows = W["n"] if n_rows is None else n_rows
    rng_w = np.random.default_rng(20240924)
    weights = [rng_w.standard_normal((p, W["k"])) for p in W["dims"]]
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((n_rows, W["k"]))
    views = []
    for w in weights:
        noise = rng.standard_normal((n_rows, w.shape[0])).astype(np.float32) * np.float32(1.0 / np.sqrt(W["snr"]))
        noise += (z @ w.T).astype(np.float32)
        views.append(noise)
    return views


def make_representations(seed: int):
    """Config 3 inputs (SURVEY.md §8d): z_i = z_l A_i + eps, z_l ~ N(0, I_16), float32, torch CPU generator."""
    import torch

    g = torch.Generator().manual_seed(seed)
    zl = torch.randn(W["n"], 16, generator=g)
    return [zl @ torch.randn(16, w, generator=g) + torch.randn(W["n"], w, generator=g) for w in W["dims"]]


# ----------------------------------------------------------------------------------------------
# clocks sampler (NVML during the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled every ~10 ms DURING the timed region (NVML; nvidia-smi fallback)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index = index
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        nv = self._nvml
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)))
        try:
            self.power.append(nv.nvmlDeviceGetPowerUsage(self._h) / 1000.0)
        except Exception:
            pass
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for bit, name in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
        if out.returncode == 0 and out.stdout.strip():
            r = [x.strip() for x in out.stdout.strip().split(",")]
            self.sm.append(float(r[0]))
            self.mx.append(float(r[1]))
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[2:]):
                if val == "Active":
                    self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml() if self._nvml else self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.01 if self._nvml else 0.2)

    def start(self):
        self._t.start()
        return self

    def stop(self):
        try:  # one sample taken by the caller's thread at the end of the timed region (the Python-side loop
            self._sample_nvml() if self._nvml else self._sample_smi()   # can starve the sampler thread)
        except Exception:
            pass
        self._stop.set()
        self._t.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                "source": "nvml" if self._nvml else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port: the same LAPACK / torch-CPU calls as the reference)
# ----------------------------------------------------------------------------------------------
def cpu_threads():
    try:
        from threadpoolctl import threadpool_info

        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_step_fn():
    """A closure running ONE full-size step of the workload with the reference's algorithm on the host cores."""
    from oracle import restatement as R

    if W["model"] == "rcca":
        views = make_views(1000)
        return lambda: R.ref_rcca_fit(views, W["k"], W["c"]), "oracle.ref_rcca_fit (numpy LAPACK: the gesdd / svd " \
            "calls of cca_zoo/linear/_rcca.py:83-101)"
    if W["model"] == "mcca":
        views = make_views(1000)
        return lambda: R.ref_mcca_fit(views, W["k"], W["c"]), "oracle.ref_mcca_fit (np.cov + scipy eigh of " \
            "cca_zoo/linear/_mcca.py:113-173)"
    import torch

    z = make_representations(0)
    return lambda: R.ref_ccaloss_torch_fwdbwd(z[0], z[1], 1e-5), "oracle.ref_ccaloss_torch_fwdbwd (torch CPU eigh + " \
        "autograd, cca_zoo/deep/objectives.py:9-21,79-102)"


def time_cpu(steps: int, warmup: int, budget_s: float = CPU_BUDGET_S):
    """Full-size CPU steps: `warmup` untimed then up to `steps` timed ones, both cut short by the wall-clock budget
    (a step that takes longer than 30 s is its own warm-up: BLAS start-up is noise against it).  Returns
    (seconds per step, timed steps, what ran)."""
    fn, what = cpu_step_fn()
    t_start = time.perf_counter()
    t0 = time.perf_counter()
    fn()
    first = time.perf_counter() - t0
    times = []
    if first > 30.0 or warmup == 0:
        times.append(first)
    else:
        for _ in range(max(warmup - 1, 0)):
            if time.perf_counter() - t_start + first > budget_s:
                break
            fn()
    while len(times) < max(steps, 1) and (not times or time.perf_counter() - t_start + np.mean(times) <= budget_s):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return float(np.mean(times)), len(times), what


def cpu_baseline_obj(steps: int = 3, warmup: int = 1, budget_s: float = CPU_BUDGET_S):
    sec, timed, what = time_cpu(steps, warmup, budget_s)
    return {"value": 1.0 / sec, "unit": W["unit"], "cores": cpu_threads(), "kind": "port", "seconds_per_step": sec,
            "sample": f"{what}: FULL workload ({W['text']}), {timed} timed step(s), no row sampling, no extrapolation"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sec, timed, what = time_cpu(args.steps, args.warmup)
    val = 1.0 / sec
    line = {
        "impl": "reference", "metric": W["metric"], "value": val, "unit": W["unit"], "n_gpus": args.gpus,
        "steps": timed, "warmup": 0 if sec > 30.0 else args.warmup, "steps_requested": args.steps,
        "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": W["text"]},
        "cpu_baseline": {"value": val, "unit": W["unit"], "cores": cpu_threads(), "kind": "port",
                         "sample": f"{what}: FULL workload, {timed} timed step(s) (wall-clock budget "
                                   f"{CPU_BUDGET_S:.0f} s), no row sampling, no extrapolation"},
        "e2e": {"value": val, "unit": W["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def parity_vs_oracle(est, views):
    """Outside the timed region: the fitted weights / canonical correlations against the float64 oracle
    (covariance form of cca_zoo/linear/_rcca.py:83-101, numpy LAPACK) on the very same float32 inputs."""
    from oracle import restatement as R

    dims, k = W["dims"], W["k"]
    X = np.hstack(views).astype(np.float64)
    n = X.shape[0]
    mu = X.mean(axis=0)
    X -= mu
    C = X.T @ X / (n - 1)
    del X
    w_ref, sv = R.cov_rcca_fit(C, dims, k, W["c"], n)
    w = [x.astype(np.float64) for x in est.weights_]
    ws = R.align_signs(w, w_ref)
    per_vec = np.concatenate([np.linalg.norm(a - b, axis=0) / np.linalg.norm(b, axis=0) for a, b in zip(ws, w_ref)])
    sub = np.random.default_rng(0).choice(n, 20_000, replace=False)
    vs = [v[sub] for v in views]
    sc = est.score(vs)
    sc_ref = R.score(vs, [mu[:dims[0]], mu[dims[0]:]], w_ref)
    return {"oracle": "oracle.restatement.cov_rcca_fit, float64, same inputs",
            "max_weight_rel_err": float(per_vec.max()), "median_weight_rel_err": float(np.median(per_vec)),
            "canonical_corr_max_rel_err": float(np.max(np.abs(sc - sc_ref) / np.abs(sc_ref))),
            "subspace_distance": float(max(R.subspace_distance(w[i], w_ref[i]) for i in range(2))),
            "min_gap_of_reference_spectrum": float(np.min(-np.diff(sv))), "tolerance_float32": 1e-3,
            "fit_route": getattr(est, "_fit_info", None)}


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def run_ours(args):
    import torch
    import torch.distributed as dist

    from cca_zoo_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: cca_zoo_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    dev = torch.device("cuda", local)
    model = W["model"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    peaks = load_peaks()
    est = None
    if model in ("rcca", "mcca"):
        from cca_zoo_b200.linear import MCCA, rCCA

        raw = make_views(1000 + rank)
        with gpu_local_cpus(dev.index if dev.index is not None else 0) as place:
            host = [torch.from_numpy(v).pin_memory() for v in raw]
        del raw
        views = [h.to(dev) for h in host]
        est = (MCCA if model == "mcca" else rCCA)(latent_dimensions=W["k"], c=W["c"], precision=args.precision)
        step_dev = lambda: est.fit(views)      # noqa: E731
        step_e2e = lambda: est.fit(host)       # noqa: E731
        h2d = sum(h.numel() * h.element_size() for h in host)
        l2_note = f"inputs ({h2d / 1e6:.0f} MB per GPU) exceed the 126 MB L2; no explicit flush"
    else:
        from cca_zoo_b200.deep import CCALoss

        raw = make_representations(rank)
        with gpu_local_cpus(dev.index if dev.index is not None else 0) as place:
            host = [z.pin_memory() for z in raw]
        del raw
        zs = [h.to(dev).requires_grad_(True) for h in host]
        fn = CCALoss(eps=1e-5)
        flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
        last = {}

        def step_dev():
            flush.zero_()                       # L2 flush between timed iterations (the batch itself is 2-16 MB)
            for z in zs:
                z.grad = None
            last["loss"] = fn(zs)
            last["loss"].backward()

        grads_host = [torch.empty_like(h).pin_memory() for h in host]
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()

        def step_e2e():
            z = [h.to(dev, non_blocking=True).requires_grad_(True) for h in host]
            loss = fn(z)
            loss.backward()
            for gh, t in zip(grads_host, z):
                gh.copy_(t.grad, non_blocking=True)
            loss_host.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()

        h2d = sum(h.numel() * h.element_size() for h in host)
        l2_note = "a 160 MB buffer is overwritten between timed iterations (L2 flush); its 0.03 ms is inside the step"

    # ---- device-resident arm (`value`) with live timing of the tcgen05 moment kernel ----
    for _ in range(args.warmup):
        step_dev()
    lib.ccab_profile_moments(1)
    k1_ms = []

    def step_prof():
        step_dev()
        k1_ms.append(lib.ccab_profile_moments_last_ms())

    sampler = ClockSampler(local).start() if rank == 0 else None
    l0 = lib.ccab_launch_count()
    total_ms = timed(step_prof, args.steps)
    launches = lib.ccab_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    lib.ccab_profile_moments(0)
    ms_per_step = total_ms / args.steps
    if args.dump_outputs and rank == 0:   # before the end-to-end leg refits the estimator
        if est is not None:
            outputs = {**{f"weights_{i}": w.copy() for i, w in enumerate(est.weights_)},
                       **{f"means_{i}": m.copy() for i, m in enumerate(est.means_)}}
        else:
            outputs = {"loss": last["loss"].detach().cpu().numpy(),
                       **{f"grad_{i}": z.grad.cpu().numpy() for i, z in enumerate(zs)}}
    value = world / (ms_per_step * 1e-3)

    # ---- end-to-end arm: pinned host inputs -> public API -> result on the host ----
    if args.no_e2e:            # profiling runs (ncu launch lists): the device-resident step only
        e2e_ms = float("nan")
    else:
        for _ in range(min(args.warmup, 2)):
            step_e2e()
        e2e_ms = timed(step_e2e, args.steps) / args.steps
    if est is not None:
        d2h = sum(w.nbytes for w in est.weights_) + sum(m.nbytes for m in est.means_)
    else:
        d2h = h2d + 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant data-parallel kernel ----
    D = sum(W["dims"])
    n = W["n"]
    k1 = float(np.mean([m for m in k1_ms if m and m > 0])) if any(m and m > 0 for m in k1_ms) else None
    roof = None
    if model in ("rcca", "mcca"):
        bf16 = peaks.get("bf16_tflops", 1590.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops/2 (TF32 runs at half the dense bf16 rate)" if peaks else \
            "fallback 1590/2 TFLOP/s (B200_PROFILING.md)"
        flops = n * D * (D + 1)  # algorithmic: symmetric product, SURVEY.md §8d (per rank)
        passes = {"tf32x3": 3, "tf32x3b": 2}.get(args.precision, 1)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "k1_traffic.json")) as f:
                tr = json.load(f)[f"{args.workload}:{args.precision}"]
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]   # one ncu --set full capture, per launch
        except Exception:
            pass
        if k1:
            ach = flops / (k1 * 1e-3) / 1e12
            kname = {"tf32x3b": "moments_x3b_persist_kernel (persistent CTA pairs; 2 bf16 cross-term + 2 tf32 MMAs per 16 samples)",
                     "tf32x3": "moments_tf32_2cta_kernel<X3> (3 tf32 MMAs per k-step)"}.get(
                         args.precision, "moments_tf32_2cta_kernel")
            roof = {"bound": "tensor", "kernel": kname, "achieved": ach, "peak": bf16 / 2,
                    "unit": "TFLOP/s", "frac": ach / (bf16 / 2), "traffic": traffic, "kernel_ms": k1,
                    "mma_passes": passes, "algorithmic_flops": flops, "algorithmic_bytes": n * D * 4,
                    "frac_of_issued": passes * ach / (bf16 / 2), "peak_source": peak_src,
                    "share_of_step": k1 / ms_per_step}
    else:
        # config 3 is HBM / latency bound (SURVEY.md §8d): algorithmic bytes = z read by the moment pass, z read again
        # and the gradients written by the backward = 3 x (2 x batch x width x 4)
        hbm = peaks.get("hbm_gbs", 6575.0)
        abytes = 3 * 2 * n * W["dims"][0] * 4
        ach = abytes / (ms_per_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "whole step (moments, small solves, backward products)", "achieved": ach,
                "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "traffic": None, "algorithmic_bytes": abytes,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback (B200_PROFILING.md)",
                "note": "latency bound: the step is a chain of small dependent launches; frac is reported, not chased"}

    line = {
        "metric": W["metric"], "value": value, "unit": W["unit"], "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": (args.precision + "+f32") if est is not None else "f32",
        "data": "synthetic",
        "config": {"workload": W["text"], "rows_per_gpu": n, "total_rows": n * world,
                   "parallelism": (f"sample-sharded x{world}, one all-reduce of the moment buffer" if est is not None
                                   else f"{world} independent replicas (per-replica batch statistics)") if world > 1
                   else "single GPU",
                   "l2": l2_note,
                   "unit_note": f"value = (n_gpus x {n}-row step-units) / step time"},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": world / (e2e_ms * 1e-3), "unit": W["unit"], "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "host_buffers": f"pinned; {place.note}"},
        "roofline": roof,
    }
    if est is not None:
        line["fit_route"] = getattr(est, "_fit_info", None)
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_obj(steps=1 if model in ("rcca", "mcca") else 5,
                                                warmup=0 if model in ("rcca", "mcca") else 1,
                                                budget_s=90.0)
        if model == "rcca":
            line["parity"] = parity_vs_oracle(est, [h.numpy() for h in host])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="tf32x3b", choices=["tf32", "tf32x3", "tf32x3b", "exact"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity legs")
    ap.add_argument("--no-e2e", action="store_true", help="profiling only: skip the end-to-end leg (the line is then "
                                                          "not a valid bench line)")
    ap.add_argument("--workload", default="rcca", choices=sorted(WORKLOADS),
                    help="rcca = BASELINE configs[1] (the headline); mcca4 = configs[3] shard; ccaloss64 / "
                         "ccaloss512 = configs[2] at the two readings of its width")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the estimator's weights_ / means_ (or the loss and its "
                                                          "gradients) of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    W.clear()
    W.update(WORKLOADS[args.workload])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

"""bench.py — NSF log_prob throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA engine)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, host cores)
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input:
``flow(c).log_prob(x)`` + the fixed-order sum of the log-densities (the per-device term of
the mean NLL) for the workload BASELINE.json quotes the metric on —
configs[1]: NSF(features=16, context=8, transforms=4, bins=8, hidden=[256]*3), batch 2^20 per
GPU.  With N > 1 (torchrun, one rank per GPU) every rank processes its own 2^20 rows (weak
scaling) and ONE NCCL all-reduce of {sum log p, count} closes the step.

Printed JSON (one line, rank 0): see the contract in the task description; additionally
``roofline`` (dominant kernel), ``kernels`` (every kernel class timed in isolation with CUDA
events), ``cpu_baseline``, ``parity`` and ``configs``: the other BASELINE.json configurations
(cfg3 MAF [512]^4 log_prob 2^20, cfg4 NSF(64, K16) rsample 2^20, cfg5 NSF(64, 16, K16, [512]^3)
log_prob with 2^21 rows per GPU = 2^24 over 8 GPUs), each timed with CUDA events after warm-up,
with its own roofline entry and oracle parity on a small slice.  Under torchrun every rank runs
cfg5 on its own 2^21-row shard, so the scaling record carries the north-star config's 1 -> 8 curve.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

# the CPU arm pins its OpenMP threads (must be in the environment before the runtime starts)
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

METRIC = "nsf_log_prob_samples_per_sec"
UNIT = "samples/s"
WORKLOAD = "NSF(features=16, context=8, transforms=4, bins=8, hidden=[256]*3) log_prob"
D, C, T, K, H = 16, 8, 4, 8, [256, 256, 256]
P = 3 * K - 1


def build_model():
    import zuko_b200 as zuko

    torch.manual_seed(0)
    return zuko.flows.NSF(D, C, transforms=T, bins=K, hidden_features=H).eval()


def measured_peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}  # fmt: skip
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU WHILE the timed region runs: an NVML
    polling thread (10 ms period by default, ZK_BENCH_CLOCK_PERIOD_MS); `nvidia-smi -lms` is the
    fallback when NVML cannot be initialised."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")  # fmt: skip
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int) -> None:
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.stop = threading.Event()
        self.source = None
        self.mode = os.environ.get("ZK_BENCH_CLOCKS", "nvml")  # nvml | smi | off
        self.period = float(os.environ.get("ZK_BENCH_CLOCK_PERIOD_MS", "10")) * 1e-3

    def _nvml_handle(self):
        import pynvml as N

        N.nvmlInit()
        try:  # CUDA_VISIBLE_DEVICES may renumber devices: address the GPU by UUID
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            return N, N.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            return N, N.nvmlDeviceGetHandleByIndex(self.index)

    def _poll_nvml(self, N, h):
        bits = [N.nvmlClocksEventReasonHwSlowdown, N.nvmlClocksEventReasonHwThermalSlowdown,
                N.nvmlClocksEventReasonSwThermalSlowdown, N.nvmlClocksEventReasonSwPowerCap]  # fmt: skip
        smax = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
        while not self.stop.is_set():
            try:
                sm = float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM))
                r = int(N.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.rows.append([sm, smax, [n for n, b in zip(self.NAMES, bits) if r & b]])
            except Exception:
                pass
            time.sleep(self.period)

    def prepare(self):
        """NVML initialisation + one full round of queries, BEFORE the warm-up: the first NVML
        calls of a process (and of a fresh box) take tens of milliseconds inside the driver and
        must not land in the timed region."""
        self._nvml = None
        if self.mode != "nvml":
            return self
        try:
            N, h = self._nvml_handle()
            N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
            N.nvmlDeviceGetCurrentClocksEventReasons(h)
            self._nvml = (N, h)
        except Exception:
            self._nvml = None
        return self

    def __enter__(self):
        if self.mode == "off":
            return self
        try:
            if self.mode == "smi":
                raise RuntimeError("nvidia-smi requested")
            N, h = getattr(self, "_nvml", None) or self._nvml_handle()
            self.thread = threading.Thread(target=self._poll_nvml, args=(N, h), daemon=True)
            self.thread.start()
            self.source = "nvml"
            t0 = time.perf_counter()
            while not self.rows and time.perf_counter() - t0 < 0.2:  # first sample landed
                time.sleep(0.001)
            return self
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(max(5, int(self.period * 1e3)))],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)  # fmt: skip
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
            self.source = "nvidia-smi"
        except OSError:
            self.proc = None
        return self

    def _read_smi(self):
        for line in self.proc.stdout:
            r = [s.strip() for s in line.split(",")]
            try:
                self.rows.append([float(r[0]), float(r[1]), [n for n, v in zip(self.NAMES, r[3:7]) if v.lower().startswith("active")]])
            except (ValueError, IndexError):
                continue

    def __exit__(self, *exc):
        self.stop.set()
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)

    def summary(self) -> dict:
        sm = [r[0] for r in self.rows]
        smax = max((r[1] for r in self.rows), default=0.0)
        reasons = sorted({n for r in self.rows for n in r[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None,
                "reasons": reasons, "samples": len(sm), "source": self.source}  # fmt: skip


def cuda_time_ms(fn, iters: int, stream=None) -> float:
    """Average device time of fn() over iters launches, CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# --------------------------------------------------------------------------- #
# CPU arm: the oracle port on the host cores
# --------------------------------------------------------------------------- #


def cpu_reference_adaptive(target_s: float, rows0: int = 1 << 15, max_rows: int = 1 << 22):
    """Sizes the bounded CPU sample so that it takes about target_s seconds on this host (the
    rate grows with the sample size on a many-core host, so the size is refined twice)."""
    rows = rows0
    rate, sec, threads = cpu_reference_rate(rows)
    for _ in range(3):
        if sec >= 0.6 * target_s or rows >= max_rows:
            break
        want = int(min(max_rows, max(rows * 2, rate * target_s)))
        rows = 1 << max(10, want.bit_length() - 1)  # power of two
        rate, sec, threads = cpu_reference_rate(rows)
    return rate, sec, threads, rows


def usable_cores() -> dict:
    """What the host really offers this process: os.cpu_count() counts the machine's logical CPUs, the
    affinity mask and the cgroup quota (containers) may allow far fewer."""
    info = {"cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        info["affinity"] = info["cpu_count"]
    quota = None
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = float(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = float(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    info["cgroup_quota"] = quota
    n = min(info["cpu_count"], info["affinity"])
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    info["threads"] = n
    return info


def cpu_reference_rate(rows: int, repeats: int = 1):
    """Times the oracle's fp32 CPU restatement of flow(c).log_prob(x) (all host threads, OpenMP)
    on `rows` rows of the bench workload.  Returns (samples/s, seconds, threads)."""
    from oracle import oracle

    threads = oracle.set_threads(int(os.environ.get("ZK_BENCH_CPU_THREADS", "0")) or usable_cores()["threads"])  # torchrun exports OMP_NUM_THREADS=1
    flow = build_model()
    spec = oracle.flowspec_from_module(flow)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(rows, D, generator=g).numpy()
    c = torch.randn(rows, C, generator=g).numpy()
    spec.log_prob(x[:256], c[:256], dtype=np.float32)  # warm-up (library load, page-in)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        spec.log_prob(x, c, dtype=np.float32)
        best = min(best, time.perf_counter() - t0)
    return rows / best, best, threads


CPU_ROWS = 1 << 19  # the bounded CPU sample of the workload: the same in the reference arm and in cpu_baseline


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one step = one pass of the oracle port over a FIXED bounded sample of the workload (the same
    # rows whatever N / steps are, so that the BENCH and SCALE reference arms agree); threads pinned
    # (OMP_PROC_BIND=close, OMP_PLACES=cores, set at import)
    rows = args.cpu_rows or CPU_ROWS
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_reference_rate(min(rows, 1 << 16))
    times = []
    threads = 1
    for _ in range(args.steps):
        _, sec, threads = cpu_reference_rate(rows)
        times.append(sec)
    sec = float(np.median(times))
    rate = rows / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows_per_step": rows, "note": "oracle port (plain C, OpenMP, threads pinned) of the reference's CPU path; fixed bounded sample per step, median step time",
                   "step_seconds_min_max": [float(min(times)), float(max(times))]},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "host": usable_cores(), "sample": f"{rows} rows of the workload per step"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }  # fmt: skip
    print(json.dumps(line))


# --------------------------------------------------------------------------- #
# the other BASELINE.json configurations (configs[2..4])
# --------------------------------------------------------------------------- #

OTHER_CONFIGS = [
    {"name": "cfg3", "workload": "MAF(features=32, transforms=8, hidden=[512]*4) log_prob, batch 2^20",
     "kind": "maf", "D": 32, "C": 0, "T": 8, "K": 0, "H": [512] * 4, "op": "log_prob", "rows": 1 << 20},
    {"name": "cfg4", "workload": "NSF(features=64, bins=16, transforms=8) rsample((2^20,)) inverse path",
     "kind": "nsf", "D": 64, "C": 0, "T": 8, "K": 16, "H": [64, 64], "op": "rsample", "rows": 1 << 20},
    {"name": "cfg5", "workload": "NSF(features=64, context=16, transforms=8, bins=16, hidden=[512]*3) log_prob, 2^21 rows per GPU (2^24 over 8)",
     "kind": "nsf", "D": 64, "C": 16, "T": 8, "K": 16, "H": [512] * 3, "op": "log_prob", "rows": 1 << 21},
]  # fmt: skip


def build_config_model(cfg):
    import zuko_b200 as zuko

    torch.manual_seed(0)
    if cfg["kind"] == "maf":
        return zuko.flows.MAF(cfg["D"], cfg["C"], transforms=cfg["T"], hidden_features=cfg["H"]).eval()
    return zuko.flows.NSF(cfg["D"], cfg["C"], transforms=cfg["T"], bins=cfg["K"], hidden_features=cfg["H"]).eval()


def tensor_peak(peaks: dict, clocks: dict) -> tuple[float, str]:
    """The denominator of a tensor-bound roofline: the measured cuBLAS burst figure (taken at the maximum SM clock) when
    the run held >= 98 % of that clock, else the same figure scaled to the clock the run actually held — the pipe's
    capacity under the power cap the timed region saw.  (MEASURED_PEAKS.json's own "sustained" figure was taken at one
    particular capped clock, 1305 MHz in round 1: dividing a run at 1935 MHz by it flatters, a run at 1680 MHz reads
    above 1.  It is reported next to the fraction as `peak_sustained`.)"""
    sm, smax = clocks.get("sm_mhz"), clocks.get("sm_max_mhz")
    burst = peaks["bf16_tflops"]
    if not sm or not smax or sm >= 0.98 * smax:
        return burst, "burst"
    return burst * sm / smax, f"burst x {sm / smax:.3f} (SM clock held {sm:.0f} of {smax:.0f} MHz)"


def fused_info(flow) -> dict:
    """Which kernel runs the flow's layers and the tensor-core work its schedules ISSUE (non-zero
    tiles only, all split terms) next to the dense work of nn.py:218 — from the packs."""
    import ctypes

    from zuko_b200 import _engine as E

    kinds, issued, dense, entries = [], 0.0, 0.0, 0
    for layer in flow.transform.transforms:
        out = (ctypes.c_double * 4)()
        k = E.lib().zk_layer_fused_info(layer._zk_layer(), out)
        kinds.append({0: "per-layer GEMM kernels", 1: "fused_layer_kernel", 2: "fused_wide_kernel", 3: "fused_dual_kernel"}.get(k, "?"))
        issued += out[2]
        dense += out[3]
        entries += int(out[1])
    return {"kernel": sorted(set(kinds)), "dense_macs_per_row": dense, "issued_macs_per_row": issued, "schedule_entries": entries}


def time_config(cfg, dev, rank, world, peaks, steps, nvml=None) -> dict:
    """One BASELINE configuration: warm-up, `steps` timed steps (CUDA events, max over ranks), oracle
    parity on a small slice (rank 0), roofline entry.  Inputs live in HBM; they rotate over buffers
    that together exceed the 126 MB L2."""
    import torch.distributed as dist

    from zuko_b200 import _engine as E
    from zuko_b200.dist import NllRing

    D, C, rows = cfg["D"], cfg["C"], cfg["rows"]
    flow_cpu = build_config_model(cfg)
    flow = build_config_model(cfg).to(dev)
    g = torch.Generator(device=dev).manual_seed(4321 + rank)
    nbuf = max(1, min(4, -(-(160 << 20) // (rows * (D + C) * 4))))  # > 126 MB in rotation
    xs = [torch.randn(rows, D, generator=g, device=dev) for _ in range(nbuf)]
    cs = [torch.randn(rows, C, generator=g, device=dev) for _ in range(nbuf)] if C else [None] * nbuf
    ring = NllRing(dev, slots=32)
    with torch.no_grad():
        if cfg["op"] == "log_prob":
            def step(i):
                return flow(cs[i % nbuf]).log_prob_and_sum(xs[i % nbuf], sum_out=ring.slot(rows))[0]
        else:  # rsample: z ~ N(0, I) supplied in HBM (RNG parity is not attempted, SURVEY §8c), x = transform.inv(z)
            t = flow(None).transform
            def step(i):
                return t.inv(xs[i % nbuf])
        parity = None
        if rank == 0:
            from oracle import oracle

            spec = oracle.flowspec_from_module(flow_cpu)
            n = 1024 if cfg["op"] == "log_prob" else 128
            xh = xs[0][:n].cpu().numpy()
            ch = None if cs[0] is None else cs[0][:n].cpu().numpy()
            if cfg["op"] == "log_prob":
                ours = flow(None if cs[0] is None else cs[0][:n]).log_prob(xs[0][:n]).cpu().numpy().astype(np.float64)
                ref = spec.log_prob(xh, ch)
            else:
                ours = flow(None).transform.inv(xs[0][:n]).cpu().numpy().astype(np.float64)
                ref = spec.inverse(xh, None)
            parity = {"rows": n, "max_rel_err_vs_fp64_oracle": float(np.max(np.abs(ours - ref) / np.maximum(np.abs(ref), 1.0)))}
        for i in range(3):
            step(i)
        ring.means()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clk = ClockSampler(dev.index or 0)
        clk._nvml = nvml
        n0 = E.lib().zk_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with clk:
            torch.cuda.synchronize()
            e0.record()
            for i in range(steps):
                step(i)
            means = ring.means()  # the collective(s) of the mean NLL close the timed region
            e1.record()
            torch.cuda.synchronize()
        launches = E.lib().zk_launch_count() - n0
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_per_step = ms.item() / steps
    clocks = clk.summary()
    out = {"name": cfg["name"], "workload": cfg["workload"], "rows_per_gpu": rows, "value": world * rows / (ms_per_step * 1e-3),
           "unit": UNIT, "ms_per_step": ms_per_step, "steps": steps, "gpu_launches": int(launches), "parity": parity, "clocks": clocks,
           "l2": f"inputs rotate over {nbuf} buffer(s) of {rows * (D + C) * 4 >> 20} MB"}  # fmt: skip
    if cfg["op"] == "log_prob":
        info = fused_info(flow)
        flops = 2.0 * info["dense_macs_per_row"] * rows
        peak, kind = tensor_peak(peaks, clocks)
        tf = flops / (ms_per_step * 1e-3) / 1e12
        out["mean_nll"] = float(means[-1].item()) if means.numel() else None
        out["roofline"] = {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "peak_kind": kind,
                           "kernel": info["kernel"], "algorithmic_flops_per_step": flops, "issued_flops_per_step": 2.0 * info["issued_macs_per_row"] * rows,
                           "frac_issued": 2.0 * info["issued_macs_per_row"] * rows / (ms_per_step * 1e-3) / 1e12 / peak,
                           "traffic": None, "algorithmic_hbm_bytes": 4.0 * (D + C + 1) * rows, "peak_sustained": peaks["bf16_tflops_sustained"]}  # fmt: skip
        tj = ncu_traffic().get(f"{cfg['name']}_layer")
        if tj:  # one `ncu --set full` capture of ONE flow layer launch of this config (bytes, and the rows that launch covered)
            out["roofline"]["traffic"] = tj.get("bytes")
            out["roofline"]["traffic_rows"] = tj.get("rows")
            out["roofline"]["traffic_note"] = "per layer launch over traffic_rows rows; algorithmic: 4 (2 D + C + 1) bytes per row"
            out["roofline"]["traffic_captured_at"] = ncu_traffic().get("git_sha")
    else:
        # every weight of the masked conditioner is visited once per sample (ar_inverse.cu): 2 FLOP per
        # non-zero weight; roofline = fp32 FMA pipe, 148 SMs x 128 lanes x 2 x SM clock (nominal)
        nnz = sum(float(m.mask.sum()) for layer in flow_cpu.transform.transforms for m in layer.hyper if hasattr(m, "mask"))
        flops = 2.0 * nnz * rows
        smax = clocks.get("sm_max_mhz") or 1965.0
        peak = 148 * 128 * 2 * smax * 1e6 / 1e12
        tf = flops / (ms_per_step * 1e-3) / 1e12
        out["roofline"] = {"bound": "fma", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "peak_kind": "nominal fp32 FMA (148 SMs x 128 lanes x 2 x max SM clock)",
                           "kernel": ["ar_inverse_kernel<RQS,16>"], "algorithmic_flops_per_step": flops, "traffic": None,
                           "algorithmic_hbm_bytes": 4.0 * 2 * D * rows}  # fmt: skip
        tj = ncu_traffic().get(f"{cfg['name']}_layer")
        if tj:
            out["roofline"]["traffic"] = tj.get("bytes")
            out["roofline"]["traffic_rows"] = tj.get("rows")
            out["roofline"]["traffic_captured_at"] = ncu_traffic().get("git_sha")
    del xs, cs, flow
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- #
# our arm
# --------------------------------------------------------------------------- #


def run_ours(args) -> None:
    import torch.distributed as dist

    import zuko_b200 as zuko  # noqa: F401
    from zuko_b200 import _engine as E

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    peaks = measured_peaks()

    flow = build_model().to(dev)
    NBUF = 4  # inputs rotate over 4 buffers: 4 x 100 MB > 126 MB L2
    g = torch.Generator().manual_seed(1234 + rank)
    xs_host = [torch.randn(B, D, generator=g).pin_memory() for _ in range(NBUF)]
    cs_host = [torch.randn(B, C, generator=g).pin_memory() for _ in range(NBUF)]
    xs = [t.to(dev) for t in xs_host]
    cs = [t.to(dev) for t in cs_host]
    from zuko_b200.dist import NllRing

    # the mean-NLL collective is off the critical path: the engine writes each step's sum log p into a
    # ring slot; one asynchronous all-reduce per bank of 32 steps runs on a side stream
    ring = NllRing(dev, slots=32)

    def step(i: int):
        d = flow(cs[i % NBUF])
        return d.log_prob_and_sum(xs[i % NBUF], sum_out=ring.slot(B))

    with torch.no_grad():
        # ---- parity of the bench workload against the oracle (small slice, outside timing)
        parity = None
        if rank == 0:
            from oracle import oracle

            spec = oracle.flowspec_from_module(build_model())
            n = 2048
            ours = flow(cs[0][:n]).log_prob(xs[0][:n]).cpu().numpy().astype(np.float64)
            ref = spec.log_prob(xs_host[0][:n].numpy(), cs_host[0][:n].numpy())
            parity = {"rows": n, "max_rel_err_vs_fp64_oracle": float(np.max(np.abs(ours - ref) / np.maximum(np.abs(ref), 1.0)))}

        clk = ClockSampler(local).prepare()
        # warm-up: at least W (>= 3) steps and never fewer than 50 (~0.25 s; the same count on every
        # rank — each step holds a collective), so that clocks / power state have settled and every
        # lazy initialisation (allocator, NVML, module loading) is behind us
        warm_steps = max(args.warmup, 3, 50)
        for i in range(warm_steps):
            step(i)
        ring.means()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches0 = E.lib().zk_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with clk:
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.steps):
                lp, lp_sum = step(i)
            nll_means = ring.means()  # waits for the outstanding mean-NLL collectives: inside the timed region
            e1.record()
            torch.cuda.synchronize()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"log_prob": lp, "log_prob_sum": lp_sum, "mean_nll": nll_means[-1:]})
        if world > 1:
            dist.barrier()
        elapsed_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
        launches = E.lib().zk_launch_count() - launches0
        ms_per_step = elapsed_ms.item() / args.steps
        value = world * B / (ms_per_step * 1e-3)
        nll_value = float(nll_means[-1].item())

        # ---- end to end through the public API with HOST buffers (H2D + compute + D2H per step)
        fc = flow(cs[0])._flow_call()[0]
        out_host = torch.empty(B, dtype=torch.float32).pin_memory()
        e2e_steps = max(2, min(args.steps, 10))
        for i in range(2):
            fc.log_prob_host(xs_host[i % NBUF], cs_host[i % NBUF], dev, out_host)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            _, tot = fc.log_prob_host(xs_host[i % NBUF], cs_host[i % NBUF], dev, out_host)  # synchronous
        e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = world * B / e2e_s.item()

        # ---- training step (forward + backward through the autograd seam), rank 0, 2^18 rows
        # (auxiliary measurements must never cost the headline line: failures are reported inside it)
        training = None
        if rank == 0 and not args.no_training_step:
            try:
                training = time_training_step(flow, xs[0], cs[0], rows=min(B, 1 << 18), iters=3)
            except Exception as e:  # noqa: BLE001
                training = {"error": f"{type(e).__name__}: {e}"[:300]}

        # ---- per-kernel timing in isolation (CUDA events), rank 0
        kernels, roofline = [], None
        peak_tf, peak_kind = tensor_peak(peaks, clk.summary())
        if rank == 0:
            try:
                kernels = time_kernels(flow, xs[0], cs[0], dev, peaks, iters=max(3, min(args.steps, 10)), peak_tf=peak_tf, peak_kind=peak_kind)
                dom = max((k for k in kernels if k["in_step"]), key=lambda k: k["ms_per_step"])
                roofline = {k: dom[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
                roofline["kernel"] = dom["name"]
                roofline["peak_source"] = peaks["source"]
                roofline["peak_kind"] = dom.get("peak_kind")
                if dom.get("bound") == "tensor":
                    roofline["peak_sustained"] = peaks["bf16_tflops_sustained"]
                roofline["traffic_captured_at"] = dom.get("traffic_captured_at")
            except Exception as e:  # noqa: BLE001
                kernels, roofline = [], {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- the other BASELINE configurations: N = 1 all three, N > 1 the north-star config (cfg5) on every rank
    configs = []
    if not args.no_configs:
        del xs, cs
        torch.cuda.empty_cache()
        for cfg in OTHER_CONFIGS:
            if world > 1 and cfg["name"] != "cfg5":
                continue
            try:
                r = time_config(cfg, dev, rank, world, peaks, steps=max(3, min(args.steps, 10)), nvml=getattr(clk, "_nvml", None))
            except Exception as e:  # noqa: BLE001
                r = {"name": cfg["name"], "workload": cfg["workload"], "error": f"{type(e).__name__}: {e}"[:300]}
                if world > 1:
                    raise
            configs.append(r)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                rows = args.cpu_rows or CPU_ROWS
                cpu_reference_rate(min(rows, 1 << 16))  # warm-up
                rate, sec, threads = cpu_reference_rate(rows, repeats=3)
                cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "host": usable_cores(),
                       "sample": f"{rows} rows of the workload, oracle fp32 C port with OpenMP (threads pinned), best of 3, {sec:.1f} s"}  # fmt: skip
            except Exception as e:  # noqa: BLE001
                cpu = {"error": f"{type(e).__name__}: {e}"[:300]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "warmup_steps_run": warm_steps,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (conditioner GEMMs: %s)" % gemm_mode_name(flow), "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": B * world,
                       "parallelism": f"dp{world}", "l2": f"inputs rotate over {NBUF} buffers ({NBUF * B * (D + C) * 4 >> 20} MB > 126 MB L2)"},
            "clocks": clk.summary(), "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * (D + C) * 4, "d2h_bytes_per_step": B * 4,
                                             "steps": e2e_steps, "api": "FlowCall.log_prob_host -> zk_flow_log_prob_host (pinned host buffers)"},
            "gpu_launches": int(launches), "mean_nll": nll_value, "roofline": roofline, "kernels": kernels,
            "cpu_baseline": cpu, "parity": parity, "training_step": training, "configs": configs,
        }  # fmt: skip
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 15 << 20  # 60 MiB of float32 log-densities: a dump stays under 64 MB


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Writes what the last timed step returned (rank 0) as out_dir/<name>.npy, in the dtype it was
    computed in (float32 / float64), so that two builds can be compared output for output on the same
    seeded inputs.  Of a batch over DUMP_ROWS rows, a fixed, seeded sample of DUMP_ROWS rows is kept
    (the same rows in every run with the same --batch)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        if a.shape[0] > DUMP_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))]
        np.save(out / f"{name}.npy", a)


def time_training_step(flow, x, c, rows: int, iters: int) -> dict:
    """One REAL training step (README.md:43-49 of the reference) on `rows` rows, CUDA events:
    `loss = -flow(c).log_prob(x).mean(); loss.backward(); optimizer.step()` — the optimizer step is
    inside the timed region, so every iteration pays the refresh of the packed weights
    (zk_layer_update_weights: split kernels only) that the new parameter versions trigger."""
    import copy

    from zuko_b200 import _engine as E

    x, c = x[:rows], c[:rows]
    model = copy.deepcopy(flow).train()  # the timed steps must not move the weights the other measurements use
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)

    def one():
        opt.zero_grad(set_to_none=True)
        (-model(c).log_prob(x).mean()).backward()
        opt.step()

    with torch.enable_grad():
        for _ in range(3):
            one()
        n0 = E.lib().zk_launch_count()
        ms = cuda_time_ms(one, iters)
        launches = (E.lib().zk_launch_count() - n0) / iters
    dims = [D + C, *H, D * P]
    flops = 2.0 * sum(a * b for a, b in zip(dims[:-1], dims[1:])) * rows * T
    return {"workload": WORKLOAD.replace("log_prob", "training step (log_prob forward + backward + Adam step)"), "rows": rows,
            "ms_per_step": ms, "samples_per_s": rows / (ms * 1e-3), "gpu_launches_per_step": launches,
            "algorithmic_tflops": 4 * flops / (ms * 1e-3) / 1e12, "optimizer_step_in_timed_region": True,
            "note": "forward + recompute + dgrad + wgrad = 4 x the dense conditioner FLOPs; backward GEMMs on linear_tc_kernel (tcgen05 split-bf16); "
                    "gpu_launches_per_step counts engine kernels only (Adam's own kernels are torch's)"}  # fmt: skip


def gemm_mode_name(flow) -> str:
    from zuko_b200 import _engine as E

    h = flow.transform.transforms[0].hyper._handle()
    return {E.ZK_GEMM_FP32: "fp32 FMA", E.ZK_GEMM_BF16X3: "tcgen05 bf16x3, fp32 accumulate", E.ZK_GEMM_BF16X1: "tcgen05 bf16"}.get(E.lib().zk_mlp_gemm_mode(h), "?")


def ncu_traffic() -> dict:
    f = ROOT / "profiles" / "ncu_traffic.json"
    return json.loads(f.read_text()) if f.exists() else {}


def time_kernels(flow, x, c, dev, peaks, iters: int, peak_tf: float | None = None, peak_kind: str = "sustained") -> list[dict]:
    """Times each kernel class of one flow layer in isolation through the C-ABI entry points
    (CUDA events on the current stream) and converts to roofline terms.  Algorithmic bytes /
    FLOPs per SURVEY §8d; a step launches each of them T = 4 times (once per flow layer)."""
    from zuko_b200 import _engine as E

    L = E.lib()
    B = x.shape[0]
    layer = flow.transform.transforms[0]
    hyper = layer.hyper
    h = hyper._handle()
    hl = layer._zk_layer()
    phi = torch.empty(B, D * P, device=dev)
    y = torch.empty_like(x)
    ladj = torch.zeros(B, device=dev)
    need = max(L.zk_mlp_workspace_bytes(h, B), L.zk_layer_workspace_bytes(hl, B), 1)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    st = E.stream_ptr(dev)

    def mlp():
        E.check(L.zk_mlp_forward(h, x.data_ptr(), D, D, c.data_ptr(), C, C, B, phi.data_ptr(), D * P, ws.data_ptr(), ws.numel(), st))

    def rqs():
        E.check(L.zk_rqs_forward(x.data_ptr(), D, phi.data_ptr(), D * P, B, D, K, 5.0, 1e-3, y.data_ptr(), D, ladj.data_ptr(), 1, st))

    def fused():
        E.check(L.zk_layer_forward(hl, x.data_ptr(), D, c.data_ptr(), C, B, y.data_ptr(), D, ladj.data_ptr(), 1, ws.data_ptr(), ws.numel(), st))


    dims = [D + C, *H, D * P]
    flops = 2.0 * sum(a * b for a, b in zip(dims[:-1], dims[1:])) * B  # dense FLOPs nn.py:218 executes
    rqs_bytes = 4.0 * (D + D * P + D + 1) * B  # SURVEY §8d: x + phi + y + ladj
    fused_bytes = 4.0 * (D + C + D + 1) * B    # fused layer: x, c in; y, ladj out
    out = []
    traffic = ncu_traffic()
    peak_tf = peak_tf or peaks["bf16_tflops_sustained"]
    info = fused_info(flow)
    issued = 2.0 * info["issued_macs_per_row"] / T * B  # one flow layer, from the pack's tile table
    fused_name = {"fused_wide_kernel": "fused_wide_kernel<RQS,8> (CTA pairs, cta_group::2)",
                  "fused_dual_kernel": "fused_dual_kernel<RQS,8> (CTA pairs, two sub-tiles in flight)"}.get(info["kernel"][0], "fused_layer_kernel<RQS,8>")
    n0 = L.zk_launch_count()
    fused()
    is_fused = (L.zk_launch_count() - n0) == 1
    if is_fused:
        fused()
        t = cuda_time_ms(fused, iters)
        tf = flops / (t * 1e-3) / 1e12
        out.append({"name": fused_name + " (conditioner 24-256-256-256-368 on tcgen05 + RQS + ladj), one flow layer",
                    "bound": "tensor", "achieved": tf, "peak": peak_tf, "peak_kind": peak_kind, "unit": "TFLOP/s",
                    "frac": tf / peak_tf, "traffic": traffic.get(info["kernel"][0] + "_cfg2", traffic.get("fused_layer_kernel") if info["kernel"][0] == "fused_layer_kernel" else None), "traffic_captured_at": traffic.get("git_sha"),
                    "ms_per_launch": t, "ms_per_step": t * T,
                    "algorithmic_flops": flops, "issued_flops": issued, "frac_issued": issued / (t * 1e-3) / 1e12 / peak_tf,
                    "algorithmic_hbm_bytes": fused_bytes, "in_step": True})  # fmt: skip
    prev = L.zk_set_fused_layers(0)
    try:
        for _ in range(2):
            mlp()
            rqs()
        t_mlp = cuda_time_ms(mlp, iters)
        t_rqs = cuda_time_ms(rqs, iters)
    finally:
        L.zk_set_fused_layers(prev)
    tf = flops / (t_mlp * 1e-3) / 1e12
    gbs = rqs_bytes / (t_rqs * 1e-3) / 1e9
    out += [
        {"name": "unfused conditioner: split_input + 4 x linear_tc_kernel (24-256-256-256-368), one flow layer", "bound": "tensor",
         "achieved": tf, "peak": peak_tf, "peak_kind": peak_kind, "unit": "TFLOP/s", "frac": tf / peak_tf,
         "traffic": traffic.get("linear_tc_kernel_stack"), "traffic_captured_at": traffic.get("git_sha"), "ms_per_launch": t_mlp, "ms_per_step": t_mlp * T, "algorithmic_flops": flops, "in_step": not is_fused},
        {"name": "uni_kernel<RQS,8> stand-alone fused RQS + ladj (phi in HBM), one flow layer", "bound": "hbm", "achieved": gbs,
         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": traffic.get("uni_kernel"),
         "traffic_captured_at": traffic.get("git_sha"), "ms_per_launch": t_rqs,
         "ms_per_step": t_rqs * T, "algorithmic_bytes": rqs_bytes, "in_step": not is_fused},
    ]  # fmt: skip
    # the HBM-roofline kernel at the cfg5 shape (D = 64, K = 16: 12 548 B per sample, SURVEY §8d)
    try:
        D5, K5, B5 = 64, 16, 1 << 19
        P5 = 3 * K5 - 1
        x5 = torch.randn(B5, D5, device=dev)
        phi5 = torch.randn(B5, D5 * P5, device=dev)
        y5 = torch.empty_like(x5)
        l5 = torch.zeros(B5, device=dev)

        def rqs5():
            E.check(L.zk_rqs_forward(x5.data_ptr(), D5, phi5.data_ptr(), D5 * P5, B5, D5, K5, 5.0, 1e-3, y5.data_ptr(), D5, l5.data_ptr(), 1, st))

        rqs5()
        t5 = cuda_time_ms(rqs5, iters)
        b5 = 4.0 * (D5 + D5 * P5 + D5 + 1) * B5
        g5 = b5 / (t5 * 1e-3) / 1e9
        out.append({"name": "uni_kernel<RQS,16> stand-alone fused RQS + ladj at the cfg5 shape (D = 64, K = 16, 2^19 rows, phi in HBM)", "bound": "hbm",
                    "achieved": g5, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": g5 / peaks["hbm_gbs"], "traffic": traffic.get("uni_kernel_rqs16"),
                    "traffic_captured_at": traffic.get("git_sha"), "ms_per_launch": t5, "ms_per_step": 0.0, "algorithmic_bytes": b5, "in_step": False})  # fmt: skip
        del x5, phi5, y5, l5
    except Exception as e:  # noqa: BLE001
        out.append({"name": "uni_kernel<RQS,16> (cfg5 shape)", "error": f"{type(e).__name__}: {e}"[:200], "in_step": False, "ms_per_step": 0.0})
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=1 << 20, help="rows per GPU")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the bounded CPU sample (0 = 2^19)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-training-step", action="store_true", help="skip the forward+backward timing (extra object)")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg3 / cfg4 / cfg5 entries of the line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the engine arm; the reference arm keeps none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

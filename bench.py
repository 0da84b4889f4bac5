#!/usr/bin/env python
"""bench.py -- headline benchmark of the newsched data-parallel block hot path on B200.

Workload (BASELINE.json configs[1], the configuration the metric is quoted on):
    null_source -> fft(N=4096, Blackman-Harris window) -> complex_to_mag -> null_sink,
    1 GiB synthetic complex64 stream (32768 vectors) PER GPU, run as ONE fused kernel launch
    per step (window + FFT + |.|).  A "step" is one pass over that stream.
`value`    = whole-job Msamples/s with the stream already resident in HBM (CUDA events, max
             over ranks).
`e2e`      = the same metric through the C-ABI host-buffer call (b200_chain_run_host): pinned
             host input -> H2D -> kernel -> D2H -> pinned host output, copies inside the region.
`roofline` = algorithmic 12 B/sample (8 in + 4 out) x samples per launch / launch duration
             against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
`extras`   = config 1 (fir_filter_ccf, 64 taps, 16 Mi samples) and the other blocks, each with
             its own roofline, for the record.
`--impl reference` times the CPU restatement (oracle/, OpenMP over all host threads) of the same
workload: the reference snapshot has no FFT/FIR block and cannot be built here (DESIGN.md 3).
`--dump-outputs DIR` writes what the timed path computed in its last step, so that two builds can be
compared output for output on the same seeded input: DIR/fft4096_window_mag.npy, float32, the
|FFT| of DUMP_VECTORS of the 32768 vectors (rank 0), picked by a fixed seed.

Multi-GPU: independent per-GPU streams (the path shards by stream / time segment), no
data-path collective; `scaling` = weak.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FFT = 4096
N_VEC = 32768                       # 32768 x 4096 complex64 = 1 GiB
SAMPLES = N_FFT * N_VEC
DUMP_VECTORS = 2048                 # 2048 x 4096 float32 = 32 MiB written by --dump-outputs
METRIC = "Msamples/s FIR-ccf & FFT-4096 flowgraph at 1/2/4/8 B200; % of HBM/FP32 roofline"
CONFIG = {
    "workload": "configs[1]: null_source -> fft(N=4096, Blackman-Harris) -> complex_to_mag -> null_sink, "
                "1 GiB synthetic complex64 stream per GPU (32768 vectors), one fused window+FFT+|.| launch per step",
    "samples_per_gpu_per_step": SAMPLES,
    "l2": "inputs (1 GiB in, 0.5 GiB out per step) are larger than the 126 MB L2; no flush needed",
    "parallelism": "one independent stream per GPU (stream / time-segment sharding), no data-path collective",
}


def blackman_harris(n):
    import numpy as np
    t = np.arange(n, dtype=np.float64) / (n - 1)
    return (0.35875 - 0.48829 * np.cos(2 * np.pi * t) + 0.14128 * np.cos(4 * np.pi * t)
            - 0.01168 * np.cos(6 * np.pi * t)).astype(np.float32)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", d
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", {}


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, torch_dev):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self._nv = pynvml
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(torch_dev).uuid)
                self._h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[torch_dev]) if vis else torch_dev
                self._h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self._err = repr(e)
            self._h = None
        self._t = None

    _NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap",
              0x8: "hw_slowdown", 0x10: "sync_boost", 0x20: "sw_thermal_slowdown",
              0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for bit, name in self._NAMES.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def sample_now(self, n=3):
        """A few synchronous samples from the caller's thread (the timed region of a fast kernel can be
        shorter than the background thread's period)."""
        if self._h is None:
            return
        nv = self._nv
        for _ in range(n):
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for bit, name in self._NAMES.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass

    def start(self):
        if self._h is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                    "note": "no NVML samples"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "n_samples": len(self.samples)}


def gpu_numa_cpus(torch, dev_index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None."""
    try:
        p = torch.cuda.get_device_properties(dev_index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None, node
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return cpus, node
    except Exception:
        return None, None


class PinnedHost:
    """Page-locked host buffer from the C-ABI (b200_host_alloc), first-touched while the process is bound to
    the GPU's NUMA node so its pages are local to the PCIe root the copies go through."""

    def __init__(self, torch, nb, nbytes, dtype, dev_index):
        import ctypes as C
        self.nb, self.ptr = nb, C.c_void_p()
        cpus, self.node = gpu_numa_cpus(torch, dev_index)
        old = None
        try:
            if cpus:
                old = os.sched_getaffinity(0)
                allowed = cpus & old
                if allowed:
                    os.sched_setaffinity(0, allowed)
            nb._check(nb.lib().b200_host_alloc(C.byref(self.ptr), nbytes))
            buf = (C.c_byte * nbytes).from_address(self.ptr.value)
            self.tensor = torch.frombuffer(buf, dtype=dtype)
            self.tensor.zero_()                                   # first touch here, on the local node
        finally:
            if old is not None:
                os.sched_setaffinity(0, old)

    def free(self):
        if self.ptr:
            self.tensor = None
            self.nb.lib().b200_host_free(self.ptr)
            self.ptr = None


def dist_env():
    return (int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)),
            int(os.environ.get("WORLD_SIZE", 1)))


def fir_executed(T, D, algo):
    """Work the selected FIR kernel EXECUTES per input sample (not the direct-form algorithmic count), and the
    pipe it runs on: algorithm 1 = direct FFMA2 form, 2 = block-Toeplitz GEMM on tcgen05 (bf16 hi/lo, four
    partial products), 3 = overlap-save (4096-point transforms, 5 N log2 N flop each plus the spectrum product)."""
    if algo == 1:
        return 4.0 * T / D, "fp32"
    if algo == 2:
        tq = -(-T // D)
        ksteps = ((tq - 1 + 15) // 16 * 16 + 64) // 16
        tile = 4096 if (D == 1 and ksteps * 16 <= 512) else 8192       # outputs per tile (tap-stationary / ring form)
        mma = 2 * 128 * (tile // 64) * 16                             # one 128 x (tile/64) x 16 MMA
        return D * ksteps * 4 * mma / (tile * D), "tensor"
    if algo == 3:
        fft = 5 * 4096 * 12 + 6 * 4096
        if D == 1 and T < 1024:
            return 2 * fft / (4096 - (T - 1)), "fp32"
        if D == 1:
            return 4 * fft / (2 * (4095 - -(-T // 2))), "fp32"
        return (D + 1) * fft / ((4096 - -(-T // D)) * D), "fp32"
    return float("nan"), "fp32"


def fir_record(gs, T, D, algo, peak_gbs, fp32_tf, bf16_tf, ms):
    """One FIR measurement as a roofline record: HBM fraction from the ALGORITHMIC bytes (8 + 8/D per input
    sample), and the executed-work fraction of the pipe the kernel runs on."""
    flop, pipe = fir_executed(T, D, algo)
    bps = 8 + 8.0 / D
    rec = {"algorithm": algo, "Msamples_s": gs * 1e3, "ms": ms, "bound": "hbm", "unit": "GB/s",
           "achieved": gs * bps, "peak": peak_gbs, "frac": gs * bps / peak_gbs,
           "algorithmic_bytes_per_sample": bps, "executed_flop_per_sample": flop,
           "executed_tflops": gs * flop / 1e3, "executed_on": pipe}
    if pipe == "tensor" and bf16_tf:
        rec["executed_frac_of_measured_bf16_peak"] = gs * flop / 1e3 / bf16_tf
    elif fp32_tf:
        rec["executed_frac_of_measured_fp32_peak"] = gs * flop / 1e3 / fp32_tf
    return rec


# ---------------------------------------------------------------------------------------------
def cpu_fft_mag_rate(steps, warmup, target_s=0.5):
    """Times the oracle's fp32 FFT+|.| (OpenMP, all host threads) on a bounded sample."""
    import numpy as np
    import oracle as o
    try:   # torchrun exports OMP_NUM_THREADS=1; the CPU arm must use every host core it may run on
        o.set_num_threads(len(os.sched_getaffinity(0)))
    except Exception:
        o.set_num_threads(os.cpu_count() or 1)
    w = blackman_harris(N_FFT)
    rng = np.random.default_rng(0x5EED)
    nv = 256
    x = (rng.uniform(-1, 1, nv * N_FFT) + 1j * rng.uniform(-1, 1, nv * N_FFT)).astype(np.complex64)
    o.fft(x, N_FFT, True, w, precise=False, mag=True, mt=True)            # thread pool up
    t0 = time.perf_counter()
    o.fft(x, N_FFT, True, w, precise=False, mag=True, mt=True)
    rate = x.size / (time.perf_counter() - t0)
    nv_step = int(min(N_VEC, max(256, 2 ** int(np.log2(max(rate * target_s / N_FFT, 256))))))
    x = np.tile(x, nv_step // nv + 1)[: nv_step * N_FFT]
    for _ in range(warmup):
        o.fft(x, N_FFT, True, w, precise=False, mag=True, mt=True)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.fft(x, N_FFT, True, w, precise=False, mag=True, mt=True)
    dt = time.perf_counter() - t0
    return {
        "value": x.size * steps / dt / 1e6, "unit": "Msamples/s", "cores": o.num_threads(),
        "kind": "port",
        "sample": f"{nv_step} vectors x {N_FFT} complex64 ({x.nbytes >> 20} MiB) per step, {steps} steps; "
                  "oracle.c fp32 radix-4 Stockham + window + |.|, OpenMP static over vectors "
                  "(CPU restatement, not VOLK/FFTW: the reference snapshot has no FFT block)",
        "ms_per_step": dt / steps * 1e3,
    }


def cpu_fft_mag_rate_tuned(steps=3, nv=2048):
    """The same workload through a tuned CPU library, for scale: scipy.fft (pocketfft, complex64 in / out,
    workers = all host threads) + window + |.|.  Labelled as such; the reference arm itself stays the C port."""
    import numpy as np
    try:
        import scipy.fft as sfft
    except Exception as e:  # pragma: no cover
        return {"value": None, "error": repr(e)}
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    w = blackman_harris(N_FFT)
    rng = np.random.default_rng(0x5EED)
    x = (rng.uniform(-1, 1, (nv, N_FFT)) + 1j * rng.uniform(-1, 1, (nv, N_FFT))).astype(np.complex64)
    np.abs(sfft.fft(x * w, axis=1, workers=cores))
    t0 = time.perf_counter()
    for _ in range(steps):
        np.abs(sfft.fft(x * w, axis=1, workers=cores))
    dt = time.perf_counter() - t0
    return {"value": x.size * steps / dt / 1e6, "unit": "Msamples/s", "cores": cores, "kind": "tuned library",
            "sample": f"{nv} vectors x {N_FFT} complex64 x {steps}: numpy window multiply + scipy.fft.fft(workers={cores}) "
                      "(pocketfft, single precision) + numpy abs"}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    steps = args.steps
    cb = cpu_fft_mag_rate(steps, max(0, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "cpu_tuned_library": cpu_fft_mag_rate_tuned(),
        "e2e": {"value": cb["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------
def timed(torch, fn, steps, warmup, barrier, during=None):
    """W warm-ups, then exactly `steps` calls between CUDA events on the current stream.  `during`
    runs on the host after everything (closing event included) has been enqueued and before the
    synchronize, i.e. while the GPU is still inside the timed region."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    if during is not None:
        during()
    torch.cuda.synchronize()
    barrier()
    return e0.elapsed_time(e1)


def run_b200(args):
    import numpy as np
    import torch

    import newsched_b200 as nb

    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    nb.lib()
    steps, warmup = args.steps, max(3, args.warmup)
    peak_gbs, peak_src, peaks = measured_peaks()
    w = blackman_harris(N_FFT)

    # ---- synthetic stream, resident in HBM (uniform[-1,1) complex64, seed 0x5EED + rank)
    g = torch.Generator(device=dev).manual_seed(0x5EED + rank)
    x = torch.view_as_complex(torch.rand(SAMPLES, 2, device=dev, generator=g) * 2 - 1)
    out = torch.empty(SAMPLES, dtype=torch.float32, device=dev)
    fft = nb.FFT(N_FFT, True, w, output=nb.OUT_MAG)

    sampler = ClockSampler(local_rank)
    l0 = nb.launch_count()
    for _ in range(warmup):
        fft.work(x, out)
    torch.cuda.synchronize()
    l_warm = nb.launch_count()
    sampler.start()
    ms = timed(torch, lambda: fft.work(x, out), steps, 0, barrier, during=sampler.sample_now)
    sampler.stop()
    launches = nb.launch_count() - l_warm
    if args.dump_outputs and rank == 0:
        # before anything else reuses `out`
        rows = np.sort(np.random.default_rng(0).choice(N_VEC, DUMP_VECTORS, replace=False))
        sample = out.view(N_VEC, N_FFT)[torch.from_numpy(rows).to(dev)].cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "fft4096_window_mag.npy"), sample)
        del sample
    ms = max_over_ranks(ms)
    value = world * SAMPLES * steps / (ms * 1e-3) / 1e6
    k_ms = ms / steps                                   # one launch per step
    achieved = 12.0 * SAMPLES / (k_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": None,
                "kernel": "fft4096_tma_kernel<fwd, mag> (TMA prefetch + window + 3x radix-16 + |.|)",
                "algorithmic_bytes_per_sample": 12, "peak_source": peak_src,
                "launch_ms": k_ms}
    # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel, stamped with the commit
    # the capture was taken at (newest file wins)
    for tf in ("r02_fft4096_traffic.json", "r01_fft4096_traffic.json"):
        traffic_file = os.path.join(ROOT, "profiles", tf)
        if os.path.exists(traffic_file):
            try:
                tj = json.load(open(traffic_file))
                roofline["traffic"] = tj.get("dram_bytes_per_launch")
                roofline["traffic_source"] = {"file": "profiles/" + tf, "captured_at_commit": tj.get("commit"),
                                              "kernel_ms_under_ncu": tj.get("kernel_ms_under_ncu")}
                break
            except Exception:
                pass

    # ---- e2e: host buffers through the C-ABI streaming call
    e2e = None
    try:
        chunk = N_FFT * 512                             # 16 MiB in / 8 MiB out per chunk (measured best of 16/64/256:
        # the pipeline runs at the box's bidirectional PCIe limit, 76-78 GB/s of 75.8 measured with plain copies)
        chain = nb.Chain([fft], in_item_bytes=8, chunk_items=chunk)
        phx = PinnedHost(torch, nb, SAMPLES * 8, torch.complex64, local_rank)
        phy = PinnedHost(torch, nb, SAMPLES * 4, torch.float32, local_rank)
        hx, hy = phx.tensor, phy.tensor
        hx.copy_(x)
        e_steps = max(1, min(steps, 10))
        for _ in range(2):
            chain.run_host(hx, hy)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            chain.run_host(hx, hy)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt = max_over_ranks(dt)
        ok = bool(torch.equal(hy[-N_FFT:], out[-N_FFT:].cpu()))
        e2e = {"value": world * SAMPLES * e_steps / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": SAMPLES * 8, "d2h_bytes_per_step": SAMPLES * 4,
               "steps": e_steps, "ms_per_step": dt / e_steps * 1e3, "matches_device_run": ok,
               "api": "b200_chain_run_host (pinned host in/out, 3-stream H2D/compute/D2H overlap)",
               "pcie_gbs": (SAMPLES * 12 * e_steps) / dt / 1e9,
               "host_buffers": f"b200_host_alloc, first touch bound to the GPU's NUMA node (node {phx.node})"}
        # the box's own ceiling for this traffic pattern: the same bytes as plain page-locked copies, H2D and D2H
        # concurrently on two streams, every rank at once, no kernel -- what the PCIe / host-memory fabric gives
        try:
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
            xin = torch.empty_like(x)

            def copies():
                with torch.cuda.stream(s_in):
                    xin.copy_(hx, non_blocking=True)
                with torch.cuda.stream(s_out):
                    hy.copy_(out, non_blocking=True)
            copies()
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                copies()
            torch.cuda.synchronize()
            dtc = time.perf_counter() - t0
            barrier()
            dtc = max_over_ranks(dtc) / 3
            e2e["ceiling"] = {"value": world * SAMPLES / dtc / 1e6, "unit": "Msamples/s", "pcie_gbs_per_gpu": SAMPLES * 12 / dtc / 1e9,
                              "what": "1 GiB H2D + 0.5 GiB D2H as plain cudaMemcpyAsync on two streams, all ranks concurrently, no kernel"}
            e2e["frac_of_ceiling"] = e2e["value"] / e2e["ceiling"]["value"]
            del xin
        except Exception as e:  # pragma: no cover
            e2e["ceiling_error"] = repr(e)
        del hx, hy, chain
        phx.free()
        phy.free()
    except Exception as e:  # pragma: no cover
        e2e = {"value": None, "unit": "Msamples/s", "error": repr(e)}

    # ---- extras: the other configs / blocks, each with its own roofline (rank 0 reports)
    extras = {}
    try:
        n1 = 1 << 24                                   # config 1: 16 Mi samples, 64 taps
        x1 = x[:n1]
        y1 = torch.empty(n1, dtype=torch.complex64, device=dev)
        rng = np.random.default_rng(1)
        fp32_tf, _ = nb.measure_fp32_tflops(8192)
        fp32_tf, _ = nb.measure_fp32_tflops(8192)
        bf16_tf = float(peaks.get("bf16_tflops", 0) or 0)
        for T in (64, 128, 256, 512, 1024):
            taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
            fir = nb.FirFilter(taps, 1)
            reps = max(3, min(steps, 20 if T <= 256 else 5))
            t = timed(torch, lambda: fir.work_segment(x1, None, y1), reps, 3, lambda: None) / reps
            extras[f"fir_ccf_{T}taps_16Mi"] = fir_record(n1 / (t * 1e-3) / 1e9, T, 1, fir.algorithm, peak_gbs, fp32_tf,
                                                         bf16_tf, t)
        # config 1's 64 taps through the SIMT direct form, for the A/B against the tensor-core form above
        taps64 = (rng.uniform(-1, 1, 64) / 64).astype(np.float32)
        fir = nb.FirFilter(taps64, 1, algorithm=1)
        t = timed(torch, lambda: fir.work_segment(x1, None, y1), 10, 3, lambda: None) / 10
        extras["fir_ccf_64taps_16Mi_simt_direct"] = fir_record(n1 / (t * 1e-3) / 1e9, 64, 1, 1, peak_gbs, fp32_tf, bf16_tf, t)
        # the same 64-tap kernel on the whole 1 GiB stream (a 16 Mi-sample call is ~50 us, a few of them ramp and tail)
        fir = nb.FirFilter(taps64, 1)
        y1b = torch.empty(SAMPLES, dtype=torch.complex64, device=dev)
        t = timed(torch, lambda: fir.work_segment(x, None, y1b), 5, 2, lambda: None) / 5
        extras["fir_ccf_64taps_128Mi"] = fir_record(SAMPLES / (t * 1e-3) / 1e9, 64, 1, fir.algorithm, peak_gbs, fp32_tf,
                                                    bf16_tf, t)
        del y1b
        # fir_filter_fff (float stream, 8 B per sample): 64 / 256 taps on the tensor cores (two 4096-sample runs per
        # tile ride through the two planes of the complex kernel), the SIMT form beside it
        xr = torch.view_as_real(x).reshape(-1)[:SAMPLES]
        yr = torch.empty(SAMPLES, dtype=torch.float32, device=dev)
        for Tr, algo_r in ((64, 0), (64, 1), (256, 0)):
            tr = (rng.uniform(-1, 1, Tr) / Tr).astype(np.float32)
            fir = nb.FirFilter(tr, 1, is_complex=False, algorithm=algo_r)
            t = timed(torch, lambda: fir.work_segment(xr, None, yr), 5, 2, lambda: None) / 5
            grs = SAMPLES / (t * 1e-3) / 1e9
            extras[f"fir_fff_{Tr}taps_128Mi" + ("_simt_direct" if algo_r == 1 else "")] = {
                "algorithm": fir.algorithm, "Mreal_samples_s": grs * 1e3, "ms": t, "bound": "hbm", "unit": "GB/s",
                "achieved": grs * 8, "peak": peak_gbs, "frac": grs * 8 / peak_gbs, "algorithmic_bytes_per_sample": 8}
        del yr
        # short decimating filters run folded into the TMA-staged SIMT kernel: HBM-bound (10 B per input at D = 4)
        for Td, Dd in ((32, 4), (64, 4), (64, 8)):
            taps = (rng.uniform(-1, 1, Td) / Td).astype(np.float32)
            fir = nb.FirFilter(taps, Dd)
            yd = torch.empty(SAMPLES // Dd, dtype=torch.complex64, device=dev)
            t = timed(torch, lambda: fir.work_segment(x, None, yd), 5, 2, lambda: None) / 5
            extras[f"fir_ccf_{Td}taps_decim{Dd}_128Mi"] = fir_record(SAMPLES / (t * 1e-3) / 1e9, Td, Dd, fir.algorithm,
                                                                     peak_gbs, fp32_tf, bf16_tf, t)
            del yd
        taps = (rng.uniform(-1, 1, 1024) / 1024).astype(np.float32)
        fir = nb.FirFilter(taps, 4, multiply_const=0.5 - 0.25j)
        n3 = 1 << 26
        y3 = torch.empty(n3 // 4, dtype=torch.complex64, device=dev)
        t = timed(torch, lambda: fir.work_segment(x[:n3], None, y3), 3, 2, lambda: None) / 3
        extras["fir_ccf_1024taps_decim4_mulc_64Mi"] = fir_record(n3 / (t * 1e-3) / 1e9, 1024, 4, fir.algorithm, peak_gbs,
                                                                 fp32_tf, bf16_tf, t)
        taps = (rng.uniform(-1, 1, 4096) / 4096).astype(np.float32)
        fir5 = nb.FirFilter(taps, 1)
        y5 = torch.empty(n3, dtype=torch.complex64, device=dev)
        t = timed(torch, lambda: fir5.work_segment(x[:n3], None, y5), 3, 2, lambda: None) / 3
        extras["fir_ccf_4096taps_64Mi"] = fir_record(n3 / (t * 1e-3) / 1e9, 4096, 1, fir5.algorithm, peak_gbs, fp32_tf,
                                                     bf16_tf, t)
        del y5
        extras["fp32_fma_tflops_measured"] = fp32_tf
        yc = torch.empty(SAMPLES, dtype=torch.complex64, device=dev)
        reps = max(3, min(steps, 20))
        for name, fn, bps in (
                ("copy_c64_1Gi", lambda: nb.copy(x, yc), 16),
                ("multiply_const_cc_1Gi", lambda: nb.multiply_const(x, 0.5 - 0.25j, yc), 16),
                ("complex_to_mag_1Gi", lambda: nb.complex_to_mag(x, False, out), 12)):
            t = timed(torch, fn, reps, 3, lambda: None) / reps
            gbs = SAMPLES * bps / (t * 1e-3) / 1e9
            extras[name] = {"Msamples_s": SAMPLES / (t * 1e-3) / 1e6, "ms": t, "hbm_gbs": gbs,
                            "frac_of_hbm": gbs / peak_gbs}
        fftc = nb.FFT(N_FFT, True, w)
        t = timed(torch, lambda: fftc.work(x, yc), reps, 3, lambda: None) / reps
        gbs = SAMPLES * 16 / (t * 1e-3) / 1e9
        extras["fft4096_window_complex_out_1Gi"] = {"Msamples_s": SAMPLES / (t * 1e-3) / 1e6, "ms": t,
                                                   "hbm_gbs": gbs, "frac_of_hbm": gbs / peak_gbs}
        import scipy.signal as sig
        pt = sig.firwin(64 * 16, 1.0 / 64).astype(np.float32)
        pfb = nb.PfbChannelizer(pt, 64)
        yp = yc.view(-1, 64)
        t = timed(torch, lambda: pfb.work_segment(x, None, yp), reps, 3, lambda: None) / reps
        gbs = SAMPLES * 16 / (t * 1e-3) / 1e9
        extras["pfb_channelizer_64ch_16tpc_1Gi"] = {"Msamples_s": SAMPLES / (t * 1e-3) / 1e6, "ms": t,
                                                   "hbm_gbs": gbs, "frac_of_hbm": gbs / peak_gbs,
                                                   "algorithm": pfb.algorithm, "form": "branch filters + 64-point DFT on the SIMT pipes"}
        # configs[3] as BASELINE words it ("filterbank + DFT as tensor-core GEMM"): the DFT across branches as a
        # bf16-split tcgen05 GEMM with the DFT matrix in tensor memory (algorithm 2), timed beside the SIMT form;
        # the library selects the faster one (DESIGN.md 4.4)
        pfb_tc = nb.PfbChannelizer(pt, 64, algorithm=2)
        ref_rows = yp[:4096].clone()
        t2 = timed(torch, lambda: pfb_tc.work_segment(x, None, yp), reps, 3, lambda: None) / reps
        torch.cuda.synchronize()
        d = (yp[:4096] - ref_rows).abs().double().pow(2).sum().sqrt() / ref_rows.abs().double().pow(2).sum().sqrt()
        gbs2 = SAMPLES * 16 / (t2 * 1e-3) / 1e9
        tc_flop = 3 * 2 * 128 * 128 / 64.0       # executed tensor flop per input sample: 3 split products of a 128 x 128 real DFT per 64-sample frame
        extras["pfb_channelizer_64ch_16tpc_1Gi_tensor_core_dft"] = {
            "Msamples_s": SAMPLES / (t2 * 1e-3) / 1e6, "ms": t2, "hbm_gbs": gbs2, "frac_of_hbm": gbs2 / peak_gbs,
            "algorithm": pfb_tc.algorithm, "form": "branch filters on the SIMT pipes, DFT across branches as a tcgen05 GEMM (A from TMEM)",
            "executed_tensor_tflops": tc_flop * SAMPLES / (t2 * 1e-3) / 1e12,
            "executed_frac_of_measured_bf16_peak": (tc_flop * SAMPLES / (t2 * 1e-3) / 1e12 / bf16_tf) if bf16_tf else None,
            "rel_rms_vs_simt_form": float(d), "selected_by_default": bool(pfb.algorithm == 2)}
        del yc, y1, y3
    except Exception as e:  # pragma: no cover
        extras["error"] = repr(e)

    # ---- the same configs as real flowgraphs: C++ blocks + device-resident edge buffers driven by
    # the thread-per-block scheduler, wall clock around start()/wait() like the reference's bm_*.cpp
    if world == 1 and rank == 0:
        try:
            import subprocess
            exe = os.path.join(ROOT, "newsched_b200", "host", "build", "bm_flowgraph")
            if not os.path.exists(exe):
                subprocess.check_call(["make", "-C", os.path.join(ROOT, "newsched_b200", "host"), "-s"])
            fgx = {}
            for name, argv in (
                    ("config2_fft4096_mag_8Gi_stream", ["--config", "2", "--samples", str(1 << 33), "--buffer_size", str(1 << 30)]),
                    ("config2_fft4096_mag_1Gi_stream", ["--config", "2", "--samples", str(1 << 30)]),
                    ("config2_unfused_fft_then_mag_1Gi", ["--config", "2", "--samples", str(1 << 30), "--fused", "0"]),
                    ("config1_fir_ccf_64taps_1Gi", ["--config", "1", "--samples", str(1 << 30)]),
                    ("config1_fir_ccf_64taps_8Gi_stream", ["--config", "1", "--samples", str(1 << 33), "--buffer_size", str(1 << 30)]),
                    ("config3_fir1024d4_mulc_fft_1Gi", ["--config", "3", "--samples", str(1 << 30)]),
                    ("config3_fir1024d4_mulc_fft_8Gi_stream", ["--config", "3", "--samples", str(1 << 33), "--buffer_size", str(1 << 30)]),
                    ("config4_pfb_channelizer_64ch_8Gi_stream", ["--config", "4", "--samples", str(1 << 33), "--buffer_size", str(1 << 30)]),
                    ("config4_pfb_channelizer_64ch_tensor_core_dft_8Gi_stream", ["--config", "4", "--fused", "2", "--samples", str(1 << 33), "--buffer_size", str(1 << 30)]),
                    ("config0_vector_source_fir64_vector_sink_16Mi", ["--config", "10", "--samples", str(1 << 24), "--buffer_size", str(1 << 25)]),
                    ("cuda_copy_x4_1Gi", ["--config", "0", "--samples", str(1 << 30)])):
                best = None
                for _ in range(3):
                    out = subprocess.run([exe] + argv, capture_output=True, text=True, timeout=120).stdout
                    rec = json.loads(out.strip().splitlines()[-1])
                    if best is None or rec["Msamples_s"] > best["Msamples_s"]:
                        best = rec
                fgx[name] = {k: best[k] for k in ("Msamples_s", "seconds", "kernel_launches", "buffer_size")}
            # the reference's own CPU-runnable case (configs[0]) beside it: the oracle's fp32 FIR on all host cores
            try:
                import oracle as o
                o.set_num_threads(len(os.sched_getaffinity(0)))
                rngc = np.random.default_rng(0)
                nc0 = 1 << 22
                xc0 = (rngc.uniform(-1, 1, nc0) + 1j * rngc.uniform(-1, 1, nc0)).astype(np.complex64)
                tc0 = np.full(64, 1.0 / 64, np.float32)
                o.fir(xc0, tc0, 1, precise=False, mt=True)
                t0 = time.perf_counter()
                for _ in range(3):
                    o.fir(xc0, tc0, 1, precise=False, mt=True)
                fgx["config0_cpu_oracle_fir64"] = {
                    "Msamples_s": 3 * nc0 / (time.perf_counter() - t0) / 1e6, "cores": o.num_threads(),
                    "sample": "4 Mi complex64 samples x 3, oracle.c fp32 64-tap FIR, OpenMP over outputs (kernel only, no scheduler)"}
            except Exception as e:  # pragma: no cover
                fgx["config0_cpu_oracle_error"] = repr(e)
            fgx["how"] = ("newsched_b200/host/bm_flowgraph: cuda::null_source -> blocks -> null_sink on D2D "
                          "device_buffer edges under scheduler_mt; wall clock start()->wait() of the second run in the process (a short "
                          "untimed run first loads the kernels' modules, which costs milliseconds once), best of 3")
            extras["flowgraph"] = fgx
        except Exception as e:  # pragma: no cover
            extras["flowgraph_error"] = repr(e)

    # ---- multi-GPU only: BASELINE config 5 (time-segmented FIR, 4096 taps, (ntaps-1) halo, NCCL gather) and
    # config 4 (64-channel channelizer, both partitions of SURVEY.md 8e).  Every rank owns one 2^27-sample
    # time segment.  The halo that precedes it is read IN PLACE from the left neighbour's buffer (PeerHalo:
    # CUDA IPC mapping + peer access, NVLink loads by the first blocks of the kernel), so a step is one
    # kernel launch; the NCCL point-to-point exchange it replaces is timed beside it.  Windows at the
    # start (where the halo matters) and the end of every rank's output are checked against the CPU oracle
    # on the same data; the trusted halo for that check comes from an all_gather, not from the path under test.
    if dist is not None:
        from newsched_b200 import multigpu as mg
        import oracle as o

        def gather_tails(n_tail):
            tails = [torch.empty(n_tail, dtype=torch.complex64, device=dev) for _ in range(world)]
            dist.all_gather([torch.view_as_real(t) for t in tails], torch.view_as_real(x[-n_tail:].contiguous()))
            return tails

        def all_max(v):
            return max_over_ranks(float(v))

        try:
            rng5 = np.random.default_rng(5)
            T5, W = 4096, 1024
            taps5 = (rng5.uniform(-1, 1, T5) / T5).astype(np.float32)
            fir5 = nb.FirFilter(taps5, 1)
            y5 = torch.empty(SAMPLES, dtype=torch.complex64, device=dev)
            sf_peer = mg.SegmentedFir(fir5, rank, world, peer=True)
            sf_p2p = mg.SegmentedFir(fir5, rank, world, peer=False)
            sf_peer.run(x, y5)                                   # collective set-up of the mapping
            t = max_over_ranks(timed(torch, lambda: sf_peer.run(x, y5), 5, 2, barrier) / 5)
            tails = gather_tails(T5 - 1)
            hist = tails[rank - 1].cpu().numpy() if rank > 0 else None
            e0 = o.rel_rms(y5[:W].cpu().numpy(), o.fir(x[:W].cpu().numpy(), taps5, 1, hist=hist))
            e1 = o.rel_rms(y5[-W:].cpu().numpy(), o.fir(x[-(W + T5 - 1):].cpu().numpy(), taps5, 1)[T5 - 1:])
            err5 = all_max(max(e0, e1))
            t_p2p = max_over_ranks(timed(torch, lambda: sf_p2p.run(x, y5), 5, 2, barrier) / 5)
            c5 = {"Msamples_s_outputs_sharded": world * SAMPLES / (t * 1e-3) / 1e6, "ms": t,
                  "halo": "read in place from the left neighbour over NVLink (peer-mapped pointer)",
                  "halo_bytes_per_rank": (T5 - 1) * 8, "algorithm": fir5.algorithm,
                  "ms_with_nccl_p2p_halo_exchange": t_p2p,
                  "parity_ok": bool(err5 < 1e-5), "rel_rms_vs_oracle": err5,
                  "parity_windows": f"first and last {W} outputs of every rank's segment vs oracle.fir (fp64), max over ranks"}
            full = mg.gather_concat(y5, rank, world, sizes=[SAMPLES] * world)   # warm-up (NCCL p2p setup)
            del full
            torch.cuda.synchronize()
            barrier()
            e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0_.record()
            full = mg.gather_concat(y5, rank, world, sizes=[SAMPLES] * world)
            e1_.record()
            torch.cuda.synchronize()
            tg = max_over_ranks(e0_.elapsed_time(e1_))
            c5["nccl_gather_ms"] = tg
            c5["Msamples_s_incl_gather"] = world * SAMPLES / ((t + tg) * 1e-3) / 1e6
            extras["config5_segmented_fir_4096taps"] = c5
            del full, y5
        except Exception as e:  # pragma: no cover
            extras["config5_error"] = repr(e)

        if 64 % world == 0:
            try:
                import scipy.signal as sig
                M, P, WF = 64, 16, 32
                pt = sig.firwin(M * P, 1 / M).astype(np.float32)
                cb, cc = mg.channel_slice(M, rank, world)
                pfb_c = nb.PfbChannelizer(pt, M, cb, cc)
                yc = torch.empty((SAMPLES // M, cc), dtype=torch.complex64, device=dev)
                t = max_over_ranks(timed(torch, lambda: pfb_c.work_segment(x, None, yc), 5, 2, barrier) / 5)
                # channel-sharded: zeros in front of the stream (no halo); first / last WF frames vs the oracle's columns
                ref0 = o.pfb_channelizer(x[:WF * M].cpu().numpy(), pt, M)[:, cb:cb + cc]
                ref1 = o.pfb_channelizer(x[-(WF + P - 1) * M:].cpu().numpy(), pt, M)[P - 1:, cb:cb + cc]
                errc = all_max(max(o.rel_rms(yc[:WF].cpu().numpy().reshape(-1), ref0.reshape(-1)),
                                   o.rel_rms(yc[-WF:].cpu().numpy().reshape(-1), ref1.reshape(-1))))
                c4 = {"channel_sharded_one_stream_Msamples_s": SAMPLES / (t * 1e-3) / 1e6, "channel_sharded_ms": t,
                      "channels_per_gpu": cc, "channel_sharded_parity_ok": bool(errc < 1e-5),
                      "channel_sharded_rel_rms_vs_oracle": errc}
                del yc
                pfb_t = nb.PfbChannelizer(pt, M)
                yt = torch.empty((SAMPLES // M, M), dtype=torch.complex64, device=dev)
                halo_len = (P - 1) * M
                st_peer = mg.SegmentedFir(pfb_t, rank, world, peer=True, halo_len=halo_len)
                st_p2p = mg.SegmentedFir(pfb_t, rank, world, peer=False, halo_len=halo_len)
                st_peer.run(x, yt)
                t = max_over_ranks(timed(torch, lambda: st_peer.run(x, yt), 5, 2, barrier) / 5)
                tails = gather_tails(halo_len)
                hist = tails[rank - 1].cpu().numpy() if rank > 0 else None
                ref0 = o.pfb_channelizer(x[:WF * M].cpu().numpy(), pt, M, hist=hist)
                ref1 = o.pfb_channelizer(x[-(WF + P - 1) * M:].cpu().numpy(), pt, M)[P - 1:]
                errt = all_max(max(o.rel_rms(yt[:WF].cpu().numpy().reshape(-1), ref0.reshape(-1)),
                                   o.rel_rms(yt[-WF:].cpu().numpy().reshape(-1), ref1.reshape(-1))))
                t_p2p = max_over_ranks(timed(torch, lambda: st_p2p.run(x, yt), 5, 2, barrier) / 5)
                c4["time_segmented_Msamples_s"] = world * SAMPLES / (t * 1e-3) / 1e6
                c4["time_segmented_ms"] = t
                c4["time_segmented_ms_with_nccl_p2p_halo_exchange"] = t_p2p
                c4["halo"] = "read in place from the left neighbour over NVLink (peer-mapped pointer)"
                c4["halo_bytes_per_rank"] = halo_len * 8
                c4["parity_ok"] = bool(errt < 1e-5)
                c4["rel_rms_vs_oracle"] = errt
                c4["parity_windows"] = f"first and last {WF} frames of every rank's segment vs oracle.pfb_channelizer (fp64), max over ranks"
                extras["config4_channelizer_64ch"] = c4
                del yt
            except Exception as e:  # pragma: no cover
                extras["config4_error"] = repr(e)

    # ---- multi-GPU only: the same configs as newsched flowgraphs on ALL GPUs of ONE process (C++ blocks, one mt
    # scheduler, every block / ring / stream on its own device; SURVEY.md 8e "single process, 8 devices"), next to
    # the one-process-per-GPU numbers above.  Rank 0 runs it; the other ranks wait on a HOST barrier (gloo), so no
    # NCCL kernel is spinning on their GPUs meanwhile.
    if dist is not None:
        try:
            torch.cuda.synchronize()
            hostgrp = dist.new_group(backend="gloo")
            dist.barrier(group=hostgrp)
            if rank == 0:
                import subprocess
                exe = os.path.join(ROOT, "newsched_b200", "host", "build", "bm_flowgraph")
                if not os.path.exists(exe):
                    subprocess.check_call(["make", "-C", os.path.join(ROOT, "newsched_b200", "host"), "-s"])
                env = dict(os.environ)
                fgm = {}
                for name, argv in (
                        ("config2_fft4096_mag_1Gi_per_gpu", ["--config", "2", "--samples", str(1 << 30)]),
                        ("config1_fir_ccf_64taps_1Gi_per_gpu", ["--config", "1", "--samples", str(1 << 30)]),
                        ("config3_fir1024d4_mulc_fft_1Gi_per_gpu", ["--config", "3", "--samples", str(1 << 30)]),
                        ("config5_time_segmented_fir4096_128Mi_per_gpu", ["--config", "5", "--samples", str(1 << 27)])):
                    best = None
                    for _ in range(2):
                        o_ = subprocess.run([exe] + argv + ["--gpus", str(world)], capture_output=True, text=True,
                                            timeout=180, env=env)
                        try:
                            rec = json.loads(o_.stdout.strip().splitlines()[-1])
                        except Exception:
                            rec = {"Msamples_s": 0.0, "error": (o_.stderr or o_.stdout)[-300:]}
                        if best is None or rec.get("Msamples_s", 0) > best.get("Msamples_s", 0):
                            best = rec
                    fgm[name] = {k: best.get(k) for k in ("Msamples_s", "seconds", "gpus", "kernel_launches", "error") if k in best}
                fgm["how"] = (f"newsched_b200/host/bm_flowgraph --gpus {world}: ONE process, one mt scheduler, {world} device-resident "
                              "replicas (config 5: time segments, halo peer-copied from the left neighbour's resident segment); "
                              "wall clock start()->wait(), aggregate over the GPUs, best of 2")
                extras["flowgraph_one_process_all_gpus"] = fgm
            dist.barrier(group=hostgrp)
        except Exception as e:  # pragma: no cover
            extras["flowgraph_multi_gpu_error"] = repr(e)

    cpu_baseline, cpu_tuned = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cb = cpu_fft_mag_rate(10, 1, target_s=1.5)
            cpu_baseline = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as e:  # pragma: no cover
            cpu_baseline = {"value": None, "error": repr(e)}
        try:
            cpu_tuned = cpu_fft_mag_rate_tuned()
        except Exception as e:  # pragma: no cover
            cpu_tuned = {"value": None, "error": repr(e)}

    # ---- the metric names "FIR-ccf & FFT-4096": every config's dominant kernel as a roofline row, at top level
    kernels = {"config2_fft4096_window_mag_1Gi": {k: roofline[k] for k in ("bound", "achieved", "peak", "frac", "unit")}}
    kernels["config2_fft4096_window_mag_1Gi"]["ms"] = k_ms
    for name, key in (("config1_fir_ccf_64taps_16Mi", "fir_ccf_64taps_16Mi"),
                      ("config1_fir_ccf_64taps_16Mi_simt_direct", "fir_ccf_64taps_16Mi_simt_direct"),
                      ("config3_head_fir_ccf_1024taps_decim4_mulc_64Mi", "fir_ccf_1024taps_decim4_mulc_64Mi"),
                      ("config5_body_fir_ccf_4096taps_64Mi", "fir_ccf_4096taps_64Mi")):
        if key in extras:
            kernels[name] = {k: extras[key][k] for k in extras[key]
                             if k in ("algorithm", "bound", "achieved", "peak", "frac", "unit", "ms", "executed_tflops",
                                      "executed_on", "executed_frac_of_measured_bf16_peak",
                                      "executed_frac_of_measured_fp32_peak")}
    if "pfb_channelizer_64ch_16tpc_1Gi" in extras:
        e4 = extras["pfb_channelizer_64ch_16tpc_1Gi"]
        kernels["config4_pfb_channelizer_64ch_1Gi"] = {"bound": "hbm", "achieved": e4["hbm_gbs"], "peak": peak_gbs,
                                                       "frac": e4["frac_of_hbm"], "unit": "GB/s", "ms": e4["ms"],
                                                       "algorithm": e4.get("algorithm")}
    if "pfb_channelizer_64ch_16tpc_1Gi_tensor_core_dft" in extras:
        e4 = extras["pfb_channelizer_64ch_16tpc_1Gi_tensor_core_dft"]
        kernels["config4_pfb_channelizer_64ch_1Gi_tensor_core_dft"] = {
            "bound": "hbm", "achieved": e4["hbm_gbs"], "peak": peak_gbs, "frac": e4["frac_of_hbm"], "unit": "GB/s",
            "ms": e4["ms"], "algorithm": 2, "executed_tflops": e4["executed_tensor_tflops"], "executed_on": "tensor",
            "executed_frac_of_measured_bf16_peak": e4["executed_frac_of_measured_bf16_peak"],
            "selected_by_default": e4["selected_by_default"]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": k_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG,
            "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu_baseline,
            "cpu_tuned_library": cpu_tuned, "e2e": e2e,
            "gpu_launches": int(launches), "clocks": sampler.summary(), "extras": extras,
            "gpu_name": torch.cuda.get_device_name(dev),
        }
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def claim_stdout():
    """Route fd 1 to stderr while the benchmark runs (NCCL / libraries print banners there) and keep
    the real stdout for the ONE JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output (a seeded sample of its vectors) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the B200 path only")
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())

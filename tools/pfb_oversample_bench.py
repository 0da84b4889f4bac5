"""Throughput of the polyphase channelizer at oversample 1, 2 and 4 against the HBM bound (DESIGN.md 4.4e).

For M in {16, 32, 64, 128, 256} and OS in {1, 2, 4}, P = 16 taps per channel (8 at M = 256), all channels:
one stateless work_segment over 2^28 complex64 input samples (2 GiB in, 2 OS GiB out: far beyond the L2),
timed with CUDA events after warm-up, `--reps` timed runs of `--calls` calls each; median and range.
The bound is the measured b200_copy bandwidth (read + write bytes over time, same call) over the bytes one
input sample moves: 8 read + 8 OS cc / M written. `--nbuf-ab` also times the OS > 1 rows with one input tile
(B200_PFB_ONEBUF) and two (B200_PFB_TWOBUF), alternated with the default handle.

    python tools/pfb_oversample_bench.py --out /tmp/pfb_oversample.json [--nbuf-ab]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def _time(torch, fn, calls, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b) / calls)
    return ms


def _stats(ms):
    s = sorted(ms)
    return {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1], "runs_ms": ms}


def _make(nb, taps, M, OS, env):
    saved = {k: os.environ.pop(k, None) for k in ("B200_PFB_ONEBUF", "B200_PFB_TWOBUF")}
    os.environ.update(env)
    try:
        return nb.PfbChannelizer(taps, M, oversample=OS)
    finally:
        for k in env:
            os.environ.pop(k, None)
        os.environ.update({k: v for k, v in saved.items() if v is not None})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2-samples", type=int, default=28)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nbuf-ab", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import torch

    import newsched_b200 as nb
    assert torch.cuda.is_available(), "this measurement needs the GPU"
    n = 1 << a.log2_samples
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=gen).mul_(2).sub_(1))
    res = {"tool": "tools/pfb_oversample_bench.py", "input_samples": n, "calls_per_run": a.calls, "runs": a.reps,
           **_device_info(torch), "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    # HBM copy bandwidth, the denominator
    cp = torch.empty_like(x)
    ms = _time(torch, lambda: nb.copy(x, cp), a.calls, a.reps, a.warmup)
    st = _stats(ms)
    copy_gbs = 2 * n * 8 / (st["median_ms"] * 1e-3) / 1e9
    res["copy"] = {**st, "GB_s": copy_gbs}
    del cp
    rows = []
    rng = np.random.default_rng(2)
    for M in (16, 32, 64, 128, 256):
        P = 8 if M == 256 else 16
        taps = (rng.uniform(-1, 1, M * P) / np.sqrt(M * P)).astype(np.float32)
        for OS in (1, 2, 4):
            D = M // OS
            out = torch.empty((n // D, M), dtype=torch.complex64, device="cuda")
            variants = {"default": {}}
            if a.nbuf_ab and OS > 1:
                variants.update({"onebuf": {"B200_PFB_ONEBUF": "1"}, "twobuf": {"B200_PFB_TWOBUF": "1"}})
            chs = {k: _make(nb, taps, M, OS, env) for k, env in variants.items()}
            runs = {k: [] for k in chs}
            for _ in range(3 if len(chs) > 1 else 1):      # alternate the variants
                for k, ch in chs.items():
                    runs[k] += _time(torch, lambda: ch.work_segment(x, None, out), a.calls,
                                     max(1, a.reps // (3 if len(chs) > 1 else 1)) if len(chs) > 1 else a.reps,
                                     a.warmup)
            bytes_per_sample = 8 + 8 * OS * M / M
            bound_gs = copy_gbs / bytes_per_sample
            row = {"M": M, "P": P, "oversample": OS, "hop": D, "bytes_per_input_sample": bytes_per_sample,
                   "hbm_bound_input_GS_s": bound_gs}
            for k, r in runs.items():
                s = _stats(r)
                gs = n / (s["median_ms"] * 1e-3) / 1e9
                row[k] = {**s, "input_GS_s": gs, "output_Gsamples_s": gs * OS,
                          "input_GS_s_range": [n / (s["max_ms"] * 1e-3) / 1e9, n / (s["min_ms"] * 1e-3) / 1e9],
                          "fraction_of_hbm_bound": gs / bound_gs}
            rows.append(row)
            print(json.dumps({"M": M, "OS": OS, **{k: round(row[k]["input_GS_s"], 1) for k in runs},
                              "fraction": round(row["default"]["fraction_of_hbm_bound"], 3)}), flush=True)
            del chs, out
            torch.cuda.empty_cache()
    res["rows"] = rows
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(json.dumps({"copy_GB_s": copy_gbs, "device": res["device"],
                      "power": res["power_limit_and_max_sm_clock"]}))


if __name__ == "__main__":
    main()

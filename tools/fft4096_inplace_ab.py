"""A/B of the FFT-4096 TMA kernel (fft4096_tma_kernel) between two builds of libb200dsp.so, on bench.py's shape:
2^27 samples (32768 vectors of 4096) resident in HBM, window + FFT + |.| (the bench kernel) and complex output.

    python tools/fft4096_inplace_ab.py build [--base REV]      # base = REV's csrc (git archive), new = working tree
    python tools/fft4096_inplace_ab.py run [--rounds 5] [--launches 50] [--json FILE]
    python tools/fft4096_inplace_ab.py profile [--lib PATH] [--trace FILE]

`build` needs git and nvcc (no GPU) and writes build_ab/{base,new}/libb200dsp.so.  `run` alternates the two libraries
(base, new, base, new, ...), one process per run, each run timing `--launches` back-to-back launches with CUDA events
after warm-up, and reports per library the median, min and max in Msamples/s (the unit of bench.py's `value`), together
with the card's name and power limit.  Every run also hashes the outputs of the last launch of several kernel forms on
the same seeded input, so the report says whether the two builds computed the same bits.  `profile` runs the bench
kernel under torch.profiler in a process of its own and reports launches, kernel duration and the start-to-start
interval of consecutive launches.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tarfile
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AB = os.path.join(ROOT, "build_ab")
LIBS = {"base": os.path.join(AB, "base", "libb200dsp.so"), "new": os.path.join(AB, "new", "libb200dsp.so")}
N = 4096
N_VEC = 32768
SAMPLES = N * N_VEC


def make_lib(csrc, build_dir, out):
    subprocess.check_call(["make", "-C", csrc, "-j8", "-s", f"BUILD={build_dir}", f"OUT={out}"])


def cmd_build(args):
    os.makedirs(AB, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        tar = os.path.join(tmp, "base.tar")
        subprocess.check_call(["git", "-C", ROOT, "archive", "-o", tar, args.base, "newsched_b200/csrc", "include"])
        with tarfile.open(tar) as t:
            t.extractall(os.path.join(tmp, "base"), filter="data")
        make_lib(os.path.join(tmp, "base", "newsched_b200", "csrc"), os.path.join(AB, "base", "obj"), LIBS["base"])
    # the working tree's sources, built apart from the package's own lib/ so that the package build is untouched
    make_lib(os.path.join(ROOT, "newsched_b200", "csrc"), os.path.join(AB, "new", "obj"), LIBS["new"])
    rev = subprocess.check_output(["git", "-C", ROOT, "rev-parse", args.base], text=True).strip()
    json.dump({"base": rev}, open(os.path.join(AB, "base", "REV.json"), "w"))
    print("built", LIBS["base"], "(", rev, ")", "and", LIBS["new"])


def bench_input(torch):
    # bench.py's synthetic stream: uniform[-1, 1) complex64, seed 0x5EED (rank 0)
    g = torch.Generator(device="cuda").manual_seed(0x5EED)
    return torch.view_as_complex(torch.rand(SAMPLES, 2, device="cuda", generator=g) * 2 - 1)


def blackman_harris():
    import numpy as np
    t = np.arange(N, dtype=np.float64) / (N - 1)
    return (0.35875 - 0.48829 * np.cos(2 * np.pi * t) + 0.14128 * np.cos(4 * np.pi * t)
            - 0.01168 * np.cos(6 * np.pi * t)).astype(np.float32)


def cmd_child(args):
    import torch
    sys.path.insert(0, ROOT)
    import newsched_b200 as nb
    nb.lib()
    x = bench_input(torch)
    w = blackman_harris()
    mag = torch.empty(SAMPLES, dtype=torch.float32, device="cuda")
    cpx = torch.empty_like(x)
    res = {"lib": os.environ["B200_LIB"]}
    for name, op, out in (("mag", nb.FFT(N, True, w, output=nb.OUT_MAG), mag), ("complex", nb.FFT(N, True, w), cpx)):
        for _ in range(args.warmup):
            op.work(x, out)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.launches):
            op.work(x, out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        res[name] = SAMPLES * args.launches / (ms * 1e-3) / 1e6
        res[name + "_us_per_launch"] = ms * 1e3 / args.launches
    if args.digests:
        dig = {}
        for name, op, out in (("mag_fwd", nb.FFT(N, True, w, output=nb.OUT_MAG), mag),
                              ("mag2_fwd", nb.FFT(N, True, w, output=nb.OUT_MAG_SQUARED), mag),
                              ("mag_rev_shift_k", nb.FFT(N, False, w, True, output=nb.OUT_MAG,
                                                         pre_multiply_const=0.5 - 0.25j), mag),
                              ("complex_fwd", nb.FFT(N, True, w), cpx),
                              ("complex_rev_shift", nb.FFT(N, False, w, True), cpx)):
            op.work(x, out)
            torch.cuda.synchronize()
            dig[name] = hashlib.sha256(out.view(torch.uint8).cpu().numpy().tobytes()).hexdigest()[:16]
        res["digests"] = dig
    print(json.dumps(res))


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                     "--format=csv,noheader"], text=True).strip().splitlines()[0]
        name, pl, clk = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001 - report what could not be read instead of failing the A/B
        return {"error": repr(e)}


def cmd_run(args):
    libs = {"base": args.base_lib or LIBS["base"], "new": args.new_lib or LIBS["new"]}
    for k, p in libs.items():
        if not os.path.exists(p):
            sys.exit(f"{k} library {p} not found: run `{sys.argv[0]} build` first")
    runs = {k: [] for k in libs}
    for r in range(args.rounds):
        for k in ("base", "new"):
            env = dict(os.environ, B200_LIB=libs[k])
            argv = [sys.executable, os.path.abspath(__file__), "child", "--launches", str(args.launches),
                    "--warmup", str(args.warmup)] + (["--digests"] if r == 0 else [])
            out = subprocess.check_output(argv, env=env, text=True)
            runs[k].append(json.loads(out.strip().splitlines()[-1]))
            print(f"round {r} {k}: mag {runs[k][-1]['mag']:.1f}  complex {runs[k][-1]['complex']:.1f} Msamples/s",
                  flush=True)
    report = {"card": card(), "shape": f"{N_VEC} x {N} complex64 (2^27 samples), {args.launches} launches per run",
              "rounds": args.rounds, "libs": {k: os.path.relpath(p, ROOT) for k, p in libs.items()}}
    for metric in ("mag", "complex"):
        m = {}
        for k in libs:
            v = [r[metric] for r in runs[k]]
            m[k] = {"median": statistics.median(v), "min": min(v), "max": max(v), "runs": v,
                    "us_per_launch_median": statistics.median(r[metric + "_us_per_launch"] for r in runs[k])}
        m["new_over_base"] = m["new"]["median"] / m["base"]["median"]
        m["spreads_overlap"] = not (m["new"]["min"] > m["base"]["max"] or m["base"]["min"] > m["new"]["max"])
        report[metric] = m
    report["bit_identical"] = runs["base"][0]["digests"] == runs["new"][0]["digests"]
    report["digests"] = {k: runs[k][0]["digests"] for k in libs}
    print(json.dumps(report, indent=1))
    if args.json:
        json.dump(report, open(args.json, "w"), indent=1)


def cmd_profile(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    if args.lib:
        os.environ["B200_LIB"] = args.lib
    sys.path.insert(0, ROOT)
    import newsched_b200 as nb
    nb.lib()
    x = bench_input(torch)
    out = torch.empty(SAMPLES, dtype=torch.float32, device="cuda")
    op = nb.FFT(N, True, blackman_harris(), output=nb.OUT_MAG)
    for _ in range(5):
        op.work(x, out)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.launches):
            op.work(x, out)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        trace = args.trace or os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(trace)
        events = json.load(open(trace))["traceEvents"]
    kernels = {}
    for e in events:
        if e.get("cat") == "kernel":
            kernels.setdefault(e["name"], []).append(e)
    rep = {"card": card(), "steps": args.launches, "kernels": []}
    for name, ev in kernels.items():
        ev.sort(key=lambda e: e["ts"])
        starts = [e["ts"] for e in ev]
        # with the dependent launch a kernel's CTAs start while its predecessor drains and wait there, so its
        # duration includes that overlap; the start-to-start interval is the time per launch
        rep["kernels"].append({"name": name, "launches": len(ev),
                               "duration_us_median": statistics.median(e["dur"] for e in ev),
                               "start_to_start_us_median": statistics.median(b - a for a, b in zip(starts, starts[1:]))
                               if len(ev) > 1 else None})
    print(json.dumps(rep, indent=1))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    sp = ap.add_subparsers(dest="cmd", required=True)
    b = sp.add_parser("build")
    b.add_argument("--base", default="HEAD", help="git revision of the base build (default HEAD)")
    r = sp.add_parser("run")
    r.add_argument("--rounds", type=int, default=5)
    r.add_argument("--launches", type=int, default=50)
    r.add_argument("--warmup", type=int, default=5)
    r.add_argument("--base-lib")
    r.add_argument("--new-lib")
    r.add_argument("--json")
    c = sp.add_parser("child")
    c.add_argument("--launches", type=int, default=50)
    c.add_argument("--warmup", type=int, default=5)
    c.add_argument("--digests", action="store_true")
    p = sp.add_parser("profile")
    p.add_argument("--lib")
    p.add_argument("--launches", type=int, default=20)
    p.add_argument("--trace")
    args = ap.parse_args()
    {"build": cmd_build, "run": cmd_run, "child": cmd_child, "profile": cmd_profile}[args.cmd](args)


if __name__ == "__main__":
    main()

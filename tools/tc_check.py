"""Tensor-core (tcgen05) FIR, algorithm 2: parity against the fp64 oracle and A/B timing against the
SIMT forms (algorithm 0 = auto: direct / overlap-save).  Algorithm 2 runs the tap-stationary kernel at
decimation 1 up to 449 taps and the ring form otherwise.  Every case runs in its own process, so a
trapped kernel poisons only that case.
usage: python tools/tc_check.py [parity|time|all]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PARITY = [(64, 1), (100, 1), (128, 1), (256, 1), (448, 1), (449, 1), (33, 1), (257, 1), (5, 1), (1024, 4)]
TIMING = [(48, 1), (64, 1), (96, 1), (128, 1), (192, 1), (256, 1), (384, 1), (512, 1), (1024, 1), (1024, 4), (512, 4), (256, 2)]


def child(kind, T, D):
    import numpy as np
    import torch
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 31 + D)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    if kind == "parity":
        import oracle as o
        n = (8192 * 301 + 1000) * D + (D - 1)          # > 2 tiles per SM for the persistent form, ragged tail
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        dx = torch.from_numpy(x).cuda()
        f = nb.FirFilter(taps, D, algorithm=2)
        y, nc = f.work(dx)
        torch.cuda.synchronize()
        ref = o.fir(x, taps, D)
        err = o.rel_rms(y.cpu().numpy(), ref)
        # streaming: two chunks must continue the history
        f2 = nb.FirFilter(taps, D, algorithm=2)
        cut = (8192 * 150 + 333) * D
        ya, _ = f2.work(dx[:cut])
        yb, _ = f2.work(dx[cut:])
        err2 = o.rel_rms(torch.cat([ya, yb]).cpu().numpy(), ref)
        # fused multiply_const epilogue
        f3 = nb.FirFilter(taps, D, algorithm=2, multiply_const=0.5 - 0.25j)
        y3, _ = f3.work(dx)
        err3 = o.rel_rms(y3.cpu().numpy(), ref * (0.5 - 0.25j))
        print(json.dumps({"kind": kind, "T": T, "D": D, "algorithm": f.algorithm, "rel_rms": err,
                          "rel_rms_chunked": err2, "rel_rms_fused": err3, "ok": bool(max(err, err2, err3) < 1e-5)}))
    else:
        n = 1 << 26
        g = torch.Generator(device="cuda").manual_seed(1)
        x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
        out = torch.empty(n // D, dtype=torch.complex64, device="cuda")
        res = {"kind": kind, "T": T, "D": D}
        for algo in (2, 3, 0):
            f = nb.FirFilter(taps, D, algorithm=algo)
            for _ in range(3):
                f.work_segment(x, None, out)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(10):
                f.work_segment(x, None, out)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            gs = n / (ms * 1e-3) / 1e9
            tag = f"algo{f.algorithm}" if algo else f"auto(algo{f.algorithm})"
            res[f"{tag}_GSs"] = round(gs, 1)
            res[f"{tag}_hbm_frac"] = round(gs * (8 + 8 / D) / 6556.5, 3)
            if algo == 2:
                # executed tensor flops: 4 MMAs of 128x128x16 per K-step, ksteps = (roundup16(ceil(T/D)-1)+64)/16 per branch
                tq = (T + D - 1) // D
                ksteps = ((tq - 1 + 15) // 16 * 16 + 64) // 16
                flop_per_tile = D * ksteps * 4 * 2 * 128 * 128 * 16
                tiles = (n // D + 8191) // 8192
                res["tensor_tflops_executed"] = round(flop_per_tile * tiles / (ms * 1e-3) / 1e12, 1)
        print(json.dumps(res))


def main():
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what == "child":
        return child(sys.argv[2], int(sys.argv[3]), int(sys.argv[4]))
    if what in ("parity", "all"):
        for T, D in PARITY:
            r = subprocess.run([sys.executable, __file__, "child", "parity", str(T), str(D)],
                               capture_output=True, text=True, timeout=300)
            line = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else ""
            print(line if line.startswith("{") else json.dumps(
                {"kind": "parity", "T": T, "D": D, "ok": False, "rc": r.returncode, "stderr": r.stderr[-400:]}), flush=True)
    if what in ("time", "all"):
        for T, D in TIMING:
            r = subprocess.run([sys.executable, __file__, "child", "time", str(T), str(D)],
                               capture_output=True, text=True, timeout=300)
            line = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else ""
            print(line if line.startswith("{") else json.dumps({"kind": "time", "T": T, "D": D, "rc": r.returncode,
                                                                 "stderr": r.stderr[-400:]}), flush=True)


if __name__ == "__main__":
    main()

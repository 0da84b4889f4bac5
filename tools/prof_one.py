"""Runs one hot-path kernel a few times on synthetic data (for ncu captures / launch lists).
usage: python tools/prof_one.py fftmag|fft|fftnN|tcT|fir64simt|fir64|firdec64d4|firdec64d5|rs32|fir1024d4|fir4096|pfb|pfbtc|pfb16|copy [reps]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import newsched_b200 as nb

what = sys.argv[1] if len(sys.argv) > 1 else "fftmag"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
N = 4096
n = N * 32768 if what in ("fftmag", "fft", "copy", "pfb") else (1 << 24)
g = torch.Generator(device="cuda").manual_seed(1)
x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
t = np.arange(N) / (N - 1)
w = (0.35875 - 0.48829 * np.cos(2 * np.pi * t) + 0.14128 * np.cos(4 * np.pi * t) - 0.01168 * np.cos(6 * np.pi * t)).astype(np.float32)
rng = np.random.default_rng(1)
if what == "fftmag":
    op = nb.FFT(N, True, w, output=nb.OUT_MAG); out = torch.empty(n, dtype=torch.float32, device="cuda"); fn = lambda: op.work(x, out)
elif what == "fft":
    op = nb.FFT(N, True, w); out = torch.empty_like(x); fn = lambda: op.work(x, out)
elif what.startswith("fftn"):
    Nn = int(what[4:]); t2 = np.arange(Nn) / (Nn - 1)
    w2 = (0.35875 - 0.48829 * np.cos(2 * np.pi * t2) + 0.14128 * np.cos(4 * np.pi * t2) - 0.01168 * np.cos(6 * np.pi * t2)).astype(np.float32)
    n = N * 32768; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.FFT(Nn, True, w2); out = torch.empty_like(x); fn = lambda: op.work(x, out)
elif what == "fir64":
    op = nb.FirFilter((rng.uniform(-1, 1, 64) / 64).astype(np.float32)); out = torch.empty_like(x); fn = lambda: op.work_segment(x, None, out)
elif what.startswith("tc"):          # tensor-core (tcgen05) FIR, e.g. tc64 / tc128 / tc256
    T = int(what[2:]); n = 1 << 26; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.FirFilter((rng.uniform(-1, 1, T) / T).astype(np.float32), algorithm=2); out = torch.empty_like(x); fn = lambda: op.work_segment(x, None, out)
elif what == "fir64simt":
    op = nb.FirFilter((rng.uniform(-1, 1, 64) / 64).astype(np.float32), algorithm=1); out = torch.empty_like(x); fn = lambda: op.work_segment(x, None, out)
elif what == "firdec64d4":
    n = N * 32768; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.FirFilter((rng.uniform(-1, 1, 64) / 64).astype(np.float32), 4); out = torch.empty(n // 4, dtype=torch.complex64, device="cuda"); fn = lambda: op.work_segment(x, None, out)
elif what == "firdec64d5":
    n = N * 32768 // 5 * 5; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.FirFilter((rng.uniform(-1, 1, 64) / 64).astype(np.float32), 5); out = torch.empty(n // 5, dtype=torch.complex64, device="cuda"); fn = lambda: op.work_segment(x, None, out)
elif what == "rs32":
    op = nb.RationalResampler((rng.uniform(-1, 1, 192) / 64).astype(np.float32), 3, 2); out = torch.empty(n // 2 * 3, dtype=torch.complex64, device="cuda"); fn = lambda: op.work_segment(x, None, out)
elif what.startswith("pfbm"):        # pfbm<M>x<P>, e.g. pfbm128x8, pfbm8x16
    import scipy.signal as sig
    Mm, Pp = (int(v) for v in what[4:].split("x"))
    n = N * 32768; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.PfbChannelizer(sig.firwin(Mm * Pp, 1 / Mm).astype(np.float32), Mm); out = torch.empty_like(x).view(-1, Mm); fn = lambda: op.work_segment(x, None, out)
elif what == "pfb16":
    import scipy.signal as sig
    n = N * 32768; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.PfbChannelizer(sig.firwin(16 * 8, 1 / 16).astype(np.float32), 16); out = torch.empty_like(x).view(-1, 16); fn = lambda: op.work_segment(x, None, out)
elif what == "fir1024d4":
    op = nb.FirFilter((rng.uniform(-1, 1, 1024) / 1024).astype(np.float32), 4); out = torch.empty(n // 4, dtype=torch.complex64, device="cuda"); fn = lambda: op.work_segment(x, None, out)
elif what == "fir4096":
    n = 1 << 26; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.FirFilter((rng.uniform(-1, 1, 4096) / 4096).astype(np.float32), 1); out = torch.empty_like(x); fn = lambda: op.work_segment(x, None, out)
elif what == "pfbtc":               # 64 channels, the DFT on the tensor cores (algorithm 2)
    import scipy.signal as sig
    n = N * 32768; x = torch.view_as_complex(torch.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    op = nb.PfbChannelizer(sig.firwin(1024, 1 / 64).astype(np.float32), 64, algorithm=2); out = torch.empty_like(x).view(-1, 64); fn = lambda: op.work_segment(x, None, out)
elif what == "pfb":
    import scipy.signal as sig
    op = nb.PfbChannelizer(sig.firwin(1024, 1 / 64).astype(np.float32), 64, algorithm=1); out = torch.empty_like(x).view(-1, 64); fn = lambda: op.work_segment(x, None, out)
else:
    out = torch.empty_like(x); fn = lambda: nb.copy(x, out)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(2): fn()
torch.cuda.synchronize(); e0.record()
for _ in range(reps): fn()
e1.record(); torch.cuda.synchronize()
print(what, "ms/launch", e0.elapsed_time(e1) / reps, "Gsamples/s", n / (e0.elapsed_time(e1) / reps * 1e-3) / 1e9)

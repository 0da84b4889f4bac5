"""The oversampled channelizer (oversample 2 and 4) on the GPU against the fp64 oracle.

b200_pfb_create with oversample OS > 1 takes the single-pass kernels only, with OS a template parameter:
    M = 64          pfb64_kernel<P4, OS> for P4 in {4, 8, 12, 16, 24, 32} (taps in registers), pfb64_kernel<0, OS>
                    (taps in shared memory) otherwise, up to the P of single_pass_max_p (test_pfb_oversampled.py)
    M = 16 .. 256   pfbm_kernel<M, P4, OS> for P4 in {4, 8, 16}, pfbm_kernel<M, 0, OS> otherwise, likewise
The input tile is TT + P4 OS - 1 rows of D = M / OS samples; branch outputs go to the U slot (i - tD) mod M.
After each work() call pfb_tail_kernel keeps the last P M - D input samples, and the handle the frame phase.

The yardstick is that of test_pfb_paths_gpu.py: random asymmetric taps; per output frame, relative to the RMS
of its M reference channels, a relative RMS error below 1e-5 and a worst channel below 1e-4; every value
finite; nothing written around the output."""
import os
import subprocess

import numpy as np
import pytest

import oracle as o
from conftest import ROOT, cplx
from test_pfb_oversampled import pfb_os_reference, single_pass_max_p
from test_pfb_paths_gpu import _Guarded, _check_frames, _device_input, _sms, _taps

gpu = pytest.mark.gpu
SWITCHES = ("B200_PFB_TWOPASS", "B200_PFB_ONEBUF", "B200_PFB_TWOBUF", "B200_PFBT_MN", "B200_PFB_TC")


def _nb():
    import newsched_b200 as nb
    return nb


def _frames(torch, M, sweeps=2):
    """Two full sweeps of the persistent grid plus two tiles and a partial one: some CTAs loop three times, the
    first tile reads the history, the last is ragged."""
    TT = 4096 // M
    grid = (1 if M >= 128 else 2) * _sms(torch)
    return (sweeps * grid + 2) * TT + TT // 3 + 1


def _channelizer(monkeypatch, taps, M, OS, cb=0, cc=0, algorithm=0, env=None):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    ch = _nb().PfbChannelizer(taps, M, channel_begin=cb, channel_count=cc, algorithm=algorithm, oversample=OS)
    assert ch.oversample == (OS or 1) and ch.hop == M // (OS or 1) and ch.algorithm == 1
    return ch


def _data(M, P, OS, n_frames, seed=0):
    rng = np.random.default_rng([M, P, OS, n_frames, seed])
    h = _taps(rng, M, P)
    D = M // OS
    x = cplx(rng, n_frames * D + D - 1)          # the trailing D - 1 items make no frame and stay unconsumed
    return h, x


def _run(torch, monkeypatch, M, P, OS, n_frames, *, cb=0, cc=0, in_offset=0, out_misaligned=False, env=None,
         record_property=None, ref=None):
    h, x = _data(M, P, OS, n_frames)
    if ref is None:
        ref = pfb_os_reference(x, h, M, OS)
    ch = _channelizer(monkeypatch, h, M, OS, cb, cc, env=env)
    n_ch = cc or M - cb
    g = _Guarded(torch, n_frames, n_ch, out_misaligned)
    y, nc = ch.work(_device_input(torch, x, in_offset), out=g.view)
    torch.cuda.synchronize()
    assert nc == n_frames * (M // OS) and tuple(y.shape) == (n_frames, n_ch)
    g.check_untouched()
    yh = y.cpu().numpy()
    _check_frames(yh, ref, slice(cb, cb + n_ch), record_property)
    return yh, ref


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ----------------------------------------------------------------------------- 1. every instantiation
def _cases():
    rows = []
    for OS in (2, 4):
        # pfb64_kernel<P4, OS>: P4 = 4, 8, 12, 16, 24, 32 in registers; P = 20 and the largest P: taps in shared memory
        for P in (3, 8, 11, 16, 21, 32, 20, single_pass_max_p(64, OS)):
            rows.append(pytest.param(64, P, OS, id=f"M64-P{P}-os{OS}"))
        # pfbm_kernel<M, P4, OS>: P4 = 4, 8, 16 in registers; P = 11 (P4 12) and the largest P: taps in shared memory
        for M in (16, 32, 128, 256):
            for P in (3, 8, 16, 11, single_pass_max_p(M, OS)):
                rows.append(pytest.param(M, P, OS, id=f"M{M}-P{P}-os{OS}"))
    return rows


@gpu
@pytest.mark.parametrize("M,P,OS", _cases())
def test_oversampled_instantiation(cuda, monkeypatch, record_property, M, P, OS):
    big = P > 32
    _run(cuda, monkeypatch, M, P, OS, _frames(cuda, M, sweeps=1 if big else 2), record_property=record_property)


@gpu
@pytest.mark.parametrize("OS", [2, 4])
@pytest.mark.parametrize("M,P", [(64, 8), (64, 16), (16, 8), (128, 16)])
def test_oversampled_tile_count_switches(cuda, monkeypatch, M, P, OS):
    """One input tile (B200_PFB_ONEBUF) and two (B200_PFB_TWOBUF) give the same bits as the default."""
    n = _frames(cuda, M, sweeps=1)
    a, ref = _run(cuda, monkeypatch, M, P, OS, n)
    for env in ({"B200_PFB_ONEBUF": "1"}, {"B200_PFB_TWOBUF": "1"}):
        b, _ = _run(cuda, monkeypatch, M, P, OS, n, env=env, ref=ref)
        assert np.array_equal(_bits(a), _bits(b)), env


# ----------------------------------------------------------------------------------- 2, 3. alignment, slices
FAMILIES = [
    pytest.param(64, 16, 2, id="pfb64-P16-os2"),
    pytest.param(64, 20, 4, id="pfb64smem-P20-os4"),
    pytest.param(16, 8, 4, id="pfbm16-P8-os4"),
    pytest.param(32, 11, 2, id="pfbm32smem-P11-os2"),
    pytest.param(128, 8, 2, id="pfbm128-P8-os2"),
    pytest.param(256, 4, 4, id="pfbm256-P4-os4"),
]


@gpu
@pytest.mark.parametrize("M,P,OS", FAMILIES)
def test_oversampled_misaligned_input_and_output(cuda, monkeypatch, record_property, M, P, OS):
    """Input 8 bytes off a 16-byte boundary (every tile staged element-wise instead of by bulk copy), then the
    output 8 bytes off: bit-equal to the aligned call."""
    n = _frames(cuda, M, sweeps=1)
    a, ref = _run(cuda, monkeypatch, M, P, OS, n)
    b, _ = _run(cuda, monkeypatch, M, P, OS, n, in_offset=1, ref=ref, record_property=record_property)
    c, _ = _run(cuda, monkeypatch, M, P, OS, n, out_misaligned=True, ref=ref)
    assert np.array_equal(_bits(a), _bits(b)) and np.array_equal(_bits(a), _bits(c))


@gpu
@pytest.mark.parametrize("which", ["first", "last", "middle"])
@pytest.mark.parametrize("M,P,OS", FAMILIES)
def test_oversampled_channel_slice(cuda, monkeypatch, record_property, M, P, OS, which):
    cb, cc = {"first": (0, 1), "last": (M - 1, 1), "middle": (M // 3, M // 3)}[which]
    n = _frames(cuda, M, sweeps=1)
    full, ref = _run(cuda, monkeypatch, M, P, OS, n)
    part, _ = _run(cuda, monkeypatch, M, P, OS, n, cb=cb, cc=cc, ref=ref, record_property=record_property)
    assert np.array_equal(_bits(part), _bits(full[:, cb:cb + cc]))


# ------------------------------------------------------------------------------------------- 4. streaming
STREAMS = [pytest.param(64, 16, 2, id="pfb64-os2"), pytest.param(64, 20, 4, id="pfb64smem-os4"),
           pytest.param(16, 8, 4, id="pfbm16-os4"), pytest.param(256, 4, 2, id="pfbm256-os2")]


def _stream_input(torch, M, P, OS):
    n = _frames(torch, M, sweeps=1)
    h, x = _data(M, P, OS, n, seed=1)
    return h, x, torch.from_numpy(x).cuda(), n


@gpu
@pytest.mark.parametrize("M,P,OS", STREAMS)
def test_oversampled_stream_in_chunks(cuda, monkeypatch, M, P, OS):
    """work() calls back to back on one stream without a host sync: one-frame calls (the history spans several),
    odd frame counts (the frame phase carries over), D - 1 leftover items, prime sizes, and calls with fewer than
    D items (nothing consumed or produced). The concatenated output equals one call over the input, bit for bit,
    and that call matches the oracle."""
    torch = cuda
    h, x, xd, n = _stream_input(torch, M, P, OS)
    D = M // OS
    one, nc = _channelizer(monkeypatch, h, M, OS).work(xd)
    assert nc == n * D
    ch = _channelizer(monkeypatch, h, M, OS)
    out = torch.full((n, M), float("nan"), dtype=torch.complex64, device="cuda")
    TT = 4096 // M
    sizes = [D] * 5 + [3 * D, D - 1, 5 * D + D - 1, 1, 7 * D + 3, 1009, 4099, TT * D + 1, 2 * TT * D - 1, 65521]
    pos = f = k = 0
    while f < n:
        size = sizes[k] if k < len(sizes) else x.size
        k += 1
        seg = xd[pos:pos + size]
        want = seg.numel() // D
        y, c = ch.work(seg, out=out[f:f + want])
        assert c == want * D and y.shape[0] == want
        pos += c
        f += want
    assert f == n and pos == n * D
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(one.cpu().numpy()))
    _check_frames(one.cpu().numpy(), pfb_os_reference(x, h, M, OS))


@gpu
@pytest.mark.parametrize("M,P,OS", STREAMS)
def test_oversampled_reset_mid_stream(cuda, monkeypatch, M, P, OS):
    """Reset after an odd number of frames zeroes the history and the frame phase: the next call equals a fresh
    handle's."""
    torch = cuda
    h, x, xd, n = _stream_input(torch, M, P, OS)
    D = M // OS
    ch = _channelizer(monkeypatch, h, M, OS)
    y0, _ = ch.work(xd[: (2 * (n // 4) + 1) * D])
    ch.reset()
    y, _ = ch.work(xd)
    fresh, _ = _channelizer(monkeypatch, h, M, OS).work(xd)
    torch.cuda.synchronize()
    assert y0.shape[0] % 2 == 1
    assert np.array_equal(_bits(y.cpu().numpy()), _bits(fresh.cpu().numpy()))


# ---------------------------------------------------------------------------------------- 5. run_segment
@gpu
@pytest.mark.parametrize("M,P,OS", STREAMS)
def test_oversampled_segments_join(cuda, monkeypatch, M, P, OS):
    """Segments starting at multiples of M input samples, each with the P M - D samples before it as halo, join
    into the one-shot output bit for bit; a segment with no halo is the oracle with zero history."""
    torch = cuda
    h, x, xd, n = _stream_input(torch, M, P, OS)
    D, nh = M // OS, P * M - M // OS
    one, _ = _channelizer(monkeypatch, h, M, OS).work(xd)
    ch = _channelizer(monkeypatch, h, M, OS)
    cuts = [0, (n * D // 3) // M * M, (2 * n * D // 3) // M * M + M, x.size]
    assert cuts[1] >= nh
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        halo = xd[lo - nh:lo] if lo else None
        parts.append(ch.work_segment(xd[lo:hi], halo=halo))
    torch.cuda.synchronize()
    joined = torch.cat(parts).cpu().numpy()
    assert joined.shape[0] == n
    assert np.array_equal(_bits(joined), _bits(one.cpu().numpy()))
    lo = cuts[1]
    seg = ch.work_segment(xd[lo:])
    torch.cuda.synchronize()
    _check_frames(seg.cpu().numpy(), pfb_os_reference(x[lo:], h, M, OS))


# ------------------------------------------------------------------------------ 6. dependent launches
@gpu
def test_alternating_oversample_rates_on_one_stream(cuda, monkeypatch):
    """OS = 2, 1 and 4 handles (M = 64, P = 16) work in turn on one stream, chunk by chunk, without a host sync:
    each handle's output equals its own one-shot run and the oracle."""
    torch = cuda
    M, P = 64, 16
    rng = np.random.default_rng(64)
    h = _taps(rng, M, P)
    n_in = 96 * 4096 * 3 + 77
    x = cplx(rng, n_in)
    xd = torch.from_numpy(x).cuda()
    rates = (2, 1, 4)
    chs = [_channelizer(monkeypatch, h, M, OS) for OS in rates]
    outs = [[] for _ in rates]
    pos = [0, 0, 0]
    for size in (4096 * 7 + 13, 1, 64 * 33 + 31, 4096 * 50 + 5, n_in):
        for k, ch in enumerate(chs):
            y, c = ch.work(xd[pos[k]:pos[k] + size])
            outs[k].append(y)
            pos[k] += c
    torch.cuda.synchronize()
    for k, OS in enumerate(rates):
        got = torch.cat(outs[k]).cpu().numpy()
        one, _ = _channelizer(monkeypatch, h, M, OS).work(xd)
        torch.cuda.synchronize()
        assert np.array_equal(_bits(got), _bits(one.cpu().numpy())), OS
        _check_frames(got, pfb_os_reference(x, h, M, OS))


# ---------------------------------------------------------------------- 7. oversample 0 / 1, algorithm 2
@gpu
@pytest.mark.parametrize("M,P", [(64, 16), (64, 20), (16, 8), (4, 8), (128, 101)])
def test_oversample_zero_and_one_are_the_critically_sampled_bank(cuda, monkeypatch, M, P):
    torch = cuda
    rng = np.random.default_rng([M, P, 3])
    h = _taps(rng, M, P)
    x = cplx(rng, M * 3000 + 5)
    xd = torch.from_numpy(x).cuda()
    a, _ = _channelizer(monkeypatch, h, M, 0).work(xd)
    b, _ = _channelizer(monkeypatch, h, M, 1).work(xd)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(a.cpu().numpy()), _bits(b.cpu().numpy()))
    _check_frames(a.cpu().numpy(), o.pfb_channelizer(x, h, M))


@gpu
@pytest.mark.parametrize("OS", [2, 4])
def test_oversampled_refuses_tensor_core_dft(cuda, monkeypatch, OS):
    nb = _nb()
    h = np.full(64 * 8, 0.01, np.float32)
    with pytest.raises(nb.B200Error, match="needs oversample 1"):
        nb.PfbChannelizer(h, 64, algorithm=2, oversample=OS)
    ch = _channelizer(monkeypatch, h, 64, OS)
    with pytest.raises(nb.B200Error, match="needs oversample 1"):
        nb._check(nb.lib().b200_pfb_set_algorithm(ch.handle, 2))
    assert ch.algorithm == 1


@gpu
def test_oversampled_refuses_two_pass_form(cuda, monkeypatch):
    nb = _nb()
    with pytest.raises(nb.B200Error, match="single-pass kernels only"):
        _channelizer(monkeypatch, np.full(64 * 8, 0.01, np.float32), 64, 2, env={"B200_PFB_TWOPASS": "1"})


# ------------------------------------------------------------------------------------------------ 8. Chain
@gpu
def test_chain_with_oversampled_stage(cuda):
    """Chain [multiply_const, PFB at OS = 2]: the PFB stage consumes whole hops (den = multiple = D); device run
    and host-streamed run against the oracle."""
    torch = cuda
    nb = _nb()
    M, P, OS = 64, 16, 2
    D = M // OS
    rng = np.random.default_rng(8)
    h = _taps(rng, M, P)
    n = D * 4096 * 24
    x = cplx(rng, n)
    k = 0.5 - 0.25j
    ref = pfb_os_reference(o.multiply_const(x, k), h, M, OS)
    ch = nb.Chain([("multiply_const_cc", k), nb.PfbChannelizer(h, M, oversample=OS)], in_item_bytes=8,
                  chunk_items=D * 4096 * 5)
    out = torch.empty((n // D, M), dtype=torch.complex64, device="cuda")
    assert ch.run(torch.from_numpy(x).cuda(), out) == out.numel() * 8
    torch.cuda.synchronize()
    _check_frames(out.cpu().numpy(), ref)
    ch2 = nb.Chain([("multiply_const_cc", k), nb.PfbChannelizer(h, M, oversample=OS)], in_item_bytes=8,
                   chunk_items=D * 4096 * 5)
    hx = torch.from_numpy(x).pin_memory()
    hy = torch.empty((n // D, M), dtype=torch.complex64).pin_memory()
    assert ch2.run_host(hx, hy) == hy.numel() * 8
    _check_frames(hy.numpy(), ref)


# ------------------------------------------------------------------------------------ 9. C++ flowgraph
@gpu
def test_cpp_flowgraph_oversampled(tmp_path):
    """tests/cpp/qa_pfb_oversampled.cpp, built here against the library with the flags of tests/cpp/Makefile."""
    exe = str(tmp_path / "qa_pfb_oversampled")
    lib = os.path.join(ROOT, "newsched_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Wno-unused-parameter",
                           "-I" + os.path.join(ROOT, "include"), "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "qa_pfb_oversampled.cpp"), "-L" + lib, "-lb200dsp",
                           "-Wl,-rpath," + lib])
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(p.stdout[-4000:], p.stderr[-2000:])
    assert p.returncode == 0 and " 0 failed" in p.stdout, p.stdout[-3000:] + p.stderr[-1000:]
    for name in ("Oversampled.Pfb64Os2", "Oversampled.Pfb16Os4Slice", "Oversampled.Rejections"):
        assert f"[  OK  ] {name}" in p.stdout

"""Every kernel path of the polyphase channelizer (pfb.cu) against the fp64 oracle.

b200_pfb_create picks the kernel family from M, P4 = P rounded up to a multiple of 4 and three create-time
environment switches (B200_PFB_TWOPASS, B200_PFB_ONEBUF, B200_PFBT_MN); pfb_launch then picks the
instantiation from P4:
    M = 64          pfb64_kernel<P4> for P4 in {4, 8, 12, 16, 24, 32} (taps in registers), pfb64_kernel<0>
                    (taps in shared memory) otherwise, up to P = 204 (220 KiB of shared memory). Two input
                    tiles only at P4 = 16 without B200_PFB_ONEBUF.
                    algorithm=2 and P <= 16: pfb64_tc_kernel<P4>, the DFT across branches as a bf16x3 tcgen05
                    GEMM, branch outputs stored MN-major, or K-major under B200_PFBT_MN=0.
    M = 4, 8        pfbs_kernel<M, P4> for P4 in {4, 8, 16}, pfbs_kernel<M, 0> otherwise, while one input tile
                    fits 110 KiB (P <= 856 / 428). Two tiles while they fit 113 KiB (P <= 132 / 64) without
                    B200_PFB_ONEBUF.
    M = 16 .. 256   pfbm_kernel<M, P4> likewise, while one tile fits 220 KiB (P <= 820, 408, 100, 48 for
                    M = 16, 32, 128, 256). M >= 128 takes two tiles while they fit 227 KiB (P <= 52 / 24)
                    without B200_PFB_ONEBUF.
    otherwise, or   pfb_generic_kernel, up to 220 KiB (P <= 3328, 1664, 832, 416, 104, 52 for M = 4 .. 256;
    under           M = 64 has no such form): the direct DFT for M = 4, 8; for M >= 16 the branch outputs go to
    B200_PFB_TWOPASS  a 32 MiB scratch, then through the library's reverse FFT, in chunks of 4 Mi input samples,
                    and pfb_slice_kernel copies a channel slice out of the full result.
After every work() call pfb_tail_kernel keeps the last (P - 1) M input samples as the next call's history.
The single-pass kernels are persistent: 2 CTAs per SM (1 for M >= 128) over tiles of 64 frames (M = 64) or
4096 samples; the first tile of a call reads the history, interior tiles arrive by bulk copy when the input
is 16-byte aligned, the last tile is ragged.

Every case uses random asymmetric taps (a prototype used back to front gives the same answer on symmetric
taps) and checks, per output frame and relative to the RMS of that frame's M reference channels: the
relative RMS error, the worst single channel, that every value is finite, and that the output buffer is
untouched before and after the n_frames * ch_count items the call owns."""
import functools

import numpy as np
import pytest

import oracle as o
from conftest import cplx

gpu = pytest.mark.gpu

TOL_RMS = 1e-5             # per frame, relative RMS error
TOL_CH = 1e-4              # per frame, worst channel / frame RMS
SENTINEL = 0x7FBADBAD      # a float32 NaN: an output item the kernel fails to write cannot pass either
LEAD_ITEMS = 32            # sentinel items in front of the output, plus the misalignment under test
GUARD_ITEMS = 8192         # sentinel items behind it: more than a whole tile of any family
TWOPASS = {"B200_PFB_TWOPASS": "1"}
ONEBUF = {"B200_PFB_ONEBUF": "1"}
KMAJOR = {"B200_PFBT_MN": "0"}
SWITCH_IDS = {"B200_PFB_TWOPASS": "twopass", "B200_PFB_ONEBUF": "onebuf", "B200_PFBT_MN": "kmajor"}
# the largest P of the single-pass kernels and of pfb_generic_kernel (shared-memory checks of b200_pfb_create)
SINGLE_PASS_MAX_P = {4: 856, 8: 428, 16: 820, 32: 408, 64: 204, 128: 100, 256: 48}
GENERIC_MAX_P = {4: 3328, 8: 1664, 16: 832, 32: 416, 128: 104, 256: 52}
TWOPASS_CHUNK = 4 << 20    # input samples per branch-filter + FFT chunk of the two-pass form (32 MiB of scratch)


def _nb():
    import newsched_b200 as nb
    return nb


def _sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _generic(M, P, env):
    return "B200_PFB_TWOPASS" in env or P > SINGLE_PASS_MAX_P[M]


def _frames(torch, M, P, env, sweeps=2):
    """Single-pass kernels: `sweeps` full sweeps of the persistent grid plus two tiles and a partial one, so
    some CTAs loop sweeps + 1 times, one tile reads the history and the last is ragged. pfb_generic_kernel
    (one CTA per tile, no persistent loop): five tiles and a partial one, and at least twice the history."""
    TT = 64 if M == 64 else 4096 // M
    if _generic(M, P, env):
        return 5 * TT + TT // 3 + 1 + 2 * P
    grid = (1 if M >= 128 else 2) * _sms(torch)
    return (sweeps * grid + 2) * TT + TT // 3 + 1


def _taps(rng, M, P, kind="random"):
    if kind == "firwin":
        import scipy.signal as sig
        return sig.firwin(M * P, 1.0 / M).astype(np.float32)
    h = (rng.uniform(-1, 1, M * P) / np.sqrt(M * P)).astype(np.float32)
    assert M * P == 1 or not np.array_equal(h, h[::-1])
    return h


def _device_input(torch, x, offset):
    """x on the device, `offset` complex items into its allocation (offset 1: 8-byte but not 16-byte aligned)."""
    buf = torch.empty(x.size + offset, dtype=torch.complex64, device="cuda")
    buf[offset:].copy_(torch.from_numpy(x))
    xd = buf[offset:]
    assert xd.data_ptr() % 16 == 8 * offset % 16
    return xd


class _Guarded:
    """An output view of [n_frames, ch] complex items inside a device buffer pre-filled with the SENTINEL bit
    pattern. misaligned: the view starts 8 bytes off a 16-byte boundary."""

    def __init__(self, torch, n_frames, ch, misaligned=False):
        self.lead = LEAD_ITEMS + (1 if misaligned else 0)
        self.n = n_frames * ch
        self.buf = torch.full((2 * (self.lead + self.n + GUARD_ITEMS),), SENTINEL, dtype=torch.int32, device="cuda")
        self.view = self.buf.view(torch.complex64)[self.lead:self.lead + self.n].view(n_frames, ch)
        assert self.view.data_ptr() % 16 == (8 if misaligned else 0)

    def check_untouched(self):
        before, after = self.buf[:2 * self.lead], self.buf[2 * (self.lead + self.n):]
        bad = (before != SENTINEL).nonzero()
        assert bad.numel() == 0, f"written before the output: word {int(bad[0])} of {before.numel()}"
        bad = (after != SENTINEL).nonzero()
        assert bad.numel() == 0, f"written past the output: word {int(bad[0])} after it"


def _check_frames(y, ref, cols=None, record_property=None):
    """y: [n, ch] output frames; ref: [n, M] reference frames, cols: the channels of ref that y holds.
    Per frame, relative to the RMS of the frame's M reference channels (so a one-channel slice is judged by the
    same yardstick as the whole frame): relative RMS error and worst single channel. The RMS error of a
    one-channel frame is that channel's error, so only the channel bound applies to it: the tensor-core form
    (bf16x3 split) keeps whole frames within 5.3e-6 but single channels reach 1.45e-5 (measured on a B200)."""
    y = np.asarray(y)
    ref = np.asarray(ref).astype(np.complex128)
    sub = ref if cols is None else ref[:, cols]
    assert y.shape == sub.shape, (y.shape, sub.shape)
    assert np.isfinite(y.view(np.float32)).all(), \
        f"frame {int(np.argmax(~np.isfinite(y.view(np.float32)).all(axis=1)))} holds a non-finite value"
    d = np.abs(y.astype(np.complex128) - sub)
    scale = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    rel_rms = np.sqrt(np.mean(d ** 2, axis=1)) / scale
    worst_ch = d.max(axis=1) / scale
    if record_property is not None:
        record_property("worst_rel_rms", float(rel_rms.max()))
        record_property("worst_channel_ratio", float(worst_ch.max()))
    f = int(rel_rms.argmax())
    assert y.shape[1] == 1 or rel_rms[f] < TOL_RMS, f"frame {f} of {len(ref)}: relative RMS error {rel_rms[f]:.3g}"
    f = int(worst_ch.argmax())
    c = int(d[f].argmax())
    assert worst_ch[f] < TOL_CH, f"frame {f} of {len(ref)}, channel {c}: |error| / rms = {worst_ch[f]:.3g}"
    return float(rel_rms.max()), float(worst_ch.max())


def _channelizer(monkeypatch, taps, M, env, algorithm=0, cb=0, cc=0):
    """A handle created with exactly the switches in `env` set (they are read by b200_pfb_create)."""
    for k in ("B200_PFB_TWOPASS", "B200_PFB_ONEBUF", "B200_PFBT_MN", "B200_PFB_TC"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ch = _nb().PfbChannelizer(taps, M, channel_begin=cb, channel_count=cc, algorithm=algorithm)
    assert ch.algorithm == (2 if algorithm == 2 else 1)
    return ch


@functools.lru_cache(maxsize=4)
def _case_data(M, P, n_frames, taps):
    """Taps, input and oracle output of a case; the variants of one test share them."""
    rng = np.random.default_rng([M, P, n_frames, int(taps == "firwin")])
    h = _taps(rng, M, P, taps)
    x = cplx(rng, n_frames * M + M - 1)          # the trailing M - 1 items make no frame and stay unconsumed
    return h, x, o.pfb_channelizer(x, h, M)


def _run_case(torch, monkeypatch, M, P, env, n_frames, *, algorithm=0, taps="random", cb=0, cc=0, in_offset=0,
              out_misaligned=False, record_property=None):
    """One work() call on n_frames * M + (M - 1) input items, checked against the oracle. Returns the
    output frames on the host (the same inputs for every in_offset / out_misaligned / slice)."""
    h, x, ref = _case_data(M, P, n_frames, taps)
    xd = _device_input(torch, x, in_offset)
    ch = _channelizer(monkeypatch, h, M, env, algorithm, cb, cc)
    n_ch = cc or M - cb
    g = _Guarded(torch, n_frames, n_ch, out_misaligned)
    y, nc = ch.work(xd, out=g.view)
    torch.cuda.synchronize()
    assert nc == n_frames * M
    assert tuple(y.shape) == (n_frames, n_ch) and y.data_ptr() == g.view.data_ptr()
    g.check_untouched()
    yh = y.cpu().numpy()
    _check_frames(yh, ref, slice(cb, cb + n_ch), record_property)
    return yh


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ----------------------------------------------------------------------------- 0. the oracle's convention
def test_oracle_tap_convention_on_asymmetric_taps():
    """The C oracle (fp64 sums, complex64 result) against the independent numpy statement on asymmetric taps:
    equal to within the complex64 rounding of the C result plus 1e-12 of the frame RMS."""
    rng = np.random.default_rng(11)
    for M, P in ((4, 3), (8, 5), (16, 2), (64, 7), (256, 3)):
        h = _taps(rng, M, P)
        x = cplx(rng, M * 37 + 3)
        hist = cplx(rng, (P - 1) * M)
        for hh in (None, hist):
            got = o.pfb_channelizer(x, h, M, hist=hh).astype(np.complex128)
            ref = o.np_pfb_channelizer(x, h, M, hist=hh)
            scale = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1, keepdims=True))
            for part in (np.real, np.imag):
                err = np.abs(part(got) - part(ref))
                assert (err <= 2.0 ** -24 * np.abs(part(ref)) + 1e-12 * scale).all(), (M, P, float(err.max()))


# ----------------------------------------------------------------------------------------- 1. path matrix
def _row(M, P, env=None, algorithm=0, taps="random"):
    env = env or {}
    name = f"M{M}-P{P}" + "".join("-" + SWITCH_IDS[k] for k in env) + ("-tc" if algorithm == 2 else "") + \
        ("-firwin" if taps == "firwin" else "")
    return pytest.param(M, P, env, algorithm, taps, id=name)


MATRIX = (
    [_row(64, P) for P in (1, 2, 3, 4, 8, 12, 16, 20, 24, 28, 32, 33, SINGLE_PASS_MAX_P[64])]
    + [_row(64, 16, ONEBUF)]
    + [_row(64, P, env, 2) for P in (1, 3, 8, 12, 16) for env in (None, KMAJOR)]
    + [_row(M, P, env) for M in (4, 8) for P in (3, 8, 11, 16, 20) for env in (None, ONEBUF)]
    + [_row(M, P) for M in (16, 32, 128, 256) for P in (3, 8, 16, 11, 21)]      # PT 4, 8, 16, 0 (P4 12, 24)
    + [_row(M, 8, ONEBUF) for M in (128, 256)]
    + [_row(128, 60), _row(256, 33)]                                           # one tile: no room for two
    + [_row(M, 9, TWOPASS) for M in (4, 8, 16, 32, 128, 256)]
    + [_row(128, SINGLE_PASS_MAX_P[128] + 1), _row(128, GENERIC_MAX_P[128]), _row(8, SINGLE_PASS_MAX_P[8] + 1)]
    + [_row(64, 16, taps="firwin"), _row(64, 16, algorithm=2, taps="firwin"), _row(8, 16, taps="firwin"),
       _row(32, 8, taps="firwin"), _row(256, 4, taps="firwin"), _row(4, 9, TWOPASS, taps="firwin"),
       _row(16, 9, TWOPASS, taps="firwin")]
)


@gpu
@pytest.mark.parametrize("M,P,env,algorithm,taps", MATRIX)
def test_pfb_path_matrix(cuda, monkeypatch, record_property, M, P, env, algorithm, taps):
    """Each instantiation past two sweeps of its persistent grid, with a partial last tile."""
    _run_case(cuda, monkeypatch, M, P, env, _frames(cuda, M, P, env), algorithm=algorithm, taps=taps,
              record_property=record_property)


# One handle of every family: the variants below run on each.
FAMILIES = [
    pytest.param(64, 12, {}, 0, id="pfb64_reg"),
    pytest.param(64, 20, {}, 0, id="pfb64_smem"),
    pytest.param(64, 12, {}, 2, id="pfb64_tc"),
    pytest.param(64, 16, KMAJOR, 2, id="pfb64_tc_kmajor"),
    pytest.param(4, 16, {}, 0, id="pfbs4"),
    pytest.param(8, 12, {}, 0, id="pfbs8"),
    pytest.param(16, 16, {}, 0, id="pfbm16"),
    pytest.param(32, 11, {}, 0, id="pfbm32"),
    pytest.param(128, 8, {}, 0, id="pfbm128"),
    pytest.param(256, 33, {}, 0, id="pfbm256_onetile"),
    pytest.param(8, 10, TWOPASS, 0, id="direct8"),
    pytest.param(16, 9, TWOPASS, 0, id="twopass16"),
    pytest.param(128, 101, {}, 0, id="twopass128"),
]


# ------------------------------------------------------------------------------------------ 2. alignment
@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_input_8_byte_aligned(cuda, monkeypatch, record_property, M, P, env, algorithm):
    """Input one complex item past a 16-byte boundary: every tile is fetched element-wise instead of by bulk
    copy. Same arithmetic per frame, so bit-equal to the aligned call."""
    n = _frames(cuda, M, P, env, sweeps=1)
    a = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm)
    b = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm, in_offset=1, record_property=record_property)
    assert np.array_equal(_bits(a), _bits(b))


@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_output_8_byte_aligned(cuda, monkeypatch, record_property, M, P, env, algorithm):
    """Output one complex item past a 16-byte boundary: pfbs_kernel stores item by item instead of 16 bytes at
    a time (out16 = 0), the FFT of the two-pass form takes its unaligned path."""
    n = _frames(cuda, M, P, env, sweeps=1)
    a = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm)
    b = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm, out_misaligned=True,
                  record_property=record_property)
    assert np.array_equal(_bits(a), _bits(b))


# -------------------------------------------------------------------------------------- 3. channel slices
def _slices(M):
    return {"first": (0, 1), "last": (M - 1, 1), "middle": (M // 3, M // 3)}


@gpu
@pytest.mark.parametrize("which", ["first", "last", "middle"])
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_channel_slice(cuda, monkeypatch, record_property, M, P, env, algorithm, which):
    """A channel slice against the oracle's columns, and bit-equal to the same columns of the whole output."""
    cb, cc = _slices(M)[which]
    n = _frames(cuda, M, P, env, sweeps=1)
    full = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm)
    part = _run_case(cuda, monkeypatch, M, P, env, n, algorithm=algorithm, cb=cb, cc=cc,
                     record_property=record_property)
    assert np.array_equal(_bits(part), _bits(full[:, cb:cb + cc]))


@gpu
@pytest.mark.parametrize("which", ["full", "first", "last", "middle"])
def test_pfb_two_pass_over_several_chunks(cuda, monkeypatch, record_property, which):
    """More than two chunks of the two-pass form at M = 16: each chunk's FFT output (whole frames) or slice
    (pfb_slice_kernel) lands at its own frame offset in the output."""
    M, P = 16, 9
    cb, cc = (0, 0) if which == "full" else _slices(M)[which]
    n = (2 * TWOPASS_CHUNK + TWOPASS_CHUNK // 3) // M + 5
    _run_case(cuda, monkeypatch, M, P, TWOPASS, n, cb=cb, cc=cc, record_property=record_property)


# ---------------------------------------------------------------------------------- 4. streams, segments
def _family_input(torch, M, P, env, sweeps=1, seed=0):
    rng = np.random.default_rng([M, P, 77, seed])
    h = _taps(rng, M, P)
    n = _frames(torch, M, P, env, sweeps=sweeps)
    x = cplx(rng, n * M + M - 1)
    return h, x, torch.from_numpy(x).cuda(), n


@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_stream_without_host_sync(cuda, monkeypatch, M, P, env, algorithm):
    """work() calls queued back to back on one stream, as a flowgraph runs them: each call's dependent launch
    reads the history pfb_tail_kernel of the call before it wrote. Six one-frame calls first, so the history
    of P - 1 frames spans several calls; chunks that end mid-frame leave their last items to the next call.
    Bit-equal to one call over the whole input."""
    torch = cuda
    h, x, xd, n = _family_input(torch, M, P, env)
    one, nc = _channelizer(monkeypatch, h, M, env, algorithm).work(xd)
    assert nc == n * M
    ch = _channelizer(monkeypatch, h, M, env, algorithm)
    out = torch.full((n, M), float("nan"), dtype=torch.complex64, device="cuda")
    TT = 64 if M == 64 else 4096 // M
    pos = f = 0
    for k, nf in enumerate([1] * 6 + [2, 3, TT + 3, 5, 2 * TT - 1, n]):
        extra = (k % 3) * (M // 4)                              # 0, M/4 or M/2 items past the last whole frame
        seg = xd[pos:pos + nf * M + extra]
        want = seg.numel() // M
        y, c = ch.work(seg, out=out[f:f + want])
        assert c == want * M and y.shape[0] == want
        pos += c
        f += want
        if f == n:
            break
    assert f == n and pos == n * M
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(one.cpu().numpy()))
    _check_frames(one.cpu().numpy(), o.pfb_channelizer(x, h, M))


@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_reset_equals_fresh_handle(cuda, monkeypatch, M, P, env, algorithm):
    torch = cuda
    h, x, xd, n = _family_input(torch, M, P, env)
    ch = _channelizer(monkeypatch, h, M, env, algorithm)
    ch.work(xd[n * M // 2:])                                   # leaves a non-zero history behind
    ch.reset()
    y, _ = ch.work(xd)
    fresh, _ = _channelizer(monkeypatch, h, M, env, algorithm).work(xd)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(y.cpu().numpy()), _bits(fresh.cpu().numpy()))


@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_segment_with_halo_equals_stream(cuda, monkeypatch, M, P, env, algorithm):
    """work_segment over the second half of the input with the (P - 1) M items before it as the halo: the
    same frames, bit for bit, as the stream, twice over."""
    torch = cuda
    h, x, xd, n = _family_input(torch, M, P, env)
    y, _ = _channelizer(monkeypatch, h, M, env, algorithm).work(xd)
    cut = n // 2 + 3
    assert cut >= P - 1
    ch = _channelizer(monkeypatch, h, M, env, algorithm)
    halo = xd[(cut - (P - 1)) * M:cut * M] if P > 1 else None
    seg = ch.work_segment(xd[cut * M:], halo=halo)
    again = ch.work_segment(xd[cut * M:], halo=halo)
    torch.cuda.synchronize()
    assert seg.shape[0] == n - cut
    assert np.array_equal(_bits(seg.cpu().numpy()), _bits(y[cut:].cpu().numpy()))
    assert np.array_equal(_bits(again.cpu().numpy()), _bits(seg.cpu().numpy()))


@gpu
@pytest.mark.parametrize("M,P,env,algorithm", FAMILIES)
def test_pfb_segment_without_halo(cuda, monkeypatch, record_property, M, P, env, algorithm):
    """work_segment with halo=None: the oracle with zero history, whatever the handle ran before."""
    torch = cuda
    h, x, xd, n = _family_input(torch, M, P, env)
    ch = _channelizer(monkeypatch, h, M, env, algorithm)
    ch.work(xd)                                                 # a non-zero history the segment must not read
    cut = n // 3 + 1
    seg = ch.work_segment(xd[cut * M:])
    torch.cuda.synchronize()
    _check_frames(seg.cpu().numpy(), o.pfb_channelizer(x[cut * M:], h, M), record_property=record_property)


# ---------------------------------------------------------------------------------- 5. coexisting handles
COEXIST = [
    pytest.param((64, 28, {}), (64, 20, {}), id="pfb64<0>-P28-P20"),
    pytest.param((16, 20, {}), (16, 12, {}), id="pfbm<16,0>-P20-P12"),
    pytest.param((8, 20, {}), (8, 12, {}), id="pfbs<8,0>-P20-P12"),
    pytest.param((16, 8, TWOPASS), (4, 8, TWOPASS), id="generic-M16-M4"),
    pytest.param((64, 16, {}), (64, 16, ONEBUF), id="pfb64<16>-twotiles-onetile"),
]


@gpu
@pytest.mark.parametrize("big,small", COEXIST)
def test_pfb_handles_of_different_sizes_coexist(cuda, monkeypatch, big, small):
    """Two live handles on one instantiation, the one with more shared memory created first, then run
    interleaved as two channelizers of one flowgraph would: the kernel's shared-memory limit must not be the
    one the last handle needed."""
    torch = cuda
    runs = []
    for i, (M, P, env) in enumerate((big, small)):
        rng = np.random.default_rng([M, P, i, 5])
        h = _taps(rng, M, P)
        n = _frames(torch, M, P, env, sweeps=1)
        x = cplx(rng, 2 * n * M)
        runs.append((M, h, x, torch.from_numpy(x).cuda(), n, _channelizer(monkeypatch, h, M, env)))
    outs = [[], []]
    for part in range(2):
        for i, (M, h, x, xd, n, ch) in enumerate(runs):
            outs[i].append(ch.work(xd[part * n * M:(part + 1) * n * M])[0])
    torch.cuda.synchronize()
    for (M, h, x, xd, n, ch), y in zip(runs, outs):
        _check_frames(torch.cat(y).cpu().numpy(), o.pfb_channelizer(x, h, M))


# ------------------------------------------------------------------------------- 6. beyond 32-bit offsets
BIG = [
    pytest.param(64, 16, {}, id="pfb64"),
    pytest.param(256, 4, {}, id="pfbm256"),
    pytest.param(4, 16, {}, id="pfbs4"),
    pytest.param(16, 8, TWOPASS, id="twopass16"),
]


@gpu
@pytest.mark.parametrize("M,P,env", BIG)
def test_pfb_beyond_32_bit_offsets(cuda, monkeypatch, record_property, M, P, env):
    """2^29 + 2^16 + 5 input samples (4 GiB and a little more in, as much out): frames around the byte offsets
    2^31 and 2^32 of input and output, the first and the last frames, against the numpy oracle with the
    history in front of them. The whole output is finite and nothing around it is written."""
    torch = cuda
    n_in = (1 << 29) + (1 << 16) + 5
    n = n_in // M
    rng = np.random.default_rng([M, P, 29])
    h = _taps(rng, M, P)
    gen = torch.Generator(device="cuda").manual_seed(M * 1000 + P)
    xd = torch.view_as_complex(torch.rand(n_in, 2, device="cuda", generator=gen).mul_(2).sub_(1))
    ch = _channelizer(monkeypatch, h, M, env)
    g = _Guarded(torch, n, M)
    y, nc = ch.work(xd, out=g.view)
    torch.cuda.synchronize()
    assert nc == n * M and y.shape[0] == n
    g.check_untouched()
    assert bool(torch.isfinite(torch.view_as_real(y)).all())
    worst = []
    for byte in (0, 1 << 31, 1 << 32, n * M * 8):
        f = byte // (8 * M)
        f0, f1 = max(f - 70, 0), min(f + 70, n)
        assert f0 == 0 or f0 >= P - 1
        hist = xd[(f0 - (P - 1)) * M:f0 * M].cpu().numpy() if f0 else None
        ref = o.np_pfb_channelizer(xd[f0 * M:f1 * M].cpu().numpy(), h, M, hist=hist)
        worst.append(_check_frames(y[f0:f1].cpu().numpy(), ref))
    record_property("worst_rel_rms", max(w[0] for w in worst))
    record_property("worst_channel_ratio", max(w[1] for w in worst))
    del xd, y, g
    torch.cuda.empty_cache()


# -------------------------------------------------------------------------------- 7. create-time checks
def _rejects(monkeypatch, match, taps, M, env=None, **kw):
    nb = _nb()
    before = nb.launch_count()
    with pytest.raises(nb.B200Error, match=match):
        _channelizer(monkeypatch, taps, M, env or {}, **kw)
    assert nb.launch_count() == before


@gpu
@pytest.mark.parametrize("M", [2, 3, 6, 512])
def test_pfb_create_rejects_channel_count(cuda, monkeypatch, M):
    _rejects(monkeypatch, "power of two", np.full(4 * M, 0.1, np.float32), M)


@gpu
@pytest.mark.parametrize("cb,cc", [(-1, 0), (-1, 4), (64, 0), (60, 5), (0, 65)])
def test_pfb_create_rejects_bad_slice(cuda, monkeypatch, cb, cc):
    _rejects(monkeypatch, "bad channel slice", np.full(64 * 4, 0.1, np.float32), 64, cb=cb, cc=cc)


@gpu
@pytest.mark.parametrize("M,P,env", [(64, SINGLE_PASS_MAX_P[64] + 1, {}), (128, GENERIC_MAX_P[128] + 1, {}),
                                     (16, GENERIC_MAX_P[16] + 1, TWOPASS)])
def test_pfb_create_rejects_too_many_taps(cuda, monkeypatch, M, P, env):
    _rejects(monkeypatch, "taps_per_channel too large", np.full(M * P, 0.01, np.float32), M, env)


@gpu
@pytest.mark.parametrize("algorithm", [3, -1])
def test_pfb_create_rejects_algorithm(cuda, monkeypatch, algorithm):
    _rejects(monkeypatch, "algorithm must be", np.full(64 * 4, 0.1, np.float32), 64, algorithm=algorithm)


@gpu
@pytest.mark.parametrize("M,P", [(16, 4), (128, 8), (64, 17)])
def test_pfb_create_rejects_tensor_core_form(cuda, monkeypatch, M, P):
    _rejects(monkeypatch, "tensor-core DFT form needs", np.full(M * P, 0.01, np.float32), M, algorithm=2)

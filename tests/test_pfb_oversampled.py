"""CPU: the oversampled analysis bank (oversample 2 and 4) as the tests state it, and the create-time
rejections of b200_pfb_create, which come before any CUDA call.

With hop D = M / OS and t the frame index since the stream start (zeros before it):
    z_c[t] = e^{-j 2 pi c tD/M} sum_{n<MP} h[n] e^{+j 2 pi n c/M} x[tD + D-1-n]          (np_pfb_os_direct)
Writing t = OS s + q, frame t reads x[sM + (q+1)D - 1 - n]: frame s of the critically sampled bank over x
delayed by M - (q+1)D samples. pfb_os_reference builds the oversampled bank from OS runs of the fp64
critically sampled oracle (oracle.pfb_channelizer: fp64 sums, complex64 result) and the phase factor, so the
GPU tests check against the same oracle as the critically sampled ones; the numpy direct formula is the
independent statement it is held to."""
import ctypes as C

import numpy as np
import pytest

import oracle as o
from conftest import cplx

B200_ERR_ARG, B200_ERR_UNSUPPORTED = -1, -4


def pfb_os_reference(x, taps, M, oversample=1, hist=None, frame0=0):
    """[len(x) // D, M] complex64 frames of the bank with hop D = M / oversample; hist: the P M - D samples
    before x[0] (None: zeros); frame0: the frame index of the first output (only its value mod oversample
    matters). At oversample 1 this is oracle.pfb_channelizer itself."""
    taps = np.asarray(taps, np.float32)
    P = taps.size // M
    D = M // oversample
    x = np.asarray(x, np.complex64)
    if oversample == 1:
        return o.pfb_channelizer(x, taps, M, hist=hist)
    pre = np.zeros(P * M - D, np.complex64) if hist is None else np.asarray(hist, np.complex64)
    assert pre.size == P * M - D
    ext = np.concatenate([pre, x])                      # ext[e] = x[e - (P M - D)]
    n_t = x.size // D
    out = np.empty((n_t, M), np.complex64)
    c = np.arange(M)
    for q in range(oversample):
        t = np.arange(q, n_t, oversample)
        if t.size == 0:
            continue
        lo = (P - 1) * M + q * D                        # x delayed by M - (q+1) D samples, and its history
        y = o.pfb_channelizer(ext[lo:], taps, M, hist=ext[lo - (P - 1) * M:lo])[: t.size]
        rot = np.exp(-2j * np.pi * np.outer((frame0 + t) * D % M, c) / M)
        out[t] = (y.astype(np.complex128) * rot).astype(np.complex64)
    return out


def np_pfb_os_direct(x, taps, M, D, hist=None, frame0=0):
    """The direct (non-polyphase) statement of the analysis bank with hop D, frame t0 = frame0 + t:
    z_c[t] = e^{-j 2 pi c t0 D / M} sum_{n<MP} h[n] e^{+j 2 pi n c / M} x[tD + D-1-n]."""
    taps = np.asarray(taps, np.float64)
    T = taps.size
    xd = np.asarray(x, np.complex128)
    pre = np.zeros(T - D, np.complex128) if hist is None else np.asarray(hist, np.complex128)
    assert pre.size == T - D
    xx = np.concatenate([pre, xd])
    n_t = xd.size // D
    n = np.arange(T)
    c = np.arange(M)
    t = np.arange(n_t)
    seg = xx[(T - D) + t[:, None] * D + (D - 1) - n[None, :]]             # x[tD + D-1-n]
    E = taps[:, None] * np.exp(2j * np.pi * np.outer(n, c) / M)
    rot = np.exp(-2j * np.pi * np.outer((frame0 + t) * D % M, c) / M)
    return rot * (seg @ E)


def _taps(rng, M, P):
    h = (rng.uniform(-1, 1, M * P) / np.sqrt(M * P)).astype(np.float32)
    assert not np.array_equal(h, h[::-1])
    return h


def _assert_reference_close(got, ref):
    """complex64 rounding of the critically sampled oracle (rotated in fp64) plus 1e-12 of the frame RMS"""
    got = np.asarray(got).astype(np.complex128)
    scale = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1, keepdims=True))
    err = np.abs(got - ref)
    assert (err <= 2.0 ** -23 * np.abs(ref) + 1e-12 * scale).all(), float((err / scale).max())


@pytest.mark.parametrize("OS", [2, 4])
@pytest.mark.parametrize("M,P", [(16, 3), (64, 5), (16, 1)])
@pytest.mark.parametrize("frame0", [0, 1, 3, 6])
def test_reference_matches_direct_statement(M, P, OS, frame0):
    """The reference built from the critically sampled oracle against the numpy direct formula, with and
    without a history."""
    rng = np.random.default_rng([M, P, OS, frame0])
    D = M // OS
    h = _taps(rng, M, P)
    x = cplx(rng, 41 * D + D - 1)
    hist = cplx(rng, P * M - D)
    for hh in (None, hist):
        got = pfb_os_reference(x, h, M, OS, hist=hh, frame0=frame0)
        assert got.shape == (41, M)
        _assert_reference_close(got, np_pfb_os_direct(x, h, M, D, hist=hh, frame0=frame0))


@pytest.mark.parametrize("M,P", [(4, 3), (16, 2), (64, 7), (256, 3)])
def test_direct_statement_at_hop_m_is_the_critically_sampled_bank(M, P):
    """At D = M the direct formula is SURVEY 8(c): it agrees with the existing numpy statement, and the
    reference is the critically sampled oracle."""
    rng = np.random.default_rng([M, P, 1])
    h = _taps(rng, M, P)
    x = cplx(rng, M * 29 + 5)
    hist = cplx(rng, (P - 1) * M)
    old = o.pfb_channelizer(x, h, M, hist=hist)
    assert np.array_equal(pfb_os_reference(x, h, M, 1, hist=hist).view(np.uint32), old.view(np.uint32))
    assert np.abs(np_pfb_os_direct(x, h, M, M, hist=hist) - o.np_pfb_channelizer(x, h, M, hist=hist)).max() \
        < 1e-12 * np.abs(old).max()


def _firwin(M, P):
    import scipy.signal as sig
    return sig.firwin(M * P, 1.0 / M).astype(np.float32)


@pytest.mark.parametrize("OS", [2, 4])
def test_centre_tone_is_a_constant_phasor(OS):
    """A tone at channel c0's centre frequency is at baseband in channel c0: a constant phasor once the filter
    has filled, and the strongest channel."""
    M, P, c0 = 16, 8, 5
    n = np.arange(300 * M)
    x = np.exp(2j * np.pi * c0 * n / M)
    h = _firwin(M, P)
    for y in (np_pfb_os_direct(x, h, M, M // OS), pfb_os_reference(x, h, M, OS)):
        y = np.asarray(y)[P * OS:]
        assert int(np.abs(y).mean(axis=0).argmax()) == c0
        z = y[:, c0].astype(np.complex128)
        assert np.ptp(np.angle(z)) < 1e-5 and np.ptp(np.abs(z)) < 1e-5 * np.abs(z).mean()


@pytest.mark.parametrize("OS", [2, 4])
def test_half_bin_tone_is_equal_in_both_neighbours(OS):
    """A tone halfway between channels c0 and c0 + 1 comes out of both at the same magnitude (about half of
    the passband gain): the signal a critically sampled bank would alias is whole in either channel."""
    M, P, c0 = 16, 8, 5
    n = np.arange(300 * M)
    x = np.exp(2j * np.pi * (c0 + 0.5) * n / M)
    y = np.abs(np_pfb_os_direct(x, _firwin(M, P), M, M // OS))[P * OS:]
    a, b = y[:, c0].mean(), y[:, c0 + 1].mean()
    assert abs(a - b) < 1e-9 * a and 0.4 < a < 0.6
    assert y[:, [c for c in range(M) if c not in (c0, c0 + 1)]].max() < 0.05 * a


@pytest.mark.parametrize("OS", [2, 4])
@pytest.mark.parametrize("M,P", [(16, 4), (64, 3)])
def test_chunked_oracle_with_carried_phase_equals_one_shot(M, P, OS):
    """Chunks that end on odd frames, each with the previous P*M - D samples as history and its first frame
    index as frame0, give the one-shot reference bit for bit; restarting the phase at 0 does not."""
    rng = np.random.default_rng([M, P, OS, 9])
    D = M // OS
    h = _taps(rng, M, P)
    x = cplx(rng, 97 * D)
    one = pfb_os_reference(x, h, M, OS)
    parts, wrong, f = [], [], 0
    for nf in (1, 3, 2, 5, 7, 11, 13, 55):
        lo = f * D
        hist = np.concatenate([np.zeros(max(0, P * M - D - lo), np.complex64), x[max(0, lo - (P * M - D)):lo]])
        seg = x[lo:lo + nf * D]
        parts.append(pfb_os_reference(seg, h, M, OS, hist=hist, frame0=f))
        wrong.append(pfb_os_reference(seg, h, M, OS, hist=hist, frame0=0))
        f += nf
    assert f == 97
    assert np.array_equal(np.concatenate(parts).view(np.uint32), one.view(np.uint32))
    assert np.abs(np.concatenate(wrong) - one).max() > 0.1 * np.abs(one).max()


# ------------------------------------------------------------------------------ create-time rejections
def single_pass_max_p(M, OS):
    """The largest P (a multiple of 4) whose one input tile fits the 220 KiB of b200_pfb_create: the tile is
    TT + 4*ceil(P/4)*OS - 1 rows of D = M/OS samples, TT = 4096/M frames (pfb_single_pass_smem in pfb.cu)."""
    def smem(P4):
        TT = 4096 // M
        x = 8 * (TT + P4 * OS - 1) * (M // OS)
        if M == 64:
            return x + 8 * 64 * 68 + (0 if P4 in (4, 8, 12, 16, 24, 32) else 4 * P4 * 64)
        return x + 8 * TT * 17 * (M // 16) + 4 * P4 * M + 16
    p = 0
    while smem(p + 4) <= 220 * 1024:
        p += 4
    return p


def _create(M, P, os_, cb=0, cc=0):
    import newsched_b200 as nb
    taps = np.full(M * P, 0.01, np.float32)
    p = nb._PfbParams(taps.ctypes.data_as(C.POINTER(C.c_float)), M, P, cb, cc, os_)
    h = C.c_void_p()
    rc = nb.lib().b200_pfb_create(C.byref(p), C.byref(h))
    return rc, nb.lib().b200_last_error().decode(), h


@pytest.mark.parametrize("os_", [-1, 3, 5, 8, 16])
def test_create_rejects_unknown_oversample(os_):
    rc, msg, h = _create(64, 16, os_)
    assert rc == B200_ERR_ARG and not h.value
    assert "oversample" in msg and "2 or 4" in msg, msg


@pytest.mark.parametrize("os_", [2, 4])
@pytest.mark.parametrize("M", [4, 8])
def test_create_rejects_oversampling_below_16_channels(M, os_):
    rc, msg, h = _create(M, 8, os_)
    assert rc == B200_ERR_UNSUPPORTED and not h.value
    assert "16, 32, 64, 128 or 256 channels" in msg, msg


@pytest.mark.parametrize("os_", [2, 4])
@pytest.mark.parametrize("M", [16, 32, 64, 128, 256])
def test_create_rejects_taps_beyond_the_single_pass_tile(M, os_):
    pmax = single_pass_max_p(M, os_)
    rc, msg, h = _create(M, pmax + 1, os_)
    assert rc == B200_ERR_UNSUPPORTED and not h.value
    assert f"at most {pmax}" in msg, msg


def test_bad_slice_is_still_reported_first():
    rc, msg, _ = _create(64, 16, 2, cb=60, cc=5)
    assert rc == B200_ERR_ARG and "bad channel slice" in msg

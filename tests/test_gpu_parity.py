"""GPU parity tests: the CUDA path (through the C-ABI) against the CPU oracle on the same seeded
inputs, against the committed golden vectors, and -- at BASELINE sizes -- through
size-independent properties.  Bars: bit-exact for copy / integer / indexing / decimation phase /
multiply_const k=1; <= 1e-6 relative for multiply_const and complex_to_mag (<= 2 ulp);
<= 1e-5 relative RMS for FIR, FFT and the channelizer (north_star)."""
import numpy as np
import pytest

import oracle as o
from conftest import cplx

pytestmark = pytest.mark.gpu

TOL_RMS = 1e-5   # north_star: FIR / FFT within 1e-5 relative RMS (fp32)
TOL_EW = 1e-6    # elementwise fp32 ops


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


# ------------------------------------------------------------------------------- copy
def test_copy_reference_ramp_bit_exact(cuda, golden):
    import newsched_b200 as nb
    x = golden["ramp_qa_cuda_copy"]            # qa_scheduler_mt_cuda_copy.cpp:24-28
    y = host(nb.copy(nb.copy(dev(cuda, x))))   # two chained copies like the reference test
    assert np.array_equal(y.view(np.uint8), x.view(np.uint8))


@pytest.mark.parametrize("nbytes", [0, 1, 15, 16, 17, 4095, 65536 + 3, (1 << 22) + 5])
@pytest.mark.parametrize("off_in,off_out", [(0, 0), (8, 8), (8, 0), (4, 12), (1, 3), (3, 3), (2, 7)])
def test_copy_any_alignment_bit_exact(cuda, nbytes, off_in, off_out):
    import newsched_b200 as nb
    rng = np.random.default_rng(nbytes + off_in * 31 + off_out)
    src = rng.integers(0, 256, nbytes + 64, dtype=np.uint8)
    d_src = dev(cuda, src)
    d_dst = cuda.full((nbytes + 64,), 0xA5, dtype=cuda.uint8, device="cuda")
    nb._check(nb.lib().b200_copy(d_dst.data_ptr() + off_out, d_src.data_ptr() + off_in, nbytes,
                                 nb._stream()))
    got = host(d_dst)
    assert np.array_equal(got[off_out:off_out + nbytes], src[off_in:off_in + nbytes])
    assert (got[:off_out] == 0xA5).all() and (got[off_out + nbytes:] == 0xA5).all()  # no overrun


def test_copy_full_size_checksum(cuda):
    import newsched_b200 as nb
    n = 1 << 24                                 # config 1 size: 16M complex64
    x = cuda.randn(n, 2, device="cuda").view(cuda.uint8).flatten()
    y = nb.copy(x)
    assert cuda.equal(x, y)


def test_copy_and_fir_beyond_32bit_byte_counts(cuda):
    """Sizes past 2^31 bytes per call: the reference computes byte counts in `int`
    (copy.hpp:37 `int size = n_items * _itemsize`) and is limited to < 2 GiB per call; the
    C-ABI takes size_t / int64 and indexes in 64 bits."""
    import newsched_b200 as nb
    n = (1 << 28) + 12345                      # complex64 samples: 2 GiB + a ragged tail
    x = cuda.empty(n, dtype=cuda.complex64, device="cuda")
    xr = cuda.view_as_real(x)
    xr[:, 0] = cuda.arange(n, device="cuda", dtype=cuda.float32) % 4093.0
    xr[:, 1] = -(cuda.arange(n, device="cuda", dtype=cuda.float32) % 611.0)
    y = nb.copy(x)
    assert cuda.equal(cuda.view_as_real(y)[-100000:], xr[-100000:]) and cuda.equal(y[:1000], x[:1000])
    assert float(cuda.view_as_real(y)[:, 0].double().sum()) == float(xr[:, 0].double().sum())
    del y
    taps = np.zeros(64, np.float32)
    taps[5] = 1.0                              # pure delay by 5 samples: exact
    z, nc = nb.FirFilter(taps, 1).work(x)
    assert nc == n and cuda.equal(z[5:], x[:-5]) and not bool(z[:5].abs().any())


# --------------------------------------------------------------------- multiply_const
def test_multiply_const_k1_exact(cuda, golden):
    import newsched_b200 as nb
    x = golden["ramp_qa_scheduler_mt"]          # qa_scheduler_mt.cpp:86-88, k = 1.0 -> exact
    d = dev(cuda, x)
    for _ in range(16):                          # qa_block_grouping.cpp chains up to 16 blocks
        d = nb.multiply_const(d, 1.0 + 0j)
    assert np.array_equal(host(d), x)


@pytest.mark.parametrize("n", [1, 2, 3, 1023, 1 << 16, (1 << 20) + 7])
def test_multiply_const_cc_matches_oracle(cuda, n):
    import newsched_b200 as nb
    rng = np.random.default_rng(n)
    x = cplx(rng, n + 1)
    k = 0.5 - 0.25j
    for off in (0, 1):                           # 16-byte aligned and 8-byte-only aligned
        xs = x[off:off + n]
        d = dev(cuda, x)[off:off + n]
        y = host(nb.multiply_const(d, k))
        ref = o.multiply_const(xs, k)
        assert np.array_equal(y, ref), "non-fused fp32 product must be bit-identical to the oracle"


def test_multiply_const_ff_ss_ii(cuda):
    import newsched_b200 as nb
    rng = np.random.default_rng(11)
    xf = rng.uniform(-4, 4, 100003).astype(np.float32)
    assert np.array_equal(host(nb.multiply_const(dev(cuda, xf), 3.25)), o.multiply_const(xf, 3.25))
    xs = rng.integers(-32768, 32767, 100001, dtype=np.int16)
    assert np.array_equal(host(nb.multiply_const(dev(cuda, xs), -7)), o.multiply_const(xs, -7))
    xi = rng.integers(-2**31, 2**31 - 1, 100002, dtype=np.int32)
    assert np.array_equal(host(nb.multiply_const(dev(cuda, xi), 1000003)), o.multiply_const(xi, 1000003))


def test_multiply_const_golden(cuda, golden):
    import newsched_b200 as nb
    y = host(nb.multiply_const(dev(cuda, golden["mulc_x"]), complex(golden["mulc_k"][0])))
    assert o.rel_rms(y, golden["mulc_y64"]) < TOL_EW


@pytest.mark.parametrize("n", [1, 3, 4097, (1 << 20) + 5])
def test_two_input_multiply_add(cuda, n):
    import newsched_b200 as nb
    rng = np.random.default_rng(n + 9)
    a, b = cplx(rng, n + 1), cplx(rng, n + 1)
    for off in (0, 1):
        da, db = dev(cuda, a)[off:off + n], dev(cuda, b)[off:off + n]
        assert np.array_equal(host(nb.multiply(da, db)), o.multiply(a[off:off + n], b[off:off + n]))
        assert np.array_equal(host(nb.add(da, db)), o.add(a[off:off + n], b[off:off + n]))
        ar, br = np.ascontiguousarray(a.real), np.ascontiguousarray(b.imag)
        dar, dbr = dev(cuda, ar)[off:off + n], dev(cuda, br)[off:off + n]
        assert np.array_equal(host(nb.multiply(dar, dbr)), o.multiply(ar[off:off + n], br[off:off + n]))
        assert np.array_equal(host(nb.add(dar, dbr)), o.add(ar[off:off + n], br[off:off + n]))


# --------------------------------------------------------------------- complex_to_mag
@pytest.mark.parametrize("n", [1, 5, 4096, (1 << 20) + 3])
def test_complex_to_mag(cuda, n):
    import newsched_b200 as nb
    rng = np.random.default_rng(n)
    x = cplx(rng, n + 1)
    for off in (0, 1):
        d = dev(cuda, x)[off:off + n]
        y = host(nb.complex_to_mag(d))
        assert np.array_equal(y, o.complex_to_mag(x[off:off + n]))  # same rounding sequence
        y2 = host(nb.complex_to_mag(d, squared=True))
        assert np.array_equal(y2, o.complex_to_mag(x[off:off + n], squared=True))


def test_complex_to_mag_golden(cuda, golden):
    import newsched_b200 as nb
    y = host(nb.complex_to_mag(dev(cuda, golden["mulc_x"])))
    assert o.rel_rms(y, golden["mag_y64"]) < TOL_EW


# ------------------------------------------------------------------------------- FIR
@pytest.mark.parametrize("name", ["fir_a", "fir_b", "fir_c"])
def test_fir_golden(cuda, golden, name):
    import newsched_b200 as nb
    taps, x, D = golden[name + "_taps"], golden[name + "_x"], int(golden[name + "_D"][0])
    T = taps.size
    f = nb.FirFilter(taps, D, is_complex=np.iscomplexobj(x))
    y, nc = f.work(dev(cuda, x))
    assert nc == (x.size // D) * D
    assert o.rel_rms(host(y), golden[name + "_y64"]) < TOL_RMS
    # preload history, then stream the rest
    f2 = nb.FirFilter(taps, D, is_complex=np.iscomplexobj(x))
    f2.set_history(dev(cuda, x[: T - 1]))
    y2, _ = f2.work(dev(cuda, x[T - 1:]))
    assert o.rel_rms(host(y2), golden[name + "_y64_hist"]) < TOL_RMS


@pytest.mark.parametrize("T,D,cplxin", [(1, 1, True), (2, 1, True), (5, 2, True), (64, 1, True),
                                        (65, 1, True), (128, 1, True), (256, 3, True),
                                        (1024, 4, True), (1000, 7, True), (64, 1, False),
                                        (63, 2, False), (513, 5, False), (64, 16, True), (300, 40, True)])
def test_fir_matches_oracle(cuda, T, D, cplxin):
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 100 + D)
    n = 40000 + 17
    x = cplx(rng, n) if cplxin else rng.uniform(-1, 1, n).astype(np.float32)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    f = nb.FirFilter(taps, D, is_complex=cplxin)
    y, nc = f.work(dev(cuda, x))
    ref = o.fir(x, taps, D)
    assert y.numel() == n // D and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS


def test_fir_impulse_and_decimation_phase_exact(cuda, golden):
    import newsched_b200 as nb
    taps = golden["fir_imp_taps"]
    imp = np.zeros(4096, np.complex64)
    imp[0] = 1
    y, _ = nb.FirFilter(taps, 1, algorithm=1).work(dev(cuda, imp))
    y = host(y)
    assert np.array_equal(y[:48].real, taps) and not y[48:].any() and not y.imag.any()
    # 48 taps at full rate are auto-routed to the tensor-core form: indexing (where the response starts and
    # ends, nothing in the imaginary plane) is exact, the values carry the bf16 hi+lo split (<= 2^-17 relative)
    f2 = nb.FirFilter(taps, 1)
    assert f2.algorithm == 2
    y2 = host(f2.work(dev(cuda, imp))[0])
    assert not y2[48:].any() and not y2.imag.any()
    assert np.allclose(y2[:48].real, taps, rtol=2.0 ** -16, atol=0)
    for D in (2, 3, 4, 7):
        yd, _ = nb.FirFilter(taps, D).work(dev(cuda, imp))
        yd = host(yd)
        k = len(taps[::D])
        assert np.array_equal(yd.real[:k], taps[::D]), "decimation phase 0: y[m] aligned to x[m*D]"
        assert not yd[k:].any()
    # an impulse at n0: the response starts at ceil(n0/D) with tap (m*D - n0)
    n0, D = 37, 4
    imp2 = np.zeros(4096, np.complex64)
    imp2[n0] = 1j
    yd = host(nb.FirFilter(taps, D).work(dev(cuda, imp2))[0])
    exp = np.zeros(1024, np.complex64)
    for m in range(1024):
        kk = m * D - n0
        if 0 <= kk < taps.size:
            exp[m] = 1j * taps[kk]
    assert np.array_equal(yd, exp)


@pytest.mark.parametrize("T,D", [(64, 1), (31, 3), (257, 4)])
def test_fir_streaming_equals_oneshot(cuda, T, D):
    import newsched_b200 as nb
    rng = np.random.default_rng(7 + T)
    n = 30000
    x = cplx(rng, n)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    ref, _ = nb.FirFilter(taps, D, algorithm=1).work(dx)   # direct form: bit-exact for any chunking
    ref = host(ref)
    for chunk in (1, T - 1 if T > 1 else 1, T, 997, 8192):
        f = nb.FirFilter(taps, D, algorithm=1)
        step = max(chunk, D)          # the scheduler re-presents unconsumed items with new ones
        outs, pos = [], 0
        while n - pos >= D:
            y, nc = f.work(dx[pos:min(pos + step, n)])
            assert nc > 0
            outs.append(host(y))
            pos += nc
        got = np.concatenate(outs)
        assert got.size == n // D
        assert np.array_equal(got, ref), f"chunk={chunk}: chunked != one-shot"


@pytest.mark.parametrize("T,D", [(2, 1), (64, 1), (65, 2), (256, 1), (1024, 4), (1000, 7), (3073, 1), (3000, 3),
                                 (3074, 1), (4096, 1), (4096, 4), (6001, 2), (1024, 8), (96, 2),
                                 (12288, 4), (13000, 4), (1024, 1), (1025, 1), (2048, 1), (6142, 1),
                                 (6143, 1), (1024, 10), (800, 12), (2048, 16), (900, 9), (1500, 14)])
def test_fir_overlap_save_matches_oracle_and_direct(cuda, T, D):
    """algorithm 3 (FFT overlap-save) against the fp64 oracle, the direct form, and itself when
    the stream is chunked or time-segmented (FFT rounding differs per blocking -> tolerance)."""
    import newsched_b200 as nb
    rng = np.random.default_rng(T + D)
    n = 3 * 4096 * 7 + 1234
    x = cplx(rng, n)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    f = nb.FirFilter(taps, D, algorithm=3)
    assert f.algorithm == 3
    y, nc = f.work(dx)
    ref = o.fir(x, taps, D)
    assert y.numel() == n // D and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS
    yd, _ = nb.FirFilter(taps, D, algorithm=1).work(dx)
    assert o.rel_rms(host(y), host(yd)) < TOL_RMS
    # streaming in ragged chunks
    f2 = nb.FirFilter(taps, D, algorithm=3)
    outs, pos = [], 0
    for chunk in (5000, 1, 4096, 33333, 10 ** 9):
        if n - pos < D:
            break
        yy, c = f2.work(dx[pos:min(pos + max(chunk, D), n)])
        outs.append(host(yy))
        pos += c
    assert o.rel_rms(np.concatenate(outs), ref[: sum(a.size for a in outs)]) < TOL_RMS
    assert sum(a.size for a in outs) == n // D
    # time segments with a halo
    if T > 1:
        L = (n // 4) // D * D
        parts = []
        for g in range(4):
            lo, hi = g * L, (n if g == 3 else (g + 1) * L)
            halo = None if g == 0 else dx[lo - (T - 1):lo]
            parts.append(host(f.work_segment(dx[lo:hi], halo)))
        assert o.rel_rms(np.concatenate(parts), ref) < TOL_RMS
    # fused multiply_const folded into the spectrum
    k = 0.5 - 0.25j
    yk, _ = nb.FirFilter(taps, D, multiply_const=k, algorithm=3).work(dx)
    assert o.rel_rms(host(yk), o.multiply_const(ref.astype(np.complex64), k)) < TOL_RMS


@pytest.mark.parametrize("T,D", [(1024, 4), (257, 2), (700, 8), (2048, 1), (4095, 1), (640, 10), (1600, 16)])
@pytest.mark.parametrize("start", [1, 2, 3])
def test_fir_polyphase_overlap_save_any_pointer_alignment(cuda, T, D, start):
    """Even-D complex filters run the polyphase overlap-save kernel, whose TMA row view depends on
    whether x[0] sits on a 16-byte boundary: every alignment must give the same stream (and the
    non-TMA path, B200_OLS_TMA=0 semantics, is what the edge blocks use in every run)."""
    import newsched_b200 as nb
    rng = np.random.default_rng(T + D + start)
    n = 4096 * D * 6 + 555
    x = cplx(rng, n + start)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)[start:]
    ref = o.fir(x[start:], taps, D)
    f = nb.FirFilter(taps, D, algorithm=3)
    y, nc = f.work(dx)
    assert y.numel() == n // D and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS
    # worst single sample too: a mis-paired phase would show up as a few wrong outputs
    assert np.max(np.abs(host(y) - ref)) < 1e-4 * np.max(np.abs(ref))
    # streaming with history across calls whose chunk starts alternate between alignments
    f2 = nb.FirFilter(taps, D, algorithm=3)
    outs, pos = [], 0
    for chunk in (4096 * D * 2 + D, 4096 * D * 3, 10 ** 9):
        yy, c = f2.work(dx[pos:min(pos + chunk, n)])
        outs.append(host(yy))
        pos += c
    got = np.concatenate(outs)
    assert got.size == n // D and o.rel_rms(got, ref) < TOL_RMS
    # output pointer 8 bytes past a 16-byte boundary (the two-phase kernel pairs its stores)
    buf = cuda.zeros(n // D + 1, dtype=cuda.complex64, device="cuda")
    f.work_segment(dx, None, buf[1:])
    assert o.rel_rms(host(buf[1:]), ref) < TOL_RMS and buf[0].item() == 0


@pytest.mark.parametrize("T,D", [(3, 1), (64, 1), (129, 2), (1024, 4), (2500, 3), (4096, 1)])
def test_fir_overlap_save_real_stream(cuda, T, D):
    """fff through algorithm 3: two real blocks per complex transform."""
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 3 + D)
    n = 4 * 4096 * 5 + 777
    x = rng.uniform(-1, 1, n).astype(np.float32)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    f = nb.FirFilter(taps, D, is_complex=False, algorithm=3)
    assert f.algorithm == 3
    y, nc = f.work(dx)
    ref = o.fir(x, taps, D)
    assert y.numel() == n // D and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS
    # chunked streaming (history carried by the handle) and an unaligned start
    f2 = nb.FirFilter(taps, D, is_complex=False, algorithm=3)
    outs, pos = [], 0
    for chunk in (4099, 1, 33333, 10 ** 9):
        if n - pos < D:
            break
        yy, c = f2.work(dx[pos:min(pos + max(chunk, D), n)])
        outs.append(host(yy))
        pos += c
    got = np.concatenate(outs)
    assert got.size == n // D and o.rel_rms(got, ref) < TOL_RMS
    yk, _ = nb.FirFilter(taps, D, is_complex=False, multiply_const=3.25, algorithm=3).work(dx)
    assert o.rel_rms(host(yk), ref * np.float32(3.25)) < TOL_RMS


@pytest.mark.parametrize("T,L,D,cplxin", [(48, 4, 1, True), (49, 3, 2, True), (160, 8, 5, False),
                                          (7, 1, 3, True), (33, 5, 5, False), (3, 7, 2, True),
                                          (1024, 16, 1, True), (2048, 4, 3, True), (256, 2, 9, False),
                                          (96, 3, 64, True), (64, 2, 1, True), (100, 3, 1, False),
                                          (33, 4, 1, False), (2000, 4, 1, True), (5, 3, 1, True),
                                          (96, 3, 2, True), (70, 2, 3, True), (320, 5, 4, True), (97, 4, 5, True),
                                          (64, 5, 3, True), (150, 3, 5, True), (40, 4, 3, True), (200, 3, 4, True),
                                          (31, 5, 2, True), (77, 2, 5, True), (96, 3, 2, False), (130, 2, 3, False),
                                          (400, 5, 4, False), (65, 4, 5, False), (90, 3, 4, False), (77, 2, 5, False),
                                          (200, 3, 5, False), (300, 4, 5, False)])
def test_resampler_matches_oracle(cuda, T, L, D, cplxin):
    """interp_fir_filter (D = 1) / rational_resampler against the fp64 oracle; streaming in ragged
    chunks (history on the device) and time segments with a halo are bit-identical to one shot."""
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 31 + L * 7 + D)
    n = 200000 + 123
    x = cplx(rng, n) if cplxin else rng.uniform(-1, 1, n).astype(np.float32)
    taps = (rng.uniform(-1, 1, T) * (L / T)).astype(np.float32)
    dx = dev(cuda, x)
    r = nb.RationalResampler(taps, L, D, is_complex=cplxin)
    y, nc = r.work(dx)
    ref = o.resample(x, taps, L, D)
    assert y.numel() == (n // D) * L and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS
    one = host(y)
    r2 = nb.RationalResampler(taps, L, D, is_complex=cplxin)
    outs, pos = [], 0
    for chunk in (5000, 1, 4097, 33333, 10 ** 9):
        if n - pos < D:
            break
        yy, c = r2.work(dx[pos:min(pos + max(chunk, D), n)])
        outs.append(host(yy))
        pos += c
    assert np.array_equal(np.concatenate(outs), one), "chunked != one-shot"
    nh = (T + L - 1) // L - 1
    seg = (n // 3) // D * D
    parts = []
    for g in range(3):
        lo, hi = g * seg, (n if g == 2 else (g + 1) * seg)
        halo = None if (g == 0 or nh == 0) else dx[lo - nh:lo]
        parts.append(host(r.work_segment(dx[lo:hi], halo)))
    assert np.array_equal(np.concatenate(parts), one), "time segments + halo != one stream"


@pytest.mark.parametrize("cplxin", [True, False])
def test_rational_fold_every_built_ratio(cuda, cplxin, monkeypatch):
    """Every (L, M) the folded rational kernel is instantiated for, forced on (the automatic choice leaves
    some ratios on the register-blocked kernel): against the fp64 oracle, and ragged chunks == one shot."""
    import newsched_b200 as nb
    monkeypatch.setenv("B200_RATIONAL_MINTQ", "1")
    rng = np.random.default_rng(77 + cplxin)
    n = 64 * 16 * 5 * 7 + 321
    x = cplx(rng, n) if cplxin else rng.uniform(-1, 1, n).astype(np.float32)
    dx = dev(cuda, x)
    for L, D in ((3, 2), (2, 3), (4, 3), (3, 4), (5, 4), (4, 5), (5, 3), (3, 5), (5, 2), (2, 5)):
        for T in (L * 7 + 1, L * 40):
            taps = (rng.uniform(-1, 1, T) * (L / T)).astype(np.float32)
            r = nb.RationalResampler(taps, L, D, is_complex=cplxin)
            y, nc = r.work(dx)
            assert y.numel() == (n // D) * L and nc == (n // D) * D
            assert o.rel_rms(host(y), o.resample(x, taps, L, D)) < TOL_RMS, (L, D, T)
            r2 = nb.RationalResampler(taps, L, D, is_complex=cplxin)
            outs, pos = [], 0
            for chunk in (4099, D, 10 ** 9):
                yy, c = r2.work(dx[pos:min(pos + max(chunk, D), n)])
                outs.append(host(yy))
                pos += c
            assert np.array_equal(np.concatenate(outs), host(y)), (L, D, T)


def test_interp_fir_impulse_exact_and_empty(cuda):
    import newsched_b200 as nb
    rng = np.random.default_rng(5)
    taps = rng.uniform(-1, 1, 45).astype(np.float32)
    imp = np.zeros(256, np.complex64)
    imp[3] = 1j
    y = host(nb.RationalResampler(taps, 5, 1).work(dev(cuda, imp))[0])
    assert np.array_equal(y[15:60].imag, taps) and not y[:15].any() and not y[60:].any() and not y.real.any()
    r = nb.RationalResampler(taps, 3, 4)
    y, nc = r.work(cuda.ones(3, dtype=cuda.complex64, device="cuda"))
    assert y.numel() == 0 and nc == 0
    with pytest.raises(nb.B200Error):
        nb.RationalResampler(taps, 1, 5000)      # plain heavy decimation belongs to fir_filter


@pytest.mark.parametrize("T,D,cplxin", [(16, 2, True), (64, 2, True), (96, 4, True), (160, 4, True), (33, 8, True),
                                        (192, 8, True), (64, 16, True), (384, 16, True), (64, 2, False),
                                        (256, 4, False), (100, 8, False), (500, 16, False), (64, 32, False),
                                        (64, 3, True), (17, 3, True), (200, 5, True), (96, 6, True), (48, 7, True),
                                        (300, 7, True), (64, 3, False), (33, 5, False), (200, 6, False),
                                        (130, 7, False), (40, 9, True), (64, 12, True), (100, 15, True),
                                        (33, 10, True), (64, 10, False), (90, 13, False), (48, 14, True)])
def test_fir_decimation_folded_into_full_rate_kernel(cuda, T, D, cplxin):
    """Decimations that divide a thread's window (2/4/8/16, 32 for fff) run in the TMA-staged
    full-rate kernel, which keeps accumulators only for every D-th position: bit-identical to the
    phase-plane kernel (same products, same order), exact decimation phase, chunk- and
    segment-invariant."""
    import os
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 7 + D + cplxin)
    n = 1024 * 37 * (D if 32 % D else 1) + 1234     # several tiles (1024 D or 512 D inputs each for non-divisors of 16 / 32)
    x = cplx(rng, n) if cplxin else rng.uniform(-1, 1, n).astype(np.float32)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    f = nb.FirFilter(taps, D, is_complex=cplxin, algorithm=1)
    y, nc = f.work(dx)
    ref = o.fir(x, taps, D)
    assert y.numel() == n // D and nc == (n // D) * D
    assert o.rel_rms(host(y), ref) < TOL_RMS
    one = host(y)
    # decimation phase: y[m] is the full-rate output at m*D, bit for bit
    os.environ["B200_FIR_REAL_SCALAR"] = "1"     # (full-rate fff normally runs the float-pair form: other sum order)
    try:
        full = host(nb.FirFilter(taps, 1, is_complex=cplxin, algorithm=1).work(dx)[0])
    finally:
        os.environ.pop("B200_FIR_REAL_SCALAR", None)
    assert np.array_equal(one, full[::D][: one.size])
    # ragged chunks (unaligned pointers -> the non-TMA staging path) and segments with a halo
    f2 = nb.FirFilter(taps, D, is_complex=cplxin, algorithm=1)
    outs, pos = [], 0
    for chunk in (4099 * D, D, 33333, 7 * D + 1, 10 ** 9):
        if n - pos < D:
            break
        yy, c = f2.work(dx[pos:min(pos + max(chunk, D), n)])
        outs.append(host(yy))
        pos += c
    assert np.array_equal(np.concatenate(outs), one), "chunked != one-shot"
    L = (n // 3) // D * D
    parts = []
    for g in range(3):
        lo, hi = g * L, (n if g == 2 else (g + 1) * L)
        halo = None if g == 0 else dx[lo - (T - 1):lo]
        parts.append(host(f.work_segment(dx[lo:hi], halo)))
    assert np.array_equal(np.concatenate(parts), one), "time segments + halo != one stream"
    k = 0.5 - 0.25j if cplxin else 3.25
    yk, _ = nb.FirFilter(taps, D, is_complex=cplxin, multiply_const=k, algorithm=1).work(dx)
    exp = o.multiply_const(one, k) if cplxin else one * np.float32(k)
    assert np.array_equal(host(yk), exp), "fused epilogue != two-block chain"
    # output pointer 8 bytes past a 16-byte boundary: plain store loop instead of the TMA store
    buf = cuda.zeros(n // D + 4, dtype=dx.dtype, device="cuda")
    off = 1 if cplxin else 3
    f.work_segment(dx, None, buf[off:off + n // D])
    assert np.array_equal(host(buf[off:off + n // D]), one) and buf[0].item() == 0 and buf[-1].item() == 0


@pytest.mark.parametrize("T", [1, 2, 3, 16, 31, 32, 33, 64, 100, 128, 255])
def test_fir_real_stream_as_float_pairs(cuda, T):
    """Full-rate fff runs as float pairs through the packed complex x real loop (even taps on the
    stream, odd taps on the stream one float later): oracle parity, odd lengths, any chunking
    bit-identical (the sum order of an output does not depend on where it falls), history, segments,
    fused constant, unaligned pointers; and within rounding of the scalar kernel it replaces."""
    import os
    import newsched_b200 as nb
    rng = np.random.default_rng(T)
    n = 4096 * 9 + 777          # odd
    x = rng.uniform(-1, 1, n).astype(np.float32)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    f = nb.FirFilter(taps, 1, is_complex=False, algorithm=1)
    y, nc = f.work(dx)
    ref = o.fir(x, taps, 1)
    assert y.numel() == n and nc == n
    assert o.rel_rms(host(y), ref) < TOL_RMS
    assert np.max(np.abs(host(y) - ref)) < 1e-5 * max(1e-3, np.max(np.abs(ref)))
    one = host(y)
    f2 = nb.FirFilter(taps, 1, is_complex=False, algorithm=1)
    outs, pos = [], 0
    for chunk in (5001, 1, 4096, 33333, 7, 2, 10 ** 9):
        if pos >= n:
            break
        yy, c = f2.work(dx[pos:min(pos + chunk, n)])
        outs.append(host(yy))
        pos += c
    assert np.array_equal(np.concatenate(outs), one), "chunked != one-shot"
    if T > 1:
        L = n // 3
        parts = []
        for g in range(3):
            lo, hi = g * L, (n if g == 2 else (g + 1) * L)
            halo = None if g == 0 else dx[lo - (T - 1):lo]
            parts.append(host(f.work_segment(dx[lo:hi], halo)))
        assert np.array_equal(np.concatenate(parts), one), "time segments + halo != one stream"
    yk, _ = nb.FirFilter(taps, 1, is_complex=False, multiply_const=3.25, algorithm=1).work(dx)
    assert np.array_equal(host(yk), one * np.float32(3.25))
    for off_in, off_out in ((1, 0), (0, 3), (3, 1)):
        xb = cuda.zeros(n + 4, dtype=cuda.float32, device="cuda")
        xb[off_in:off_in + n] = dx
        ob = cuda.zeros(n + 8, dtype=cuda.float32, device="cuda")
        f.work_segment(xb[off_in:off_in + n], None, ob[off_out:off_out + n])
        assert np.array_equal(host(ob[off_out:off_out + n]), one) and ob[off_out + n].item() == 0
    os.environ["B200_FIR_REAL_SCALAR"] = "1"
    try:
        ys, _ = nb.FirFilter(taps, 1, is_complex=False, algorithm=1).work(dx)
    finally:
        os.environ.pop("B200_FIR_REAL_SCALAR", None)
    assert o.rel_rms(one, host(ys)) < TOL_RMS


@pytest.mark.parametrize("T,D", [(5, 1), (33, 1), (64, 1), (100, 1), (128, 1), (256, 1), (384, 1), (448, 1), (449, 1),
                                 (1024, 1), (96, 3), (512, 2), (1024, 4), (2048, 8)])
def test_fir_tensor_core_form(cuda, T, D):
    """algorithm 2: block-Toeplitz GEMM on tcgen05 (bf16 hi/lo split, fp32 accumulation in TMEM).  Tap-stationary
    persistent kernel for D = 1 and K <= 512 (T <= 448), ring form beyond and for D > 1.  Against the fp64
    oracle: one shot, any 8-byte pointer alignment (a ring hands out windows on item boundaries), chunked
    streaming with ragged chunks, a time segment with its halo, and the fused multiply_const epilogue."""
    import newsched_b200 as nb
    rng = np.random.default_rng(T * 7 + D)
    n = (4096 * 150 * 2 + 1234) * D + (D - 1)           # > 2 tiles per SM for the persistent form, ragged tail
    x = cplx(rng, n + 1)
    taps = (rng.uniform(-1, 1, T) / np.sqrt(T)).astype(np.float32)
    dx = dev(cuda, x)
    ref = o.fir(x[:n], taps, D, mt=True)
    f = nb.FirFilter(taps, D, algorithm=2)
    assert f.algorithm == 2
    y, nc = f.work(dx[:n])
    assert nc == (n // D) * D and o.rel_rms(host(y), ref) < TOL_RMS
    # an 8-byte-only aligned input / output window
    f1 = nb.FirFilter(taps, D, algorithm=2)
    buf = cuda.zeros(n // D + 3, dtype=cuda.complex64, device="cuda")
    y1, _ = f1.work(dx[1:], buf[1:1 + n // D])
    assert o.rel_rms(host(y1), o.fir(x[1:], taps, D, mt=True)) < TOL_RMS and buf[0].item() == 0 and buf[-1].item() == 0
    # streaming in ragged chunks: the history carries over
    f2 = nb.FirFilter(taps, D, algorithm=2)
    outs, pos = [], 0
    for c in (7 * D, 4096 * D + D, 100003 * D, n):
        c = min(c, n - pos)
        if c <= 0:
            break
        yy, used = f2.work(dx[pos:pos + c])
        outs.append(host(yy))
        pos += used
    got = np.concatenate(outs)
    assert o.rel_rms(got, ref[: got.size]) < TOL_RMS and got.size >= ref.size - 1
    # a time segment with its halo (multi-GPU sharding) == the same outputs of the whole stream
    cut = (4096 * 100 + 8) * D
    seg = f.work_segment(dx[cut:n], dx[cut - (T - 1):cut] if T > 1 else None)
    assert o.rel_rms(host(seg), ref[cut // D:]) < TOL_RMS
    # fused multiply_const epilogue
    k = 0.5 - 0.25j
    yk, _ = nb.FirFilter(taps, D, algorithm=2, multiply_const=k).work(dx[:n])
    assert o.rel_rms(host(yk), ref * np.complex64(k)) < TOL_RMS


def test_fir_tensor_core_form_rejects_what_it_cannot_do(cuda):
    import newsched_b200 as nb
    with pytest.raises(nb.B200Error):
        nb.FirFilter(np.ones(64, np.float32), 2, is_complex=False, algorithm=2)    # float streams: decimation 1 only
    with pytest.raises(nb.B200Error):
        nb.FirFilter(np.ones(450, np.float32), 1, is_complex=False, algorithm=2)   # ... and taps resident in TMEM (K <= 512)
    with pytest.raises(nb.B200Error):
        nb.FirFilter(np.ones(64, np.float32), 9, algorithm=2)                      # decimation > 8


@pytest.mark.parametrize("algorithm", [-1, 5, 6, 7])
def test_fir_rejects_unknown_algorithm(cuda, algorithm):
    """algorithm is 0 (auto) or one of the forms 1..4; any other value is an error, not a silent direct form."""
    import newsched_b200 as nb
    with pytest.raises(nb.B200Error, match="algorithm must be"):
        nb.FirFilter(np.ones(64, np.float32), 1, algorithm=algorithm)


@pytest.mark.parametrize("T", [33, 64, 100, 256, 448, 5])
def test_fir_fff_tensor_core_form(cuda, T):
    """fir_filter_fff on the tensor cores: the tap-stationary block-Toeplitz kernel with two 4096-sample runs of the
    float stream riding through its two planes.  Against the fp64 oracle: one shot, streamed in ragged chunks,
    fused constant, a 4-byte-aligned stream (element-wise tiles), time segments with a halo, tiny inputs."""
    import newsched_b200 as nb
    rng = np.random.default_rng(900 + T)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    n = 8192 * 37 + 4097 + 13                         # whole tiles, a tile with only its first run complete, a ragged end
    x = rng.uniform(-1, 1, n).astype(np.float32)
    dx = dev(cuda, x)
    ref = o.fir(x, taps, 1)
    f = nb.FirFilter(taps, 1, is_complex=False, algorithm=2)
    assert f.algorithm == 2
    y, nc = f.work(dx)
    assert nc == n and o.rel_rms(host(y), ref) < TOL_RMS
    # streaming: the history carries over calls of any length (shorter than a tile, shorter than the history, one item)
    g = nb.FirFilter(taps, 1, is_complex=False, algorithm=2)
    outs, pos = [], 0
    for m in (1, 7, T - 1 if T > 1 else 1, 4096, 8191, 8192, 8193, 100000, 10 ** 9):
        if pos >= n:
            break
        yy, c = g.work(dx[pos:pos + m])
        outs.append(host(yy))
        pos += c
    assert pos == n and o.rel_rms(np.concatenate(outs), ref) < TOL_RMS
    # fused multiply_const (real constant)
    yk, _ = nb.FirFilter(taps, 1, is_complex=False, algorithm=2, multiply_const=0.375).work(dx)
    assert o.rel_rms(host(yk), ref * np.float32(0.375)) < TOL_RMS
    # a stream that is only 4-byte aligned (a ring hands out windows on item boundaries): the bulk copies start up to
    # three samples early; same numbers for every alignment
    for sh in (1, 2, 3):
        xo = cuda.empty(n + sh, dtype=cuda.float32, device="cuda")
        xo[sh:] = dx
        yo, _ = nb.FirFilter(taps, 1, is_complex=False, algorithm=2).work(xo[sh:])
        assert np.array_equal(host(yo), host(y)), sh
    # time segment with its halo == the same outputs of the stream
    cut = 8192 * 11 + 16
    if T > 1:
        seg = nb.FirFilter(taps, 1, is_complex=False, algorithm=2).work_segment(dx[cut:], dx[cut - (T - 1):cut])
        assert o.rel_rms(host(seg), ref[cut:]) < TOL_RMS
    for m in (0, 1, 63, 64, 4095, 4096, 4097):
        ys, c = nb.FirFilter(taps, 1, is_complex=False, algorithm=2).work(dx[:m])
        assert c == m and ys.numel() == m
        if m:
            assert o.rel_rms(host(ys), ref[:m]) < TOL_RMS or np.abs(host(ys) - ref[:m]).max() < 1e-6


def test_fir_auto_algorithm_choice(cuda):
    import newsched_b200 as nb
    assert nb.FirFilter(np.ones(32, np.float32), 1).algorithm == 1     # short: direct FFMA2 form (HBM-bound)
    assert nb.FirFilter(np.ones(64, np.float32), 1).algorithm == 2     # config 1: block-Toeplitz GEMM on tcgen05
    assert nb.FirFilter(np.ones(384, np.float32), 1).algorithm == 2
    assert nb.FirFilter(np.ones(385, np.float32), 1).algorithm == 3    # beyond: overlap-save
    assert nb.FirFilter(np.ones(32, np.float32), 1, is_complex=False).algorithm == 1   # float streams: the same rule ...
    assert nb.FirFilter(np.ones(64, np.float32), 1, is_complex=False).algorithm == 2
    assert nb.FirFilter(np.ones(448, np.float32), 1, is_complex=False).algorithm == 2  # ... while the taps fit TMEM
    assert nb.FirFilter(np.ones(449, np.float32), 1, is_complex=False).algorithm == 3
    assert nb.FirFilter(np.ones(64, np.float32), 4, is_complex=False).algorithm == 1   # decimating float streams stay SIMT
    assert nb.FirFilter(np.ones(64, np.float32), 1, algorithm=1).algorithm == 1        # and the SIMT forms stay selectable
    assert nb.FirFilter(np.ones(1024, np.float32), 4).algorithm == 3   # config 3: overlap-save
    assert nb.FirFilter(np.ones(1024, np.float32), 4, is_complex=False).algorithm == 3
    assert nb.FirFilter(np.ones(300, np.float32), 40).algorithm == 3   # huge D: overlap-save instead of the fallback
    assert nb.FirFilter(np.ones(100, np.float32), 40, algorithm=4).algorithm == 4   # the fallback stays selectable
    assert nb.FirFilter(np.ones(256, np.float32), 4).algorithm == 3    # polyphase overlap-save beyond 160 taps at D = 4
    assert nb.FirFilter(np.ones(128, np.float32), 4).algorithm == 1    # decimation folded into the full-rate kernel
    assert nb.FirFilter(np.ones(256, np.float32), 16).algorithm == 1
    assert nb.FirFilter(np.ones(300, np.float32), 3).algorithm == 3    # D = 3: folded kernel up to 208 taps
    assert nb.FirFilter(np.ones(64, np.float32), 3).algorithm == 1
    assert nb.FirFilter(np.ones(64, np.float32), 6).algorithm == 1     # D = 3, 5, 6, 7 fold too (D rows per thread)
    assert nb.FirFilter(np.ones(256, np.float32), 6).algorithm == 3
    assert nb.FirFilter(np.ones(64, np.float32), 10).algorithm == 1    # ... and 9 ... 15
    assert nb.FirFilter(np.ones(256, np.float32), 10).algorithm == 3
    assert nb.FirFilter(np.ones(512, np.float32), 11, is_complex=False).algorithm == 1   # real streams fold further out
    assert nb.FirFilter(np.ones(1024, np.float32), 11, is_complex=False).algorithm == 3


def test_fir_empty_and_short(cuda):
    import newsched_b200 as nb
    f = nb.FirFilter(np.ones(8, np.float32), 4)
    y, nc = f.work(cuda.zeros(0, dtype=cuda.complex64, device="cuda"))
    assert y.numel() == 0 and nc == 0
    y, nc = f.work(cuda.ones(3, dtype=cuda.complex64, device="cuda"))
    assert y.numel() == 0 and nc == 0


def test_fir_segment_halo_equals_stream(cuda):
    import newsched_b200 as nb
    rng = np.random.default_rng(21)
    T, D, n = 200, 2, 1 << 16
    x = cplx(rng, n)
    taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
    dx = dev(cuda, x)
    f = nb.FirFilter(taps, D, algorithm=1)   # direct form: bit-exact across any segmentation
    ref = host(f.work(dx)[0])
    segs = 8
    L = n // segs
    parts = []
    for g in range(segs):
        halo = None if g == 0 else dx[g * L - (T - 1):g * L]
        parts.append(host(f.work_segment(dx[g * L:(g + 1) * L], halo)))
    assert np.array_equal(np.concatenate(parts), ref), "time-segment sharding must equal one stream"


def test_fir_fused_multiply_const(cuda):
    import newsched_b200 as nb
    rng = np.random.default_rng(9)
    x = cplx(rng, 50000)
    taps = (rng.uniform(-1, 1, 100) / 100).astype(np.float32)
    k = 0.5 - 0.25j
    dx = dev(cuda, x)
    a = nb.multiply_const(nb.FirFilter(taps, 4).work(dx)[0], k)
    b = nb.FirFilter(taps, 4, multiply_const=k).work(dx)[0]
    assert cuda.equal(a, b), "fused epilogue must equal the two-block chain bit for bit"


def test_fir_config1_size_linearity(cuda):
    """BASELINE config 1 size (16M samples, 64 taps): linearity + spot check vs the oracle."""
    import newsched_b200 as nb
    n = 1 << 24
    g = cuda.Generator(device="cuda").manual_seed(1)
    x1 = cuda.view_as_complex(cuda.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    x2 = cuda.view_as_complex(cuda.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    rng = np.random.default_rng(1)
    taps = (rng.uniform(-1, 1, 64) / 64).astype(np.float32)
    y1 = nb.FirFilter(taps).work(x1)[0]
    y2 = nb.FirFilter(taps).work(x2)[0]
    y12 = nb.FirFilter(taps).work(x1 + x2)[0]
    err = (y12 - (y1 + y2)).abs().pow(2).mean().sqrt() / y12.abs().pow(2).mean().sqrt()
    assert float(err) < TOL_RMS
    for s in (0, 5_000_000, n - 4096):
        seg = host(x1[max(s - 63, 0):s + 4096])
        ref = o.fir(seg, taps, 1)[(63 if s else 0):]
        assert o.rel_rms(host(y1[s:s + 4096]), ref) < TOL_RMS


@pytest.mark.parametrize("T,D,log2n,algo", [(1024, 4, 28, 3), (4096, 1, 27, 3), (512, 1, 26, 3), (256, 1, 26, 2),
                                             (64, 1, 27, 2)])
def test_fir_long_filters_full_size_properties(cuda, T, D, log2n, algo):
    """BASELINE config 3 head (2^28 samples, 1024 taps, decim 4: polyphase overlap-save), config 5
    per-GPU segment (2^27 samples, 4096 taps: two-phase overlap-save), a one-phase overlap-save
    size and two tensor-core (tcgen05 block-Toeplitz) sizes incl. config 1's 64 taps on a 1 GiB stream,
    through size-independent properties: linearity, oracle spot checks on windows at the
    start / middle / end of the stream, and the response to impulses placed deep in the stream
    (output index = input index / D exactly: decimation phase and 64-bit indexing)."""
    import newsched_b200 as nb
    n = 1 << log2n
    g = cuda.Generator(device="cuda").manual_seed(T + D)
    x1 = cuda.view_as_complex(cuda.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    x2 = cuda.view_as_complex(cuda.rand(n, 2, device="cuda", generator=g) * 2 - 1)
    rng = np.random.default_rng(T)
    taps = (rng.uniform(-1, 1, T) / np.sqrt(T)).astype(np.float32)
    f = nb.FirFilter(taps, D)
    assert f.algorithm == algo
    y1 = f.work_segment(x1)
    y2 = f.work_segment(x2)
    x1 += x2
    y12 = f.work_segment(x1)
    x1 -= x2                                     # (fp32: x1 is back to within 1 ulp; only used for windows below)
    y1 += y2
    err = (y12 - y1).abs().pow(2).mean().sqrt() / y12.abs().pow(2).mean().sqrt()
    assert float(err) < TOL_RMS
    del y1, y12
    # oracle on windows: outputs [m0, m0 + 2048) need inputs [m0*D - (T-1), (m0 + 2048)*D)
    for m0 in (0, (n // D) // 2 + 12345, n // D - 2048):
        skip = -(-(T - 1) // D) if m0 else 0        # whole outputs of lead-in, so the window starts on phase 0
        lo = (m0 - skip) * D
        seg = host(x2[lo:(m0 + 2048) * D])
        ref = o.fir(seg, taps, D)
        assert o.rel_rms(host(y2[m0:m0 + 2048]), ref[skip:skip + 2048]) < TOL_RMS
    del y2
    # impulses deep in the stream: h[k] appears at output (g0 + k) / D when D divides g0 + k
    x1.zero_()
    spots = [7, n // 2 + 3 * D + 1, n - 2 * T - 5]
    for i, g0 in enumerate(spots):
        x1[g0] = complex(1 + i, -(1 + i))
    y = f.work_segment(x1)
    hn = float(np.sqrt(np.sum(taps.astype(np.float64) ** 2)))   # FFT rounding scales with ||h||_2 * |amplitude|
    for i, g0 in enumerate(spots):
        m_lo = -(-g0 // D)
        k = np.arange(m_lo * D - g0, T, D)
        exp = taps[k].astype(np.complex64) * np.complex64(complex(1 + i, -(1 + i)))
        got = host(y[m_lo:m_lo + k.size])
        assert np.max(np.abs(got - exp)) < 2e-6 * hn * (1 + i) * np.sqrt(2), (T, D, g0)
    # and nothing anywhere else (between the second and third response)
    quiet = y[(spots[1] + T) // D + 4096:(spots[2]) // D - 4096]
    assert float(quiet.abs().max()) < 1e-6 * hn


# ------------------------------------------------------------------------------- FFT
@pytest.mark.parametrize("key,fwd,shift", [("fft_fwd", True, False), ("fft_fwd_shift", True, True),
                                           ("fft_rev", False, False), ("fft_rev_shift", False, True)])
def test_fft4096_golden(cuda, golden, key, fwd, shift):
    import newsched_b200 as nb
    x, w = golden["fft_x"], golden["bh4096"].astype(np.float32)
    y = host(nb.FFT(4096, fwd, w, shift).work(dev(cuda, x)))
    for v in range(2):
        assert o.rel_rms(y[v * 4096:(v + 1) * 4096], golden[key][v * 4096:(v + 1) * 4096]) < TOL_RMS


@pytest.mark.parametrize("N", [8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192])
@pytest.mark.parametrize("fwd", [True, False])
def test_fft_matches_oracle(cuda, N, fwd):
    import newsched_b200 as nb
    rng = np.random.default_rng(N)
    nv = 37 if N <= 1024 else 5
    x = cplx(rng, nv * N)
    w = rng.uniform(0.1, 1, N).astype(np.float32)
    for shift in (False, True):
        y = host(nb.FFT(N, fwd, w, shift).work(dev(cuda, x)))
        ref = o.fft(x, N, fwd, w, shift)
        for v in range(nv):
            assert o.rel_rms(y[v * N:(v + 1) * N], ref[v * N:(v + 1) * N]) < TOL_RMS
    y = host(nb.FFT(N, fwd).work(dev(cuda, x)))      # no window
    assert o.rel_rms(y, o.fft(x, N, fwd)) < TOL_RMS


def test_fft_impulse_tone_exact_structure(cuda):
    import newsched_b200 as nb
    N = 4096
    imp = np.zeros(N, np.complex64)
    imp[0] = 1
    y = host(nb.FFT(N).work(dev(cuda, imp)))
    assert np.abs(y - 1).max() < 1e-6                 # flat spectrum
    k0 = 1234
    tone = np.exp(2j * np.pi * k0 * np.arange(N) / N).astype(np.complex64)
    y = host(nb.FFT(N).work(dev(cuda, tone)))
    assert int(np.argmax(np.abs(y))) == k0            # bin index exact
    ys = host(nb.FFT(N, shift=True).work(dev(cuda, tone)))
    assert int(np.argmax(np.abs(ys))) == (k0 + N // 2) % N   # DC lands on N/2


@pytest.mark.parametrize("N", [8, 16, 64, 128, 256, 512, 1024, 2048, 4096, 8192])
def test_fft_mag_fused_and_premultiply(cuda, golden, N):
    import newsched_b200 as nb
    rng = np.random.default_rng(N + 1)
    x = cplx(rng, 9 * N)
    w = o.window_blackmanharris(N)
    dx = dev(cuda, x)
    ref = o.fft(x, N, True, w)
    m = host(nb.FFT(N, True, w, output=nb.OUT_MAG).work(dx))
    assert o.rel_rms(m, np.abs(ref.astype(np.complex128))) < TOL_RMS
    m2 = host(nb.FFT(N, True, w, output=nb.OUT_MAG_SQUARED).work(dx))
    assert o.rel_rms(m2, np.abs(ref.astype(np.complex128)) ** 2) < 2 * TOL_RMS
    k = 0.5 - 0.25j
    y = host(nb.FFT(N, True, w, pre_multiply_const=k).work(dx))
    ref2 = o.fft(o.multiply_const(x, k), N, True, w)
    assert o.rel_rms(y, ref2) < TOL_RMS


def test_fft_config2_size_roundtrip(cuda):
    """BASELINE config 2 size (1 GiB = 32768 x 4096): reverse(forward(x)) == N x, and Parseval."""
    import newsched_b200 as nb
    N, nv = 4096, 32768
    g = cuda.Generator(device="cuda").manual_seed(2)
    x = cuda.view_as_complex(cuda.rand(nv * N, 2, device="cuda", generator=g) * 2 - 1)
    X = nb.FFT(N, True).work(x)
    e_t = x[: 64 * N].abs().pow(2).sum().double()
    e_f = X[: 64 * N].abs().pow(2).sum().double() / N
    assert abs(float(e_t / e_f) - 1) < 1e-5
    xr = nb.FFT(N, False).work(X)
    err = (xr / N - x).abs().pow(2).mean().sqrt() / x.abs().pow(2).mean().sqrt()
    assert float(err) < TOL_RMS
    # last vector against the oracle (tail handling at full size)
    ref = o.fft(host(x[-N:]), N)
    assert o.rel_rms(host(X[-N:]), ref) < TOL_RMS


def test_fft8192_many_vectors_roundtrip(cuda):
    """N = 8192 (radix-2 split in front of two 4096-point transforms): more vectors than CTAs, so the
    persistent loop and the two-half TMA refill run; forward -> reverse returns N x; Parseval;
    first / middle / last vectors against the oracle, with a window, shift and fused |.|."""
    import newsched_b200 as nb
    N, nv = 8192, 1000
    g = cuda.Generator(device="cuda").manual_seed(8)
    x = cuda.view_as_complex(cuda.rand(nv * N, 2, device="cuda", generator=g) * 2 - 1)
    X = nb.FFT(N, True).work(x)
    e_t = x.abs().pow(2).sum().double()
    e_f = X.abs().pow(2).sum().double() / N
    assert abs(float(e_t / e_f) - 1) < 1e-5
    xr = nb.FFT(N, False).work(X)
    err = (xr / N - x).abs().pow(2).mean().sqrt() / x.abs().pow(2).mean().sqrt()
    assert float(err) < TOL_RMS
    w = o.window_blackmanharris(N)
    for shift in (False, True):
        Y = nb.FFT(N, True, w, shift).work(x)
        M = nb.FFT(N, True, w, shift, output=nb.OUT_MAG).work(x)
        for v in (0, 499, nv - 1):
            ref = o.fft(host(x[v * N:(v + 1) * N]), N, True, w, shift)
            assert o.rel_rms(host(Y[v * N:(v + 1) * N]), ref) < TOL_RMS
            assert o.rel_rms(host(M[v * N:(v + 1) * N]), np.abs(ref.astype(np.complex128))) < TOL_RMS
    # unaligned input pointer: falls back to the generic kernel, same numbers within tolerance
    xo = cuda.empty(4 * N + 1, dtype=cuda.complex64, device="cuda")
    xo[1:] = x[: 4 * N]
    assert o.rel_rms(host(nb.FFT(N, True).work(xo[1:])), host(X[: 4 * N])) < TOL_RMS


# ------------------------------------------------------------------------ channelizer
@pytest.mark.parametrize("name", ["pfb_a", "pfb_b"])
def test_pfb_golden(cuda, golden, name):
    import newsched_b200 as nb
    taps, x, M = golden[name + "_taps"], golden[name + "_x"], int(golden[name + "_M"][0])
    y, nc = nb.PfbChannelizer(taps, M).work(dev(cuda, x))
    assert nc == x.size
    assert o.rel_rms(host(y), golden[name + "_y64"]) < TOL_RMS


@pytest.mark.parametrize("M,P", [(64, 16), (64, 3), (64, 32), (16, 8), (256, 4), (4, 7), (16, 16), (16, 5),
                                 (32, 16), (32, 4), (128, 8), (128, 13), (256, 16), (8, 12), (8, 16), (8, 4), (4, 16), (4, 3)])
def test_pfb_matches_oracle_and_streams(cuda, M, P):
    import scipy.signal as sig
    import newsched_b200 as nb
    rng = np.random.default_rng(M + P)
    taps = sig.firwin(M * P, 1.0 / M).astype(np.float32)
    x = cplx(rng, M * max(333, 3 * 4096 // M + 77) + 5)     # several 4096-sample tiles for every M
    dx = dev(cuda, x)
    ref = o.pfb_channelizer(x, taps, M)
    y, nc = nb.PfbChannelizer(taps, M).work(dx)
    assert nc == (x.size // M) * M and o.rel_rms(host(y), ref) < TOL_RMS
    ch = nb.PfbChannelizer(taps, M)
    outs, pos = [], 0
    for n_fr in (1, 2, 64, 100, 166, 4096 // M + 3, 10 ** 6):
        if pos + M > x.size:
            break
        yy, c = ch.work(dx[pos:pos + n_fr * M])
        outs.append(host(yy))
        pos += c
    got = np.concatenate(outs)
    assert np.array_equal(got, host(y)[: got.shape[0]]), "chunked channelizer != one-shot"
    # channel slice == the same columns of the full output
    part, _ = nb.PfbChannelizer(taps, M, channel_begin=M // 4, channel_count=M // 2).work(dx)
    assert np.array_equal(host(part), host(y)[:, M // 4:M // 4 + M // 2])


@pytest.mark.parametrize("P", [16, 3, 8, 12])
def test_pfb_dft_on_tensor_cores(cuda, P):
    """BASELINE configs[3] 'filterbank + DFT as tensor-core GEMM': algorithm 2 (the 64-point DFT across branches as a
    bf16-split tcgen05 GEMM, DFT matrix in tensor memory) against the fp64 oracle, the SIMT form, chunked streaming,
    a channel slice and time segments with a halo."""
    import scipy.signal as sig
    import newsched_b200 as nb
    M = 64
    rng = np.random.default_rng(640 + P)
    taps = sig.firwin(M * P, 1.0 / M).astype(np.float32)
    x = cplx(rng, M * (64 * 7 + 29) + 11)                   # several 64-frame tiles and a ragged one
    dx = dev(cuda, x)
    ref = o.pfb_channelizer(x, taps, M)
    tc = nb.PfbChannelizer(taps, M, algorithm=2)
    assert tc.algorithm == 2
    y, nc = tc.work(dx)
    err = o.rel_rms(host(y), ref)
    assert nc == (x.size // M) * M and err < TOL_RMS, err
    # per channel too: no channel (row of the DFT matrix) may hide behind the others
    yh = host(y).astype(np.complex128)
    per_ch = np.sqrt((np.abs(yh - ref) ** 2).sum(axis=0) / (np.abs(ref) ** 2).sum(axis=0).clip(1e-30))
    assert per_ch.max() < 4 * TOL_RMS, per_ch.max()         # stop-band channels carry little energy: looser
    y1, _ = nb.PfbChannelizer(taps, M, algorithm=1).work(dx)
    assert o.rel_rms(host(y), host(y1).astype(np.complex128)) < TOL_RMS
    # chunked == one-shot, bit for bit (same arithmetic per frame whatever the tiling)
    ch = nb.PfbChannelizer(taps, M, algorithm=2)
    outs, pos = [], 0
    for n_fr in (1, 2, 64, 100, 166, 67, 10 ** 6):
        if pos + M > x.size:
            break
        yy, c = ch.work(dx[pos:pos + n_fr * M])
        outs.append(host(yy))
        pos += c
    got = np.concatenate(outs)
    assert np.array_equal(got, host(y)[: got.shape[0]]), "chunked tensor-core channelizer != one-shot"
    part, _ = nb.PfbChannelizer(taps, M, channel_begin=16, channel_count=32, algorithm=2).work(dx)
    assert np.array_equal(host(part), host(y)[:, 16:48])
    # time segment with a halo == the same frames of the stream
    cut = M * 200
    seg = nb.PfbChannelizer(taps, M, algorithm=2).work_segment(dx[cut:], halo=dx[cut - (P - 1) * M:cut] if P > 1 else None)
    assert np.array_equal(host(seg), host(y)[200:200 + seg.shape[0]])
    # 8-byte aligned (not 16) input pointer: the tile is fetched without the bulk copy
    xo = cuda.empty(x.size + 1, dtype=cuda.complex64, device="cuda")
    xo[1:] = dx
    yo, _ = nb.PfbChannelizer(taps, M, algorithm=2).work(xo[1:])
    assert np.array_equal(host(yo), host(y))


def test_pfb_tensor_core_form_rejects_what_it_cannot_do(cuda):
    import scipy.signal as sig
    import newsched_b200 as nb
    with pytest.raises(nb.B200Error):
        nb.PfbChannelizer(sig.firwin(32 * 8, 1 / 32).astype(np.float32), 32, algorithm=2)
    with pytest.raises(nb.B200Error):
        nb.PfbChannelizer(sig.firwin(64 * 32, 1 / 64).astype(np.float32), 64, algorithm=2)
    tone = np.exp(2j * np.pi * 5 / 64 * np.arange(64 * 600)).astype(np.complex64)
    y = host(nb.PfbChannelizer(sig.firwin(64 * 16, 1 / 64).astype(np.float32), 64, algorithm=2).work(dev(cuda, tone))[0])
    p = (np.abs(y[16:]) ** 2).mean(axis=0)
    assert int(np.argmax(p)) == 5 and p[5] > 1e3 * np.delete(p, 5).max()


def test_pfb_tone(cuda):
    import scipy.signal as sig
    import newsched_b200 as nb
    for M, P, c0 in ((64, 16, 5), (16, 8, 3), (32, 8, 21), (128, 8, 77), (256, 4, 200), (8, 16, 6), (4, 16, 1)):
        taps = sig.firwin(M * P, 1.0 / M).astype(np.float32)
        x = np.exp(2j * np.pi * c0 / M * np.arange(M * 600)).astype(np.complex64)
        y = host(nb.PfbChannelizer(taps, M).work(dev(cuda, x))[0])
        p = (np.abs(y[P:]) ** 2).mean(axis=0)
        assert int(np.argmax(p)) == c0 and p[c0] > 1e3 * np.delete(p, c0).max(), (M, c0)


def test_small_and_ragged_sizes_for_the_tiled_kernels(cuda):
    """Sizes around the tile / grid granularities of the single-pass kernels: fewer items than one tile,
    one more than a whole number of tiles, one more vector than resident CTAs."""
    import scipy.signal as sig
    import newsched_b200 as nb
    rng = np.random.default_rng(77)
    # decimation folded into the full-rate kernel: tiles of 2048 inputs
    for D, T in ((4, 64), (16, 33), (2, 5)):
        taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
        for n in (0, 1, D - 1, D, D + 1, 2047, 2048, 2049, 2048 * 3 + D + 1):
            x = cplx(rng, n)
            y, nc = nb.FirFilter(taps, D, algorithm=1).work(dev(cuda, x))
            assert y.numel() == n // D and nc == (n // D) * D
            if n >= D:
                assert o.rel_rms(host(y), o.fir(x, taps, D)) < TOL_RMS
    # interpolation folded into the full-rate kernel
    for L, T in ((2, 64), (3, 10)):
        taps = rng.uniform(-1, 1, T).astype(np.float32)
        for n in (1, 17, 2047, 2049, 4096 + 5):
            x = cplx(rng, n)
            y, nc = nb.RationalResampler(taps, L, 1).work(dev(cuda, x))
            assert y.numel() == n * L and nc == n
            assert o.rel_rms(host(y), o.resample(x, taps, L, 1)) < TOL_RMS
    # single-pass channelizers: tiles of 4096 samples
    for M, P in ((16, 8), (32, 4), (128, 8), (256, 4), (64, 16), (8, 8), (4, 16)):
        taps = sig.firwin(M * P, 1.0 / M).astype(np.float32)
        TT = 4096 // M
        for nf in (1, TT - 1, TT, TT + 1, 3 * TT + 2):
            x = cplx(rng, nf * M + M // 2)
            y, nc = nb.PfbChannelizer(taps, M).work(dev(cuda, x))
            assert y.shape[0] == nf and nc == nf * M
            assert o.rel_rms(host(y), o.pfb_channelizer(x, taps, M)) < TOL_RMS
    # FFT 8192 / 8: one vector, and one more than a multiple of the resident grid
    sms = cuda.cuda.get_device_properties(0).multi_processor_count
    for N, counts in ((8192, (1, 2, 2 * sms + 1)), (8, (1, 255, 256 * 16 * sms + 3))):
        w = rng.uniform(0.1, 1, N).astype(np.float32)
        for nv in counts:
            x = cplx(rng, nv * N)
            y = host(nb.FFT(N, True, w).work(dev(cuda, x)))
            pick = sorted({0, nv // 2, nv - 1})
            for v in pick:
                assert o.rel_rms(y[v * N:(v + 1) * N], o.fft(x[v * N:(v + 1) * N], N, True, w)) < TOL_RMS
    # polyphase overlap-save at a large decimation, fewer outputs than one block
    taps = (rng.uniform(-1, 1, 2000) / 2000).astype(np.float32)
    for n in (16, 16 * 100 + 3, 16 * 5000 + 1):
        x = cplx(rng, n)
        y, _ = nb.FirFilter(taps, 16, algorithm=3).work(dev(cuda, x))
        assert y.numel() == n // 16 and o.rel_rms(host(y), o.fir(x, taps, 16)) < TOL_RMS


# ------------------------------------------------------------------------ ring / chain
def test_ring_double_mapping(cuda):
    import newsched_b200 as nb
    ring = nb.DeviceRing(1 << 20)
    assert ring.size >= 1 << 20 and ring.size % (1 << 16) == 0
    n = ring.size
    src = cuda.arange(n // 4, dtype=cuda.int32, device="cuda")
    L = nb.lib()
    # write through the low mapping, read the same bytes through the high mapping
    nb._check(L.b200_copy(ring.base, src.data_ptr(), n, nb._stream()))
    dst = cuda.empty_like(src)
    nb._check(L.b200_copy(dst.data_ptr(), ring.base + n, n, nb._stream()))
    assert cuda.equal(src, dst)
    # a window that wraps: write starting at 3/4 n for n/2 bytes, read back via wrapped offsets
    half = src[: n // 8]
    nb._check(L.b200_copy(ring.base + 3 * n // 4, half.data_ptr(), n // 2, nb._stream()))
    back = cuda.empty(n // 16, dtype=cuda.int32, device="cuda")
    nb._check(L.b200_copy(back.data_ptr(), ring.base, n // 4, nb._stream()))
    assert cuda.equal(back, half[n // 16:]), "bytes written past the end must appear at the start"


def test_chain_device_and_host_equal_blocks(cuda):
    import newsched_b200 as nb
    rng = np.random.default_rng(33)
    N = 4096
    n = N * 64 * 4
    x = cplx(rng, n)
    taps = (rng.uniform(-1, 1, 128) / 128).astype(np.float32)
    w = o.window_blackmanharris(N)
    k = 0.5 - 0.25j
    dx = dev(cuda, x)
    # config-3 style chain, block by block
    a = nb.FirFilter(taps, 4).work(dx)[0]
    a = nb.multiply_const(a, k)
    a = nb.FFT(N, True, w).work(a)
    # the same through the chain driver (unfused ops), chunked
    ch = nb.Chain([nb.FirFilter(taps, 4), ("multiply_const_cc", k), nb.FFT(N, True, w)],
                  in_item_bytes=8, chunk_items=N * 4 * 8)
    out = cuda.empty(n // 4, dtype=cuda.complex64, device="cuda")
    nbytes = ch.run(dx, out)
    assert nbytes == out.numel() * 8 and cuda.equal(out, a)
    # host-resident streaming: pinned in, pinned out
    ch2 = nb.Chain([nb.FirFilter(taps, 4), ("multiply_const_cc", k), nb.FFT(N, True, w)],
                   in_item_bytes=8, chunk_items=N * 4 * 8)
    hx = cuda.from_numpy(x).pin_memory()
    hy = cuda.empty(n // 4, dtype=cuda.complex64).pin_memory()
    assert ch2.run_host(hx, hy) == hy.numel() * 8
    assert cuda.equal(hy, a.cpu())
    # fused form (FIR epilogue k, nothing else) stays within tolerance of the oracle
    ref = o.fft(o.multiply_const(o.fir(x, taps, 4), k), N, True, w)
    assert o.rel_rms(host(a), ref) < TOL_RMS
    fused = nb.FFT(N, True, w, pre_multiply_const=k).work(nb.FirFilter(taps, 4).work(dx)[0])
    assert o.rel_rms(host(fused), ref) < TOL_RMS


def test_launch_counter_moves(cuda):
    import newsched_b200 as nb
    before = nb.launch_count()
    nb.copy(cuda.zeros(1024, device="cuda"))
    assert nb.launch_count() > before

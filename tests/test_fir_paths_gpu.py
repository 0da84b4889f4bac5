"""Every kernel path of the FIR family (fir.cu, fir_direct.cuh with fir_dg_* / fir_ll_*, fir_ols.cu, fir_tc.cu,
resampler.cu) against the fp64 oracle.

b200_fir_create (FirFilter) picks the form from T taps, decimation D, the stream type and `algorithm`; the launch
then picks the instantiation:
    algorithm 1   fir_direct_kernel<2, false>        complex, D = 1, T <= 32 (33..384 go to the tensor cores)
                  fir_direct_kernel<2, ..., RP>      real, D = 1, T <= 32: the stream as float pairs
                  fir_direct_kernel<1, false>        real, D = 1 under B200_FIR_REAL_SCALAR
                  fir_direct_kernel<V, false, DD>    D divides the 16 (complex) / 32 (real) positions of a thread
                                                     (dd: 2, 4, 8, 16 / 2 ... 32) while T is below the overlap-save
                                                     crossover (complex 96 / 160 / 192 / 384, real 256 / 512 / 768)
                  fir_direct_kernel<V, ..., DG>      D = 3, 5, 6, 7, 9 ... 15 (up to B200_FIR_DG_MAX), T <= tx_c[D] /
                                                     tx_r[D] (dg: fir_dg_c.cu / fir_dg_r.cu; even D of complex
                                                     streams and real D = 12 use the padded row layout)
                  fir_direct_kernel<V, true>         phase planes: only under B200_FIR_PLANES (D <= 12 fits 200 KiB)
                                                     or with D beyond B200_FIR_DG_MAX; automatic selection never
                                                     reaches it (D >= 17 needs more than 200 KiB and falls back)
    algorithm 4   fir_naive_kernel<2> / <1>          the phase planes would need more than 200 KiB and overlap-save
                                                     does not apply (complex D >= 17 at T = 1, real D >= 17 while
                                                     T / D < 96), or algorithm = 4
    algorithm 2   fir_tc_ts_kernel<false> / <true>   complex 33..384 taps / real 33..448 taps at D = 1: tap-stationary
                  fir_tc_pipe_kernel                 algorithm = 2 at D = 2..8 or beyond 449 taps
    algorithm 3   fir_olsd_kernel                    complex, D = 2..16 (B200_OLS_POLY=0 turns it off); 2 CTAs per SM,
                                                     1 for D > 10; bulk-copied rows for even D unless B200_OLS_TMA=0
                                                     (read at launch)
                  fir_ols2_kernel                    complex, D = 1, T >= 1024 (B200_OLS_TWO sets that bound, 0 = off)
                  fir_ols4096_kernel<false> / <true> everything else (complex / real), in (T - 1) / 2048 + 1
                                                     partitions once the overlap leaves less than 1024 samples
                                                     (T <= 32768: 16 partitions), grid 2 SMs
    B200_FIR_TMA=0 keeps every tile of the direct kernels on the register-staged path.
RationalResampler (b200_resampler_create, interpolation L, decimation D):
    fir_direct_kernel<V, false, 1, L, false, D>      the 13 (L, D) pairs of fir_ll_{c,r}{23,45}.cu: L = 2, 3 at D = 1
                                                     and L = 4 from B200_INTERP_L4_MIN (192) taps; rational pairs
                                                     from fir_ratio_min_tq's taps per phase (B200_RATIONAL_MINTQ
                                                     overrides it; B200_RATIONAL_RB and B200_INTERP_RB turn the
                                                     folds off)
    resample_rb_kernel<V, D, R>                      otherwise for D <= 4 (R = 15, 7, 6, 3)
    resample_kernel<V>                               otherwise, or under B200_RESAMPLER_SIMPLE
Every work() call with outputs ends with fir_hist_kernel / rs_hist_kernel, which keeps the last T - 1 (ceil(T/L) - 1)
inputs as the next call's history; fir_hist_kernel is a dependent launch that the next call's overlap-save and
tap-stationary kernels overlap with.  All switches are read at create except B200_OLS_TMA.

Every case of the path matrix and of the persistent loops asserts, from the kernel names torch.profiler records,
that its call launched exactly the kernel its id names (and the history kernel).

Every case uses random asymmetric taps scaled by 1/sqrt(T) and white uniform input, writes into a view of a
device buffer pre-filled with a NaN bit pattern with more than one tile of guard items on each side, and checks
per block of 4096 output items the relative RMS error and the worst item against that block's reference RMS."""
import functools

import numpy as np
import pytest

import oracle as o
from conftest import cplx

gpu = pytest.mark.gpu

TOL_RMS = 1e-5            # per block, relative RMS error
TOL_ITEM = 1e-4           # per block, worst item / block reference RMS
BLOCK = 4096              # output items per checked block
SENTINEL = 0x7FBADBAD     # a float32 NaN: an output item the kernel fails to write cannot pass
GUARD = 16384             # sentinel items on each side of an output: more than a tile of any family
MAC_BUDGET = 2e8          # oracle multiply-adds per case
SWITCHES = ("B200_FIR_TMA", "B200_FIR_PLANES", "B200_FIR_DG_MAX", "B200_FIR_REAL_SCALAR", "B200_OLS_POLY",
            "B200_OLS_TWO", "B200_OLS_TMA", "B200_RESAMPLER_SIMPLE", "B200_INTERP_RB", "B200_RATIONAL_RB",
            "B200_RATIONAL_MINTQ", "B200_INTERP_L4_MIN")
TX_C = (0, 0, 0, 208, 0, 304, 176, 368, 0, 448, 208, 544, 288, 448, 224, 512)   # fir.cu: fold / overlap-save
TX_R = (0, 0, 0, 352, 0, 608, 608, 640, 0, 640, 576, 640, 480, 448, 448, 512)   # crossovers (taps)
DG = (3, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15)
RB_R = {1: 15, 2: 7, 3: 6, 4: 3}                                                 # resampler.cu: Rtab


def _nb():
    import newsched_b200 as nb
    return nb


def _sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------ geometry
def _dg_nt(D):
    return 32 if D >= 9 else 64 if D >= 3 else 128


def _ols_block(T, D, real, env):
    """(outputs per overlap-save block, kernel) as fir_ols.cu lays them out."""
    if not real and 2 <= D <= 16 and env.get("B200_OLS_POLY", "1") != "0" and 4096 - -(-T // D) >= 1024:
        return 4096 - -(-T // D), "olsd"
    two = int(env.get("B200_OLS_TWO", "1024"))
    if not real and D == 1 and T >= (two if two > 0 else 1 << 30) and 4095 - (T + 1) // 2 >= 1024:
        return 2 * (4095 - (T + 1) // 2), "ols2"
    q = 4 if real else 2
    Tp = T if -(-(T - 1) // q) * q <= 3072 else 2048
    ov = -(-(Tp - 1) // q) * q
    V = (4096 - ov) // (q * D) * (q * D)
    return V * (2 if real else 1) // D, "ols4096"


class Case:
    """One handle: a FirFilter (L == 1) or a RationalResampler (L > 1), the switches set at its creation, the
    algorithm it must report, the kernel its calls must launch (name with its template arguments, no spaces) and
    its tile (outputs per tile or block of that kernel)."""

    def __init__(self, name, T, D=1, cplxin=True, L=1, env=None, algorithm=0, expect=None, tile=None, kernel=None):
        self.env, self.algorithm, self.expect, self.kernel = dict(env or {}), algorithm, expect, kernel
        self.name = name + "".join(f"-{k[5:].lower()}={v}" for k, v in self.env.items())
        self.T, self.D, self.cplx, self.L = T, D, cplxin, L
        self.resampler = L > 1
        self.tile = tile                      # outputs
        self.tile_in = -(-tile * D // L)      # inputs
        self.simt = self.resampler or expect in (1, 4)

    @property
    def hist_len(self):
        return -(-self.T // self.L) - 1

    def n_out(self, n_in):
        return n_in // self.D * self.L

    def __repr__(self):
        return self.name


R_C, R_R = 16, 32   # outputs per thread row: complex / real


def _fd(V, decim=False, DD=1, LL=1, RP=False, DG=1):
    """fir_direct_kernel<VEC, DECIM, DD, LL, RP, DG> as the profiler names it."""
    b = lambda v: "true" if v else "false"
    return f"fir_direct_kernel<{V},{b(decim)},{DD},{LL},{b(RP)},{DG}>"


def direct(T, cplxin=True, scalar=False):
    if cplxin:
        return Case(f"fir_direct<2,false>-T{T}", T, expect=1, tile=128 * R_C, kernel=_fd(2))
    if scalar:
        return Case(f"fir_direct<1,false>-T{T}", T, cplxin=False, env={"B200_FIR_REAL_SCALAR": "1"}, expect=1,
                    tile=128 * R_R, kernel=_fd(1))
    return Case(f"fir_direct<RP>-T{T}", T, cplxin=False, expect=1, tile=128 * R_R, kernel=_fd(2, RP=True))


def dd(D, T, cplxin):
    R = R_C if cplxin else R_R
    return Case(f"fir_direct<{2 if cplxin else 1},false,DD={D}>-T{T}", T, D, cplxin, expect=1, tile=128 * R // D,
                kernel=_fd(2 if cplxin else 1, DD=D))


def dg(D, T, cplxin):
    R = R_C if cplxin else R_R
    return Case(f"fir_direct<{2 if cplxin else 1},DG={D}>-T{T}", T, D, cplxin, expect=1, tile=_dg_nt(D) * R,
                kernel=_fd(2 if cplxin else 1, DG=D))


def planes(D, T, cplxin):
    R = R_C if cplxin else R_R
    return Case(f"fir_direct<{2 if cplxin else 1},true>-D{D}-T{T}", T, D, cplxin, env={"B200_FIR_PLANES": "1"},
                expect=1, tile=128 * R, kernel=_fd(2 if cplxin else 1, decim=True))


def naive(D, T, cplxin, algorithm=0):
    how = "algo4" if algorithm else "auto"
    return Case(f"fir_naive<{2 if cplxin else 1}>-{how}-D{D}-T{T}", T, D, cplxin, algorithm=algorithm, expect=4,
                tile=256, kernel=f"fir_naive_kernel<{2 if cplxin else 1}>")


def ll(L, M, T, cplxin, env=None):
    R = R_C if cplxin else R_R
    nt = 64 if (L > 1 and M > 1) or L >= 4 else _dg_nt(M)
    return Case(f"fir_ll<{'c' if cplxin else 'r'},{L}/{M}>-T{T}", T, M, cplxin, L, env, tile=nt * R * L,
                kernel=_fd(2 if cplxin else 1, LL=L, DG=M))


def rb(D, cplxin, L=7, T=60, env=None):
    return Case(f"resample_rb<{2 if cplxin else 1},{D},{RB_R[D]}>-L{L}-T{T}", T, D, cplxin, L, env,
                tile=(256 // L * L) * RB_R[D], kernel=f"resample_rb_kernel<{2 if cplxin else 1},{D},{RB_R[D]}>")


def simple(cplxin, L=3, D=7, T=30, env=None):
    room = (6144 - -(-T // L) - 2) * L // D
    return Case(f"resample<{2 if cplxin else 1}>-L{L}-D{D}-T{T}", T, D, cplxin, L, env, tile=min(1024, room),
                kernel=f"resample_kernel<{2 if cplxin else 1}>")


def ols(T, D, cplxin, env=None, algorithm=0, tag=""):
    env = dict(env or {})
    blk, kern = _ols_block(T, D, not cplxin, env)
    if kern == "ols4096":
        kern = f"ols4096<{'false' if cplxin else 'true'}>"
    return Case(f"fir_{kern}{tag}-D{D}-T{T}", T, D, cplxin, env=env, algorithm=algorithm, expect=3, tile=blk,
                kernel=f"fir_{kern.replace('<', '_kernel<') if '<' in kern else kern + '_kernel'}")


def tc(T, D=1, cplxin=True, algorithm=0):
    ts = D == 1 and ((T - 1 + 15) // 16 * 16 + 64 <= 512)
    kern = f"tc_ts<{'false' if cplxin else 'true'}>" if ts else "tc_pipe"
    tile = (4096 if cplxin else 8192) if ts else 8192
    return Case(f"fir_{kern}-D{D}-T{T}", T, D, cplxin, algorithm=algorithm, expect=2, tile=tile,
                kernel=f"fir_{kern.replace('<', '_kernel<') if '<' in kern else kern + '_kernel'}")


# ------------------------------------------------------------------------------------------ helpers
def _taps(rng, T):
    h = (rng.uniform(-1, 1, T) / np.sqrt(T)).astype(np.float32)
    assert T == 1 or not np.array_equal(h, h[::-1])
    return h


def _signal(rng, n, cplxin):
    return cplx(rng, n) if cplxin else rng.uniform(-1, 1, n).astype(np.float32)


def _oracle(c, x, h, hist=None):
    if c.resampler:
        return o.resample(x, h, c.L, c.D, hist=hist)
    return o.fir(x, h, c.D, hist=hist, mt=bool(np.iscomplexobj(x)))   # (the fp64 oracle has threads for ccf only)


@functools.lru_cache(maxsize=8)
def _data(seed, T, D, L, cplxin, n, with_hist=False):
    """Taps, input (and a random history) of n items and the fp64 oracle output; shorter runs use prefixes
    (the filter is causal, so the oracle of a prefix is the prefix of the oracle)."""
    c = Case("", T, D, cplxin, L, tile=1)
    rng = np.random.default_rng([seed, T, D, L, int(cplxin), n])
    h = _taps(rng, T)
    x = _signal(rng, n, cplxin)
    hist = _signal(rng, c.hist_len, cplxin) if with_hist and c.hist_len > 0 else None
    return h, x, hist, _oracle(c, x, h, hist)


def _budget_n(c, n_in):
    """n_in capped so that the oracle does about MAC_BUDGET multiply-adds, but at least a tile and a bit."""
    cap = int(MAC_BUDGET / (c.T / c.L)) * c.D // c.L
    return max(min(n_in, cap), c.tile_in + 3 * c.D)


def _device(torch, x, off_bytes=0):
    """x on the device, starting off_bytes past a 16-byte boundary."""
    isz = x.itemsize
    assert off_bytes % isz == 0
    k = off_bytes // isz
    buf = torch.empty(x.size + k + 1, dtype=torch.complex64 if np.iscomplexobj(x) else torch.float32, device="cuda")
    xd = buf[k:k + x.size]
    if x.size:
        xd.copy_(torch.from_numpy(x))
    assert xd.data_ptr() % 16 == off_bytes % 16
    return xd


class _Guarded:
    """An output view of n items inside a device buffer pre-filled with the SENTINEL bit pattern, GUARD items on
    each side; the view starts off_bytes past a 16-byte boundary."""

    def __init__(self, torch, n, cplxin, off_bytes=0, device="cuda"):
        w = 2 if cplxin else 1
        assert off_bytes % (4 * w) == 0
        self.lead = GUARD * w + off_bytes // 4
        self.words = n * w
        self.buf = torch.full((self.lead + self.words + GUARD * w,), SENTINEL, dtype=torch.int32, device=device)
        self.view = self.buf[self.lead:self.lead + self.words].view(torch.complex64 if cplxin else torch.float32)
        assert self.view.data_ptr() % 16 == off_bytes % 16

    def check_untouched(self):
        before, after = self.buf[:self.lead], self.buf[self.lead + self.words:]
        bad = (before != SENTINEL).nonzero()
        assert bad.numel() == 0, f"written before the output: word {int(bad[0]) - self.lead} (of -{self.lead})"
        bad = (after != SENTINEL).nonzero()
        assert bad.numel() == 0, f"written past the output: word {int(bad[0])} after it"

    def host(self):
        return self.view.cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _blocks(n):
    """[lo, hi) of every 4096-item block; a ragged last block is the last 4096 items."""
    out = [(b, b + BLOCK) for b in range(0, n - n % BLOCK, BLOCK)]
    if n % BLOCK:
        out.append((max(n - BLOCK, 0), n))
    return out


def _check(y, ref, record_property=None, what=""):
    """Per block of 4096 output items: relative RMS error < TOL_RMS and worst item < TOL_ITEM of the block's
    reference RMS; every value finite.  Returns (worst relative RMS, worst item ratio)."""
    y = np.asarray(y)
    ref = np.asarray(ref)
    assert y.shape == ref.shape, (what, y.shape, ref.shape)
    if y.size == 0:
        return 0.0, 0.0
    fin = np.isfinite(y.view(np.float32))
    if not fin.all():
        i = int(np.argmin(fin)) // (2 if np.iscomplexobj(y) else 1)
        raise AssertionError(f"{what}item {i} of {y.size} is not finite ({y[i]})")
    wide = np.complex128 if np.iscomplexobj(y) else np.float64
    d = np.abs(y.astype(wide) - ref.astype(wide))
    r = np.abs(ref.astype(wide))
    worst_rms = worst_item = 0.0
    for b, (lo, hi) in enumerate(_blocks(y.size)):
        scale = np.sqrt(np.mean(r[lo:hi] ** 2))
        dd_ = d[lo:hi]
        if scale == 0:
            assert dd_.max() == 0, f"{what}block {b} (items {lo}..{hi}): reference zero, |error| {dd_.max():.3g}"
            continue
        rel = np.sqrt(np.mean(dd_ ** 2)) / scale
        item = dd_.max() / scale
        assert rel < TOL_RMS, f"{what}block {b} (items {lo}..{hi}) of {y.size}: relative RMS error {rel:.3g}"
        assert item < TOL_ITEM, \
            f"{what}block {b}, item {lo + int(dd_.argmax())} of {y.size}: |error| / block rms = {item:.3g}"
        worst_rms, worst_item = max(worst_rms, rel), max(worst_item, item)
    if record_property is not None:
        record_property("worst_rel_rms", float(worst_rms))
        record_property("worst_item_ratio", float(worst_item))
    return worst_rms, worst_item


def _make(monkeypatch, c, h, multiply_const=None, env=None):
    """The handle of case c, created with exactly the switches of c.env (and env) set."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in {**c.env, **(env or {})}.items():
        monkeypatch.setenv(k, v)
    nb = _nb()
    if c.resampler:
        assert multiply_const is None
        return nb.RationalResampler(h, c.L, c.D, is_complex=c.cplx)
    f = nb.FirFilter(h, c.D, is_complex=c.cplx, multiply_const=multiply_const, algorithm=c.algorithm)
    assert f.algorithm == c.expect, (c.name, f.algorithm)
    return f


def _launched(torch, fn):
    """fn() under torch.profiler: its result and the set of library kernels it launched, each named as in
    Case.kernel (the demangled name after the b200:: namespace, without its parameter list or spaces)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name.split("b200::", 1)[1].split("(", 1)[0].replace(" ", "") for e in prof.events()
             if "b200::" in e.name}
    return out, names


def _check_kernels(c, names, history=True):
    """The case's kernel ran, and nothing else but the history kernel of a stream call."""
    want = {c.kernel}
    if history and c.hist_len > 0:
        want.add("rs_hist_kernel" if c.resampler else "fir_hist_kernel")
    assert names == want, f"{c.name}: launched {sorted(names)}, expected {sorted(want)}"


def _work(torch, f, c, xd, off_bytes=0, segment=False, halo=None):
    """One call into a guarded output; returns the output on the host (the guard is checked)."""
    n_out = c.n_out(xd.numel())
    g = _Guarded(torch, n_out, c.cplx, off_bytes)
    if segment:
        y = f.work_segment(xd, halo, out=g.view)
    else:
        y, nc = f.work(xd, out=g.view)
        assert nc == xd.numel() // c.D * c.D
    torch.cuda.synchronize()
    assert y.numel() == n_out and (n_out == 0 or y.data_ptr() == g.view.data_ptr())
    g.check_untouched()
    return g.host()


# ----------------------------------------------------------------------------- 0. the helpers themselves
def test_block_check_and_guard_layout():
    """The block check finds a wrong item, a non-finite item and an error confined to one short block; the
    sentinel is a NaN; the block split covers a ragged tail with a whole block."""
    assert np.isnan(np.array([SENTINEL], np.uint32).view(np.float32)[0])
    assert _blocks(0) == [] and _blocks(5) == [(0, 5)] and _blocks(8192) == [(0, 4096), (4096, 8192)]
    assert _blocks(9000) == [(0, 4096), (4096, 8192), (9000 - 4096, 9000)]
    rng = np.random.default_rng(1)
    for cplxin in (True, False):
        c = Case("", 37, 3, cplxin, tile=1)
        h, x, hist, ref = _data(0, 37, 3, 1, cplxin, 3 * 5000 + 2, True)
        assert ref.size == 5000 and hist.size == 36
        assert np.array_equal(ref, _oracle(c, x, h, hist))
        y = ref.copy()
        _check(y, ref)
        y[4321] += np.float32(3e-4) * np.sqrt(np.mean(np.abs(ref) ** 2))     # 3e-4 of the rms, 4.7e-6 of the block
        with pytest.raises(AssertionError, match="item 4321"):
            _check(y, ref)
        y = ref.copy()
        y[17] = np.nan
        with pytest.raises(AssertionError, match="item 17 "):
            _check(y, ref)
        y = ref.copy()
        y[:BLOCK] *= np.float32(1 + 3e-5)        # a relative error of 3e-5 in one block only
        with pytest.raises(AssertionError, match="block 0 "):
            _check(y, ref)
    r = _data(0, 24, 2, 3, True, 1001)
    assert r[3].size == 1001 // 2 * 3 and np.array_equal(r[3], o.resample(r[1], r[0], 3, 2))
    assert Case("", 10, 7, L=3, tile=1).hist_len == 3 and rb(2, True).tile == 252 * 7
    assert _ols_block(512, 1, False, {}) == (3584, "ols4096") and _ols_block(512, 1, True, {}) == (2 * 3584, "ols4096")
    assert _ols_block(2048, 1, False, {})[1] == "ols2" and _ols_block(2048, 1, False, {"B200_OLS_TWO": "0"})[1] == "ols4096"
    assert _ols_block(32768, 1, True, {}) == (2 * 2048, "ols4096") and _ols_block(256, 4, False, {}) == (4032, "olsd")


def test_guarded_output_detects_stray_writes():
    """The sentinel buffer (on the host here) passes a write that stays inside the view and reports the first
    word written before or after it."""
    import torch
    for cplxin, off in ((True, 0), (True, 8), (False, 4), (False, 12)):
        g = _Guarded(torch, 7, cplxin, off, device="cpu")
        assert g.view.numel() == 7 and np.isnan(g.host().view(np.float32)).all()
        g.view.fill_(1)
        g.check_untouched()
        g.buf[g.lead - 1] = 0
        with pytest.raises(AssertionError, match="written before the output: word -1 "):
            g.check_untouched()
        g.buf[g.lead - 1] = SENTINEL
        g.buf[g.lead + g.words + 2] = 0
        with pytest.raises(AssertionError, match="written past the output: word 2 "):
            g.check_untouched()


# --------------------------------------------------------------------------- 1. every instantiation once
MATRIX = (
    [direct(32), direct(32, False), direct(32, False, scalar=True), direct(7), direct(7, False)]
    + [dd(D, 64, True) for D in (2, 4, 8, 16)] + [dd(D, 64, False) for D in (2, 4, 8, 16, 32)]
    + [dd(4, 5, True), dd(32, 9, False)]
    + [dg(D, TX_C[D], True) for D in DG] + [dg(D, 7, True) for D in DG]
    + [dg(D, TX_R[D], False) for D in DG] + [dg(D, 7, False) for D in DG]
    + [planes(D, 48, cplxin) for D in (2, 3, 5, 12) for cplxin in (True, False)]
    + [naive(20, 64, False), naive(17, 1, True), naive(3, 100, True, 4), naive(1, 100, False, 4)]
    + [ll(2, 1, 48, True), ll(3, 1, 48, True), ll(4, 1, 192, True), ll(2, 3, 48, True), ll(2, 5, 48, True),
       ll(3, 2, 48, True), ll(3, 4, 48, True), ll(3, 5, 48, True), ll(4, 3, 48, True), ll(4, 5, 48, True),
       ll(5, 2, 50, True, {"B200_RATIONAL_MINTQ": "1"}), ll(5, 3, 48, True), ll(5, 4, 240, True)]
    + [ll(2, 1, 48, False), ll(3, 1, 48, False), ll(4, 1, 192, False), ll(2, 3, 64, False), ll(2, 5, 48, False),
       ll(3, 5, 96, False), ll(4, 5, 256, False)]
    + [ll(L, M, 48, False, {"B200_RATIONAL_MINTQ": "1"}) for L, M in ((3, 2), (3, 4), (4, 3), (5, 2), (5, 3), (5, 4))]
    + [ll(4, 1, 64, True, {"B200_INTERP_L4_MIN": "64"})]
    + [rb(D, cplxin) for D in (1, 2, 3, 4) for cplxin in (True, False)]
    + [simple(True), simple(False), simple(True, 8, 5, 64), simple(False, 8, 5, 64), rb(2, True, 3, 48, {"B200_RATIONAL_RB": "1"}),
       simple(True, 3, 2, 48, {"B200_RATIONAL_RB": "1", "B200_RESAMPLER_SIMPLE": "1"})]
    + [ols(512, 1, True), ols(4000, 1, True, {"B200_OLS_TWO": "0"}, tag="-2parts"),
       ols(32768, 1, True, tag="-16parts"), ols(600, 1, False), ols(4000, 1, False, tag="-2parts"),
       ols(32768, 1, False, tag="-16parts"), ols(1024, 4, False)]
    + [ols(128, 2, True), ols(256, 4, True), ols(1024, 16, True), ols(300, 3, True), ols(600, 11, True),
       ols(500, 13, True), ols(600, 15, True), ols(2048, 1, True)]
    + [tc(64), tc(64, cplxin=False), tc(128, 2, algorithm=2), tc(600, 1, algorithm=2)]
)


@gpu
@pytest.mark.parametrize("c", MATRIX, ids=repr)
def test_fir_path_matrix(cuda, monkeypatch, record_property, c):
    """Three tiles, a third of one and a ragged end in one call; a FIR handle starts from a random history."""
    n = _budget_n(c, 3 * c.tile_in + c.tile_in // 3 + 1 + (c.D - 1))
    h, x, hist, ref = _data(1, c.T, c.D, c.L, c.cplx, n, not c.resampler)
    f = _make(monkeypatch, c, h)
    if hist is not None:
        f.set_history(cuda.from_numpy(hist).cuda())
    xd = _device(cuda, x)
    y, names = _launched(cuda, lambda: _work(cuda, f, c, xd))
    _check_kernels(c, names)
    _check(y, ref, record_property)


# ---------------------------------------------------------------------------- one handle of every family
FAMILIES = [
    direct(32), direct(32, False), direct(32, False, scalar=True), dd(4, 64, True), dd(32, 64, False),
    dg(12, 64, True), dg(7, 48, True), dg(12, 64, False), dg(5, 33, False), planes(5, 48, True), planes(12, 48, False),
    naive(3, 40, True, 4), naive(20, 64, False), ll(3, 2, 48, True), ll(2, 1, 48, False), ll(4, 1, 192, True),
    ll(2, 5, 48, False), rb(2, True), rb(3, False), simple(True), simple(False, 8, 5, 64), ols(512, 1, True), ols(600, 1, False),
    ols(4000, 1, True, {"B200_OLS_TWO": "0"}, tag="-2parts"), ols(256, 4, True), ols(300, 3, True),
    ols(2048, 1, True), tc(64), tc(64, cplxin=False), tc(128, 2, algorithm=2),
]


def _fam_n(c):
    return _budget_n(c, max(2 * c.tile_in + c.tile_in // 3 + 1, 6 * c.T + 2 * c.tile_in + 101))


# ------------------------------------------------------------------------------------------- 2. tile edges
@gpu
@pytest.mark.parametrize("c", FAMILIES, ids=repr)
def test_fir_tile_edges(cuda, monkeypatch, record_property, c):
    """Input lengths 0, 1, D - 1, D, D + 1 and a tile - 1, a tile, a tile + 1 (and of outputs: a tile + D), each
    after reset() from zero history; a call without outputs launches nothing and writes nothing."""
    nb = _nb()
    k = c.tile_in
    lengths = sorted({m for m in (0, 1, c.D - 1, c.D, c.D + 1, k - 1, k, k + 1, k + c.D) if m >= 0})
    h, x, _, ref = _data(2, c.T, c.D, c.L, c.cplx, lengths[-1])
    f = _make(monkeypatch, c, h)
    xd = _device(cuda, x)
    worst = [0.0, 0.0]
    for m in lengths:
        f.reset()
        cuda.cuda.synchronize()
        before = nb.launch_count()
        y = _work(cuda, f, c, xd[:m])
        if c.n_out(m) == 0:
            assert nb.launch_count() == before, f"{m} inputs, no output: launched"
        w = _check(y, ref[:c.n_out(m)], what=f"{m} inputs: ")
        worst = [max(worst[0], w[0]), max(worst[1], w[1])]
    record_property("worst_rel_rms", worst[0])
    record_property("worst_item_ratio", worst[1])


# --------------------------------------------------------------------------------------- 3. persistent loops
PERSISTENT = [
    ols(16, 1, True, algorithm=3), ols(16, 1, False, algorithm=3), ols(32, 4, True, algorithm=3),
    ols(44, 11, True, algorithm=3), ols(32, 1, True, {"B200_OLS_TWO": "2"}, algorithm=3),
    tc(16, algorithm=2), tc(16, cplxin=False, algorithm=2), tc(16, 2, algorithm=2),
]


def _grid(torch, c):
    sms = _sms(torch)
    if c.expect == 2:
        return sms
    return sms if "olsd" in c.name and c.D > 10 else 2 * sms


@gpu
@pytest.mark.parametrize("which", ["grid-1", "grid+1", "2grid+1"])
@pytest.mark.parametrize("c", PERSISTENT, ids=repr)
def test_fir_persistent_loop(cuda, monkeypatch, record_property, c, which):
    """grid - 1, grid + 1 and 2 grid + 1 blocks (tiles) with a ragged last one: some CTAs run a second and a
    third iteration (mbarrier phase flips, the prefetch of the next block)."""
    grid = _grid(cuda, c)
    blocks = {"grid-1": grid - 1, "grid+1": grid + 1, "2grid+1": 2 * grid + 1}[which]
    n_out = (blocks - 1) * c.tile + c.tile // 2 + 1
    h, x, _, ref = _data(3, c.T, c.D, c.L, c.cplx, (2 * grid + 1) * c.tile * c.D)
    f = _make(monkeypatch, c, h)
    xd = _device(cuda, x[:n_out * c.D])
    y, names = _launched(cuda, lambda: _work(cuda, f, c, xd))
    _check_kernels(c, names)
    _check(y, ref[:n_out], record_property)


# ------------------------------------------------------------------------------------------- 4. alignment
def _align_rows():
    rows = []
    for c in FAMILIES:
        offs = ["in8", "out8"] if c.cplx else ["in4", "in8", "in12", "out4"]
        if c.expect == 1:
            offs.append("fir_tma0")
        if "olsd" in c.name and c.D % 2 == 0:
            offs.append("ols_tma0")
        rows += [pytest.param(c, v, id=f"{c.name}-{v}") for v in offs]
    return rows


@gpu
@pytest.mark.parametrize("c,variant", _align_rows())
def test_fir_alignment(cuda, monkeypatch, record_property, c, variant):
    """Input 8 (complex) or 4 / 8 / 12 (real) bytes off a 16-byte boundary, output 8 / 4 bytes off, or the bulk
    copies switched off with aligned pointers: against the oracle, and bit-equal to the aligned call for the
    SIMT forms and the resampler (same sums, whatever the staging)."""
    n = _fam_n(c)
    h, x, _, ref = _data(4, c.T, c.D, c.L, c.cplx, n)
    aligned = _work(cuda, _make(monkeypatch, c, h), c, _device(cuda, x))
    in_off = int(variant[2:]) if variant.startswith("in") else 0
    out_off = int(variant[3:]) if variant.startswith("out") else 0
    f = _make(monkeypatch, c, h, env={"B200_FIR_TMA": "0"} if variant == "fir_tma0" else None)
    if variant == "ols_tma0":
        monkeypatch.setenv("B200_OLS_TMA", "0")                 # read at launch
    y = _work(cuda, f, c, _device(cuda, x, in_off), out_off)
    _check(y, ref, record_property)
    if c.simt:
        assert np.array_equal(_bits(y), _bits(aligned))


# ---------------------------------------------------------------------------------- 5. streams, history
def _stream(torch, f, c, xd, g, chunks):
    """Feed xd in the given chunk lengths (then the rest) into consecutive views of g, without a sync."""
    pos = o_ = 0
    n = xd.numel()
    for m in list(chunks) + [n]:
        m = min(m, n - pos)
        seg = xd[pos:pos + m]
        k = c.n_out(m)
        y, used = f.work(seg, out=g.view[o_:o_ + k])
        assert used == m // c.D * c.D and y.numel() == k
        pos += used
        o_ += k
        if n - pos < c.D:
            break
    return pos, o_


@gpu
@pytest.mark.parametrize("c", FAMILIES, ids=repr)
def test_fir_stream_without_host_sync(cuda, monkeypatch, record_property, c):
    """Chunks of 1, T - 1, T, a tile - 1, a tile + 1 and the rest queued back to back into one guarded output,
    one synchronise at the end: each call's filter kernel overlaps the history kernel of the call before it.
    Against the oracle; bit-identical to one call for the SIMT forms and the resampler.  Then the handle's
    history is the last T - 1 inputs exactly, a fresh handle given that history continues the stream as the
    oracle does, and after reset() the handle equals a fresh one."""
    torch = cuda
    n = _fam_n(c)
    h, x, _, ref = _data(5, c.T, c.D, c.L, c.cplx, n)
    xd = _device(torch, x)
    f = _make(monkeypatch, c, h)
    g = _Guarded(torch, c.n_out(n), c.cplx)
    pos, n_o = _stream(torch, f, c, xd, g, (1, c.T - 1, c.T, c.tile_in - 1, c.tile_in + 1))
    torch.cuda.synchronize()
    g.check_untouched()
    assert pos == n // c.D * c.D and n_o == c.n_out(n)
    y = g.host()
    _check(y, ref, record_property)
    if c.simt:
        one = _work(torch, _make(monkeypatch, c, h), c, xd)
        assert np.array_equal(_bits(y), _bits(one)), "chunked != one shot"
    x2 = _data(6, c.T, c.D, c.L, c.cplx, c.tile_in + 3 * c.D + c.T)[1]
    x2d = _device(torch, x2)
    if not c.resampler and c.T > 1:
        hist = f.get_history()
        torch.cuda.synchronize()
        assert np.array_equal(_bits(hist.cpu().numpy()), _bits(x[pos - (c.T - 1):pos])), "history != last T-1 inputs"
        f2 = _make(monkeypatch, c, h)
        f2.set_history(hist)
        _check(_work(torch, f2, c, x2d), _oracle(c, x2, h, x[pos - (c.T - 1):pos]), what="set_history: ")
    f.reset()
    after = _work(torch, f, c, x2d)
    fresh = _work(torch, _make(monkeypatch, c, h), c, x2d)
    assert np.array_equal(_bits(after), _bits(fresh)), "reset() != fresh handle"


# ---------------------------------------------------------------------------------------- 6. time segments
@gpu
@pytest.mark.parametrize("c", FAMILIES, ids=repr)
def test_fir_segments_with_halo(cuda, monkeypatch, record_property, c):
    """Three time segments, each with the inputs before it as the halo (the first with none), run by one handle
    after a call that left a history the segments must not read: against the oracle, and bit-identical to one
    stream for the SIMT forms and the resampler."""
    torch = cuda
    n = _fam_n(c)
    h, x, _, ref = _data(7, c.T, c.D, c.L, c.cplx, n)
    xd = _device(torch, x)
    f = _make(monkeypatch, c, h)
    f.work(xd[n // 2:])                                         # a non-zero history
    H = c.hist_len
    cuts = [0, (n // 3) // c.D * c.D + c.D * 3, (2 * n // 3) // c.D * c.D + c.D, n // c.D * c.D]
    parts = []
    for lo, hi in zip(cuts, cuts[1:]):
        halo = xd[lo - H:lo] if lo and H else None
        parts.append(_work(torch, f, c, xd[lo:hi], segment=True, halo=halo))
    y = np.concatenate(parts)
    _check(y, ref[:y.size], record_property)
    if c.simt:
        one = _work(torch, _make(monkeypatch, c, h), c, xd)
        assert np.array_equal(_bits(y), _bits(one[:y.size])), "segments != one stream"


# ------------------------------------------------------------------------------------ 7. two handles, one stream
PAIRS = [
    pytest.param(tc(64), ols(2048, 1, True), id="tc_ts-T64+ols2-T2048"),
    pytest.param(dg(12, 64, True), ll(3, 2, 48, True), id="dg12+fir_ll<c,3/2>"),
    pytest.param(ols(600, 1, False), direct(32, False), id="ols4096<true>+RP"),
]


@gpu
@pytest.mark.parametrize("a,b", PAIRS)
def test_fir_two_handles_on_one_stream(cuda, monkeypatch, a, b):
    """Chunks of two handles of different forms alternate on one stream with one synchronise at the end, as two
    blocks of a flowgraph run: each output is bit-identical to the same chunks run by its handle alone, and
    matches the oracle."""
    torch = cuda
    runs = []
    for i, c in enumerate((a, b)):
        n = _fam_n(c)
        h, x, _, ref = _data(8 + i, c.T, c.D, c.L, c.cplx, n)
        runs.append((c, h, _device(torch, x), ref))
    chunks = (1, 63, 4097, 10001, 30011)

    def go(cs):
        state = [(_make(monkeypatch, c, h), _Guarded(torch, c.n_out(xd.numel()), c.cplx), 0, 0)
                 for c, h, xd, _ in cs]
        for m in list(chunks) + [1 << 40]:
            for i, (c, h, xd, _) in enumerate(cs):
                f, g, pos, o_ = state[i]
                mm = min(m, xd.numel() - pos)
                k = c.n_out(mm)
                _, used = f.work(xd[pos:pos + mm], out=g.view[o_:o_ + k])
                state[i] = (f, g, pos + used, o_ + k)
        torch.cuda.synchronize()
        for f, g, _, _ in state:
            g.check_untouched()
        return [g.host() for _, g, _, _ in state]

    together = go(runs)
    for r, y in zip(runs, together):
        alone = go([r])[0]
        assert np.array_equal(_bits(y), _bits(alone)), r[0].name
        _check(y, r[3], what=r[0].name + ": ")


# ----------------------------------------------------------------------------------- 8. fused multiply_const
FUSED = [c for c in FAMILIES if not c.resampler] + [naive(17, 1, True)]


@gpu
@pytest.mark.parametrize("c", FUSED, ids=repr)
def test_fir_fused_multiply_const(cuda, monkeypatch, record_property, c):
    """multiply_const fused into the epilogue: bit-exact against the two-block chain (filter, then multiply_const)
    for the SIMT forms (algorithms 1 and 4), within tolerance of the oracle times the constant for the tensor-core
    and overlap-save forms (whose constant is folded into the taps or the spectrum)."""
    n = _fam_n(c)
    h, x, _, ref = _data(10, c.T, c.D, c.L, c.cplx, n)
    xd = _device(cuda, x)
    k = (0.5 - 0.25j) if c.cplx else 3.25
    y = _work(cuda, _make(monkeypatch, c, h, multiply_const=k), c, xd)
    if c.simt:
        plain = _work(cuda, _make(monkeypatch, c, h), c, xd)
        chain = o.multiply_const(plain, k) if c.cplx else plain * np.float32(k)
        assert np.array_equal(_bits(y), _bits(chain)), "fused epilogue != two-block chain"
    wide = np.complex128 if c.cplx else np.float64
    _check(y, ref.astype(wide) * k, record_property)

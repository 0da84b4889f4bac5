"""Every FFT kernel path of b200_fft_run (fft.cu) against the fp64 oracle.

b200_fft_run picks one of seven kernel families from N, the pointer alignments and two create-time
switches, each instantiated for forward / reverse x {complex, |.|, |.|^2}:
    N = 8          fft8_kernel (in and out 16-byte aligned), else fft_generic_kernel
    N = 16..128    fft_small_kernel (4096 samples per CTA loop iteration, TMA-staged when the input is
                   16-byte aligned and the block is full, direct loads otherwise)
    N = 256..2048  fft_r0_kernel (same scheme)
    N = 4096       fft4096_tma_kernel (input 16-byte aligned, B200_FFT_TMA not 0), else fft4096_kernel
    N = 8192       fft8192_kernel (in and out 16-byte aligned, B200_FFT_GENERIC unset), else fft_generic_kernel
The shift, the reverse-shift sign and a fused multiply_const are folded into each family's tables at
create time, each family differently, so every combination is checked at every N.

Every case checks, per vector: the relative RMS error, the worst single bin relative to the RMS of its
reference vector (one wrong bin or one stale vector cannot hide behind the others), and that the
output buffer is untouched before and after the n_vec * N items the call owns."""
import numpy as np
import pytest

import oracle as o
from conftest import cplx

pytestmark = pytest.mark.gpu

NS = [8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
BLOCKED_NS = [16, 32, 64, 128, 256, 512, 1024, 2048]   # fft_small_kernel / fft_r0_kernel
OUTS = ["complex", "mag", "mag2"]
TOL_RMS = {"complex": 1e-5, "mag": 1e-5, "mag2": 2e-5}
TOL_BIN = 1e-4
K = 0.5 - 0.25j
SENTINEL = 0x7FBADBAD      # a float32 NaN: an output item the kernel fails to write cannot pass either
LEAD_BYTES = 256           # sentinel words in front of the output, plus the misalignment under test
GUARD_ITEMS = 8192         # sentinel items behind it: a whole stray vector or 4096-sample block


def _nb():
    import newsched_b200 as nb
    return nb


def _mode(out):
    nb = _nb()
    return {"complex": nb.OUT_COMPLEX, "mag": nb.OUT_MAG, "mag2": nb.OUT_MAG_SQUARED}[out]


def _sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _grid(torch):
    # persistent grid of the blocked, 4096 and 8192 kernels: two CTAs per SM (fft.cu, b200_fft_create)
    return 2 * _sms(torch)


def _block_vectors(N):
    # vectors per loop iteration of fft_small_kernel / fft_r0_kernel: one 4096-sample block
    return 4096 // N


def _device_input(torch, x, offset):
    """x on the device, `offset` complex items into its allocation (offset 1: 8-byte but not 16-byte aligned)."""
    buf = torch.empty(x.size + offset, dtype=torch.complex64, device="cuda")
    buf[offset:].copy_(torch.from_numpy(x))
    xd = buf[offset:]
    assert xd.data_ptr() % 16 == 8 * offset % 16
    return xd


class _Guarded:
    """An output view of n items inside a device buffer pre-filled with the SENTINEL bit pattern.
    misaligned: the view starts 8 bytes (complex) or 4 bytes (float) off a 16-byte boundary."""

    def __init__(self, torch, out, n, misaligned=False):
        self.item = 8 if out == "complex" else 4
        self.lead = LEAD_BYTES // self.item + (1 if misaligned else 0)
        self.n = n
        words = self.item // 4
        self.buf = torch.full(((self.lead + n + GUARD_ITEMS) * words,), SENTINEL, dtype=torch.int32, device="cuda")
        dtype = torch.complex64 if out == "complex" else torch.float32
        self.view = self.buf.view(dtype)[self.lead:self.lead + n]
        assert self.view.data_ptr() % 16 == (self.item if misaligned else 0)

    def check_untouched(self):
        words = self.buf.cpu().numpy()
        w = self.item // 4
        before, after = words[:self.lead * w], words[(self.lead + self.n) * w:]
        assert (before == SENTINEL).all(), f"written before the output: word {int(np.argmax(before != SENTINEL))}"
        assert (after == SENTINEL).all(), f"written past the output: word {int(np.argmax(after != SENTINEL))}"


def _reference(x, N, fwd, w, shift, out, k):
    ref = o.fft(o.multiply_const(x, k) if k is not None else x, N, fwd, w, shift).astype(np.complex128)
    if out == "mag":
        return np.abs(ref)
    if out == "mag2":
        return np.abs(ref) ** 2
    return ref


def _check_vectors(y, ref, N, out, record_property=None):
    """Per vector: relative RMS error and worst single bin, both relative to the reference vector's RMS."""
    y = np.asarray(y).reshape(-1, N)
    ref = ref.reshape(-1, N)
    assert y.shape == ref.shape
    assert np.isfinite(y).all(), f"vector {int(np.argmax(~np.isfinite(y).all(axis=1)))} holds a non-finite value"
    d = np.abs(y.astype(ref.dtype) - ref)
    scale = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    rel_rms = np.sqrt(np.mean(d ** 2, axis=1)) / scale
    worst_bin = d.max(axis=1) / scale
    if record_property is not None:
        record_property("worst_rel_rms", float(rel_rms.max()))
        record_property("worst_bin_ratio", float(worst_bin.max()))
    v = int(rel_rms.argmax())
    assert rel_rms[v] < TOL_RMS[out], f"vector {v} of {len(ref)}: relative RMS error {rel_rms[v]:.3g}"
    v = int(worst_bin.argmax())
    b = int(d[v].argmax())
    assert worst_bin[v] < TOL_BIN, f"vector {v} of {len(ref)}, bin {b}: |error| / rms = {worst_bin[v]:.3g}"


def _run_case(torch, N, n_vec, *, fwd=True, shift=False, out="complex", k=None, window=True, in_offset=0,
              out_misaligned=False, tail=0, seed=0, record_property=None):
    """One call of FFT.work on n_vec * N + tail input items, checked against the oracle."""
    nb = _nb()
    rng = np.random.default_rng([N, n_vec, int(fwd), int(shift), len(out), int(k is not None), int(window),
                                 in_offset, int(out_misaligned), tail, seed])
    x = cplx(rng, n_vec * N + tail)
    w = rng.uniform(0.1, 1, N).astype(np.float32) if window else None
    xd = _device_input(torch, x, in_offset)
    g = _Guarded(torch, out, n_vec * N, out_misaligned)
    fft = nb.FFT(N, fwd, w, shift, output=_mode(out), pre_multiply_const=k)
    y = fft.work(xd, out=g.view)
    torch.cuda.synchronize()
    assert y.data_ptr() == g.view.data_ptr() and y.numel() == n_vec * N
    g.check_untouched()
    _check_vectors(y.cpu().numpy(), _reference(x[:n_vec * N], N, fwd, w, shift, out, k), N, out, record_property)


def _matrix_vectors(torch, N):
    """Group 1 sizes: for the blocked kernels every CTA runs more than one loop iteration and the last block
    is partial; at 4096 and 8192 a few CTAs run a second vector."""
    if N <= 2048:
        return (2 * _grid(torch) + 1) * _block_vectors(N) - 3
    return _grid(torch) + 3


# ---------------------------------------------------------------------------------- 1. fused-form matrix
@pytest.mark.parametrize("k", [None, K], ids=["nok", "k"])
@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("shift", [False, True], ids=["noshift", "shift"])
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", NS)
def test_fft_fused_forms(cuda, record_property, N, fwd, shift, out, k):
    """Window in (0.1, 1) x direction x shift x output form x fused multiply_const."""
    _run_case(cuda, N, _matrix_vectors(cuda, N), fwd=fwd, shift=shift, out=out, k=k,
              record_property=record_property)


@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", NS)
def test_fft_fused_forms_no_window(cuda, record_property, N, fwd, out):
    """No window: the shift alone is folded into a table of +-1 (forward) or the output sign (reverse)."""
    _run_case(cuda, N, _matrix_vectors(cuda, N), fwd=fwd, shift=True, out=out, window=False,
              record_property=record_property)


# ------------------------------------------------------------------------ 2. persistent loop of each size
BLOCK_COUNTS = ["one", "grid_minus_1", "grid_plus_1", "two_grids_plus_1", "three_grids_plus_2"]


@pytest.mark.parametrize("out", ["complex", "mag"])
@pytest.mark.parametrize("last", ["full", "partial"])
@pytest.mark.parametrize("blocks", BLOCK_COUNTS)
@pytest.mark.parametrize("N", BLOCKED_NS)
def test_fft_persistent_loop(cuda, record_property, N, blocks, last, out):
    """Block counts around one, two and three grids: CTAs with no block, one, two and three loop iterations
    (the mbarrier phase goes 0 -> 1 -> 0), and a TMA-staged block followed by a partial one loaded directly."""
    g = _grid(cuda)
    nb_ = {"one": 1, "grid_minus_1": g - 1, "grid_plus_1": g + 1, "two_grids_plus_1": 2 * g + 1,
           "three_grids_plus_2": 3 * g + 2}[blocks]
    n_vec = nb_ * _block_vectors(N) - (1 if last == "partial" else 0)
    _run_case(cuda, N, n_vec, out=out, record_property=record_property)


@pytest.mark.parametrize("out", OUTS)
def test_fft8_grid_stride_loop(cuda, record_property, out):
    """fft8_kernel runs at most 16 blocks of 256 threads per SM, one vector per thread per iteration: a count
    past two full sweeps makes some threads loop three times."""
    cap = 16 * _sms(cuda) * 256
    _run_case(cuda, 8, 2 * cap + 3, out=out, record_property=record_property)


# ----------------------------------------------------------------------------------- 3. fallback kernels
def _fallback_vectors(torch, N):
    if N <= 2048:
        return (_grid(torch) + 1) * _block_vectors(N) - 3   # one CTA loops twice, last block partial
    if N == 4096:
        return _grid(torch) + 5                                # fft4096_kernel loops
    return 5


@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", NS)
def test_fft_input_8_byte_aligned(cuda, record_property, N, fwd, out):
    """Input one complex item past a 16-byte boundary: direct loads in the blocked kernels, fft4096_kernel at
    4096, fft_generic_kernel at 8 and 8192."""
    _run_case(cuda, N, _fallback_vectors(cuda, N), fwd=fwd, shift=True, out=out, k=K, in_offset=1,
              record_property=record_property)


@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", NS)
def test_fft_output_not_16_byte_aligned(cuda, record_property, N, fwd, out):
    """Output 8 bytes (complex) or 4 bytes (float) past a 16-byte boundary: fft_generic_kernel at 8 and 8192."""
    n_vec = 3 * _block_vectors(N) - 1 if N <= 2048 else 3
    _run_case(cuda, N, n_vec, fwd=fwd, shift=True, out=out, k=K, out_misaligned=True,
              record_property=record_property)


FORCED = {4096: ("B200_FFT_TMA", "0"), 8192: ("B200_FFT_GENERIC", "1")}


@pytest.mark.parametrize("k", [None, K], ids=["nok", "k"])
@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("shift", [False, True], ids=["noshift", "shift"])
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", sorted(FORCED))
def test_fft_forced_fallback_fused_forms(cuda, monkeypatch, record_property, N, fwd, shift, out, k):
    """Aligned pointers, fallback chosen at create time: fft4096_kernel (B200_FFT_TMA=0) and fft_generic_kernel
    at 8192 (B200_FFT_GENERIC=1), over the fused-form matrix."""
    monkeypatch.setenv(*FORCED[N])
    _run_case(cuda, N, _fallback_vectors(cuda, N), fwd=fwd, shift=shift, out=out, k=k,
              record_property=record_property)


@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", sorted(FORCED))
def test_fft_forced_fallback_no_window(cuda, monkeypatch, record_property, N, fwd, out):
    monkeypatch.setenv(*FORCED[N])
    _run_case(cuda, N, _fallback_vectors(cuda, N), fwd=fwd, shift=True, out=out, window=False,
              record_property=record_property)


# ------------------------------------------------------------------------------------------- 4. bounds
@pytest.mark.parametrize("N", NS)
def test_fft_zero_vectors_writes_nothing(cuda, N):
    """Fewer than N input items: no vector, no launch, nothing written."""
    nb = _nb()
    torch = cuda
    for n_in in (0, N - 1):
        x = _device_input(torch, cplx(np.random.default_rng(n_in), n_in), 0)
        for out in ("complex", "mag"):
            fft = nb.FFT(N, output=_mode(out))
            g = _Guarded(torch, out, 0)
            before = nb.launch_count()
            assert fft.work(x, out=g.view).numel() == 0
            assert fft.work(x).numel() == 0
            assert nb.launch_count() == before
            torch.cuda.synchronize()
            g.check_untouched()


@pytest.mark.parametrize("out", ["complex", "mag"])
@pytest.mark.parametrize("N", NS)
def test_fft_trailing_partial_vector_is_ignored(cuda, record_property, N, out):
    """An input of 3 N + N/2 + 1 items is 3 vectors: the trailing items produce no output."""
    _run_case(cuda, N, 3, fwd=False, shift=True, out=out, k=K, tail=N // 2 + 1, record_property=record_property)
    x = _device_input(cuda, cplx(np.random.default_rng(N), 3 * N + N // 2 + 1), 0)
    assert _nb().FFT(N, output=_mode(out)).work(x).numel() == 3 * N


@pytest.mark.parametrize("out", OUTS)
@pytest.mark.parametrize("fwd", [True, False], ids=["fwd", "rev"])
@pytest.mark.parametrize("N", NS)
def test_fft_one_vector(cuda, record_property, N, fwd, out):
    _run_case(cuda, N, 1, fwd=fwd, shift=True, out=out, k=K, record_property=record_property)


# ------------------------------------------------------------------------------- 5. dependent launches
@pytest.mark.parametrize("N", [8, 64, 1024, 8192])
def test_fft_dependent_launches(cuda, N):
    """Launches queued on one stream without a host synchronisation, each reading what the one before it
    wrote. The blocked and 8192 kernels are dependent launches: their prologue overlaps the previous
    kernel's tail, their loads must not."""
    nb = _nb()
    torch = cuda
    rng = np.random.default_rng(N + 5)
    if N == 8:
        n_vec = 16 * _sms(torch) * 256 + 77    # past one sweep of fft8_kernel's grid
    elif N == 8192:
        n_vec = _grid(torch) + 7
    else:
        n_vec = _matrix_vectors(torch, N)
    x = cplx(rng, n_vec * N)
    w = rng.uniform(0.1, 1, N).astype(np.float32)
    fwd_c = nb.FFT(N, True, w)
    rev_c = nb.FFT(N, False)
    mag = nb.FFT(N, True, w, output=nb.OUT_MAG)
    mag2 = nb.FFT(N, False, w, True, output=nb.OUT_MAG_SQUARED)
    a = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    chain = []
    for _ in range(3):
        b = fwd_c.work(a)          # X = FFT(w x)
        c = rev_c.work(b)          # N * (w x)
        m = mag.work(c)            # |FFT(w N w x)|
        m2 = mag2.work(b)          # |IFFT(ifftshift(w X))|^2
        chain.append((a, b, c, m, m2))
        a = c * (1.0 / N)
    torch.cuda.synchronize()
    for a, b, c, m, m2 in chain:
        ah, bh, ch = a.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy()
        _check_vectors(bh, o.fft(ah, N, True, w).astype(np.complex128), N, "complex")
        _check_vectors(ch, o.fft(bh, N, False).astype(np.complex128), N, "complex")
        _check_vectors(m.cpu().numpy(), np.abs(o.fft(ch, N, True, w).astype(np.complex128)), N, "mag")
        _check_vectors(m2.cpu().numpy(), np.abs(o.fft(bh, N, False, w, True).astype(np.complex128)) ** 2, N, "mag2")


# -------------------------------------------------------------------------------- 6. create-time checks
@pytest.mark.parametrize("N", [0, 4, 12, 16384])
def test_fft_create_rejects_unsupported_length(cuda, N):
    nb = _nb()
    before = nb.launch_count()
    with pytest.raises(nb.B200Error, match="power of two"):
        nb.FFT(N)
    assert nb.launch_count() == before


@pytest.mark.parametrize("mode", [3, -1])
def test_fft_create_rejects_output_mode(cuda, mode):
    nb = _nb()
    before = nb.launch_count()
    with pytest.raises(nb.B200Error, match="output mode"):
        nb.FFT(4096, output=mode)
    assert nb.launch_count() == before

"""FFT-4096 TMA kernel (fft4096_tma_kernel): each vector is transformed in place in the input tile its
bulk copy landed in, with three tiles per CTA for the |.| / |.|^2 forms and two for complex output.
These tests drive the persistent loop through every tile and both mbarrier parities (vector counts
below, at and well above the grid, not multiples of three grids), every output form, both directions,
the folded shift and multiply_const, and dependent launches back to back on one stream."""
import numpy as np
import pytest

import oracle as o
from conftest import cplx

pytestmark = pytest.mark.gpu

N = 4096
TOL_RMS = 1e-5


def _grid(torch):
    # the launch's grid: two CTAs per SM (fft.cu, b200_fft_create)
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count


def _per_vector_rel_rms(y, ref):
    y = np.asarray(y).reshape(-1, N).astype(np.complex128)
    ref = np.asarray(ref).reshape(-1, N).astype(np.complex128)
    num = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1))
    den = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    return num / den


def _reference(x, fwd, w, shift, out, k=None):
    import newsched_b200 as nb
    ref = o.fft(o.multiply_const(x, k) if k is not None else x, N, fwd, w, shift).astype(np.complex128)
    if out == nb.OUT_MAG:
        return np.abs(ref)
    if out == nb.OUT_MAG_SQUARED:
        return np.abs(ref) ** 2
    return ref


def _run(torch, x, fwd, w, shift, out, k=None):
    import newsched_b200 as nb
    y = nb.FFT(N, fwd, w, shift, output=out, pre_multiply_const=k).work(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    return y.cpu().numpy()


def _outs():
    import newsched_b200 as nb
    return {"complex": nb.OUT_COMPLEX, "mag": nb.OUT_MAG, "mag2": nb.OUT_MAG_SQUARED}


@pytest.mark.parametrize("out", ["mag", "mag2", "complex"])
@pytest.mark.parametrize("shift", [False, True])
@pytest.mark.parametrize("fwd", [True, False])
def test_fft4096_inplace_matches_oracle(cuda, fwd, shift, out):
    """7 grids + 41 vectors: every CTA runs 7 or 8 vectors, i.e. wraps its tiles at least twice."""
    rng = np.random.default_rng(4096 + 4 * fwd + 2 * shift + len(out))
    n_vec = 7 * _grid(cuda) + 41
    x = cplx(rng, n_vec * N)
    w = o.window_blackmanharris(N)
    mode = _outs()[out]
    err = _per_vector_rel_rms(_run(cuda, x, fwd, w, shift, mode), _reference(x, fwd, w, shift, mode))
    assert err.max() < TOL_RMS, (int(err.argmax()), float(err.max()))


@pytest.mark.parametrize("out", ["mag", "mag2", "complex"])
@pytest.mark.parametrize("fwd", [True, False])
def test_fft4096_inplace_fused_multiply_const(cuda, fwd, out):
    rng = np.random.default_rng(77 + fwd + len(out))
    n_vec = 3 * _grid(cuda) + 5
    x = cplx(rng, n_vec * N)
    w = rng.uniform(0.1, 1, N).astype(np.float32)
    k = 0.5 - 0.25j
    mode = _outs()[out]
    err = _per_vector_rel_rms(_run(cuda, x, fwd, w, False, mode, k), _reference(x, fwd, w, False, mode, k))
    assert err.max() < TOL_RMS, (int(err.argmax()), float(err.max()))


@pytest.mark.parametrize("which", ["one", "third_of_grid", "grid_minus_1", "grid_plus_1", "three_grids_minus_1",
                                   "three_grids_plus_1", "six_grids_plus_2"])
@pytest.mark.parametrize("out", ["mag", "mag2", "complex"])
def test_fft4096_inplace_vector_counts(cuda, which, out):
    """Vector counts around the grid and around three grids: CTAs with no vector, with fewer vectors than
    tiles (no refill issued), and the last refill of every CTA."""
    g = _grid(cuda)
    n_vec = {"one": 1, "third_of_grid": g // 3, "grid_minus_1": g - 1, "grid_plus_1": g + 1,
             "three_grids_minus_1": 3 * g - 1, "three_grids_plus_1": 3 * g + 1, "six_grids_plus_2": 6 * g + 2}[which]
    rng = np.random.default_rng(n_vec)
    x = cplx(rng, n_vec * N)
    w = o.window_blackmanharris(N)
    mode = _outs()[out]
    err = _per_vector_rel_rms(_run(cuda, x, True, w, False, mode), _reference(x, True, w, False, mode))
    assert err.max() < TOL_RMS, (int(err.argmax()), float(err.max()))


def test_fft4096_inplace_back_to_back_launches(cuda):
    """Launches queued on one stream without a host synchronisation, each reading what the one before it
    wrote (dependent launch: a kernel's prologue overlaps its predecessor's tail, its loads must not)."""
    import newsched_b200 as nb
    torch = cuda
    rng = np.random.default_rng(5)
    n_vec = 2 * _grid(torch) + 77
    x = cplx(rng, n_vec * N)
    w = o.window_blackmanharris(N)
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
        for y, ref in ((bh, o.fft(ah, N, True, w)), (ch, o.fft(bh, N, False)),
                       (m.cpu().numpy(), np.abs(o.fft(ch, N, True, w).astype(np.complex128))),
                       (m2.cpu().numpy(), np.abs(o.fft(bh, N, False, w, True).astype(np.complex128)) ** 2)):
            err = _per_vector_rel_rms(y, ref)
            assert err.max() < TOL_RMS, (int(err.argmax()), float(err.max()))

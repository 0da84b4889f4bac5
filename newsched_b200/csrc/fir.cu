// fir.cu -- decimating FIR filter, ccf (complex64 stream, real taps) and fff (float stream).
//
//   y[m] = sum_{k<T} h[k] x[m*D - k],  m = 0 .. floor(n_in/D)-1      (SURVEY.md 8c)
//
// The reference snapshot has no FIR block (SURVEY.md 0.1); the work() contract it plugs
// into is gr::block::work (runtime/include/gnuradio/block.hpp:81-85) with
// n_consumed = n_produced*D set by the block (block_work_io.hpp:21,36).
//
// Direct-form SIMT kernel (algorithm 1), FP32-pipe bound for T >= 32 (SURVEY.md 8d):
//   * polyphase split: y = sum_p (h_p * x_p), h_p[q] = h[qD+p], x_p[j] = x[jD-p]; the
//     input tile is staged once into shared memory de-interleaved by phase, so every phase
//     is a unit-stride FIR and decimated-away products are never formed;
//   * each thread owns 32 fp32 accumulators (16 complex / 32 real consecutive outputs) and a
//     64-float circular register window over x_p; one step = 16 (32) taps = 512 (1024) FFMA
//     fed by 8 LDS.128 of samples + 4 (8) LDS.128 of taps (warp-uniform broadcast): the inner
//     loop is > 96 % FFMA issue slots;
//   * shared layout is padded 16 B per 128 B so that the per-thread 128 B-strided LDS.128
//     window reads are bank-conflict free;
//   * outputs go back through shared memory so global stores are fully coalesced.
// History (the T-1 samples before the next input item) lives in a ping-pong pair of small
// device buffers owned by the handle; nothing is re-read from the host and the caller may
// chunk the stream arbitrarily.
#include "fir_direct.cuh"

namespace b200 {

// Fallback for parameter combinations the tiled kernel cannot stage (very large D):
// one thread per output straight from global memory.
template <int VEC>
__global__ void __launch_bounds__(256)
    fir_naive_kernel(const float* __restrict__ x, const float* __restrict__ hist,
                     float* __restrict__ y, const float* __restrict__ taps, int T, int D,
                     long long n_in, long long n_out, fir_epilogue ep)
{
    long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_out)
        return;
    float a0 = 0.f, a1 = 0.f;
    for (int k = 0; k < T; k++) {
        float v[2];
        fir_fetch<VEC>(x, hist, T - 1, m * D - k, n_in, v);
        float h = __ldg(taps + k);
        a0 = fmaf(h, v[0], a0);
        if (VEC == 2)
            a1 = fmaf(h, v[1], a1);
    }
    if (VEC == 2) {
        float2 v = make_float2(a0, a1);
        if (ep.fuse)
            v = cmul_nofma(v, ep.kre, ep.kim);
        reinterpret_cast<float2*>(y)[m] = v;
    } else {
        y[m] = ep.fuse ? __fmul_rn(a0, ep.kre) : a0;
    }
}

// new_hist[j] = sample (n_consumed - Tm1 + j) of the stream (old history ++ x)
__global__ void fir_hist_kernel(const float* __restrict__ x, const float* __restrict__ hist_old,
                                float* __restrict__ hist_new, long long n_consumed, int Tm1, int VEC)
{
    // launched with programmatic stream serialization (B200_LAUNCH_PDL): the filter kernel of the NEXT work() call may
    // start its prologue right away; this kernel waits for the filter kernel in front of it (which still reads
    // hist_old's twin) before it touches anything
    pdl_launch_dependents();
    pdl_wait();
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Tm1)
        return;
    long long s = n_consumed - Tm1 + j;
    for (int c = 0; c < VEC; c++)
        hist_new[j * VEC + c] = (s >= 0) ? x[s * VEC + c] : hist_old[(Tm1 + s) * VEC + c];
}

} // namespace b200

using namespace b200;

struct b200_fir {
    int T = 0, D = 1, vec = 2;
    int TQ = 0;      // taps per phase, padded
    int plane_rows = 0, box_rows = 0, n_boxes = 0; // smem plane geometry (rows of 128 B)
    size_t smem = 0;
    int use_tma = 1;
    int rp = 0;      // real stream through the packed complex x real loop (fir_direct_kernel<..., RP>)
    int interp = 0;  // > 1: interpolation folded into the full-rate kernel (created by fir_interp_create)
    int dg = 0;      // > 1: decimation by a non-divisor of 16 folded into the full-rate kernel (D rows per thread)
    int dd = 0;      // > 1: decimation folded into the TMA-staged full-rate kernel (geometry as for D = 1)
    ols_plan* ols = nullptr; // algorithm 3
    tc_plan* tc = nullptr;   // algorithm 2
    int algorithm = 1;
    fir_epilogue ep{ 0, 1.f, 0.f };
    float* d_taps_pp = nullptr; // [D][TQ] reversed per phase
    float* d_taps = nullptr;    // [T] natural order (naive kernel)
    float* d_hist[2] = { nullptr, nullptr };
    int cur = 0;
    int device = 0;
};

// 2-D view of the input stream for TMA: rows of 32 floats (128 B), SWIZZLE_128B, box = box_rows
static int fir_make_tmap(CUtensorMap* tmap, const void* d_in, long long full_rows, int box_rows)
{
    tmap_encode_fn enc = tmap_encode_tiled();
    if (!enc)
        return set_err(B200_ERR_CUDA, "fir: cuTensorMapEncodeTiled unavailable");
    cuuint64_t gdim[2] = { 32, (cuuint64_t)full_rows };
    cuuint64_t gstride[1] = { 128 };
    cuuint32_t box[2] = { 32, (cuuint32_t)box_rows };
    cuuint32_t estr[2] = { 1, 1 };
    CUresult r = enc(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(d_in), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return set_err(B200_ERR_CUDA, "fir: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return B200_OK;
}

static int fir_launch(b200_fir* h, const float* d_hist, const void* d_in, void* d_out,
                      long long n_in, long long n_out, cudaStream_t s)
{
    if (n_out <= 0)
        return B200_OK;
    const float* x = (const float*)d_in;
    float* y = (float*)d_out;
    if (h->algorithm == 3)
        return ols_launch(h->ols, d_hist, d_in, d_out, n_in, n_out, s);
    if (h->algorithm == 2)
        return tc_launch(h->tc, d_hist, d_in, d_out, n_in, n_out, s);
    if (h->algorithm == 1 && h->rp) {
        // real stream as float pairs: tiles of 2048 pairs = 4096 real outputs
        const long long pairs_out = (n_out + 1) / 2, pairs_in = (n_in + 1) / 2;
        const int MTp = FIR_NT * (FIR_ACC / 2);
        const long long tiles = (pairs_out + MTp - 1) / MTp;
        if (tiles > 0x7fffffffLL)
            return set_err(B200_ERR_ARG, "fir: too many items for one call");
        fir_geom gm{};
        gm.Tm1 = h->T - 1;
        gm.D = 1;
        gm.TQ = h->TQ;
        gm.plane_rows = h->plane_rows;
        gm.box_rows = h->box_rows;
        gm.n_boxes = h->n_boxes;
        gm.n_in = pairs_in;
        gm.n_out = pairs_out;
        gm.n_in_f = n_in;
        gm.n_out_f = n_out;
        gm.full_rows = n_in / 32;
        gm.full_out_rows = n_out / 32;
        CUtensorMap tmap, tmap_out;
        memset(&tmap, 0, sizeof(tmap));
        memset(&tmap_out, 0, sizeof(tmap_out));
        if (h->use_tma && gm.full_rows >= h->plane_rows && (uintptr_t)d_in % 16 == 0 &&
            fir_make_tmap(&tmap, d_in, gm.full_rows, h->box_rows) == B200_OK)
            gm.tma_ok = 1;
        if (h->use_tma && gm.full_out_rows >= FIR_NT && (uintptr_t)d_out % 16 == 0 &&
            fir_make_tmap(&tmap_out, d_out, gm.full_out_rows, FIR_NT) == B200_OK)
            gm.tma_out_ok = 1;
        B200_LAUNCH((fir_direct_kernel<2, false, 1, 1, true>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,
                    h->d_taps_pp, tmap, tmap_out, gm, h->ep);
        return B200_OK;
    }
    if (h->algorithm == 1) {
        const int NTt = h->dg ? fir_dg_nt(h->dg) : FIR_NT;             // threads per tile
        const int MT = NTt * (FIR_ACC / h->vec) / (h->dd ? h->dd : 1); // outputs per tile
        long long tiles = (n_out + MT - 1) / MT;
        if (tiles > 0x7fffffffLL)
            return set_err(B200_ERR_ARG, "fir: too many items for one call");
        fir_geom gm{};
        gm.Tm1 = h->T - 1;
        gm.D = (h->dd || h->dg) ? 1 : h->D;
        gm.TQ = h->TQ;
        gm.plane_rows = h->plane_rows;
        gm.box_rows = h->box_rows;
        gm.n_boxes = h->n_boxes;
        gm.n_in = n_in;
        gm.n_out = n_out;
        gm.full_rows = n_in * h->vec / 32;
        gm.tma_ok = 0;
        CUtensorMap tmap;
        memset(&tmap, 0, sizeof(tmap));
        if (h->use_tma && (h->D == 1 || h->dd || h->dg) && gm.full_rows >= h->plane_rows && (uintptr_t)d_in % 16 == 0) {
            int rc = fir_make_tmap(&tmap, d_in, gm.full_rows, h->box_rows);
            if (rc != B200_OK)
                return rc;
            gm.tma_ok = 1;
        }
        CUtensorMap tmap_out;
        memset(&tmap_out, 0, sizeof(tmap_out));
        gm.full_out_rows = n_out * h->vec / 32;
        gm.tma_out_ok = 0;
        const int out_rows = NTt / (h->dd ? h->dd : 1); // rows of the output tile
        if (h->use_tma && out_rows >= 8 && gm.full_out_rows >= out_rows && (uintptr_t)d_out % 16 == 0) {
            int rc = fir_make_tmap(&tmap_out, d_out, gm.full_out_rows, out_rows);
            if (rc != B200_OK)
                return rc;
            gm.tma_out_ok = 1;
        }
        const bool decim = h->D > 1;
        if (h->dg) {
            const fir_args fa{ x, d_hist, y, h->d_taps_pp, tmap, tmap_out, gm, h->ep };
            const int rc = h->vec == 2 ? fir_dg_launch_c(h->dg, (unsigned)tiles, h->smem, s, fa)
                                       : fir_dg_launch_r(h->dg, (unsigned)tiles, h->smem, s, fa);
            if (rc != B200_OK)
                return rc;
        } else if (h->dd) {
#define FIR_DD(V, DDV)                                                                                     \
    B200_LAUNCH((fir_direct_kernel<V, false, DDV>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,     \
                h->d_taps_pp, tmap, tmap_out, gm, h->ep)
            if (h->vec == 2) {
                switch (h->dd) {
                case 2: FIR_DD(2, 2); break;
                case 4: FIR_DD(2, 4); break;
                case 8: FIR_DD(2, 8); break;
                default: FIR_DD(2, 16); break;
                }
            } else {
                switch (h->dd) {
                case 2: FIR_DD(1, 2); break;
                case 4: FIR_DD(1, 4); break;
                case 8: FIR_DD(1, 8); break;
                case 16: FIR_DD(1, 16); break;
                default: FIR_DD(1, 32); break;
                }
            }
#undef FIR_DD
        } else if (h->vec == 2) {
            if (decim)
                B200_LAUNCH((fir_direct_kernel<2, true>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,
                            h->d_taps_pp, tmap, tmap_out, gm, h->ep);
            else
                B200_LAUNCH((fir_direct_kernel<2, false>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,
                            h->d_taps_pp, tmap, tmap_out, gm, h->ep);
        } else {
            if (decim)
                B200_LAUNCH((fir_direct_kernel<1, true>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,
                            h->d_taps_pp, tmap, tmap_out, gm, h->ep);
            else
                B200_LAUNCH((fir_direct_kernel<1, false>), (unsigned)tiles, FIR_NT, h->smem, s, x, d_hist, y,
                            h->d_taps_pp, tmap, tmap_out, gm, h->ep);
        }
    } else {
        long long blocks = (n_out + 255) / 256;
        if (h->vec == 2)
            B200_LAUNCH((fir_naive_kernel<2>), (unsigned)blocks, 256, 0, s, x, d_hist, y, h->d_taps,
                        h->T, h->D, n_in, n_out, h->ep);
        else
            B200_LAUNCH((fir_naive_kernel<1>), (unsigned)blocks, 256, 0, s, x, d_hist, y, h->d_taps,
                        h->T, h->D, n_in, n_out, h->ep);
    }
    return B200_OK;
}

namespace b200 {

// (L, M) pairs the rational fold is instantiated for, and from how many taps per phase it beats the
// register-blocked resampler kernel (tools/resampler_sweep.py with RATIOS=1 and B200_RATIONAL_MINTQ=1 against
// B200_RATIONAL_RB=1; TFLOP/s fold vs kernel at 16 / 32 / 64 taps per phase): 3/2 17.7 / 28.7 / 41.6 vs 15.4 /
// 24.7 / 32.9, 2/3 15.5 / 25.4 / 37.2 vs 11.4 / 18.3 / 24.4, 4/3 12.5 / 20.4 / 28.4 vs 10.8 / 14.3 / 15.8,
// 3/4 10.5 / 17.1 / 24.7 vs 7.4 / 10.0 / 11.0, 4/5 6.6 / 11.5 / 17.6 vs 4.9 / 6.4 / 6.9, 5/3 14.8 / 23.4 / 30.4
// vs 10.9 / 14.2 / 15.8, 3/5 9.1 / 15.9 / 23.9 vs 4.3 / 6.1 / 6.7, 2/5 7.9 / 13.7 / 21.8 vs 3.5 / 5.4 / 6.4;
// 5/4 only from long phases (8.8 / 14.3 / 20.9 vs 10.7 / 15.1 / 18.4); 5/2 never (16.3 / 25.6 / 30.5 vs
// 16.6 / 25.8 / 33.5: its 5 x 64-row output tile leaves 3 two-warp CTAs per SM).
// Real streams (32 samples per row, scalar FMAs): the register-blocked kernel is the faster one except for
// the strongly decimating ratios (out GS/s fold vs kernel at 16 / 32 / 64 taps per phase: 2/5 137 / 136 / 113 vs
// 111 / 75 / 43, 3/5 121 / 122 / 97 vs 124 / 80 / 44, 4/5 74 / 74 / 58 vs 135 / 83 / 45, 2/3 218 / 220 / 162 vs
// 257 / 212 / 147; 5/3 136 vs 311, 4/3 141 vs 284 at 16).
static int fir_ratio_min_tq(int L, int M, int is_complex)
{
    if (!is_complex) {
        switch (L * 8 + M) {
        case 2 * 8 + 5: return 1;
        case 3 * 8 + 5:
        case 2 * 8 + 3: return 32;
        case 4 * 8 + 5: return 64;
        case 3 * 8 + 2:
        case 3 * 8 + 4:
        case 4 * 8 + 3:
        case 5 * 8 + 2:
        case 5 * 8 + 3:
        case 5 * 8 + 4: return 1 << 20;
        }
        return 0;
    }
    switch (L * 8 + M) {
    case 2 * 8 + 3:
    case 2 * 8 + 5:
    case 3 * 8 + 2:
    case 3 * 8 + 4:
    case 3 * 8 + 5:
    case 4 * 8 + 3:
    case 4 * 8 + 5:
    case 5 * 8 + 3: return 1;
    case 5 * 8 + 4: return 48;
    case 5 * 8 + 2: return 1 << 20; // (built, selectable with B200_RATIONAL_MINTQ)
    }
    return 0; // not built
}

bool fir_interp_supported(int T, int L, int M, int is_complex)
{
    if (T < 1 || getenv("B200_INTERP_RB"))
        return false;
    const int vec = is_complex ? 2 : 1, CH = FIR_ACC / vec;
    const int TQ = ((T + L - 1) / L + CH - 1) / CH * CH;
    if (M > 1) {
        int mq = fir_ratio_min_tq(L, M, is_complex);
        if (const char* e = getenv("B200_RATIONAL_MINTQ")) // (measurement: fold from this many taps per phase)
            mq = mq > 0 ? atoi(e) : 0;
        return mq > 0 && (T + L - 1) / L >= mq && TQ / CH <= 64 && !getenv("B200_RATIONAL_RB");
    }
    if (L < 2 || L > 4)
        return false;
    // measured against the register-blocked resampler kernel (tools/resampler_sweep.py): +22..47 % for
    // L = 2, 3 at any length; at L = 4 the 64 KiB output tile leaves 2 CTAs per SM and short phases lose
    // (128 taps: 230 vs 259 GS/s out), so L = 4 folds only once the phases are FMA-bound
    if (L == 4 && T < (getenv("B200_INTERP_L4_MIN") ? atoi(getenv("B200_INTERP_L4_MIN")) : 192))
        return false;
    return TQ / CH <= 64;
}

int fir_interp_create(const float* taps, int T, int L, int M, int is_complex, b200_fir** out)
{
    *out = nullptr;
    if (!fir_interp_supported(T, L, M, is_complex))
        return set_err(B200_ERR_UNSUPPORTED, "fir resampling fold: %d / %d, %d taps not supported", L, M, T);
    b200_fir* h = new b200_fir();
    h->T = T;
    h->D = 1;
    h->interp = L;
    h->dg = M > 1 ? M : 0;
    h->vec = is_complex ? 2 : 1;
    const int CH = FIR_ACC / h->vec;
    const int NTt = fir_tile_nt(L, M);
    h->TQ = ((T + L - 1) / L + CH - 1) / CH * CH;
    const int need = NTt * M + h->TQ / CH;
    h->n_boxes = (need + 255) / 256;
    h->box_rows = (need + h->n_boxes - 1) / h->n_boxes;
    h->plane_rows = h->box_rows * h->n_boxes;
    if (const int gr = fir_dg_group(h->dg, h->vec)) {
        h->n_boxes = (need + gr - 1) / gr;
        h->box_rows = gr;
        h->plane_rows = h->n_boxes * (gr + 1);
    }
    h->smem = 16 + sizeof(float) * ((size_t)L * h->TQ + (size_t)h->plane_rows * 32 + 256) + 2048 +
              (size_t)L * NTt * 128;
    // tap row r = phase (r M) mod L of the filter, reversed (row r makes the outputs L n + r)
    std::vector<float> pp((size_t)L * h->TQ, 0.f);
    for (int r = 0; r < L; r++) {
        const int ph = (int)(((long long)r * M) % L);
        for (int qr = 0; qr < h->TQ; qr++) {
            const long long k = (long long)(h->TQ - 1 - qr) * L + ph;
            pp[(size_t)r * h->TQ + qr] = k < T ? taps[k] : 0.f;
        }
    }
    cudaError_t e = cudaMalloc(&h->d_taps_pp, pp.size() * sizeof(float));
    if (e == cudaSuccess)
        e = cudaMemcpy(h->d_taps_pp, pp.data(), pp.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = h->vec == 2 ? (L <= 3 ? fir_ll_attr_c23() : fir_ll_attr_c45()) : (L <= 3 ? fir_ll_attr_r23() : fir_ll_attr_r45());
    if (e != cudaSuccess) {
        b200_fir_destroy(h);
        return set_err(B200_ERR_CUDA, "fir resampling fold: %s", cudaGetErrorString(e));
    }
    // the uploads above went through the legacy default stream (cudaMemcpy / cudaMemset); the caller's streams are
    // non-blocking and not ordered against it, so finish them before the handle can be used
    if (cudaDeviceSynchronize() != cudaSuccess) {
        b200_fir_destroy(h);
        return set_err(B200_ERR_CUDA, "fir_interp_create: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = h;
    return B200_OK;
}

int fir_interp_launch(b200_fir* h, const float* d_hist, const void* d_in, void* d_out, long long n_in,
                      cudaStream_t s)
{
    if (n_in <= 0)
        return B200_OK;
    const int L = h->interp, M = h->dg ? h->dg : 1;
    const int NTt = fir_tile_nt(L, M);
    const int MT = NTt * (FIR_ACC / h->vec) * M; // inputs per tile
    const long long tiles = (n_in + MT - 1) / MT;
    if (tiles > 0x7fffffffLL)
        return set_err(B200_ERR_ARG, "resampler: too many items for one call");
    fir_geom gm{};
    gm.Tm1 = (h->T + L - 1) / L - 1; // history is counted in input samples of a phase filter
    gm.D = 1;
    gm.TQ = h->TQ;
    gm.plane_rows = h->plane_rows;
    gm.box_rows = h->box_rows;
    gm.n_boxes = h->n_boxes;
    gm.n_in = n_in;
    gm.n_out = n_in / M * L;
    gm.full_rows = n_in * h->vec / 32;
    gm.full_out_rows = gm.n_out * h->vec / 32;
    CUtensorMap tmap, tmap_out;
    memset(&tmap, 0, sizeof(tmap));
    memset(&tmap_out, 0, sizeof(tmap_out));
    if (h->use_tma && gm.full_rows >= h->plane_rows && (uintptr_t)d_in % 16 == 0 &&
        fir_make_tmap(&tmap, d_in, gm.full_rows, h->box_rows) == B200_OK)
        gm.tma_ok = 1;
    if (h->use_tma && gm.full_out_rows >= NTt && (uintptr_t)d_out % 16 == 0 &&
        fir_make_tmap(&tmap_out, d_out, gm.full_out_rows, NTt) == B200_OK)
        gm.tma_out_ok = 1;
    const float* x = (const float*)d_in;
    float* y = (float*)d_out;
    fir_epilogue ep{ 0, 1.f, 0.f };
    const fir_args fa{ x, d_hist, y, h->d_taps_pp, tmap, tmap_out, gm, ep };
    if (h->vec == 2)
        return L <= 3 ? fir_ll_launch_c23(L, M, (unsigned)tiles, h->smem, s, fa)
                      : fir_ll_launch_c45(L, M, (unsigned)tiles, h->smem, s, fa);
    return L <= 3 ? fir_ll_launch_r23(L, M, (unsigned)tiles, h->smem, s, fa)
                  : fir_ll_launch_r45(L, M, (unsigned)tiles, h->smem, s, fa);
    return B200_OK;
}

} // namespace b200

extern "C" {

int b200_fir_destroy(b200_fir* h)
{
    if (!h)
        return B200_OK;
    cudaFree(h->d_taps_pp);
    cudaFree(h->d_taps);
    cudaFree(h->d_hist[0]);
    cudaFree(h->d_hist[1]);
    ols_destroy(h->ols);
    tc_destroy(h->tc);
    delete h;
    return B200_OK;
}

int b200_fir_create(const b200_fir_params* p, b200_fir** out)
{
    if (!p || !out)
        return set_err(B200_ERR_ARG, "fir_create: null argument");
    *out = nullptr;
    if (!p->taps || p->n_taps < 1 || p->decimation < 1)
        return set_err(B200_ERR_ARG, "fir_create: need n_taps >= 1, decimation >= 1, taps != NULL");
    if (p->algorithm < 0 || p->algorithm > 4)
        return set_err(B200_ERR_ARG, "fir_create: algorithm must be 0 (auto), 1 (direct SIMT), 2 (tensor core), 3 (overlap-save) "
                                     "or 4 (one thread per output)");
    if (p->algorithm == 2 && !tc_supported(p->n_taps, p->decimation, !p->is_complex))
        return set_err(B200_ERR_UNSUPPORTED,
                       "fir_create: the tensor-core form needs decimation 1..8 and <= 2048 taps per branch (complex stream), or "
                       "decimation 1 and <= 449 taps (float stream)");
    b200_fir* h = new b200_fir();
    h->T = p->n_taps;
    h->D = p->decimation;
    h->vec = p->is_complex ? 2 : 1;
    h->ep = fir_epilogue{ p->fuse_multiply_const ? 1 : 0, p->k_re, p->k_im };
    cudaGetDevice(&h->device);

    // full-rate real streams run as float pairs through the packed complex x real loop
    if (h->vec == 1 && h->D == 1 && !getenv("B200_FIR_REAL_SCALAR"))
        h->rp = 1;
    const int CH = FIR_ACC / (h->rp ? 2 : h->vec);
    const int MT = FIR_NT * (FIR_ACC / h->vec);
    // decimations that divide the 16 (32) window positions of a thread run in the full-rate kernel
    if (h->D > 1 && (FIR_ACC / h->vec) % h->D == 0 && !getenv("B200_FIR_PLANES"))
        h->dd = h->D;
    // ... and the other decimations up to 15 (3, 5, 6, 7, 9 ... 15) with D rows per thread
    if (!h->dd && h->D > 1 && h->D <= (getenv("B200_FIR_DG_MAX") ? atoi(getenv("B200_FIR_DG_MAX")) : 15) && !getenv("B200_FIR_PLANES"))
        h->dg = h->D;
    const int Dg = h->rp ? 2 : (h->dd || h->dg) ? 1 : h->D; // phases the plane / tap geometry is built for
    int tq = (h->T + Dg - 1) / Dg;
    h->TQ = (tq + CH - 1) / CH * CH; // whole 16- (32-) tap steps
    (void)MT;
    {
        int need = (h->dg ? fir_dg_nt(h->dg) * h->dg : FIR_NT) + h->TQ / CH; // rows per plane: per thread + one per tap step
        h->n_boxes = (need + 255) / 256;
        h->box_rows = (need + h->n_boxes - 1) / h->n_boxes;
        h->plane_rows = h->box_rows * h->n_boxes;
        if (const int gr = fir_dg_group(h->dg, h->vec)) { // padded layout: one TMA box per group, one spare row behind each
            h->n_boxes = (need + gr - 1) / gr;
            h->box_rows = gr;
            h->plane_rows = h->n_boxes * (gr + 1);
        }
    }
    h->smem = 16 + sizeof(float) * ((size_t)Dg * h->TQ + (size_t)Dg * (h->plane_rows * 32 + 8)) + 1024;
    if (const char* e = getenv("B200_FIR_TMA"))
        h->use_tma = atoi(e);
    h->algorithm = 1;
    if (h->smem > 200 * 1024 || p->algorithm == 4)
        h->algorithm = 4; // naive global-memory fallback
    // block-Toeplitz GEMM on the tensor cores (algorithm 2, fir_tc.cu).  Measured on B200 (tools/tc_check.py,
    // 64 Mi samples, input rate in GS/s, tensor form vs the best SIMT form): full-rate complex filters of
    // 48 / 64 / 96 / 128 / 192 / 256 / 384 taps run 354 / 347 / 323 / 312 / 280 / 245 / 193 against
    // 294 / 229 / 193 / 194 / 190 / 188 / 183 (direct FFMA2 kernel up to 64 taps, overlap-save beyond), i.e.
    // 0.86 .. 0.60 of the HBM roofline where the SIMT forms reach 0.56 .. 0.45; at 512 taps it loses
    // (133 vs 177) and so do the decimating cases (T=1024/D=4: 163 vs 252), which stay on overlap-save.
    // Its results carry the bf16 hi/lo split error, 3.1e-6 .. 3.6e-6 relative RMS against the fp64 oracle
    // (bar: 1e-5); the SIMT forms (~1e-7 / 3e-7) remain selectable with algorithm = 1 / 3 for callers that
    // want bit-reproducible chunking or an exact impulse response.
    {
        bool want2 = p->algorithm == 2;
        if (p->algorithm == 0 && h->vec == 2 && h->D == 1 && h->T >= 33 && h->T <= 384 && tc_supported(h->T, h->D, 0))
            want2 = true;
        // float streams (fff): the same kernel with two 4096-sample runs per tile; crossovers measured with tools/real_tc_ab.py
        if (p->algorithm == 0 && h->vec == 1 && h->D == 1 && h->T >= 33 && h->T <= 448 && tc_supported(h->T, h->D, 1))
            want2 = true;
        if (want2) {
            int rc = tc_create(p->taps, h->T, h->D, h->vec == 1, h->ep.fuse, h->ep.kre, h->ep.kim, &h->tc);
            if (rc != B200_OK) {
                b200_fir_destroy(h);
                return rc;
            }
            h->algorithm = 2;
        }
    }

    // overlap-save fast convolution: complex streams, enough taps per output to pay for two
    // FFTs per block (crossover measured on B200: ~100 taps per output sample)
    {
        const bool can = ols_supported(h->T, h->D, h->vec == 1);
        bool want = (p->algorithm == 3);
        // measured crossovers on B200 (tools/fir_sweep.py, tools/olsd_sweep.py): the full-rate form
        // beats the direct kernel from ~96 taps per output; the polyphase form of a decimating
        // complex filter already from ~40 (even D, TMA-staged; at 32 the two are within 5 %) / ~64 (odd D)
        const int poly = can ? ols_polyphase(h->T, h->D, h->vec == 1) : 0;
        // full-rate filters: the direct kernel pays for taps in pairs of 16-tap steps (64, 96, 128 ...), so
        // 65..96 taps cost 1.5x 64 taps (151 vs 214 GS/s at 16 Mi samples) while overlap-save stays at
        // ~185 (tools/cross_ab.py): switch right after 64 taps, complex and real alike
        const int cross = poly == 1 ? 40 : poly == 2 ? 64 : h->D == 1 ? 65 : 96;
        if (p->algorithm == 0 && can && h->T / h->D >= cross)
            want = true;
        if (p->algorithm == 0 && h->dg && can) {
            // D = 3, 5, 6, 7, 9 ... 15 folded into the full-rate kernel with D rows per thread (tools/decim_ab.py
            // with DS=..., tools/dg_ab.py): complex 400-660 GS/s at 32 taps against 93-280 for overlap-save, real
            // 0.83-1.25 TS/s against ~200; its cost grows with T, overlap-save is flat: measured crossovers (taps)
            static const short tx_c[16] = { 0, 0, 0, 208, 0, 304, 176, 368, 0, 448, 208, 544, 288, 448, 224, 512 };
            static const short tx_r[16] = { 0, 0, 0, 352, 0, 608, 608, 640, 0, 640, 576, 640, 480, 448, 448, 512 };
            const int tx = (h->vec == 2 ? tx_c : tx_r)[h->dg];
            want = h->T > tx;
        } else if (p->algorithm == 0 && !h->dd && h->vec == 2 && h->D > 1 && can) {
            // decimations that do not fold (beyond 15, or B200_FIR_PLANES / B200_FIR_DG_MAX set): the phase-plane kernel
            // stages with per-sample copies and sits at 150-290 GS/s; the polyphase overlap-save is flat at
            // 130-280.  Even D = 6, 10, 12, 14 (TMA-staged polyphase form): from 64 taps; D = 3, 5, 7: beyond 96 taps;
            // larger D: from 192 taps, and whenever the phase planes would not fit shared memory
            if (poly == 1)
                want = h->T >= 64; // (shorter filters stay on the direct kernel: exact impulse response)
            else if (poly == 2)
                want = h->D <= 7 ? h->T > 96 : h->T >= 192;
            else
                want = h->T >= 192 || h->algorithm == 4;
        }
        if (p->algorithm == 0 && h->dd) {
            // decimation folded into the full-rate kernel (dd): short filters are HBM-bound there and
            // its cost grows with T, not T/D; measured crossovers against overlap-save
            // (tools/decim_ab.py, taps): complex 96 / 160 / 192 / 384 for D = 2 / 4 / 8 / 16, real
            // 256 / 512 / 768 / 768 / 768 for D = 2 / 4 / 8 / 16 / 32
            int tx;
            if (h->vec == 2)
                tx = h->dd == 2 ? 96 : h->dd == 4 ? 160 : h->dd == 8 ? 192 : 384;
            else
                tx = h->dd == 2 ? 256 : h->dd == 4 ? 512 : 768;
            want = can && h->T > tx;
        }
        if (h->algorithm == 2)
            want = false; // the tensor-core form was chosen above
        if (want && !can && p->algorithm == 3) {
            b200_fir_destroy(h);
            return set_err(B200_ERR_UNSUPPORTED, "fir_create: overlap-save needs 2..32768 taps");
        }
        if (want && can) {
            int rc = ols_create(p->taps, h->T, h->D, h->vec == 1, h->ep.fuse, h->ep.kre, h->ep.kim, &h->ols);
            if (rc != B200_OK) {
                b200_fir_destroy(h);
                return rc;
            }
            h->algorithm = 3;
        }
    }

#define FIR_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            b200_fir_destroy(h);                                                         \
            return set_err(e__ == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA, \
                           "fir_create: %s -> %s", #call, cudaGetErrorString(e__));      \
        }                                                                                \
    } while (0)

    std::vector<float> pp((size_t)Dg * h->TQ, 0.f);
    for (int ph = 0; ph < Dg; ph++)
        for (int qr = 0; qr < h->TQ; qr++) {
            long long k = (long long)(h->TQ - 1 - qr) * Dg + ph;
            pp[(size_t)ph * h->TQ + qr] = (k < h->T) ? p->taps[k] : 0.f;
        }
    FIR_CUDA(cudaMalloc(&h->d_taps_pp, pp.size() * sizeof(float)));
    FIR_CUDA(cudaMemcpy(h->d_taps_pp, pp.data(), pp.size() * sizeof(float), cudaMemcpyHostToDevice));
    FIR_CUDA(cudaMalloc(&h->d_taps, (size_t)h->T * sizeof(float)));
    FIR_CUDA(cudaMemcpy(h->d_taps, p->taps, (size_t)h->T * sizeof(float), cudaMemcpyHostToDevice));
    size_t hb = sizeof(float) * (size_t)h->vec * (size_t)(h->T > 1 ? h->T - 1 : 1);
    for (int i = 0; i < 2; i++) {
        FIR_CUDA(cudaMalloc(&h->d_hist[i], hb));
        FIR_CUDA(cudaMemset(h->d_hist[i], 0, hb));
    }
    if (h->algorithm == 1 && h->dg) {
        FIR_CUDA(h->vec == 2 ? fir_dg_attr_c() : fir_dg_attr_r());
    }
    if (h->algorithm == 1 && h->dd) {
#define FIR_DD_ATTR(V, DDV) \
    FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<V, false, DDV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024))
        FIR_DD_ATTR(2, 2);
        FIR_DD_ATTR(2, 4);
        FIR_DD_ATTR(2, 8);
        FIR_DD_ATTR(2, 16);
        FIR_DD_ATTR(1, 2);
        FIR_DD_ATTR(1, 4);
        FIR_DD_ATTR(1, 8);
        FIR_DD_ATTR(1, 16);
        FIR_DD_ATTR(1, 32);
#undef FIR_DD_ATTR
    }
    if (h->algorithm == 1 && h->rp)
        FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<2, false, 1, 1, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (h->algorithm == 1) {
        if (h->vec == 2)
        {
            FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<2, true>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<2, false>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
        else
        {
            FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<1, true>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            FIR_CUDA(cudaFuncSetAttribute(fir_direct_kernel<1, false>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
    }
#undef FIR_CUDA
    // the uploads above went through the legacy default stream (cudaMemcpy / cudaMemset); the caller's streams are
    // non-blocking and not ordered against it, so finish them before the handle can be used
    if (cudaDeviceSynchronize() != cudaSuccess) {
        b200_fir_destroy(h);
        return set_err(B200_ERR_CUDA, "fir_create: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = h;
    return B200_OK;
}

int b200_fir_algorithm(const b200_fir* h) { return h ? h->algorithm : 0; }

int b200_fir_geometry(const b200_fir* h, int* decimation, int* item_bytes)
{
    if (!h)
        return set_err(B200_ERR_ARG, "fir_geometry: null handle");
    if (decimation)
        *decimation = h->D;
    if (item_bytes)
        *item_bytes = 4 * h->vec;
    return B200_OK;
}

int b200_fir_run(b200_fir* h, const void* d_in, void* d_out, int64_t n_in_items,
                 int64_t* n_consumed, int64_t* n_produced, b200_stream_t s)
{
    if (!h || n_in_items < 0 || (n_in_items > 0 && !d_in) || (n_in_items >= h->D && !d_out))
        return set_err(B200_ERR_ARG, "fir_run: bad argument");
    long long n_out = n_in_items / h->D;
    long long n_cons = n_out * h->D;
    int rc = fir_launch(h, h->d_hist[h->cur], d_in, d_out, n_in_items, n_out, cs(s));
    if (rc != B200_OK)
        return rc;
    if (h->T > 1 && n_cons > 0) {
        int Tm1 = h->T - 1;
        B200_LAUNCH_PDL(fir_hist_kernel, (Tm1 + 255) / 256, 256, 0, cs(s), (const float*)d_in,
                        (const float*)h->d_hist[h->cur], h->d_hist[h->cur ^ 1], (long long)n_cons, Tm1, h->vec);
        h->cur ^= 1;
    }
    if (n_consumed)
        *n_consumed = n_cons;
    if (n_produced)
        *n_produced = n_out;
    return B200_OK;
}

int b200_fir_run_segment(b200_fir* h, const void* d_halo, const void* d_in, void* d_out,
                         int64_t n_in_items, int64_t* n_produced, b200_stream_t s)
{
    if (!h || n_in_items < 0 || (n_in_items > 0 && !d_in) || (n_in_items >= h->D && !d_out))
        return set_err(B200_ERR_ARG, "fir_run_segment: bad argument");
    long long n_out = n_in_items / h->D;
    int rc = fir_launch(h, (const float*)d_halo, d_in, d_out, n_in_items, n_out, cs(s));
    if (rc == B200_OK && n_produced)
        *n_produced = n_out;
    return rc;
}

int b200_fir_reset(b200_fir* h, b200_stream_t s)
{
    if (!h)
        return set_err(B200_ERR_ARG, "fir_reset: null handle");
    size_t hb = sizeof(float) * (size_t)h->vec * (size_t)(h->T > 1 ? h->T - 1 : 1);
    B200_CUDA(cudaMemsetAsync(h->d_hist[h->cur], 0, hb, cs(s)));
    return B200_OK;
}

int b200_fir_set_history(b200_fir* h, const void* d_hist, b200_stream_t s)
{
    if (!h || !d_hist)
        return set_err(B200_ERR_ARG, "fir_set_history: null argument");
    if (h->T > 1)
        B200_CUDA(cudaMemcpyAsync(h->d_hist[h->cur], d_hist,
                                  sizeof(float) * (size_t)h->vec * (size_t)(h->T - 1),
                                  cudaMemcpyDeviceToDevice, cs(s)));
    return B200_OK;
}

int b200_fir_get_history(b200_fir* h, void* d_hist, b200_stream_t s)
{
    if (!h || !d_hist)
        return set_err(B200_ERR_ARG, "fir_get_history: null argument");
    if (h->T > 1)
        B200_CUDA(cudaMemcpyAsync(d_hist, h->d_hist[h->cur],
                                  sizeof(float) * (size_t)h->vec * (size_t)(h->T - 1),
                                  cudaMemcpyDeviceToDevice, cs(s)));
    return B200_OK;
}

} // extern "C"

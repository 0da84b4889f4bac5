// fir_direct.cuh -- the TMA-staged, register-blocked direct-form FIR kernel (all its modes) shared by the
// translation units that instantiate it: fir.cu (full-rate, divisor decimations, real-pair form, phase
// planes), fir_dg_*.cu (decimation by 3, 5, 6, 7, 9 ... 15) and fir_ll_*.cu (interpolation / rational
// resampling).  One kernel per translation unit would take minutes to compile in a single nvcc run.
#pragma once
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "fir_interp.cuh"
#include "fir_ols.cuh"
#include "fir_tc.cuh"

namespace b200 {

// minimum resident CTAs the compiler must leave room for: 6 caps the kernel at 85 registers (with the
// odd tail step it would otherwise take 96 and drop to 5 CTAs/SM: -7 % on HBM-bound short filters)
#ifndef FIR_MINB
#define FIR_MINB 6
#endif
#ifndef B200_FIR_NT
#define B200_FIR_NT 128
#endif
constexpr int FIR_NT = B200_FIR_NT; // threads per CTA
constexpr int FIR_ACC = 32;  // fp32 accumulators per thread
constexpr int FIR_RING = 64; // register window (floats)

// Shared-memory tile layout = what TMA SWIZZLE_128B produces: rows of 32 floats (128 B), the
// 16-byte chunk c of row r stored at chunk position c ^ (r & 7).  Thread t's window starts at
// row t, so the 8 lanes of a quarter-warp hit 8 different chunk positions: the per-thread
// 128 B-strided LDS.128 reads are bank-conflict free without padding.
__host__ __device__ __forceinline__ int swz(int f)
{
    const int row = f >> 5, c = (f >> 2) & 7;
    return (row << 5) | ((c ^ (row & 7)) << 2) | (f & 3);
}

struct fir_epilogue {
    int fuse;
    float kre, kim;
};

struct fir_geom {
    int Tm1, D, TQ;
    int plane_rows;   // rows (of 32 floats) per phase plane
    int box_rows;     // rows per TMA box
    int n_boxes;      // TMA boxes per tile (D == 1 only)
    int tma_ok;       // input tensor map valid (input 16-byte aligned, enough full rows)
    int tma_out_ok;   // output tensor map valid
    long long full_rows;     // rows of the input that are completely inside [0, n_in)
    long long full_out_rows; // rows of the output completely inside [0, n_out)
    long long n_in, n_out;
    long long n_in_f, n_out_f; // RP mode: bounds in floats (n_in / n_out are in float PAIRS there)
};

// x value at global sample index g (may be negative -> history, or >= n_in -> 0)
template <int VEC>
__device__ __forceinline__ void fir_fetch(const float* __restrict__ x, const float* __restrict__ hist,
                                          int Tm1, long long g, long long n_in, float* v)
{
    const float* src = nullptr;
    if (g >= 0) {
        if (g < n_in)
            src = x + g * VEC;
    } else if (hist && g >= -(long long)Tm1) {
        src = hist + ((long long)Tm1 + g) * VEC;
    }
    if (VEC == 2) {
        float2 t = src ? __ldg(reinterpret_cast<const float2*>(src)) : make_float2(0.f, 0.f);
        v[0] = t.x;
        v[1] = t.y;
    } else {
        v[0] = src ? __ldg(src) : 0.f;
        v[1] = 0.f;
    }
}

// One step of CH taps against the register ring.  OFF = ring offset (floats) of the thread's row;
// tap q' of the step meets ring element (q'+1): the window is read from one sample early so that
// BOTH the input window and the output tile start on 128-byte rows (TMA load and TMA store).
// DD > 1 (decimation folded into the full-rate kernel): only every DD-th output position of the
// window owns an accumulator, the taps stay in natural order.
template <int VEC, int CH, int OFF, int DD = 1>
__device__ __forceinline__ void fir_step(float (&acc)[FIR_ACC], const float (&W)[FIR_RING],
                                         const float* __restrict__ hs)
{
#pragma unroll
    for (int q4 = 0; q4 < CH; q4 += 4) {
        float4 h4 = *reinterpret_cast<const float4*>(hs + q4);
        const float hv[4] = { h4.x, h4.y, h4.z, h4.w };
#pragma unroll
        for (int u = 0; u < 4; u++) {
            if (VEC == 2) {
                // complex sample x real tap = one packed FFMA2 (fma.rn.f32x2, tap broadcast):
                // half the issue slots of two FFMAs, so staging / epilogue instructions of the
                // other resident warps issue underneath the FMA pipe
                const float2 h2 = make_float2(hv[u], hv[u]);
#pragma unroll
                for (int l = 0; l < FIR_ACC; l += 2 * DD) {
                    const int i = (OFF + (q4 + u + 1) * VEC + l) % FIR_RING;
                    float2 a = __ffma2_rn(make_float2(W[i], W[i + 1]), h2, make_float2(acc[l], acc[l + 1]));
                    acc[l] = a.x;
                    acc[l + 1] = a.y;
                }
            } else {
#pragma unroll
                for (int l = 0; l < FIR_ACC; l += DD)
                    acc[l] = fmaf(hv[u], W[(OFF + (q4 + u + 1) * VEC + l) % FIR_RING], acc[l]);
            }
        }
    }
}

// 32 floats of row `row` of a swizzled plane into one half of the register ring
template <int HALF>
__device__ __forceinline__ void fir_load_half(float (&W)[FIR_RING], const float* __restrict__ plane, int row)
{
    const float* rb = plane + (row << 5);
    const int s = (row & 7) << 2;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        float4 t = *reinterpret_cast<const float4*>(rb + ((j << 2) ^ s));
        W[HALF * 32 + 4 * j + 0] = t.x;
        W[HALF * 32 + 4 * j + 1] = t.y;
        W[HALF * 32 + 4 * j + 2] = t.z;
        W[HALF * 32 + 4 * j + 3] = t.w;
    }
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1,
                                            uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(smem_dst)),
                 "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}

// Tile k produces outputs [k*MT, (k+1)*MT).  Plane element 0 is x_p[k*MT - TQ] (one sample before
// the oldest sample the taps reach), so every thread's window and every thread's 128 B of outputs
// start on a 128-byte row: interior tiles are staged by ONE TMA tensor load (D == 1) and written
// back by ONE TMA tensor store.
// smem: [mbarrier 16 B][taps D*TQ floats][pad to 1024 B][D planes of plane_rows*32 floats]
// DECIM = false: D == 1 instantiation (TMA for interior tiles, register-staged loads for the few
// edge tiles).  DECIM = true: decimating filters -- phase de-interleave with cp.async.  (Keeping
// the cp.async path out of the D == 1 kernel is worth ~10 % on short filters: measured A/B.)
// ---- decimation by ANY small D folded into the full-rate kernel (DG) --------------------------------
// A thread owns D consecutive 16-sample rows of the input tile = exactly 16 outputs (one output row).
// Row c of the thread starts at input 16 (D t + c), so its outputs sit at the compile-time positions
// p0(c), p0(c) + D, ... with p0(c) = (-16 c) mod D, and they are the thread's outputs
// off(c) .. off(c) + n(c) - 1 with off(c) = ceil(16 c / D): D passes of the register-window loop, each
// over its own row window, accumulate disjoint slices of the SAME 16 accumulators, and the epilogue
// (row per thread, one TMA store) is the full-rate one.  Same products as the phase-plane kernel, no
// de-interleaving copies; the window loads per input sample equal those of the full-rate filter.
// threads per tile: D rows of 128 B per thread, so these kernels run 64-thread tiles (32 threads from D = 9;
// 24-60 KB, 3-8 CTAs per SM; with 128 threads D = 7 fits one CTA per SM: 64 taps 338 -> 492 GS/s, D = 5 471 -> 558, D = 3 476 -> 494)
#ifndef B200_FIR_DG_SMALL
#define B200_FIR_DG_SMALL 3
#endif
__host__ __device__ constexpr int fir_dg_nt(int dg) { return dg >= 9 ? FIR_NT / 4 : dg >= B200_FIR_DG_SMALL ? FIR_NT / 2 : FIR_NT; }
// Even D: the rows D t + k of the 8 lanes that share a shared-memory wavefront take only 8 / gcd(D, 8)
// different values of (row & 7), i.e. of the 128-byte swizzle: a 2-way (D = 6) bank conflict on every
// window load.  One unused row after every P = 8 / gcd(D, 8) threads' rows (P D rows, one TMA box each)
// makes lanes t and t + P differ by 1 (mod 8): fir_dg_group = rows per group, 0 = no padding.
#ifndef B200_FIR_DG_PAD
#define B200_FIR_DG_PAD 1
#endif
#ifndef B200_FIR_DG_PAD_REAL
#define B200_FIR_DG_PAD_REAL 9 // real streams: pad multiples of 4 from this D on (i.e. D = 12)
#endif
// (Real streams: only D = 12, where the conflict is 4-way -- 32 taps 671 -> 835 GS/s; the 2-way cases are
// FMA-bound in the scalar loop and the padding costs them a resident CTA per SM: D = 6 at 512 taps
// 194 -> 168, D = 10 at 32 taps 1017 -> 870.)
__host__ __device__ constexpr int fir_dg_group(int dg, int vec)
{
    return (!B200_FIR_DG_PAD || (vec != 2 && (dg < B200_FIR_DG_PAD_REAL || dg % 4)) || dg < 2 || dg % 2)
               ? 0
               : (dg % 8 == 0 ? 1 : dg % 4 == 0 ? 2 : 4) * dg;
}
template <int GR>
__device__ __forceinline__ int fir_prow(int r) { return GR ? r + r / GR : r; }

// S (rational resampling, 0 <= S < DG): the thread's output j reads the input DG j + S instead of DG j.
#ifndef B200_FIR_LL4_NT
#define B200_FIR_LL4_NT (FIR_NT / 2) // threads per tile of the interpolate-by-4 fold (64: 41 KB, 5 CTAs per SM;
                                     // 192 taps 190 -> 213 GS/s out against 128-thread tiles, same from 256)
#endif
__host__ __device__ constexpr int fir_tile_nt(int ll, int dg)
{
    return ll > 1 && dg > 1 ? FIR_NT / 2 : ll >= 4 ? B200_FIR_LL4_NT : fir_dg_nt(dg);
}

template <int DG, int C, int R = 16, int S = 0> // R = samples per row: 16 complex, 32 real
struct fir_dg {
    static constexpr int P0 = ((S - R * C) % DG + DG) % DG;
    static constexpr int OFF_OUT = (R * C + P0 - S) / DG;
    static constexpr int N = (R - P0 + DG - 1) / DG;
};

template <int VEC, int OFF, int DG, int C, int S = 0>
__device__ __forceinline__ void fir_step_dg(float (&acc)[FIR_ACC], const float (&W)[FIR_RING],
                                            const float* __restrict__ hs)
{
    constexpr int CH = FIR_ACC / VEC;
    using G = fir_dg<DG, C, CH, S>;
#pragma unroll
    for (int q4 = 0; q4 < CH; q4 += 4) {
        float4 h4 = *reinterpret_cast<const float4*>(hs + q4);
        const float hv[4] = { h4.x, h4.y, h4.z, h4.w };
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const float2 h2 = make_float2(hv[u], hv[u]);
#pragma unroll
            for (int j = 0; j < G::N; j++) {
                const int i = (OFF + (q4 + u + 1 + G::P0 + j * DG) * VEC) % FIR_RING;
                const int l = (G::OFF_OUT + j) * VEC;
                if (VEC == 2) {
                    float2 a = __ffma2_rn(make_float2(W[i], W[i + 1]), h2, make_float2(acc[l], acc[l + 1]));
                    acc[l] = a.x;
                    acc[l + 1] = a.y;
                } else
                    acc[l] = fmaf(hv[u], W[i], acc[l]);
            }
        }
    }
}

template <int HALF>
__device__ __forceinline__ void fir_load_half(float (&W)[FIR_RING], const float* __restrict__ plane, int row);

template <int VEC, int DG, int C = 0, int S = 0>
__device__ __forceinline__ void fir_passes_dg(float (&acc)[FIR_ACC], float (&W)[FIR_RING],
                                              const float* __restrict__ plane, const float* __restrict__ hp,
                                              int nsteps, int tid)
{
    if constexpr (C < DG) {
        constexpr int CH = FIR_ACC / VEC;
        constexpr int GR = fir_dg_group(DG, VEC);
        const int r0 = tid * DG + C;
        fir_load_half<0>(W, plane, fir_prow<GR>(r0));
        int b = 0;
        for (; b + 1 < nsteps; b += 2) {
            fir_load_half<1>(W, plane, fir_prow<GR>(r0 + b + 1));
            fir_step_dg<VEC, 0, DG, C, S>(acc, W, hp + b * CH);
            fir_load_half<0>(W, plane, fir_prow<GR>(r0 + b + 2));
            fir_step_dg<VEC, 32, DG, C, S>(acc, W, hp + (b + 1) * CH);
        }
        if (b < nsteps) {
            fir_load_half<1>(W, plane, fir_prow<GR>(r0 + b + 1));
            fir_step_dg<VEC, 0, DG, C, S>(acc, W, hp + b * CH);
        }
        fir_passes_dg<VEC, DG, C + 1, S>(acc, W, plane, hp, nsteps, tid);
    }
}

// Row-major order of the same work: the D passes of a thread re-read each other's rows (pass c, step b needs
// rows c + b and c + b + 1: D (nsteps + 1) row loads for D + nsteps distinct rows).  Walking the rows once
// and running, for row rho, the step b = rho - c of every pass c that has one, loads each row exactly once
// (D = 5, 64 taps: 25 -> 9 row loads per thread; these kernels are LSU-bound, profiles/r01_firdec64d5).  Every
// accumulator still sees its taps in the same order, so the results are bit-identical.
#ifndef B200_FIR_DG_ROWS
#define B200_FIR_DG_ROWS 1
#endif
template <int VEC, int OFF, int DG, int S, int C = 0>
__device__ __forceinline__ void fir_row_steps(float (&acc)[FIR_ACC], const float (&W)[FIR_RING],
                                              const float* __restrict__ hp, int rho, int nsteps)
{
    if constexpr (C < DG) {
        constexpr int CH = FIR_ACC / VEC;
        const int b = rho - C;
        if (b >= 0 && b < nsteps)
            fir_step_dg<VEC, OFF, DG, C, S>(acc, W, hp + b * CH);
        fir_row_steps<VEC, OFF, DG, S, C + 1>(acc, W, hp, rho, nsteps);
    }
}

template <int VEC, int DG, int S = 0>
__device__ __forceinline__ void fir_rows_dg(float (&acc)[FIR_ACC], float (&W)[FIR_RING],
                                            const float* __restrict__ plane, const float* __restrict__ hp,
                                            int nsteps, int tid)
{
#if B200_FIR_DG_ROWS
    // the row walk tests DG guards per row: with few steps and many passes that costs more than the repeated
    // loads (complex D = 15, 32 taps: 465 -> 393 GS/s; real D = 12, 32 taps: 835 -> 737), so short filters at
    // large D keep the pass-major order
    if (DG > 6 && 2 * nsteps < DG - 4) {
        fir_passes_dg<VEC, DG, 0, S>(acc, W, plane, hp, nsteps, tid);
        return;
    }
    constexpr int GR = fir_dg_group(DG, VEC);
    const int r0 = tid * DG;
    const int nrows = DG - 1 + nsteps;
    fir_load_half<0>(W, plane, fir_prow<GR>(r0));
    int rho = 0;
    for (; rho + 1 < nrows; rho += 2) {
        fir_load_half<1>(W, plane, fir_prow<GR>(r0 + rho + 1));
        fir_row_steps<VEC, 0, DG, S>(acc, W, hp, rho, nsteps);
        fir_load_half<0>(W, plane, fir_prow<GR>(r0 + rho + 2));
        fir_row_steps<VEC, 32, DG, S>(acc, W, hp, rho + 1, nsteps);
    }
    if (rho < nrows) {
        fir_load_half<1>(W, plane, fir_prow<GR>(r0 + rho + 1));
        fir_row_steps<VEC, 0, DG, S>(acc, W, hp, rho, nsteps);
    }
#else
    fir_passes_dg<VEC, DG, 0, S>(acc, W, plane, hp, nsteps, tid);
#endif
}

// Rational resampling by LL / DG (LL and DG coprime) = both folds at once.  Output m = LL n + r is
//   y[LL n + r] = sum_q h[q LL + (r DG) mod LL] x[DG n + floor(r DG / LL) - q],
// a decimate-by-DG filter with the taps of phase (r DG) mod LL whose input is shifted by S_r = floor(r DG / LL):
// LL x DG passes over the thread's DG rows, each set of DG passes filling the 16 accumulators of residue r, which
// are scattered into the thread's LL output rows like the interpolator's.
template <int VEC, int LL, int DG, int RR = 0>
__device__ __forceinline__ void fir_passes_ll_dg(float (&acc)[FIR_ACC], float (&W)[FIR_RING],
                                                 const float* __restrict__ plane, const float* __restrict__ hs,
                                                 int TQ, int nsteps, int tid, float* __restrict__ otile)
{
    if constexpr (RR < LL) {
        constexpr int R = FIR_ACC / VEC;
#pragma unroll
        for (int l = 0; l < FIR_ACC; l++)
            acc[l] = 0.f;
        fir_rows_dg<VEC, DG, (RR * DG) / LL>(acc, W, plane, hs + RR * TQ, nsteps, tid);
#pragma unroll
        for (int pz = 0; pz < R; pz++) {
            const int f = ((tid * R + pz) * LL + RR) * VEC;
            if (VEC == 2)
                *reinterpret_cast<float2*>(otile + swz(f)) = make_float2(acc[2 * pz], acc[2 * pz + 1]);
            else
                otile[swz(f)] = acc[pz];
        }
        fir_passes_ll_dg<VEC, LL, DG, RR + 1>(acc, W, plane, hs, TQ, nsteps, tid, otile);
    }
}

// DD > 1 (with DECIM = false): decimation by a divisor of the 16 (32) window positions of a thread.
// The tile is the SAME 2048-sample (4096 for fff) input tile as for D = 1, staged by the same single
// TMA tensor load with the taps in natural order; a thread simply keeps accumulators only for the
// positions 0, DD, 2 DD ... of its row, i.e. 16/DD outputs, and the output tile shrinks to 128/DD rows.
// No phase planes, no per-sample de-interleaving copies: a short decimating filter becomes HBM-bound
// like a short full-rate one (64 taps, decimation 4: 197 -> 400+ GS/s input rate).
// LL > 1 (with DECIM = false, DD = 1): interpolation by LL folded into the same kernel.  Output
// phase r of an interpolator, y[n LL + r] = sum_q h[q LL + r] x[n - q], is a full-rate filter over the
// SAME input tile with the taps of phase r: LL passes of the register-blocked loop over one
// TMA-staged tile, each scattering its 16 results per thread into the thread's own LL rows of a
// separate output tile (16 LL consecutive outputs), which then leaves by LL TMA tensor stores.
// RP ("real pairs", with VEC = 2, DECIM = false): a REAL stream f[] run through the packed
// complex x real loop.  With the float pairs P0[j] = (f[2j], f[2j+1]) (the stream itself) and
// P1[j] = (f[2j-1], f[2j]) (the stream one float later), (y[2m], y[2m+1]) = h_e * P0 + h_o * P1 with the
// even / odd taps: two passes of the FFMA2 loop, i.e. half the issue slots of the scalar fff loop.
// P0 is staged by the same TMA tensor load as a complex stream; P1 is derived from it in shared memory
// (each thread shifts its own row by one float).
template <int VEC, bool DECIM, int DD = 1, int LL = 1, bool RP = false, int DG = 1>
__global__ void __launch_bounds__(fir_tile_nt(LL, DG), (LL > 1 && DG > 1) ? 4 : DG > 1 ? 8 : FIR_MINB) // (DG: 1-2 warp CTAs)
    fir_direct_kernel(const float* __restrict__ x, const float* __restrict__ hist,
                      float* __restrict__ y, const float* __restrict__ taps_pp,
                      const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_out,
                      fir_geom gm, fir_epilogue ep)
{
    constexpr int NT = fir_tile_nt(LL, DG); // threads (= output rows) per tile
    constexpr int R = FIR_ACC / VEC;  // window positions per thread (= outputs per thread for DD == 1)
    constexpr int CH = FIR_ACC / VEC; // taps per step
    constexpr int MT = NT * R * DG; // input-rate positions per tile
    constexpr int MTO = MT / DD / DG;   // outputs per tile
    static_assert(DG == 1 || (!DECIM && DD == 1 && !RP), "DG is a mode of its own (or, with LL, the rational resampler)");
    static_assert(!DECIM || DD == 1, "DD applies to the TMA-staged full-rate kernel only");
    static_assert(R % DD == 0, "decimation must divide the positions per thread");
    static_assert(LL == 1 || (!DECIM && DD == 1), "LL applies to the TMA-staged full-rate kernel only");
    static_assert(!RP || (VEC == 2 && !DECIM && DD == 1 && LL == 1), "RP is the full-rate real-stream mode");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    float* hs = reinterpret_cast<float*>(smem_raw + 16);
    const int D = DECIM ? gm.D : 1, TQ = gm.TQ;
    const int NTAPROWS = RP ? 2 : LL > 1 ? LL : D; // tap rows: one per decimation / interpolation phase
    float* planes;
    {
        uint32_t a = smem_u32(hs + NTAPROWS * TQ);
        uint32_t aligned = (a + 1023u) & ~1023u;
        planes = hs + NTAPROWS * TQ + (aligned - a) / 4;
    }
    // phase planes are skewed by 32 B each so that the de-interleaving stores of one warp (same
    // element, different phase) land in different banks
    const int plane_f = (gm.plane_rows << 5) + (DECIM ? 8 : 0);
    const int tid = threadIdx.x;
    const long long tile = blockIdx.x;
    const long long B0 = tile * MT - TQ; // x_p index of plane element 0
    const long long O0 = tile * MTO;     // first output of this tile
    constexpr int GR = fir_dg_group(DG, VEC);              // DG, even D: one pad row per GR rows
    const int PLs = ((gm.box_rows * gm.n_boxes) << 5) / VEC; // samples per plane

    // interior tile of a D == 1 filter: one TMA tensor copy stages the whole window
    const long long row0 = B0 * VEC / 32;
    const bool use_tma = !DECIM && gm.tma_ok && B0 >= 0 &&
                         row0 + (long long)gm.box_rows * gm.n_boxes <= gm.full_rows;
    if (use_tma && tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        mbar_arrive_expect_tx(bar, (uint32_t)(gm.box_rows * gm.n_boxes) * 128u);
        for (int bx = 0; bx < gm.n_boxes; bx++)
            tma_load_2d(planes + (size_t)bx * (gm.box_rows + (GR ? 1 : 0)) * 32, &tmap, 0, (int)(row0 + (long long)bx * gm.box_rows),
                        bar);
    }
    for (int i = tid; i < NTAPROWS * TQ; i += NT)
        hs[i] = __ldg(taps_pp + i);
    if (DECIM) {
        // decimating filters: every sample inside the input goes global -> shared with cp.async
        // (LDGSTS: asynchronous, no register staging, all of a thread's copies in flight at once)
        // and is de-interleaved by phase on the way in; samples before the stream start come from
        // the history buffer
        const long long g_lo = B0 * D - (D - 1);
        const int total = PLs * D;
        for (int i = tid; i < total; i += NT) {
            const int e = i / D;
            const int p = D - 1 - (i - e * D);
            float* dst = planes + p * plane_f + swz(e * VEC);
            const long long g = g_lo + i;
            if (g >= 0 && g < gm.n_in) {
                if (VEC == 2)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)),
                                 "l"(x + g * 2)
                                 : "memory");
                else
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(x + g)
                                 : "memory");
            } else {
                float v[2];
                fir_fetch<VEC>(x, hist, gm.Tm1, g, gm.n_in, v);
                if (VEC == 2)
                    *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
                else
                    dst[0] = v[0];
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (!use_tma) {
        // D == 1 edge tiles / unaligned input: coalesced loads, 8 independent loads in flight
        const long long g_lo = B0;
        const int total = PLs;
        for (int i0 = tid; i0 < total; i0 += NT * 8) {
            float v[8][2];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = i0 + u * NT;
                if (i < total) {
                    if (RP) { // pair g = floats 2g, 2g+1 of the real stream, each with its own bounds
                        float t0[2], t1_[2];
                        fir_fetch<1>(x, hist, gm.Tm1, 2 * (g_lo + i), gm.n_in_f, t0);
                        fir_fetch<1>(x, hist, gm.Tm1, 2 * (g_lo + i) + 1, gm.n_in_f, t1_);
                        v[u][0] = t0[0];
                        v[u][1] = t1_[0];
                    } else
                        fir_fetch<VEC>(x, hist, gm.Tm1, g_lo + i, gm.n_in, v[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = i0 + u * NT;
                if (i < total) {
                    const int fl = i * VEC;
                    float* dst = planes + swz(GR ? (fir_prow<GR>(fl >> 5) << 5) | (fl & 31) : fl);
                    if (VEC == 2)
                        *reinterpret_cast<float2*>(dst) = make_float2(v[u][0], v[u][1]);
                    else
                        dst[0] = v[u][0];
                }
            }
        }
    }
    __syncthreads();
    if (use_tma)
        mbar_wait(bar, 0);
    if (RP) {
        // plane 1 = plane 0 one float later: row r = [last float of row r-1, first 31 floats of row r]
        float first[2];
        fir_fetch<1>(x, hist, gm.Tm1, 2 * B0 - 1, gm.n_in_f, first); // the float in front of the tile
        float* P1 = planes + plane_f;
        for (int r = tid; r < gm.plane_rows; r += NT) {
            const float* rb = planes + (r << 5);
            const int sw = (r & 7) << 2;
            float a[32];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 t = *reinterpret_cast<const float4*>(rb + ((j << 2) ^ sw));
                a[4 * j] = t.x, a[4 * j + 1] = t.y, a[4 * j + 2] = t.z, a[4 * j + 3] = t.w;
            }
            const float prev = r > 0 ? planes[swz(32 * r - 1)] : first[0];
            float* wb = P1 + (r << 5);
            *reinterpret_cast<float4*>(wb + (0 ^ sw)) = make_float4(prev, a[0], a[1], a[2]);
#pragma unroll
            for (int j = 1; j < 8; j++)
                *reinterpret_cast<float4*>(wb + ((j << 2) ^ sw)) =
                    make_float4(a[4 * j - 1], a[4 * j], a[4 * j + 1], a[4 * j + 2]);
        }
        __syncthreads();
    }

    // ---- register-blocked multiply-accumulate -----------------------------------------
    float acc[FIR_ACC];
#pragma unroll
    for (int l = 0; l < FIR_ACC; l++)
        acc[l] = 0.f;
    float W[FIR_RING];
    const int nsteps = TQ / CH; // any count >= 1: an odd tail step runs alone
    if (LL > 1) {
        // output tile: LL * NT rows behind the input plane (1024-byte aligned for the TMA stores)
        float* otile = planes + (((gm.plane_rows << 5) + 255) & ~255);
        if constexpr (DG > 1)
            fir_passes_ll_dg<VEC, LL, DG>(acc, W, planes, hs, TQ, nsteps, tid, otile);
        else
#pragma unroll 1
        for (int r = 0; r < LL; r++) {
#pragma unroll
            for (int l = 0; l < FIR_ACC; l++)
                acc[l] = 0.f;
            const float* hp = hs + r * TQ;
            fir_load_half<0>(W, planes, tid);
            int b = 0;
            for (; b + 1 < nsteps; b += 2) {
                fir_load_half<1>(W, planes, tid + b + 1);
                fir_step<VEC, CH, 0, 1>(acc, W, hp + b * CH);
                fir_load_half<0>(W, planes, tid + b + 2);
                fir_step<VEC, CH, 32, 1>(acc, W, hp + (b + 1) * CH);
            }
            if (b < nsteps) {
                fir_load_half<1>(W, planes, tid + b + 1);
                fir_step<VEC, CH, 0, 1>(acc, W, hp + b * CH);
            }
            // position p of the thread is output (tid R + p) LL + r of the tile
#pragma unroll
            for (int pz = 0; pz < R; pz++) {
                const int f = ((tid * R + pz) * LL + r) * VEC;
                if (VEC == 2)
                    *reinterpret_cast<float2*>(otile + swz(f)) = make_float2(acc[2 * pz], acc[2 * pz + 1]);
                else
                    otile[swz(f)] = acc[pz];
            }
        }
        const long long orow0 = tile * (NT * LL);
        if (gm.tma_out_ok && orow0 + NT * LL <= gm.full_out_rows) {
            fence_proxy_async();
            __syncthreads();
            if (tid == 0) {
#pragma unroll 1
                for (int r = 0; r < LL; r++)
                    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                                     &tmap_out),
                                 "r"(0), "r"((int)(orow0 + (long long)r * NT)),
                                 "r"(smem_u32(otile + (size_t)r * NT * 32))
                                 : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
            return;
        }
        __syncthreads();
        const long long OL = tile * (long long)(NT * R * LL);
#pragma unroll 4
        for (int i = tid; i < NT * R * LL; i += NT) {
            const long long m = OL + i;
            if (m >= gm.n_out)
                break;
            const float* src = otile + swz(i * VEC);
            if (VEC == 2)
                __stcs(reinterpret_cast<float2*>(y) + m, *reinterpret_cast<const float2*>(src));
            else
                __stcs(y + m, src[0]);
        }
        return;
    }
    if constexpr (DG > 1) {
        fir_rows_dg<VEC, DG>(acc, W, planes, hs, nsteps, tid);
    } else
    for (int p = 0; p < (RP ? 2 : D); p++) {
        const float* plane = planes + p * plane_f;
        const float* hp = hs + p * TQ;
        fir_load_half<0>(W, plane, tid);
        int b = 0;
        for (; b + 1 < nsteps; b += 2) { // pairs of steps: the loop body the scheduler pipelines
            fir_load_half<1>(W, plane, tid + b + 1);
            fir_step<VEC, CH, 0, DD>(acc, W, hp + b * CH);
            fir_load_half<0>(W, plane, tid + b + 2);
            fir_step<VEC, CH, 32, DD>(acc, W, hp + (b + 1) * CH);
        }
        if (b < nsteps) { // odd tail step (ring half 0 holds row tid + b)
            fir_load_half<1>(W, plane, tid + b + 1);
            fir_step<VEC, CH, 0, DD>(acc, W, hp + b * CH);
        }
    }
    __syncthreads();

    // ---- outputs: registers -> shared (swizzled row per thread) -> global ----------------------
    if (ep.fuse && RP) {
#pragma unroll
        for (int l = 0; l < FIR_ACC; l++)
            acc[l] = __fmul_rn(acc[l], ep.kre);
    } else if (ep.fuse) {
        if (VEC == 2) {
#pragma unroll
            for (int l = 0; l < FIR_ACC; l += 2 * DD) {
                float2 v = cmul_nofma(make_float2(acc[l], acc[l + 1]), ep.kre, ep.kim);
                acc[l] = v.x;
                acc[l + 1] = v.y;
            }
        } else {
#pragma unroll
            for (int l = 0; l < FIR_ACC; l += DD)
                acc[l] = __fmul_rn(acc[l], ep.kre);
        }
    }
    if (DD == 1) {
        float* rb = planes + (tid << 5);
        const int s = (tid & 7) << 2;
#pragma unroll
        for (int j = 0; j < 8; j++)
            *reinterpret_cast<float4*>(rb + ((j << 2) ^ s)) =
                make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
    } else {
        // the thread's FIR_ACC/DD output floats, compacted, at their place in the (swizzled) output tile
        constexpr int NF = FIR_ACC / DD; // floats per thread
        float o[NF];
#pragma unroll
        for (int j = 0; j < NF; j++)
            o[j] = acc[(j / VEC) * DD * VEC + (j % VEC)];
        const int f0 = tid * NF;
        if (NF >= 4) {
#pragma unroll
            for (int j = 0; j < NF; j += 4)
                *reinterpret_cast<float4*>(planes + swz(f0 + j)) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < NF; j++)
                planes[swz(f0 + j)] = o[j];
        }
    }
    const long long orow0 = tile * (NT / DD); // output rows per tile
    if (NT / DD >= 8 && gm.tma_out_ok && orow0 + NT / DD <= gm.full_out_rows) {
        // whole tile inside the output: one TMA tensor store from the swizzled rows
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                             &tmap_out),
                         "r"(0), "r"((int)orow0), "r"(smem_u32(planes))
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        return;
    }
    __syncthreads();
#pragma unroll 4
    for (int i = tid; i < MTO; i += NT) {
        const long long m = O0 + i;
        if (m >= gm.n_out)
            break;
        const float* src = planes + swz(i * VEC);
        if (RP) { // the last pair of an odd-length real stream is half a pair
            __stcs(y + 2 * m, src[0]);
            if (2 * m + 1 < gm.n_out_f)
                __stcs(y + 2 * m + 1, src[1]);
        } else if (VEC == 2)
            __stcs(reinterpret_cast<float2*>(y) + m, *reinterpret_cast<const float2*>(src));
        else
            __stcs(y + m, src[0]);
    }
}

// ---- instantiations that live in their own translation units ----------------------------------------------
struct fir_args {
    const float* x;
    const float* hist;
    float* y;
    const float* taps;
    CUtensorMap tmap, tmap_out;
    fir_geom gm;
    fir_epilogue ep;
};
// decimation DG folded (fir_dg_c.cu: complex, fir_dg_r.cu: real)
int fir_dg_launch_c(int dg, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
int fir_dg_launch_r(int dg, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
cudaError_t fir_dg_attr_c();
cudaError_t fir_dg_attr_r();
// interpolation L (M == 1) / rational L / M (fir_ll_{c,r}{23,45}.cu: complex / real, L in {2,3} / {4,5})
int fir_ll_launch_c23(int L, int M, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
int fir_ll_launch_c45(int L, int M, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
int fir_ll_launch_r23(int L, int M, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
int fir_ll_launch_r45(int L, int M, unsigned tiles, size_t smem, cudaStream_t s, const fir_args& a);
cudaError_t fir_ll_attr_c23();
cudaError_t fir_ll_attr_c45();
cudaError_t fir_ll_attr_r23();
cudaError_t fir_ll_attr_r45();

} // namespace b200

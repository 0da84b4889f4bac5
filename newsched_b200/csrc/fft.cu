// fft.cu -- complex64 FFT of vector length N (power of two), forward / reverse, optional real
// window, optional shift, optional fused complex_to_mag epilogue and fused upstream
// multiply_const.  Hand-written shared-memory Stockham kernels; cuFFT is not used.
//
// Semantics (SURVEY.md 8c, GNU Radio fft_vcc): t = x*w; X[k] = sum_n t[n] e^{-/+ j 2 pi k n/N};
// no 1/N scaling; forward+shift = fftshift of the output; reverse+shift = ifftshift of the
// input.  Both shifts are folded into tables at create time:
//     forward+shift : w_eff[n] = w[n] * (-1)^n            (X[k+N/2] = FFT{x (-1)^n}[k])
//     reverse+shift : w_eff[m] = w[(m+N/2) mod N], output * (-1)^k
// and a fused upstream multiply_const k = |k| e^{j phi} becomes w_eff *= |k| plus a constant
// output phasor -- so none of them costs a pass over memory.
//
// N = 4096 (the BASELINE config): one CTA of 256 threads per vector, three radix-16 passes
// with 16 points per thread in registers (4096 = 16*16*16):
//   pass 1  thread L=(n1,n0) loads x[n2*256+L] straight from HBM (coalesced 8 B/thread, 16
//           loads in flight), window in registers, DFT16 over n2, twiddle W4096^{L k0} from
//           registers (loaded once per CTA, reused for every vector), store A[k0][n1][n0];
//   pass 2  thread (k0,n0) DFT16 over n1 IN PLACE, twiddle W256^{n0 k1} from a 2 KB shared
//           table;
//   pass 3  thread (k1,k0) DFT16 over n0, writes X[k0+16k1+256k2] (coalesced) or |X|.
// Exactly one HBM read and one HBM write per sample (16 B, or 12 B with the fused |.|).
// fft4096_kernel exchanges through a buffer with a row stride of 257 complex so all three access
// patterns are bank-conflict free; fft4096_tma_kernel transforms in place in its input tile and
// swizzles the pass-2 stores instead (see there).
// Other N (8..8192): generic radix-2 shared-memory Stockham kernel.
#include <cmath>
#include <cstdlib>
#include <vector>

#include "fft_core.cuh"

// pass-2 twiddles of fft4096_tma_kernel: 0 = shared table read at use, 1 = held in registers for the
// lifetime of the CTA (measured +5.5 %: 451 -> 476 GS/s fused |.|), 2 = re-fetched before the barrier (-3 %)
#ifndef B200_FFT_TW2
#define B200_FFT_TW2 1
#endif

namespace b200 {

template <bool FWD, int OUT>
__global__ void __launch_bounds__(256, 2)
    fft4096_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                   const float* __restrict__ weff, const float2* __restrict__ tw1,
                   const float2* __restrict__ tw2)
{
    __shared__ float2 sA[16 * F4K_STRIDE];
    __shared__ float2 sT2[256];
    const int tid = threadIdx.x;

    // per-thread constants, reused for every vector this CTA transforms
    float wreg[16];
    float2 t1[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        wreg[i] = __ldg(weff + i * 256 + tid);
        t1[i] = __ldg(tw1 + i * 256 + tid);
    }
    sT2[tid] = __ldg(tw2 + tid);
    __syncthreads();

    for (long long vec = blockIdx.x; vec < n_vec; vec += gridDim.x) {
        const float2* x = in + vec * 4096;
        float2 v[16];
        // pull the NEXT vector into L2 while this one is transformed (one bulk prefetch, no smem)
        if (tid == 0 && vec + gridDim.x < n_vec && ((uintptr_t)in % 16 == 0))
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(in + (vec + gridDim.x) * 4096),
                         "r"(4096 * 8)
                         : "memory");
        // ---- pass 1: over n2, thread = L = n1*16+n0
#pragma unroll
        for (int i = 0; i < 16; i++)
            v[i] = __ldcs(x + i * 256 + tid);
#pragma unroll
        for (int i = 0; i < 16; i++)
            v[i] = __fmul2_rn(v[i], make_float2(wreg[i], wreg[i]));
        dft16<FWD>(v);
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++)
            sA[k0 * F4K_STRIDE + tid] = cmul(v[pos16(k0)], t1[k0]);
        __syncthreads();
        // ---- pass 2: over n1, thread = (k0, n0), in place
        {
            const int k0 = tid >> 4, n0 = tid & 15;
            float2* row = sA + k0 * F4K_STRIDE + n0;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i * 16];
            dft16<FWD>(v);
            row[0] = v[pos16(0)];
#pragma unroll
            for (int k1 = 1; k1 < 16; k1++)
                row[k1 * 16] = cmul(v[pos16(k1)], sT2[k1 * 16 + n0]);
        }
        __syncthreads();
        // ---- pass 3: over n0, thread = (k1, k0)
        {
            const int k0 = tid & 15, k1 = tid >> 4;
            const float2* row = sA + k0 * F4K_STRIDE + k1 * 16;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i];
            dft16<FWD>(v);
            if (OUT == B200_FFT_OUT_COMPLEX) {
                float2* y = reinterpret_cast<float2*>(out) + vec * 4096;
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++)
                    __stcs(y + k2 * 256 + tid, v[pos16(k2)]);
            } else {
                float* y = reinterpret_cast<float*>(out) + vec * 4096;
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++) {
                    float2 z = v[pos16(k2)];
                    float p = fmaf(z.x, z.x, z.y * z.y);
                    __stcs(y + k2 * 256 + tid, OUT == B200_FFT_OUT_MAG ? sqrt_approx(p) : p);
                }
            }
        }
        __syncthreads(); // pass-3 reads done before the next vector's pass-1 writes
    }
}

// Same three passes, but the vectors arrive by the TMA engine (1-D bulk copy, 32 KiB, completion on
// an mbarrier) into NT input tiles, and each vector is transformed IN PLACE in its tile: global-load
// latency is off the critical path and costs no registers or issue slots, and there is no separate
// exchange buffer.  Vector i of a CTA (i = 0, 1, ...) uses tile i % NT:
//   pass 1  thread tid reads tile[n2*256 + tid] and writes its 16 results back to tile[k0*256 + tid]:
//           the same slots, which no other thread touches, so no barrier between the loads and stores;
//   -- barrier 1 --
//   pass 2  row k0 is read and rewritten by the 16 lanes tid >> 4 == k0 alone (half a warp):
//           __syncwarp() between its loads and its stores; the stores are swizzled (f4k_swz);
//   -- barrier 2 --
//   pass 3  thread (k1, k0) reads its 16 contiguous values as 8 LDS.128, conflict-free thanks to the
//           swizzle.
// Vector i + 1 lives in another tile, so its pass 1 never touches what pass 3 of vector i reads: no
// third barrier.  Tile t of vector i is refilled with vector i + NT once every thread has passed
// barrier 1 of vector i + 1, i.e. once all pass-3 reads of vector i are over; thread 0 is the one
// that issues that copy, right after the barrier.
// smem: NT tiles of 32 KiB | sT2 2 KiB | NT mbarriers.
// Tiles per CTA, i.e. copies in flight = NT - 1 vectors ahead.  The fused |.| forms write half as many
// bytes as they read and are limited on chip: copies two vectors ahead remove the exposed mbarrier
// wait (measured +1.8 %, DESIGN.md 4.3).  The complex-output form is HBM-bound and LOSES 11 % with that
// deeper read prefetch (more reads in flight against the write stream), so its copies stay one vector
// ahead.
constexpr int f4k_ntile(int out) { return out == B200_FFT_OUT_COMPLEX ? 2 : 3; }
constexpr size_t f4k_tma_smem(int out) { return (size_t)f4k_ntile(out) * (4096 * 8 + 8) + 256 * 8; }

// Position of element n0 (0..15) of a 16-element segment of row k0 after the pass-2 stores: the
// 16-byte chunk index n0 >> 1 is XORed with k0 & 7.  Pass 3 reads a segment as 8 LDS.128 (8 lanes
// per phase, k0 = 0..7 or 8..15, same k1): unswizzled, all 8 would hit the same chunk of a 2 KiB-
// aligned row, an 8-way bank conflict; swizzled, they hit 8 different chunks.
__device__ __forceinline__ int f4k_swz(int n0, int k0) { return (((n0 >> 1) ^ (k0 & 7)) << 1) | (n0 & 1); }

template <bool FWD, int OUT>
__global__ void __launch_bounds__(256, 2)
    fft4096_tma_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                       const float* __restrict__ weff, const float2* __restrict__ tw1,
                       const float2* __restrict__ tw2)
{
    constexpr int NT = f4k_ntile(OUT);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* sTile0 = reinterpret_cast<float2*>(smem_raw);
    float2* sT2 = sTile0 + 4096 * NT;
    uint64_t* bar0 = reinterpret_cast<uint64_t*>(sT2 + 256);
    const int tid = threadIdx.x;

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < NT; i++)
            mbar_init(bar0 + i, 1);
        fence_mbar_init();
    }
    float wreg[16];
    float2 t1[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        wreg[i] = __ldg(weff + i * 256 + tid);
        t1[i] = __ldg(tw1 + i * 256 + tid);
    }
    sT2[tid] = __ldg(tw2 + tid);
    __syncthreads();
#if B200_FFT_TW2 == 1
    // pass-2 twiddles W256^{n0 k1} depend on the thread (n0 = tid & 15) only: keep them in registers
    float2 t2r[16];
#pragma unroll
    for (int k1 = 1; k1 < 16; k1++)
        t2r[k1] = sT2[k1 * 16 + (tid & 15)];
#endif
    // programmatic dependent launch (B200_LAUNCH_PDL): the prologue above ran while the previous kernel in the
    // stream drained; nothing below may start before that kernel has completed and flushed
    pdl_wait();
    pdl_launch_dependents();
    long long vec = blockIdx.x;
    if (tid == 0) {
        // the first NT - 1 vectors; the loop then issues one copy per vector, NT - 1 vectors ahead
#pragma unroll
        for (int i = 0; i < NT - 1; i++)
            if (vec + (long long)i * gridDim.x < n_vec) {
                mbar_arrive_expect_tx(bar0 + i, 4096 * 8);
                bulk_copy_g2s(sTile0 + 4096 * i, in + (vec + (long long)i * gridDim.x) * 4096, 4096 * 8, bar0 + i);
            }
    }
    int t = 0;        // tile of this CTA's vector i: i % NT
    uint32_t par = 0; // parity of that tile's mbarrier phase: (i / NT) & 1
    for (; vec < n_vec; vec += gridDim.x) {
        float2 v[16];
        float2* tile = sTile0 + t * 4096;
        mbar_wait(bar0 + t, par);
        // ---- pass 1: over n2, thread = L = n1*16+n0, results back into the slots it read
#pragma unroll
        for (int i = 0; i < 16; i++)
            v[i] = tile[i * 256 + tid];
#pragma unroll
        for (int i = 0; i < 16; i++)
            v[i] = __fmul2_rn(v[i], make_float2(wreg[i], wreg[i]));
        dft16<FWD>(v);
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++)
            tile[k0 * 256 + tid] = cmul(v[pos16(k0)], t1[k0]);
#if B200_FFT_TW2 == 2
        // v[] is dead until pass 2 reloads it: fetch this thread's pass-2 twiddles now, so that the
        // barrier below covers their shared-memory latency
        float2 t2r[16];
#pragma unroll
        for (int k1 = 1; k1 < 16; k1++)
            t2r[k1] = sT2[k1 * 16 + (tid & 15)];
#endif
        __syncthreads(); // rows complete for pass 2; every thread is past pass 3 of the previous vector
        const int tn = t == 0 ? NT - 1 : t - 1; // the previous vector's tile, now free
        if (tid == 0 && vec + (long long)(NT - 1) * gridDim.x < n_vec) {
            fence_proxy_async(); // the generic-proxy accesses of that tile before the async-proxy copy into it
            mbar_arrive_expect_tx(bar0 + tn, 4096 * 8);
            bulk_copy_g2s(sTile0 + tn * 4096, in + (vec + (long long)(NT - 1) * gridDim.x) * 4096, 4096 * 8,
                          bar0 + tn);
        }
        // ---- pass 2: over n1, thread = (k0, n0), in place within row k0
        {
            const int k0 = tid >> 4, n0 = tid & 15;
            float2* row = tile + k0 * 256;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i * 16 + n0];
            __syncwarp(); // the other 15 lanes of this row have read it before it is overwritten
            dft16<FWD>(v);
            float2* dst = row + f4k_swz(n0, k0);
            dst[0] = v[pos16(0)];
#pragma unroll
            for (int k1 = 1; k1 < 16; k1++)
#if B200_FFT_TW2
                dst[k1 * 16] = cmul(v[pos16(k1)], t2r[k1]);
#else
                dst[k1 * 16] = cmul(v[pos16(k1)], sT2[k1 * 16 + n0]);
#endif
        }
        __syncthreads();
        // ---- pass 3: over n0, thread = (k1, k0)
        {
            const int k0 = tid & 15, k1 = tid >> 4, s = k0 & 7;
            const float4* seg = reinterpret_cast<const float4*>(tile + k0 * 256 + k1 * 16);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 q = seg[j ^ s];
                v[2 * j] = make_float2(q.x, q.y);
                v[2 * j + 1] = make_float2(q.z, q.w);
            }
            dft16<FWD>(v);
            if (OUT == B200_FFT_OUT_COMPLEX) {
                float2* y = reinterpret_cast<float2*>(out) + vec * 4096;
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++)
                    __stcs(y + k2 * 256 + tid, v[pos16(k2)]);
            } else {
                float* y = reinterpret_cast<float*>(out) + vec * 4096;
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++) {
                    float2 z = v[pos16(k2)];
                    float p = fmaf(z.x, z.x, z.y * z.y);
                    __stcs(y + k2 * 256 + tid, OUT == B200_FFT_OUT_MAG ? sqrt_approx(p) : p);
                }
            }
        }
        if (++t == NT) {
            t = 0;
            par ^= 1;
        }
    }
}

// ---- N = 8192: one radix-2 decimation-in-frequency stage in front of two 4096-point transforms ---
//   a[n] = x'[n] + x'[n+4096]                    ->  X[2k]   = FFT4096(a)[k]
//   b[n] = (x'[n] - x'[n+4096]) W8192^n          ->  X[2k+1] = FFT4096(b)[k]        (x' = windowed input)
// One CTA per vector: the 64 KiB vector arrives in two halves by TMA; every thread forms its 16 a's
// (kept in registers) and b's (parked in the first half of the input buffer, own slots), runs the
// three radix-16 passes on a, then on b, and stores (X[2k], X[2k+1]) pairs as one 16-byte store each,
// so the output is written in whole lines.  The second half of the buffer is refilled for the
// next vector right after the first barrier, the first half as soon as the b's have been read back.
// W8192^{tid + 256 i} = W8192^{tid} * W32^{i}: one per-thread register pair times compile-time
// constants.  One HBM read and one HBM write per sample (the generic radix-2 kernel it replaces for
// this size was latency-bound at 11 % of HBM).
// B200_F8K_EARLY=1 (A/B, tools/f8k_ab.py): the even bins leave as 8-byte stores right after their transform, so that
// their 32 registers are free during the odd transform.  Measured on the B200: 321 -> 256 GS/s (complex output), 358 ->
// 330 (|.|): half-written 32-byte sectors cost more than the registers give.  Off.
#ifndef B200_F8K_EARLY
#define B200_F8K_EARLY 0
#endif
constexpr size_t F8K_SMEM = 8192 * 8 + 16 * F4K_STRIDE * 8 + 256 * 8 + 32;

template <bool FWD, int I>
__device__ __forceinline__ float2 mul_w32(float2 z) // z * e^{-+ j 2 pi I / 32}
{
    constexpr double kPi = 3.14159265358979323846;
    // cos / sin of 2 pi I / 32 for I = 0..15 as compile-time constants
    constexpr float cr[16] = { 1.f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f,
                               0.70710678118654752f, 0.55557023301960218f, 0.38268343236508977f,
                               0.19509032201612825f, 0.f, -0.19509032201612825f, -0.38268343236508977f,
                               -0.55557023301960218f, -0.70710678118654752f, -0.83146961230254524f,
                               -0.92387953251128674f, -0.98078528040323043f };
    constexpr float si[16] = { 0.f, 0.19509032201612825f, 0.38268343236508977f, 0.55557023301960218f,
                               0.70710678118654752f, 0.83146961230254524f, 0.92387953251128674f,
                               0.98078528040323043f, 1.f, 0.98078528040323043f, 0.92387953251128674f,
                               0.83146961230254524f, 0.70710678118654752f, 0.55557023301960218f,
                               0.38268343236508977f, 0.19509032201612825f };
    (void)kPi;
    if (I == 0)
        return z;
    constexpr float wr = cr[I], wi = FWD ? -si[I] : si[I];
    return make_float2(fmaf(-z.y, wi, z.x * wr), fmaf(z.x, wi, z.y * wr));
}

template <bool FWD, int I = 0>
__device__ __forceinline__ void f8k_split(float2 (&a)[16], float2* sIn, const float* __restrict__ w0,
                                          const float* __restrict__ w1, float2 wt, int tid)
{
    if constexpr (I < 16) {
        const float2 x0 = __fmul2_rn(sIn[I * 256 + tid], make_float2(w0[I], w0[I]));
        const float2 x1 = __fmul2_rn(sIn[4096 + I * 256 + tid], make_float2(w1[I], w1[I]));
        a[I] = x0 + x1;
        sIn[I * 256 + tid] = cmul(mul_w32<FWD, I>(x0 - x1), wt);
        f8k_split<FWD, I + 1>(a, sIn, w0, w1, wt, tid);
    }
}

template <bool FWD, int OUT>
__global__ void __launch_bounds__(256, 2)
    fft8192_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                   const float* __restrict__ weff, const float2* __restrict__ tw1,
                   const float2* __restrict__ tw2, float odd_sign)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* sIn = reinterpret_cast<float2*>(smem_raw);
    float2* sA = sIn + 8192;
    float2* sT2 = sA + 16 * F4K_STRIDE;
    uint64_t* bar = reinterpret_cast<uint64_t*>(sT2 + 256); // [0]: first half, [1]: second half
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_mbar_init();
    }
    float2 t1[16];
#pragma unroll
    for (int i = 0; i < 16; i++)
        t1[i] = __ldg(tw1 + i * 256 + tid);
    sT2[tid] = __ldg(tw2 + tid);
    float2 wt; // W8192^{tid}, with the sign of the odd bins of a reverse-shifted transform folded in
    {
        float sn, cs_;
        sincospif((float)tid / 4096.0f, &sn, &cs_);
        wt = make_float2(cs_ * odd_sign, (FWD ? -sn : sn) * odd_sign);
    }
    __syncthreads();
    pdl_wait();              // programmatic dependent launch: everything above overlapped the previous kernel's tail
    pdl_launch_dependents();
    long long vec = blockIdx.x;
    if (tid == 0 && vec < n_vec) {
        mbar_arrive_expect_tx(bar, 4096 * 8);
        bulk_copy_g2s(sIn, in + vec * 8192, 4096 * 8, bar);
        mbar_arrive_expect_tx(bar + 1, 4096 * 8);
        bulk_copy_g2s(sIn + 4096, in + vec * 8192 + 4096, 4096 * 8, bar + 1);
    }
    uint32_t phase = 0;
    for (; vec < n_vec; vec += gridDim.x) {
        float2 e[16], v[16];
        {
            float w0[16], w1[16];
#pragma unroll
            for (int i = 0; i < 16; i++) {
                w0[i] = __ldg(weff + i * 256 + tid);
                w1[i] = __ldg(weff + 4096 + i * 256 + tid);
            }
            mbar_wait(bar, phase);
            mbar_wait(bar + 1, phase);
            phase ^= 1;
            f8k_split<FWD>(e, sIn, w0, w1, wt, tid);
        }
        // ---- even bins: three passes on a (in e[])
        dft16<FWD>(e);
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++)
            sA[k0 * F4K_STRIDE + tid] = cmul(e[pos16(k0)], t1[k0]);
        __syncthreads(); // every thread is done with the second half of sIn
        const long long nxt = vec + gridDim.x;
        if (tid == 0 && nxt < n_vec) {
            mbar_arrive_expect_tx(bar + 1, 4096 * 8);
            bulk_copy_g2s(sIn + 4096, in + nxt * 8192 + 4096, 4096 * 8, bar + 1);
        }
        {
            const int k0 = tid >> 4, n0 = tid & 15;
            float2* row = sA + k0 * F4K_STRIDE + n0;
#pragma unroll
            for (int i = 0; i < 16; i++)
                e[i] = row[i * 16];
            dft16<FWD>(e);
            row[0] = e[pos16(0)];
#pragma unroll
            for (int k1 = 1; k1 < 16; k1++)
                row[k1 * 16] = cmul(e[pos16(k1)], sT2[k1 * 16 + n0]);
        }
        __syncthreads();
        {
            const int k0 = tid & 15, k1 = tid >> 4;
            const float2* row = sA + k0 * F4K_STRIDE + k1 * 16;
#pragma unroll
            for (int i = 0; i < 16; i++)
                e[i] = row[i];
            dft16<FWD>(e); // X[2 (tid + 256 k2)] in e[pos16(k2)]
        }
#if B200_F8K_EARLY
        // A/B: the even bins leave as 8-byte stores now (the odd ones fill the other half of each 16-byte pair
        // later; the pairs merge in L2), so e[] is dead during the odd transform: 32 registers back
        if (OUT == B200_FFT_OUT_COMPLEX) {
            float2* y = reinterpret_cast<float2*>(out) + vec * 8192;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++)
                __stcs(y + 2 * (k2 * 256 + tid), e[pos16(k2)]);
        } else {
            float* y = reinterpret_cast<float*>(out) + vec * 8192;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++) {
                const float2 p = e[pos16(k2)];
                const float pe = fmaf(p.x, p.x, p.y * p.y);
                __stcs(y + 2 * (k2 * 256 + tid), OUT == B200_FFT_OUT_MAG ? sqrt_approx(pe) : pe);
            }
        }
#endif
        __syncthreads(); // pass-3 reads of sA done
        // ---- odd bins: the b's come back from this thread's own slots
#pragma unroll
        for (int i = 0; i < 16; i++)
            v[i] = sIn[i * 256 + tid];
        dft16<FWD>(v);
#pragma unroll
        for (int k0 = 0; k0 < 16; k0++)
            sA[k0 * F4K_STRIDE + tid] = cmul(v[pos16(k0)], t1[k0]);
        __syncthreads(); // every thread has read its b's: the first half of sIn is free
        if (tid == 0 && nxt < n_vec) {
            mbar_arrive_expect_tx(bar, 4096 * 8);
            bulk_copy_g2s(sIn, in + nxt * 8192, 4096 * 8, bar);
        }
        {
            const int k0 = tid >> 4, n0 = tid & 15;
            float2* row = sA + k0 * F4K_STRIDE + n0;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i * 16];
            dft16<FWD>(v);
            row[0] = v[pos16(0)];
#pragma unroll
            for (int k1 = 1; k1 < 16; k1++)
                row[k1 * 16] = cmul(v[pos16(k1)], sT2[k1 * 16 + n0]);
        }
        __syncthreads();
        {
            const int k0 = tid & 15, k1 = tid >> 4;
            const float2* row = sA + k0 * F4K_STRIDE + k1 * 16;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i];
            dft16<FWD>(v); // X[2 (tid + 256 k2) + 1] in v[pos16(k2)]
        }
#if B200_F8K_EARLY
        if (OUT == B200_FFT_OUT_COMPLEX) {
            float2* y = reinterpret_cast<float2*>(out) + vec * 8192;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++)
                __stcs(y + 2 * (k2 * 256 + tid) + 1, v[pos16(k2)]);
        } else {
            float* y = reinterpret_cast<float*>(out) + vec * 8192;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++) {
                const float2 q = v[pos16(k2)];
                const float po = fmaf(q.x, q.x, q.y * q.y);
                __stcs(y + 2 * (k2 * 256 + tid) + 1, OUT == B200_FFT_OUT_MAG ? sqrt_approx(po) : po);
            }
        }
#else
        if (OUT == B200_FFT_OUT_COMPLEX) {
            float4* y = reinterpret_cast<float4*>(out) + vec * 4096;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++) {
                const float2 p = e[pos16(k2)], q = v[pos16(k2)];
                __stcs(y + k2 * 256 + tid, make_float4(p.x, p.y, q.x, q.y));
            }
        } else {
            float2* y = reinterpret_cast<float2*>(out) + vec * 4096;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++) {
                const float2 p = e[pos16(k2)], q = v[pos16(k2)];
                const float pe = fmaf(p.x, p.x, p.y * p.y), po = fmaf(q.x, q.x, q.y * q.y);
                __stcs(y + k2 * 256 + tid, OUT == B200_FFT_OUT_MAG ? make_float2(sqrt_approx(pe), sqrt_approx(po))
                                                                   : make_float2(pe, po));
            }
        }
#endif
        __syncthreads(); // pass-3 reads done before the next vector's pass-1 writes
    }
}

// ---- N = 256, 512, 1024, 2048: same machinery, N = R0 * 256 ------------------------------------
// A CTA always works on 4096 contiguous samples = V = 16/R0 vectors.  Pass 1 is V radix-R0
// butterflies per thread (16 points in registers, as before) with twiddle W_N^{L k0}; that leaves
// 16 rows of 256 points, and passes 2-3 are exactly the N = 4096 ones.  Output index is
// k = k0 + R0 (k1 + 16 k2); pass 3 maps lanes to (k0 fastest, then k1) so stores are contiguous.
// Rows are padded (column stride 17, row stride 272 + 16/R0) to keep every pattern conflict-free.
template <int R0>
struct fr0 {
    static constexpr int V = 16 / R0;
    static constexpr int SK = 17;
    static constexpr int SR = 16 * 17 + (16 / R0);
    static constexpr int N = R0 * 256;
    static constexpr size_t SMEM = 4096 * 8 + 16 * SR * 8 + 256 * 8 + 16;
};

template <bool FWD>
__device__ __forceinline__ void dft2(float2& a, float2& b)
{
    float2 s = a + b, d = a - b;
    a = s;
    b = d;
}

// natural-order 8-point DFT
template <bool FWD>
__device__ __forceinline__ void dft8(float2 (&z)[8])
{
    float2 e0 = z[0], e1 = z[2], e2 = z[4], e3 = z[6];
    float2 o0 = z[1], o1 = z[3], o2 = z[5], o3 = z[7];
    dft4<FWD>(e0, e1, e2, e3);
    dft4<FWD>(o0, o1, o2, o3);
    o1 = mul_w16<FWD, 2>(o1); // W8^1 = W16^2
    o2 = mul_w16<FWD, 4>(o2);
    o3 = mul_w16<FWD, 6>(o3);
    z[0] = e0 + o0;
    z[4] = e0 - o0;
    z[1] = e1 + o1;
    z[5] = e1 - o1;
    z[2] = e2 + o2;
    z[6] = e2 - o2;
    z[3] = e3 + o3;
    z[7] = e3 - o3;
}

template <int R0, bool FWD, int OUT>
__global__ void __launch_bounds__(256, 2)
    fft_r0_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                  const float* __restrict__ weff, const float2* __restrict__ tw1,
                  const float2* __restrict__ tw2, int tma_ok)
{
    using G = fr0<R0>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* sIn = reinterpret_cast<float2*>(smem_raw);
    float2* sA = sIn + 4096;
    float2* sT2 = sA + 16 * G::SR;
    uint64_t* bar = reinterpret_cast<uint64_t*>(sT2 + 256);
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    float wreg[R0];
    float2 t1[R0];
#pragma unroll
    for (int i = 0; i < R0; i++) {
        wreg[i] = __ldg(weff + i * 256 + tid);
        t1[i] = __ldg(tw1 + i * 256 + tid);
    }
    sT2[tid] = __ldg(tw2 + tid);
    __syncthreads();
    const long long n_blocks = (n_vec + G::V - 1) / G::V;
    auto tma_block = [&](long long b) { return tma_ok && (b + 1) * G::V <= n_vec; };
    pdl_wait();              // programmatic dependent launch: everything above overlapped the previous kernel's tail
    pdl_launch_dependents();
    long long blk = blockIdx.x;
    if (tid == 0 && blk < n_blocks && tma_block(blk)) {
        mbar_arrive_expect_tx(bar, 4096 * 8);
        bulk_copy_g2s(sIn, in + blk * 4096, 4096 * 8, bar);
    }
    uint32_t phase = 0;
    for (; blk < n_blocks; blk += gridDim.x) {
        const long long vec0 = blk * G::V;
        float2 v[16];
        if (tma_block(blk)) {
            mbar_wait(bar, phase);
            phase ^= 1;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = sIn[i * 256 + tid];
        } else {
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const long long vv = vec0 + i / R0; // element i*256+tid belongs to vector i / R0
                v[i] = vv < n_vec ? __ldcs(in + blk * 4096 + i * 256 + tid) : make_float2(0.f, 0.f);
            }
        }
        // ---- pass 1: V radix-R0 butterflies; v[vv*R0 + n2]
#pragma unroll
        for (int vv = 0; vv < G::V; vv++) {
            float2 z[R0];
#pragma unroll
            for (int n2 = 0; n2 < R0; n2++)
                z[n2] = __fmul2_rn(v[vv * R0 + n2], make_float2(wreg[n2], wreg[n2]));
            if (R0 == 2)
                dft2<FWD>(z[0], z[R0 > 1 ? 1 : 0]);
            if (R0 == 4)
                dft4<FWD>(z[0], z[R0 > 1 ? 1 : 0], z[R0 > 2 ? 2 : 0], z[R0 > 3 ? 3 : 0]);
            if (R0 == 8)
                dft8<FWD>(reinterpret_cast<float2(&)[8]>(z));
            const int n1 = tid >> 4, n0 = tid & 15;
#pragma unroll
            for (int k0 = 0; k0 < R0; k0++)
                sA[(vv * R0 + k0) * G::SR + n1 * G::SK + n0] = cmul(z[k0], t1[k0]);
        }
        __syncthreads();
        if (tid == 0 && blk + gridDim.x < n_blocks && tma_block(blk + gridDim.x)) {
            mbar_arrive_expect_tx(bar, 4096 * 8);
            bulk_copy_g2s(sIn, in + (blk + gridDim.x) * 4096, 4096 * 8, bar);
        }
        // ---- pass 2: per row, DFT16 over n1, in place
        {
            const int r = tid >> 4, n0 = tid & 15;
            float2* row = sA + r * G::SR + n0;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i * G::SK];
            dft16<FWD>(v);
#pragma unroll
            for (int k1 = 0; k1 < 16; k1++)
                row[k1 * G::SK] = cmul(v[pos16(k1)], sT2[k1 * 16 + n0]);
        }
        __syncthreads();
        // ---- pass 3: lanes = (k0 fastest, k1, vector)
        {
            const int k0 = tid % R0, k1 = (tid / R0) & 15, vv = tid / (R0 * 16);
            const float2* row = sA + (vv * R0 + k0) * G::SR + k1 * G::SK;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i];
            dft16<FWD>(v);
            if (vec0 + vv < n_vec) {
                const long long base = blk * 4096 + vv * G::N + (tid % (R0 * 16));
                if (OUT == B200_FFT_OUT_COMPLEX) {
                    float2* y = reinterpret_cast<float2*>(out) + base;
#pragma unroll
                    for (int k2 = 0; k2 < 16; k2++)
                        __stcs(y + k2 * 16 * R0, v[pos16(k2)]);
                } else {
                    float* y = reinterpret_cast<float*>(out) + base;
#pragma unroll
                    for (int k2 = 0; k2 < 16; k2++) {
                        float2 z = v[pos16(k2)];
                        float p = fmaf(z.x, z.x, z.y * z.y);
                        __stcs(y + k2 * 16 * R0, OUT == B200_FFT_OUT_MAG ? sqrt_approx(p) : p);
                    }
                }
            }
        }
        __syncthreads();
    }
}

// ---- N = 16, 32, 64, 128: two passes (radix R0 then radix 16), N = R0 * 16 ----------------------
// Same block shape again: a CTA transforms 4096 contiguous samples = 4096/N vectors staged by one
// TMA bulk copy.  Pass 1: each thread does 16/R0 radix-R0 butterflies (over n2, n = 16 n2 + n0) and
// applies W_N^{n0 k0}; pass 2: thread p = (vector, k0) does the DFT16 over n0.  k = k0 + R0 k1.
// Results go through a padded shared tile so the global stores are fully coalesced even for N = 16.
template <int R0>
struct fsm {
    static constexpr int N = R0 * 16;
    static constexpr int V = 4096 / N;        // vectors per block
    static constexpr int OS = N + R0;         // padded output row (keeps the scatter conflict-free)
    static constexpr size_t SMEM = 4096 * 8 + 256 * 17 * 8 + (size_t)V * OS * 8 + 128 * 8 + 128 * 4 + 16;
};

template <int R0, bool FWD, int OUT>
__global__ void __launch_bounds__(256, 2)
    fft_small_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                     const float* __restrict__ weff, const float2* __restrict__ tw /* [k0][n0] */, int flip,
                     int tma_ok)
{
    using G = fsm<R0>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* sIn = reinterpret_cast<float2*>(smem_raw);
    float2* sA = sIn + 4096;
    float2* sO = sA + 256 * 17;
    float2* sTw = sO + G::V * G::OS;
    float* sW = reinterpret_cast<float*>(sTw + 128);
    uint64_t* bar = reinterpret_cast<uint64_t*>(sW + 128);
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (tid < G::N) {
        sW[tid] = __ldg(weff + tid);
        sTw[tid] = __ldg(tw + tid);
    }
    __syncthreads();
    const long long n_blocks = (n_vec + G::V - 1) / G::V;
    auto tma_block = [&](long long b) { return tma_ok && (b + 1) * G::V <= n_vec; };
    pdl_wait();              // programmatic dependent launch: everything above overlapped the previous kernel's tail
    pdl_launch_dependents();
    long long blk = blockIdx.x;
    if (tid == 0 && blk < n_blocks && tma_block(blk)) {
        mbar_arrive_expect_tx(bar, 4096 * 8);
        bulk_copy_g2s(sIn, in + blk * 4096, 4096 * 8, bar);
    }
    uint32_t phase = 0;
    for (; blk < n_blocks; blk += gridDim.x) {
        const long long vec0 = blk * G::V;
        const bool staged = tma_block(blk);
        if (staged) {
            mbar_wait(bar, phase);
            phase ^= 1;
        }
        // ---- pass 1: butterflies beta = j*256 + tid -> (vector, n0)
#pragma unroll
        for (int j = 0; j < 16 / R0; j++) {
            const int beta = j * 256 + tid;
            const int vv = beta >> 4, n0 = beta & 15;
            float2 z[R0];
#pragma unroll
            for (int n2 = 0; n2 < R0; n2++) {
                const int e = vv * G::N + n2 * 16 + n0;
                float2 xv;
                if (staged)
                    xv = sIn[e];
                else
                    xv = (vec0 + vv < n_vec) ? __ldcs(in + blk * 4096 + e) : make_float2(0.f, 0.f);
                const float w = sW[n2 * 16 + n0];
                z[n2] = __fmul2_rn(xv, make_float2(w, w));
            }
            if (R0 == 2)
                dft2<FWD>(z[0], z[R0 > 1 ? 1 : 0]);
            if (R0 == 4)
                dft4<FWD>(z[0], z[R0 > 1 ? 1 : 0], z[R0 > 2 ? 2 : 0], z[R0 > 3 ? 3 : 0]);
            if (R0 == 8)
                dft8<FWD>(reinterpret_cast<float2(&)[8]>(z));
#pragma unroll
            for (int k0 = 0; k0 < R0; k0++)
                sA[(vv * R0 + k0) * 17 + n0] = cmul(z[k0], sTw[k0 * 16 + n0]);
        }
        __syncthreads(); // sA complete, sIn consumed
        if (tid == 0 && blk + gridDim.x < n_blocks && tma_block(blk + gridDim.x)) {
            mbar_arrive_expect_tx(bar, 4096 * 8);
            bulk_copy_g2s(sIn, in + (blk + gridDim.x) * 4096, 4096 * 8, bar);
        }
        // ---- pass 2: thread p = vector*R0 + k0, DFT16 over n0
        {
            float2 v[16];
            const float2* row = sA + tid * 17;
#pragma unroll
            for (int i = 0; i < 16; i++)
                v[i] = row[i];
            dft16<FWD>(v);
            const int vv = tid / R0, k0 = tid % R0;
            float2* orow = sO + vv * G::OS + k0;
#pragma unroll
            for (int k1 = 0; k1 < 16; k1++)
                orow[k1 * R0] = v[pos16(k1)];
        }
        __syncthreads();
        // ---- coalesced copy-out of the 4096 results (natural order within each vector)
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const int e = i * 256 + tid;
            const int vv = e / G::N, k = e % G::N;
            if (vec0 + vv < n_vec) {
                float2 z = sO[vv * G::OS + k];
                if (OUT == B200_FFT_OUT_COMPLEX) {
                    if (flip && (k & 1))
                        z = make_float2(-z.x, -z.y);
                    __stcs(reinterpret_cast<float2*>(out) + blk * 4096 + e, z);
                } else {
                    float p = fmaf(z.x, z.x, z.y * z.y);
                    __stcs(reinterpret_cast<float*>(out) + blk * 4096 + e, OUT == B200_FFT_OUT_MAG ? sqrt_approx(p) : p);
                }
            }
        }
        __syncthreads(); // sO / sA free for the next block
    }
}

// ---- N = 8: one thread per vector ---------------------------------------------------------------
// A vector is 64 contiguous bytes: four 16-byte loads, the 8-point DFT in registers, four 16-byte
// stores (two for |.|).  Neighbouring threads touch neighbouring 64-byte blocks, so every sector is
// used; several independent vectors per thread keep enough loads in flight.
template <bool FWD, int OUT>
__global__ void __launch_bounds__(256)
    fft8_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec,
                const float* __restrict__ weff, float2 post, int flip)
{
    float w[8];
#pragma unroll
    for (int i = 0; i < 8; i++)
        w[i] = __ldg(weff + i);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += stride) {
        const float4* src = reinterpret_cast<const float4*>(in + v * 8);
        float2 z[8];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float4 t = __ldcs(src + i);
            z[2 * i] = make_float2(t.x * w[2 * i], t.y * w[2 * i]);
            z[2 * i + 1] = make_float2(t.z * w[2 * i + 1], t.w * w[2 * i + 1]);
        }
        dft8<FWD>(z);
        if (OUT == B200_FFT_OUT_COMPLEX) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                z[k] = cmul(z[k], post);
                if (flip && (k & 1))
                    z[k] = make_float2(-z[k].x, -z[k].y);
            }
            float4* dst = reinterpret_cast<float4*>(out) + v * 4;
#pragma unroll
            for (int i = 0; i < 4; i++)
                __stcs(dst + i, make_float4(z[2 * i].x, z[2 * i].y, z[2 * i + 1].x, z[2 * i + 1].y));
        } else {
            float m[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const float pw = fmaf(z[k].x, z[k].x, z[k].y * z[k].y);
                m[k] = OUT == B200_FFT_OUT_MAG ? sqrt_approx(pw) : pw;
            }
            float4* dst = reinterpret_cast<float4*>(out) + v * 2;
            __stcs(dst, make_float4(m[0], m[1], m[2], m[3]));
            __stcs(dst + 1, make_float4(m[4], m[5], m[6], m[7]));
        }
    }
}

// ---- generic power-of-two radix-2 Stockham (N = 8 .. 8192) ----------------------------------
template <bool FWD, int OUT>
__global__ void __launch_bounds__(512)
    fft_generic_kernel(const float2* __restrict__ in, void* __restrict__ out, long long n_vec, int N,
                       int log2n, int vpb, const float* __restrict__ weff,
                       const float2* __restrict__ tw, float2 post, int flip)
{
    extern __shared__ __align__(16) float2 sbuf[];
    const int per_cta = vpb * N;
    float2* bx = sbuf;
    float2* by = sbuf + per_cta;
    const long long v0 = (long long)blockIdx.x * vpb;
    const int nv = (int)((n_vec - v0) < vpb ? (n_vec - v0) : vpb);
    if (nv <= 0)
        return;
    const int tot = nv * N;
    const float2* x = in + v0 * N;
    for (int i = threadIdx.x; i < tot; i += blockDim.x) {
        float2 t = __ldcs(x + i);
        float w = __ldg(weff + (i & (N - 1)));
        bx[i] = make_float2(t.x * w, t.y * w);
    }
    __syncthreads();
    const int half = N >> 1;
    int s_log = 0;
    for (int n_log = log2n; n_log >= 1; n_log--, s_log++) {
        const int m = 1 << (n_log - 1);
        const int s = 1 << s_log;
        for (int i = threadIdx.x; i < nv * half; i += blockDim.x) {
            int vi = i / half;
            int bi = i - vi * half;
            int p = bi >> s_log;
            int q = bi & (s - 1);
            const float2* xb = bx + vi * N;
            float2* yb = by + vi * N;
            float2 a = xb[q + s * p];
            float2 b = xb[q + s * (p + m)];
            float2 w = __ldg(tw + (p << (log2n - n_log)));
            float2 d = a - b;
            yb[q + s * 2 * p] = a + b;
            yb[q + s * (2 * p + 1)] = cmul(d, w);
        }
        __syncthreads();
        float2* t = bx;
        bx = by;
        by = t;
    }
    for (int i = threadIdx.x; i < tot; i += blockDim.x) {
        float2 z = bx[i];
        int k = i & (N - 1);
        if (OUT == B200_FFT_OUT_COMPLEX) {
            z = cmul(z, post);
            if (flip && (k & 1))
                z = make_float2(-z.x, -z.y);
            __stcs(reinterpret_cast<float2*>(out) + v0 * N + i, z);
        } else {
            float pw = fmaf(z.x, z.x, z.y * z.y);
            __stcs(reinterpret_cast<float*>(out) + v0 * N + i,
                   OUT == B200_FFT_OUT_MAG ? sqrt_approx(pw) : pw);
        }
    }
}

} // namespace b200

using namespace b200;

struct b200_fft {
    int N = 0, log2n = 0;
    int forward = 1, out_mode = 0;
    int flip = 0;
    float2 post{ 1.f, 0.f };
    float* d_weff = nullptr;
    float2* d_tw1 = nullptr; // 4096 path: [16][256]
    float2* d_tw2 = nullptr; // 4096 path: [16][16]
    float2* d_tw = nullptr;  // generic: N/2
    int vpb = 1;
    int grid_4k = 296;
    int use_tma = 1; // TMA-prefetch kernel for N = 4096 when the input is 16-byte aligned
};

template <bool FWD, int OUT>
static int fft_run_t(b200_fft* h, const void* d_in, void* d_out, long long n_vec, cudaStream_t s)
{
    if (h->N == 4096) {
        long long g = n_vec < h->grid_4k ? n_vec : h->grid_4k;
        if (h->use_tma && (uintptr_t)d_in % 16 == 0)
            B200_LAUNCH_PDL((fft4096_tma_kernel<FWD, OUT>), (unsigned)g, 256, f4k_tma_smem(OUT), s,
                        (const float2*)d_in, d_out, n_vec, h->d_weff, h->d_tw1, h->d_tw2);
        else
            B200_LAUNCH((fft4096_kernel<FWD, OUT>), (unsigned)g, 256, 0, s, (const float2*)d_in, d_out,
                        n_vec, h->d_weff, h->d_tw1, h->d_tw2);
    } else if (h->N == 16 || h->N == 32 || h->N == 64 || h->N == 128) {
        const int R0 = h->N / 16, V = 4096 / h->N;
        long long nb = (n_vec + V - 1) / V;
        long long g = nb < h->grid_4k ? nb : h->grid_4k;
        const int tma_ok = (uintptr_t)d_in % 16 == 0;
#define FFT_SM_GO(R)                                                                                     \
    B200_LAUNCH_PDL((fft_small_kernel<R, FWD, OUT>), (unsigned)g, 256, fsm<R>::SMEM, s, (const float2*)d_in, \
                d_out, n_vec, h->d_weff, h->d_tw1, h->flip, tma_ok)
        switch (R0) {
        case 1: FFT_SM_GO(1); break;
        case 2: FFT_SM_GO(2); break;
        case 4: FFT_SM_GO(4); break;
        default: FFT_SM_GO(8); break;
        }
#undef FFT_SM_GO
    } else if (h->N == 256 || h->N == 512 || h->N == 1024 || h->N == 2048) {
        const int R0 = h->N / 256, V = 16 / R0;
        long long nb = (n_vec + V - 1) / V;
        long long g = nb < h->grid_4k ? nb : h->grid_4k;
        const int tma_ok = (uintptr_t)d_in % 16 == 0;
#define FFT_R0_GO(R)                                                                                  \
    B200_LAUNCH_PDL((fft_r0_kernel<R, FWD, OUT>), (unsigned)g, 256, fr0<R>::SMEM, s, (const float2*)d_in, \
                d_out, n_vec, h->d_weff, h->d_tw1, h->d_tw2, tma_ok)
        switch (R0) {
        case 1: FFT_R0_GO(1); break;
        case 2: FFT_R0_GO(2); break;
        case 4: FFT_R0_GO(4); break;
        default: FFT_R0_GO(8); break;
        }
#undef FFT_R0_GO
    } else if (h->N == 8 && (uintptr_t)d_in % 16 == 0 && (uintptr_t)d_out % 16 == 0) {
        long long blocks = (n_vec + 255) / 256;
        const long long cap = 16LL * sm_count();
        B200_LAUNCH((fft8_kernel<FWD, OUT>), (unsigned)(blocks < cap ? blocks : cap), 256, 0, s, (const float2*)d_in,
                    d_out, n_vec, h->d_weff, h->post, h->flip);
    } else if (h->N == 8192 && h->d_tw1 && (uintptr_t)d_in % 16 == 0 && (uintptr_t)d_out % 16 == 0) {
        long long g = n_vec < h->grid_4k ? n_vec : h->grid_4k;
        B200_LAUNCH_PDL((fft8192_kernel<FWD, OUT>), (unsigned)g, 256, F8K_SMEM, s, (const float2*)d_in, d_out, n_vec,
                    h->d_weff, h->d_tw1, h->d_tw2, h->flip ? -1.f : 1.f);
    } else {
        long long blocks = (n_vec + h->vpb - 1) / h->vpb;
        if (blocks > 0x7fffffffLL)
            return set_err(B200_ERR_ARG, "fft: too many vectors for one call");
        int work = h->vpb * h->N / 2;
        int nt = work < 512 ? (work < 32 ? 32 : work) : 512;
        size_t smem = sizeof(float2) * 2 * (size_t)h->vpb * h->N;
        B200_LAUNCH((fft_generic_kernel<FWD, OUT>), (unsigned)blocks, nt, smem, s,
                    (const float2*)d_in, d_out, n_vec, h->N, h->log2n, h->vpb, h->d_weff, h->d_tw,
                    h->post, h->flip);
    }
    return B200_OK;
}

template <bool FWD>
static int fft_run_o(b200_fft* h, const void* d_in, void* d_out, long long n_vec, cudaStream_t s)
{
    switch (h->out_mode) {
    case B200_FFT_OUT_COMPLEX:
        return fft_run_t<FWD, B200_FFT_OUT_COMPLEX>(h, d_in, d_out, n_vec, s);
    case B200_FFT_OUT_MAG:
        return fft_run_t<FWD, B200_FFT_OUT_MAG>(h, d_in, d_out, n_vec, s);
    default:
        return fft_run_t<FWD, B200_FFT_OUT_MAG_SQUARED>(h, d_in, d_out, n_vec, s);
    }
}

template <bool FWD, int OUT>
static cudaError_t fft_tma_attr()
{
    return cudaFuncSetAttribute(fft4096_tma_kernel<FWD, OUT>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f4k_tma_smem(OUT));
}

template <int R0, bool FWD, int OUT>
static cudaError_t fft_r0_attr()
{
    return cudaFuncSetAttribute(fft_r0_kernel<R0, FWD, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)fr0<R0>::SMEM);
}
template <int R0>
static cudaError_t fft_r0_attr_all()
{
    cudaError_t e = cudaSuccess;
    if ((e = fft_r0_attr<R0, true, 0>()) != cudaSuccess) return e;
    if ((e = fft_r0_attr<R0, true, 1>()) != cudaSuccess) return e;
    if ((e = fft_r0_attr<R0, true, 2>()) != cudaSuccess) return e;
    if ((e = fft_r0_attr<R0, false, 0>()) != cudaSuccess) return e;
    if ((e = fft_r0_attr<R0, false, 1>()) != cudaSuccess) return e;
    return fft_r0_attr<R0, false, 2>();
}

template <int R0, bool FWD, int OUT>
static cudaError_t fft_small_attr()
{
    return cudaFuncSetAttribute(fft_small_kernel<R0, FWD, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)fsm<R0>::SMEM);
}
template <int R0>
static cudaError_t fft_small_attr_all()
{
    cudaError_t e = cudaSuccess;
    if ((e = fft_small_attr<R0, true, 0>()) != cudaSuccess) return e;
    if ((e = fft_small_attr<R0, true, 1>()) != cudaSuccess) return e;
    if ((e = fft_small_attr<R0, true, 2>()) != cudaSuccess) return e;
    if ((e = fft_small_attr<R0, false, 0>()) != cudaSuccess) return e;
    if ((e = fft_small_attr<R0, false, 1>()) != cudaSuccess) return e;
    return fft_small_attr<R0, false, 2>();
}

template <bool FWD, int OUT>
static cudaError_t fft_generic_attr()
{
    return cudaFuncSetAttribute(fft_generic_kernel<FWD, OUT>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
}

extern "C" {

int b200_fft_destroy(b200_fft* h)
{
    if (!h)
        return B200_OK;
    cudaFree(h->d_weff);
    cudaFree(h->d_tw1);
    cudaFree(h->d_tw2);
    cudaFree(h->d_tw);
    delete h;
    return B200_OK;
}

int b200_fft_create(const b200_fft_params* p, b200_fft** out)
{
    if (!p || !out)
        return set_err(B200_ERR_ARG, "fft_create: null argument");
    *out = nullptr;
    const int N = p->n;
    if (N < 8 || N > 8192 || (N & (N - 1)))
        return set_err(B200_ERR_UNSUPPORTED, "fft_create: N must be a power of two in [8, 8192], got %d", N);
    if (p->output < 0 || p->output > 2)
        return set_err(B200_ERR_ARG, "fft_create: bad output mode %d", p->output);
    b200_fft* h = new b200_fft();
    h->N = N;
    while ((1 << h->log2n) < N)
        h->log2n++;
    h->forward = p->forward ? 1 : 0;
    h->out_mode = p->output;
    const double sgn = h->forward ? -1.0 : 1.0;

    // effective window: window, shift folding, |k| of a fused upstream multiply_const
    double kmag = 1.0, kph_re = 1.0, kph_im = 0.0;
    if (p->fuse_pre_multiply_const) {
        kmag = std::hypot((double)p->k_re, (double)p->k_im);
        if (kmag > 0.0) {
            kph_re = p->k_re / kmag;
            kph_im = p->k_im / kmag;
        }
    }
    std::vector<float> weff(N);
    for (int n = 0; n < N; n++) {
        double w;
        if (!h->forward && p->shift) {
            // t[n'] = x[(n'+N/2)%N] w[n']  ->  input element n meets w[(n - N/2) mod N]
            w = p->window ? (double)p->window[(n + N - N / 2) % N] : 1.0;
        } else {
            w = p->window ? (double)p->window[n] : 1.0;
            if (h->forward && p->shift && (n & 1))
                w = -w;
        }
        weff[n] = (float)(w * kmag);
    }
    h->flip = (!h->forward && p->shift) ? 1 : 0;
    h->post = make_float2((float)kph_re, (float)kph_im);

#define FFT_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            b200_fft_destroy(h);                                                         \
            return set_err(e__ == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA, \
                           "fft_create: %s -> %s", #call, cudaGetErrorString(e__));      \
        }                                                                                \
    } while (0)

    FFT_CUDA(cudaMalloc(&h->d_weff, sizeof(float) * N));
    FFT_CUDA(cudaMemcpy(h->d_weff, weff.data(), sizeof(float) * N, cudaMemcpyHostToDevice));
    if (N == 4096) {
        std::vector<float2> t1(16 * 256), t2(256);
        for (int k0 = 0; k0 < 16; k0++)
            for (int L = 0; L < 256; L++) {
                double ang = sgn * 2.0 * M_PI * (double)((L * k0) % 4096) / 4096.0;
                double wr = std::cos(ang), wi = std::sin(ang);
                // fold the output phasor and the reverse-shift (-1)^k (k parity = k0 parity)
                double pr = kph_re, pi = kph_im;
                if (h->flip && (k0 & 1)) {
                    pr = -pr;
                    pi = -pi;
                }
                t1[k0 * 256 + L] = make_float2((float)(wr * pr - wi * pi), (float)(wr * pi + wi * pr));
            }
        for (int k1 = 0; k1 < 16; k1++)
            for (int n0 = 0; n0 < 16; n0++) {
                double ang = sgn * 2.0 * M_PI * (double)(n0 * k1) / 256.0;
                t2[k1 * 16 + n0] = make_float2((float)std::cos(ang), (float)std::sin(ang));
            }
        FFT_CUDA(cudaMalloc(&h->d_tw1, sizeof(float2) * t1.size()));
        FFT_CUDA(cudaMemcpy(h->d_tw1, t1.data(), sizeof(float2) * t1.size(), cudaMemcpyHostToDevice));
        FFT_CUDA(cudaMalloc(&h->d_tw2, sizeof(float2) * t2.size()));
        FFT_CUDA(cudaMemcpy(h->d_tw2, t2.data(), sizeof(float2) * t2.size(), cudaMemcpyHostToDevice));
        h->grid_4k = 2 * sm_count();
        if (const char* e = getenv("B200_FFT_TMA"))
            h->use_tma = atoi(e);
        if (const char* e = getenv("B200_FFT_GRID_PER_SM"))
            h->grid_4k = atoi(e) * sm_count();
        FFT_CUDA((fft_tma_attr<true, 0>()));
        FFT_CUDA((fft_tma_attr<true, 1>()));
        FFT_CUDA((fft_tma_attr<true, 2>()));
        FFT_CUDA((fft_tma_attr<false, 0>()));
        FFT_CUDA((fft_tma_attr<false, 1>()));
        FFT_CUDA((fft_tma_attr<false, 2>()));
    } else if (N == 16 || N == 32 || N == 64 || N == 128) {
        const int R0 = N / 16;
        std::vector<float2> t1((size_t)R0 * 16);
        for (int k0 = 0; k0 < R0; k0++)
            for (int n0 = 0; n0 < 16; n0++) {
                double ang = sgn * 2.0 * M_PI * (double)(n0 * k0) / (double)N;
                double wr = std::cos(ang), wi = std::sin(ang);
                t1[(size_t)k0 * 16 + n0] =
                    make_float2((float)(wr * kph_re - wi * kph_im), (float)(wr * kph_im + wi * kph_re));
            }
        FFT_CUDA(cudaMalloc(&h->d_tw1, sizeof(float2) * 128));
        FFT_CUDA(cudaMemset(h->d_tw1, 0, sizeof(float2) * 128));
        FFT_CUDA(cudaMemcpy(h->d_tw1, t1.data(), sizeof(float2) * t1.size(), cudaMemcpyHostToDevice));
        h->grid_4k = 2 * sm_count();
        FFT_CUDA(fft_small_attr_all<1>());
        FFT_CUDA(fft_small_attr_all<2>());
        FFT_CUDA(fft_small_attr_all<4>());
        FFT_CUDA(fft_small_attr_all<8>());
    } else if (N == 256 || N == 512 || N == 1024 || N == 2048) {
        const int R0 = N / 256;
        std::vector<float2> t1((size_t)R0 * 256), t2(256);
        for (int k0 = 0; k0 < R0; k0++)
            for (int L = 0; L < 256; L++) {
                double ang = sgn * 2.0 * M_PI * (double)((L * k0) % N) / (double)N;
                double wr = std::cos(ang), wi = std::sin(ang);
                double pr = kph_re, pi = kph_im;
                if (h->flip && R0 > 1 && (k0 & 1)) { // (-1)^k, k = k0 + R0 (k1 + 16 k2), R0 even
                    pr = -pr;
                    pi = -pi;
                }
                t1[(size_t)k0 * 256 + L] = make_float2((float)(wr * pr - wi * pi), (float)(wr * pi + wi * pr));
            }
        for (int k1 = 0; k1 < 16; k1++)
            for (int n0 = 0; n0 < 16; n0++) {
                double ang = sgn * 2.0 * M_PI * (double)(n0 * k1) / 256.0;
                double f = (h->flip && R0 == 1 && (k1 & 1)) ? -1.0 : 1.0; // N = 256: parity of k is k1's
                t2[k1 * 16 + n0] = make_float2((float)(f * std::cos(ang)), (float)(f * std::sin(ang)));
            }
        FFT_CUDA(cudaMalloc(&h->d_tw1, sizeof(float2) * t1.size()));
        FFT_CUDA(cudaMemcpy(h->d_tw1, t1.data(), sizeof(float2) * t1.size(), cudaMemcpyHostToDevice));
        FFT_CUDA(cudaMalloc(&h->d_tw2, sizeof(float2) * t2.size()));
        FFT_CUDA(cudaMemcpy(h->d_tw2, t2.data(), sizeof(float2) * t2.size(), cudaMemcpyHostToDevice));
        h->grid_4k = 2 * sm_count();
        FFT_CUDA(fft_r0_attr_all<1>());
        FFT_CUDA(fft_r0_attr_all<2>());
        FFT_CUDA(fft_r0_attr_all<4>());
        FFT_CUDA(fft_r0_attr_all<8>());
    } else {
        std::vector<float2> tw(N / 2);
        for (int j = 0; j < N / 2; j++) {
            double ang = sgn * 2.0 * M_PI * (double)j / (double)N;
            tw[j] = make_float2((float)std::cos(ang), (float)std::sin(ang));
        }
        FFT_CUDA(cudaMalloc(&h->d_tw, sizeof(float2) * tw.size()));
        FFT_CUDA(cudaMemcpy(h->d_tw, tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice));
        h->vpb = N >= 1024 ? 1 : 1024 / N;
        FFT_CUDA((fft_generic_attr<true, 0>()));
        FFT_CUDA((fft_generic_attr<true, 1>()));
        FFT_CUDA((fft_generic_attr<true, 2>()));
        FFT_CUDA((fft_generic_attr<false, 0>()));
        FFT_CUDA((fft_generic_attr<false, 1>()));
        FFT_CUDA((fft_generic_attr<false, 2>()));
        if (N == 8192 && !getenv("B200_FFT_GENERIC")) {
            // tables of the two 4096-point sub-transforms of fft8192_kernel: the output phasor of a
            // fused upstream multiply_const is folded in; the reverse-shift (-1)^k is the parity of the
            // radix-2 split and goes into the odd branch's twiddle (odd_sign), not into these
            std::vector<float2> t1(16 * 256), t2(256);
            for (int k0 = 0; k0 < 16; k0++)
                for (int L = 0; L < 256; L++) {
                    double ang = sgn * 2.0 * M_PI * (double)((L * k0) % 4096) / 4096.0;
                    double wr = std::cos(ang), wi = std::sin(ang);
                    t1[k0 * 256 + L] =
                        make_float2((float)(wr * kph_re - wi * kph_im), (float)(wr * kph_im + wi * kph_re));
                }
            for (int k1 = 0; k1 < 16; k1++)
                for (int n0 = 0; n0 < 16; n0++) {
                    double ang = sgn * 2.0 * M_PI * (double)(n0 * k1) / 256.0;
                    t2[k1 * 16 + n0] = make_float2((float)std::cos(ang), (float)std::sin(ang));
                }
            FFT_CUDA(cudaMalloc(&h->d_tw1, sizeof(float2) * t1.size()));
            FFT_CUDA(cudaMemcpy(h->d_tw1, t1.data(), sizeof(float2) * t1.size(), cudaMemcpyHostToDevice));
            FFT_CUDA(cudaMalloc(&h->d_tw2, sizeof(float2) * t2.size()));
            FFT_CUDA(cudaMemcpy(h->d_tw2, t2.data(), sizeof(float2) * t2.size(), cudaMemcpyHostToDevice));
            h->grid_4k = 2 * sm_count();
#define F8K_ATTR(FW, O) \
    FFT_CUDA(cudaFuncSetAttribute(fft8192_kernel<FW, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F8K_SMEM))
            F8K_ATTR(true, 0);
            F8K_ATTR(true, 1);
            F8K_ATTR(true, 2);
            F8K_ATTR(false, 0);
            F8K_ATTR(false, 1);
            F8K_ATTR(false, 2);
#undef F8K_ATTR
        }
    }
#undef FFT_CUDA
    // the uploads above went through the legacy default stream (cudaMemcpy / cudaMemset); the caller's streams are
    // non-blocking and not ordered against it, so finish them before the handle can be used
    if (cudaDeviceSynchronize() != cudaSuccess) {
        b200_fft_destroy(h);
        return set_err(B200_ERR_CUDA, "fft_create: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = h;
    return B200_OK;
}

int b200_fft_geometry(const b200_fft* h, int* n, int* out_item_bytes)
{
    if (!h)
        return set_err(B200_ERR_ARG, "fft_geometry: null handle");
    if (n)
        *n = h->N;
    if (out_item_bytes)
        *out_item_bytes = h->out_mode == B200_FFT_OUT_COMPLEX ? 8 : 4;
    return B200_OK;
}

int b200_fft_run(b200_fft* h, const void* d_in, void* d_out, int64_t n_vectors, b200_stream_t s)
{
    if (!h || n_vectors < 0 || (n_vectors > 0 && (!d_in || !d_out)))
        return set_err(B200_ERR_ARG, "fft_run: bad argument");
    if (n_vectors == 0)
        return B200_OK;
    if ((uintptr_t)d_in % 8 || (uintptr_t)d_out % (h->out_mode == B200_FFT_OUT_COMPLEX ? 8 : 4))
        return set_err(B200_ERR_ARG, "fft_run: misaligned buffer");
    return h->forward ? fft_run_o<true>(h, d_in, d_out, n_vectors, cs(s))
                      : fft_run_o<false>(h, d_in, d_out, n_vectors, cs(s));
}

} // extern "C"

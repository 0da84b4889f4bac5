// pfb.cu -- critically sampled polyphase analysis channelizer (M channels, P taps/branch).
//
//   u_i[t] = sum_{r<P} h[i + r M] x[(t-r) M + (M-1-i)]
//   y_c[t] = sum_{i<M} u_i[t] e^{+j 2 pi i c / M}              out[t*M + c]      (SURVEY.md 8c)
//
// Absent from the reference snapshot (SURVEY.md 0.1); plugs into gr::block::work
// (runtime/include/gnuradio/block.hpp:81-85) as a rate-changing block
// (n_consumed = M * n_produced).
//
// Algorithmically 4P + 5 log2 M flop and 16 B per input sample (AI ~ 6 flop/B for M=64,
// P=16): HBM bound, so the kernel is the polyphase form -- branch FIRs from a shared-memory
// tile with a register sliding window over time, then an M-point DFT across branches done
// in shared memory/registers (radix 4 x 16 for M = 64) -- one HBM read and one HBM write
// per sample.  A dense filterbank*DFT GEMM would execute 8T = 8192 flop/sample and cannot
// reach the HBM bound of this form (SURVEY.md 8d), so it is not used here.
#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"
#include "tc_ptx.cuh"

// (the stage-1 DFT twiddles of pfb64_kernel live in registers: measured +2.9 % over a shared table, 359 -> 369 GS/s)
#ifndef B200_PK_ROT
#define B200_PK_ROT 1 // +-j rotations as one packed add: bit-identical results, +0.5-1 % (measured)
#endif
#ifndef B200_PK_W16
#define B200_PK_W16 0 // packed constant twiddles: within +-2 % either way per kernel (measured), off
#endif

namespace b200 {

__device__ __forceinline__ float2 f2add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }

// reverse (e^{+j}) 4-point DFT
__device__ __forceinline__ void idft4(float2& a, float2& b, float2& c, float2& d)
{
    float2 t0 = f2add(a, c), t1 = f2sub(a, c), t2 = f2add(b, d), t3 = f2sub(b, d);
    a = f2add(t0, t2);
    c = f2sub(t0, t2);
#if B200_PK_ROT
    b = __fadd2_rn(t1, make_float2(-t3.y, t3.x)); // t1 + j t3: one packed add, swap + negate operand modifier
    d = __fadd2_rn(t1, make_float2(t3.y, -t3.x));
#else
    b = make_float2(t1.x - t3.y, t1.y + t3.x);
    d = make_float2(t1.x + t3.y, t1.y - t3.x);
#endif
}

__device__ __forceinline__ float2 cmulc(float2 z, float wr, float wi)
{
#if B200_PK_W16
    const float2 r = __fmul2_rn(z, make_float2(wr, wr)); // two packed instructions, see cmul (common.cuh)
    return __ffma2_rn(make_float2(-z.y, z.x), make_float2(wi, wi), r);
#else
    return make_float2(fmaf(-z.y, wi, z.x * wr), fmaf(z.x, wi, z.y * wr));
#endif
}

// reverse 16-point DFT, output X[k] in v[4*(k&3) + (k>>2)]
__device__ __forceinline__ void idft16(float2 (&v)[16])
{
    constexpr float C8 = 0.92387953251128674f, S8 = 0.38268343236508977f, R2 = 0.70710678118654752f;
#pragma unroll
    for (int b = 0; b < 4; b++)
        idft4(v[b], v[4 + b], v[8 + b], v[12 + b]);
    v[5] = cmulc(v[5], C8, S8);
    v[6] = cmulc(v[6], R2, R2);
    v[7] = cmulc(v[7], S8, C8);
    v[9] = cmulc(v[9], R2, R2);
    v[10] = make_float2(-v[10].y, v[10].x);
    v[11] = cmulc(v[11], -R2, R2);
    v[13] = cmulc(v[13], S8, C8);
    v[14] = cmulc(v[14], -R2, R2);
    v[15] = cmulc(v[15], -C8, -S8);
#pragma unroll
    for (int c = 0; c < 4; c++)
        idft4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}

// stream sample g relative to the new input (g < 0 -> halo of nh samples, oldest first)
__device__ __forceinline__ float2 pfb_fetch(const float2* __restrict__ x, const float2* __restrict__ halo,
                                            long long nh, long long g, long long n_in)
{
    if (g >= 0)
        return g < n_in ? __ldcs(x + g) : make_float2(0.f, 0.f);
    if (halo && g >= -nh)
        return __ldg(halo + (nh + g));
    return make_float2(0.f, 0.f);
}

constexpr int PFB64_TT = 64;  // frames per tile
constexpr int PFB64_RS = 68;  // u row stride (complex): 68 = 4 mod 16 keeps the 4-lane-contiguous DFT accesses conflict-free

// M = 64.  256 threads, persistent over 64-frame tiles.
// smem: X[(TT+P4-1)][64] | U[TT][65] | taps[P4][64] | tw64[64] | mbarrier
// The input tile is one contiguous span of the stream, so interior tiles are staged by a 1-D TMA
// bulk copy issued as soon as the branch filters of the previous tile have consumed X -- it lands
// while the 64-point DFTs and the output stores of that tile run.
// OS = 2, 4 (oversampled bank, DESIGN.md 4.4e): frames advance by D = 64 / OS samples, the input tile is
// TT + P4 OS - 1 rows of D samples, and branch outputs go to their circularly shifted U slot.
template <int P4T, int OS = 1> // P4T > 0: taps per branch known at compile time (fully unrolled filters)
__global__ void __launch_bounds__(256, 2)
    pfb64_kernel(const float2* __restrict__ x, const float2* __restrict__ halo, float2* __restrict__ out,
                 const float* __restrict__ taps_rm /* [P4][64] */, int P4, int Ptrue,
                 long long n_frames, long long n_in, int ch_begin, int ch_count, int tma_ok, int nbuf,
                 int phase0 /* OS > 1: (frame index of out[0]) mod OS */)
{
    constexpr int D = 64 / OS; // hop: input samples per frame = samples per row of the input tile
    // nbuf = 2 (P4T > 0 and P <= 16, see b200_pfb_create): TWO input tiles, the copy of tile i+1 is issued a whole tile
    // ahead of its use.  With one buffer the copy only had the DFT stage to hide behind and 10.5 % of all warp samples
    // sat on the input mbarrier (ncu r02_pfb64_v4).  Two tiles + U are exactly the 115 712 bytes a CTA may use with two
    // CTAs per SM, so the taps live in registers for the lifetime of the CTA (no shared copy) and the two mbarriers sit
    // in the padding of U's first row (elements 64..67 of a row are never touched).
    extern __shared__ __align__(128) float2 sm[];
    const int rows = PFB64_TT + P4 * OS - 1;
    float2* X0 = sm;
    float2* U = X0 + nbuf * rows * D;
    uint64_t* bar = reinterpret_cast<uint64_t*>(U + 64);
    float* hT = reinterpret_cast<float*>(U + PFB64_TT * PFB64_RS); // only when P4T == 0 (taps not in registers)
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_mbar_init();
    }
    if (P4T == 0)
        for (int i = tid; i < P4 * 64; i += 256)
            hT[i] = __ldg(taps_rm + i);
    float hreg[P4T > 0 ? P4T : 1];
    if (P4T > 0) {
#pragma unroll
        for (int r = 0; r < P4T; r++)
            hreg[r] = __ldg(taps_rm + r * 64 + (tid & 63));
    }
    const long long nh = (long long)(Ptrue - 1) * 64 + (64 - D); // P M - D samples of history
    const long long n_tiles = (n_frames + PFB64_TT - 1) / PFB64_TT;
    // stage-1 twiddles W64^{i0 c1} depend on the thread only (i0 = tid & 3): register resident
    float2 twr[16];
#pragma unroll
    for (int c1 = 1; c1 < 16; c1++) {
        float sn, cs_;
        sincospif((float)(((tid & 3) * c1) & 63) / 32.0f, &sn, &cs_); // e^{+j 2 pi i0 c1 / 64}
        twr[c1] = make_float2(cs_, sn);
    }
    const uint32_t tile_bytes = (uint32_t)rows * (uint32_t)D * 8u;
    // can tile `t` be staged by TMA?  (whole span inside [0, n_in), 16-byte aligned source)
    auto tma_tile = [&](long long t) {
        const long long g0 = (t * PFB64_TT - (P4 * OS - 1)) * D;
        return tma_ok && g0 >= 0 && g0 + (long long)rows * D <= n_in;
    };
    __syncthreads();
    // programmatic dependent launch (B200_LAUNCH_PDL): the prologue above ran while the previous kernel in the
    // stream drained; nothing below may start before that kernel has completed and flushed
    pdl_wait();
    pdl_launch_dependents();
    long long tile = blockIdx.x;
    if (tid == 0)
        for (int b = 0; b < nbuf; b++) {
            const long long t = tile + (long long)b * gridDim.x;
            if (t < n_tiles && tma_tile(t)) {
                mbar_arrive_expect_tx(bar + b, tile_bytes);
                bulk_copy_g2s(X0 + b * rows * D, x + (t * PFB64_TT - (P4 * OS - 1)) * D, tile_bytes, bar + b);
            }
        }
    uint32_t phase = 0; // bit b: parity of the next completion of bar[b]
    int it = 0;

    for (; tile < n_tiles; tile += gridDim.x, it++) {
        const long long f0 = tile * PFB64_TT; // first frame of the tile
        const int xb = nbuf == 2 ? (it & 1) : 0;
        float2* X = X0 + xb * rows * D;
        // rows: row j holds samples [(f0 - (P4 OS - 1) + j) D, ... + D); at OS = 1 frame (f0 - (P4-1) + j)
        if (tma_tile(tile)) {
            mbar_wait(bar + xb, (phase >> xb) & 1u);
            phase ^= 1u << xb;
        } else {
            const long long g0 = (f0 - (P4 * OS - 1)) * D;
            for (int i0 = tid; i0 < rows * D; i0 += 256 * 8) {
                float2 v[8];
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * D)
                        v[u] = pfb_fetch(x, halo, nh, g0 + i0 + u * 256, n_in);
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * D)
                        X[i0 + u * 256] = v[u];
            }
            __syncthreads();
        }

        // ---- branch filters: thread = (branch i, 16 consecutive frames) ------------------
        {
            const int i = tid & 63, tg = tid >> 6;
            // branch i = a D + b, frame j of the thread, tap r: column D-1-b of row tg*16 + j + (P4-1-r) OS + (OS-1-a)
            // (OS = 1: a = 0, b = i, row tg*16 + j + (P4-1) - r)
            const int a = i / D, b = i % D;
            const float2* col = X + (D - 1 - b) + (tg * 16 + OS - 1 - a) * D;
            float2 acc[16];
#pragma unroll
            for (int j = 0; j < 16; j++)
                acc[j] = make_float2(0.f, 0.f);
            if (P4T > 0) {
                // taps in registers, every input row read exactly once: row rho feeds the
                // (frame j, tap r) pairs with j + (P4-1 - r) OS == rho
#pragma unroll
                for (int rho = 0; rho < 16 + (P4T - 1) * OS; rho++) {
                    const float2 v = col[rho * D];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const int r = P4T - 1 - (rho - j) / OS;
                        if ((rho - j) % OS == 0 && r >= 0 && r < P4T)
                            acc[j] = __ffma2_rn(v, make_float2(hreg[r], hreg[r]), acc[j]);
                    }
                }
            } else {
                for (int rc = 0; rc < P4; rc += 4) {
                    // taps r = rc..rc+3 ; rows needed: j + (P4-1 - r) OS for j in 0..15
                    const float h0 = hT[(rc + 0) * 64 + i], h1 = hT[(rc + 1) * 64 + i];
                    const float h2 = hT[(rc + 2) * 64 + i], h3 = hT[(rc + 3) * 64 + i];
                    const float2* base = col + (P4 - 1 - rc - 3) * OS * D;
                    float2 w[16 + 3 * OS];
#pragma unroll
                    for (int q = 0; q < 16 + 3 * OS; q++)
                        w[q] = base[q * D];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        acc[j] = __ffma2_rn(w[j + 3 * OS], make_float2(h0, h0), acc[j]);
                        acc[j] = __ffma2_rn(w[j + 2 * OS], make_float2(h1, h1), acc[j]);
                        acc[j] = __ffma2_rn(w[j + OS], make_float2(h2, h2), acc[j]);
                        acc[j] = __ffma2_rn(w[j], make_float2(h3, h3), acc[j]);
                    }
                }
            }
            // circular shift of the branches: u_i[t] goes to slot (i - t D) mod 64, t = phase0 + f0 + tg*16 + j, and
            // f0 + tg*16 is a multiple of OS.  Consecutive lanes still write a contiguous run (mod 64) of a row.
#pragma unroll
            for (int j = 0; j < 16; j++)
                U[(tg * 16 + j) * PFB64_RS + (OS == 1 ? i : (i - (phase0 + j) * D) & 63)] = acc[j];
        }
        __syncthreads(); // U complete; X fully consumed
        {
            const long long nxt = tile + (long long)nbuf * gridDim.x; // refill the buffer just consumed
            if (tid == 0 && nxt < n_tiles && tma_tile(nxt)) {
                mbar_arrive_expect_tx(bar + xb, tile_bytes);
                bulk_copy_g2s(X, x + (nxt * PFB64_TT - (P4 * OS - 1)) * D, tile_bytes, bar + xb);
            }
        }

        // ---- 64-point reverse DFT across branches: i = 4 i1 + i0, c = c1 + 16 c0 -----------
        //   stage 1, thread (frame t, i0):  A_{i0}[c1] = W64^{i0 c1} sum_{i1} u[4 i1 + i0] W16^{i1 c1}
        //   stage 2, thread (4 frames, c1): y[c1 + 16 c0] = sum_{i0} A_{i0}[c1] W4^{i0 c0}
        // Stage 2 puts 16 consecutive channels on 16 consecutive lanes, so every output store
        // instruction writes whole 128-byte lines (the radix 4 x 16 order wrote 32-byte pieces of
        // eight lines per instruction, and the store wavefronts were a quarter of the LSU traffic).
        // Rows are warp-local (warp w owns frames 8w..8w+7) in both stages: __syncwarp suffices.
        {
            const int t = tid >> 2, i0 = tid & 3;
            float2* row = U + t * PFB64_RS;
            float2 v[16];
#pragma unroll
            for (int i1 = 0; i1 < 16; i1++)
                v[i1] = row[4 * i1 + i0];
            idft16(v); // A[c1] in v[4*(c1&3) + (c1>>2)]
            __syncwarp();
            row[i0] = v[0];
#pragma unroll
            for (int c1 = 1; c1 < 16; c1++) {
                const float2 w = twr[c1];
                row[4 * c1 + i0] = cmulc(v[4 * (c1 & 3) + (c1 >> 2)], w.x, w.y);
            }
            __syncwarp();
        }
        {
            const int lane = tid & 31, c1 = lane & 15;
            const int fq = (tid >> 5) * 8 + (lane >> 4) * 4; // first of this thread's four frames
            const int swap = (c1 >> 2) & 1;                  // bank-conflict-free order of the two 16-byte halves
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const float4* src = reinterpret_cast<const float4*>(U + (fq + q) * PFB64_RS + 4 * c1);
                const float4 p0 = src[swap], p1 = src[swap ^ 1];
                const float4 lo = swap ? p1 : p0, hi = swap ? p0 : p1;
                float2 a = make_float2(lo.x, lo.y), b = make_float2(lo.z, lo.w);
                float2 c = make_float2(hi.x, hi.y), d = make_float2(hi.z, hi.w);
                idft4(a, b, c, d); // y[c1 + 16 c0], c0 = 0..3
                const long long f = f0 + fq + q;
                if (f < n_frames) {
                    float2* y = out + f * ch_count - ch_begin;
                    const float2 r[4] = { a, b, c, d };
#pragma unroll
                    for (int c0 = 0; c0 < 4; c0++) {
                        const int ch = c1 + 16 * c0;
                        if (ch >= ch_begin && ch < ch_begin + ch_count)
                            __stcs(y + ch, r[c0]);
                    }
                }
            }
        }
        __syncthreads(); // U free for the next tile's branch filters
    }
}

// ---- M = 64, the 64-point DFT across branches as a GEMM on the tensor cores (algorithm 2) -------
// BASELINE.json configs[3]: "64-channel polyphase channelizer (filterbank + DFT as tensor-core GEMM)";
// SURVEY.md 8(d): build the GEMM form, measure it against the SIMT DFT and keep the faster one.
// Only the DFT is a dense contraction worth the tensor pipe (the fused filterbank x DFT matrix executes
// 8T = 8192 flop/sample x 3 split products: 57 GS/s at the measured bf16 peak, against ~370 measured for
// this form), so the branch filters stay the register-window FFMA2 code of pfb64_kernel and
//
//   [y_re ; y_im][c][t] = sum_k A[2c + part][k] * B[t][k],   k = 2 i + (re | im) of branch output u_i[t]
//   A[2c][2i] = cos th, A[2c][2i+1] = -sin th, A[2c+1][2i] = sin th, A[2c+1][2i+1] = cos th, th = 2 pi i c / 64
//
// is one 128 x 64 x 128 GEMM per 64-frame tile: M = 128 rows (channel, re/im), N = 64 frames, K = 128.
// Precision: both operands split into bf16 hi + lo; hi*hi + lo*hi + hi*lo (lo*lo is below fp32 rounding)
// = 3 x 8 MMAs of 128 x 64 x 16 per tile, fp32 accumulation in TMEM.  The DFT matrix never changes: it is
// written once per CTA into tensor memory (A from TMEM: 64 + 64 columns), the MMAs read only the branch
// outputs from shared memory.  B is K-major SWIZZLE_128B: a frame's 128 k-values are two 128-byte rows
// (K-atoms: branches 0..31 / 32..63); the filter thread of branch i writes (re, im) of a frame as ONE
// 32-bit store per plane, a warp covers a whole row -- the same 8 B/sample of shared-memory stores the SIMT
// kernel spends on U, and nothing else: no DFT loads, stores, twiddles or butterflies.
// Epilogue: TMEM lane 2c + part holds y_part[c] of 32 frames per warp, i.e. the lanes of a warp are the 32
// consecutive floats (16 channels x re, im) of a frame: every store instruction writes one whole 128-byte line,
// with no exchange between lanes.  Tiles are software-pipelined: the MMAs of tile i run while the CTA drains tile
// i-1 and filters tile i+1, whose input arrived a whole tile earlier (two input buffers: with one, the copy had only
// the short epilogue to hide behind and a fifth of all warp samples sat on its mbarrier).  2 CTAs/SM, 256 TMEM
// columns each (DFT matrix 128 + 2 accumulator stages of 64); the branch taps live in registers.
constexpr int PFBT_PLANE = 2 * 64 * 128; // one plane (hi or lo) of a tile: 2 K-atoms x 64 frames x 128 bytes
constexpr int PFBT_TMEM_COLS = 256;
constexpr uint32_t PFBT_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

// shared-memory descriptor of an MN-major SWIZZLE_128B operand: atoms of 8 k-rows x 64 n-elements (1 KiB), SBO = stride
// between the atoms along K; LBO (stride between 64-element groups along N) is not used with N = 64
__device__ __forceinline__ uint64_t pfbt_desc_mn(uint32_t saddr)
{
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)(8192 >> 4) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

constexpr int PFBT_THREADS = 288; // 8 worker warps (filters, conversion, epilogue) + 1 issuer warp (TMA refills, MMAs)

__device__ __forceinline__ void pfbt_bar_arrive(int id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(PFBT_THREADS) : "memory"); }
__device__ __forceinline__ void pfbt_bar_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(PFBT_THREADS) : "memory"); }
__device__ __forceinline__ void pfbt_workers_sync() { asm volatile("bar.sync 3, 256;" ::: "memory"); }

template <int P4T>
__global__ void __launch_bounds__(PFBT_THREADS, 2)
    pfb64_tc_kernel(const float2* __restrict__ x, const float2* __restrict__ halo, float2* __restrict__ out,
                    const float* __restrict__ taps_rm /* [P4][64] */, const uint4* __restrict__ gA /* [128][hi 128 | lo 128] bf16 */,
                    int P4, int Ptrue, long long n_frames, long long n_in, int ch_begin, int ch_count, int tma_ok, int mn)
{
    // mn = 1: the branch outputs are stored MN-major (frames contiguous, layout verified by tools/mn_probe.cu): a
    // filter thread holds 16 consecutive frames of ONE branch, i.e. two 16-byte runs per (re | im, hi | lo) plane row --
    // 8 STS.128 per thread and tile instead of the 32 STS.32 of the K-major layout (mn = 0, kept for the A/B).  K is then
    // ordered planar (k = i: re of branch i, k = 64 + i: im), which the host-built DFT matrix gA matches.
    extern __shared__ uint8_t pfbt_raw[];
    uint8_t* planes = tc_align1024(pfbt_raw);                       // [hi, lo] planes of the tile being multiplied
    const int rows = PFB64_TT + P4 - 1;
    float2* X0 = reinterpret_cast<float2*>(planes + 2 * PFBT_PLANE); // two input tiles: the copy of tile i+1 lands while tile i is filtered
    uint64_t* bar = reinterpret_cast<uint64_t*>(X0 + 2 * rows * 64); // [0], [1]: input tile landed; [2], [3]: accumulator stage complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 4);
    const int tid = threadIdx.x, warp = tc_warp_idx(), lane = tid & 31;
    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < 4; b++)
            mbar_init(bar + b, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        __syncwarp();
        tc_alloc(tmem_slot, PFBT_TMEM_COLS);
    }
    // this thread's branch taps: constants of the thread, register resident for the lifetime of the CTA
    float hreg[P4T];
#pragma unroll
    for (int r = 0; r < P4T; r++)
        hreg[r] = __ldg(taps_rm + r * 64 + (tid & 63));
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0); // warp-uniform for the compiler (MMA operands)
    if (warp < 4) {
        // one-off: row m = 32 warp + lane of the DFT matrix -> this thread's TMEM lane, hi then lo
        const uint4* row = gA + (size_t)(warp * 32 + lane) * 32;
        const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 4
        for (int k = 0; k < 16; k++) {
            const uint4 a = __ldg(row + 2 * k), b = __ldg(row + 2 * k + 1);
            const uint32_t v[8] = { a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w };
            tc_st8(tl + k * 8, v);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const long long nh = (long long)(Ptrue - 1) * 64;
    const long long n_tiles = (n_frames + PFB64_TT - 1) / PFB64_TT;
    const uint32_t tile_bytes = (uint32_t)rows * 64u * 8u;
    auto tma_tile = [&](long long t) {
        const long long g0 = (t * PFB64_TT - (P4 - 1)) * 64;
        return tma_ok && g0 >= 0 && g0 + (long long)rows * 64 <= n_in;
    };
    auto issue = [&](long long t, int b) { // one elected thread
        mbar_arrive_expect_tx(bar + b, tile_bytes);
        bulk_copy_g2s(X0 + b * rows * 64, x + (t * PFB64_TT - (P4 - 1)) * 64, tile_bytes, bar + b);
    };
    // drain accumulator stage `st` (tile starting at frame f0) into out; the caller has waited for its MMAs
    auto epilogue = [&](int st, long long f0) {
        const int quarter = warp & 3, half = warp >> 2;
        float v[32];
        tc_ld32(tmem + ((uint32_t)(quarter * 32) << 16) + 128 + st * 64 + half * 32, v);
        tc_wait_ld();
        tc_fence_before();
        // lane 2c + part of the quarter holds y_part[c] of 32 frames: lanes store their own float, so a warp writes
        // the 16 (re, im) pairs of one frame as ONE contiguous 128-byte line per instruction -- no exchange at all
        const int c = quarter * 16 + (lane >> 1);
        float* y = reinterpret_cast<float*>(out + (f0 + half * 32) * ch_count - ch_begin + c) + (lane & 1);
        if (ch_count == 64 && f0 + PFB64_TT <= n_frames) {
#pragma unroll
            for (int n = 0; n < 32; n++)
                __stcs(y + n * 128, v[n]);
        } else {
            const bool ch_ok = c >= ch_begin && c < ch_begin + ch_count;
#pragma unroll
            for (int n = 0; n < 32; n++)
                if (ch_ok && f0 + half * 32 + n < n_frames)
                    __stcs(y + (long long)n * 2 * ch_count, v[n]);
        }
    };

    // programmatic dependent launch (B200_LAUNCH_PDL): the prologue above ran while the previous kernel in the
    // stream drained; nothing below may start before that kernel has completed and flushed
    pdl_wait();
    pdl_launch_dependents();
    long long tile = blockIdx.x;
    const uint32_t planes_s = smem_u32(planes);
    if (warp == 8) {
        // ================= issuer warp: input copies and MMAs =================
        if (lane == 0) {
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const long long t = tile + (long long)b * gridDim.x;
                if (t < n_tiles && tma_tile(t))
                    issue(t, b);
            }
        }
        __syncwarp();
        for (int it = 0; tile < n_tiles; tile += gridDim.x, it++) {
            const int st = it & 1;
            // every worker has written its part of the planes (and fenced it for the async proxy), is done with
            // input buffer st, and has drained accumulator stage st (tile it-2)
            pfbt_bar_sync(1 + st);
            tc_fence_after();
            const long long nxt = tile + 2LL * gridDim.x; // refill the buffer just consumed: two tiles ahead
            if (lane == 0 && nxt < n_tiles && tma_tile(nxt))
                issue(nxt, st);
            __syncwarp();
            const uint32_t d = tmem + 128 + st * 64;
#pragma unroll
            const uint32_t idesc = mn ? (PFBT_IDESC | (1u << 16)) : PFBT_IDESC; // bit 16: B is MN-major
            for (int ks = 0; ks < 8; ks++) {
                // K-major: K-step = 32 bytes inside the 128-byte rows of a K-atom; MN-major: two 8-row atoms of 1 KiB
                const uint32_t boff = mn ? ks * 2048 : (ks >> 2) * 8192 + (ks & 3) * 32;
                const uint64_t bh = mn ? pfbt_desc_mn(planes_s + boff) : tc_desc(planes_s + boff);
                const uint64_t bl = mn ? pfbt_desc_mn(planes_s + PFBT_PLANE + boff) : tc_desc(planes_s + PFBT_PLANE + boff);
                tc_mma_bf16_ts_w(d, tmem + ks * 8, bh, idesc, ks != 0);   // F_hi u_hi
                tc_mma_bf16_ts_w(d, tmem + 64 + ks * 8, bh, idesc, 1);    // F_lo u_hi
                tc_mma_bf16_ts_w(d, tmem + ks * 8, bl, idesc, 1);         // F_hi u_lo
            }
            tc_commit_w(smem_u32(bar + 2 + st));
        }
    } else {
        // ================= worker warps: no barrier among themselves in the steady state =================
        uint32_t xph = 0; // bit b: parity of the next completion of bar[b]
        int it = 0;
        long long prev_f0 = 0;
        for (; tile < n_tiles; tile += gridDim.x, it++) {
            const long long f0 = tile * PFB64_TT;
            const int st = it & 1;
            float2* X = X0 + st * rows * 64;
            if (tma_tile(tile)) {
                mbar_wait(bar + st, (xph >> st) & 1u);
                xph ^= 1u << st;
            } else {
                // edge tile (history in front of the call, ragged end, unaligned stream): fetched element-wise.  The
                // buffer is free: the issuer refills it only for tiles that pass tma_tile
                const long long g0 = (f0 - (P4 - 1)) * 64;
                pfbt_workers_sync(); // nobody still filters the tile that used this buffer two tiles ago
                for (int i0 = tid; i0 < rows * 64; i0 += 256 * 8) {
                    float2 v[8];
#pragma unroll
                    for (int u = 0; u < 8; u++)
                        if (i0 + u * 256 < rows * 64)
                            v[u] = pfb_fetch(x, halo, nh, g0 + i0 + u * 256, n_in);
#pragma unroll
                    for (int u = 0; u < 8; u++)
                        if (i0 + u * 256 < rows * 64)
                            X[i0 + u * 256] = v[u];
                }
                pfbt_workers_sync();
            }
            // ---- branch filters: thread = (branch i, 16 consecutive frames), as in pfb64_kernel
            const int i = tid & 63, tg = tid >> 6;
            const float2* col = X + (63 - i) + (tg * 16) * 64;
            float2 acc[16];
#pragma unroll
            for (int j = 0; j < 16; j++)
                acc[j] = make_float2(0.f, 0.f);
#pragma unroll
            for (int rho = 0; rho < 16 + P4T - 1; rho++) {
                const float2 v = col[rho * 64];
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    const int r = j + P4T - 1 - rho;
                    if (r >= 0 && r < P4T)
                        acc[j] = __ffma2_rn(v, make_float2(hreg[r], hreg[r]), acc[j]);
                }
            }
            // the MMAs of the previous tile must have read the planes before they are overwritten (they were
            // issued a whole filter pass ago: this wait is normally over already); it also publishes that
            // tile's accumulator stage for the epilogue below
            if (it > 0) {
                mbar_wait(bar + 2 + (st ^ 1), (uint32_t)(((it - 1) >> 1) & 1));
                tc_fence_after();
            }
            if (mn) {
                // MN-major planes: row k = i (re) / 64 + i (im) of atom k / 8, the thread's frames 16 tg .. 16 tg + 15 are
                // the 16-byte chunks 2 tg and 2 tg + 1 of that row (XOR-swizzled by the row inside the atom).  The eight
                // lanes of a quarter-warp sit on the eight rows of one atom: conflict-free 16-byte stores.
                uint8_t* rowre = planes + (i >> 3) * 1024 + (i & 7) * 128;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    uint32_t rh[4], rl[4], ih[4], il[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const float2 a0 = acc[8 * h + 2 * q], a1 = acc[8 * h + 2 * q + 1];
                        const __nv_bfloat162 hr = __floats2bfloat162_rn(a0.x, a1.x), hi_ = __floats2bfloat162_rn(a0.y, a1.y);
                        const float2 hrf = __bfloat1622float2(hr), hif = __bfloat1622float2(hi_);
                        const __nv_bfloat162 lr = __floats2bfloat162_rn(a0.x - hrf.x, a1.x - hrf.y);
                        const __nv_bfloat162 li = __floats2bfloat162_rn(a0.y - hif.x, a1.y - hif.y);
                        rh[q] = *reinterpret_cast<const uint32_t*>(&hr);
                        ih[q] = *reinterpret_cast<const uint32_t*>(&hi_);
                        rl[q] = *reinterpret_cast<const uint32_t*>(&lr);
                        il[q] = *reinterpret_cast<const uint32_t*>(&li);
                    }
                    const int off = ((2 * tg + h) ^ (i & 7)) << 4;
                    *reinterpret_cast<uint4*>(rowre + off) = make_uint4(rh[0], rh[1], rh[2], rh[3]);
                    *reinterpret_cast<uint4*>(rowre + PFBT_PLANE + off) = make_uint4(rl[0], rl[1], rl[2], rl[3]);
                    *reinterpret_cast<uint4*>(rowre + 8192 + off) = make_uint4(ih[0], ih[1], ih[2], ih[3]);
                    *reinterpret_cast<uint4*>(rowre + 8192 + PFBT_PLANE + off) = make_uint4(il[0], il[1], il[2], il[3]);
                }
            } else {
            // (re, im) of u_i[t] -> k = 2i, 2i + 1 of frame row t: bf16 hi and lo planes
            uint8_t* pl = planes + (i >> 5) * 8192 + (i & 3) * 4;
            const int chunk = (i & 31) >> 2;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const int n = tg * 16 + j;
                const __nv_bfloat162 hi = __floats2bfloat162_rn(acc[j].x, acc[j].y);
                const float2 hf = __bfloat1622float2(hi);
                const __nv_bfloat162 lo = __floats2bfloat162_rn(acc[j].x - hf.x, acc[j].y - hf.y);
                const int off = n * 128 + ((chunk ^ (n & 7)) << 4);
                *reinterpret_cast<__nv_bfloat162*>(pl + off) = hi;
                *reinterpret_cast<__nv_bfloat162*>(pl + PFBT_PLANE + off) = lo;
            }
            }
            fence_proxy_async(); // generic-proxy stores -> visible to the tensor core's async-proxy reads
            tc_fence_before();
            pfbt_bar_arrive(1 + st); // hand the tile to the issuer and carry on: no wait here
            if (it > 0)
                epilogue(st ^ 1, prev_f0);
            prev_f0 = f0;
        }
        if (it > 0) {
            mbar_wait(bar + 2 + ((it - 1) & 1), (uint32_t)(((it - 1) >> 1) & 1));
            tc_fence_after();
            epilogue((it - 1) & 1, prev_f0);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tc_dealloc(tmem, PFBT_TMEM_COLS);
    }
}

// ---- M = 16, 32, 128, 256: the same single-pass structure as pfb64_kernel -----------------------
// 4096-sample tiles (TT = 4096/M frames), branch filters with register-resident taps and a
// 16-frame sliding window per thread, then the M-point reverse DFT across branches as radix 16
// (over i1, i = S i1 + i0, S = M/16; thread = frame x i0, twiddles W_M^{i0 c1} in registers) followed by
// radix S over i0 with thread = (frame, c1): 16 consecutive channels on 16 consecutive lanes, i.e.
// whole-line output stores.  Stage 1 leaves A_{i0}[c1] at row[17 i0 + c1] (row stride 17 S): both its
// 4-lane-contiguous accesses and stage 2's lane-contiguous LDS.64 reads are bank-conflict free.
// One HBM read and one HBM write per sample (the two-kernel form it replaces made two round trips).
template <int M>
struct pfbm {
    static constexpr int S = M / 16;
    static constexpr int TT = 4096 / M;
    static constexpr int RS = 17 * S;
};

// reverse 8-point DFT, natural order in and out
__device__ __forceinline__ void idft8(float2 (&z)[8])
{
    constexpr float R2 = 0.70710678118654752f;
    float2 e0 = z[0], e1 = z[2], e2 = z[4], e3 = z[6];
    float2 o0 = z[1], o1 = z[3], o2 = z[5], o3 = z[7];
    idft4(e0, e1, e2, e3);
    idft4(o0, o1, o2, o3);
    o1 = cmulc(o1, R2, R2);                 // W8^-1 = e^{+j pi/4}
    o2 = make_float2(-o2.y, o2.x);          // e^{+j pi/2}
    o3 = cmulc(o3, -R2, R2);                // e^{+j 3 pi/4}
    z[0] = f2add(e0, o0), z[4] = f2sub(e0, o0);
    z[1] = f2add(e1, o1), z[5] = f2sub(e1, o1);
    z[2] = f2add(e2, o2), z[6] = f2sub(e2, o2);
    z[3] = f2add(e3, o3), z[7] = f2sub(e3, o3);
}

// OS = 2, 4: oversampled bank, the same changes as pfb64_kernel (rows of D = M / OS samples, shifted U slots).
template <int M, int P4T, int OS = 1>
__global__ void __launch_bounds__(256, (M >= 128 ? 1 : 2))
    pfbm_kernel(const float2* __restrict__ x, const float2* __restrict__ halo, float2* __restrict__ out,
                const float* __restrict__ taps_rm /* [P4][M] */, int P4, int Ptrue, long long n_frames,
                long long n_in, int ch_begin, int ch_count, int tma_ok, int nbuf,
                int phase0 /* OS > 1: (frame index of out[0]) mod OS */)
{
    // nbuf = 2 (when shared memory allows, see b200_pfb_create): two input tiles, the copy of tile i+1 is issued a
    // whole tile ahead.  With one buffer it only had the DFT stage to hide behind: M = 128 (one CTA per SM) spent
    // 17 % of its warp samples on the input mbarrier (ncu, round 2).
    constexpr int S = pfbm<M>::S, TT = pfbm<M>::TT, RS = pfbm<M>::RS, D = M / OS;
    extern __shared__ __align__(128) float2 sm[];
    const int rows = TT + P4 * OS - 1;
    float2* X0 = sm;
    float2* U = X0 + nbuf * rows * D;
    float* hT = reinterpret_cast<float*>(U + TT * RS);
    uint64_t* bar = reinterpret_cast<uint64_t*>(hT + P4 * M);
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_mbar_init();
    }
    for (int i = tid; i < P4 * M; i += 256)
        hT[i] = __ldg(taps_rm + i);
    // stage-1 twiddles e^{+j 2 pi i0 c1 / M} of this thread (i0 = tid % S): register resident
    float2 twr[16];
#pragma unroll
    for (int c1 = 0; c1 < 16; c1++) {
        float sn, cs_;
        sincospif(2.0f * (float)(((tid % S) * c1) % M) / (float)M, &sn, &cs_);
        twr[c1] = make_float2(cs_, sn);
    }
    const long long nh = (long long)(Ptrue - 1) * M + (M - D); // P M - D samples of history
    const long long n_tiles = (n_frames + TT - 1) / TT;
    const uint32_t tile_bytes = (uint32_t)rows * (uint32_t)D * 8u;
    auto tma_tile = [&](long long t) {
        const long long g0 = (t * TT - (P4 * OS - 1)) * D;
        return tma_ok && g0 >= 0 && g0 + (long long)rows * D <= n_in;
    };
    __syncthreads();
    pdl_wait();              // programmatic dependent launch: everything above overlapped the previous kernel's tail
    pdl_launch_dependents();
    long long tile = blockIdx.x;
    if (tid == 0)
        for (int b = 0; b < nbuf; b++) {
            const long long t = tile + (long long)b * gridDim.x;
            if (t < n_tiles && tma_tile(t)) {
                mbar_arrive_expect_tx(bar + b, tile_bytes);
                bulk_copy_g2s(X0 + b * rows * D, x + (t * TT - (P4 * OS - 1)) * D, tile_bytes, bar + b);
            }
        }
    uint32_t phase = 0; // bit b: parity of the next completion of bar[b]
    for (int it = 0; tile < n_tiles; tile += gridDim.x, it++) {
        const long long f0 = tile * TT;
        const int xb = nbuf == 2 ? (it & 1) : 0;
        float2* X = X0 + xb * rows * D;
        if (tma_tile(tile)) {
            mbar_wait(bar + xb, (phase >> xb) & 1u);
            phase ^= 1u << xb;
        } else {
            const long long g0 = (f0 - (P4 * OS - 1)) * D;
            for (int i0 = tid; i0 < rows * D; i0 += 256 * 8) {
                float2 v[8];
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * D)
                        v[u] = pfb_fetch(x, halo, nh, g0 + i0 + u * 256, n_in);
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * D)
                        X[i0 + u * 256] = v[u];
            }
            __syncthreads();
        }
        // ---- branch filters: thread = (branch i, 16 consecutive frames)
        {
            const int i = tid % M, tg = tid / M;
            const int a = i / D, b = i % D; // branch i = a D + b: column D-1-b, rows shifted by OS-1-a (see pfb64_kernel)
            const float2* col = X + (D - 1 - b) + (tg * 16 + OS - 1 - a) * D;
            float2 acc[16];
#pragma unroll
            for (int j = 0; j < 16; j++)
                acc[j] = make_float2(0.f, 0.f);
            if (P4T > 0) {
                float hreg[P4T > 0 ? P4T : 1];
#pragma unroll
                for (int r = 0; r < P4T; r++)
                    hreg[r] = hT[r * M + i];
#pragma unroll
                for (int rho = 0; rho < 16 + (P4T - 1) * OS; rho++) {
                    const float2 v = col[rho * D];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const int r = P4T - 1 - (rho - j) / OS;
                        if ((rho - j) % OS == 0 && r >= 0 && r < P4T)
                            acc[j] = __ffma2_rn(v, make_float2(hreg[r], hreg[r]), acc[j]);
                    }
                }
            } else {
                for (int rc = 0; rc < P4; rc += 4) {
                    const float h0 = hT[(rc + 0) * M + i], h1 = hT[(rc + 1) * M + i];
                    const float h2 = hT[(rc + 2) * M + i], h3 = hT[(rc + 3) * M + i];
                    const float2* base = col + (P4 - 1 - rc - 3) * OS * D;
                    float2 w[16 + 3 * OS];
#pragma unroll
                    for (int q = 0; q < 16 + 3 * OS; q++)
                        w[q] = base[q * D];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        acc[j] = __ffma2_rn(w[j + 3 * OS], make_float2(h0, h0), acc[j]);
                        acc[j] = __ffma2_rn(w[j + 2 * OS], make_float2(h1, h1), acc[j]);
                        acc[j] = __ffma2_rn(w[j + OS], make_float2(h2, h2), acc[j]);
                        acc[j] = __ffma2_rn(w[j], make_float2(h3, h3), acc[j]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 16; j++) // circular shift of the branches: slot (i - t D) mod M
                U[(tg * 16 + j) * RS + (OS == 1 ? i : (i - (phase0 + j) * D) & (M - 1))] = acc[j];
        }
        __syncthreads(); // U complete; X fully consumed
        {
            const long long nxt = tile + (long long)nbuf * gridDim.x; // refill the buffer just consumed
            if (tid == 0 && nxt < n_tiles && tma_tile(nxt)) {
                mbar_arrive_expect_tx(bar + xb, tile_bytes);
                bulk_copy_g2s(X, x + (nxt * TT - (P4 * OS - 1)) * D, tile_bytes, bar + xb);
            }
        }
        // ---- stage 1: radix 16 over i1 (rows are warp-local: a warp owns 32/S whole frames)
        {
            const int t = tid / S, i0 = tid % S;
            float2* row = U + t * RS;
            float2 v[16];
#pragma unroll
            for (int i1 = 0; i1 < 16; i1++)
                v[i1] = row[S * i1 + i0];
            idft16(v); // A[c1] in v[4*(c1&3) + (c1>>2)]
            __syncwarp();
#pragma unroll
            for (int c1 = 0; c1 < 16; c1++) {
                const float2 a = v[4 * (c1 & 3) + (c1 >> 2)];
                row[17 * i0 + c1] = (S > 1 && c1 > 0) ? cmulc(a, twr[c1].x, twr[c1].y) : a;
            }
            __syncwarp();
        }
        const int lane = tid & 31, warp = tid >> 5;
        if (S == 1) {
            // M = 16: the row already is the frame's 16 channels; the warp stores its 32 frames
            // (4 KiB contiguous in the output) cooperatively
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const int idx = k * 32 + lane, fr = warp * 32 + (idx >> 4), ch = idx & 15;
                const long long f = f0 + fr;
                if (f < n_frames && ch >= ch_begin && ch < ch_begin + ch_count)
                    __stcs(out + f * ch_count - ch_begin + ch, U[fr * RS + ch]);
            }
        } else {
            // ---- stage 2: radix S over i0, thread = (frame, c1)
            constexpr int FW = 32 / S; // frames per warp
            const int c1 = lane & 15;
#pragma unroll
            for (int q = 0; q < FW / 2; q++) {
                const int fr = warp * FW + (lane >> 4) + 2 * q;
                const float2* row = U + fr * RS + c1;
                float2 z[S > 1 ? S : 2];
#pragma unroll
                for (int i0 = 0; i0 < S; i0++)
                    z[i0] = row[17 * i0];
                if constexpr (S == 2) {
                    const float2 a = f2add(z[0], z[1]), b = f2sub(z[0], z[1]);
                    z[0] = a, z[1] = b;
                } else if constexpr (S == 8) {
                    idft8(z);
                } else if constexpr (S == 16) {
                    idft16(z);
                }
                const long long f = f0 + fr;
                if (f < n_frames) {
                    float2* y = out + f * ch_count - ch_begin;
#pragma unroll
                    for (int c0 = 0; c0 < S; c0++) {
                        const int ch = c1 + 16 * c0;
                        const float2 r = (S == 16) ? z[4 * (c0 & 3) + (c0 >> 2)] : z[c0];
                        if (ch >= ch_begin && ch < ch_begin + ch_count)
                            __stcs(y + ch, r);
                    }
                }
            }
        }
        __syncthreads(); // U free for the next tile's branch filters
    }
}

// ---- M = 4, 8: same tiles and branch filters, the whole DFT in one thread --------------------------
// 4096-sample tiles (TT = 4096/M frames); the branch outputs go to shared memory branch-major
// (U[i][frame], row stride TT + 1), so the DFT thread of a frame reads its M values with lane-contiguous
// LDS.64 and writes the frame's M channels as 16-byte stores (neighbouring lanes = neighbouring frames:
// whole lines).
template <int M, int P4T>
__global__ void __launch_bounds__(256, 2)
    pfbs_kernel(const float2* __restrict__ x, const float2* __restrict__ halo, float2* __restrict__ out,
                const float* __restrict__ taps_rm /* [P4][M] */, int P4, int Ptrue, long long n_frames,
                long long n_in, int ch_begin, int ch_count, int tma_ok, int out16, int nbuf)
{
    // Shared-memory layout (round 2, from the ncu capture of M = 8: 30 M bank conflicts, mio_throttle 4.2 warps per
    // issue): a warp holds M branches x 32/M frame groups, and the groups' rows are 16 rows = a multiple of 128 bytes
    // apart, so the filter loads of the groups hit the same banks (4-way for M = 8, 8-way for M = 4).  One spare
    // row after every 16 rows of the input tile (the tile arrives as one bulk copy per 16-row block) and one spare
    // slot after every 16 frames of a branch's outputs (row stride = 2 mod 16) make filter loads, output stores
    // and the DFT's loads conflict-free.
    constexpr int TT = 4096 / M, US = TT + TT / 16 + 2;
    extern __shared__ __align__(128) float2 sm[];
    const int rows = TT + P4 - 1;
    const int prows = rows + (rows >> 4) + 1; // padded rows of one input tile
    float2* X0 = sm;
    float2* U = X0 + nbuf * prows * M;
    float* hT = reinterpret_cast<float*>(U + M * US);
    uint64_t* bar = reinterpret_cast<uint64_t*>(hT + P4 * M + ((P4 * M) & 1));
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_mbar_init();
    }
    for (int i = tid; i < P4 * M; i += 256)
        hT[i] = __ldg(taps_rm + i);
    const long long nh = (long long)(Ptrue - 1) * M;
    const long long n_tiles = (n_frames + TT - 1) / TT;
    const uint32_t tile_bytes = (uint32_t)rows * (uint32_t)M * 8u;
    auto tma_tile = [&](long long t) {
        const long long g0 = (t * TT - (P4 - 1)) * M;
        return tma_ok && g0 >= 0 && g0 + (long long)rows * M <= n_in;
    };
    __syncthreads();
    pdl_wait();              // programmatic dependent launch: everything above overlapped the previous kernel's tail
    pdl_launch_dependents();
    auto issue = [&](long long t, int b) { // one elected thread: one bulk copy per 16-row block, padded destination
        mbar_arrive_expect_tx(bar + b, tile_bytes);
        const float2* src = x + (t * TT - (P4 - 1)) * M;
        float2* dst = X0 + b * prows * M;
        for (int r = 0; r < rows; r += 16) {
            const int nr = rows - r < 16 ? rows - r : 16;
            bulk_copy_g2s(dst + (r + (r >> 4)) * M, src + r * M, (uint32_t)(nr * M * 8), bar + b);
        }
    };
    long long tile = blockIdx.x;
    if (tid == 0)
        for (int b = 0; b < nbuf; b++) {
            const long long t = tile + (long long)b * gridDim.x;
            if (t < n_tiles && tma_tile(t))
                issue(t, b);
        }
    uint32_t phase = 0; // bit b: parity of the next completion of bar[b]
    for (int it = 0; tile < n_tiles; tile += gridDim.x, it++) {
        const long long f0 = tile * TT;
        const int xb = nbuf == 2 ? (it & 1) : 0;
        float2* X = X0 + xb * prows * M;
        if (tma_tile(tile)) {
            mbar_wait(bar + xb, (phase >> xb) & 1u);
            phase ^= 1u << xb;
        } else {
            const long long g0 = (f0 - (P4 - 1)) * M;
            for (int i0 = tid; i0 < rows * M; i0 += 256 * 8) {
                float2 v[8];
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * M)
                        v[u] = pfb_fetch(x, halo, nh, g0 + i0 + u * 256, n_in);
#pragma unroll
                for (int u = 0; u < 8; u++)
                    if (i0 + u * 256 < rows * M) {
                        const int e = i0 + u * 256, r = e / M;
                        X[e + (r >> 4) * M] = v[u];
                    }
            }
            __syncthreads();
        }
        {
            const int i = tid % M, tg = tid / M; // 256 / M groups of 16 frames = TT frames
            const float2* col = X + (M - 1 - i) + (tg * 17) * M; // group tg starts at row 16 tg = padded row 17 tg
            float2 acc[16];
#pragma unroll
            for (int j = 0; j < 16; j++)
                acc[j] = make_float2(0.f, 0.f);
            if (P4T > 0) {
                float hreg[P4T > 0 ? P4T : 1];
#pragma unroll
                for (int r = 0; r < P4T; r++)
                    hreg[r] = hT[r * M + i];
#pragma unroll
                for (int rho = 0; rho < 16 + P4T - 1; rho++) {
                    const float2 v = col[(rho + (rho >> 4)) * M];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const int r = j + P4T - 1 - rho;
                        if (r >= 0 && r < P4T)
                            acc[j] = __ffma2_rn(v, make_float2(hreg[r], hreg[r]), acc[j]);
                    }
                }
            } else {
                for (int rc = 0; rc < P4; rc += 4) {
                    const float h0 = hT[(rc + 0) * M + i], h1 = hT[(rc + 1) * M + i];
                    const float h2 = hT[(rc + 2) * M + i], h3 = hT[(rc + 3) * M + i];
                    const int a0 = P4 - 1 - rc - 3;
                    float2 w[19];
#pragma unroll
                    for (int q = 0; q < 19; q++)
                        w[q] = col[(a0 + q + ((a0 + q) >> 4)) * M];
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        acc[j] = __ffma2_rn(w[j + 3], make_float2(h0, h0), acc[j]);
                        acc[j] = __ffma2_rn(w[j + 2], make_float2(h1, h1), acc[j]);
                        acc[j] = __ffma2_rn(w[j + 1], make_float2(h2, h2), acc[j]);
                        acc[j] = __ffma2_rn(w[j], make_float2(h3, h3), acc[j]);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 16; j++)
                U[i * US + tg * 17 + j] = acc[j];
        }
        __syncthreads(); // U complete; X fully consumed
        {
            const long long nxt = tile + (long long)nbuf * gridDim.x; // refill the buffer just consumed
            if (tid == 0 && nxt < n_tiles && tma_tile(nxt))
                issue(nxt, xb);
        }
#pragma unroll 1
        for (int fr = tid; fr < TT; fr += 256) {
            float2 z[M];
#pragma unroll
            for (int i = 0; i < M; i++)
                z[i] = U[i * US + fr + (fr >> 4)];
            if constexpr (M == 8)
                idft8(z);
            else
                idft4(z[0], z[1], z[2], z[3]);
            const long long f = f0 + fr;
            if (f < n_frames) {
                if (out16 && ch_begin == 0 && ch_count == M) {
                    float4* y = reinterpret_cast<float4*>(out + f * M);
#pragma unroll
                    for (int c = 0; c < M; c += 2)
                        __stcs(y + c / 2, make_float4(z[c].x, z[c].y, z[c + 1].x, z[c + 1].y));
                } else {
                    float2* y = out + f * ch_count - ch_begin;
#pragma unroll
                    for (int c = 0; c < M; c++)
                        if (c >= ch_begin && c < ch_begin + ch_count)
                            __stcs(y + c, z[c]);
                }
            }
        }
        __syncthreads(); // U free for the next tile's branch filters
    }
}

// generic M (power of two, 4..256): straightforward shared-memory version
__global__ void __launch_bounds__(256)
    pfb_generic_kernel(const float2* __restrict__ x, const float2* __restrict__ halo,
                       float2* __restrict__ out, const float* __restrict__ taps /* [P][M] */, int M,
                       int P, int TT, long long n_frames, long long n_in, int ch_begin, int ch_count,
                       float2* __restrict__ u_out /* != NULL: write the branch outputs [t][i], skip the DFT */,
                       long long frame_offset)
{
    extern __shared__ __align__(16) float2 sm[];
    const int rows = TT + P - 1;
    float2* X = sm;
    float2* U = X + rows * M;
    float2* tw = U + TT * M;
    const int tid = threadIdx.x;
    for (int i = tid; i < M; i += blockDim.x) {
        float s, c;
        sincospif(2.0f * (float)i / (float)M, &s, &c);
        tw[i] = make_float2(c, s);
    }
    const long long nh = (long long)(P - 1) * M;
    const long long f0 = frame_offset + (long long)blockIdx.x * TT;
    const long long g0 = (f0 - (P - 1)) * M;
    for (int i0 = tid; i0 < rows * M; i0 += blockDim.x * 8) { // 8 independent loads in flight
        float2 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u * (int)blockDim.x < rows * M)
                v[u] = pfb_fetch(x, halo, nh, g0 + i0 + u * (int)blockDim.x, n_in);
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u * (int)blockDim.x < rows * M)
                X[i0 + u * (int)blockDim.x] = v[u];
    }
    float* hS = reinterpret_cast<float*>(tw + M); // taps [P][M] staged once per CTA
    for (int i = tid; i < P * M; i += blockDim.x)
        hS[i] = __ldg(taps + i);
    __syncthreads();
    for (int e = tid; e < TT * M; e += blockDim.x) {
        int t = e / M, i = e - t * M;
        float2 a = make_float2(0.f, 0.f);
        for (int r = 0; r < P; r++) {
            float h = hS[r * M + i];
            float2 v = X[(t + P - 1 - r) * M + (M - 1 - i)];
            a = __ffma2_rn(v, make_float2(h, h), a);
        }
        if (u_out) {
            if (f0 + t < n_frames)
                u_out[((long long)blockIdx.x * TT + t) * M + i] = a; // coalesced across i
        } else {
            U[e] = a;
        }
    }
    if (u_out)
        return;
    __syncthreads();
    for (int e = tid; e < TT * ch_count; e += blockDim.x) {
        int t = e / ch_count, cc = e - t * ch_count;
        int c = cc + ch_begin;
        long long f = f0 + t;
        if (f >= n_frames)
            continue;
        float2 a = make_float2(0.f, 0.f);
        for (int i = 0; i < M; i++) {
            float2 w = tw[(i * c) & (M - 1)];
            float2 u = U[t * M + i];
            a.x += u.x * w.x - u.y * w.y;
            a.y += u.x * w.y + u.y * w.x;
        }
        out[f * ch_count + cc] = a;
    }
}

// out[t][c - ch_begin] = full[t][c] for a channel slice of the FFT-based generic path
__global__ void pfb_slice_kernel(const float2* __restrict__ full, float2* __restrict__ out, long long n_frames,
                                 int M, int ch_begin, int ch_count)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_frames * ch_count)
        return;
    long long t = e / ch_count;
    int c = (int)(e - t * ch_count);
    out[e] = full[t * M + ch_begin + c];
}

// new_tail[j] = sample (n_consumed - nh + j) of (old tail ++ x), complex64
__global__ void pfb_tail_kernel(const float2* __restrict__ x, const float2* __restrict__ old_tail,
                                float2* __restrict__ new_tail, long long n_consumed, long long nh)
{
    long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nh)
        return;
    long long s = n_consumed - nh + j;
    new_tail[j] = (s >= 0) ? x[s] : old_tail[nh + s];
}

} // namespace b200

using namespace b200;

// auto-selection of the M = 64 form: 0 = SIMT DFT, 1 = tensor-core DFT (set from the measured A/B, DESIGN.md 4.4)
#ifndef PFB64_TC_DEFAULT
#define PFB64_TC_DEFAULT 0
#endif

// MaxDynamicSharedMemorySize of every channelizer kernel: the most a block may have on sm_100.  The attribute belongs
// to the kernel, and handles with different shared-memory sizes share an instantiation (pfb64_kernel<0> at P = 20
// and 28, every pfb_generic_kernel handle, ...): a per-handle value set by the last b200_pfb_create would make the
// launches of an older, larger handle fail.  Each launch passes its own h->smem, which the create-time checks keep
// within 220 KiB (227 KiB for the two-tile pfbm_kernel).
constexpr int PFB_SMEM_ATTR = 227 * 1024;

// shared memory of pfbs_kernel: one (padded) input tile, and everything else
static inline size_t pfbs_xbytes(int M, int P4)
{
    const int rows = 4096 / M + P4 - 1;
    return sizeof(float2) * (size_t)(rows + (rows >> 4) + 1) * M;
}
static inline size_t pfbs_rest(int M, int P4)
{
    const int TT = 4096 / M;
    return sizeof(float2) * (size_t)M * (TT + TT / 16 + 2) + sizeof(float) * ((size_t)P4 * M + 1) + 32;
}

// shared memory of the single-pass M = 16 .. 256 kernels (pfb64_kernel, pfbm_kernel) with `nbuf` input tiles of
// TT + P4 os - 1 rows of D = M / os samples (TT = 4096 / M frames)
static inline size_t pfb_single_pass_smem(int M, int P4, int os, int nbuf)
{
    const int TT = 4096 / M;
    const size_t xbytes = sizeof(float2) * (size_t)(TT + P4 * os - 1) * (M / os);
    if (M == 64) {
        const bool regtaps = P4 == 4 || P4 == 8 || P4 == 12 || P4 == 16 || P4 == 24 || P4 == 32;
        return nbuf * xbytes + sizeof(float2) * (size_t)PFB64_TT * PFB64_RS + (regtaps ? 0 : sizeof(float) * (size_t)P4 * 64);
    }
    return nbuf * xbytes + sizeof(float2) * (size_t)TT * 17 * (M / 16) + sizeof(float) * (size_t)P4 * M + 16;
}

static inline uint16_t pfb_bf16_rn(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static inline float pfb_bf16_f(uint16_t b)
{
    const uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}

struct b200_pfb {
    int M = 0, P = 0, P4 = 0;
    int ch_begin = 0, ch_count = 0;
    float* d_taps_rm = nullptr; // [P4][M], zero padded rows
    float2* d_tail[2] = { nullptr, nullptr };
    int cur = 0;
    size_t smem = 0;
    int TT = 0;
    int grid = 296;
    int tc = 0;            // M = 64: 1 = DFT across branches on the tensor cores (pfb64_tc_kernel), 0 = SIMT DFT
    int tc_ok = 0;         // the tensor-core form exists for this (M, P)
    uint4* d_dft = nullptr; // [128 rows = (channel, re/im)][hi 128 | lo 128] bf16 DFT matrix
    size_t smem_tc = 0;
    int tc_mn = 1;         // pfb64_tc_kernel: branch outputs stored MN-major (16-byte stores), DFT matrix with planar K
    int nbuf = 1;          // input tiles in shared memory (pfbm_kernel)
    int fusedM = 0; // 1: M = 16 / 32 / 128 / 256 on pfbm_kernel; 2: M = 4 / 8 on pfbs_kernel (single pass both)
    int os = 1;            // oversample rate: one frame per D = M / os input samples
    int D = 0;
    int phase = 0;         // frames produced since creation or the last reset, mod os (the branch rotation)
    // generic M >= 16: branch filters -> scratch -> the library's own reverse FFT of length M
    b200_fft* ifft = nullptr;
    float2* d_u = nullptr;    // [chunk_frames][M] branch outputs
    float2* d_full = nullptr; // [chunk_frames][M] FFT output when a channel slice is requested
    long long chunk_frames = 0;
};

static int pfb_launch(b200_pfb* h, const void* d_halo, const void* d_in, void* d_out,
                      long long n_in, long long n_frames, int phase0, cudaStream_t s)
{
    if (n_frames <= 0)
        return B200_OK;
    if (h->M == 64 && h->tc) {
        long long tiles = (n_frames + PFB64_TT - 1) / PFB64_TT;
        long long g = tiles < h->grid ? tiles : h->grid;
#define PFBT_GO(PT)                                                                               \
    B200_LAUNCH_PDL(pfb64_tc_kernel<PT>, (unsigned)g, PFBT_THREADS, h->smem_tc, s, (const float2*)d_in,           \
                (const float2*)d_halo, (float2*)d_out, h->d_taps_rm, h->d_dft, h->P4, h->P, n_frames, \
                n_in, h->ch_begin, h->ch_count, (int)((uintptr_t)d_in % 16 == 0), h->tc_mn)
        switch (h->P4) {
        case 4: PFBT_GO(4); break;
        case 8: PFBT_GO(8); break;
        case 12: PFBT_GO(12); break;
        default: PFBT_GO(16); break;
        }
#undef PFBT_GO
    } else if (h->M == 64) {
        long long tiles = (n_frames + PFB64_TT - 1) / PFB64_TT;
        long long g = tiles < h->grid ? tiles : h->grid;
#define PFB64_GO(PT, OS)                                                                          \
    B200_LAUNCH_PDL((pfb64_kernel<PT, OS>), (unsigned)g, 256, h->smem, s, (const float2*)d_in,            \
                (const float2*)d_halo, (float2*)d_out, h->d_taps_rm, h->P4, h->P, n_frames, n_in,     \
                h->ch_begin, h->ch_count, (int)((uintptr_t)d_in % 16 == 0), h->nbuf, phase0)
#define PFB64_P(OS)                    \
    switch (h->P4) {                   \
    case 4: PFB64_GO(4, OS); break;    \
    case 8: PFB64_GO(8, OS); break;    \
    case 12: PFB64_GO(12, OS); break;  \
    case 16: PFB64_GO(16, OS); break;  \
    case 24: PFB64_GO(24, OS); break;  \
    case 32: PFB64_GO(32, OS); break;  \
    default: PFB64_GO(0, OS); break;   \
    }
        switch (h->os) {
        case 2: PFB64_P(2); break;
        case 4: PFB64_P(4); break;
        default: PFB64_P(1); break;
        }
#undef PFB64_P
#undef PFB64_GO
    } else if (h->fusedM == 2) {
        const int TT = 4096 / h->M;
        long long tiles = (n_frames + TT - 1) / TT;
        long long g = tiles < h->grid ? tiles : h->grid;
#define PFBS_GO(MM, PT)                                                                               \
    B200_LAUNCH_PDL((pfbs_kernel<MM, PT>), (unsigned)g, 256, h->smem, s, (const float2*)d_in,             \
                (const float2*)d_halo, (float2*)d_out, h->d_taps_rm, h->P4, h->P, n_frames, n_in,     \
                h->ch_begin, h->ch_count, (int)((uintptr_t)d_in % 16 == 0), (int)((uintptr_t)d_out % 16 == 0), h->nbuf)
        if (h->M == 8) {
            switch (h->P4) {
            case 4: PFBS_GO(8, 4); break;
            case 8: PFBS_GO(8, 8); break;
            case 16: PFBS_GO(8, 16); break;
            default: PFBS_GO(8, 0); break;
            }
        } else {
            switch (h->P4) {
            case 4: PFBS_GO(4, 4); break;
            case 8: PFBS_GO(4, 8); break;
            case 16: PFBS_GO(4, 16); break;
            default: PFBS_GO(4, 0); break;
            }
        }
#undef PFBS_GO
    } else if (h->fusedM) {
        const int TT = 4096 / h->M;
        long long tiles = (n_frames + TT - 1) / TT;
        long long g = tiles < h->grid ? tiles : h->grid;
#define PFBM_GO(MM, PT, OS)                                                                           \
    B200_LAUNCH_PDL((pfbm_kernel<MM, PT, OS>), (unsigned)g, 256, h->smem, s, (const float2*)d_in,         \
                (const float2*)d_halo, (float2*)d_out, h->d_taps_rm, h->P4, h->P, n_frames, n_in,     \
                h->ch_begin, h->ch_count, (int)((uintptr_t)d_in % 16 == 0), h->nbuf, phase0)
#define PFBM_P(MM, OS)                     \
    switch (h->P4) {                       \
    case 4: PFBM_GO(MM, 4, OS); break;     \
    case 8: PFBM_GO(MM, 8, OS); break;     \
    case 16: PFBM_GO(MM, 16, OS); break;   \
    default: PFBM_GO(MM, 0, OS); break;    \
    }
#define PFBM_OS(MM)                        \
    switch (h->os) {                       \
    case 2: PFBM_P(MM, 2); break;          \
    case 4: PFBM_P(MM, 4); break;          \
    default: PFBM_P(MM, 1); break;         \
    }
        switch (h->M) {
        case 16: PFBM_OS(16); break;
        case 32: PFBM_OS(32); break;
        case 128: PFBM_OS(128); break;
        default: PFBM_OS(256); break;
        }
#undef PFBM_OS
#undef PFBM_P
#undef PFBM_GO
    } else if (h->ifft) {
        // branch filters into a scratch tile, then the M-point reverse FFT of fft.cu; chunked so the
        // scratch allocated at create time is enough for any call
        const bool slice = h->ch_count != h->M;
        for (long long f0 = 0; f0 < n_frames; f0 += h->chunk_frames) {
            const long long nf = std::min(h->chunk_frames, n_frames - f0);
            const long long tiles = (nf + h->TT - 1) / h->TT;
            B200_LAUNCH(pfb_generic_kernel, (unsigned)tiles, 256, h->smem, s, (const float2*)d_in,
                        (const float2*)d_halo, (float2*)nullptr, h->d_taps_rm, h->M, h->P, h->TT, n_frames,
                        n_in, h->ch_begin, h->ch_count, h->d_u, f0);
            float2* dst = slice ? h->d_full : (float2*)d_out + f0 * h->M;
            int rc = b200_fft_run(h->ifft, h->d_u, dst, nf, reinterpret_cast<b200_stream_t>(s));
            if (rc != B200_OK)
                return rc;
            if (slice) {
                const long long tot = nf * h->ch_count;
                B200_LAUNCH(pfb_slice_kernel, (unsigned)((tot + 255) / 256), 256, 0, s, h->d_full,
                            (float2*)d_out + f0 * h->ch_count, nf, h->M, h->ch_begin, h->ch_count);
            }
        }
    } else {
        long long tiles = (n_frames + h->TT - 1) / h->TT;
        if (tiles > 0x7fffffffLL)
            return set_err(B200_ERR_ARG, "pfb: too many items for one call");
        B200_LAUNCH(pfb_generic_kernel, (unsigned)tiles, 256, h->smem, s, (const float2*)d_in,
                    (const float2*)d_halo, (float2*)d_out, h->d_taps_rm, h->M, h->P, h->TT, n_frames,
                    n_in, h->ch_begin, h->ch_count, (float2*)nullptr, 0LL);
    }
    return B200_OK;
}

extern "C" {

int b200_pfb_destroy(b200_pfb* h)
{
    if (!h)
        return B200_OK;
    cudaFree(h->d_taps_rm);
    cudaFree(h->d_tail[0]);
    cudaFree(h->d_tail[1]);
    cudaFree(h->d_u);
    cudaFree(h->d_full);
    cudaFree(h->d_dft);
    b200_fft_destroy(h->ifft);
    delete h;
    return B200_OK;
}

int b200_pfb_create(const b200_pfb_params* p, b200_pfb** out)
{
    if (!p || !out)
        return set_err(B200_ERR_ARG, "pfb_create: null argument");
    *out = nullptr;
    const int M = p->n_channels, P = p->taps_per_channel;
    if (!p->taps || M < 4 || M > 256 || (M & (M - 1)) || P < 1)
        return set_err(B200_ERR_ARG, "pfb_create: need M power of two in [4,256], P >= 1, taps != NULL");
    int cb = p->channel_begin, cc = p->channel_count ? p->channel_count : M - p->channel_begin;
    if (cb < 0 || cc < 1 || cb + cc > M)
        return set_err(B200_ERR_ARG, "pfb_create: bad channel slice [%d, %d)", cb, cb + cc);
    const int os = p->oversample ? p->oversample : 1;
    if (os != 1 && os != 2 && os != 4)
        return set_err(B200_ERR_ARG, "pfb_create: oversample %d: need 0 or 1 (critically sampled), 2 or 4", p->oversample);
    if (os > 1) {
        // the oversampled bank exists on the single-pass kernels of M = 16 .. 256 only
        if (M < 16)
            return set_err(B200_ERR_UNSUPPORTED, "pfb_create: oversample %d needs 16, 32, 64, 128 or 256 channels, not %d", os, M);
        if (getenv("B200_PFB_TWOPASS"))
            return set_err(B200_ERR_UNSUPPORTED, "pfb_create: oversample %d runs on the single-pass kernels only, and B200_PFB_TWOPASS is set", os);
        const int P4 = (P + 3) / 4 * 4;
        if (pfb_single_pass_smem(M, P4, os, 1) > 220 * 1024) {
            int pmax = 0;
            while (pfb_single_pass_smem(M, pmax + 4, os, 1) <= 220 * 1024)
                pmax += 4;
            return set_err(B200_ERR_UNSUPPORTED, "pfb_create: taps_per_channel %d too large for oversample %d at M=%d: at most %d", P,
                           os, M, pmax);
        }
    }
    b200_pfb* h = new b200_pfb();
    h->os = os;
    h->D = M / os;
    h->M = M;
    h->P = P;
    h->P4 = (P + 3) / 4 * 4;
    h->ch_begin = cb;
    h->ch_count = cc;
#define PFB_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            b200_pfb_destroy(h);                                                         \
            return set_err(e__ == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA, \
                           "pfb_create: %s -> %s", #call, cudaGetErrorString(e__));      \
        }                                                                                \
    } while (0)
    std::vector<float> rm((size_t)h->P4 * M, 0.f);
    for (int r = 0; r < P; r++)
        for (int i = 0; i < M; i++)
            rm[(size_t)r * M + i] = p->taps[i + r * M];
    PFB_CUDA(cudaMalloc(&h->d_taps_rm, rm.size() * sizeof(float)));
    PFB_CUDA(cudaMemcpy(h->d_taps_rm, rm.data(), rm.size() * sizeof(float), cudaMemcpyHostToDevice));
    size_t nh = (size_t)P * M - h->D;
    for (int i = 0; i < 2; i++) {
        PFB_CUDA(cudaMalloc(&h->d_tail[i], sizeof(float2) * (nh ? nh : 1)));
        PFB_CUDA(cudaMemset(h->d_tail[i], 0, sizeof(float2) * (nh ? nh : 1)));
    }
    if (M == 64) {
        int rows = PFB64_TT + h->P4 * os - 1;
        const bool regtaps = h->P4 == 4 || h->P4 == 8 || h->P4 == 12 || h->P4 == 16 || h->P4 == 24 || h->P4 == 32;
        const size_t xb64 = sizeof(float2) * (size_t)rows * h->D, u64 = sizeof(float2) * (size_t)PFB64_TT * PFB64_RS;
        const size_t taps64 = regtaps ? 0 : sizeof(float) * (size_t)h->P4 * 64;
        // second input tile when two CTAs per SM still fit: (233472 - 2 * 1024) / 2 = 115712 bytes per CTA
        // ... and only for 16 taps per channel: the shorter (HBM-bound) filters LOSE with the deeper read prefetch
        // (P = 8: 413 -> 353 GS/s, P = 12: 400 -> 374), P = 16 gains 1.5 % (372.6 -> 378.3)
        // oversampled: B200_PFB_TWOBUF asks for two tiles at any P4 with taps in registers (the A/B of DESIGN.md 4.4e)
        h->nbuf = (regtaps && (h->P4 == 16 || (os > 1 && getenv("B200_PFB_TWOBUF"))) && 2 * xb64 + u64 <= 115712 &&
                   !getenv("B200_PFB_ONEBUF")) ? 2 : 1;
        h->smem = h->nbuf * xb64 + u64 + taps64;
        if (h->smem > 220 * 1024) {
            b200_pfb_destroy(h);
            return set_err(B200_ERR_UNSUPPORTED, "pfb_create: taps_per_channel too large for M=64 tile");
        }
#define PFB64_ATTR(OS)                                                                                              \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<0, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));  \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<4, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));  \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<8, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));  \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<12, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<16, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<24, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfb64_kernel<32, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR))
        if (os == 2) {
            PFB64_ATTR(2);
        } else if (os == 4) {
            PFB64_ATTR(4);
        } else {
            PFB64_ATTR(1);
        }
#undef PFB64_ATTR
        h->grid = 2 * sm_count();
        if (h->P4 <= 16 && os == 1) { // the tensor-core form exists for the critically sampled bank only
            // tensor-core DFT form: DFT matrix rows m = 2c + part; columns k = 2i + (re | im) for the K-major planes,
            // k = i (re) / 64 + i (im) for the MN-major ones; bf16 hi | lo
            h->tc_mn = 1;
            if (const char* e = getenv("B200_PFBT_MN"))
                h->tc_mn = atoi(e) != 0;
            std::vector<uint16_t> F((size_t)128 * 256);
            for (int m = 0; m < 128; m++)
                for (int k = 0; k < 128; k++) {
                    const int c = m >> 1, po = m & 1, i = h->tc_mn ? (k & 63) : (k >> 1), pi = h->tc_mn ? (k >> 6) : (k & 1);
                    const double th = 2.0 * M_PI * (double)((i * c) & 63) / 64.0;
                    const double v = po == pi ? std::cos(th) : (po ? std::sin(th) : -std::sin(th));
                    const float f = (float)v;
                    const uint16_t hi = pfb_bf16_rn(f);
                    F[(size_t)m * 256 + k] = hi;
                    F[(size_t)m * 256 + 128 + k] = pfb_bf16_rn(f - pfb_bf16_f(hi));
                }
            PFB_CUDA(cudaMalloc(&h->d_dft, F.size() * 2));
            PFB_CUDA(cudaMemcpy(h->d_dft, F.data(), F.size() * 2, cudaMemcpyHostToDevice));
            h->smem_tc = 1024 + 2 * (size_t)PFBT_PLANE + 2 * sizeof(float2) * (size_t)rows * 64 + 64;
            PFB_CUDA(cudaFuncSetAttribute(pfb64_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));
            PFB_CUDA(cudaFuncSetAttribute(pfb64_tc_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));
            PFB_CUDA(cudaFuncSetAttribute(pfb64_tc_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));
            PFB_CUDA(cudaFuncSetAttribute(pfb64_tc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));
            h->tc_ok = 1;
            h->tc = PFB64_TC_DEFAULT;
            if (const char* e = getenv("B200_PFB_TC"))
                h->tc = atoi(e) != 0;
        }
    } else if ((M == 4 || M == 8) && !getenv("B200_PFB_TWOPASS") &&
               pfbs_xbytes(M, h->P4) + pfbs_rest(M, h->P4) <= 110 * 1024) {
        h->fusedM = 2;
        h->nbuf = (2 * pfbs_xbytes(M, h->P4) + pfbs_rest(M, h->P4) <= 113 * 1024 && !getenv("B200_PFB_ONEBUF")) ? 2 : 1;
        h->smem = h->nbuf * pfbs_xbytes(M, h->P4) + pfbs_rest(M, h->P4);
#define PFBS_ATTR(MM)                                                                                          \
    PFB_CUDA(cudaFuncSetAttribute(pfbs_kernel<MM, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbs_kernel<MM, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbs_kernel<MM, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbs_kernel<MM, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR))
        if (M == 8) {
            PFBS_ATTR(8);
        } else {
            PFBS_ATTR(4);
        }
#undef PFBS_ATTR
        h->grid = 2 * sm_count();
    } else if ((M == 16 || M == 32 || M == 128 || M == 256) && !getenv("B200_PFB_TWOPASS") &&
               pfb_single_pass_smem(M, h->P4, os, 1) <= 220 * 1024) {
        h->fusedM = 1;
        const size_t xbytes = sizeof(float2) * (size_t)(4096 / M + h->P4 * os - 1) * h->D;
        const size_t rest = sizeof(float2) * (size_t)(4096 / M) * 17 * (M / 16) + sizeof(float) * (size_t)h->P4 * M + 16;
        // a second input tile for M >= 128 (one CTA per SM: 321 -> 391 GS/s at M = 128 / P = 8, 335 -> 411 at M = 256 /
        // P = 4).  M = 16 / 32 run two CTAs per SM and LOSE with it (M = 16 / P = 8: 399 -> 345 GS/s; the deeper read
        // prefetch works against the write stream of these HBM-bound kernels), so they keep one.
        // oversampled: B200_PFB_TWOBUF asks for two tiles at M = 16 / 32 too while two CTAs per SM still fit
        h->nbuf = ((M >= 128 || (os > 1 && getenv("B200_PFB_TWOBUF") && 2 * xbytes + rest <= 115712)) &&
                   2 * xbytes + rest <= 227 * 1024 && !getenv("B200_PFB_ONEBUF")) ? 2 : 1;
        h->smem = h->nbuf * xbytes + rest;
#define PFBM_ATTR(MM, OS)                                                                                          \
    PFB_CUDA(cudaFuncSetAttribute(pfbm_kernel<MM, 0, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbm_kernel<MM, 4, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbm_kernel<MM, 8, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR)); \
    PFB_CUDA(cudaFuncSetAttribute(pfbm_kernel<MM, 16, OS>, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR))
#define PFBM_ATTR_OS(MM)  \
    if (os == 2) {        \
        PFBM_ATTR(MM, 2); \
    } else if (os == 4) { \
        PFBM_ATTR(MM, 4); \
    } else {              \
        PFBM_ATTR(MM, 1); \
    }
        if (M == 16) {
            PFBM_ATTR_OS(16);
        } else if (M == 32) {
            PFBM_ATTR_OS(32);
        } else if (M == 128) {
            PFBM_ATTR_OS(128);
        } else {
            PFBM_ATTR_OS(256);
        }
#undef PFBM_ATTR_OS
#undef PFBM_ATTR
        h->grid = (M >= 128 ? 1 : 2) * sm_count();
    } else {
        h->TT = 4096 / M;
        if (h->TT < 1)
            h->TT = 1;
        h->smem = sizeof(float2) * ((size_t)(h->TT + P - 1) * M + (size_t)h->TT * M + M) +
                  sizeof(float) * (size_t)P * M;
        if (h->smem > 220 * 1024) {
            b200_pfb_destroy(h);
            return set_err(B200_ERR_UNSUPPORTED, "pfb_create: taps_per_channel too large");
        }
        PFB_CUDA(cudaFuncSetAttribute(pfb_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PFB_SMEM_ATTR));
        if (M >= 16) {
            b200_fft_params fp{};
            fp.n = M;
            fp.forward = 0; // e^{+j}: the channelizer applies an un-normalised reverse DFT across branches
            fp.output = B200_FFT_OUT_COMPLEX;
            if (b200_fft_create(&fp, &h->ifft) != B200_OK) {
                b200_pfb_destroy(h);
                return B200_ERR_CUDA;
            }
            h->chunk_frames = (32ll << 20) / (8ll * M) / h->TT * h->TT; // 32 MiB of branch outputs
            PFB_CUDA(cudaMalloc(&h->d_u, sizeof(float2) * (size_t)h->chunk_frames * M));
            if (h->ch_count != M)
                PFB_CUDA(cudaMalloc(&h->d_full, sizeof(float2) * (size_t)h->chunk_frames * M));
        }
    }
#undef PFB_CUDA
    // the uploads above went through the legacy default stream (cudaMemcpy / cudaMemset); the caller's streams are
    // non-blocking and not ordered against it, so finish them before the handle can be used
    if (cudaDeviceSynchronize() != cudaSuccess) {
        b200_pfb_destroy(h);
        return set_err(B200_ERR_CUDA, "pfb_create: %s", cudaGetErrorString(cudaGetLastError()));
    }
    *out = h;
    return B200_OK;
}

int b200_pfb_run(b200_pfb* h, const void* d_in, void* d_out, int64_t n_in_items,
                 int64_t* n_consumed, int64_t* n_produced_vectors, b200_stream_t s)
{
    if (!h || n_in_items < 0 || (n_in_items > 0 && !d_in) || (n_in_items >= h->D && !d_out))
        return set_err(B200_ERR_ARG, "pfb_run: bad argument");
    long long n_frames = n_in_items / h->D;
    long long n_cons = n_frames * h->D;
    int rc = pfb_launch(h, h->d_tail[h->cur], d_in, d_out, n_in_items, n_frames, h->phase, cs(s));
    if (rc != B200_OK)
        return rc;
    h->phase = (int)((h->phase + n_frames) % h->os);
    long long nh = (long long)h->P * h->M - h->D;
    if (nh > 0 && n_cons > 0) {
        B200_LAUNCH(pfb_tail_kernel, (unsigned)((nh + 255) / 256), 256, 0, cs(s), (const float2*)d_in,
                    h->d_tail[h->cur], h->d_tail[h->cur ^ 1], n_cons, nh);
        h->cur ^= 1;
    }
    if (n_consumed)
        *n_consumed = n_cons;
    if (n_produced_vectors)
        *n_produced_vectors = n_frames;
    return B200_OK;
}

int b200_pfb_run_segment(b200_pfb* h, const void* d_halo, const void* d_in, void* d_out,
                         int64_t n_in_items, int64_t* n_produced_vectors, b200_stream_t s)
{
    if (!h || n_in_items < 0 || (n_in_items > 0 && !d_in) || (n_in_items >= h->D && !d_out))
        return set_err(B200_ERR_ARG, "pfb_run_segment: bad argument");
    long long n_frames = n_in_items / h->D;
    int rc = pfb_launch(h, d_halo, d_in, d_out, n_in_items, n_frames, 0, cs(s)); // d_in[0] starts frame phase 0
    if (rc == B200_OK && n_produced_vectors)
        *n_produced_vectors = n_frames;
    return rc;
}

int b200_pfb_set_algorithm(b200_pfb* h, int32_t algorithm)
{
    if (!h)
        return set_err(B200_ERR_ARG, "pfb_set_algorithm: null handle");
    if (algorithm < 0 || algorithm > 2)
        return set_err(B200_ERR_ARG, "pfb_set_algorithm: algorithm must be 0 (auto), 1 (SIMT DFT) or 2 (tensor-core DFT)");
    if (algorithm == 2 && h->os > 1)
        return set_err(B200_ERR_UNSUPPORTED, "pfb_set_algorithm: the tensor-core DFT form needs oversample 1 (this handle: %d); "
                       "oversampled banks run algorithm 0 or 1", h->os);
    if (algorithm == 2 && !h->tc_ok)
        return set_err(B200_ERR_UNSUPPORTED, "pfb_set_algorithm: the tensor-core DFT form needs 64 channels and <= 16 taps per channel");
    h->tc = algorithm == 2 ? 1 : algorithm == 1 ? 0 : (h->tc_ok ? PFB64_TC_DEFAULT : 0);
    return B200_OK;
}

int b200_pfb_get_algorithm(const b200_pfb* h, int32_t* algorithm)
{
    if (!h || !algorithm)
        return set_err(B200_ERR_ARG, "pfb_get_algorithm: null argument");
    *algorithm = h->tc ? 2 : 1;
    return B200_OK;
}

int b200_pfb_get_oversample(const b200_pfb* h, int32_t* oversample)
{
    if (!h || !oversample)
        return set_err(B200_ERR_ARG, "pfb_get_oversample: null argument");
    *oversample = h->os;
    return B200_OK;
}

int b200_pfb_geometry(const b200_pfb* h, int* n_channels, int* channel_count)
{
    if (!h)
        return set_err(B200_ERR_ARG, "pfb_geometry: null handle");
    if (n_channels)
        *n_channels = h->M;
    if (channel_count)
        *channel_count = h->ch_count;
    return B200_OK;
}

int b200_pfb_reset(b200_pfb* h, b200_stream_t s)
{
    if (!h)
        return set_err(B200_ERR_ARG, "pfb_reset: null handle");
    size_t nh = (size_t)h->P * h->M - h->D;
    B200_CUDA(cudaMemsetAsync(h->d_tail[h->cur], 0, sizeof(float2) * (nh ? nh : 1), cs(s)));
    h->phase = 0;
    return B200_OK;
}

} // extern "C"

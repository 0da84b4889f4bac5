// fir_tc.cu -- ccf FIR as a block-Toeplitz GEMM on the 5th-generation tensor cores (algorithm 2).
//
//   y[m] = sum_{k<T} h[k] x[m*D - k]          (SURVEY.md 8c; real taps, complex stream)
//
// The reference snapshot has no FIR block and no tensor-core code at all (SURVEY.md 0.1, 2.2); the
// block interface this stands behind is gr::block::work, runtime/include/gnuradio/block.hpp:81-85.
// BASELINE.json north_star: "long-tap FIR expressed as Toeplitz/polyphase GEMM".
//
// Formulation.  Real taps act on the real and the imaginary stream separately, so a tile of outputs
// is two real problems (planes "re" and "im").  Write an output index in the tile as m = 64 r + c
// (r = 0..127, c = 0..63) and, per polyphase branch p (h_p[q] = h[qD+p], x_p[j] = x[jD-p]),
//
//     Y[c][r] = sum_j  A_p[c][j] * X_p[r][j],   A_p[c][j] = h_p[c + P - j],   X_p[r][j] = xs_p[64 r + j]
//
// with xs_p the branch's samples starting P before the tile.  X_p is a HANKEL matrix: row r is the
// same linear signal shifted by 64 samples = 128 bytes of bf16, which is exactly the row pitch of
// the tensor core's canonical K-major SWIZZLE_128B shared-memory layout.  So the signal is stored
// ONCE, linearly (in that swizzle), and the 128 x K operand the MMA reads is produced by the shared
// memory descriptor alone: K-atom a / K-step t start at byte a*128 + t*32 of the plane.  No im2col
// copy exists anywhere.  A_p (64 phases x K, a Toeplitz band of the taps) is built on the host at
// create time.
//
// Precision.  fp32 -> bf16 hi + bf16 lo (x = hi + lo + O(2^-18 |x|)).  The tap operand carries
// [h_hi phases 0..63 ; h_lo phases 0..63] as its M = 128 rows, the signal operand is x_hi, then x_lo:
// two MMAs per K-step per plane give all FOUR partial products (hi*hi, hi*lo, lo*hi, lo*lo), and the
// epilogue adds the hi-tap and the lo-tap sums of each phase.  fp32 accumulation in TMEM.
//
// Two kernels run this formulation.  Both are persistent (one CTA per SM) and warp-specialised, so the
// conversion (fp32 -> 4 swizzled bf16 planes in shared memory), the MMAs and the epilogue of successive
// tiles overlap; each is described above its code.
//   fir_tc_ts_kernel    tap-stationary: decimation 1 and K <= 512 (up to 449 taps).  The taps sit in tensor
//                       memory for the whole call and tiles are 4096 outputs.  A float stream, which only
//                       this kernel takes, runs 8192 per tile: two 4096-sample runs ride through the planes
//                       "re" and "im", the same MMAs at twice the sample rate.  tc_create picks this kernel
//                       whenever it applies, so auto selection (at most 448 taps) reaches only this one.
//   fir_tc_pipe_kernel  ring form: decimation 1..8, up to 2048 taps per branch, tiles of 8192 outputs.  The
//                       pre-swizzled tap atoms stream from L2 through a shared-memory ring by 1-D bulk
//                       copies (16 KiB per 64-wide K-atom).  It serves explicit algorithm 2 at D > 1 or
//                       beyond 449 taps.
#include <cuda_bf16.h>

#include <vector>

#include "common.cuh"
#include "fir_tc.cuh"
#include "tc_ptx.cuh"

namespace b200 {

constexpr int TC_NROW = 128;             // signal rows per tile (MMA N)
constexpr int TC_PH = 64;                // outputs per row = bf16 elements per 128-byte swizzle row
constexpr int TC_TILE = TC_NROW * TC_PH; // outputs per tile
constexpr int TC_ATOM_BYTES = 128 * 128; // one K-atom of the tap operand: 128 rows x 64 bf16
constexpr int TC_TMEM_COLS = 256;        // re accumulator: columns 0..127, im: 128..255
constexpr int TC_MAX_STAGES = 4;

// Both kernels take this as a __grid_constant__ and read it in place from the parameter bank.  As a plain by-value
// struct, how the compiler stages it depends on its size: at this size the float-stream converter loop came out
// 4 instructions longer and fir_fff at 64 taps ran 1.2 % slower (B200, 1000 W power limit).
struct tc_args {
    const float2* x;
    const float2* hist;
    float2* y;
    const uint8_t* gA; // [D][KA] tap atoms, pre-swizzled
    long long n_in, n_out;
    int Tm1;         // T - 1: length of hist
    int D;           // decimation = polyphase branches
    int P;           // samples of the branch signal in front of the tile
    int ksteps;      // 16-wide K-steps per branch
    int KA;          // 64-wide K-atoms per branch
    int plane_elems; // converted samples per plane: 64*127 + 16*ksteps
    int plane_bytes; // multiple of 1024
    int stages;      // tap-atom ring depth
    int fuse;
    float kre, kim;
    const uint32_t* gAt; // TMEM-resident form: tap matrix [128 lanes][16*ksteps / 2] bf16 pairs, K contiguous
    int ts_plane_elems, ts_plane_bytes, ts_stages, ts_stage_bytes;
};

// instruction descriptor: bf16 x bf16 -> fp32, both operands K-major, M = 128, N = 128
constexpr uint32_t TC_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC_NROW >> 3) << 17) | ((128u >> 4) << 24);

// =================================================================================================
// Pipelined form: one persistent CTA per SM, warp-specialised.
//   warp 0       MMA issuer (one elected lane), owns the TMEM allocation (2 accumulator stages x 256 columns)
//   warp 1       tap-atom producer (1-D bulk copies into a ring)
//   warps 2..5   epilogue: TMEM -> registers, hi-/lo-tap halves combined through a 16 KiB exchange
//                buffer, coalesced 8-byte stores straight to global memory
//   warps 6..13  converters: fp32 stream -> four swizzled bf16 planes, two plane stages
// so the conversion of tile i+1, the MMAs of tile i and the epilogue of tile i-1 run concurrently;
// all hand-offs are mbarriers (tcgen05.commit on the tensor-core side).
constexpr int TCP_THREADS = 14 * 32;
constexpr int TCP_CONVERTERS = 8 * 32;
constexpr int TCP_XBUF = 32 * 64 * 8; // one exchange buffer: 32 columns x 64 phases x complex64
constexpr int TCP_LOADS = 18;         // loads in flight per converter thread: 256 x 18 x 16 B = 72 KiB >= one tile

__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int TCP_CONV, int TCP_LD>
__device__ __forceinline__ void tc_convert(const tc_args& a, uint8_t* planes, int plane_elems, int plane_bytes,
                                           long long m0, int p, int ctid)
{
    const long long j0 = m0 - a.P;
    if (a.D == 1 && j0 >= 0 && j0 + plane_elems <= a.n_in && (reinterpret_cast<uintptr_t>(a.x) & 15) == 0) {
        // the whole tile (64-80 KB) is requested before the first conversion: TCP_LD independent 16-byte loads per thread
        const float4* src = reinterpret_cast<const float4*>(a.x + j0);
        const int npairs = plane_elems >> 1;
#pragma unroll 1
        for (int base = 0; base < npairs; base += TCP_CONV * TCP_LD) {
            float4 v[TCP_LD];
#pragma unroll
            for (int u = 0; u < TCP_LD; u++) {
                const int q = base + u * TCP_CONV + ctid;
                v[u] = q < npairs ? __ldg(src + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < TCP_LD; u++) {
                const int q = base + u * TCP_CONV + ctid;
                if (q < npairs) {
                    const __nv_bfloat162 rh = __floats2bfloat162_rn(v[u].x, v[u].z);
                    const __nv_bfloat162 ih = __floats2bfloat162_rn(v[u].y, v[u].w);
                    const float2 rhf = __bfloat1622float2(rh), ihf = __bfloat1622float2(ih);
                    const __nv_bfloat162 rl = __floats2bfloat162_rn(v[u].x - rhf.x, v[u].z - rhf.y);
                    const __nv_bfloat162 il = __floats2bfloat162_rn(v[u].y - ihf.x, v[u].w - ihf.y);
                    const uint32_t off = tc_plane_off(2u * q);
                    *reinterpret_cast<__nv_bfloat162*>(planes + off) = rh;
                    *reinterpret_cast<__nv_bfloat162*>(planes + plane_bytes + off) = rl;
                    *reinterpret_cast<__nv_bfloat162*>(planes + 2 * plane_bytes + off) = ih;
                    *reinterpret_cast<__nv_bfloat162*>(planes + 3 * plane_bytes + off) = il;
                }
            }
        }
        return;
    }
    const bool interior = j0 * a.D - p >= 0 && (j0 + plane_elems - 1) * a.D - p < a.n_in;
#pragma unroll 1
    for (int base = 0; base < plane_elems; base += TCP_CONV * 8) {
        float2 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int i = base + u * TCP_CONV + ctid;
            const long long n = (j0 + i) * a.D - p;
            v[u] = make_float2(0.f, 0.f);
            if (i < plane_elems) {
                if (interior || (n >= 0 && n < a.n_in))
                    v[u] = __ldg(a.x + n);
                else if (n < 0 && a.hist != nullptr && n >= -(long long)a.Tm1)
                    v[u] = __ldg(a.hist + (a.Tm1 + n));
            }
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int i = base + u * TCP_CONV + ctid;
            if (i < plane_elems) {
                __nv_bfloat16 rh, rl, ih, il;
                tc_split(v[u].x, rh, rl);
                tc_split(v[u].y, ih, il);
                const uint32_t off = tc_plane_off((uint32_t)i);
                *reinterpret_cast<__nv_bfloat16*>(planes + off) = rh;
                *reinterpret_cast<__nv_bfloat16*>(planes + plane_bytes + off) = rl;
                *reinterpret_cast<__nv_bfloat16*>(planes + 2 * plane_bytes + off) = ih;
                *reinterpret_cast<__nv_bfloat16*>(planes + 3 * plane_bytes + off) = il;
            }
        }
    }
}

__global__ void __launch_bounds__(TCP_THREADS, 1) fir_tc_pipe_kernel(const __grid_constant__ tc_args a)
{
    extern __shared__ uint8_t tc_smem_raw[];
    uint8_t* smem = tc_align1024(tc_smem_raw);
    uint8_t* planes = smem;                                          // [2 stages][re_hi, re_lo, im_hi, im_lo]
    uint8_t* ring = smem + 8 * (size_t)a.plane_bytes;                // tap atoms
    uint8_t* xbuf = ring + (size_t)a.stages * TC_ATOM_BYTES;         // [2] exchange buffers
    uint64_t* bars = reinterpret_cast<uint64_t*>(xbuf + 2 * TCP_XBUF);
    uint64_t* taps_full = bars;                                      // [TC_MAX_STAGES]
    uint64_t* taps_empty = bars + TC_MAX_STAGES;                     // [TC_MAX_STAGES]
    uint64_t* planes_full = bars + 2 * TC_MAX_STAGES;                // [2]
    uint64_t* planes_empty = planes_full + 2;                        // [2]
    uint64_t* tmem_full = planes_empty + 2;                          // [2]
    uint64_t* tmem_empty = tmem_full + 2;                            // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int tid = threadIdx.x, warp = tc_warp_idx(), lane = tid & 31;
    const long long n_tiles = (a.n_out + TC_TILE - 1) / TC_TILE;
    const int my_tiles = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);

    if (tid == 0) {
        for (int s = 0; s < a.stages; s++) {
            mbar_init(&taps_full[s], 1);
            mbar_init(&taps_empty[s], 1);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(&planes_full[b], TCP_CONVERTERS / 32);
            mbar_init(&planes_empty[b], 1);
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], 4);
        }
        fence_mbar_init();
    }
    if (warp == 0) {
        __syncwarp();
        tc_alloc(tmem_slot, 2 * TC_TMEM_COLS);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // the CTA owns all 512 columns, so the allocation starts at column 0 / lane 0: using the literal keeps
    // every MMA operand warp-uniform for the compiler (a value loaded from shared memory is not)
    if (*tmem_slot != 0)
        __trap();
    constexpr uint32_t tmem = 0;
    const int atoms_per_tile = a.D * a.KA;

    if (warp == 0) {
        // ================= MMA issuer =================
        const uint32_t planes_s = smem_u32(planes), ring_s = smem_u32(ring);
        int g = 0, u = 0;
        for (int it = 0; it < my_tiles; it++) {
            const int acc = it & 1;
            mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d_re = tmem + acc * TC_TMEM_COLS, d_im = d_re + TC_NROW;
            for (int p = 0; p < a.D; p++, u++) {
                const int ps = u & 1;
                mbar_wait(&planes_full[ps], (u >> 1) & 1);
                tc_fence_after();
                const uint32_t pl = planes_s + ps * 4 * a.plane_bytes;
                for (int at = 0; at < a.KA; at++, g++) {
                    const int s = g % a.stages;
                    mbar_wait(&taps_full[s], (g / a.stages) & 1);
                    tc_fence_after();
                    const int nst = min(4, a.ksteps - 4 * at);
                    if (tc_elect_one()) {
                        const uint64_t pstep = (uint64_t)(a.plane_bytes >> 4);
                        uint64_t adesc = tc_desc(ring_s + s * TC_ATOM_BYTES), b0 = tc_desc(pl + at * 128);
                        for (int t = 0; t < nst; t++, adesc += 2, b0 += 2) {
                            const uint32_t accum = (p | at | t) != 0;
                            tc_mma_bf16(d_re, adesc, b0, TC_IDESC, accum);
                            tc_mma_bf16(d_re, adesc, b0 + pstep, TC_IDESC, 1);
                            tc_mma_bf16(d_im, adesc, b0 + 2 * pstep, TC_IDESC, accum);
                            tc_mma_bf16(d_im, adesc, b0 + 3 * pstep, TC_IDESC, 1);
                        }
                        tc_commit(&taps_empty[s]);
                        if (at == a.KA - 1) {
                            tc_commit(&planes_empty[ps]);
                            if (p == a.D - 1)
                                tc_commit(&tmem_full[acc]);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        // ================= tap-atom producer =================
        const int total = my_tiles * atoms_per_tile;
        for (int g = 0; g < total; g++) {
            const int s = g % a.stages;
            mbar_wait(&taps_empty[s], ((g / a.stages) & 1) ^ 1);
            if (lane == 0) {
                mbar_arrive_expect_tx(&taps_full[s], TC_ATOM_BYTES);
                bulk_copy_g2s(ring + (size_t)s * TC_ATOM_BYTES, a.gA + (size_t)(g % atoms_per_tile) * TC_ATOM_BYTES,
                              TC_ATOM_BYTES, &taps_full[s]);
            }
            __syncwarp();
        }
    } else if (warp < 6) {
        // ================= epilogue =================
        const int quarter = warp & 3;                 // TMEM lanes 32*quarter .. +31
        const int part = quarter >> 1;                // 0: hi-tap rows, 1: lo-tap rows
        const int c = (quarter & 1) * 32 + lane;      // phase
        const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16);
        int cq = 0;
        for (int it = 0; it < my_tiles; it++) {
            const int acc = it & 1;
            const long long m0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * TC_TILE;
            const long long left = a.n_out - m0;
            const int count = left < TC_TILE ? (int)left : TC_TILE;
            float2* dst = a.y + m0;
            mbar_wait(&tmem_full[acc], (it >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int q = 0; q < 4; q++, cq++) {
                float re[32], im[32];
                tc_ld32(tl + acc * TC_TMEM_COLS + q * 32, re);
                tc_ld32(tl + acc * TC_TMEM_COLS + TC_NROW + q * 32, im);
                tc_wait_ld();
                if (q == 3) { // this warp has drained its lanes of the accumulator stage
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0)
                        mbar_arrive(&tmem_empty[acc]);
                }
                float2* xb = reinterpret_cast<float2*>(xbuf + (cq & 1) * TCP_XBUF);
                const bool writer = part == ((cq & 1) ^ 1);
                if (writer) {
#pragma unroll
                    for (int i = 0; i < 32; i++)
                        xb[i * 64 + c] = make_float2(re[i], im[i]);
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (!writer) {
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        float2 v = xb[i * 64 + c];
                        v.x += re[i];
                        v.y += im[i];
                        if (a.fuse)
                            v = cmul_nofma(v, a.kre, a.kim);
                        const int o = (q * 32 + i) * 64 + c;
                        if (o < count)
                            __stcs(dst + o, v);
                    }
                }
            }
        }
    } else {
        // ================= converters =================
        const int ctid = tid - 6 * 32;
        int u = 0;
        for (int it = 0; it < my_tiles; it++) {
            const long long m0 = ((long long)blockIdx.x + (long long)it * gridDim.x) * TC_TILE;
            for (int p = 0; p < a.D; p++, u++) {
                const int ps = u & 1;
                mbar_wait(&planes_empty[ps], ((u >> 1) & 1) ^ 1);
                tc_convert<TCP_CONVERTERS, TCP_LOADS>(a, planes + (size_t)ps * 4 * a.plane_bytes, a.plane_elems,
                                                      a.plane_bytes, m0, p, ctid);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0)
                    mbar_arrive(&planes_full[ps]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tc_dealloc(tmem, 2 * TC_TMEM_COLS);
    }
}

// =================================================================================================
// Tap-stationary form (decimation 1, K <= 512, i.e. up to 448 taps): the tap operand never changes, so it
// is written ONCE per CTA into tensor memory (A operand from TMEM, 128 lanes x K/2 columns) and the
// MMAs read only the signal from shared memory -- half the shared-memory traffic of the ring form and
// no tap streaming at all.  Tiles are 64 Hankel rows (4096 outputs, MMA 128x64x16), so an accumulator
// stage is 128 TMEM columns (re 64 + im 64): 256 columns of taps + 2 accumulator stages = 512.
// The tap rows are permuted so that the hi- and lo-tap partial sums of a phase sit 16 lanes apart in the
// same warp: the epilogue adds them with one shuffle, no shared-memory exchange and no CTA barrier.
//   warp 0        MMA issuer (one elected lane), TMEM allocation
//   warp 1        input producer: one 1-D bulk copy (TMA) per tile, raw fp32, into a 3-deep staging ring --
//                 two to three tiles (70-100 KB) are in flight per SM whatever the other warps are doing
//   warps 4..11   epilogue: (warp & 3) = TMEM lane quarter, two warps per quarter split the 64 columns
//                 (warps 4..7 also do the one-off tap upload into TMEM)
//   warps 2, 3, 12..15  converters: staging (fp32) -> four swizzled bf16 planes, 3 plane stages
// Measured on the way here (roles switched off one at a time, per 4096-sample tile and SM): with register-staged
// global loads in the converters (two groups x 36 KB in flight) the conversion alone took 1.5 us and did not
// overlap the epilogue's stores (both latency-bound on the same memory system): 266 GS/s at 64 taps.
constexpr int TS_NROW = 64;
constexpr int TS_TILE = TS_NROW * TC_PH;  // 4096 outputs
constexpr int TS_THREADS = 16 * 32;
constexpr int TS_EPI_WARPS = 8;
constexpr int TS_EPI_WARP0 = 4;
constexpr int TS_CONV_WARPS = 6;
constexpr int TS_CONV = TS_CONV_WARPS * 32;
constexpr int TS_MAX_STAGES = 4;          // plane stages
constexpr int TS_IN_STAGES = 3;           // staging ring (raw input tiles)
constexpr int TS_A_COLS = 256;
constexpr uint32_t TS_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TS_NROW >> 3) << 17) | ((128u >> 4) << 24);

// interior tile: its whole input span [j0, j0 + plane_elems) lies inside this call's stream, so it can travel as
// ONE bulk copy; edge tiles (history in front, ragged end) are read element-wise.  A ring hands out windows
// that start on any item (8 bytes): when x is only 8-byte aligned the copy starts one sample early (`shift` = 1,
// the bulk copy needs 16-byte alignment) and the converters skip that sample.
// samples between the 16-byte boundary at or below x[0] and x[0]: 0 / 1 for a complex stream, 0 .. 3 for a float stream
template <bool REAL>
__device__ __forceinline__ int ts_shift(const tc_args& a)
{
    return REAL ? (int)((reinterpret_cast<uintptr_t>(a.x) >> 2) & 3) : (int)((reinterpret_cast<uintptr_t>(a.x) >> 3) & 1);
}
// head tile of a call: its first P samples are history (or zeros), the others are x[0 .. tile).  The producer
// warp copies the history part itself and sends the rest as a bulk copy, so the tile runs through the same staged
// conversion as an interior one (the element-wise path costs ~3 us, on the CTA that has the most tiles).
template <bool REAL>
__device__ __forceinline__ bool ts_head_tile(const tc_args& a, long long j0)
{
    if (REAL)
        return j0 == -(long long)a.P && a.P > 0 && ts_shift<REAL>(a) == 0 && 2 * TS_TILE <= a.n_in;
    return j0 == -(long long)a.P && a.P > 0 && ts_shift<REAL>(a) == 0 && a.ts_plane_elems - a.P <= a.n_in;
}
// REAL: a tile's input is the 8192 + P floats from j0 on (run A: [j0, j0 + plane_elems), run B: 4096 further); the
// bulk copies need a 16-byte aligned stream, j0 is a multiple of 16 samples
template <bool REAL>
__device__ __forceinline__ bool ts_fast_tile(const tc_args& a, long long j0)
{
    if (REAL) {
        // a ring hands out windows that start on any item (4 bytes): the copy then starts `sh` samples early and ends
        // (4 - sh) % 4 samples late, so that both ends sit on 16-byte boundaries, and the converters skip the lead
        const int sh = ts_shift<REAL>(a);
        return (j0 - sh >= 0 && j0 + 2 * TS_TILE + a.P + ((4 - sh) & 3) <= a.n_in) || ts_head_tile<REAL>(a, j0);
    }
    const int sh = ts_shift<REAL>(a);
    return (j0 - sh >= 0 && j0 + a.ts_plane_elems + sh <= a.n_in) || ts_head_tile<REAL>(a, j0);
}

// element-wise conversion of an edge tile of a REAL stream: plane "re" <- samples j0 + i, plane "im" <- j0 + 4096 + i
template <int NCONV>
__device__ __forceinline__ void tc_convert_real(const tc_args& a, uint8_t* planes, int plane_elems, int plane_bytes,
                                                long long m0, int ctid)
{
    const float* x = reinterpret_cast<const float*>(a.x);
    const float* hist = reinterpret_cast<const float*>(a.hist);
    const long long j0 = m0 - a.P;
    auto fetch = [&](long long n) -> float {
        if (n >= 0)
            return n < a.n_in ? __ldg(x + n) : 0.f;
        return (hist != nullptr && n >= -(long long)a.Tm1) ? __ldg(hist + (a.Tm1 + n)) : 0.f;
    };
#pragma unroll 1
    for (int base = 0; base < plane_elems; base += NCONV * 4) {
        float va[4], vb[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = base + u * NCONV + ctid;
            va[u] = i < plane_elems ? fetch(j0 + i) : 0.f;
            vb[u] = i < plane_elems ? fetch(j0 + TS_TILE + i) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = base + u * NCONV + ctid;
            if (i < plane_elems) {
                __nv_bfloat16 rh, rl, ih, il;
                tc_split(va[u], rh, rl);
                tc_split(vb[u], ih, il);
                const uint32_t off = tc_plane_off((uint32_t)i);
                *reinterpret_cast<__nv_bfloat16*>(planes + off) = rh;
                *reinterpret_cast<__nv_bfloat16*>(planes + plane_bytes + off) = rl;
                *reinterpret_cast<__nv_bfloat16*>(planes + 2 * plane_bytes + off) = ih;
                *reinterpret_cast<__nv_bfloat16*>(planes + 3 * plane_bytes + off) = il;
            }
        }
    }
}

template <bool REAL>
__global__ void __launch_bounds__(TS_THREADS, 1) fir_tc_ts_kernel(const __grid_constant__ tc_args a)
{
    extern __shared__ uint8_t tc_smem_raw[];
    uint8_t* smem = tc_align1024(tc_smem_raw);
    uint8_t* planes = smem;                                          // [stages][re_hi, re_lo, im_hi, im_lo]
    uint8_t* staging = planes + (size_t)a.ts_stages * 4 * a.ts_plane_bytes; // [TS_IN_STAGES] raw complex64 tiles
    uint64_t* bars = reinterpret_cast<uint64_t*>(staging + (size_t)TS_IN_STAGES * a.ts_stage_bytes);
    uint64_t* planes_full = bars;                                    // [TS_MAX_STAGES]
    uint64_t* planes_empty = bars + TS_MAX_STAGES;                   // [TS_MAX_STAGES]
    uint64_t* tmem_full = bars + 2 * TS_MAX_STAGES;                  // [2]
    uint64_t* tmem_empty = tmem_full + 2;                            // [2]
    uint64_t* in_full = tmem_empty + 2;                              // [TS_IN_STAGES]
    uint64_t* in_empty = in_full + TS_IN_STAGES;                     // [TS_IN_STAGES]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_empty + TS_IN_STAGES);

    const int tid = threadIdx.x, warp = tc_warp_idx(), lane = tid & 31;
    constexpr int TILE_OUT = REAL ? 2 * TS_TILE : TS_TILE; // outputs (items) per tile
    const long long n_tiles = (a.n_out + TILE_OUT - 1) / TILE_OUT;
    // CTA order reversed: the head tile (history in front of the call) goes to the LAST CTA, which has one tile
    // fewer than the first ones whenever the tiles do not divide evenly
    const long long bid = (long long)(gridDim.x - 1 - blockIdx.x);
    const int my_tiles = (int)((n_tiles - bid + gridDim.x - 1) / gridDim.x);
    const int S = a.ts_stages;

    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(&planes_full[s], TS_CONV_WARPS);
            mbar_init(&planes_empty[s], 1);
        }
        for (int s = 0; s < TS_IN_STAGES; s++) {
            mbar_init(&in_full[s], 1);
            mbar_init(&in_empty[s], TS_CONV_WARPS);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], TS_EPI_WARPS);
        }
        fence_mbar_init();
    }
    if (warp == 0) {
        __syncwarp();
        tc_alloc(tmem_slot, 512);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (*tmem_slot != 0) // all 512 columns are ours: the allocation starts at 0 (keeps MMA operands warp-uniform)
        __trap();
    constexpr uint32_t tmem = 0;
    if (warp >= TS_EPI_WARP0 && warp < TS_EPI_WARP0 + 4) {
        // one-off: this thread's tap row -> its TMEM lane, 8 columns (16 bf16) per K-step
        const int quarter = warp & 3;
        const uint32_t* row = a.gAt + (size_t)(quarter * 32 + lane) * (a.ksteps * 8);
        const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16);
        for (int k = 0; k < a.ksteps; k++) {
            const uint4 lo4 = __ldg(reinterpret_cast<const uint4*>(row + k * 8));
            const uint4 hi4 = __ldg(reinterpret_cast<const uint4*>(row + k * 8 + 4));
            const uint32_t v[8] = { lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w };
            tc_st8(tl + k * 8, v);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t d_base = tmem + TS_A_COLS;
    // programmatic dependent launch: everything above (barriers, TMEM, the tap upload) overlapped the tail of
    // the previous kernel in the stream; nothing below may start before that kernel has completed and flushed
    pdl_wait();
    pdl_launch_dependents();

    if (warp == 0) {
        // ================= MMA issuer =================
        const uint32_t planes_s = smem_u32(planes);
        for (int it = 0; it < my_tiles; it++) {
            const int acc = it & 1, ps = it % S;
            mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
            mbar_wait(&planes_full[ps], (it / S) & 1);
            tc_fence_after();
            const uint32_t d_re = d_base + acc * 2 * TS_NROW, d_im = d_re + TS_NROW;
            // descriptors of the four planes at K-step 0; a K-step advances the start address by 32 bytes = 2 units
            uint64_t b0 = tc_desc(planes_s + ps * 4 * a.ts_plane_bytes);
            const uint64_t pstep = (uint64_t)(a.ts_plane_bytes >> 4);
            if (tc_elect_one()) {
#pragma unroll 2
                for (int k = 0; k < a.ksteps; k++, b0 += 2) {
                    const uint32_t at = tmem + k * 8, accum = k != 0;
                    tc_mma_bf16_ts(d_re, at, b0, TS_IDESC, accum);
                    tc_mma_bf16_ts(d_re, at, b0 + pstep, TS_IDESC, 1);
                    tc_mma_bf16_ts(d_im, at, b0 + 2 * pstep, TS_IDESC, accum);
                    tc_mma_bf16_ts(d_im, at, b0 + 3 * pstep, TS_IDESC, 1);
                }
                tc_commit(&planes_empty[ps]);
                tc_commit(&tmem_full[acc]);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ================= input producer =================
        int nf = 0;
        for (int it = 0; it < my_tiles; it++) {
            const long long j0 = (bid + (long long)it * gridDim.x) * TILE_OUT - a.P;
            if (!ts_fast_tile<REAL>(a, j0))
                continue;                                            // edge tile: the converters read it themselves
            const int slot = nf % TS_IN_STAGES;
            mbar_wait(&in_empty[slot], ((nf / TS_IN_STAGES) & 1) ^ 1);
            if (REAL) {
                // float stream: 8192 + P samples per tile; the head tile's first P come from the history
                float* st = reinterpret_cast<float*>(staging + (size_t)slot * a.ts_stage_bytes);
                const float* xr = reinterpret_cast<const float*>(a.x);
                const float* hr = reinterpret_cast<const float*>(a.hist);
                if (j0 < 0) {
                    for (int i = lane; i < a.P; i += 32) {
                        const int n = i - a.P;
                        st[i] = (hr != nullptr && n >= -a.Tm1) ? __ldg(hr + (a.Tm1 + n)) : 0.f;
                    }
                    __syncwarp();
                }
                if (lane == 0) {
                    const int sh = j0 < 0 ? 0 : ts_shift<REAL>(a);
                    const uint32_t bytes = (uint32_t)(2 * TS_TILE + (j0 < 0 ? 0 : a.P) + sh + ((4 - sh) & 3)) * 4u;
                    mbar_arrive_expect_tx(&in_full[slot], bytes);
                    bulk_copy_g2s(j0 < 0 ? st + a.P : st, j0 < 0 ? xr : xr + j0 - sh, bytes, &in_full[slot]);
                }
            } else if (j0 < 0) {
                // head tile: history (or zeros) by this warp, x[0 .. 4096) as a bulk copy behind it; the mbarrier
                // arrive below releases the generic stores to the converters
                float2* st = reinterpret_cast<float2*>(staging + (size_t)slot * a.ts_stage_bytes);
                for (int i = lane; i < a.P; i += 32) {
                    const int n = i - a.P;
                    st[i] = (a.hist != nullptr && n >= -a.Tm1) ? __ldg(a.hist + (a.Tm1 + n)) : make_float2(0.f, 0.f);
                }
                __syncwarp();
                if (lane == 0) {
                    const uint32_t bytes = (uint32_t)(a.ts_plane_elems - a.P) * 8u;
                    mbar_arrive_expect_tx(&in_full[slot], bytes);
                    bulk_copy_g2s(st + a.P, a.x, bytes, &in_full[slot]);
                }
            } else if (lane == 0) {
                const int sh = ts_shift<REAL>(a);
                const uint32_t bytes = (uint32_t)(a.ts_plane_elems + 2 * sh) * 8u;
                mbar_arrive_expect_tx(&in_full[slot], bytes);
                bulk_copy_g2s(staging + (size_t)slot * a.ts_stage_bytes, a.x + j0 - sh, bytes, &in_full[slot]);
            }
            __syncwarp();
            nf++;
        }
    } else if (warp >= TS_EPI_WARP0 && warp < TS_EPI_WARP0 + TS_EPI_WARPS) {
        // ================= epilogue =================
        const int quarter = warp & 3, ch = (warp - TS_EPI_WARP0) >> 2;   // this warp drains columns 32 ch .. 32 ch + 31
        const int c = quarter * 16 + (lane & 15);     // phase; lanes l and l+16 hold its hi- / lo-tap sums
        const bool lower = lane < 16;
        const uint32_t tl = d_base + ((uint32_t)(quarter * 32) << 16);
        for (int it = 0; it < my_tiles; it++) {
            const int acc = it & 1;
            const long long m0 = (bid + (long long)it * gridDim.x) * TILE_OUT;
            const long long left = a.n_out - m0;
            const int count = left < TILE_OUT ? (int)left : TILE_OUT;
            float2* dst = a.y + m0;
            float* dstr = reinterpret_cast<float*>(a.y) + m0; // REAL: run A at dstr, run B 4096 floats further
            mbar_wait(&tmem_full[acc], (it >> 1) & 1);
            tc_fence_after();
            {
                float re[32], im[32];
                tc_ld32(tl + acc * 2 * TS_NROW + ch * 32, re);
                tc_ld32(tl + acc * 2 * TS_NROW + TS_NROW + ch * 32, im);
                tc_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0)
                    mbar_arrive(&tmem_empty[acc]);
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    // lower half-warp finishes column 2j, upper half column 2j+1: each sends what the other needs
                    const float sr = lower ? re[2 * j + 1] : re[2 * j], si = lower ? im[2 * j + 1] : im[2 * j];
                    const float rr = __shfl_xor_sync(0xffffffffu, sr, 16), ri = __shfl_xor_sync(0xffffffffu, si, 16);
                    float2 v = make_float2((lower ? re[2 * j] : re[2 * j + 1]) + rr, (lower ? im[2 * j] : im[2 * j + 1]) + ri);
                    const int o = (ch * 32 + 2 * j + (lower ? 0 : 1)) * 64 + c;
                    if (REAL) {
                        if (a.fuse) {
                            v.x = __fmul_rn(v.x, a.kre);
                            v.y = __fmul_rn(v.y, a.kre);
                        }
                        if (o < count)
                            __stcs(dstr + o, v.x);
                        if (TS_TILE + o < count)
                            __stcs(dstr + TS_TILE + o, v.y);
                    } else {
                        if (a.fuse)
                            v = cmul_nofma(v, a.kre, a.kim);
                        if (o < count)
                            __stcs(dst + o, v);
                    }
                }
            }
        }
    } else {
        // ================= converters (warps 2, 3, 12..15) =================
        const int ctid = (warp < 4 ? warp - 2 : warp - 10) * 32 + lane;
        int nf = 0;
        for (int it = 0; it < my_tiles; it++) {
            const long long m0 = (bid + (long long)it * gridDim.x) * TILE_OUT;
            const int ps = it % S;
            uint8_t* pl = planes + (size_t)ps * 4 * a.ts_plane_bytes;
            mbar_wait(&planes_empty[ps], ((it / S) & 1) ^ 1);
            if (ts_fast_tile<REAL>(a, m0 - a.P)) {
                const int slot = nf % TS_IN_STAGES;
                mbar_wait(&in_full[slot], (nf / TS_IN_STAGES) & 1);
                const float2* src = reinterpret_cast<const float2*>(staging + (size_t)slot * a.ts_stage_bytes) + ts_shift<REAL>(a);
                const int npairs = a.ts_plane_elems >> 1;
                const bool al16 = ts_shift<REAL>(a) == 0;
#pragma unroll 4
                for (int q = ctid; q < npairs; q += TS_CONV) {
                    float4 v;
                    if (REAL) {
                        // samples 2q, 2q+1 of run A and of run B (4096 floats = 2048 float2 further)
                        if (al16) {
                            const float2* s2 = reinterpret_cast<const float2*>(staging + (size_t)slot * a.ts_stage_bytes);
                            const float2 ra = s2[q], rb = s2[TS_TILE / 2 + q];
                            v = make_float4(ra.x, rb.x, ra.y, rb.y);
                        } else {
                            const float* s1 = reinterpret_cast<const float*>(staging + (size_t)slot * a.ts_stage_bytes) +
                                              ts_shift<REAL>(a);
                            v = make_float4(s1[2 * q], s1[TS_TILE + 2 * q], s1[2 * q + 1], s1[TS_TILE + 2 * q + 1]);
                        }
                    } else if (al16) {
                        v = *reinterpret_cast<const float4*>(src + 2 * q);
                    } else {
                        const float2 s0 = src[2 * q], s1 = src[2 * q + 1];
                        v = make_float4(s0.x, s0.y, s1.x, s1.y);
                    }
                    const __nv_bfloat162 rh = __floats2bfloat162_rn(v.x, v.z);
                    const __nv_bfloat162 ih = __floats2bfloat162_rn(v.y, v.w);
                    const float2 rhf = __bfloat1622float2(rh), ihf = __bfloat1622float2(ih);
                    const __nv_bfloat162 rl = __floats2bfloat162_rn(v.x - rhf.x, v.z - rhf.y);
                    const __nv_bfloat162 il = __floats2bfloat162_rn(v.y - ihf.x, v.w - ihf.y);
                    const uint32_t off = tc_plane_off(2u * q);
                    *reinterpret_cast<__nv_bfloat162*>(pl + off) = rh;
                    *reinterpret_cast<__nv_bfloat162*>(pl + a.ts_plane_bytes + off) = rl;
                    *reinterpret_cast<__nv_bfloat162*>(pl + 2 * a.ts_plane_bytes + off) = ih;
                    *reinterpret_cast<__nv_bfloat162*>(pl + 3 * a.ts_plane_bytes + off) = il;
                }
                __syncwarp();
                if (lane == 0)
                    mbar_arrive(&in_empty[slot]);                    // this warp has read its share of the slot
                nf++;
            } else {
                if (REAL)
                    tc_convert_real<TS_CONV>(a, pl, a.ts_plane_elems, a.ts_plane_bytes, m0, ctid);
                else
                    tc_convert<TS_CONV, 8>(a, pl, a.ts_plane_elems, a.ts_plane_bytes, m0, 0, ctid);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0)
                mbar_arrive(&planes_full[ps]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tc_dealloc(tmem, 512);
    }
}

// ---- host side ---------------------------------------------------------------------------------
struct tc_plan {
    int T = 0, D = 1;
    int Tq = 0, P = 0, ksteps = 0, KA = 0, plane_elems = 0, plane_bytes = 0;
    int fuse = 0;
    float kre = 1.f, kim = 0.f;
    int real = 0;          // float stream (fff): tap-stationary kernel only
    int ts = 0;            // 1: tap-stationary kernel (fir_tc_ts_kernel): D = 1, K <= 512; 0: ring form (fir_tc_pipe_kernel)
    int ts_plane_elems = 0, ts_plane_bytes = 0, ts_stages = 0, ts_stage_bytes = 0;
    size_t ts_smem = 0;
    uint32_t* d_at = nullptr;
    int pipe_stages = 2;
    size_t pipe_smem = 0;
    uint8_t* d_atoms = nullptr;
};

static inline uint16_t tc_bf16_rn(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u)
        return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static inline float tc_bf16_f(uint16_t b)
{
    uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}

bool tc_supported(int n_taps, int decimation, int real)
{
    if (n_taps < 1 || decimation < 1 || decimation > 8)
        return false;
    const int tq = (n_taps + decimation - 1) / decimation;
    if (real) // float streams: the tap-stationary kernel only (decimation 1, K = roundup16(T - 1) + 64 <= 512)
        return decimation == 1 && (n_taps - 1 + 15) / 16 * 16 + TC_PH <= 2 * TS_A_COLS;
    return tq <= 2048;
}

int tc_create(const float* taps, int n_taps, int decimation, int real, int fuse, float kre, float kim, tc_plan** out)
{
    *out = nullptr;
    if (!tc_supported(n_taps, decimation, real))
        return set_err(B200_ERR_UNSUPPORTED, "fir(tensor core): complex stream, decimation 1..8, <= 2048 taps per branch");
    tc_plan* p = new tc_plan();
    p->T = n_taps;
    p->D = decimation;
    p->real = real;
    p->Tq = (n_taps + decimation - 1) / decimation;
    p->P = (p->Tq - 1 + 15) / 16 * 16;
    const int kneed = p->P + TC_PH;
    p->ksteps = kneed / 16;
    p->KA = (kneed + 63) / 64;
    p->plane_elems = TC_PH * (TC_NROW - 1) + kneed;
    p->plane_bytes = ((p->plane_elems + 63) / 64 * 128 + 1023) / 1024 * 1024;
    p->fuse = fuse;
    p->kre = kre;
    p->kim = kim;
    const int total_atoms = p->D * p->KA;
    // ring form: two plane stages + the deepest tap ring that still fits.  At 2048 taps per branch a 2-deep ring
    // needs 230 656 bytes, so every filter tc_supported accepts fits; the check guards that arithmetic.
    {
        const size_t fixed = 1024 + 8 * (size_t)p->plane_bytes + 2 * TCP_XBUF + 256;
        int st = TC_MAX_STAGES;
        while (st > 1 && fixed + (size_t)st * TC_ATOM_BYTES > 227 * 1024)
            st--;
        if (st > total_atoms)
            st = total_atoms;
        p->pipe_stages = st;
        p->pipe_smem = fixed + (size_t)st * TC_ATOM_BYTES;
        if (p->pipe_smem > 227 * 1024) {
            delete p;
            return set_err(B200_ERR_UNSUPPORTED, "fir(tensor core): the tap ring does not fit shared memory");
        }
    }

    // tap atoms: [branch][atom][row 0..127][64 bf16], rows 0..63 = hi part of phase c, 64..127 = lo part,
    // element e of atom at <-> j = 64 at + e, tap index q = c + P - j of the branch; SWIZZLE_128B order
    std::vector<uint16_t> atoms((size_t)total_atoms * TC_ATOM_BYTES / 2, 0);
    for (int br = 0; br < p->D; br++)
        for (int at = 0; at < p->KA; at++) {
            uint16_t* dst = atoms.data() + ((size_t)br * p->KA + at) * (TC_ATOM_BYTES / 2);
            for (int row = 0; row < 128; row++) {
                const int c = row & 63, lo = row >> 6;
                for (int e = 0; e < 64; e++) {
                    const int j = 64 * at + e;
                    const long long q = (long long)c + p->P - j;
                    const long long k = q * p->D + br;
                    float hv = 0.f;
                    if (q >= 0 && k < n_taps)
                        hv = taps[k];
                    const uint16_t hi = tc_bf16_rn(hv);
                    const uint16_t v = lo ? tc_bf16_rn(hv - tc_bf16_f(hi)) : hi;
                    const size_t off = (size_t)row * 64 + (size_t)(((e >> 3) ^ (row & 7)) << 3) + (e & 7);
                    dst[off] = v;
                }
            }
        }
    // tap-stationary form: [128 TMEM lanes][K] bf16, K contiguous; lane 32 q + l carries phase 16 q + (l & 15),
    // hi part for l < 16 and lo part for l >= 16
    std::vector<uint16_t> at_rows;
    if (p->D == 1 && p->ksteps * 16 <= 2 * TS_A_COLS) {
        const int K = p->ksteps * 16;
        at_rows.assign((size_t)128 * K, 0);
        for (int m = 0; m < 128; m++) {
            const int q4 = m >> 5, l = m & 31, c = 16 * q4 + (l & 15), lo = l >> 4;
            for (int j = 0; j < K; j++) {
                const long long k = (long long)c + p->P - j;
                const float hv = (k >= 0 && k < n_taps) ? taps[k] : 0.f;
                const uint16_t hi = tc_bf16_rn(hv);
                at_rows[(size_t)m * K + j] = lo ? tc_bf16_rn(hv - tc_bf16_f(hi)) : hi;
            }
        }
        p->ts_plane_elems = TC_PH * (TS_NROW - 1) + K;
        p->ts_plane_bytes = ((p->ts_plane_elems + 63) / 64 * 128 + 1023) / 1024 * 1024;
        p->ts_stage_bytes = (p->ts_plane_elems * 8 + 16 + 1023) / 1024 * 1024; // + one sample each side for 8-byte-aligned streams
        int st = TS_MAX_STAGES;
        while (st > 2 && 1024 + (size_t)st * 4 * p->ts_plane_bytes + (size_t)TS_IN_STAGES * p->ts_stage_bytes + 256 > 227 * 1024)
            st--;
        p->ts_stages = st;
        p->ts_smem = 1024 + (size_t)st * 4 * p->ts_plane_bytes + (size_t)TS_IN_STAGES * p->ts_stage_bytes + 256;
        p->ts = 1;
    }
    cudaError_t e = cudaMalloc(&p->d_atoms, atoms.size() * 2);
    if (e == cudaSuccess)
        e = cudaMemcpy(p->d_atoms, atoms.data(), atoms.size() * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && !at_rows.empty()) {
        e = cudaMalloc(&p->d_at, at_rows.size() * 2);
        if (e == cudaSuccess)
            e = cudaMemcpy(p->d_at, at_rows.data(), at_rows.size() * 2, cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(fir_tc_ts_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(fir_tc_ts_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    }
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(fir_tc_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess)
        e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        tc_destroy(p);
        return set_err(e == cudaErrorMemoryAllocation ? B200_ERR_NOMEM : B200_ERR_CUDA, "fir(tensor core) create: %s",
                       cudaGetErrorString(e));
    }
    *out = p;
    return B200_OK;
}

void tc_destroy(tc_plan* p)
{
    if (!p)
        return;
    cudaFree(p->d_atoms);
    cudaFree(p->d_at);
    delete p;
}

int tc_launch(tc_plan* p, const float* d_hist, const void* d_in, void* d_out, long long n_in, long long n_out,
              cudaStream_t s)
{
    if (n_out <= 0)
        return B200_OK;
    const long long tiles = (n_out + TC_TILE - 1) / TC_TILE;
    if (tiles > 0x7fffffffLL)
        return set_err(B200_ERR_ARG, "fir(tensor core): too many items for one call");
    tc_args a{};
    a.x = (const float2*)d_in;
    a.hist = (const float2*)d_hist;
    a.y = (float2*)d_out;
    a.gA = p->d_atoms;
    a.n_in = n_in;
    a.n_out = n_out;
    a.Tm1 = p->T - 1;
    a.D = p->D;
    a.P = p->P;
    a.ksteps = p->ksteps;
    a.KA = p->KA;
    a.plane_elems = p->plane_elems;
    a.plane_bytes = p->plane_bytes;
    a.stages = p->pipe_stages;
    a.fuse = p->fuse;
    a.kre = p->kre;
    a.kim = p->kim;
    const long long sms = sm_count();
    if (p->ts) {
        a.gAt = p->d_at;
        a.ts_plane_elems = p->ts_plane_elems;
        a.ts_plane_bytes = p->ts_plane_bytes;
        a.ts_stages = p->ts_stages;
        a.ts_stage_bytes = p->ts_stage_bytes;
        const long long tile_out = p->real ? 2 * TS_TILE : TS_TILE;
        const long long ts_tiles = (n_out + tile_out - 1) / tile_out;
        const unsigned grid = (unsigned)(ts_tiles < sms ? ts_tiles : sms);
        if (p->real)
            B200_LAUNCH_PDL(fir_tc_ts_kernel<true>, grid, TS_THREADS, p->ts_smem, s, a);
        else
            B200_LAUNCH_PDL(fir_tc_ts_kernel<false>, grid, TS_THREADS, p->ts_smem, s, a);
        return B200_OK;
    }
    B200_LAUNCH(fir_tc_pipe_kernel, (unsigned)(tiles < sms ? tiles : sms), TCP_THREADS, p->pipe_smem, s, a);
    return B200_OK;
}

} // namespace b200

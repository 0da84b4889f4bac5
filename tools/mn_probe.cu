// mn_probe.cu -- groundwork for DESIGN.md section 9 "next (1)": does tcgen05.mma read a B operand that is stored
// MN-major (N contiguous, K strided) in the SWIZZLE_128B shared-memory layout, and with which descriptor fields?
// One CTA, one 128 x 64 x 64 product (4 K-steps), A K-major (the layout every kernel of the library uses), B MN-major:
//   element (n, k) of B at byte  (k / 8) * SBO  +  (k % 8) * 128  +  ((n / 8) ^ (k % 8)) * 16  +  (n % 8) * 2
// i.e. atoms of 8 k-rows x 64 n-elements (1024 bytes), 16-byte chunks XOR-swizzled by the row inside the atom.
// Prints the number of mismatches against a CPU product of the same small-integer (bf16-exact) operands.
//   build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -I newsched_b200/csrc -o /tmp/mn_probe tools/mn_probe.cu
//   run:   /tmp/mn_probe [mode]    mode 0: LBO = 8192, SBO = 1024 (hypothesis), 1: swapped, 2: K-major B (sanity check)
#include <cuda_bf16.h>

#include <cstdio>
#include <cstdlib>
#include <vector>

#include "tc_ptx.cuh"

namespace b200 {
char* err_buf() { static thread_local char b[256]; return b; }
int set_err(int code, const char*, ...) { return code; }
std::atomic<int64_t> g_launches{ 0 };
} // namespace b200
using namespace b200;

__device__ __forceinline__ uint64_t probe_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61; // SWIZZLE_128B
    return d;
}

__global__ void __launch_bounds__(128, 1) mn_probe_kernel(const uint16_t* gA, const uint16_t* gB, float* out, int mode)
{
    extern __shared__ uint8_t raw[];
    uint8_t* smem = tc_align1024(raw);
    uint8_t* sA = smem;          // 128 rows x 128 bytes (64 bf16), K-major SW128
    uint8_t* sB = smem + 16384;  // 8 KB
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 16384 + 8192);
    uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < 128 * 64; i += 128) { // A[m][k]
        const int m = i >> 6, k = i & 63;
        const uint32_t off = m * 128 + ((((k >> 3) ^ (m & 7))) << 4) + (k & 7) * 2;
        *reinterpret_cast<uint16_t*>(sA + off) = gA[i];
    }
    for (int i = tid; i < 64 * 64; i += 128) { // B[n][k]
        const int n = i >> 6, k = i & 63;
        uint32_t off;
        if (mode == 2) // K-major, as A
            off = n * 128 + ((((k >> 3) ^ (n & 7))) << 4) + (k & 7) * 2;
        else
            off = (k >> 3) * 1024 + (k & 7) * 128 + ((((n >> 3) ^ (k & 7))) << 4) + (n & 7) * 2;
        *reinterpret_cast<uint16_t*>(sB + off) = gB[i];
    }
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        __syncwarp();
        tc_alloc(slot, 64);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot;
    if (tid == 0) {
        // bf16 x bf16 -> fp32, M = 128, N = 64; bit 16: B is MN-major
        uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
        if (mode != 2)
            idesc |= 1u << 16;
        for (int s = 0; s < 4; s++) {
            const uint64_t ad = tc_desc(smem_u32(sA) + s * 32);
            uint64_t bd;
            if (mode == 2)
                bd = tc_desc(smem_u32(sB) + s * 32);
            else if (mode == 0)
                bd = probe_desc(smem_u32(sB) + s * 2048, 8192, 1024);
            else
                bd = probe_desc(smem_u32(sB) + s * 2048, 1024, 8192);
            tc_mma_bf16(tmem, ad, bd, idesc, s != 0);
        }
        tc_commit(bar);
    }
    mbar_wait(bar, 0);
    tc_fence_after();
    float v[32];
    for (int h = 0; h < 2; h++) {
        tc_ld32(tmem + ((uint32_t)(warp * 32) << 16) + h * 32, v);
        tc_wait_ld();
        for (int j = 0; j < 32; j++)
            out[(size_t)tid * 64 + h * 32 + j] = v[j];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tc_dealloc(tmem, 64);
    }
}

static uint16_t bf16_of(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    return (uint16_t)(u >> 16); // exact for the small integers used here
}

int main(int argc, char** argv)
{
    const int mode = argc > 1 ? atoi(argv[1]) : 0;
    std::vector<float> A(128 * 64), B(64 * 64), ref(128 * 64, 0.f);
    std::vector<uint16_t> hA(128 * 64), hB(64 * 64);
    for (int i = 0; i < 128 * 64; i++) {
        A[i] = (float)((i * 7 + (i >> 6) * 3) % 9 - 4);
        hA[i] = bf16_of(A[i]);
    }
    for (int i = 0; i < 64 * 64; i++) {
        B[i] = (float)((i * 5 + (i >> 6) * 11) % 7 - 3);
        hB[i] = bf16_of(B[i]);
    }
    for (int m = 0; m < 128; m++)
        for (int n = 0; n < 64; n++) {
            float acc = 0;
            for (int k = 0; k < 64; k++)
                acc += A[m * 64 + k] * B[n * 64 + k];
            ref[m * 64 + n] = acc;
        }
    uint16_t *dA, *dB;
    float* dO;
    cudaMalloc(&dA, hA.size() * 2);
    cudaMalloc(&dB, hB.size() * 2);
    cudaMalloc(&dO, ref.size() * 4);
    cudaMemcpy(dA, hA.data(), hA.size() * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, hB.data(), hB.size() * 2, cudaMemcpyHostToDevice);
    cudaMemset(dO, 0, ref.size() * 4);
    cudaFuncSetAttribute(mn_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 40 * 1024);
    mn_probe_kernel<<<1, 128, 40 * 1024>>>(dA, dB, dO, mode);
    cudaError_t e = cudaDeviceSynchronize();
    std::vector<float> got(ref.size());
    cudaMemcpy(got.data(), dO, got.size() * 4, cudaMemcpyDeviceToHost);
    int bad = 0;
    for (size_t i = 0; i < ref.size(); i++)
        bad += got[i] != ref[i];
    std::printf("{\"mode\": %d, \"cuda\": \"%s\", \"mismatches\": %d, \"of\": %zu, \"got0\": %g, \"ref0\": %g, \"got_last\": %g, \"ref_last\": %g}\n",
                mode, cudaGetErrorString(e), bad, ref.size(), got[0], ref[0], got.back(), ref.back());
    return 0;
}

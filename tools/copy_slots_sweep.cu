// How copy_slots_kernel (csrc/mgw_deploy.cu) was sized: its body (the full-slot case, no size lookup) at unroll 1 / 2 / 4 / 8
// and 1 / 2 / 4 / 8 / 16 blocks per SM spread over 64 slots of 1080p BGR, host to device and device to host through the mapped
// address of pinned memory, against cudaMemcpyAsync of the same pool; 20 back-to-back calls per timing, two rounds.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/copy_slots_sweep tools/copy_slots_sweep.cu
// Result on a B200: profiles/copy_slots_sweep.txt.
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>
#include <stdint.h>
template <int U>
__global__ void __launch_bounds__(256) k(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int stride, int n)
{
    const size_t off = (size_t)blockIdx.y * stride; src += off; dst += off;
    const int head = min((int)((16 - (off & 15)) & 15), n);
    const int n16 = (n - head) >> 4, tail = head + (n16 << 4);
    const int t = blockIdx.x * 256 + threadIdx.x, nt = gridDim.x * 256;
    if (t < head) dst[t] = __ldcs(src + t);
    if (t < n - tail) dst[tail + t] = __ldcs(src + tail + t);
    const uint4* s4 = reinterpret_cast<const uint4*>(src + head); uint4* d4 = reinterpret_cast<uint4*>(dst + head);
    int i = t;
    for (; i + (U - 1) * nt < n16; i += U * nt) {
        uint4 v[U];
#pragma unroll
        for (int q = 0; q < U; ++q) v[q] = __ldcs(s4 + i + q * nt);
#pragma unroll
        for (int q = 0; q < U; ++q) __stcs(d4 + i + q * nt, v[q]);
    }
    for (; i < n16; i += nt) __stcs(d4 + i, __ldcs(s4 + i));
}
template <int U> float run(const uint8_t* s, uint8_t* d, int S, int stride, int bps, int sms, cudaEvent_t a, cudaEvent_t b, int reps)
{
    long long full = (stride + 256LL * U * 16 - 1) / (256LL * U * 16), spread = ((long long)sms * bps + S - 1) / S;
    dim3 g((unsigned)(full < spread ? full : spread), S);
    for (int r = 0; r < 3; ++r) k<U><<<g, 256>>>(s, d, stride, stride);
    cudaEventRecord(a);
    for (int r = 0; r < reps; ++r) k<U><<<g, 256>>>(s, d, stride, stride);
    cudaEventRecord(b); cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b); return ms / reps;
}
int main()
{
    const int S = 64, stride = 1080 * 1920 * 3; const size_t bytes = (size_t)S * stride;
    uint8_t *h, *dv; cudaHostAlloc(&h, bytes, 0); cudaMalloc(&dv, bytes);
    memset(h, 1, bytes); cudaMemset(dv, 2, bytes);
    int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    const int reps = 20;
    for (int dir = 0; dir < 2; ++dir) {
        const uint8_t* s = dir == 0 ? h : dv; uint8_t* d = dir == 0 ? dv : h;
        for (int round = 0; round < 2; ++round) {
            cudaMemcpyAsync(d, s, bytes, dir == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost);
            cudaEventRecord(a);
            for (int r = 0; r < reps; ++r) cudaMemcpyAsync(d, s, bytes, dir == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost);
            cudaEventRecord(b); cudaEventSynchronize(b);
            float ms; cudaEventElapsedTime(&ms, a, b); ms /= reps;
            printf("%s memcpy        %.3f ms %.1f GB/s\n", dir ? "D2H" : "H2D", ms, bytes / ms / 1e6);
            for (int bps : {1, 2, 4, 8, 16}) {
                float m1 = run<1>(s, d, S, stride, bps, sms, a, b, reps), m2 = run<2>(s, d, S, stride, bps, sms, a, b, reps);
                float m4 = run<4>(s, d, S, stride, bps, sms, a, b, reps), m8 = run<8>(s, d, S, stride, bps, sms, a, b, reps);
                printf("%s bps=%2d  U1 %.1f  U2 %.1f  U4 %.1f  U8 %.1f GB/s\n", dir ? "D2H" : "H2D", bps, bytes / m1 / 1e6, bytes / m2 / 1e6,
                       bytes / m4 / 1e6, bytes / m8 / 1e6);
            }
        }
    }
    printf("err %s\n", cudaGetErrorString(cudaGetLastError()));
    cudaFree(dv); cudaFreeHost(h);
    return 0;
}

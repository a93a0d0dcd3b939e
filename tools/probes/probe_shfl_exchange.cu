// probe_shfl_exchange.cu -- is a lane-pair shuffle cheaper than a shared-memory exchange on sm_100a?
// The 8192-point line transform of the stepper (16 warps per SM, 16 complex values per thread) can end either with a
// third shared-memory exchange followed by the radix-2 stage, or with the radix-2 stage split across lanes l, l ^ 16
// (8 complex values each way: 16 shfl.xor per thread plus lane-parity selects).  Timed per SM:
//   (a) exchange : 16 STS.64 at padpos(16 t + s) and 16 LDS.64 at padpos(t + 512 k) of a 64 KB line, two barriers
//   (b) shuffle  : 16 shfl.xor(16) per thread with the selects of the lane-pair stage
//   (c) neither  : the same arithmetic alone, the floor both share
// One CTA of 512 threads per SM, 148 CTAs.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o probe_shfl_exchange probe_shfl_exchange.cu
#include <cstdio>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)

constexpr int L = 8192, G = 512, ITERS = 2048;
__device__ __forceinline__ int padpos(int p) { return p + (p >> 4); }

// a cheap butterfly that keeps every value live and dependent on the moved ones
__device__ __forceinline__ void mix(float2 (&v)[16])
{
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float2 a = v[i], b = v[i + 8];
        v[i] = make_float2(a.x + b.x, a.y + b.y);
        v[i + 8] = make_float2(a.x - b.x, a.y - b.y);
    }
}

template <int MODE>
__global__ void __launch_bounds__(512, 1) k_probe(float2 *out)
{
    extern __shared__ float2 sm[];
    const int t = threadIdx.x;
    const bool h = (t >> 4) & 1;
    float2 v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = make_float2(t + k, blockIdx.x - k);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it) {
        mix(v);
        if (MODE == 0) {
            float2 *dst = sm + padpos(16 * t);
#pragma unroll
            for (int s = 0; s < 16; ++s) dst[s] = v[s];
            __syncthreads();
            const float2 *src = sm + padpos(t);
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = src[k * (G + G / 16)];
            __syncthreads();
        } else if (MODE == 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float2 r = make_float2(__shfl_xor_sync(0xffffffffu, v[8 + i].x, 16), __shfl_xor_sync(0xffffffffu, v[8 + i].y, 16));
                const float2 e = h ? r : v[i], o = h ? v[i] : r;
                v[i] = e;
                v[8 + i] = o;
            }
        }
    }
    float2 s = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 16; ++k) { s.x += v[k].x; s.y += v[k].y; }
    out[blockIdx.x * blockDim.x + t] = s;
}

template <typename F>
static float time_ms(F f)
{
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    f(); f();
    cudaDeviceSynchronize();
    cudaEventRecord(e0);
    for (int r = 0; r < 10; ++r) f();
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    return ms / 10;
}

int main()
{
    const int blocks = 148, threads = 512, smem = (L + L / 16) * (int)sizeof(float2);
    float2 *out;
    CK(cudaMalloc(&out, sizeof(float2) * blocks * threads));
    CK(cudaFuncSetAttribute(k_probe<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int clk_khz = 0;
    CK(cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0));
    const char *name[3] = {"(a) shared-memory exchange", "(b) 16 shfl.xor + selects ", "(c) arithmetic only       "};
    float ms[3];
    ms[0] = time_ms([&] { k_probe<0><<<blocks, threads, smem>>>(out); });
    ms[1] = time_ms([&] { k_probe<1><<<blocks, threads>>>(out); });
    ms[2] = time_ms([&] { k_probe<2><<<blocks, threads>>>(out); });
    CK(cudaDeviceSynchronize());
    for (int m = 0; m < 3; ++m) {
        const double ns = ms[m] * 1e6 / ITERS, extra = (ms[m] - ms[2]) * 1e6 / ITERS;
        printf("%s: %.3f ms  %.1f ns/iter  %.1f ns/iter over (c)  ~%.0f SM cycles/iter over (c) at %d MHz\n", name[m], ms[m], ns, extra,
               extra * clk_khz * 1e-6, clk_khz / 1000);
    }
    return 0;
}

// Micro-benchmark (B200): cost of parking 12 fp32 per thread for one step in tensor memory (tcgen05.st /
// tcgen05.ld, SASS STTM / LDTM), against keeping them in registers or bouncing them through shared memory
// (STS.128 / LDS.128).  Shape of the fused 3-D pass: 148 CTAs x 384 threads, one CTA per SM; each warp owns
// 128 TMEM columns of its lane quarter (warp w: lanes 32*(w%4), columns (w/4)*128).
// Per step every thread produces 12 values (6 packed pairs), parks them, fetches the 12 parked one step
// earlier and adds them into its accumulators, with WORK independent packed adds in between.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tmem_window tmem_window.cu -lnvidia-ml
#include <cstdio>
#include <cuda_runtime.h>
#include <nvml.h>
typedef unsigned long long u64;
#define THREADS 384
#define STEPS 4096

__device__ __forceinline__ void fadd2(u64& a, u64 b) { asm volatile("add.rn.f32x2 %0, %0, %1;" : "+l"(a) : "l"(b)); }

__device__ __forceinline__ void tm_st12(unsigned taddr, const u64* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"((unsigned)v[0]), "r"((unsigned)(v[0] >> 32)), "r"((unsigned)v[1]),
                    "r"((unsigned)(v[1] >> 32)), "r"((unsigned)v[2]), "r"((unsigned)(v[2] >> 32)),
                    "r"((unsigned)v[3]), "r"((unsigned)(v[3] >> 32)) : "memory");
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};"
                 :: "r"(taddr + 8), "r"((unsigned)v[4]), "r"((unsigned)(v[4] >> 32)), "r"((unsigned)v[5]),
                    "r"((unsigned)(v[5] >> 32)) : "memory");
}

__device__ __forceinline__ void tm_ld12(unsigned taddr, u64* v) {
    unsigned r[12];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]) : "r"(taddr + 8) : "memory");
#pragma unroll
    for (int c = 0; c < 6; ++c) v[c] = ((u64)r[2 * c + 1] << 32) | r[2 * c];
}

__device__ __forceinline__ void sm_st12(unsigned a, const u64* v) {
#pragma unroll
    for (int q = 0; q < 3; ++q)
        asm volatile("st.shared.v2.b64 [%0], {%1,%2};" :: "r"(a + q * 16 * THREADS), "l"(v[2 * q]), "l"(v[2 * q + 1]) : "memory");
}

__device__ __forceinline__ void sm_ld12(unsigned a, u64* v) {
#pragma unroll
    for (int q = 0; q < 3; ++q)
        asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];" : "=l"(v[2 * q]), "=l"(v[2 * q + 1]) : "r"(a + q * 16 * THREADS) : "memory");
}

// MODE 0: registers, 1: tensor memory, 2: shared memory, 3: tensor-memory round-trip latency (one chain)
template <int MODE, int WORK>
__global__ void __launch_bounds__(THREADS, 1) k(float* out, long long* clocks, float seed, int steps) {
    __shared__ unsigned tmem_base;
    __shared__ __align__(16) u64 park[2][3][THREADS][2];       // [slot][quad][thread]: 16 bytes per thread
    const int warp = threadIdx.x / 32;
    if (MODE == 1 || MODE == 3) {
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;"
                         :: "r"((unsigned)__cvta_generic_to_shared(&tmem_base)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    const unsigned tcol = tmem_base + ((unsigned)(32 * (warp % 4)) << 16) + (warp / 4) * 128;
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(&park[0][0][threadIdx.x][0]);
    u64 inc = ((u64)__float_as_uint(seed) << 32) | __float_as_uint(seed);
    u64 acc[6], cur[6], old[6], prev[6], w[WORK > 0 ? WORK : 1];
#pragma unroll
    for (int c = 0; c < 6; ++c) { acc[c] = inc + c + threadIdx.x; old[c] = acc[c]; }
#pragma unroll
    for (int c = 0; c < (WORK > 0 ? WORK : 1); ++c) w[c] = inc + 7 * c;
    if (MODE == 1) tm_st12(tcol + 12, old);
    if (MODE == 2) sm_st12(sbase + 6 * 8 * THREADS, old);
    __syncthreads();
    long long t0 = clock64();
    if (MODE == 3) {
        // dependent chain: store, wait, load, wait, add, ... (one round trip per iteration)
        for (int s = 0; s < steps; ++s) {
            tm_st12(tcol, acc);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tm_ld12(tcol, cur);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            fadd2(acc[0], cur[0]);
        }
    } else {
        for (int s = 0; s < steps; s += 2) {
#pragma unroll
            for (int u = 0; u < 2; ++u) {   // unroll 2: slot of step s is static
#pragma unroll
                for (int c = 0; c < 6; ++c) { cur[c] = acc[c]; fadd2(cur[c], inc); }
                if (MODE == 1) {
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");  // previous step's store
                    tm_ld12(tcol + 12 * (1 - u), prev);                           // parked one step earlier
                    tm_st12(tcol + 12 * u, cur);
                } else if (MODE == 2) {
                    sm_ld12(sbase + (1 - u) * 6 * 8 * THREADS, prev);
                    sm_st12(sbase + u * 6 * 8 * THREADS, cur);
                }
#pragma unroll
                for (int c = 0; c < WORK; ++c) fadd2(w[c], inc);
                if (MODE == 1) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (MODE == 0) {
#pragma unroll
                    for (int c = 0; c < 6; ++c) { prev[c] = old[c]; old[c] = cur[c]; }
                }
#pragma unroll
                for (int c = 0; c < 6; ++c) fadd2(acc[c], prev[c]);
            }
        }
    }
    long long t1 = clock64();
    if (threadIdx.x == 0) clocks[blockIdx.x] = t1 - t0;
    float r = 0;
#pragma unroll
    for (int c = 0; c < 6; ++c) r += __uint_as_float((unsigned)acc[c]) + __uint_as_float((unsigned)(acc[c] >> 32));
#pragma unroll
    for (int c = 0; c < WORK; ++c) r += __uint_as_float((unsigned)w[c]);
    out[blockIdx.x * THREADS + threadIdx.x] = r;
    if (MODE == 1 || MODE == 3) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (warp == 0)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" :: "r"(tmem_base) : "memory");
    }
}

template <int MODE, int WORK>
bool run(const char* what) {
    float* out; long long* clocks;
    cudaMalloc(&out, 148 * THREADS * sizeof(float));
    cudaMalloc(&clocks, 148 * sizeof(long long));
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    k<MODE, WORK><<<148, THREADS>>>(out, clocks, 1.0f, 64);
    cudaDeviceSynchronize();
    cudaEventRecord(e0);
    k<MODE, WORK><<<148, THREADS>>>(out, clocks, 1.0f, STEPS);
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        printf("%-46s failed: %s\n", what, cudaGetErrorString(err));
        return false;
    }
    long long h[148]; cudaMemcpy(h, clocks, sizeof(h), cudaMemcpyDeviceToHost);
    long long mx = 0; double mean = 0;
    for (int b = 0; b < 148; ++b) { mx = h[b] > mx ? h[b] : mx; mean += h[b] / 148.0; }
    printf("%-46s %8.3f ms  %7.2f clocks/step (mean over CTAs)  %7.2f (slowest CTA)\n", what, ms,
           mean / STEPS, (double)mx / STEPS);
    cudaFree(out); cudaFree(clocks);
    return true;
}

int main() {
    cudaDeviceProp p; cudaGetDeviceProperties(&p, 0);
    unsigned mw = 0, clk = 0;
    nvmlDevice_t dev;
    if (nvmlInit() == NVML_SUCCESS && nvmlDeviceGetHandleByIndex(0, &dev) == NVML_SUCCESS) {
        nvmlDeviceGetEnforcedPowerLimit(dev, &mw);
        nvmlDeviceGetMaxClockInfo(dev, NVML_CLOCK_SM, &clk);
    }
    printf("card: %s, %d SMs, power limit %.0f W, max SM clock %u MHz\n", p.name, p.multiProcessorCount, mw / 1000.0, clk);
    printf("148 CTAs x %d threads, %d steps; per step per thread: park 12 fp32, fetch the 12 parked a step earlier\n",
           THREADS, STEPS);
    bool ok = run<0, 0>("registers,     0 extra FADD2") && run<1, 0>("tensor memory, 0 extra FADD2") &&
              run<2, 0>("shared memory, 0 extra FADD2") && run<0, 24>("registers,    24 extra FADD2") &&
              run<1, 24>("tensor memory, 24 extra FADD2") && run<2, 24>("shared memory, 24 extra FADD2") &&
              run<0, 48>("registers,    48 extra FADD2") && run<1, 48>("tensor memory, 48 extra FADD2") &&
              run<2, 48>("shared memory, 48 extra FADD2") &&
              run<3, 0>("tensor memory round trip (st, wait, ld, wait)");
    if (!ok) return 1;
    return 0;
}

// Micro-benchmark behind DESIGN.md section 4 ("128 bytes of DRAM traffic per random 4-byte access"): random single-word
// reads over a table far larger than the L2, one kernel per load flavour.  Run under
//   ncu --metrics dram__bytes_read.sum,lts__t_sectors_srcunit_tex_op_read.sum,lts__t_requests_srcunit_tex_op_read.sum,gpu__time_duration.sum
// to see how many DRAM bytes and L2 sectors ONE access costs for each flavour; without ncu it prints the rate.
//   gather [log2 words = 28] [loads per thread = 64] [L2 fetch granularity limit = 0 (leave)] [policy window: 0 none, 1 streaming, 2 normal]
// Build: nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o scripts/ubench/gather scripts/ubench/gather.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); exit(1); } } while (0)

__device__ __forceinline__ uint32_t mix(uint32_t x) { x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16; return x; }

template <int V>
__device__ __forceinline__ uint32_t load(const uint32_t* p, unsigned long long pol) {
    uint32_t r, a, b, c, d, e, f, g;
    if (V == 0) { asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 1) { asm volatile("ld.global.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 2) { asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol)); return r; }
    if (V == 3) { asm volatile("ld.global.nc.L1::no_allocate.L2::64B.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 4) { asm volatile("ld.global.cg.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 5) { asm volatile("ld.global.cv.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 6) {
        const uint32_t* q = (const uint32_t*)((uintptr_t)p & ~(uintptr_t)15);
        asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r), "=r"(a), "=r"(b), "=r"(c) : "l"(q));
        return r ^ a ^ b ^ c;
    }
    if (V == 7) {
        const uint32_t* q = (const uint32_t*)((uintptr_t)p & ~(uintptr_t)31);
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                     : "=r"(r), "=r"(a), "=r"(b), "=r"(c), "=r"(d), "=r"(e), "=r"(f), "=r"(g) : "l"(q), "l"(pol));
        return r ^ a ^ b ^ c ^ d ^ e ^ f ^ g;
    }
    if (V == 8) {
        const uint32_t* q = (const uint32_t*)((uintptr_t)p & ~(uintptr_t)31);
        asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r), "=r"(a), "=r"(b), "=r"(c), "=r"(d), "=r"(e), "=r"(f), "=r"(g) : "l"(q));
        return r ^ a ^ b ^ c ^ d ^ e ^ f ^ g;
    }
    if (V == 9) { asm volatile("ld.global.lu.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 10) { asm volatile("ld.relaxed.gpu.global.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 11) { asm volatile("ld.global.nc.L1::evict_first.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 12) { asm volatile("ld.global.nc.L1::no_allocate.b8 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    if (V == 13) { asm volatile("ld.global.nc.L1::no_allocate.L2::128B.b32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
    return 0;
}

template <int V, int POL>
__global__ void __launch_bounds__(256) k_gather(const uint32_t* __restrict__ tab, uint32_t mask, int per_thread, uint32_t* out) {
    unsigned long long pol = 0;
    if (POL == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    if (POL == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    if (POL == 3) asm volatile("createpolicy.fractional.L2::evict_unchanged.b64 %0, 1.0;" : "=l"(pol));
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t acc = 0, x = mix(t * 2654435761u + 12345u);
    for (int i = 0; i < per_thread; i += 4) {
        const uint32_t i0 = x & mask, i1 = mix(x + 1u) & mask, i2 = mix(x + 2u) & mask, i3 = mix(x + 3u) & mask;
        const uint32_t a = load<V>(tab + i0, pol), b = load<V>(tab + i1, pol), c = load<V>(tab + i2, pol), d = load<V>(tab + i3, pol);
        acc ^= a ^ b ^ c ^ d;
        x = mix(x + 4u + (acc & 1u));
    }
    if (acc == 0x12345678u) out[0] = acc;
}

template <int V, int POL>
void run(const char* name, const uint32_t* tab, uint32_t mask, int per_thread, uint32_t* out, cudaStream_t st) {
    const int grid = 148 * 16, block = 256;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    k_gather<V, POL><<<grid, block, 0, st>>>(tab, mask, 8, out);          // warm-up (code, TLB)
    CK(cudaEventRecord(e0, st));
    k_gather<V, POL><<<grid, block, 0, st>>>(tab, mask, per_thread, out);
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double n = (double)grid * block * per_thread;
    printf("{\"variant\": \"%s\", \"ms\": %.4f, \"G_loads_per_s\": %.2f}\n", name, ms, n / ms / 1e6);
}

int main(int argc, char** argv) {
    const int lg = argc > 1 ? atoi(argv[1]) : 28, per_thread = argc > 2 ? atoi(argv[2]) : 64;
    const int gran = argc > 3 ? atoi(argv[3]) : 0, window = argc > 4 ? atoi(argv[4]) : 0;
    if (gran) { cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)gran); cudaGetLastError(); }
    size_t g = 0; cudaDeviceGetLimit(&g, cudaLimitMaxL2FetchGranularity);
    const size_t words = (size_t)1 << lg;
    uint32_t *tab, *out;
    CK(cudaMalloc(&tab, words * 4)); CK(cudaMalloc(&out, 64));
    CK(cudaMemset(tab, 0x5A, words * 4));
    cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    if (window) {
        cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
        cudaStreamAttrValue attr; memset(&attr, 0, sizeof(attr));
        attr.accessPolicyWindow.base_ptr = tab;
        attr.accessPolicyWindow.num_bytes = words * 4 < (size_t)prop.accessPolicyMaxWindowSize ? words * 4 : (size_t)prop.accessPolicyMaxWindowSize;
        attr.accessPolicyWindow.hitRatio = 1.0f;
        attr.accessPolicyWindow.hitProp = window == 1 ? cudaAccessPropertyStreaming : cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        CK(cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr));
    }
    printf("{\"table_MiB\": %zu, \"loads_per_thread\": %d, \"l2_fetch_granularity\": %zu, \"policy_window\": %d}\n", words * 4 >> 20, per_thread, g, window);
    const uint32_t mask = (uint32_t)(words - 1);
    run<0, 0>("b32 nc L1::no_allocate (K1 today)", tab, mask, per_thread, out, st);
    run<1, 0>("b32 plain ld.global", tab, mask, per_thread, out, st);
    run<2, 1>("b32 nc no_allocate + L2 evict_first hint", tab, mask, per_thread, out, st);
    run<2, 2>("b32 nc no_allocate + L2 evict_last hint", tab, mask, per_thread, out, st);
    run<2, 3>("b32 nc no_allocate + L2 evict_unchanged hint", tab, mask, per_thread, out, st);
    run<3, 0>("b32 nc no_allocate L2::64B", tab, mask, per_thread, out, st);
    run<13, 0>("b32 nc no_allocate L2::128B", tab, mask, per_thread, out, st);
    run<4, 0>("b32 ld.global.cg", tab, mask, per_thread, out, st);
    run<5, 0>("b32 ld.global.cv", tab, mask, per_thread, out, st);
    run<9, 0>("b32 ld.global.lu", tab, mask, per_thread, out, st);
    run<10, 0>("b32 ld.relaxed.gpu", tab, mask, per_thread, out, st);
    run<11, 0>("b32 nc L1::evict_first", tab, mask, per_thread, out, st);
    run<12, 0>("b8 nc no_allocate", tab, mask, per_thread, out, st);
    run<6, 0>("v4.b32 (16 B) nc no_allocate", tab, mask, per_thread, out, st);
    run<8, 0>("v8.b32 (32 B) nc no_allocate", tab, mask, per_thread, out, st);
    run<7, 1>("v8.b32 (32 B) nc no_allocate + L2 evict_first hint (layout 0's load)", tab, mask, per_thread, out, st);
    return 0;
}

// Shared device/host helpers for libhipr_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <type_traits>
#include "hipr_b200.h"

#ifndef __CUDA_ARCH__
#define HIPR_HOST_ONLY 1
#endif

namespace hipr {

constexpr int kNumSMsB200 = 148;

extern std::atomic<int64_t> g_launches;   // kernels launched by this library (bench.py reads it)

inline int sm_count() {
    static int cached = 0;
    if (cached > 0) return cached;
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return kNumSMsB200;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
        return kNumSMsB200;
    cached = n;
    return n;
}

// cudaFuncSetAttribute is per device: true the first time the calling site runs on the current device
// (one process per GPU is the normal deployment; a process driving several devices must still work).
inline bool first_use_on_device(std::atomic<uint64_t> &mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return true;
    const uint64_t bit = 1ull << (dev & 63);
    return (mask.fetch_or(bit, std::memory_order_relaxed) & bit) == 0;
}

// Returns the launch error (if any) as the ABI's positive code and counts the launch.
inline int after_launch() {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? HIPR_OK : (int)e;
}

#define HIPR_CUDA(expr)                                   \
    do {                                                  \
        cudaError_t _e = (expr);                          \
        if (_e != cudaSuccess) return (int)_e;            \
    } while (0)

// ---------------------------------------------------------------------------------------
// Order-preserving 64-bit key of a double, so a global max is one atomicMax on uint64.
// key(a) < key(b)  <=>  a < b for all non-NaN doubles; key 0 is below every real number.
// ---------------------------------------------------------------------------------------
__host__ __device__ inline uint64_t key_of_double(double v) {
#ifdef __CUDA_ARCH__
    uint64_t b = (uint64_t)__double_as_longlong(v);
#else
    uint64_t b;
    memcpy(&b, &v, 8);
#endif
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double double_of_key(uint64_t k) {
    uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double v;
    memcpy(&v, &b, 8);
    return v;
#endif
}

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP), streaming loads.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes,
                                         uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float ldg_stream(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_stream4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
// Sum of C consecutive floats in shared memory, in float64; sixteen loads are issued before the
// first add so the LDS latency is paid once per batch.
// PAIRS = false: every channel is converted and added in float64 (the float32 result is then the
//   correctly rounded sum).  The float->double conversion runs on the XU pipe at 16 lanes/clk/SM:
//   95 per pixel make XU the busiest pipe of K1 (ncu: 42 %), which K1 can afford (HBM-bound).
// PAIRS = true: channels are added in pairs in float32 first (one rounding of <= 0.5 ulp of a
//   ~S/48 partial, ~6e-9 relative on the total), halving the XU work; used by the fused kernel,
//   whose stencil also needs the XU pipe.
template <bool PAIRS>
__device__ __forceinline__ double sum_channels(const float *__restrict__ p, int C) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int c = 0;
    for (; c + 16 <= C; c += 16) {
        float v[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) v[u] = p[c + u];
        if (PAIRS) {
            a0 += (double)(v[0] + v[1]);
            a1 += (double)(v[2] + v[3]);
            a2 += (double)(v[4] + v[5]);
            a3 += (double)(v[6] + v[7]);
            a0 += (double)(v[8] + v[9]);
            a1 += (double)(v[10] + v[11]);
            a2 += (double)(v[12] + v[13]);
            a3 += (double)(v[14] + v[15]);
        } else {
#pragma unroll
            for (int u = 0; u < 16; u += 4) {
                a0 += (double)v[u];
                a1 += (double)v[u + 1];
                a2 += (double)v[u + 2];
                a3 += (double)v[u + 3];
            }
        }
    }
    if (c + 8 <= C) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = p[c + u];
        if (PAIRS) {
            a0 += (double)(v[0] + v[1]);
            a1 += (double)(v[2] + v[3]);
            a2 += (double)(v[4] + v[5]);
            a3 += (double)(v[6] + v[7]);
        } else {
            a0 += (double)v[0] + (double)v[4];
            a1 += (double)v[1] + (double)v[5];
            a2 += (double)v[2] + (double)v[6];
            a3 += (double)v[3] + (double)v[7];
        }
        c += 8;
    }
    if (PAIRS) {
        for (; c + 2 <= C; c += 2) a0 += (double)(p[c] + p[c + 1]);
        if (c < C) a1 += (double)p[c];
    } else {
        for (; c < C; ++c) a0 += (double)p[c];
    }
    return (a0 + a1) + (a2 + a3);
}

// Raw detector counts -> the float32 value python-bioformats' load_image(rescale=True) hands the
// scripts: image.astype(np.float32) / float(scale), one correctly rounded float32 divide per sample.
template <typename InT>
__device__ __forceinline__ float raw_value(InT v, float scale) {
    return __fdiv_rn((float)v, scale);
}
template <typename InT>
__device__ __forceinline__ double sum_channels_raw(const InT *__restrict__ p, int C, float scale) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int c = 0;
    for (; c + 8 <= C; c += 8) {
        InT v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = p[c + u];
        a0 += (double)raw_value(v[0], scale);
        a1 += (double)raw_value(v[1], scale);
        a2 += (double)raw_value(v[2], scale);
        a3 += (double)raw_value(v[3], scale);
        a0 += (double)raw_value(v[4], scale);
        a1 += (double)raw_value(v[5], scale);
        a2 += (double)raw_value(v[6], scale);
        a3 += (double)raw_value(v[7], scale);
    }
    for (; c < C; ++c) a0 += (double)raw_value(p[c], scale);
    return (a0 + a1) + (a2 + a3);
}

// sum_c p[c] / q[c]: the flat-field divide of syn/..._measurement.py:104 followed by the channel sum
// of :105.  numpy divides in float64; a float64 divide per channel (MUFU.RCP64H + ~10 dependent
// DFMA) made the kernel latency-bound at a third of the HBM rate, so the quotient is formed as
//   v / w = v*r0 * (1 + e + e^2 + O(e^3)),  r0 = RCP(w) in float32 (|e| <= ~1.2e-7),  e = 1 - w*r0
// with v*r0 taken exactly in float64 (two 24-bit significands) and the O(1e-7) correction in
// float32: four float32 roundings (e, e + e^2, v*r0, the fma into the accumulator), each <= 2^-24
// relative, of a correction <= 2^-23 of the term (rcp.approx is within 1 ulp) put a term within
// 2^-45 + 2^-52 = 2.9e-14 of numpy's float64 quotient (tests/test_gpu_quotients.py checks every
// divisor significand), far inside what the fixed-point stencil resolves (4.6e-10 of the image
// range).  One DFMA, three XU operations and four FFMA per channel.
__device__ __forceinline__ float rcp_approx(float w) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(w));   // one MUFU.RCP, <= 1 ulp
    return r;
}
__device__ __forceinline__ void div_accum(float v, float w, double &acc, float &corr) {
    const float r0 = rcp_approx(w);
    const float e = fmaf(-w, r0, 1.0f);          // exact up to one rounding of a ~1e-7 quantity
    const float pf = v * r0;
    corr = fmaf(pf, fmaf(e, e, e), corr);
    acc = fma((double)v, (double)r0, acc);
}
static __device__ __noinline__ double sum_channels_div_exact(const float *__restrict__ p, const float *__restrict__ q, int C) {
    double a = 0.0;
    for (int c = 0; c < C; ++c) a += (double)p[c] / (double)q[c];
    return a;
}
__device__ __forceinline__ double sum_channels_div(const float *__restrict__ p, const float *__restrict__ q, int C) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    float k0 = 0.f, k1 = 0.f, k2 = 0.f, k3 = 0.f;
    int c = 0;
    for (; c + 8 <= C; c += 8) {
        float v[8], w[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            v[u] = p[c + u];
            w[u] = q[c + u];
        }
        div_accum(v[0], w[0], a0, k0);
        div_accum(v[1], w[1], a1, k1);
        div_accum(v[2], w[2], a2, k2);
        div_accum(v[3], w[3], a3, k3);
        div_accum(v[4], w[4], a0, k0);
        div_accum(v[5], w[5], a1, k1);
        div_accum(v[6], w[6], a2, k2);
        div_accum(v[7], w[7], a3, k3);
    }
    for (; c < C; ++c) div_accum(p[c], q[c], a0, k0);
    const double total = ((a0 + a1) + (a2 + a3)) + (double)((k0 + k1) + (k2 + k3));
    // A divisor that is zero, denormal (flushed) or non-finite, or a non-finite numerator, makes r0 or e
    // infinite / NaN and therefore the total non-finite: that pixel is redone with numpy's own float64
    // quotients, channel by channel (never taken on real flat fields).  So is a non-zero total below 2^-90:
    // there the float32 correction terms (<= 2^-23 of a quotient) fall below 2^-126, and each denormal rounding
    // loses up to 2^-150 absolute -- for denormal numerators the whole correction, up to 2^-23 of the total.
    // Above 2^-90 those roundings stay below 2^-52 of the total.  A divisor above 2^126 has its reciprocal
    // flushed to zero: the term becomes 0 instead of ~v * 1e-38 (the exact path, when taken, keeps it).
    const double mag = fabs(total);
    if (!(mag < 1.7e308) || (mag < 0x1p-90 && mag != 0.0)) return sum_channels_div_exact(p, q, C);
    return total;
}

// ---------------------------------------------------------------------------------------
// Grid barrier of the persistent cooperative kernels (K8, K11).  *counter is zeroed before the launch; every CTA
// adds one per barrier and waits until the count reaches its target (gridDim.x per barrier passed so far).  The
// comparison is wrap-safe, so the count may pass 2^32 in a long run.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void grid_barrier(unsigned int *counter, unsigned int &target) {
    __syncthreads();
    target += (unsigned)gridDim.x;
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        while ((int)(ld_acquire_gpu(counter) - target) < 0) {}
    }
    __syncthreads();
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// f(std::integral_constant<int, i>{}) for i = I .. N-1: the index is a constant expression inside f (LDS immediates,
// compile-time register indices)
template <int I, int N, typename F>
__device__ __forceinline__ void static_for(F &&f) {
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}
#endif  // __CUDACC__

}  // namespace hipr

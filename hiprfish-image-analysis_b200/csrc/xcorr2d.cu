// K9: integer registration shifts by a float64 FFT cross-correlation.
//
// Replaces skimage.feature.register_translation(src, target)[0] with upsample_factor=1, space="real", as the
// scripts call it on the excitations' channel-sum images (syn/..._measurement.py:83-85):
//     cc = ifftn(fftn(src) * conj(fftn(target)));  peak = argmax |cc| (numpy's: first NaN, else first maximum)
//     shift = peak, minus the axis length where peak > axis // 2
// H and W are powers of two in [2, 8192].  Every transform is a hand-written radix-2/4 decimation-in-time FFT in
// shared memory, all in float64 (twiddles from sincospi, one table per call in the workspace):
//   xc_rows_forward  per image: load a row (real, optional log(x + eps)), bit-reversed into shared memory, FFT
//   xc_cols          per image: load a column tile, FFT; for the source image store its spectrum F; for a target
//                    image form F * conj(G) in place, bit-reverse it and run the inverse column FFT on chip
//   xc_rows_inverse  per target: inverse row FFT, |cc| / (H W), per-CTA (value, flat index) argmax
//   xc_finish        per target: the final argmax and the wrap rule -> (row, col) float64
// HBM traffic per target image: 8 B/px read + 16 written (rows), 32 read + 16 written (columns: G and F), 16 read
// (+8 written for |cc|) -- the column pass of the forward transform, the spectrum product and the column pass of
// the inverse share one trip through shared memory.
#include <algorithm>
#include <cmath>
#include "hipr_common.cuh"

namespace hipr {

constexpr int XC_MAX_IMG = 8;
constexpr int XC_MAX_N = 8192;
constexpr int XC_THREADS = 256;
constexpr int XC_TILE = 4096;       // complex elements per CTA (64 KB + padding) unless one line is longer

struct XcInputs {
    const void *img[XC_MAX_IMG];    // real (H, W) images of the input dtype
};

__device__ __forceinline__ double2 c_add(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 c_sub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 c_mul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ int bit_reverse(int k, int logn) { return (int)(__brev((unsigned)k) >> (32 - logn)); }

// tw[j] = exp(-2 pi i j / nt), j < nt / 2
__global__ void xc_twiddles(double2 *__restrict__ tw, int nt) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nt / 2) {
        double s, c;
        sincospi(-2.0 * (double)j / (double)nt, &s, &c);
        tw[j] = make_double2(c, s);
    }
}

// In-place FFT of `lines` lines of length n = 2^logn in shared memory (line l at s + l * stride), input in
// bit-reversed order, output in natural order.  Stages are taken two at a time (a radix-4 butterfly built from two
// radix-2 stages: no barrier between them), after one plain radix-2 stage when logn is odd.  INV: exp(+2 pi i ...).
template <bool INV>
__device__ void fft_lines(double2 *s, int logn, int stride, int lines, const double2 *__restrict__ tw, int lognt) {
    const int n = 1 << logn;
    int m = 1;
    if (logn & 1) {
        for (int q = threadIdx.x; q < lines << (logn - 1); q += blockDim.x) {
            double2 *p = s + (q >> (logn - 1)) * stride + 2 * (q & ((n >> 1) - 1));
            const double2 a = p[0], b = p[1];
            p[0] = c_add(a, b);
            p[1] = c_sub(a, b);
        }
        __syncthreads();
        m = 2;
    }
    for (; m < n; m <<= 2) {
        const int lm = __ffs(m) - 1;
        for (int q = threadIdx.x; q < lines << (logn - 2); q += blockDim.x) {
            const int r = q & ((n >> 2) - 1);
            const int j = r & (m - 1);
            double2 *p = s + (q >> (logn - 2)) * stride + ((r - j) << 2) + j;
            double2 w1 = __ldg(tw + (j << (lognt - lm - 1)));     // exp(-2 pi i j / 2m)
            double2 w2 = __ldg(tw + (j << (lognt - lm - 2)));     // exp(-2 pi i j / 4m)
            if (INV) { w1.y = -w1.y; w2.y = -w2.y; }
            const double2 w3 = INV ? make_double2(-w2.y, w2.x) : make_double2(w2.y, -w2.x);   // w2 * (-+i)
            double2 a0 = p[0], a1 = p[m], a2 = p[2 * m], a3 = p[3 * m];
            double2 t = c_mul(w1, a1);
            a1 = c_sub(a0, t);
            a0 = c_add(a0, t);
            t = c_mul(w1, a3);
            a3 = c_sub(a2, t);
            a2 = c_add(a2, t);
            t = c_mul(w2, a2);
            p[0] = c_add(a0, t);
            p[2 * m] = c_sub(a0, t);
            t = c_mul(w3, a3);
            p[m] = c_add(a1, t);
            p[3 * m] = c_sub(a1, t);
        }
        __syncthreads();
    }
}

// ---- pass 1: real rows -> complex row spectra.  grid (H / lines, n_images).
template <typename T>
__global__ void __launch_bounds__(XC_THREADS)
xc_rows_forward(const __grid_constant__ XcInputs in, int logh, int logw, int lines, int transform, double eps,
                const double2 *__restrict__ tw, int lognt, double2 *__restrict__ spec) {
    extern __shared__ double2 xc_smem[];
    const int W = 1 << logw, stride = W + 1;
    const int64_t hw = (int64_t)1 << (logh + logw);
    const T *src = static_cast<const T *>(in.img[blockIdx.y]) + (int64_t)blockIdx.x * lines * W;
    for (int i = threadIdx.x; i < lines * W; i += blockDim.x) {
        const int l = i >> logw, k = i & (W - 1);
        double v = (double)src[i];
        if (transform == 1) v = log(v + eps);
        xc_smem[l * stride + bit_reverse(k, logw)] = make_double2(v, 0.0);
    }
    __syncthreads();
    fft_lines<false>(xc_smem, logw, stride, lines, tw, lognt);
    double2 *dst = spec + blockIdx.y * hw + (int64_t)blockIdx.x * lines * W;
    for (int i = threadIdx.x; i < lines * W; i += blockDim.x) dst[i] = xc_smem[(i >> logw) * stride + (i & (W - 1))];
}

// ---- pass 2: column FFTs of a tile of `lines` adjacent columns.  grid (W / lines, n).  Image blockIdx.y + first.
// CORRELATE: spec[img] <- inverse column FFT of F * conj(G), F = spec[0] (complete: stream-ordered after the
// source's own column pass), G = the forward column FFT of spec[img]; else spec[img] <- forward column FFT.
template <bool CORRELATE>
__global__ void __launch_bounds__(XC_THREADS)
xc_cols(int logh, int logw, int lines, int first, const double2 *__restrict__ tw, int lognt, double2 *spec) {
    extern __shared__ double2 xc_smem[];
    const int H = 1 << logh, W = 1 << logw, stride = H + 1;
    const int logl = __ffs(lines) - 1;
    const int64_t hw = (int64_t)1 << (logh + logw);
    const int c0 = blockIdx.x * lines;
    double2 *col = spec + (blockIdx.y + first) * hw + c0;
    for (int i = threadIdx.x; i < lines * H; i += blockDim.x) {
        const int l = i & (lines - 1), k = i >> logl;
        xc_smem[l * stride + bit_reverse(k, logh)] = col[(int64_t)k * W + l];
    }
    __syncthreads();
    fft_lines<false>(xc_smem, logh, stride, lines, tw, lognt);
    if (CORRELATE) {
        const double2 *f = spec + c0;
        for (int i = threadIdx.x; i < lines * H; i += blockDim.x) {
            const int l = i & (lines - 1), k = i >> logl;
            double2 g = xc_smem[l * stride + k];
            g.y = -g.y;
            xc_smem[l * stride + k] = c_mul(f[(int64_t)k * W + l], g);
        }
        __syncthreads();
        // bit-reversal permutation in place: the owner of the smaller index of each pair swaps it
        for (int i = threadIdx.x; i < lines * H; i += blockDim.x) {
            const int l = i >> logh, k = i & (H - 1), kr = bit_reverse(k, logh);
            if (k < kr) {
                double2 *p = xc_smem + l * stride;
                const double2 a = p[k];
                p[k] = p[kr];
                p[kr] = a;
            }
        }
        __syncthreads();
        fft_lines<true>(xc_smem, logh, stride, lines, tw, lognt);
    }
    for (int i = threadIdx.x; i < lines * H; i += blockDim.x) {
        const int l = i & (lines - 1), k = i >> logl;
        col[(int64_t)k * W + l] = xc_smem[l * stride + k];
    }
}

// numpy's argmax order on |cc|: a NaN beats every number, a larger value beats a smaller one, ties (and NaN
// against NaN) go to the lower flat index
__device__ __forceinline__ bool xc_better(double va, long long ia, double vb, long long ib) {
    if (isnan(va)) return !isnan(vb) || ia < ib;
    if (isnan(vb)) return false;
    return va > vb || (va == vb && ia < ib);
}

__device__ __forceinline__ void xc_block_argmax(double &v, long long &idx, double *red_v, long long *red_i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (xc_better(ov, oi, v, idx)) { v = ov; idx = oi; }
    }
    const int warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    __syncthreads();              // red_* may alias the FFT buffer
    if ((threadIdx.x & 31) == 0) { red_v[warp] = v; red_i[warp] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < nwarps; ++w)
            if (xc_better(red_v[w], red_i[w], v, idx)) { v = red_v[w]; idx = red_i[w]; }
    }
}

// ---- pass 3: inverse row FFTs of target spec[1 + blockIdx.y], |cc| and the per-CTA argmax.  grid (H / lines, n-1).
__global__ void __launch_bounds__(XC_THREADS)
xc_rows_inverse(int logh, int logw, int lines, const double2 *__restrict__ tw, int lognt,
                const double2 *__restrict__ spec, double *__restrict__ corr, double2 *__restrict__ partial) {
    extern __shared__ double2 xc_smem[];
    const int W = 1 << logw, stride = W + 1;
    const int64_t hw = (int64_t)1 << (logh + logw);
    const int64_t row0 = (int64_t)blockIdx.x * lines * W;
    const double2 *src = spec + (blockIdx.y + 1) * hw + row0;
    for (int i = threadIdx.x; i < lines * W; i += blockDim.x)
        xc_smem[(i >> logw) * stride + bit_reverse(i & (W - 1), logw)] = src[i];
    __syncthreads();
    fft_lines<true>(xc_smem, logw, stride, lines, tw, lognt);
    const double scale = 1.0 / (double)hw;          // numpy's ifftn normalisation: a power of two, exact
    double best = -INFINITY;
    long long best_i = 0x7fffffffffffffffll;
    for (int i = threadIdx.x; i < lines * W; i += blockDim.x) {
        const double2 c = xc_smem[(i >> logw) * stride + (i & (W - 1))];
        const double a = hypot(c.x, c.y) * scale;
        if (corr != nullptr) corr[row0 + i] = a;
        if (xc_better(a, row0 + i, best, best_i)) { best = a; best_i = row0 + i; }
    }
    double *red_v = reinterpret_cast<double *>(xc_smem);
    xc_block_argmax(best, best_i, red_v, reinterpret_cast<long long *>(red_v + 32));
    if (threadIdx.x == 0)
        partial[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = make_double2(best, __longlong_as_double(best_i));
}

// ---- final argmax over the CTAs of pass 3 and the wrap rule.  grid (n - 1).
__global__ void __launch_bounds__(XC_THREADS)
xc_finish(const double2 *__restrict__ partial, int nparts, int logh, int logw, double *__restrict__ shifts) {
    __shared__ double red_v[32];
    __shared__ long long red_i[32];
    double best = -INFINITY;
    long long best_i = 0x7fffffffffffffffll;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        const double2 p = partial[(int64_t)blockIdx.x * nparts + i];
        const long long pi = __double_as_longlong(p.y);
        if (xc_better(p.x, pi, best, best_i)) { best = p.x; best_i = pi; }
    }
    xc_block_argmax(best, best_i, red_v, red_i);
    if (threadIdx.x == 0) {
        const int H = 1 << logh, W = 1 << logw;
        int r = (int)(best_i >> logw), c = (int)(best_i & (W - 1));
        if (r > H / 2) r -= H;                       // np.fix(n / 2) == n // 2: a peak at exactly n / 2 stays +n / 2
        if (c > W / 2) c -= W;
        shifts[2 * blockIdx.x] = (double)r;
        shifts[2 * blockIdx.x + 1] = (double)c;
    }
}

static int xc_log2(int n) {
    if (n < 2 || n > XC_MAX_N || (n & (n - 1))) return -1;
    int l = 0;
    while ((1 << l) < n) ++l;
    return l;
}

struct XcLayout {
    int64_t tw, partial, sums, spec, total;   // byte offsets in the workspace
};

static int xc_layout(int H, int W, int n, XcLayout *lay) {
    if (xc_log2(H) < 0 || xc_log2(W) < 0) return HIPR_E_UNSUPPORTED;
    if (n < 1) return HIPR_E_ARG;
    if (n > XC_MAX_IMG) return HIPR_E_RANGE;
    auto up = [](int64_t b) { return (b + 255) & ~(int64_t)255; };
    const int64_t hw = (int64_t)H * W;
    lay->tw = 0;
    lay->partial = up((int64_t)XC_MAX_N / 2 * 16);
    lay->sums = lay->partial + up((int64_t)n * H * 16);
    lay->spec = lay->sums + up(n * hw * 8);
    lay->total = lay->spec + n * hw * 16;
    return HIPR_OK;
}

static int xc_lines(int n_line, int n_lines) {
    int l = n_line >= XC_TILE ? 1 : XC_TILE / n_line;
    return l < n_lines ? l : n_lines;
}

// The whole chain for n real images of dtype on the device: shifts of images 1 .. n-1 against image 0, written to
// shifts_dev[2 (i - 1) + {0, 1}]; corr_dev (n == 2 only) receives |cc|.
static int xc_run(const XcInputs &in, int dtype, int n, int H, int W, int transform, double eps, char *work,
                  const XcLayout &lay, double *shifts_dev, double *corr_dev, cudaStream_t st) {
    const int logh = xc_log2(H), logw = xc_log2(W);
    const int nt = H > W ? H : W, lognt = logh > logw ? logh : logw;
    double2 *tw = reinterpret_cast<double2 *>(work + lay.tw);
    double2 *partial = reinterpret_cast<double2 *>(work + lay.partial);
    double2 *spec = reinterpret_cast<double2 *>(work + lay.spec);
    const int lr = xc_lines(W, H), lc = xc_lines(H, W);
    // (at least 512 B: xc_rows_inverse reuses the buffer for its 32 + 32 reduction slots)
    const size_t smem_r = std::max<size_t>((size_t)lr * (W + 1) * sizeof(double2), 512);
    const size_t smem_c = (size_t)lc * (H + 1) * sizeof(double2);
    const int smem_max = (XC_TILE + XC_MAX_N) * (int)sizeof(double2);
    static std::atomic<uint64_t> attr_once;
    if (first_use_on_device(attr_once)) {
        HIPR_CUDA(cudaFuncSetAttribute(xc_rows_forward<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        HIPR_CUDA(cudaFuncSetAttribute(xc_rows_forward<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        HIPR_CUDA(cudaFuncSetAttribute(xc_cols<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        HIPR_CUDA(cudaFuncSetAttribute(xc_cols<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        HIPR_CUDA(cudaFuncSetAttribute(xc_rows_inverse, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    }
    int rc;
    xc_twiddles<<<(nt / 2 + 255) / 256, 256, 0, st>>>(tw, nt);
    if ((rc = after_launch()) != HIPR_OK) return rc;
    const dim3 grid_r(H / lr, n), grid_c(W / lc, 1), grid_ct(W / lc, n - 1), grid_ri(H / lr, n - 1);
    if (dtype == HIPR_F32)
        xc_rows_forward<float><<<grid_r, XC_THREADS, smem_r, st>>>(in, logh, logw, lr, transform, eps, tw, lognt, spec);
    else
        xc_rows_forward<double><<<grid_r, XC_THREADS, smem_r, st>>>(in, logh, logw, lr, transform, eps, tw, lognt, spec);
    if ((rc = after_launch()) != HIPR_OK) return rc;
    xc_cols<false><<<grid_c, XC_THREADS, smem_c, st>>>(logh, logw, lc, 0, tw, lognt, spec);
    if ((rc = after_launch()) != HIPR_OK) return rc;
    xc_cols<true><<<grid_ct, XC_THREADS, smem_c, st>>>(logh, logw, lc, 1, tw, lognt, spec);
    if ((rc = after_launch()) != HIPR_OK) return rc;
    xc_rows_inverse<<<grid_ri, XC_THREADS, smem_r, st>>>(logh, logw, lr, tw, lognt, spec, corr_dev, partial);
    if ((rc = after_launch()) != HIPR_OK) return rc;
    xc_finish<<<n - 1, XC_THREADS, 0, st>>>(partial, H / lr, logh, logw, shifts_dev);
    return after_launch();
}

}  // namespace hipr

using namespace hipr;

extern "C" int64_t hipr_xcorr2d_workspace_bytes(int H, int W, int n_images) {
    XcLayout lay;
    const int rc = xc_layout(H, W, n_images, &lay);
    return rc != HIPR_OK ? rc : lay.total;
}

extern "C" int hipr_register_translation_2d(const void *src_dev, const void *target_dev, int dtype, int H, int W,
                                            void *work_dev, int64_t work_bytes, double *shift_dev, double *corr_dev,
                                            void *stream) {
    if (!src_dev || !target_dev || !work_dev || !shift_dev || H <= 0 || W <= 0) return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    const uintptr_t elem = dtype == HIPR_F32 ? 3u : 7u;
    if ((((uintptr_t)src_dev) & elem) || (((uintptr_t)target_dev) & elem) || (((uintptr_t)work_dev) & 15u) ||
        (((uintptr_t)shift_dev) & 7u) || (((uintptr_t)corr_dev) & 7u))
        return HIPR_E_ALIGN;
    XcLayout lay;
    int rc = xc_layout(H, W, 2, &lay);
    if (rc != HIPR_OK) return rc;
    if (work_bytes < lay.total) return HIPR_E_RANGE;
    XcInputs in = {};
    in.img[0] = src_dev;
    in.img[1] = target_dev;
    return xc_run(in, dtype, 2, H, W, 0, 0.0, static_cast<char *>(work_dev), lay, shift_dev, corr_dev,
                  (cudaStream_t)stream);
}

extern "C" int hipr_excitation_shifts(const float *const *stacks_dev, const int32_t *chans, int n_stacks, int H, int W,
                                      int transform, double eps, void *work_dev, int64_t work_bytes, double *shifts_dev,
                                      void *stream) {
    if (!stacks_dev || !chans || !work_dev || !shifts_dev || n_stacks <= 0 || H <= 0 || W <= 0) return HIPR_E_ARG;
    if (transform != 0 && transform != 1) return HIPR_E_ARG;
    if ((((uintptr_t)work_dev) & 15u) || (((uintptr_t)shifts_dev) & 7u)) return HIPR_E_ALIGN;
    for (int e = 0; e < n_stacks; ++e)
        if (!stacks_dev[e] || chans[e] <= 0) return HIPR_E_ARG;
    XcLayout lay;
    int rc = xc_layout(H, W, n_stacks, &lay);
    if (rc != HIPR_OK) return rc;
    if (work_bytes < lay.total) return HIPR_E_RANGE;
    cudaStream_t st = (cudaStream_t)stream;
    char *work = static_cast<char *>(work_dev);
    HIPR_CUDA(cudaMemsetAsync(shifts_dev, 0, 2 * sizeof(double), st));     // the first excitation is the reference
    if (n_stacks == 1) return HIPR_OK;
    const int64_t hw = (int64_t)H * W;
    double *sums = reinterpret_cast<double *>(work + lay.sums);
    XcInputs in = {};
    for (int e = 0; e < n_stacks; ++e) {
        if ((rc = hipr_chansum(stacks_dev[e], nullptr, hw, chans[e], sums + e * hw, HIPR_F64, nullptr, stream)) != HIPR_OK)
            return rc;
        in.img[e] = sums + e * hw;
    }
    return xc_run(in, HIPR_F64, n_stacks, H, W, transform, eps, work, lay, shifts_dev + 2, nullptr, st);
}

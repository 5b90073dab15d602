// K3q: the 2-D stencil + epilogue on a 31-bit FIXED-POINT copy of the sum image.
//
// Why: the score is (centre - min) / (max - min) along each line, and on real data the line
// range is ~1/10 of the value, so any rounding of the sum image is amplified ~10-20x.  A
// float32 sum image (6e-8 relative) lands at ~6e-6 in the score -- outside the 1e-5 parity gate
// on some pixels -- and a float64 stencil costs 3-4x the instructions (no DMNMX on sm_100).
// Instead the tile loader maps the float64 channel sums onto the 31-bit fixed-point grid of
// lne_fixed.cuh, with the global min / max that K1 produced or the tile's own.  The 11-sample
// min / max run on FMNMX3 exactly as a float kernel would -- but every min, max and difference is
// EXACT; the only roundings left are two int->float conversions and one divide per line (~1e-7).
// Quantisation step: (max - min) * 4.7e-10.
//
// With the pinned (11, 9) table the sample offsets are compile-time immediates of the LDS
// instructions (baked_tables.cuh); any other 11x9 table takes the parameter-bank variant.
#include "hipr_common.cuh"
#include "lne_math.cuh"
#include "lne_fixed.cuh"

namespace hipr {

constexpr int Q_TW = 32, Q_TH = 32, Q_P = 11, Q_R = 9, Q_HALF = 5;
constexpr int Q_SW = Q_TW + Q_P - 1;  // 42
constexpr int Q_SH = Q_TH + Q_P - 1;  // 42

struct TableQ {
    int off[Q_R * Q_P];  // dy * Q_SW + dx
};

// T and LI are compile-time, so the baked offset is a constant expression (an LDS immediate)
template <bool BAKED, int T, int LI>
__device__ __forceinline__ int q_off(const TableQ &tab) {
    if constexpr (BAKED) {
        constexpr int off = baked2d_off<Q_SW>(T, LI);
        return off;
    } else {
        return tab.off[T * Q_P + LI];
    }
}

// Marked pixels (~0.3 % of a synthetic field of view, see the bound in lne_fixed.cuh) are recomputed from the float64
// image by lne2d_refine_kernel, which packs them densely (refining inside the stencil CTA was measured slower: its
// shared-memory footprint and its thinly populated warps kept the stencil from running beside the channel sum of the
// next field of view; a list in global memory needs an allocation per call).
constexpr int Q_RPIX = 28;     // marked pixels per refinement round of a CTA: 28 * 9 = 252 (pixel, line) pairs

// n / d to ~1e-14 relative without the float64 divide subroutine: float32 reciprocal + one Newton step in float64
// (q0 = n * rc, q = q0 + (n - q0 * d) * rc has relative error eps_rc^2).  0 / 0 -> NaN, as the true quotient.
__device__ __forceinline__ double q_fast_div(double n, double d) {
    const double rc = (double)__fdividef(1.0f, (float)d);
    const double q0 = n * rc;
    return fma(fma(-q0, d, n), rc, q0);
}

// inv[t] = 1 / (range of line t in grid units) = e_t
template <int FLAVOUR, bool REFINE>
__device__ __forceinline__ float q_reduce(float (&r)[Q_R], const float (&inv)[Q_R]) {
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < Q_R; ++i) sum += r[i];
    const float mean = sum * (1.0f / Q_R);
    float r0[Q_R];                     // line order, for the refinement test
    if (REFINE) {
#pragma unroll
        for (int i = 0; i < Q_R; ++i) r0[i] = r[i];
    }
    sort_network<float, Q_R>(r);
    const float lq = r[2], uq = r[6];  // np.percentile(.., 25 / 75) of 9 values: order statistics 2 and 6
    float A, B;
    bool unit;
    const float factor = q_factor<FLAVOUR>(lq, uq, A, B, unit);
    if (REFINE) {
        // First with e_max for the e of every line (cheap, passes ~97 % of the pixels); the rest look up the e of the
        // lines that gave lq and uq and sum the exact mean term.
        float e_max = inv[0];
#pragma unroll
        for (int i = 1; i < Q_R; ++i) e_max = fmaxf(e_max, inv[i]);
        bool mark = q_mark<true>(unit, mean, q_err(lq, e_max), q_err(uq, e_max), fmaf(mean, e_max, e_max), A, B);
        if (mark) {
            // exact terms: d_mean = sum over the lines of their bound / 9, e of the lines that gave lq and uq (ties: the
            // largest)
            float d_sum = 0.f, e_lq = 0.f, e_uq = 0.f;
#pragma unroll
            for (int i = 0; i < Q_R; ++i) {
                d_sum += q_err(r0[i], inv[i]);
                e_lq = (r0[i] == lq) ? fmaxf(e_lq, inv[i]) : e_lq;
                e_uq = (r0[i] == uq) ? fmaxf(e_uq, inv[i]) : e_uq;
            }
            const float d_mean = d_sum * (1.0f / Q_R);
            mark = q_mark<true>(unit, mean, q_err(lq, e_lq), q_err(uq, e_uq), d_mean, A, B);
        }
        if (mark) return Q_SENTINEL;
    }
    return mean * factor;
}

template <typename SrcT, int FLAVOUR, bool BAKED, bool REFINE>
__global__ void __launch_bounds__(256)
lne2d_q_kernel(const SrcT *__restrict__ img, int Hs, int Ws, int64_t ld, int src_off, int y_begin, int H, int W,
               const __grid_constant__ TableQ tab, const unsigned long long *__restrict__ range,
               float *__restrict__ out) {
    __shared__ __align__(16) float tile[Q_SH * Q_SW];
    __shared__ double red[16];
    const int x0 = blockIdx.x * Q_TW, y0 = y_begin + blockIdx.y * Q_TH;
    // one pass over the tile: each thread keeps its (at most 7) samples in registers, so the
    // tile-local range costs no second read
    constexpr int PER = (Q_SH * Q_SW + 255) / 256;
    double vals[PER];
    double vmax = -__longlong_as_double(0x7ff0000000000000ll), vmin = -vmax;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        const int i = threadIdx.x + 256 * k;
        vals[k] = 0.0;
        if (i < Q_SH * Q_SW) {
            const int ly = i / Q_SW, lx = i - ly * Q_SW;
            const int sy = min(max(y0 + ly - Q_HALF + src_off, 0), Hs - 1);
            const int sx = min(max(x0 + lx - Q_HALF + src_off, 0), Ws - 1);
            double v = (double)img[(int64_t)sy * ld + sx];
            if (v != v) v = 0.0;  // nan_to_num; NaN is not representable in fixed point (see DESIGN.md)
            vals[k] = v;
            vmax = fmax(vmax, v);
            vmin = fmin(vmin, v);
        }
    }
    if (range != nullptr) {
        vmax = double_of_key(range[0]);
        vmin = double_of_key(range[1]);
    } else {
        // LOCAL range: F1/F2 are invariant to any affine map, so the tile's own min/max serve (and
        // give a finer grid); the stencil then does not depend on a global reduction
        block8_minmax(vmax, vmin, red, threadIdx.x, [] { __syncthreads(); });
    }
    const double K = q_scale(vmax, vmin);
    const float eps_q = q_eps(vmax, K);
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        const int i = threadIdx.x + 256 * k;
        if (i < Q_SH * Q_SW) tile[i] = q_encode(vals[k], vmin, K);
    }
    __syncthreads();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll 1
    for (int k = 0; k < Q_TH / 8; ++k) {
        const int py = ty + 8 * k;
        const int x = x0 + tx, y = y0 + py;
        if (x >= W || y >= H) continue;
        const float *base = tile + py * Q_SW + tx;
        float r[Q_R], e[Q_R];
        static_for<0, Q_R>([&](auto tc) {
            constexpr int t = decltype(tc)::value;
            float mn = base[q_off<BAKED, t, 0>(tab)], mx = mn;
            static_for<1, Q_P>([&](auto lc) {
                constexpr int li = decltype(lc)::value;
                const float s = base[q_off<BAKED, t, li>(tab)];
                mn = fminf(mn, s);
                mx = fmaxf(mx, s);
            });
            r[t] = q_line<FLAVOUR>(base[q_off<BAKED, t, Q_HALF>(tab)], mn, mx, eps_q, &e[t]);
        });
        out[(int64_t)y * W + x] = q_reduce<FLAVOUR, REFINE>(r, e);   // Q_SENTINEL where marked
    }
}

// Refinement of the marked pixels from the source image in float64 (the arithmetic of the float64 stencil,
// csrc/lne2d.cu, with the fixed-point loader's NaN -> 0 and edge clamp).  A CTA scans a 128 x 32 region of the score
// map for the sentinel and collects the positions in shared memory, then takes 28 of them per round: phase A gives
// every (pixel, line) pair a thread -- 11 samples straight from global memory (the image is L2-resident), min / max,
// one quotient -- and parks the nine line values per pixel in shared memory; phase B gives every pixel one thread
// for the mean / quartile epilogue.  No workspace, no global atomics.
constexpr int RF_W = 128, RF_H = 32;

template <typename SrcT, int FLAVOUR>
__global__ void __launch_bounds__(256)
lne2d_refine_kernel(const SrcT *__restrict__ img, int Hs, int Ws, int64_t ld, int src_off, int y_begin, int H, int W,
                    const __grid_constant__ TableQ tab /* dy * Q_SW + dx */, const unsigned long long *__restrict__ range,
                    float *__restrict__ out) {
    __shared__ double rbuf[Q_RPIX][Q_R];
    __shared__ unsigned short marked[RF_W * RF_H];
    __shared__ unsigned int n_marked;
    const int x0 = blockIdx.x * RF_W, y0 = y_begin + blockIdx.y * RF_H;
    if (threadIdx.x == 0) n_marked = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < RF_W * RF_H; i += 256) {
        const int py = i / RF_W, px = i - py * RF_W;
        const int x = x0 + px, y = y0 + py;
        if (x < W && y < H && out[(int64_t)y * W + x] == Q_SENTINEL) marked[atomicAdd(&n_marked, 1u)] = (unsigned short)i;
    }
    __syncthreads();
    const int n = (int)n_marked;
    if (n == 0) return;
    // F3: the reference adds 1e-8 to the range of the image already divided by its max
    const double eps = (range != nullptr) ? 1e-8 * fabs(double_of_key(range[0])) : 1e-8;
    for (int j0 = 0; j0 < n; j0 += Q_RPIX) {
        const int nj = min(Q_RPIX, n - j0);
        if ((int)threadIdx.x < nj * Q_R) {
            const int j = threadIdx.x / Q_R, t = threadIdx.x - j * Q_R;
            const int i = marked[j0 + j];
            const int y = y0 + i / RF_W, x = x0 + i % RF_W;
            const int by = y - Q_HALF + src_off, bx = x - Q_HALF + src_off;     // patch origin in the source image
            double v[Q_P];
#pragma unroll
            for (int li = 0; li < Q_P; ++li) {
                const int o = tab.off[t * Q_P + li];
                const int dy = o / Q_SW, dx = o - dy * Q_SW;
                const int sy = min(max(by + dy, 0), Hs - 1), sx = min(max(bx + dx, 0), Ws - 1);
                const double s = (double)img[(int64_t)sy * ld + sx];
                v[li] = (s != s) ? 0.0 : s;
            }
            double mn = v[0], mx = v[0];
#pragma unroll
            for (int li = 1; li < Q_P; ++li) {
                mn = fmin(mn, v[li]);
                mx = fmax(mx, v[li]);
            }
            const double den = q_den<FLAVOUR>(mx - mn, eps);
            rbuf[j][t] = q_fast_div(v[Q_HALF] - mn, den);
        }
        __syncthreads();
        if ((int)threadIdx.x < nj) {
            const int j = threadIdx.x;
            double rr[Q_R];
            double sum = 0.0;
#pragma unroll
            for (int t = 0; t < Q_R; ++t) {
                rr[t] = rbuf[j][t];
                sum += rr[t];
            }
            const double mean = sum * (1.0 / Q_R);
            sort_network<double, Q_R>(rr);
            const double lq = rr[2], uq = rr[6];
            double factor;
            if (FLAVOUR == HIPR_FLAVOUR_F1) factor = (uq > 0.0) ? q_fast_div(2.0 * lq + 1e-8, uq + lq + 1e-8) : 1.0;
            else if (FLAVOUR == HIPR_FLAVOUR_F2 || FLAVOUR == HIPR_FLAVOUR_ME2) factor = (uq + lq == 0.0) ? 1.0 : q_fast_div(2.0 * lq, uq + lq);
            else factor = q_fast_div(2.0 * lq + 1e-8, uq + lq + 1e-8);
            const int i = marked[j0 + j];
            out[(int64_t)(y0 + i / RF_W) * W + (x0 + i % RF_W)] = (float)(mean * factor);
        }
        __syncthreads();
    }
}

// mode: refine_mode("HIPR_LNE2D_REFINE"); without the refinement the fixed-point result alone holds rtol 1e-5 + atol 5e-7
template <typename SrcT, bool BAKED>
static int lne2d_q_launch(const SrcT *img, int Hs, int Ws, int64_t ld, int src_off, int y_begin, int H, int W,
                          const TableQ &tab, int flavour, const unsigned long long *range, float *out, int mode,
                          cudaStream_t st) {
    // rows [y_begin, H) of the output are computed
    dim3 grid((W + Q_TW - 1) / Q_TW, (H - y_begin + Q_TH - 1) / Q_TH);
    dim3 grid_rf((W + RF_W - 1) / RF_W, (H - y_begin + RF_H - 1) / RF_H);
    const bool refine = mode != 0;
#define HIPR_Q_LAUNCH(F)                                                                                                    \
    if (refine) {                                                                                                           \
        lne2d_q_kernel<SrcT, F, BAKED, true><<<grid, 256, 0, st>>>(img, Hs, Ws, ld, src_off, y_begin, H, W, tab, range, out); \
        if (mode == 1) {                                                                                                    \
            g_launches.fetch_add(1, std::memory_order_relaxed);                                                             \
            lne2d_refine_kernel<SrcT, F><<<grid_rf, 256, 0, st>>>(img, Hs, Ws, ld, src_off, y_begin, H, W, tab, range, out); \
        }                                                                                                                   \
    } else {                                                                                                                \
        lne2d_q_kernel<SrcT, F, BAKED, false><<<grid, 256, 0, st>>>(img, Hs, Ws, ld, src_off, y_begin, H, W, tab, range, out); \
    }
    switch (flavour) {
        case HIPR_FLAVOUR_F1: HIPR_Q_LAUNCH(HIPR_FLAVOUR_F1) break;
        case HIPR_FLAVOUR_F2: HIPR_Q_LAUNCH(HIPR_FLAVOUR_F2) break;
        case HIPR_FLAVOUR_F3: HIPR_Q_LAUNCH(HIPR_FLAVOUR_F3) break;
        default:
            return HIPR_E_FLAVOUR;
    }
#undef HIPR_Q_LAUNCH
    return after_launch();
}

}  // namespace hipr

namespace hipr {
// rows [y_begin, y_end) of the score of an UNPADDED (padded == 0) or padded image; range_dev NULL =
// tile-local quantisation (F1 / F2 only)
int lne2d_q_rows(const void *image_dev, int Hs, int Ws, int64_t ld, int padded, int dtype, const int32_t *table_host,
                 int flavour, const uint64_t *range_dev, float *out_dev, int y_begin, int y_end, cudaStream_t st) {
    const int H = padded ? Hs - (Q_P - 1) : Hs, W = padded ? Ws - (Q_P - 1) : Ws;
    const int src_off = padded ? Q_HALF : 0;
    if (H < 1 || W < 1) return HIPR_E_PATCH;
    if (y_begin < 0 || y_end > H || y_begin >= y_end) return HIPR_E_ARG;
    if (!range_dev && flavour != HIPR_FLAVOUR_F1 && flavour != HIPR_FLAVOUR_F2) return HIPR_E_FLAVOUR;
    TableQ tab;
    bool baked = true;
    for (int i = 0; i < Q_R * Q_P; ++i) {
        const int dy = table_host[2 * i], dx = table_host[2 * i + 1];
        if (dy < 0 || dy >= Q_P || dx < 0 || dx >= Q_P) return HIPR_E_TABLE;
        tab.off[i] = dy * Q_SW + dx;
        baked = baked && dy == kBaked2D[2 * i] && dx == kBaked2D[2 * i + 1];
    }
    const unsigned long long *rg = reinterpret_cast<const unsigned long long *>(range_dev);
    static const int mode = refine_mode("HIPR_LNE2D_REFINE");
    if (dtype == HIPR_F64) {
        if (baked) return lne2d_q_launch<double, true>((const double *)image_dev, Hs, Ws, ld, src_off, y_begin, y_end, W, tab, flavour, rg, out_dev, mode, st);
        return lne2d_q_launch<double, false>((const double *)image_dev, Hs, Ws, ld, src_off, y_begin, y_end, W, tab, flavour, rg, out_dev, mode, st);
    }
    if (baked) return lne2d_q_launch<float, true>((const float *)image_dev, Hs, Ws, ld, src_off, y_begin, y_end, W, tab, flavour, rg, out_dev, mode, st);
    return lne2d_q_launch<float, false>((const float *)image_dev, Hs, Ws, ld, src_off, y_begin, y_end, W, tab, flavour, rg, out_dev, mode, st);
}
}  // namespace hipr

using namespace hipr;

extern "C" int hipr_lne2d_q(const void *image_dev, int Hs, int Ws, int64_t ld, int padded, int dtype, int patch_size,
                            int n_dirs, const int32_t *table_host, int flavour, const uint64_t *range_dev,
                            float *out_dev, void *stream) {
    if (!image_dev || !out_dev || !table_host || Hs < 1 || Ws < 1 || ld < Ws) return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    if (patch_size != Q_P || n_dirs != Q_R) return HIPR_E_TABLE;   // callers use hipr_lne2d otherwise
    const int H = padded ? Hs - (Q_P - 1) : Hs;
    if (H < 1) return HIPR_E_PATCH;
    return lne2d_q_rows(image_dev, Hs, Ws, ld, padded, dtype, table_host, flavour, range_dev, out_dev, 0, H,
                        (cudaStream_t)stream);
}

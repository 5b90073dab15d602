// The fixed-point format of the stencils (K3q in lne2d_q.cu, lne3d_q_kernel in lne3d.cu, K13 in fused2d.cu) and the
// error bound that decides which pixels are recomputed in float64.  DESIGN.md, K3q, gives the reasoning.
//
// Format: a tile's float64 samples are mapped affinely onto 31-bit integers,
//     q = (S - min) * (SPAN / (max - min)) + BIAS,
// stored as the bit patterns of positive normal floats, whose ordering is the integer ordering: min and max run on
// FMNMX like a float kernel, but every min, max and difference is exact.  F1/F2 scores are invariant under that map;
// F3 and ME2 carry their 1e-8 epsilon into grid units (eps_q).  NaN is not representable: callers map it to 0 before
// they take the range.
#pragma once
#include <cstdlib>
#include "hipr_common.cuh"
#include "baked_tables.cuh"

namespace hipr {

constexpr uint32_t Q_BIAS = 0x00800000u;          // smallest positive normal float
constexpr double Q_SPAN = (double)0x7E000000u;    // BIAS + SPAN = 0x7E800000 < +inf

// grid units per unit of the image; 0 for a flat range
__device__ __forceinline__ double q_scale(double vmax, double vmin) {
    return (vmax > vmin) ? Q_SPAN / (vmax - vmin) : 0.0;
}
__device__ __forceinline__ float q_encode(double v, double vmin, double K) {
    const double qd = fmin(fmax((v - vmin) * K, 0.0), Q_SPAN);
    return __uint_as_float(__double2uint_rn(qd) + Q_BIAS);
}
// the flavours' 1e-8 epsilon of an image whose max is vmax, in grid units
__device__ __forceinline__ float q_eps(double vmax, double K) {
    return (K > 0.0) ? (float)(1e-8 * fabs(vmax) * K) : 1.0f;
}

// max / min over the 8 warps of a 256-thread group; tid: the thread's index in the group, `red`: 16 doubles of shared
// memory, `sync`: the group's barrier
template <typename Sync>
__device__ __forceinline__ void block8_minmax(double &vmax, double &vmin, double *red, unsigned tid, Sync sync) {
    vmax = warp_max(vmax);
    vmin = -warp_max(-vmin);
    if ((tid & 31) == 0) {
        red[(tid >> 5) * 2] = vmax;
        red[(tid >> 5) * 2 + 1] = vmin;
    }
    sync();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        vmax = fmax(vmax, red[2 * j]);
        vmin = fmin(vmin, red[2 * j + 1]);
    }
}

// Denominator of a line value, (centre - min) / den, per flavour: the fixed-point lines (in grid units) and the float64
// refinement lines (in image units) share it.
template <int FLAVOUR, typename T>
__device__ __forceinline__ T q_den(T range, T eps) {
    if (FLAVOUR == HIPR_FLAVOUR_F1 || FLAVOUR == HIPR_FLAVOUR_F2) return range;   // 0/0 -> NaN on a flat line
    if (FLAVOUR == HIPR_FLAVOUR_F3) return range + eps;
    return fmax(range, eps);                                                     // ME2
}

// One line of the fixed-point tile: its value r = dq / den and, where asked, inv = 1 / den, the e of the error bound
// below.  Either way one MUFU.RCP and one FMUL: dq * inv is what __fdividef(dq, den) does.
template <int FLAVOUR>
__device__ __forceinline__ float q_line(float centre, float mn, float mx, float eps_q, float *inv = nullptr) {
    const float dq = __uint2float_rn(__float_as_uint(centre) - __float_as_uint(mn));
    const float rq = __uint2float_rn(__float_as_uint(mx) - __float_as_uint(mn));
    const float den = q_den<FLAVOUR>(rq, eps_q);
    if (inv == nullptr) return __fdividef(dq, den);
    *inv = __fdividef(1.0f, den);
    return dq * *inv;
}

// Score factor 1 - qcv without the cancellation: 1 - (uq - lq) / (uq + lq + eps) = A / B, A = 2 lq + eps,
// B = uq + lq + eps.  unit: the factor is exactly 1 (F1 with uq <= 0; F2 / ME2's nan_to_num(0 / 0) = 0).
template <int FLAVOUR>
__device__ __forceinline__ float q_factor(float lq, float uq, float &A, float &B, bool &unit) {
    if (FLAVOUR == HIPR_FLAVOUR_F1 || FLAVOUR == HIPR_FLAVOUR_F3) {
        A = 2.f * lq + 1e-8f;
        B = uq + lq + 1e-8f;
        unit = (FLAVOUR == HIPR_FLAVOUR_F1) && !(uq > 0.f);
    } else {
        A = 2.f * lq;
        B = uq + lq;
        unit = (B == 0.f);
    }
    return unit ? 1.f : __fdiv_rn(A, B);
}

// Pixels the grid cannot resolve to 1e-5 RELATIVE.  Every sample is off by at most half a grid unit, so a line value
// r = dq / den is off by at most (1 + r) e, e = 1 / den, whatever the size of r; a value that is exactly 0 on the grid is
// exact (the grid preserves order, so the centre is the line's minimum).  The mean and the order statistics are
// 1-Lipschitz in the line values, so the bound carries through mean * A / B.  A pixel whose bound on the relative error
// exceeds Q_REFINE_THR (2e-6 are left for the float32 roundings of the epilogue) is written as Q_SENTINEL, which no
// score takes, and recomputed from the float64 image.
constexpr float Q_REFINE_THR = 8e-6f;
constexpr float Q_SENTINEL = -2.0f;

// the bound on one line value or order statistic x whose line has e
__device__ __forceinline__ float q_err(float x, float e) {
    return (x > 0.f) ? fmaf(x, e, e) : 0.f;
}
// d_mean / mean + d_A / A + d_B / B > thr with the divisions multiplied out (d_A = 2 d_lq, d_B = d_lq + d_uq).  2-D
// multiplies the threshold out as ((thr * mean) * A) * B, 3-D as ((thr * A) * B) * mean (MEAN_FIRST = false): the two
// round differently, so each keeps its own.  NaN (a flat line) compares false and keeps the fixed-point result's NaN.
template <bool MEAN_FIRST>
__device__ __forceinline__ bool q_mark(bool unit, float mean, float d_lq, float d_uq, float d_mean, float A, float B) {
    if (unit) return d_mean > Q_REFINE_THR * mean;
    return fmaf(mean, 2.f * d_lq * B + (d_lq + d_uq) * A, d_mean * A * B) >
           (MEAN_FIRST ? Q_REFINE_THR * mean * A * B : Q_REFINE_THR * A * B * mean);
}

// HIPR_LNE2D_REFINE / HIPR_LNE3D_REFINE: 1 (default) = mark and recompute in float64, 0 = the fixed-point result alone,
// 2 = mark only, leaving the sentinels in the output (diagnostic)
inline int refine_mode(const char *env_var) {
    const char *e = getenv(env_var);
    return (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1;
}

// offset of sample li of line t of the pinned (11, 9) table in a 2-D tile of row stride STRIDE (an LDS immediate)
template <int STRIDE>
constexpr int baked2d_off(int t, int li) {
    return kBaked2D[(t * 11 + li) * 2] * STRIDE + kBaked2D[(t * 11 + li) * 2 + 1];
}

}  // namespace hipr

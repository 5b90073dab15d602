// 3-D stencils (biofilm z-stacks), bio/neighbor.pyx.
//   line_profile_3d : literal 5-D gather, bio/neighbor.pyx:171-180 (shares K2's gather kernel)
//   lne3d_dirs      : line_profile_memory_efficient_v2, bio/neighbor.pyx:246-262
//   lne3d           : stencil + epilogue (F2 / F3 / ME2 / V3)
// Fast path: P = 11, 72 directions; a (TX+10) x (8+10) x (32+10) brick of the volume sits in
// shared memory (z fastest, lanes along z: conflict-free), each thread walks TX voxels.  The
// 792-entry offset table rides in the kernel parameter bank.  This kernel is shared-memory /
// min-max-ALU bound (792 samples + a 72-value rank selection per voxel), not HBM bound.
#include "hipr_common.cuh"
#include "lne_math.cuh"
#include "lne_fixed.cuh"

namespace hipr {

template <typename T>
int gather_launch(const T *src, int64_t stride_a, int64_t stride_b, int inner, int64_t nrows, int rowlen,
                  int K, const int *lin, T *out, cudaStream_t st);
int check_table(const int32_t *table, int n_dirs, int P, int ndim);

struct Table3D {
    int off[HIPR_MAX_TABLE];
};
// the generic kernel's (t, li, 3) table, by value in the kernel parameter bank (11.5 KB; the limit is 32 KB since
// CUDA 12.1): no device copy to keep coherent with streams, devices or threads
struct Table3DFull {
    int v[HIPR_MAX_TABLE * 3];
};

constexpr int L3_P = 11, L3_T = 72, L3_HALF = 5;
constexpr int L3_TY = 8, L3_TZ = 32;
constexpr int L3_SY = L3_TY + L3_P - 1;  // 18
constexpr int L3_SZ = L3_TZ + L3_P - 1;  // 42

constexpr int l3_baked_off(int t, int li) {
    return (kBaked3D[(t * L3_P + li) * 3] * L3_SY + kBaked3D[(t * L3_P + li) * 3 + 1]) * L3_SZ +
           kBaked3D[(t * L3_P + li) * 3 + 2];
}
// Lines of the pinned table that repeat an earlier line (same 11 voxels, in either order): 6 of the 72.  Their
// min, max and centre are the earlier line's, so their value is copied instead of recomputed.
constexpr int l3_dup_of(int t) {
    for (int u = 0; u < t; ++u) {
        bool same = true, rev = true;
        for (int li = 0; li < L3_P; ++li) {
            same = same && (l3_baked_off(t, li) == l3_baked_off(u, li));
            rev = rev && (l3_baked_off(t, li) == l3_baked_off(u, L3_P - 1 - li));
        }
        if (same || rev) return u;
    }
    return -1;
}

constexpr int l3_mult(int t) {      // 1 + number of later lines that repeat line t
    int m = 1;
    for (int u = t + 1; u < L3_T; ++u)
        if (l3_dup_of(u) == t) ++m;
    return m;
}

// float32 lines use the fast reciprocal divide (2 ulp): one of 72 per voxel, far inside the gate
template <typename T> __device__ __forceinline__ T l3_div(T a, T b) { return a / b; }
template <> __device__ __forceinline__ float l3_div<float>(float a, float b) { return __fdividef(a, b); }

template <typename T, int FLAVOUR>
__device__ __forceinline__ T l3_line_rel(T centre, T mn, T mx, bool bad) {
    const T range = mx - mn;
    T r;
    if (FLAVOUR == HIPR_FLAVOUR_F2) r = l3_div<T>(centre - mn, range);
    else if (FLAVOUR == HIPR_FLAVOUR_F3) r = l3_div<T>(centre - mn, range + (T)1e-8);
    else r = l3_div<T>(centre - mn, Num<T>::mx(range, (T)1e-8));
    if (FLAVOUR != HIPR_FLAVOUR_F2 && bad) r = Num<T>::nan();
    return r;
}

// MODE 0: write the 72 per-direction values (me_v2); MODE 1: write the fused score.
// BAKED: the host's table equals the pinned (11, 9, 9) table, whose 792 offsets are then
// compile-time immediates of the LDS instructions (no table fetch, no address arithmetic).
template <typename T, int FLAVOUR, int MODE, int TX, bool BAKED>
__global__ void __launch_bounds__(256)
lne3d_p11t72_kernel(const T *__restrict__ vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
                    const __grid_constant__ Table3D tab,  // (dx * SY + dy) * SZ + dz, patch coords
                    const unsigned long long *__restrict__ maxkey, T *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw3[];
    T *tile = reinterpret_cast<T *>(smem_raw3);
    constexpr int SX = TX + L3_P - 1;
    const int nzb = (Z + L3_TZ - 1) / L3_TZ;
    const int z0 = (blockIdx.x % nzb) * L3_TZ;
    const int y0 = (blockIdx.x / nzb) * L3_TY;
    const int x0 = blockIdx.y * TX;
    const bool scale = (maxkey != nullptr);
    const T vmax = scale ? (T)double_of_key(*maxkey) : (T)1;
    for (int i = threadIdx.x; i < SX * L3_SY * L3_SZ; i += 256) {
        const int lz = i % L3_SZ, rest = i / L3_SZ;
        const int ly = rest % L3_SY, lx = rest / L3_SY;
        int sx = x0 + lx - L3_HALF + src_off, sy = y0 + ly - L3_HALF + src_off, sz = z0 + lz - L3_HALF + src_off;
        sx = min(max(sx, 0), Xs - 1);
        sy = min(max(sy, 0), Ys - 1);
        sz = min(max(sz, 0), Zs - 1);
        T v = vol[((int64_t)sx * Ys + sy) * Zs + sz];
        if (scale) v = Num<T>::div(v, vmax);
        if (FLAVOUR == HIPR_FLAVOUR_F2) v = nan_to_num<T>(v);
        tile[i] = v;
    }
    __syncthreads();
    const int tz = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int z = z0 + tz, y = y0 + ty;
    if (z >= Z || y >= Y) return;
#pragma unroll 1
    for (int lx = 0; lx < TX; ++lx) {
        const int x = x0 + lx;
        if (x >= X) break;
        const T *base = tile + (lx * L3_SY + ty) * L3_SZ + tz;
        T r[L3_T];
        if constexpr (BAKED) {
            static_for<0, L3_T>([&](auto tc) {
                constexpr int t = decltype(tc)::value;
                constexpr int o0 = l3_baked_off(t, 0);
                T mn = base[o0], mx = mn;
                bool bad = (mn != mn);
                static_for<1, L3_P>([&](auto lc) {
                    constexpr int off = l3_baked_off(t, decltype(lc)::value);
                    const T s = base[off];
                    mn = Num<T>::mn(mn, s);
                    mx = Num<T>::mx(mx, s);
                    if (FLAVOUR != HIPR_FLAVOUR_F2) bad |= (s != s);
                });
                constexpr int oc = l3_baked_off(t, L3_HALF);
                r[t] = l3_line_rel<T, FLAVOUR>(base[oc], mn, mx, bad);
            });
        } else {
#pragma unroll
            for (int t = 0; t < L3_T; ++t) {
                T mn = base[tab.off[t * L3_P]], mx = mn, centre = mn;
                bool bad = (mn != mn);
#pragma unroll
                for (int li = 1; li < L3_P; ++li) {
                    const T s = base[tab.off[t * L3_P + li]];
                    mn = Num<T>::mn(mn, s);
                    mx = Num<T>::mx(mx, s);
                    if (li == L3_HALF) centre = s;
                    if (FLAVOUR != HIPR_FLAVOUR_F2) bad |= (s != s);
                }
                r[t] = l3_line_rel<T, FLAVOUR>(centre, mn, mx, bad);
            }
        }
        const int64_t v = ((int64_t)x * Y + y) * Z + z;
        if (MODE == 0) {
            T *o = out + v * L3_T;
#pragma unroll
            for (int t = 0; t < L3_T; ++t) o[t] = r[t];
        } else {
            out[v] = reduce_dirs<T, L3_T, FLAVOUR>(r);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Fixed-point variant: the brick is mapped onto the 31-bit grid of lne_fixed.cuh with the BRICK's
// own min/max; min / max / differences along the 72 lines are exact, so float64 channel sums keep
// their precision at float32 speed and no NaN bookkeeping is needed (NaN samples become 0).  F2 is
// invariant to the affine map; F3 / ME2 carry their 1e-8 into q units with the global max
// (`maxkey`; NULL = the volume is already normalised).  Baked (11, 9, 9) table only.
// Strict relative parity, as in 2-D: e_max, the largest e_t, stands in for the e of the quartile
// lines, and a voxel whose bound exceeds Q_REFINE_THR is written as a sentinel and recomputed in
// float64 by lne3d_refine_kernel (~2 % of a synthetic z-stack).
// ---------------------------------------------------------------------------------------
// mean * (1 - qcv) over the 72 directions without the cancellation of 1 - (uq - lq) / (uq + lq)
struct L3QResult {
    float score, mean, r17, r18, r53, r54;
    bool mark;
};
template <int FLAVOUR, bool REFINE>
__device__ __forceinline__ L3QResult l3q_reduce(float (&r)[L3_T], float e_max) {
    L3QResult res;
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < L3_T; ++i) sum += r[i];
    const float mean = sum * (1.0f / L3_T);
    sort_network<float, L3_T>(r);
    const float lq = quartile_sorted<float, L3_T, 1>(r);
    const float uq = quartile_sorted<float, L3_T, 3>(r);
    float A, B;
    bool unit;
    res.score = mean * q_factor<FLAVOUR>(lq, uq, A, B, unit);
    res.mean = mean;
    res.r17 = r[17];
    res.r18 = r[18];
    res.r53 = r[53];
    res.r54 = r[54];
    res.mark = false;
    if (REFINE) {
        // first opinion: e_max, the largest e_t of the voxel, stands in for the e of the quartile lines
        const float d_mean = fmaf(mean, e_max, e_max);
        res.mark = q_mark<false>(unit, mean, q_err(lq, e_max), q_err(uq, e_max), d_mean, A, B);
    }
    return res;
}

// a voxel the first opinion marked, parked for the second opinion
struct L3QPending {
    float score, mean, r17, r18, r53, r54;
    int local;                               // (lx * L3_TY + ty) * L3_TZ + tz
};
constexpr int L3Q_PENDING = 224;             // per CTA; beyond that a marked voxel goes straight to the refinement

template <typename SrcT, int FLAVOUR, int MODE, int TX, bool REFINE>
__global__ void __launch_bounds__(256)
lne3d_q_kernel(const SrcT *__restrict__ vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
               const unsigned long long *__restrict__ maxkey, float *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw3q[];
    float *tile = reinterpret_cast<float *>(smem_raw3q);
    __shared__ double red[16];
    __shared__ L3QPending pending[(REFINE && MODE == 1) ? L3Q_PENDING : 1];
    __shared__ unsigned int n_pending;
    constexpr int SX = TX + L3_P - 1;
    const int nzb = (Z + L3_TZ - 1) / L3_TZ;
    const int z0 = (blockIdx.x % nzb) * L3_TZ;
    const int y0 = (blockIdx.x / nzb) * L3_TY;
    const int x0 = blockIdx.y * TX;
    if (threadIdx.x == 0) n_pending = 0;
    double bmax = -__longlong_as_double(0x7ff0000000000000ll), bmin = -bmax;
    for (int i = threadIdx.x; i < SX * L3_SY * L3_SZ; i += 256) {
        const int lz = i % L3_SZ, rest = i / L3_SZ;
        const int ly = rest % L3_SY, lx = rest / L3_SY;
        const int sx = min(max(x0 + lx - L3_HALF + src_off, 0), Xs - 1);
        const int sy = min(max(y0 + ly - L3_HALF + src_off, 0), Ys - 1);
        const int sz = min(max(z0 + lz - L3_HALF + src_off, 0), Zs - 1);
        double v = (double)vol[((int64_t)sx * Ys + sy) * Zs + sz];
        if (v != v) v = 0.0;
        bmax = fmax(bmax, v);
        bmin = fmin(bmin, v);
    }
    block8_minmax(bmax, bmin, red, threadIdx.x, [] { __syncthreads(); });
    const double K = q_scale(bmax, bmin);
    const float eps_q = q_eps(maxkey ? fabs(double_of_key(*maxkey)) : 1.0, K);
    for (int i = threadIdx.x; i < SX * L3_SY * L3_SZ; i += 256) {
        const int lz = i % L3_SZ, rest = i / L3_SZ;
        const int ly = rest % L3_SY, lx = rest / L3_SY;
        const int sx = min(max(x0 + lx - L3_HALF + src_off, 0), Xs - 1);
        const int sy = min(max(y0 + ly - L3_HALF + src_off, 0), Ys - 1);
        const int sz = min(max(z0 + lz - L3_HALF + src_off, 0), Zs - 1);
        double v = (double)vol[((int64_t)sx * Ys + sy) * Zs + sz];   // second read: L1/L2 hit
        if (v != v) v = 0.0;
        tile[i] = q_encode(v, bmin, K);
    }
    __syncthreads();
    const int tz = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int z = z0 + tz, y = y0 + ty;
    // one line of the fixed-point tile: value and e = 1 / (denominator in grid units)
    auto line = [&](const float *base, auto tc, float &rv, float &inv) {
        constexpr int t = decltype(tc)::value;
        constexpr int o0 = l3_baked_off(t, 0);
        float mn = base[o0], mx = mn;
        static_for<1, L3_P>([&](auto lc) {
            constexpr int off = l3_baked_off(t, decltype(lc)::value);
            const float s = base[off];
            mn = fminf(mn, s);
            mx = fmaxf(mx, s);
        });
        constexpr int oc = l3_baked_off(t, L3_HALF);
        rv = q_line<FLAVOUR>(base[oc], mn, mx, eps_q, &inv);
    };
    if (z < Z && y < Y) {
#pragma unroll 1
        for (int lx = 0; lx < TX; ++lx) {
            const int x = x0 + lx;
            if (x >= X) break;
            const float *base = tile + (lx * L3_SY + ty) * L3_SZ + tz;
            float r[L3_T];
            float e_max = 0.f;
            static_for<0, L3_T>([&](auto tc) {
                constexpr int t = decltype(tc)::value;
                constexpr int dup = l3_dup_of(t);
                if constexpr (dup >= 0) {
                    r[t] = r[dup];
                } else {
                    float rv, inv;
                    line(base, tc, rv, inv);
                    if (REFINE) {
                        if (MODE == 0) {
                            // per-direction output: mark the value itself when (1 + r) e > thr * r
                            if (rv > 0.f && fmaf(rv, inv, inv) > Q_REFINE_THR * rv) rv = Q_SENTINEL;
                        } else {
                            e_max = fmaxf(e_max, inv);
                        }
                    }
                    r[t] = rv;
                }
            });
            const int64_t v = ((int64_t)x * Y + y) * Z + z;
            if (MODE == 0) {
                float *o = out + v * L3_T;
#pragma unroll
                for (int t = 0; t < L3_T; ++t) o[t] = r[t];
            } else {
                const L3QResult res = l3q_reduce<FLAVOUR, REFINE>(r, e_max);
                float score = res.score;
                if (REFINE && res.mark) {
                    const unsigned int slot = atomicAdd(&n_pending, 1u);
                    if (slot < L3Q_PENDING) {
                        pending[slot] = L3QPending{res.score, res.mean, res.r17, res.r18, res.r53, res.r54,
                                                   (lx * L3_TY + ty) * L3_TZ + tz};
                        continue;                       // written after the second opinion
                    }
                    score = Q_SENTINEL;
                }
                out[v] = score;
            }
        }
    }
    if (!(REFINE && MODE == 1)) return;
    // ---- second opinion for the marked voxels, packed into full warps: the 72 lines again, this time keeping the e of
    // the lines that gave the quartile order statistics and the exact sum for the mean -------------------------------
    __syncthreads();
    const int np = (int)min(n_pending, (unsigned int)L3Q_PENDING);
    for (int p = threadIdx.x; p < np; p += 256) {
        const L3QPending pd = pending[p];
        const int ptz = pd.local % L3_TZ, rest = pd.local / L3_TZ;
        const int pty = rest % L3_TY, plx = rest / L3_TY;
        const float *base = tile + (plx * L3_SY + pty) * L3_SZ + ptz;
        float e17 = 0.f, e18 = 0.f, e53 = 0.f, e54 = 0.f, d_sum = 0.f;
        static_for<0, L3_T>([&](auto tc) {
            constexpr int t = decltype(tc)::value;
            if constexpr (l3_dup_of(t) < 0) {
                float rv, inv;
                line(base, tc, rv, inv);
                constexpr float mult = (float)l3_mult(t);
                d_sum += mult * q_err(rv, inv);
                e17 = (rv == pd.r17) ? fmaxf(e17, inv) : e17;
                e18 = (rv == pd.r18) ? fmaxf(e18, inv) : e18;
                e53 = (rv == pd.r53) ? fmaxf(e53, inv) : e53;
                e54 = (rv == pd.r54) ? fmaxf(e54, inv) : e54;
            }
        });
        const float lq = quartile_pair<float, 1>(pd.r17, pd.r18), uq = quartile_pair<float, 3>(pd.r53, pd.r54);
        float A, B;
        bool unit;
        q_factor<FLAVOUR>(lq, uq, A, B, unit);
        const float d_mean = d_sum * (1.0f / L3_T);
        // |d lq| <= 0.25 (1 + r17) e17 + 0.75 (1 + r18) e18, |d uq| <= 0.75 (1 + r53) e53 + 0.25 (1 + r54) e54
        const float d_lq = 0.25f * q_err(pd.r17, e17) + 0.75f * q_err(pd.r18, e18);
        const float d_uq = 0.75f * q_err(pd.r53, e53) + 0.25f * q_err(pd.r54, e54);
        const bool mark = q_mark<false>(unit, pd.mean, d_lq, d_uq, d_mean, A, B);
        const int64_t v = ((int64_t)(x0 + plx) * Y + (y0 + pty)) * Z + (z0 + ptz);
        out[v] = mark ? Q_SENTINEL : pd.score;
    }
}

// the pinned table for run-time indexing on the device (kBaked3D itself only exists in constant expressions)
struct Baked3DCopy {
    int v[L3_T * L3_P * 3];
};
constexpr Baked3DCopy make_baked3d_copy() {
    Baked3DCopy a{};
    for (int i = 0; i < L3_T * L3_P * 3; ++i) a.v[i] = kBaked3D[i];
    return a;
}
__constant__ Baked3DCopy c_baked3d = make_baked3d_copy();

// One line value in float64 from the source volume (edge clamp, NaN -> 0: the fixed-point loader's semantics);
// `tab` = the (72, 11, 3) table as bytes.
template <typename SrcT, int FLAVOUR>
__device__ __forceinline__ double l3_line_value_f64(const SrcT *__restrict__ vol, int Xs, int Ys, int Zs, int bx, int by,
                                                   int bz, const signed char *__restrict__ tab, int t, double eps) {
    double v[L3_P];
#pragma unroll
    for (int li = 0; li < L3_P; ++li) {
        const signed char *o = tab + (t * L3_P + li) * 3;
        const int sx = min(max(bx + o[0], 0), Xs - 1), sy = min(max(by + o[1], 0), Ys - 1), sz = min(max(bz + o[2], 0), Zs - 1);
        const double s = (double)vol[((int64_t)sx * Ys + sy) * Zs + sz];
        v[li] = (s != s) ? 0.0 : s;
    }
    double mn = v[0], mx = v[0];
#pragma unroll
    for (int li = 1; li < L3_P; ++li) {
        mn = fmin(mn, v[li]);
        mx = fmax(mx, v[li]);
    }
    const double den = q_den<FLAVOUR>(mx - mn, eps);
    return (v[L3_HALF] - mn) / den;
}

// Refinement of the marked voxels of a fused score volume, in float64.  A CTA scans 16384 consecutive voxels for the
// sentinel, collects them in shared memory and takes 4 per round with 72 threads per voxel: phase A, thread t
// computes the value of line t; phase B, thread t counts the values below its own (ties by index): the threads that
// hold ranks 17, 18, 53 and 54 publish them, thread 0 of the voxel adds up the mean and writes the score.  Small
// register and shared-memory footprint, so many CTAs are resident.
constexpr int RF3_SPAN = 16384, RF3_VOX = 4, RF3_THREADS = RF3_VOX * L3_T;   // 288

template <typename SrcT, int FLAVOUR>
__global__ void __launch_bounds__(RF3_THREADS, 3)
lne3d_refine_kernel(const SrcT *__restrict__ vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
                    const unsigned long long *__restrict__ maxkey, float *__restrict__ out) {
    __shared__ double rbuf[RF3_VOX][L3_T];
    __shared__ double sel[RF3_VOX][4];
    __shared__ int has_nan[RF3_VOX];
    __shared__ signed char tab[L3_T * L3_P * 3];
    __shared__ unsigned short marked[RF3_SPAN];
    __shared__ unsigned int n_marked;
    const int64_t nvox = (int64_t)X * Y * Z;
    const int64_t v0 = (int64_t)blockIdx.x * RF3_SPAN;
    if (threadIdx.x == 0) n_marked = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < RF3_SPAN; i += RF3_THREADS)
        if (v0 + i < nvox && out[v0 + i] == Q_SENTINEL) marked[atomicAdd(&n_marked, 1u)] = (unsigned short)i;
    __syncthreads();
    const int n = (int)n_marked;
    if (n == 0) return;
    for (int i = threadIdx.x; i < L3_T * L3_P * 3; i += RF3_THREADS) tab[i] = (signed char)c_baked3d.v[i];
    const double eps = 1e-8 * (maxkey ? fabs(double_of_key(*maxkey)) : 1.0);
    const int j = threadIdx.x / L3_T, t = threadIdx.x - j * L3_T;
    for (int j0 = 0; j0 < n; j0 += RF3_VOX) {
        const bool active = (j0 + j < n);
        __syncthreads();                     // table staged; previous round's buffers consumed
        double mine = 0.0;
        int64_t v = 0;
        if (active) {
            v = v0 + marked[j0 + j];
            const int z = (int)(v % Z);
            const int64_t rest = v / Z;
            const int y = (int)(rest % Y), x = (int)(rest / Y);
            mine = l3_line_value_f64<SrcT, FLAVOUR>(vol, Xs, Ys, Zs, x - L3_HALF + src_off, y - L3_HALF + src_off,
                                                    z - L3_HALF + src_off, tab, t, eps);
            rbuf[j][t] = mine;
            if (t == 0) has_nan[j] = 0;
        }
        __syncthreads();
        if (active) {
            if (mine != mine) has_nan[j] = 1;
            int below = 0;
#pragma unroll 4
            for (int u = 0; u < L3_T; ++u) {
                const double o = rbuf[j][u];
                below += (o < mine || (o == mine && u < t)) ? 1 : 0;
            }
            if (below == 17) sel[j][0] = mine;
            if (below == 18) sel[j][1] = mine;
            if (below == 53) sel[j][2] = mine;
            if (below == 54) sel[j][3] = mine;
        }
        __syncthreads();
        if (active && t == 0) {
            double sum = 0.0;
#pragma unroll 4
            for (int u = 0; u < L3_T; ++u) sum += rbuf[j][u];
            const double mean = sum / L3_T;
            // numpy 'linear' percentiles at virtual indices 17.75 and 53.25 (numpy's _lerp)
            const double a1 = sel[j][0], b1 = sel[j][1], a3 = sel[j][2], b3 = sel[j][3];
            const double lq = b1 - (b1 - a1) * 0.25, uq = a3 + (b3 - a3) * 0.25;
            double score;
            if (has_nan[j]) score = __longlong_as_double(0x7ff8000000000000ll);
            else if (FLAVOUR == HIPR_FLAVOUR_F3) score = mean * (1.0 - (uq - lq) / (uq + lq + 1e-8));
            else {
                const double qcv = (uq + lq == 0.0) ? 0.0 : (uq - lq) / (uq + lq);     // nan_to_num(0 / 0) = 0
                score = mean * (1.0 - qcv);
            }
            out[v] = (float)score;
        }
    }
}

// Refinement of the marked per-direction values of a (X, Y, Z, 72) output: thread per value.
template <typename SrcT>
__global__ void __launch_bounds__(256)
lne3d_refine_dirs_kernel(const SrcT *__restrict__ vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
                         const unsigned long long *__restrict__ maxkey, float *__restrict__ out) {
    __shared__ signed char tab[L3_T * L3_P * 3];
    for (int i = threadIdx.x; i < L3_T * L3_P * 3; i += 256) tab[i] = (signed char)c_baked3d.v[i];
    __syncthreads();
    const int64_t n = (int64_t)X * Y * Z * L3_T;
    const double eps = 1e-8 * (maxkey ? fabs(double_of_key(*maxkey)) : 1.0);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (out[i] != Q_SENTINEL) continue;
        const int t = (int)(i % L3_T);
        const int64_t v = i / L3_T;
        const int z = (int)(v % Z);
        const int64_t rest = v / Z;
        const int y = (int)(rest % Y), x = (int)(rest / Y);
        out[i] = (float)l3_line_value_f64<SrcT, HIPR_FLAVOUR_ME2>(vol, Xs, Ys, Zs, x - L3_HALF + src_off, y - L3_HALF + src_off,
                                                                 z - L3_HALF + src_off, tab, t, eps);
    }
}

// Generic path: any table; thread per voxel from global memory.  `flat` != 0 reproduces the
// v3 function's flat addressing: table entries may leave the patch, the address is taken in
// the padded buffer and a read past its end gives NaN (undefined behaviour in the reference).
template <typename T>
__global__ void __launch_bounds__(128)
lne3d_generic_kernel(const T *__restrict__ vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
                     int P, int Tn, const __grid_constant__ Table3DFull tabp /* (t, li, 3) */, int flavour, int mode,
                     int flat, const unsigned long long *__restrict__ maxkey, T *__restrict__ out) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)X * Y * Z) return;
    const int z = (int)(idx % Z);
    const int64_t rest = idx / Z;
    const int y = (int)(rest % Y), x = (int)(rest / Y);
    const int half = (P - 1) / 2;
    const bool scale = (maxkey != nullptr);
    const T vmax = scale ? (T)double_of_key(*maxkey) : (T)1;
    const bool n2n = (flavour == HIPR_FLAVOUR_F2);
    const int64_t nvox = (int64_t)Xs * Ys * Zs;
    T r[HIPR_MAX_DIRS];
    for (int t = 0; t < Tn; ++t) {
        T mn = (T)0, mx = (T)0, centre = (T)0;
        bool bad = false;
        for (int li = 0; li < P; ++li) {
            const int *o = tabp.v + (t * P + li) * 3;
            T s;
            if (flat) {
                const int64_t a = ((int64_t)(x + o[0]) * Ys + (y + o[1])) * Zs + (z + o[2]);
                s = (a >= 0 && a < nvox) ? vol[a] : Num<T>::nan();
            } else {
                int sx = x + o[0] - half + src_off, sy = y + o[1] - half + src_off, sz = z + o[2] - half + src_off;
                sx = min(max(sx, 0), Xs - 1);
                sy = min(max(sy, 0), Ys - 1);
                sz = min(max(sz, 0), Zs - 1);
                s = vol[((int64_t)sx * Ys + sy) * Zs + sz];
            }
            if (scale) s = Num<T>::div(s, vmax);
            if (n2n) s = nan_to_num<T>(s);
            bad |= (s != s);
            if (li == 0) { mn = s; mx = s; }
            else { mn = Num<T>::mn(mn, s); mx = Num<T>::mx(mx, s); }
            if (li == half) centre = s;
        }
        switch (flavour) {
            case HIPR_FLAVOUR_F2: r[t] = line_rel<T, HIPR_FLAVOUR_F2>(centre, mn, mx, bad); break;
            case HIPR_FLAVOUR_F3: r[t] = line_rel<T, HIPR_FLAVOUR_F3>(centre, mn, mx, bad); break;
            default: r[t] = line_rel<T, HIPR_FLAVOUR_ME2>(centre, mn, mx, bad); break;
        }
    }
    if (mode == 0) {
        for (int t = 0; t < Tn; ++t) out[idx * Tn + t] = r[t];
    } else {
        out[idx] = reduce_dirs_runtime<T>(r, Tn, flavour);
    }
}

template <typename T, int FLAVOUR, int MODE, bool BAKED>
static int launch_fast3d_b(const T *vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z, const Table3D &tab,
                           const unsigned long long *maxkey, T *out, cudaStream_t st) {
    constexpr int TX = (sizeof(T) == 4) ? 8 : 4;
    constexpr int SX = TX + L3_P - 1;
    const size_t smem = (size_t)SX * L3_SY * L3_SZ * sizeof(T);
    auto kern = lne3d_p11t72_kernel<T, FLAVOUR, MODE, TX, BAKED>;
    static std::atomic<uint64_t> attr_done{0};
    if (first_use_on_device(attr_done)) HIPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int nzb = (Z + L3_TZ - 1) / L3_TZ, nyb = (Y + L3_TY - 1) / L3_TY, nxb = (X + TX - 1) / TX;
    if ((int64_t)nzb * nyb > 0x7fffffffLL || nxb > 65535) return HIPR_E_RANGE;
    dim3 grid((unsigned)(nzb * nyb), (unsigned)nxb);
    kern<<<grid, 256, smem, st>>>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, maxkey, out);
    return after_launch();
}

template <typename T, int FLAVOUR, int MODE>
static int launch_fast3d(const T *vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z, const Table3D &tab,
                         bool baked, const unsigned long long *maxkey, T *out, cudaStream_t st) {
    if (baked) return launch_fast3d_b<T, FLAVOUR, MODE, true>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, maxkey, out, st);
    return launch_fast3d_b<T, FLAVOUR, MODE, false>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, maxkey, out, st);
}

template <typename T>
static int lne3d_dispatch(const T *vol, int Xs, int Ys, int Zs, int padded, int P, int Tn, const int32_t *table,
                          int flavour, int mode, const unsigned long long *maxkey, T *out, cudaStream_t st) {
    const int X = padded ? Xs - (P - 1) : Xs, Y = padded ? Ys - (P - 1) : Ys, Z = padded ? Zs - (P - 1) : Zs;
    const int src_off = padded ? (P - 1) / 2 : 0;
    if (X < 1 || Y < 1 || Z < 1) return HIPR_E_PATCH;
    const bool flat = (flavour == HIPR_FLAVOUR_V3);
    if (flat && !padded) return HIPR_E_ARG;
    bool in_patch = true;
    for (int i = 0; i < Tn * P * 3; ++i)
        if (table[i] < 0 || table[i] >= P) in_patch = false;
    if (!in_patch && !flat) return HIPR_E_TABLE;
    if (flat)
        for (int i = 0; i < Tn * P * 3; ++i)
            if (table[i] < -4 * P || table[i] > 4 * P) return HIPR_E_TABLE;
    if (P == L3_P && Tn == L3_T && in_patch && !flat) {
        Table3D tab;
        bool baked = true;
        for (int i = 0; i < Tn * P; ++i)
            tab.off[i] = (table[3 * i] * L3_SY + table[3 * i + 1]) * L3_SZ + table[3 * i + 2];
        for (int i = 0; i < Tn * P * 3; ++i) baked = baked && (table[i] == kBaked3D[i]);
        if (mode == 0)
            return launch_fast3d<T, HIPR_FLAVOUR_ME2, 0>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, baked, maxkey, out, st);
        switch (flavour) {
            case HIPR_FLAVOUR_F2: return launch_fast3d<T, HIPR_FLAVOUR_F2, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, baked, maxkey, out, st);
            case HIPR_FLAVOUR_F3: return launch_fast3d<T, HIPR_FLAVOUR_F3, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, baked, maxkey, out, st);
            case HIPR_FLAVOUR_ME2: return launch_fast3d<T, HIPR_FLAVOUR_ME2, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, tab, baked, maxkey, out, st);
            default: return HIPR_E_FLAVOUR;
        }
    }
    if (flavour != HIPR_FLAVOUR_F2 && flavour != HIPR_FLAVOUR_F3 && flavour != HIPR_FLAVOUR_ME2 && !flat)
        return HIPR_E_FLAVOUR;
    if (Tn * P * 3 > HIPR_MAX_TABLE * 3) return HIPR_E_TABLE;
    static_assert(sizeof(Table3DFull) <= 32000, "kernel parameter bank");
    Table3DFull tabp;
    memcpy(tabp.v, table, (size_t)Tn * P * 3 * sizeof(int));
    const int64_t nv = (int64_t)X * Y * Z;
    if ((nv + 127) / 128 > 0x7fffffffLL) return HIPR_E_RANGE;
    lne3d_generic_kernel<T><<<(unsigned)((nv + 127) / 128), 128, 0, st>>>(vol, Xs, Ys, Zs, src_off, X, Y, Z, P, Tn,
                                                                         tabp, flavour, mode, flat ? 1 : 0,
                                                                         maxkey, out);
    return after_launch();
}

// refine: refine_mode("HIPR_LNE3D_REFINE")
template <typename SrcT, int FLAVOUR, int MODE>
static int launch_q3d(const SrcT *vol, int Xs, int Ys, int Zs, int src_off, int X, int Y, int Z,
                      const unsigned long long *maxkey, float *out, int refine, cudaStream_t st) {
    constexpr int TX = 8;
    constexpr int SX = TX + L3_P - 1;
    const size_t smem = (size_t)SX * L3_SY * L3_SZ * sizeof(float);
    auto kern = refine ? lne3d_q_kernel<SrcT, FLAVOUR, MODE, TX, true> : lne3d_q_kernel<SrcT, FLAVOUR, MODE, TX, false>;
    static std::atomic<uint64_t> attr_done{0};
    if (first_use_on_device(attr_done)) {
        HIPR_CUDA(cudaFuncSetAttribute(lne3d_q_kernel<SrcT, FLAVOUR, MODE, TX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HIPR_CUDA(cudaFuncSetAttribute(lne3d_q_kernel<SrcT, FLAVOUR, MODE, TX, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const int nzb = (Z + L3_TZ - 1) / L3_TZ, nyb = (Y + L3_TY - 1) / L3_TY, nxb = (X + TX - 1) / TX;
    if ((int64_t)nzb * nyb > 0x7fffffffLL || nxb > 65535) return HIPR_E_RANGE;
    dim3 grid((unsigned)(nzb * nyb), (unsigned)nxb);
    kern<<<grid, 256, smem, st>>>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out);
    int e = after_launch();
    if (e || refine != 1) return e;
    const int64_t nvox = (int64_t)X * Y * Z;
    if (MODE == 0) {
        lne3d_refine_dirs_kernel<SrcT><<<sm_count() * 8, 256, 0, st>>>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out);
    } else {
        const int64_t nb = (nvox + RF3_SPAN - 1) / RF3_SPAN;
        if (nb > 0x7fffffffLL) return HIPR_E_RANGE;
        lne3d_refine_kernel<SrcT, FLAVOUR><<<(unsigned)nb, RF3_THREADS, 0, st>>>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out);
    }
    return after_launch();
}

template <typename SrcT>
static int lne3d_q_dispatch(const SrcT *vol, int Xs, int Ys, int Zs, int padded, int flavour, int mode,
                            const unsigned long long *maxkey, float *out, int refine, cudaStream_t st) {
    const int P = L3_P;
    const int X = padded ? Xs - (P - 1) : Xs, Y = padded ? Ys - (P - 1) : Ys, Z = padded ? Zs - (P - 1) : Zs;
    const int src_off = padded ? L3_HALF : 0;
    if (X < 1 || Y < 1 || Z < 1) return HIPR_E_PATCH;
    if (mode == 0) return launch_q3d<SrcT, HIPR_FLAVOUR_ME2, 0>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out, refine, st);
    switch (flavour) {
        case HIPR_FLAVOUR_F2: return launch_q3d<SrcT, HIPR_FLAVOUR_F2, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out, refine, st);
        case HIPR_FLAVOUR_F3: return launch_q3d<SrcT, HIPR_FLAVOUR_F3, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out, refine, st);
        case HIPR_FLAVOUR_ME2: return launch_q3d<SrcT, HIPR_FLAVOUR_ME2, 1>(vol, Xs, Ys, Zs, src_off, X, Y, Z, maxkey, out, refine, st);
        default: return HIPR_E_FLAVOUR;
    }
}

}  // namespace hipr

using namespace hipr;

// mode 1: fused score (X, Y, Z); mode 0: per-direction values (X, Y, Z, 72).  float32 out.
extern "C" int hipr_lne3d_q(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype, int patch_size,
                            int n_dirs, const int32_t *table_host, int flavour, int dirs_only,
                            const uint64_t *maxkey_dev, float *out_dev, void *stream) {
    if (!volume_dev || !out_dev || !table_host || Xs < 1 || Ys < 1 || Zs < 1) return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    if (patch_size != L3_P || n_dirs != L3_T) return HIPR_E_UNSUPPORTED;
    for (int i = 0; i < L3_T * L3_P * 3; ++i)
        if (table_host[i] != kBaked3D[i]) return HIPR_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long *mk = reinterpret_cast<const unsigned long long *>(maxkey_dev);
    static const int refine = refine_mode("HIPR_LNE3D_REFINE");
    if (dtype == HIPR_F64)
        return lne3d_q_dispatch<double>((const double *)volume_dev, Xs, Ys, Zs, padded, flavour, dirs_only ? 0 : 1, mk,
                                        out_dev, refine, st);
    return lne3d_q_dispatch<float>((const float *)volume_dev, Xs, Ys, Zs, padded, flavour, dirs_only ? 0 : 1, mk,
                                   out_dev, refine, st);
}

extern "C" int hipr_line_profile_3d(const void *volume_padded_dev, int Xp, int Yp, int Zp, int dtype, int patch_size,
                                    int n_dirs, const int32_t *table_host, void *out_dev, void *stream) {
    if (!volume_padded_dev || !out_dev) return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    int e = check_table(table_host, n_dirs, patch_size, 3);
    if (e) return e;
    const int P = patch_size, X = Xp - (P - 1), Y = Yp - (P - 1), Z = Zp - (P - 1);
    if (X < 1 || Y < 1 || Z < 1) return HIPR_E_PATCH;
    int lin[HIPR_MAX_TABLE];
    for (int i = 0; i < n_dirs * P; ++i) {
        const int a = table_host[3 * i], b = table_host[3 * i + 1], c = table_host[3 * i + 2];
        if (a < 0 || a >= P || b < 0 || b >= P || c < 0 || c >= P) return HIPR_E_TABLE;
        const int64_t l = ((int64_t)a * Yp + b) * Zp + c;
        if (l > 0x7fffffffLL) return HIPR_E_RANGE;
        lin[i] = (int)l;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t sa = (int64_t)Yp * Zp, sb = Zp;
    if (dtype == HIPR_F32)
        return gather_launch<float>((const float *)volume_padded_dev, sa, sb, Y, (int64_t)X * Y, Z, n_dirs * P, lin,
                                    (float *)out_dev, st);
    return gather_launch<double>((const double *)volume_padded_dev, sa, sb, Y, (int64_t)X * Y, Z, n_dirs * P, lin,
                                 (double *)out_dev, st);
}

static int lne3d_entry(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype, int patch_size,
                       int n_dirs, const int32_t *table_host, int flavour, int mode, const uint64_t *maxkey_dev,
                       void *out_dev, void *stream) {
    if (!volume_dev || !out_dev || Xs < 1 || Ys < 1 || Zs < 1) return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    int e = check_table(table_host, n_dirs, patch_size, 3);
    if (e) return e;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long *mk = reinterpret_cast<const unsigned long long *>(maxkey_dev);
    if (dtype == HIPR_F32)
        return lne3d_dispatch<float>((const float *)volume_dev, Xs, Ys, Zs, padded, patch_size, n_dirs, table_host,
                                     flavour, mode, mk, (float *)out_dev, st);
    return lne3d_dispatch<double>((const double *)volume_dev, Xs, Ys, Zs, padded, patch_size, n_dirs, table_host,
                                  flavour, mode, mk, (double *)out_dev, st);
}

extern "C" int hipr_lne3d_dirs(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype, int patch_size,
                               int n_dirs, const int32_t *table_host, const uint64_t *maxkey_dev, void *out_dev,
                               void *stream) {
    return lne3d_entry(volume_dev, Xs, Ys, Zs, padded, dtype, patch_size, n_dirs, table_host, HIPR_FLAVOUR_ME2, 0,
                       maxkey_dev, out_dev, stream);
}

extern "C" int hipr_lne3d(const void *volume_dev, int Xs, int Ys, int Zs, int padded, int dtype, int patch_size,
                          int n_dirs, const int32_t *table_host, int flavour, const uint64_t *maxkey_dev,
                          void *out_dev, void *stream) {
    return lne3d_entry(volume_dev, Xs, Ys, Zs, padded, dtype, patch_size, n_dirs, table_host, flavour, 1, maxkey_dev,
                       out_dev, stream);
}

// 1-D k-means thresholding of a score / intensity image (SURVEY.md 8f rank 3): replaces
//   KMeans(n_clusters = k, random_state = 0).fit_predict(image.reshape(-1, 1))
// as the measurement scripts call it on image_final, the denoised sum and their logarithms
// (syn/..._measurement.py:125-149; bio/..._analysis.py:367-392, 463-486, 819-846; eco/..._measurement.py:73-85),
// with scikit-learn 1.9.0 (installed here) as the pinned reference of the parity tests: k-means++ seeding driven by the caller's
// uniform random numbers (numpy RandomState(seed) on the host, in the order scikit-learn consumes them), Lloyd
// iterations with scikit-learn's two stopping rules (labels unchanged; squared centre shift <= tol * var(x)),
// labels from the final centres, best of n_init by inertia.
//
// One persistent cooperative kernel: every phase is "one pass over the image + a grid barrier".  The image
// (<= a few tens of MB) stays in L2 between passes.  A CTA owns a contiguous chunk and a warp a contiguous piece of
// it, so that prefix sums in raster order (np.cumsum + searchsorted of the seeding) only need the per-block and
// per-warp partial sums, which stay in shared memory across the barriers.  Block partials are reduced in a fixed
// order by every CTA, so all CTAs take the same decisions and results do not depend on scheduling.  In one
// dimension clusters are intervals, so "labels unchanged" is "cluster sizes unchanged" (centre order is
// preserved by the Lloyd update): no label array is kept between iterations.
#include <math.h>
#include <string.h>
#include "hipr_common.cuh"

namespace hipr {

constexpr int KM_THREADS = 512;
constexpr int KM_WARPS = KM_THREADS / 32;
constexpr int KM_MAXK = 8;
constexpr int KM_MAXTRIALS = 4;      // 2 + int(log(k)) for k <= 8
constexpr int KM_MAXU = 256;         // uniforms: n_init * (1 + trials * (k - 1))
constexpr int KM_MAXGRID = 2048;
constexpr int KM_SLOT = 2 * KM_MAXK; // doubles per block per parity

struct KmUniforms {
    double u[KM_MAXU];
};

struct KmWork {                       // global scratch, zeroed (first 64 bytes) before the launch
    unsigned int barrier;
    unsigned int pad[15];
    double cand[KM_MAXTRIALS];        // centred values of the seeding candidates
    double first;                     // centred value of the first seed
    double blockcnt[KM_MAXGRID];      // valid samples per block (pass 0), kept for the first-seed rank search
    double part[2][KM_MAXGRID][KM_SLOT];
};

struct KmCtx {
    const void *x;
    int dtype;         // HIPR_F32 / HIPR_F64
    int transform;     // 0 none, 1 log10(x + eps), 2 ln(x + eps)
    int positive_only;
    double eps;
};

__device__ __forceinline__ bool km_load(const KmCtx &c, int64_t i, double &v, double &raw) {
    raw = (c.dtype == HIPR_F32) ? (double)reinterpret_cast<const float *>(c.x)[i] : reinterpret_cast<const double *>(c.x)[i];
    if (c.positive_only && !(raw > 0.0)) return false;
    v = raw;
    if (c.transform == 1) v = log10(raw + c.eps);
    else if (c.transform == 2) v = log(raw + c.eps);
    return true;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// result layout (doubles)
enum { KR_STATUS = 0, KR_NVALID = 1, KR_MEAN = 2, KR_TOL = 3, KR_NITER = 4, KR_INERTIA = 5, KR_BEST_INIT = 6, KR_BRIGHT = 7,
       KR_CENTERS = 8, KR_COUNTS = 16, KR_POSMEAN = 24, KR_SIZE = 32 };

__global__ void __launch_bounds__(KM_THREADS)
kmeans1d_kernel(KmCtx ctx, int64_t n, int k, int n_init, int max_iter, double tol_rel, const __grid_constant__ KmUniforms U,
                KmWork *__restrict__ work, int32_t *__restrict__ labels_out, int fill_label, uint8_t *__restrict__ mask_out,
                double *__restrict__ result) {
    __shared__ double s_warp[KM_WARPS][KM_SLOT];     // per-warp partials of the current pass
    __shared__ double s_red[KM_SLOT + 4];
    __shared__ double s_cnt_warp[KM_WARPS];          // valid samples per warp piece (fixed for the whole call)
    const int G = gridDim.x, b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned int bar_target = 0;
    int parity = 0;

    // contiguous chunk per CTA, contiguous piece per warp (multiples of 32 elements)
    const int64_t chunk = ((n + G - 1) / G + 32 * KM_WARPS - 1) / (32 * KM_WARPS) * (32 * KM_WARPS);
    const int64_t piece = chunk / KM_WARPS;
    const int64_t c0 = (int64_t)b * chunk;
    const int64_t w0 = c0 + (int64_t)warp * piece;
    const int64_t w1 = (w0 + piece < n) ? w0 + piece : n;

    auto grid_barrier = [&]() { hipr::grid_barrier(&work->barrier, bar_target); };
    // every thread holds `nv` partial values v[0..nv): reduce over the block, publish the block partial in this
    // parity's slot, barrier, then every CTA sums all block partials in block order into tot[] (identical everywhere)
    auto reduce_all = [&](double *v, int nv, double *tot) {
        for (int j = 0; j < nv; ++j) {
            const double s = warp_sum(v[j]);
            if (lane == 0) s_warp[warp][j] = s;
        }
        __syncthreads();
        if (tid < nv) {
            double s = 0.0;
            for (int w = 0; w < KM_WARPS; ++w) s += s_warp[w][tid];
            work->part[parity][b][tid] = s;
        }
        grid_barrier();
        if (tid < nv) {
            double s = 0.0;
            for (int g = 0; g < G; ++g) s += __ldcg(&work->part[parity][g][tid]);
            s_red[tid] = s;
        }
        __syncthreads();
        for (int j = 0; j < nv; ++j) tot[j] = s_red[j];
        __syncthreads();
        parity ^= 1;
    };
    // after reduce_all(v, 1, ..) of a pass whose v[0] is a weight sum: finds, for each of `nt` targets r[m], the first
    // sample (raster order over the valid samples) whose inclusive prefix sum of weights reaches r[m], and stores its
    // centred value in out_global[m].  weight(i, value) is re-evaluated by the owning warp.  Uses the partials of the
    // pass just reduced: slot index 0 of parity^1 (block sums) and s_warp[.][0] (warp sums).  Blocks and warps without
    // a valid sample are skipped (their sums are exactly 0, so the prefixes do not change): a target r <= 0, which
    // k-means++ draws once the seeds cover every distinct value, then picks the first valid sample, as searchsorted
    // does.  Where rounding leaves r above every prefix of the blocks, or of the chosen block's warps, the last valid
    // sample there is taken (numpy clips to the last index).  Exactly one warp writes out_global[m].
    auto locate = [&](const double *r, int nt, double mean, auto weight, double *out_global) {
        const int pp = parity ^ 1;
        for (int m = 0; m < nt; ++m) {
            // block: first g with prefix_inclusive >= r (all CTAs agree)
            double target = r[m], before = 0.0;
            int gb = -1, glast = -1;
            for (int g = 0; g < G; ++g) {
                if (!(__ldcg(&work->blockcnt[g]) > 0.0)) continue;
                glast = g;
                const double s = __ldcg(&work->part[pp][g][0]);
                if (before + s >= target) { gb = g; break; }
                before += s;
            }
            if (gb < 0) { gb = glast; target = INFINITY; }
            if (gb != b) continue;
            double wbefore = before;
            int wb = -1, wlast = -1;
            for (int w = 0; w < KM_WARPS; ++w) {
                if (!(s_cnt_warp[w] > 0.0)) continue;
                wlast = w;
                if (wbefore + s_warp[w][0] >= target) { wb = w; break; }
                wbefore += s_warp[w][0];
            }
            if (wb < 0) { wb = wlast; target = INFINITY; }
            if (wb != warp) continue;
            // this warp: walk the piece 32 samples at a time with an inclusive warp scan
            double run = wbefore, found_val = 0.0, last_valid = 0.0;
            bool found = false;
            for (int64_t i0 = w0; i0 < w1 && !found; i0 += 32) {
                const int64_t i = i0 + lane;
                double v = 0.0, raw, wgt = 0.0;
                bool ok = false;
                if (i < w1 && km_load(ctx, i, v, raw)) {
                    ok = true;
                    v -= mean;
                    wgt = weight(v);
                }
                double inc = wgt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const double t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, ok && (run + inc >= target));
                const unsigned okm = __ballot_sync(0xffffffffu, ok);
                if (okm) last_valid = __shfl_sync(0xffffffffu, v, 31 - __clz(okm));
                if (hit) {
                    found = true;
                    found_val = __shfl_sync(0xffffffffu, v, __ffs(hit) - 1);
                }
                run += __shfl_sync(0xffffffffu, inc, 31);
            }
            // rounding can leave the target just above the warp's last prefix: the warp has a valid sample, take its last
            if (lane == 0) out_global[m] = found ? found_val : last_valid;
        }
    };

    // ---- pass 0: valid count, sum -> mean; then variance -> tolerance -----------------------------------------
    double acc[KM_SLOT], tot[KM_SLOT];
    {
        double cnt = 0.0, sum = 0.0, bad = 0.0;
        for (int64_t i = w0 + lane; i < w1; i += 32) {
            double v, raw;
            if (km_load(ctx, i, v, raw)) {
                cnt += 1.0;
                sum += v;
                if (!(fabs(v) < 1.7e308)) bad += 1.0;
            }
        }
        const double wc = warp_sum(cnt);
        if (lane == 0) s_cnt_warp[warp] = wc;
        acc[0] = cnt; acc[1] = sum; acc[2] = bad;
        reduce_all(acc, 3, tot);
    }
    const double n_valid = tot[0];
    // keep this block's valid count where later passes do not overwrite it (read after the next grid barrier)
    if (tid == 0) work->blockcnt[b] = work->part[parity ^ 1][b][0];
    int status = 0;
    if (tot[2] > 0.0) status = 2;                     // NaN / inf among the samples (scikit-learn raises)
    else if (n_valid < (double)k) status = 4;
    const double mean = (n_valid > 0.0) ? tot[1] / n_valid : 0.0;
    if (status) {
        if (b == 0 && tid == 0) {
            for (int j = 0; j < KR_SIZE; ++j) result[j] = 0.0;
            result[KR_STATUS] = (double)status;
            result[KR_NVALID] = n_valid;
        }
        return;
    }
    {
        double ss = 0.0;
        for (int64_t i = w0 + lane; i < w1; i += 32) {
            double v, raw;
            if (km_load(ctx, i, v, raw)) ss += (v - mean) * (v - mean);
        }
        acc[0] = ss;
        reduce_all(acc, 1, tot);
    }
    const double tol_abs = tol_rel * tot[0] / n_valid;    // np.mean(np.var(X, axis=0)) * tol

    const int trials = 2 + (int)log((double)k);
    const int u_per_init = 1 + trials * (k - 1);
    double best_inertia = 0.0, best_c[KM_MAXK];
    int best_init = -1, best_iter = 0;
    double best_cnt[KM_MAXK];
    for (int j = 0; j < KM_MAXK; ++j) { best_c[j] = 0.0; best_cnt[j] = 0.0; }

    for (int init = 0; init < n_init && status == 0; ++init) {
        const double *u = U.u + init * u_per_init;
        double cen[KM_MAXK];
        // ---- k-means++ : first seed = sample floor(u * n_valid) of the valid samples, raster order ---------------
        {
            double rank = floor(u[0] * n_valid);
            if (rank > n_valid - 1.0) rank = n_valid - 1.0;
            // weights = 1 per valid sample; the per-warp counts are in s_cnt_warp, block counts from pass 0
            const double target = rank + 1.0;
            // block search on the pass-0 counts
            {
                double before = 0.0;
                int gb = G - 1;
                for (int g = 0; g < G; ++g) {
                    const double s = __ldcg(&work->blockcnt[g]);
                    if (before + s >= target) { gb = g; break; }
                    before += s;
                }
                if (gb == b) {
                    double wbefore = before;
                    int wb = KM_WARPS - 1;
                    for (int w = 0; w < KM_WARPS; ++w) {
                        if (wbefore + s_cnt_warp[w] >= target) { wb = w; break; }
                        wbefore += s_cnt_warp[w];
                    }
                    if (wb == warp) {
                        double run = wbefore;
                        bool found = false;
                        for (int64_t i0 = w0; i0 < w1 && !found; i0 += 32) {
                            const int64_t i = i0 + lane;
                            double v = 0.0, raw;
                            const bool ok = (i < w1) && km_load(ctx, i, v, raw);
                            const unsigned okm = __ballot_sync(0xffffffffu, ok);
                            const double inc = run + (double)__popc(okm & ((2u << lane) - 1u));
                            const unsigned hit = __ballot_sync(0xffffffffu, ok && inc >= target);
                            if (hit) {
                                found = true;
                                const double fv = __shfl_sync(0xffffffffu, v, __ffs(hit) - 1);
                                if (lane == 0) work->first = fv - mean;
                            }
                            run += (double)__popc(okm);
                        }
                    }
                }
            }
            grid_barrier();
            cen[0] = __ldcg(&work->first);
        }
        double pot = 0.0;
        for (int c = 1; c < k; ++c) {
            // closest squared distance to the seeds chosen so far, recomputed on the fly (no per-sample storage)
            auto closest = [&](double v) {
                double d = (v - cen[0]) * (v - cen[0]);
                for (int j = 1; j < c; ++j) d = fmin(d, (v - cen[j]) * (v - cen[j]));
                return d;
            };
            {
                double s = 0.0;
                for (int64_t i = w0 + lane; i < w1; i += 32) {
                    double v, raw;
                    if (km_load(ctx, i, v, raw)) s += closest(v - mean);
                }
                acc[0] = s;
                reduce_all(acc, 1, tot);
            }
            if (c == 1) pot = tot[0];           // later rounds carry the chosen candidate's potential, as scikit-learn does
            double r[KM_MAXTRIALS];
            for (int m = 0; m < trials; ++m) r[m] = u[1 + (c - 1) * trials + m] * pot;
            locate(r, trials, mean, closest, work->cand);
            grid_barrier();
            double cand[KM_MAXTRIALS];
            for (int m = 0; m < trials; ++m) cand[m] = __ldcg(&work->cand[m]);
            {
                for (int m = 0; m < trials; ++m) acc[m] = 0.0;
                for (int64_t i = w0 + lane; i < w1; i += 32) {
                    double v, raw;
                    if (km_load(ctx, i, v, raw)) {
                        v -= mean;
                        const double d = closest(v);
                        for (int m = 0; m < trials; ++m) acc[m] += fmin(d, (v - cand[m]) * (v - cand[m]));
                    }
                }
                reduce_all(acc, trials, tot);
            }
            int bestm = 0;
            for (int m = 1; m < trials; ++m)
                if (tot[m] < tot[bestm]) bestm = m;
            pot = tot[bestm];
            cen[c] = cand[bestm];
        }
        // ---- Lloyd ------------------------------------------------------------------------------------------------
        double cnt_old[KM_MAXK];
        for (int j = 0; j < k; ++j) cnt_old[j] = -1.0;
        int n_iter = 0;
        for (int it = 0; it < max_iter; ++it) {
            double c2[KM_MAXK];
            for (int j = 0; j < k; ++j) c2[j] = cen[j] * cen[j];
            for (int j = 0; j < 2 * k; ++j) acc[j] = 0.0;
            for (int64_t i = w0 + lane; i < w1; i += 32) {
                double v, raw;
                if (km_load(ctx, i, v, raw)) {
                    v -= mean;
                    int lab = 0;
                    double dbest = c2[0] - 2.0 * v * cen[0];
                    for (int j = 1; j < k; ++j) {
                        const double d = c2[j] - 2.0 * v * cen[j];
                        if (d < dbest) { dbest = d; lab = j; }
                    }
#pragma unroll
                    for (int j = 0; j < KM_MAXK; ++j)
                        if (j == lab) { acc[2 * j] += 1.0; acc[2 * j + 1] += v; }
                }
            }
            reduce_all(acc, 2 * k, tot);
            n_iter = it + 1;
            double shift = 0.0;
            bool same = true, empty = false;
            for (int j = 0; j < k; ++j) {
                if (tot[2 * j] <= 0.0) { empty = true; continue; }
                const double cn = tot[2 * j + 1] / tot[2 * j];
                shift += (cn - cen[j]) * (cn - cen[j]);
                cen[j] = cn;
                same = same && (tot[2 * j] == cnt_old[j]);
                cnt_old[j] = tot[2 * j];
            }
            if (empty) { status = 3; break; }            // scikit-learn relocates empty clusters: not reproduced
            if (same) break;                             // strict convergence: labels did not change
            if (shift <= tol_abs) break;
        }
        if (status) break;
        // ---- inertia and cluster sizes under the final centres -------------------------------------------------------
        {
            double c2[KM_MAXK];
            for (int j = 0; j < k; ++j) c2[j] = cen[j] * cen[j];
            for (int j = 0; j <= k; ++j) acc[j] = 0.0;
            for (int64_t i = w0 + lane; i < w1; i += 32) {
                double v, raw;
                if (km_load(ctx, i, v, raw)) {
                    v -= mean;
                    int lab = 0;
                    double dbest = c2[0] - 2.0 * v * cen[0];
                    for (int j = 1; j < k; ++j) {
                        const double d = c2[j] - 2.0 * v * cen[j];
                        if (d < dbest) { dbest = d; lab = j; }
                    }
                    double cl = cen[0];
#pragma unroll
                    for (int j = 0; j < KM_MAXK; ++j)
                        if (j == lab) { acc[j] += 1.0; cl = cen[j]; }
                    acc[k] += (v - cl) * (v - cl);
                }
            }
            reduce_all(acc, k + 1, tot);
        }
        // best of n_init: better inertia and a different clustering (in 1-D the cluster sizes in centre order identify it)
        bool take = (best_init < 0);
        if (!take && tot[k] < best_inertia) {
            double a[KM_MAXK], bb[KM_MAXK], ca[KM_MAXK], cb[KM_MAXK];
            for (int j = 0; j < k; ++j) { a[j] = tot[j]; ca[j] = cen[j]; bb[j] = best_cnt[j]; cb[j] = best_c[j]; }
            for (int p = 1; p < k; ++p)              // insertion sort of (centre, size) pairs by centre
                for (int q = p; q > 0; --q) {
                    if (ca[q] < ca[q - 1]) { double t = ca[q]; ca[q] = ca[q - 1]; ca[q - 1] = t; t = a[q]; a[q] = a[q - 1]; a[q - 1] = t; }
                    if (cb[q] < cb[q - 1]) { double t = cb[q]; cb[q] = cb[q - 1]; cb[q - 1] = t; t = bb[q]; bb[q] = bb[q - 1]; bb[q - 1] = t; }
                }
            bool same_clustering = true;
            for (int j = 0; j < k; ++j) same_clustering = same_clustering && (a[j] == bb[j]);
            take = !same_clustering;
        }
        if (take) {
            best_init = init;
            best_inertia = tot[k];
            best_iter = n_iter;
            for (int j = 0; j < k; ++j) { best_c[j] = cen[j]; best_cnt[j] = tot[j]; }
        }
    }

    if (status) {
        if (b == 0 && tid == 0) {
            for (int j = 0; j < KR_SIZE; ++j) result[j] = 0.0;
            result[KR_STATUS] = (double)status;
            result[KR_NVALID] = n_valid;
        }
        return;
    }
    // ---- per-cluster mean of the positive raw values (the scripts orient their masks by it), then labels / mask ----
    {
        double c2[KM_MAXK];
        for (int j = 0; j < k; ++j) c2[j] = best_c[j] * best_c[j];
        for (int j = 0; j < 2 * k; ++j) acc[j] = 0.0;
        for (int64_t i = w0 + lane; i < w1; i += 32) {
            double v, raw;
            if (km_load(ctx, i, v, raw)) {
                v -= mean;
                int lab = 0;
                double dbest = c2[0] - 2.0 * v * best_c[0];
                for (int j = 1; j < k; ++j) {
                    const double d = c2[j] - 2.0 * v * best_c[j];
                    if (d < dbest) { dbest = d; lab = j; }
                }
                if (raw > 0.0) {
#pragma unroll
                    for (int j = 0; j < KM_MAXK; ++j)
                        if (j == lab) { acc[2 * j] += 1.0; acc[2 * j + 1] += raw; }
                }
            }
        }
        reduce_all(acc, 2 * k, tot);
    }
    int bright = 0;
    double pm[KM_MAXK];
    for (int j = 0; j < k; ++j) pm[j] = (tot[2 * j] > 0.0) ? tot[2 * j + 1] / tot[2 * j] : -1.7e308;
    for (int j = 1; j < k; ++j)
        if (pm[j] > pm[bright]) bright = j;              // np.argmax: first maximum
    if (labels_out || mask_out) {
        double c2[KM_MAXK];
        for (int j = 0; j < k; ++j) c2[j] = best_c[j] * best_c[j];
        for (int64_t i = w0 + lane; i < w1; i += 32) {
            double v, raw;
            int lab = fill_label;
            bool ok = km_load(ctx, i, v, raw);
            if (ok) {
                v -= mean;
                lab = 0;
                double dbest = c2[0] - 2.0 * v * best_c[0];
                for (int j = 1; j < k; ++j) {
                    const double d = c2[j] - 2.0 * v * best_c[j];
                    if (d < dbest) { dbest = d; lab = j; }
                }
            }
            if (labels_out) labels_out[i] = lab;
            if (mask_out) mask_out[i] = (ok && lab == bright) ? 1 : 0;
        }
    }
    if (b == 0 && tid == 0) {
        for (int j = 0; j < KR_SIZE; ++j) result[j] = 0.0;
        result[KR_STATUS] = 0.0;
        result[KR_NVALID] = n_valid;
        result[KR_MEAN] = mean;
        result[KR_TOL] = tol_abs;
        result[KR_NITER] = (double)best_iter;
        result[KR_INERTIA] = best_inertia;
        result[KR_BEST_INIT] = (double)best_init;
        result[KR_BRIGHT] = (double)bright;
        for (int j = 0; j < k; ++j) {
            result[KR_CENTERS + j] = best_c[j] + mean;
            result[KR_COUNTS + j] = best_cnt[j];
            result[KR_POSMEAN + j] = pm[j];
        }
    }
}

}  // namespace hipr

using namespace hipr;

extern "C" int64_t hipr_kmeans1d_workspace_bytes(void) { return (int64_t)sizeof(KmWork); }

extern "C" int hipr_kmeans1d_uniforms(int k, int n_init) {
    if (k < 2 || k > KM_MAXK || n_init < 1) return HIPR_E_ARG;
    const int trials = 2 + (int)log((double)k);
    const int64_t n = (int64_t)n_init * (1 + trials * (k - 1));
    return n > KM_MAXU ? HIPR_E_RANGE : (int)n;
}

extern "C" int hipr_kmeans1d(const void *image_dev, int dtype, int64_t n, int transform, double eps, int positive_only,
                             int k, int n_init, const double *uniforms_host, int max_iter, double tol,
                             void *workspace_dev, int32_t *labels_out_dev, int fill_label, uint8_t *mask_out_dev,
                             double *result_dev, void *stream) {
    if (!image_dev || !uniforms_host || !workspace_dev || !result_dev || n < 1 || max_iter < 1 || !(tol >= 0.0))
        return HIPR_E_ARG;
    if (dtype != HIPR_F32 && dtype != HIPR_F64) return HIPR_E_DTYPE;
    if (transform < 0 || transform > 2) return HIPR_E_ARG;
    const int nu = hipr_kmeans1d_uniforms(k, n_init);
    if (nu < 0) return nu;
    cudaStream_t st = (cudaStream_t)stream;
    KmUniforms U;
    memset(&U, 0, sizeof(U));
    for (int i = 0; i < nu; ++i) {
        if (!(uniforms_host[i] >= 0.0 && uniforms_host[i] < 1.0)) return HIPR_E_ARG;
        U.u[i] = uniforms_host[i];
    }
    int dev = 0, sms = 0, per_sm = 0, coop = 0;
    HIPR_CUDA(cudaGetDevice(&dev));
    HIPR_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) return HIPR_E_UNSUPPORTED;
    HIPR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    HIPR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kmeans1d_kernel, KM_THREADS, 0));
    if (per_sm < 1) return HIPR_E_UNSUPPORTED;
    if (per_sm > 2) per_sm = 2;
    int64_t grid = (int64_t)sms * per_sm;
    const int64_t min_chunk = 32 * KM_WARPS;
    if (grid > (n + min_chunk - 1) / min_chunk) grid = (n + min_chunk - 1) / min_chunk;
    if (grid > KM_MAXGRID) grid = KM_MAXGRID;
    HIPR_CUDA(cudaMemsetAsync(workspace_dev, 0, 64, st));
    KmCtx ctx{image_dev, dtype, transform, positive_only ? 1 : 0, eps};
    KmWork *work = reinterpret_cast<KmWork *>(workspace_dev);
    void *args[] = {&ctx, &n, &k, &n_init, &max_iter, &tol, &U, &work, &labels_out_dev, &fill_label, &mask_out_dev, &result_dev};
    HIPR_CUDA(cudaLaunchCooperativeKernel((const void *)kmeans1d_kernel, dim3((unsigned)grid), dim3(KM_THREADS), args, 0, st));
    return after_launch();
}

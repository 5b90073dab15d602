// K7: per-cell geometry and paint-by-label, the consumers of the label image next to the per-cell spectra.
//
// cell geometry: skimage.measure.regionprops(segmentation) -> label, area, centroid, major / minor axis
//   length, eccentricity, orientation: syn/hiprfish_imaging_classify_spectra.py:38-46,
//   bio/..._analysis.py:1232-1240.  One pass over the label image accumulates, per label, the integer raw
//   moments (count, sum r, sum c, sum r^2, sum c^2, sum r c) with 64-bit integer atomics -- exact, order
//   independent -- and a finalize kernel derives the float64 properties for the labels present, ascending.
// paint by label: `image[segmentation == label] = value` for every cell (an O(cells x pixels) numpy loop at
//   eco/hiprfish_imaging_image_classification.py:64-70, bio/..._analysis.py:1247-1257) as one LUT gather.
#include "hipr_common.cuh"

namespace hipr {

constexpr int CG_STRIP = 32;   // consecutive pixels walked by one thread

// A thread walks CG_STRIP consecutive pixels, summing the moments of a run of equal labels in registers and
// flushing a run with six atomics (labels come from a watershed: runs are long).
template <typename LabelT>
__global__ void __launch_bounds__(256)
cell_moments_kernel(const LabelT *__restrict__ labels, int64_t npix, int W, int64_t max_label,
                    unsigned long long *__restrict__ mom /* (max_label + 1, 6) */) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t p0 = t * CG_STRIP;
    if (p0 >= npix) return;
    const int64_t p1 = (p0 + CG_STRIP < npix) ? p0 + CG_STRIP : npix;
    unsigned long long r = (unsigned long long)(p0 / W), c = (unsigned long long)(p0 % W);
    long long cur = 0;
    unsigned long long n = 0, sr = 0, sc = 0, srr = 0, scc = 0, src = 0;
    auto flush = [&]() {
        if (cur > 0 && n > 0) {
            unsigned long long *m = mom + cur * 6;
            atomicAdd(m + 0, n);
            atomicAdd(m + 1, sr);
            atomicAdd(m + 2, sc);
            atomicAdd(m + 3, srr);
            atomicAdd(m + 4, scc);
            atomicAdd(m + 5, src);
        }
        n = sr = sc = srr = scc = src = 0;
    };
    for (int64_t p = p0; p < p1; ++p) {
        long long lab = (long long)labels[p];
        if (lab > max_label) lab = 0;
        if (lab != cur) {
            flush();
            cur = lab;
        }
        if (lab > 0) {
            ++n;
            sr += r;
            sc += c;
            srr += r * r;
            scc += c * c;
            src += r * c;
        }
        if (++c == (unsigned long long)W) { c = 0; ++r; }
    }
    flush();
}

// One thread per present label (labels_out / n_cells from cell_compact_kernel's ordering): float64 properties.
// Central moments are formed exactly from the integer sums (128-bit products) before going to float64.
__global__ void __launch_bounds__(128)
cell_geometry_kernel(const unsigned long long *__restrict__ mom, const int *__restrict__ n_cells,
                     const long long *__restrict__ labels_out, double *__restrict__ geom /* (n, 9) */) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= *n_cells) return;
    const unsigned long long *m = mom + labels_out[row] * 6;
    const unsigned __int128 n = m[0];
    const double nd = (double)m[0];
    // n * sum(x^2) - (sum x)^2 >= 0 and n * sum(xy) - sum(x) sum(y), exact
    const unsigned __int128 a2 = n * m[3] - (unsigned __int128)m[1] * m[1];
    const unsigned __int128 c2 = n * m[4] - (unsigned __int128)m[2] * m[2];
    const __int128 b2 = (__int128)(n * m[5]) - (__int128)((unsigned __int128)m[1] * m[2]);
    const double mu20 = (double)a2 / nd, mu02 = (double)c2 / nd, mu11 = (double)b2 / nd;   // central moments
    const double a = mu20 / nd, c = mu02 / nd, b = mu11 / nd;                              // covariance of (r, c)
    const double tr = a + c, df = a - c;
    const double root = sqrt(df * df + 4.0 * b * b);
    const double l1 = fmax(0.5 * (tr + root), 0.0), l2 = fmax(0.5 * (tr - root), 0.0);
    double *g = geom + (int64_t)row * 9;
    g[0] = (double)m[1] / nd;                      // centroid row
    g[1] = (double)m[2] / nd;                      // centroid column
    g[2] = 4.0 * sqrt(l1);                         // major_axis_length
    g[3] = 4.0 * sqrt(l2);                         // minor_axis_length
    g[4] = (l1 == 0.0) ? 0.0 : sqrt(1.0 - l2 / l1);   // eccentricity
    // orientation, skimage >= 0.16 ('rc' coordinates): inertia tensor [[mu02, -mu11], [-mu11, mu20]] / n,
    // a_ = mu02 / n, b_ = -mu11 / n, c_ = mu20 / n;  a_ == c_: -pi/4 if b_ < 0 else pi/4;
    // else 0.5 * atan2(-2 b_, c_ - a_)
    const double ta = c, tb = -b, tc = a;
    const double quarter_pi = 0.78539816339744830962;
    g[5] = (ta - tc == 0.0) ? (tb < 0.0 ? -quarter_pi : quarter_pi) : 0.5 * atan2(-2.0 * tb, tc - ta);
    g[6] = mu20;
    g[7] = mu02;
    g[8] = mu11;
}

template <typename LabelT, typename T>
__global__ void __launch_bounds__(256)
paint_kernel(const LabelT *__restrict__ labels, int64_t npix, const T *__restrict__ values, int K, int64_t max_label,
             T *__restrict__ out) {
    const int64_t total = npix * K;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = i / K;
        const int k = (int)(i - p * K);
        long long lab = (long long)labels[p];
        if (lab < 0 || lab > max_label) lab = 0;
        out[i] = values[lab * K + k];
    }
}

// cell_spectra.cu: the labels present, ascending, and their pixel counts
int cell_compact_launch(const int *counts, int64_t max_label, int *n_cells, long long *labels_out, long long *area_out,
                        cudaStream_t st);

__global__ void __launch_bounds__(256)
moments_counts_kernel(const unsigned long long *__restrict__ mom, int64_t max_label, int *__restrict__ counts) {
    for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l <= max_label; l += (int64_t)gridDim.x * blockDim.x)
        counts[l] = (int)mom[l * 6];
}

}  // namespace hipr

using namespace hipr;

extern "C" int hipr_cell_moments(const void *labels_dev, int label_bytes, int H, int W, int64_t max_label,
                                 uint64_t *moments_dev, void *stream) {
    if (!labels_dev || !moments_dev || H < 1 || W < 1 || max_label < 0) return HIPR_E_ARG;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    const int64_t npix = (int64_t)H * W;
    if (npix > 0x7fffffffLL) return HIPR_E_RANGE;
    cudaStream_t st = (cudaStream_t)stream;
    HIPR_CUDA(cudaMemsetAsync(moments_dev, 0, (size_t)(max_label + 1) * 6 * sizeof(uint64_t), st));
    const int64_t threads = (npix + CG_STRIP - 1) / CG_STRIP;
    const unsigned blocks = (unsigned)((threads + 255) / 256);
    unsigned long long *mom = reinterpret_cast<unsigned long long *>(moments_dev);
    if (label_bytes == 4)
        cell_moments_kernel<int><<<blocks, 256, 0, st>>>((const int *)labels_dev, npix, W, max_label, mom);
    else
        cell_moments_kernel<long long><<<blocks, 256, 0, st>>>((const long long *)labels_dev, npix, W, max_label, mom);
    return after_launch();
}

extern "C" int hipr_cell_geometry_finalize(const uint64_t *moments_dev, int64_t max_label, int32_t *counts_scratch_dev,
                                           int32_t *n_cells_dev, int64_t *labels_out, int64_t *area_out,
                                           double *geometry_out, void *stream) {
    if (!moments_dev || !counts_scratch_dev || !n_cells_dev || !labels_out || !area_out || !geometry_out || max_label < 0)
        return HIPR_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long *mom = reinterpret_cast<const unsigned long long *>(moments_dev);
    int64_t blocks = (max_label + 256) / 256;
    if (blocks > 1184) blocks = 1184;
    moments_counts_kernel<<<(unsigned)blocks, 256, 0, st>>>(mom, max_label, counts_scratch_dev);
    int e = after_launch();
    if (e) return e;
    if ((e = cell_compact_launch(counts_scratch_dev, max_label, n_cells_dev, (long long *)labels_out,
                                 (long long *)area_out, st)))
        return e;
    const int64_t rows = max_label > 0 ? max_label : 1;
    cell_geometry_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(mom, n_cells_dev, (const long long *)labels_out,
                                                                       geometry_out);
    return after_launch();
}

extern "C" int hipr_paint_labels(const void *labels_dev, int label_bytes, int64_t npix, const void *values_dev, int K,
                                 int64_t max_label, int dtype, void *out_dev, void *stream) {
    if (!labels_dev || !values_dev || !out_dev || npix < 1 || K < 1 || max_label < 0) return HIPR_E_ARG;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    if (dtype < HIPR_F32 || dtype > HIPR_U8) return HIPR_E_DTYPE;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t blocks = (npix * K + 1023) / 1024;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
#define HIPR_PAINT(LT, VT)                                                                                         \
    paint_kernel<LT, VT><<<(unsigned)blocks, 256, 0, st>>>((const LT *)labels_dev, npix, (const VT *)values_dev, K, \
                                                          max_label, (VT *)out_dev)
#define HIPR_PAINT_VALUES(LT)                                 \
    switch (dtype) {                                          \
        case HIPR_F32: HIPR_PAINT(LT, float); break;          \
        case HIPR_F64: HIPR_PAINT(LT, double); break;         \
        case HIPR_I32: HIPR_PAINT(LT, int); break;            \
        case HIPR_I64: HIPR_PAINT(LT, long long); break;      \
        default: HIPR_PAINT(LT, uint8_t); break;              \
    }
    if (label_bytes == 4) { HIPR_PAINT_VALUES(int) }
    else { HIPR_PAINT_VALUES(long long) }
#undef HIPR_PAINT_VALUES
#undef HIPR_PAINT
    return after_launch();
}

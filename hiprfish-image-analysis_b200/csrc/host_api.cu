// ABI housekeeping and the host-buffer entry points: what a numpy caller binds.  The cube is
// streamed host -> device in row bands on a copy stream while the channel sum (or the per-cell
// accumulation) of the previous band runs on a compute stream, so the end-to-end time is the
// PCIe time of the cube plus a short tail.  Every entry point on the per-device workspace opens a
// CallScope; cubes go up through upload_bands, large results come down through banded_to_host,
// and the 2-D score tail is score2d.
#include <mutex>
#include <string.h>
#include <cstdlib>
#include <thread>
#include <vector>
#include <cstdio>
#include "hipr_common.cuh"

// in this file a failing CUDA call also reports where, when HIPR_DEBUG is set (the host pipelines enqueue dozens of
// calls per entry point; the ABI's return value only carries the code)
#undef HIPR_CUDA
#define HIPR_CUDA(expr)                                                                             \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            if (getenv("HIPR_DEBUG")) fprintf(stderr, "hipr: %s:%d: %s -> %s\n", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return (int)_e;                                                                         \
        }                                                                                           \
    } while (0)

namespace hipr {

std::atomic<int64_t> g_launches{0};

int chansum_band(const void *cube, int sample_bytes, float scale, int64_t npix, int C, double *out,
                 unsigned long long *maxkey, cudaStream_t st);
template <typename T>
int gather_launch(const T *src, int64_t stride_a, int64_t stride_b, int inner, int64_t nrows, int rowlen, int K,
                  const int *offs, T *out, cudaStream_t st);
int check_table(const int32_t *table, int n_dirs, int P, int ndim);

// A grow-only device (or page-locked host) buffer.  The recorded size is 0 until a new allocation has succeeded, so a
// failed reserve is retried by the next call.
template <bool HOST>
struct Buf {
    void *p = nullptr;
    size_t bytes = 0;
    int reserve(size_t n) {
        if (n <= bytes) return HIPR_OK;
        release();
        HIPR_CUDA(HOST ? cudaHostAlloc(&p, n, cudaHostAllocDefault) : cudaMalloc(&p, n));
        bytes = n;
        return HIPR_OK;
    }
    void release() {
        if (p) HOST ? cudaFreeHost(p) : cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};
using DevBuf = Buf<false>;
using HostBuf = Buf<true>;

// An error return after the first enqueue must not leave copies from the caller's buffers (or into them) in flight:
// the caller may free them.  Unless disarmed, the guard synchronises its streams on scope exit.
struct Drain {
    cudaStream_t s[3] = {};
    bool armed = true;
    ~Drain() {
        if (!armed) return;
        for (cudaStream_t st : s)
            if (st) cudaStreamSynchronize(st);
    }
};

constexpr int NBUF = 3;
struct Workspace {
    std::mutex mu;
    cudaStream_t copy = nullptr, comp = nullptr;
    cudaEvent_t copied[NBUF] = {}, freed[NBUF] = {};
    cudaEvent_t staged_out[NBUF] = {};   // the copy out of stage[i] has completed
    cudaEvent_t t0 = nullptr, t1 = nullptr;   // device-side timing of the last host call
    float last_ms = -1.f;
    DevBuf band[NBUF];
    // pageable callers: page-locked staging ring the caller's array is copied through by a few host threads
    HostBuf stage[NBUF];
    // batch entry point (hipr_neighbor2d_host_batch): a third stream for denoise + stencil + score read-back of FOV i
    // while FOV i + 1 is uploaded and summed, and two sets of per-image buffers (the other entry points use img[0])
    cudaStream_t post = nullptr;
    cudaEvent_t summed[2] = {}, post_done[2] = {};
    struct Image {
        DevBuf sum;       // float64 channel sums
        DevBuf score;     // float32 score, then the float32 normalised sum
        DevBuf keys;      // range keys (64 bytes)
        DevBuf scratch;   // float64: the denoised image, then the float64 score
    } img[2];
    DevBuf input;         // an input uploaded whole: the padded gather input, a label image
    DevBuf extra;         // the 3-D denoise's padded copy
    // the cell table of the last hipr_cell_spectra_host call stays here for hipr_cell_spectra_host_fetch
    DevBuf cells;
    int64_t last_cells = -1, last_max_label = 0;
    int last_C = 0;
    bool ready = false;

    void release() {
        for (int i = 0; i < NBUF; ++i) {
            band[i].release();
            stage[i].release();
        }
        for (Image &m : img)
            for (DevBuf *b : {&m.sum, &m.score, &m.keys, &m.scratch}) b->release();
        for (DevBuf *b : {&input, &extra, &cells}) b->release();
    }
};
// One workspace per device: its streams, events and buffers belong to the device that was current when they were
// created, so a process that drives several GPUs (or switches devices between calls) never shares them.
constexpr int kMaxDevices = 32;
static Workspace g_ws_dev[kMaxDevices];
static thread_local float t_last_ms = -1.f;      // hipr_host_last_elapsed_ms: the calling thread's last host call

// host threads that copy a pageable array into the page-locked staging ring (HIPR_HOST_COPY_THREADS overrides)
static int host_copy_threads() {
    int n = (int)std::thread::hardware_concurrency();
    n = n > 8 ? 8 : n;                                      // measured with 8: 143 -> 48 ms per 1.59 GB cube
    if (const char *ev = getenv("HIPR_HOST_COPY_THREADS")) n = atoi(ev);
    return n > 16 ? 16 : (n < 1 ? 1 : n);
}

static int ws_init(Workspace &w) {
    if (w.ready) return HIPR_OK;
    HIPR_CUDA(cudaStreamCreateWithFlags(&w.copy, cudaStreamNonBlocking));
    // the compute stream (channel sums of the bands as they arrive) has the highest priority: the hardware dispatches a
    // later kernel's CTAs only when the earlier one has none left to dispatch, unless its stream's priority is higher --
    // without it a band's channel sum waits behind the whole denoise grid of the previous FOV on the `post` stream, the
    // band ring fills and the upload stalls (batch entry point: 33.6 ms per FOV instead of the PCIe time)
    int prio_lo = 0, prio_hi = 0;
    HIPR_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    HIPR_CUDA(cudaStreamCreateWithPriority(&w.comp, cudaStreamNonBlocking, prio_hi));
    for (int i = 0; i < NBUF; ++i) {
        HIPR_CUDA(cudaEventCreateWithFlags(&w.copied[i], cudaEventDisableTiming));
        HIPR_CUDA(cudaEventCreateWithFlags(&w.freed[i], cudaEventDisableTiming));
        HIPR_CUDA(cudaEventCreateWithFlags(&w.staged_out[i], cudaEventDisableTiming));
    }
    HIPR_CUDA(cudaStreamCreateWithFlags(&w.post, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        HIPR_CUDA(cudaEventCreateWithFlags(&w.summed[i], cudaEventDisableTiming));
        HIPR_CUDA(cudaEventCreateWithFlags(&w.post_done[i], cudaEventDisableTiming));
    }
    HIPR_CUDA(cudaEventCreate(&w.t0));
    HIPR_CUDA(cudaEventCreate(&w.t1));
    w.ready = true;
    return HIPR_OK;
}

// One entry point's use of the current device's workspace: open() finds it, takes its lock, creates its streams and
// events on first use and arms the drain over its three streams.  finish(last) ends a timed call: t1 on `last`, every
// stream synchronised, the device time from t0 stored for hipr_host_last_elapsed_ms.  done() ends an untimed one.
struct CallScope {
    Workspace *w = nullptr;
    std::unique_lock<std::mutex> lock;
    Drain drain{{}, false};          // armed by open(); declared after the lock, so it drains before the unlock
    int open() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return HIPR_E_NODEVICE;
        w = &g_ws_dev[dev];
        lock = std::unique_lock<std::mutex>(w->mu);
        int e = ws_init(*w);
        if (e) return e;
        drain.s[0] = w->copy;
        drain.s[1] = w->comp;
        drain.s[2] = w->post;
        drain.armed = true;
        return HIPR_OK;
    }
    int done() {
        for (cudaStream_t st : drain.s) HIPR_CUDA(cudaStreamSynchronize(st));
        drain.armed = false;
        return HIPR_OK;
    }
    int finish(cudaStream_t last) {
        HIPR_CUDA(cudaEventRecord(w->t1, last));
        int e = done();
        if (e) return e;
        HIPR_CUDA(cudaEventElapsedTime(&w->last_ms, w->t0, w->t1));
        t_last_ms = w->last_ms;
        return HIPR_OK;
    }
};

// band ring (and, for a pageable source or destination, the staging ring) of `bytes` per band
static int ws_ring(Workspace &w, size_t bytes, bool staged) {
    int e;
    for (int i = 0; i < NBUF; ++i) {
        if ((e = w.band[i].reserve(bytes))) return e;
        if (staged && (e = w.stage[i].reserve(bytes))) return e;
    }
    return HIPR_OK;
}

// true when `p` is ordinary pageable host memory (numpy's allocator): a direct cudaMemcpyAsync from it is staged by
// the driver at ~11 GB/s (measured: 143 ms for a 1.59 GB cube); page-locked memory goes at the PCIe rate
static bool is_pageable(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return attr.type == cudaMemoryTypeUnregistered;
}

// dst <- src with a few threads (one slice each)
static void parallel_copy(void *dst, const void *src, size_t bytes, int nthreads) {
    if (nthreads <= 1 || bytes < (4u << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    std::vector<std::thread> th;
    const size_t slice = ((bytes + nthreads - 1) / nthreads + 4095) & ~(size_t)4095;
    for (int t = 1; t < nthreads; ++t) {
        const size_t o = (size_t)t * slice;
        if (o >= bytes) break;
        const size_t n = (bytes - o < slice) ? bytes - o : slice;
        th.emplace_back([=] { memcpy((char *)dst + o, (const char *)src + o, n); });
    }
    memcpy(dst, src, slice < bytes ? slice : bytes);
    for (auto &t : th) t.join();
}

// rows per band so that a band is ~32 MiB and a whole number of rows
static int band_rows(int64_t row_bytes, int64_t nrows) {
    int64_t r = (32ll << 20) / (row_bytes > 0 ? row_bytes : 1);
    if (r < 1) r = 1;
    if (r > nrows) r = nrows;
    return (int)r;
}

// Host -> device in bands: `units` units of `unit_bytes` from src, `units_per_band` per band, through the band ring on
// the copy stream, while `consume(u0, nu, band_dev, comp)` reads the previous band on the compute stream.  A pageable
// src goes through the staging ring: host threads copy band b into it while band b - 1 crosses PCIe and band b - 2
// is consumed.  `band` counts the bands since the start of the call, so the ring slots carry over from one upload to
// the next.  The caller reserves the rings (ws_ring) for units_per_band units.
template <typename Consume>
static int upload_bands(Workspace &w, const void *src, int64_t units, int64_t unit_bytes, int64_t units_per_band,
                        int &band, Consume consume) {
    int e;
    const bool pageable = is_pageable(src);
    const int copy_threads = host_copy_threads();
    for (int64_t u0 = 0; u0 < units; u0 += units_per_band, ++band) {
        const int64_t nu = (units - u0 < units_per_band) ? units - u0 : units_per_band;
        const size_t bytes = (size_t)(nu * unit_bytes);
        const int slot = band % NBUF;
        const void *from = (const char *)src + u0 * unit_bytes;
        if (pageable) {
            if (band >= NBUF) HIPR_CUDA(cudaEventSynchronize(w.staged_out[slot]));
            parallel_copy(w.stage[slot].p, from, bytes, copy_threads);
            from = w.stage[slot].p;
        }
        if (band >= NBUF) HIPR_CUDA(cudaStreamWaitEvent(w.copy, w.freed[slot], 0));
        HIPR_CUDA(cudaMemcpyAsync(w.band[slot].p, from, bytes, cudaMemcpyHostToDevice, w.copy));
        if (pageable) HIPR_CUDA(cudaEventRecord(w.staged_out[slot], w.copy));
        HIPR_CUDA(cudaEventRecord(w.copied[slot], w.copy));
        HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.copied[slot], 0));
        if ((e = consume(u0, nu, (const void *)w.band[slot].p, w.comp))) return e;
        HIPR_CUDA(cudaEventRecord(w.freed[slot], w.comp));
    }
    return HIPR_OK;
}

// range keys before the first channel sum: max 0, min all ones
static int reset_keys(unsigned long long *keys, cudaStream_t st) {
    HIPR_CUDA(cudaMemsetAsync(keys, 0x00, 8, st));
    HIPR_CUDA(cudaMemsetAsync(keys + 1, 0xff, 8, st));
    return HIPR_OK;
}

// The 2-D score of an (H, W) float64 channel-sum image with its range keys, into the float32 `score` on `st`.
// denoise_h > 0: syn/..._measurement.py:106-124 in full, /max (in place) -> NL-means -> float64 stencil (the denoised
// image is too smooth for the fixed-point grid, DESIGN.md).  Otherwise the fixed-point stencil for the (11, 9) table
// every pipeline uses (F1 / F2: every tile quantised with its own range, the finest grid and the same as the
// device-resident pipeline, bit for bit; F3's epsilon needs the global range), and the float64 stencil for other
// parameters.  The float64 routes reserve `scratch` for 2 H W doubles: the denoised image, then the float64 score.
static int score2d(double *sum, const unsigned long long *keys, int H, int W, int patch_size, int n_dirs,
                   const int32_t *table, int flavour, double denoise_h, DevBuf &scratch, float *score, cudaStream_t st) {
    const int64_t npix = (int64_t)H * W;
    const uint64_t *range = (const uint64_t *)keys;
    int e;
    if (denoise_h <= 0.0) {
        const bool tile_local = (flavour == HIPR_FLAVOUR_F1 || flavour == HIPR_FLAVOUR_F2);
        e = hipr_lne2d_q(sum, H, W, W, 0, HIPR_F64, patch_size, n_dirs, table, flavour, tile_local ? nullptr : range,
                         score, st);
        if (e != HIPR_E_TABLE || (patch_size == 11 && n_dirs == 9)) return e;
    }
    if ((e = scratch.reserve((size_t)npix * 2 * sizeof(double)))) return e;
    double *den = (double *)scratch.p, *score64 = den + npix;
    const double *src = sum;
    if (denoise_h > 0.0) {
        if ((e = hipr_normalize(sum, HIPR_F64, npix, range, st))) return e;
        if ((e = hipr_denoise_nl_means_2d(sum, H, W, HIPR_F64, 7, 11, denoise_h, den, st))) return e;
        src = den;
        range = nullptr;
    }
    if ((e = hipr_lne2d(src, H, W, W, 0, HIPR_F64, patch_size, n_dirs, table, flavour, range, score64, st))) return e;
    return hipr_normalize_cast(score64, npix, nullptr, score, st);
}

// Per-cell table in one device buffer: the accumulators (sums (max_label + 1, C) float64, counts int32 padded to 16
// bytes, 16 bytes more; zeroed before the pass), then the finalized table: n (16 bytes), labels and areas (max_label)
// int64, avgint and avgint_norm (max_label, C) float64 -- the first n rows are valid.
struct CellTable {
    double *sums;
    int32_t *counts, *n;
    int64_t *labels, *area;
    double *avg, *norm;
    size_t acc_bytes;
};
static int cell_table(DevBuf &buf, int64_t max_label, int C, CellTable &t) {
    const size_t row_bytes = (size_t)C * 8, sums_bytes = (size_t)(max_label + 1) * row_bytes;
    const size_t cnt_bytes = ((size_t)(max_label + 1) * 4 + 15) & ~(size_t)15;
    t.acc_bytes = sums_bytes + cnt_bytes + 16;
    int e = buf.reserve(t.acc_bytes + 16 + (size_t)max_label * (16 + 2 * row_bytes));
    if (e) return e;
    char *base = (char *)buf.p, *fin = base + t.acc_bytes;
    t.sums = (double *)base;
    t.counts = (int32_t *)(base + sums_bytes);
    t.n = (int32_t *)fin;
    t.labels = (int64_t *)(fin + 16);
    t.area = t.labels + max_label;
    t.avg = (double *)(t.area + max_label);
    t.norm = t.avg + (size_t)max_label * C;
    return HIPR_OK;
}
static int copy_cell_table(const CellTable &t, int64_t n, int C, int64_t *labels_out, int64_t *area_out,
                           double *avgint_out, double *avgint_norm_out, cudaStream_t st) {
    HIPR_CUDA(cudaMemcpyAsync(labels_out, t.labels, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    HIPR_CUDA(cudaMemcpyAsync(area_out, t.area, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    HIPR_CUDA(cudaMemcpyAsync(avgint_out, t.avg, (size_t)n * C * 8, cudaMemcpyDeviceToHost, st));
    HIPR_CUDA(cudaMemcpyAsync(avgint_norm_out, t.norm, (size_t)n * C * 8, cudaMemcpyDeviceToHost, st));
    return HIPR_OK;
}
// finalize the accumulated table, read n back (*n_cells), and enqueue the copy of the table when it fits the caller's
// capacity; HIPR_E_RANGE when it does not (everything enqueued has then completed)
static int finalize_cells(const CellTable &t, int64_t max_label, int C, int64_t capacity, int64_t *n_cells,
                          int64_t *labels_out, int64_t *area_out, double *avgint_out, double *avgint_norm_out,
                          cudaStream_t st) {
    int e = hipr_cell_spectra_finalize(t.sums, t.counts, max_label, C, t.n, t.labels, t.area, t.avg, t.norm, st);
    if (e) return e;
    int32_t n = 0;
    HIPR_CUDA(cudaMemcpyAsync(&n, t.n, 4, cudaMemcpyDeviceToHost, st));
    HIPR_CUDA(cudaStreamSynchronize(st));
    *n_cells = n;
    if (n > capacity) return HIPR_E_RANGE;
    return n ? copy_cell_table(t, n, C, labels_out, area_out, avgint_out, avgint_norm_out, st) : HIPR_OK;
}

}  // namespace hipr

using namespace hipr;

extern "C" int hipr_abi_version(void) { return HIPR_ABI_VERSION; }

extern "C" int64_t hipr_launch_count(void) { return g_launches.load(); }

extern "C" int hipr_sm_count(void) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return HIPR_E_NODEVICE;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return HIPR_E_NODEVICE;
    return n;
}

extern "C" const char *hipr_error_string(int code) {
    switch (code) {
        case HIPR_OK: return "ok";
        case HIPR_E_ARG: return "invalid argument (null pointer or non-positive size)";
        case HIPR_E_DTYPE: return "unsupported dtype code";
        case HIPR_E_PATCH: return "patch_size must be odd, 3..31, and no larger than the image";
        case HIPR_E_TABLE: return "line table entry outside the patch, or table too large";
        case HIPR_E_FLAVOUR: return "unknown epilogue flavour for this entry point";
        case HIPR_E_ALIGN: return "pointer not aligned to its element type";
        case HIPR_E_RANGE: return "size exceeds the index range or the caller's capacity";
        case HIPR_E_NODEVICE: return "no CUDA device";
        case HIPR_E_UNSUPPORTED: return "request outside this entry point's fast path";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown error";
}

extern "C" int hipr_host_alloc(void **ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) return HIPR_E_ARG;
    HIPR_CUDA(cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault));
    return HIPR_OK;
}
extern "C" int hipr_host_free(void *ptr) {
    if (!ptr) return HIPR_OK;
    HIPR_CUDA(cudaFreeHost(ptr));
    return HIPR_OK;
}
static void fov_cache_release_current_device();
extern "C" int hipr_host_release_workspace(void) {
    fov_cache_release_current_device();
    CallScope call;
    int e = call.open();
    if (e) return e;
    cudaDeviceSynchronize();
    call.w->release();
    return call.done();
}

// cube_host: (H, W, C) samples of `sample_bytes` (4 = float32; 2 / 1 = raw uint16 / uint8 counts, value =
// float32(count) / float32(scale))
static int neighbor2d_host_impl(const void *cube_host, int sample_bytes, float scale, int H, int W, int C,
                                int patch_size, int n_dirs, const int32_t *table_host, int flavour, float *score_host,
                                float *sum_host, double denoise_h = 0.0) {
    if (!cube_host || !score_host || H < 1 || W < 1 || C < 1) return HIPR_E_ARG;
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    Workspace::Image &m = w.img[0];
    const int64_t row_bytes = (int64_t)W * C * sample_bytes;
    const int rows = band_rows(row_bytes, H);
    const size_t img_bytes = (size_t)H * W * 4;
    if ((e = ws_ring(w, (size_t)rows * row_bytes, is_pageable(cube_host))) || (e = m.sum.reserve(2 * img_bytes)) ||
        (e = m.score.reserve(img_bytes)) || (e = m.keys.reserve(64)))
        return e;
    double *sum_dev = (double *)m.sum.p;
    float *score_dev = (float *)m.score.p;
    unsigned long long *key = (unsigned long long *)m.keys.p;
    HIPR_CUDA(cudaEventRecord(w.t0, w.copy));            // device clock starts before the first H2D
    HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.t0, 0));
    if ((e = reset_keys(key, w.comp))) return e;
    int b = 0;
    e = upload_bands(w, cube_host, H, row_bytes, rows, b, [&](int64_t r0, int64_t nr, const void *band, cudaStream_t st) {
        return chansum_band(band, sample_bytes, scale, nr * W, C, sum_dev + r0 * W, key, st);
    });
    if (e || (e = score2d(sum_dev, key, H, W, patch_size, n_dirs, table_host, flavour, denoise_h, m.scratch, score_dev,
                          w.comp)))
        return e;
    HIPR_CUDA(cudaMemcpyAsync(score_host, score_dev, img_bytes, cudaMemcpyDeviceToHost, w.comp));
    if (sum_host) {
        // the normalised denoised image, or the sums with the range keys
        const bool den = denoise_h > 0.0;
        if ((e = hipr_normalize_cast(den ? (const double *)m.scratch.p : sum_dev, (int64_t)H * W,
                                     den ? nullptr : (const uint64_t *)key, score_dev, w.comp)))
            return e;
        HIPR_CUDA(cudaMemcpyAsync(sum_host, score_dev, img_bytes, cudaMemcpyDeviceToHost, w.comp));
    }
    return call.finish(w.comp);                          // ... and stops after the last D2H
}

extern "C" int hipr_neighbor2d_host(const float *cube_host, int H, int W, int C, int patch_size, int n_dirs,
                                    const int32_t *table_host, int flavour, float *score_host, float *sum_host) {
    return neighbor2d_host_impl(cube_host, 4, 1.f, H, W, C, patch_size, n_dirs, table_host, flavour, score_host, sum_host);
}

// Results that are far larger than their inputs (the literal gathers: 792 B per pixel, 576 B per voxel) leave the
// device in row bands: `produce(r0, nr, band_dev, stream)` fills a band of `nr` rows on the compute stream while the
// previous bands cross PCIe on the copy stream -- straight into out_host when it is page-locked, otherwise through
// the page-locked staging ring and a few host threads (a direct device -> pageable copy is staged by the driver at
// a few GB/s; measured 1.58 s for a 3.3 GB result against 0.10 s this way and 0.06 s into page-locked memory).
template <typename Produce>
static int banded_to_host(Workspace &w, int64_t nrows, int64_t row_bytes, void *out_host, Produce produce) {
    int e;
    const int rows = band_rows(row_bytes, nrows);
    const bool pageable = is_pageable(out_host);
    const int copy_threads = host_copy_threads();
    if ((e = ws_ring(w, (size_t)rows * row_bytes, pageable))) return e;
    struct Pending { int slot; int64_t off; size_t bytes; };
    std::vector<Pending> pend;          // pageable: bands whose staged copy still has to reach out_host
    size_t drained = 0;
    auto drain = [&](size_t upto) -> int {
        for (; drained < upto; ++drained) {
            const Pending &q = pend[drained];
            HIPR_CUDA(cudaEventSynchronize(w.staged_out[q.slot]));
            parallel_copy((char *)out_host + q.off, w.stage[q.slot].p, q.bytes, copy_threads);
        }
        return HIPR_OK;
    };
    int b = 0;
    for (int64_t r0 = 0; r0 < nrows; r0 += rows, ++b) {
        const int nr = (int)((nrows - r0 < rows) ? nrows - r0 : rows);
        const int slot = b % NBUF;
        const size_t bytes = (size_t)nr * row_bytes;
        void *band = w.band[slot].p;
        if (b >= NBUF) HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.freed[slot], 0));   // its previous band has left the device
        if ((e = produce(r0, nr, band, w.comp))) return e;
        HIPR_CUDA(cudaEventRecord(w.copied[slot], w.comp));
        HIPR_CUDA(cudaStreamWaitEvent(w.copy, w.copied[slot], 0));
        if (pageable) {
            // stage[slot] is free once the host has copied band b - NBUF out of it
            if (b >= NBUF && (e = drain((size_t)(b - NBUF + 1)))) return e;
            HIPR_CUDA(cudaMemcpyAsync(w.stage[slot].p, band, bytes, cudaMemcpyDeviceToHost, w.copy));
            HIPR_CUDA(cudaEventRecord(w.staged_out[slot], w.copy));
            pend.push_back(Pending{slot, r0 * row_bytes, bytes});
        } else {
            HIPR_CUDA(cudaMemcpyAsync((char *)out_host + r0 * row_bytes, band, bytes, cudaMemcpyDeviceToHost, w.copy));
        }
        HIPR_CUDA(cudaEventRecord(w.freed[slot], w.copy));
    }
    if (pageable && (e = drain(pend.size()))) return e;
    return HIPR_OK;
}

// The host gathers: the padded float64 input (`in_count` values) is uploaded once, then banded_to_host runs
// `produce(in_dev, r0, nr, band_dev, stream)` over `nrows` output rows of `row_bytes`.
template <typename Produce>
static int gather_to_host(const double *in_host, size_t in_count, int64_t nrows, int64_t row_bytes, double *out_host,
                          Produce produce) {
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    if ((e = w.input.reserve(in_count * sizeof(double)))) return e;
    const double *in_dev = (const double *)w.input.p;
    HIPR_CUDA(cudaEventRecord(w.t0, w.comp));
    HIPR_CUDA(cudaMemcpyAsync(w.input.p, in_host, in_count * sizeof(double), cudaMemcpyHostToDevice, w.comp));
    e = banded_to_host(w, nrows, row_bytes, out_host, [&](int64_t r0, int nr, void *band, cudaStream_t st) {
        return produce(in_dev, r0, nr, band, st);
    });
    return e ? e : call.finish(w.copy);
}

// The strict drop-in of line_profile_2d_v2 (eco/neighbor2d.pyx:8-64) from and to HOST arrays: padded float64 image in,
// the literal (H, W, n_dirs, P) float64 gather out -- 792 B per pixel at (11, 9), 3.3 GB for a 2048^2 image, so the
// call is the PCIe time of the OUTPUT.  The image is uploaded once; the gather runs in row bands of ~32 MiB of output.
extern "C" int hipr_line_profile_2d_host(const double *image_padded_host, int Hp, int Wp, int patch_size, int n_dirs,
                                         const int32_t *table_host, double *out_host) {
    if (!image_padded_host || !out_host) return HIPR_E_ARG;
    int e = check_table(table_host, n_dirs, patch_size, 2);
    if (e) return e;
    const int P = patch_size, H = Hp - (P - 1), W = Wp - (P - 1), K = n_dirs * P;
    if (H < 1 || W < 1) return HIPR_E_PATCH;
    int lin[HIPR_MAX_TABLE];
    for (int i = 0; i < K; ++i) {
        const int dy = table_host[2 * i], dx = table_host[2 * i + 1];
        if (dy < 0 || dy >= P || dx < 0 || dx >= P) return HIPR_E_TABLE;
        lin[i] = dy * Wp + dx;
    }
    return gather_to_host(image_padded_host, (size_t)Hp * Wp, H, (int64_t)W * K * sizeof(double), out_host,
                          [&](const double *img_dev, int64_t r0, int nr, void *band, cudaStream_t st) {
                              return gather_launch<double>(img_dev + r0 * Wp, Wp, 0, 1, nr, W, K, lin, (double *)band, st);
                          });
}

// line_profile_v2 (bio/neighbor.pyx:115-181) from and to host arrays: (X, Y, Z, n_dirs, P) float64, 6,336 B per voxel at
// (11, 9, 9) -- the reference's callers chunk the volume to 100^2 / 200^2 columns for that reason
// (bio/..._analysis.py:900-904, 1105-1112); a 100 x 100 x 64 chunk is a 4 GB result.  Bands of whole x-planes.
extern "C" int hipr_line_profile_3d_host(const double *volume_padded_host, int Xp, int Yp, int Zp, int patch_size, int n_dirs,
                                         const int32_t *table_host, double *out_host) {
    if (!volume_padded_host || !out_host || patch_size < 1) return HIPR_E_ARG;
    const int P = patch_size, X = Xp - (P - 1), Y = Yp - (P - 1), Z = Zp - (P - 1);
    if (X < 1 || Y < 1 || Z < 1) return HIPR_E_PATCH;
    return gather_to_host(volume_padded_host, (size_t)Xp * Yp * Zp, X, (int64_t)Y * Z * n_dirs * P * sizeof(double),
                          out_host, [&](const double *vol_dev, int64_t x0, int nx, void *band, cudaStream_t st) {
                              return hipr_line_profile_3d(vol_dev + x0 * (int64_t)Yp * Zp, nx + P - 1, Yp, Zp, HIPR_F64, P,
                                                          n_dirs, table_host, band, st);
                          });
}

// The same for line_profile_memory_efficient_v2 (bio/neighbor.pyx:186-263), the 3-D stencil the z-stack pipelines
// call (bio/..._analysis.py:456, :812): padded float64 volume (Xp, Yp, Zp) in, the (X, Y, Z, n_dirs) float64
// per-direction values out (576 B per voxel at 72 directions), in bands of whole x-planes.
extern "C" int hipr_lne3d_dirs_host(const double *volume_padded_host, int Xp, int Yp, int Zp, int patch_size, int n_dirs,
                                    const int32_t *table_host, double *out_host) {
    if (!volume_padded_host || !out_host || patch_size < 1) return HIPR_E_ARG;
    const int P = patch_size, X = Xp - (P - 1), Y = Yp - (P - 1), Z = Zp - (P - 1);
    if (X < 1 || Y < 1 || Z < 1) return HIPR_E_PATCH;
    return gather_to_host(volume_padded_host, (size_t)Xp * Yp * Zp, X, (int64_t)Y * Z * n_dirs * sizeof(double), out_host,
                          [&](const double *vol_dev, int64_t x0, int nx, void *band, cudaStream_t st) {
                              // output planes [x0, x0 + nx) read padded planes [x0, x0 + nx + P - 1)
                              return hipr_lne3d_dirs(vol_dev + x0 * (int64_t)Yp * Zp, nx + P - 1, Yp, Zp, 1, HIPR_F64, P,
                                                     n_dirs, table_host, nullptr, band, st);
                          });
}

// 3-D: cube_host (X, Y, Z, C) float32 -> score_host (X, Y, Z) float32: channel sum -> /max -> edge pad -> 72 x 11 line
// profiles -> epilogue, bio/..._analysis.py:807-817 (ME2), :900-917 (F2), :1102-1125 (F3), the cube streamed in bands
// of whole x-planes under the channel sum.
static int neighbor3d_host_impl(const float *cube_host, int X, int Y, int Z, int C, int patch_size, int n_dirs,
                                const int32_t *table_host, int flavour, float *score_host, double denoise_h,
                                int denoise_distance) {
    if (!cube_host || !score_host || !table_host || X < 1 || Y < 1 || Z < 1 || C < 1) return HIPR_E_ARG;
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    Workspace::Image &m = w.img[0];
    const int64_t plane_px = (int64_t)Y * Z, plane_bytes = plane_px * C * 4, nvox = (int64_t)X * plane_px;
    const int planes = band_rows(plane_bytes, X);
    if ((e = ws_ring(w, (size_t)planes * plane_bytes, is_pageable(cube_host))) || (e = m.sum.reserve((size_t)nvox * 8)) ||
        (e = m.score.reserve((size_t)nvox * 4)) || (e = m.keys.reserve(64)))
        return e;
    double *sum_dev = (double *)m.sum.p;
    float *score_dev = (float *)m.score.p;
    unsigned long long *key = (unsigned long long *)m.keys.p;
    HIPR_CUDA(cudaEventRecord(w.t0, w.copy));
    HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.t0, 0));
    if ((e = reset_keys(key, w.comp))) return e;
    int b = 0;
    e = upload_bands(w, cube_host, X, plane_bytes, planes, b, [&](int64_t x0, int64_t nx, const void *band, cudaStream_t st) {
        return chansum_band(band, 4, 1.f, nx * plane_px, C, sum_dev + x0 * plane_px, key, st);
    });
    if (e) return e;
    if (denoise_h > 0.0) {
        // bio/..._analysis.py:452-462 in full: /max -> 3-D NL-means -> float64 stencil (the denoised volume is too smooth
        // for the fixed-point grid, as in 2-D) -> float32 score.  scratch: denoised volume; the float64 score goes back
        // into the sums; extra: the reflect-padded copy the denoise works on
        const int64_t wbytes = hipr_denoise_nl_means_3d_workspace(X, Y, Z, denoise_distance);
        if (wbytes < 0) return HIPR_E_UNSUPPORTED;
        if ((e = m.scratch.reserve((size_t)nvox * 8)) || (e = w.extra.reserve((size_t)wbytes))) return e;
        double *den = (double *)m.scratch.p;
        if ((e = hipr_normalize(sum_dev, HIPR_F64, nvox, (const uint64_t *)key, w.comp))) return e;
        if ((e = hipr_denoise_nl_means_3d(sum_dev, X, Y, Z, HIPR_F64, 7, denoise_distance, denoise_h, den, w.extra.p, wbytes, w.comp)))
            return e;
        if ((e = hipr_lne3d(den, X, Y, Z, 0, HIPR_F64, patch_size, n_dirs, table_host, flavour, nullptr, sum_dev, w.comp))) return e;
        if ((e = hipr_normalize_cast(sum_dev, nvox, nullptr, score_dev, w.comp))) return e;
    } else {
        // fixed-point stencil for the reference's (11, 9, 9) table; the float64 stencil for any other table
        e = hipr_lne3d_q(sum_dev, X, Y, Z, 0, HIPR_F64, patch_size, n_dirs, table_host, flavour, 0, (const uint64_t *)key,
                         score_dev, w.comp);
        if (e == HIPR_E_UNSUPPORTED) {
            if ((e = m.scratch.reserve((size_t)nvox * 8))) return e;
            double *score64 = (double *)m.scratch.p;
            if ((e = hipr_lne3d(sum_dev, X, Y, Z, 0, HIPR_F64, patch_size, n_dirs, table_host, flavour, (const uint64_t *)key,
                                score64, w.comp)))
                return e;
            e = hipr_normalize_cast(score64, nvox, nullptr, score_dev, w.comp);
        }
        if (e) return e;
    }
    HIPR_CUDA(cudaMemcpyAsync(score_host, score_dev, (size_t)nvox * 4, cudaMemcpyDeviceToHost, w.comp));
    return call.finish(w.comp);
}

extern "C" int hipr_neighbor3d_host(const float *cube_host, int X, int Y, int Z, int C, int patch_size, int n_dirs,
                                    const int32_t *table_host, int flavour, float *score_host) {
    return neighbor3d_host_impl(cube_host, X, Y, Z, C, patch_size, n_dirs, table_host, flavour, score_host, 0.0, 11);
}

extern "C" int hipr_neighbor3d_host_denoise(const float *cube_host, int X, int Y, int Z, int C, int patch_size, int n_dirs,
                                            const int32_t *table_host, int flavour, double denoise_h, int denoise_distance,
                                            float *score_host) {
    if (!(denoise_h > 0.0)) return HIPR_E_ARG;
    return neighbor3d_host_impl(cube_host, X, Y, Z, C, patch_size, n_dirs, table_host, flavour, score_host, denoise_h,
                                denoise_distance);
}

extern "C" int hipr_neighbor2d_host_denoise(const float *cube_host, int H, int W, int C, int patch_size, int n_dirs,
                                            const int32_t *table_host, int flavour, double denoise_h, float *score_host,
                                            float *sum_host) {
    if (!(denoise_h > 0.0)) return HIPR_E_ARG;
    return neighbor2d_host_impl(cube_host, 4, 1.f, H, W, C, patch_size, n_dirs, table_host, flavour, score_host, sum_host,
                                denoise_h);
}

// A batch of fields of view from host memory (config 3: hundreds of FOVs per run; the scripts process them one after
// another, syn/..._measurement.py:161-173 inside the Snakefile's per-sample loop).  FOV i + 1 is uploaded band by band
// and summed on the copy / compute streams while FOV i's normalisation, NL-means denoise (denoise_h > 0: lines 106-124
// in full), stencil and score read-back run on a third stream from a second set of buffers: per FOV the call costs the
// PCIe time of the cube, where one hipr_neighbor2d_host_denoise call per FOV costs that plus ~6 ms of denoise + stencil.
// Results are bit-identical to the single-FOV entry points.
extern "C" int hipr_neighbor2d_host_batch(const float *const *cubes_host, int n_fov, int H, int W, int C, int patch_size,
                                          int n_dirs, const int32_t *table_host, int flavour, double denoise_h,
                                          float *const *scores_host) {
    if (!cubes_host || !scores_host || n_fov < 1 || H < 1 || W < 1 || C < 1 || denoise_h < 0.0) return HIPR_E_ARG;
    for (int i = 0; i < n_fov; ++i)
        if (!cubes_host[i] || !scores_host[i]) return HIPR_E_ARG;
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    const int64_t row_bytes = (int64_t)W * C * 4;
    const int rows = band_rows(row_bytes, H);
    const size_t img_bytes = (size_t)H * W * 4;
    bool any_pageable = false;
    for (int i = 0; i < n_fov; ++i) any_pageable = any_pageable || is_pageable(cubes_host[i]);
    if ((e = ws_ring(w, (size_t)rows * row_bytes, any_pageable))) return e;
    for (Workspace::Image &m : w.img)
        if ((e = m.sum.reserve(2 * img_bytes)) || (e = m.score.reserve(img_bytes)) || (e = m.keys.reserve(64))) return e;
    HIPR_CUDA(cudaEventRecord(w.t0, w.copy));
    HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.t0, 0));
    HIPR_CUDA(cudaStreamWaitEvent(w.post, w.t0, 0));
    int b = 0;                                                 // bands since the start of the call (ring slots carry over)
    for (int i = 0; i < n_fov; ++i) {
        const int k = i & 1;
        Workspace::Image &m = w.img[k];
        double *sum_dev = (double *)m.sum.p;
        float *score_dev = (float *)m.score.p;
        unsigned long long *key = (unsigned long long *)m.keys.p;
        if (i >= 2) HIPR_CUDA(cudaStreamWaitEvent(w.comp, w.post_done[k], 0));   // FOV i - 2 has left this set
        if ((e = reset_keys(key, w.comp))) return e;
        e = upload_bands(w, cubes_host[i], H, row_bytes, rows, b,
                         [&](int64_t r0, int64_t nr, const void *band, cudaStream_t st) {
                             return chansum_band(band, 4, 1.f, nr * W, C, sum_dev + r0 * W, key, st);
                         });
        if (e) return e;
        HIPR_CUDA(cudaEventRecord(w.summed[k], w.comp));
        HIPR_CUDA(cudaStreamWaitEvent(w.post, w.summed[k], 0));
        if ((e = score2d(sum_dev, key, H, W, patch_size, n_dirs, table_host, flavour, denoise_h, m.scratch, score_dev,
                         w.post)))
            return e;
        HIPR_CUDA(cudaMemcpyAsync(scores_host[i], score_dev, img_bytes, cudaMemcpyDeviceToHost, w.post));
        HIPR_CUDA(cudaEventRecord(w.post_done[k], w.post));
    }
    return call.finish(w.post);
}

extern "C" int hipr_neighbor2d_host_raw(const void *cube_host, int sample_bytes, double scale, int H, int W, int C,
                                        int patch_size, int n_dirs, const int32_t *table_host, int flavour,
                                        float *score_host, float *sum_host) {
    if (sample_bytes != 1 && sample_bytes != 2) return HIPR_E_DTYPE;
    if (!(scale > 0.0)) return HIPR_E_ARG;
    if (sample_bytes == 2 && (((uintptr_t)cube_host) & 1u)) return HIPR_E_ALIGN;
    return neighbor2d_host_impl(cube_host, sample_bytes, (float)scale, H, W, C, patch_size, n_dirs, table_host, flavour,
                                score_host, sum_host);
}

extern "C" double hipr_host_last_elapsed_ms(void) { return (double)t_last_ms; }

extern "C" int hipr_cell_spectra_host(const float *cube_host, const void *labels_host, int label_bytes, int64_t npix,
                                      int64_t row_len, int C, int64_t capacity, int64_t *n_cells, int64_t *labels_out,
                                      int64_t *area_out, double *avgint_out, double *avgint_norm_out) {
    if (!cube_host || !labels_host || !n_cells || !labels_out || !area_out || !avgint_out || !avgint_norm_out ||
        npix < 1 || C < 1 || capacity < 0)
        return HIPR_E_ARG;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    // labels first (small), max label back to the host to size the accumulators
    if ((e = w.input.reserve((size_t)npix * label_bytes)) || (e = w.img[0].keys.reserve(64))) return e;
    const void *labels_dev = w.input.p;
    int64_t *scalar_dev = (int64_t *)w.img[0].keys.p;
    HIPR_CUDA(cudaMemcpyAsync(w.input.p, labels_host, (size_t)npix * label_bytes, cudaMemcpyHostToDevice, w.comp));
    if ((e = hipr_label_max(labels_dev, label_bytes, npix, scalar_dev, w.comp))) return e;
    int64_t max_label = 0;
    HIPR_CUDA(cudaMemcpyAsync(&max_label, scalar_dev, 8, cudaMemcpyDeviceToHost, w.comp));
    HIPR_CUDA(cudaStreamSynchronize(w.comp));
    *n_cells = 0;
    if (max_label <= 0) return call.done();
    w.last_cells = -1;                                   // the table buffer is rewritten from here on
    CellTable t;
    if ((e = cell_table(w.cells, max_label, C, t))) return e;
    HIPR_CUDA(cudaMemsetAsync(t.sums, 0, t.acc_bytes, w.comp));
    const int64_t px_bytes = (int64_t)C * 4;
    int64_t band_px = (32ll << 20) / px_bytes;
    const int64_t W = (row_len > 0 && npix % row_len == 0) ? row_len : npix;
    if (W < npix) {
        band_px = (band_px / W) / 32 * 32 * W;   // whole 32-row tiles per band
        if (band_px < W) band_px = W;
    } else {
        band_px &= ~31ll;
        if (band_px < 32) band_px = 32;
    }
    if ((e = ws_ring(w, (size_t)(band_px * px_bytes), is_pageable(cube_host)))) return e;
    int b = 0;
    e = upload_bands(w, cube_host, npix, px_bytes, band_px, b, [&](int64_t p0, int64_t np, const void *band, cudaStream_t st) {
        return hipr_cell_spectra_accumulate((const float *)band, (const char *)labels_dev + p0 * label_bytes, label_bytes,
                                            np, (W < npix) ? W : 0, C, max_label, t.sums, t.counts, nullptr, st);
    });
    if (e) return e;
    e = finalize_cells(t, max_label, C, capacity, n_cells, labels_out, area_out, avgint_out, avgint_norm_out, w.comp);
    if (e && e != HIPR_E_RANGE) return e;
    w.last_cells = *n_cells;              // HIPR_E_RANGE: the table stays on the device (hipr_cell_spectra_host_fetch)
    w.last_max_label = max_label;
    w.last_C = C;
    const int d = call.done();
    return d ? d : e;
}

extern "C" int hipr_cell_spectra_host_fetch(int64_t capacity, int64_t *labels_out, int64_t *area_out, double *avgint_out,
                                            double *avgint_norm_out) {
    if (!labels_out || !area_out || !avgint_out || !avgint_norm_out) return HIPR_E_ARG;
    CallScope call;
    int e = call.open();
    if (e) return e;
    Workspace &w = *call.w;
    if (w.last_cells < 0 || !w.cells.p) return HIPR_E_ARG;      // no table to fetch
    const int64_t n = w.last_cells;
    if (n > capacity) return HIPR_E_RANGE;
    if (n == 0) return HIPR_OK;
    CellTable t;
    if ((e = cell_table(w.cells, w.last_max_label, w.last_C, t))) return e;   // the buffer already holds it
    if ((e = copy_cell_table(t, n, w.last_C, labels_out, area_out, avgint_out, avgint_norm_out, w.comp))) return e;
    return call.done();
}


// ---------------------------------------------------------------------------------------------------------------
// Field-of-view handle: ONE upload of the cube for the score map and the per-cell spectra.
// The scripts hold `image_registered` across both steps (syn/..._measurement.py:161-173: generate_2d_segmentation
// returns it, the regionprops loop reads it again after the watershed); with the two host entry points above the
// cube crosses PCIe twice (29 + 32 ms per 2048^2 FOV).  hipr_fov_upload streams it to the device once, in row bands
// under the channel sum, and keeps cube, sums and range resident; hipr_fov_score and hipr_fov_cell_spectra then cost
// a stencil / a label upload + one pass over the resident cube.
// ---------------------------------------------------------------------------------------------------------------
namespace hipr {
struct Fov {
    int device = 0, H = 0, W = 0, C = 0;
    float *cube = nullptr;
    double *sum = nullptr;
    float *score = nullptr;            // (H, W) float32 scratch: score, then the normalised sum
    unsigned long long *keys = nullptr;
    DevBuf scratch;                    // float64 score, general stencil parameters only
    DevBuf labels;
    DevBuf cells;                      // the cell table
    cudaStream_t copy = nullptr, comp = nullptr;
    cudaEvent_t copied = nullptr, t0 = nullptr, t1 = nullptr;
    float last_ms = -1.f;
    std::mutex mu;
};
struct DeviceScope {                   // run on the handle's device, restore the caller's afterwards
    int prev = -1;
    bool ok = true;
    explicit DeviceScope(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceScope() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
static void fov_free(Fov *f) {
    if (!f) return;
    if (f->comp) cudaStreamSynchronize(f->comp);
    if (f->copy) cudaStreamSynchronize(f->copy);
    cudaFree(f->cube);
    cudaFree(f->sum);
    cudaFree(f->score);
    cudaFree(f->keys);
    for (DevBuf *b : {&f->scratch, &f->labels, &f->cells}) b->release();
    if (f->copied) cudaEventDestroy(f->copied);
    if (f->t0) cudaEventDestroy(f->t0);
    if (f->t1) cudaEventDestroy(f->t1);
    if (f->copy) cudaStreamDestroy(f->copy);
    if (f->comp) cudaStreamDestroy(f->comp);
    delete f;
}
// the end of a timed handle call: t1 after the last read-back, the device time from t0
static int fov_finish(Fov *f, Drain &drain) {
    HIPR_CUDA(cudaEventRecord(f->t1, f->comp));
    HIPR_CUDA(cudaStreamSynchronize(f->comp));
    drain.armed = false;
    HIPR_CUDA(cudaEventElapsedTime(&f->last_ms, f->t0, f->t1));
    t_last_ms = f->last_ms;
    return HIPR_OK;
}
}  // namespace hipr

// A released handle's buffers are kept (one per device) for the next upload of the same shape: allocating and freeing
// 1.6 GB of device memory costs more than the upload itself (measured 128 ms per FOV without this, 31 ms with).
static Fov *g_fov_cache[kMaxDevices] = {};
static std::mutex g_fov_cache_mu;

static void fov_cache_release_current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return;
    Fov *c = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_fov_cache_mu);
        c = g_fov_cache[dev];
        g_fov_cache[dev] = nullptr;
    }
    fov_free(c);
}

extern "C" int hipr_fov_upload(const float *cube_host, int H, int W, int C, void **handle_out) {
    if (!cube_host || !handle_out || H < 1 || W < 1 || C < 1) return HIPR_E_ARG;
    *handle_out = nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return HIPR_E_NODEVICE;
    Fov *f = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_fov_cache_mu);
        Fov *c = g_fov_cache[dev];
        if (c) {
            g_fov_cache[dev] = nullptr;
            if (c->H == H && c->W == W && c->C == C) f = c;
            else fov_free(c);
        }
    }
    const bool reused = (f != nullptr);
    if (!f) f = new Fov;
    f->device = dev;
    f->H = H; f->W = W; f->C = C;
    const size_t npix = (size_t)H * W;
    int e = HIPR_OK;
    auto fail = [&](int code) {
        fov_free(f);
        return code;
    };
#define HIPR_FOV(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return fail((int)_e); } while (0)
    if (!reused) {
        HIPR_FOV(cudaMalloc((void **)&f->cube, npix * C * sizeof(float)));
        HIPR_FOV(cudaMalloc((void **)&f->sum, npix * sizeof(double)));
        HIPR_FOV(cudaMalloc((void **)&f->score, npix * sizeof(float)));
        HIPR_FOV(cudaMalloc((void **)&f->keys, 64));
        HIPR_FOV(cudaStreamCreateWithFlags(&f->copy, cudaStreamNonBlocking));
        HIPR_FOV(cudaStreamCreateWithFlags(&f->comp, cudaStreamNonBlocking));
        HIPR_FOV(cudaEventCreateWithFlags(&f->copied, cudaEventDisableTiming));
        HIPR_FOV(cudaEventCreate(&f->t0));
        HIPR_FOV(cudaEventCreate(&f->t1));
    }
    HIPR_FOV(cudaEventRecord(f->t0, f->copy));
    HIPR_FOV(cudaStreamWaitEvent(f->comp, f->t0, 0));
    if ((e = reset_keys(f->keys, f->comp))) return fail(e);
    // bands of ~32 MiB straight into the resident cube; the channel sum of band b runs under the copy of band b + 1.
    // Page-locked memory (hipr_host_alloc) goes at the PCIe rate; pageable memory is staged by the driver.
    const int64_t row_bytes = (int64_t)W * C * 4;
    const int rows = band_rows(row_bytes, H);
    for (int r0 = 0; r0 < H; r0 += rows) {
        const int nr = (H - r0 < rows) ? H - r0 : rows;
        float *dst = f->cube + (size_t)r0 * W * C;
        HIPR_FOV(cudaMemcpyAsync(dst, (const char *)cube_host + (int64_t)r0 * row_bytes, (size_t)nr * row_bytes,
                                 cudaMemcpyHostToDevice, f->copy));
        HIPR_FOV(cudaEventRecord(f->copied, f->copy));
        HIPR_FOV(cudaStreamWaitEvent(f->comp, f->copied, 0));
        if ((e = chansum_band(dst, 4, 1.f, (int64_t)nr * W, C, f->sum + (size_t)r0 * W, f->keys, f->comp))) return fail(e);
    }
    HIPR_FOV(cudaEventRecord(f->t1, f->comp));
    HIPR_FOV(cudaStreamSynchronize(f->comp));      // the caller may reuse cube_host
    HIPR_FOV(cudaEventElapsedTime(&f->last_ms, f->t0, f->t1));
#undef HIPR_FOV
    t_last_ms = f->last_ms;
    *handle_out = f;
    return HIPR_OK;
}

extern "C" int hipr_fov_release(void *handle) {
    Fov *f = reinterpret_cast<Fov *>(handle);
    if (!f) return HIPR_OK;
    DeviceScope scope(f->device);
    cudaStreamSynchronize(f->comp);
    cudaStreamSynchronize(f->copy);
    Fov *old = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_fov_cache_mu);
        old = g_fov_cache[f->device];
        g_fov_cache[f->device] = f;          // keep the newest; hipr_host_release_workspace frees it
    }
    fov_free(old);
    return HIPR_OK;
}

// device pointers of a handle's resident arrays (for callers that continue on the device): cube (H, W, C) float32,
// channel sums (H, W) float64, range keys (2 uint64)
extern "C" int hipr_fov_device_arrays(void *handle, const float **cube_dev, const double **sum_dev, const uint64_t **range_dev) {
    Fov *f = reinterpret_cast<Fov *>(handle);
    if (!f) return HIPR_E_ARG;
    if (cube_dev) *cube_dev = f->cube;
    if (sum_dev) *sum_dev = f->sum;
    if (range_dev) *range_dev = reinterpret_cast<const uint64_t *>(f->keys);
    return HIPR_OK;
}

extern "C" int hipr_fov_score(void *handle, int patch_size, int n_dirs, const int32_t *table_host, int flavour,
                              float *score_host, float *sum_host) {
    Fov *f = reinterpret_cast<Fov *>(handle);
    if (!f || !score_host || !table_host) return HIPR_E_ARG;
    std::lock_guard<std::mutex> lock(f->mu);
    DeviceScope scope(f->device);
    if (!scope.ok) return HIPR_E_NODEVICE;
    const int H = f->H, W = f->W;
    const size_t img_bytes = (size_t)H * W * 4;
    Drain drain{{f->comp}};
    HIPR_CUDA(cudaEventRecord(f->t0, f->comp));
    int e = score2d(f->sum, f->keys, H, W, patch_size, n_dirs, table_host, flavour, 0.0, f->scratch, f->score, f->comp);
    if (e) return e;
    HIPR_CUDA(cudaMemcpyAsync(score_host, f->score, img_bytes, cudaMemcpyDeviceToHost, f->comp));
    if (sum_host) {
        if ((e = hipr_normalize_cast(f->sum, (int64_t)H * W, reinterpret_cast<const uint64_t *>(f->keys), f->score, f->comp)))
            return e;
        HIPR_CUDA(cudaMemcpyAsync(sum_host, f->score, img_bytes, cudaMemcpyDeviceToHost, f->comp));
    }
    return fov_finish(f, drain);
}

extern "C" int hipr_fov_cell_spectra(void *handle, const void *labels_host, int label_bytes, int64_t capacity,
                                     int64_t *n_cells, int64_t *labels_out, int64_t *area_out, double *avgint_out,
                                     double *avgint_norm_out) {
    Fov *f = reinterpret_cast<Fov *>(handle);
    if (!f || !labels_host || !n_cells || !labels_out || !area_out || !avgint_out || !avgint_norm_out || capacity < 0)
        return HIPR_E_ARG;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    std::lock_guard<std::mutex> lock(f->mu);
    DeviceScope scope(f->device);
    if (!scope.ok) return HIPR_E_NODEVICE;
    const int64_t npix = (int64_t)f->H * f->W;
    const int C = f->C;
    Drain drain{{f->comp}};
    int e = f->labels.reserve((size_t)npix * label_bytes);
    if (e) return e;
    HIPR_CUDA(cudaEventRecord(f->t0, f->comp));
    HIPR_CUDA(cudaMemcpyAsync(f->labels.p, labels_host, (size_t)npix * label_bytes, cudaMemcpyHostToDevice, f->comp));
    int64_t *scalar_dev = reinterpret_cast<int64_t *>(f->keys + 4);      // the handle's 64-byte scratch, past the keys
    if ((e = hipr_label_max(f->labels.p, label_bytes, npix, scalar_dev, f->comp))) return e;
    int64_t max_label = 0;
    HIPR_CUDA(cudaMemcpyAsync(&max_label, scalar_dev, 8, cudaMemcpyDeviceToHost, f->comp));
    HIPR_CUDA(cudaStreamSynchronize(f->comp));
    *n_cells = 0;
    if (max_label <= 0) {
        drain.armed = false;
        return HIPR_OK;
    }
    CellTable t;
    if ((e = cell_table(f->cells, max_label, C, t))) return e;
    HIPR_CUDA(cudaMemsetAsync(t.sums, 0, t.acc_bytes, f->comp));
    if ((e = hipr_cell_spectra_accumulate(f->cube, f->labels.p, label_bytes, npix, f->W, C, max_label, t.sums, t.counts,
                                          nullptr, f->comp)))
        return e;
    e = finalize_cells(t, max_label, C, capacity, n_cells, labels_out, area_out, avgint_out, avgint_norm_out, f->comp);
    if (e == HIPR_E_RANGE || (!e && *n_cells == 0)) {
        drain.armed = false;
        return e;                              // HIPR_E_RANGE: call again with capacity >= *n_cells (the cube is resident)
    }
    return e ? e : fov_finish(f, drain);
}

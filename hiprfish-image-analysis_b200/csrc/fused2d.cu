// K13: the whole 2-D front end in ONE launch: cube (H, W, C) -> score map (H, W).
//
//   channel sum (syn/..._measurement.py:105) -> [/max: a no-op for F1/F2, which are invariant to
//   any affine map of the image] -> edge pad (:109) -> line_profile_2d_v2 (eco/neighbor2d.pyx:56-63)
//   -> epilogue F1 (:111-124) or F2 (bio/..._analysis.py:671-683).
//
// HBM-bound on the cube read (380 B/px at C = 95); the point of fusing is that the stencil's
// shared-memory/ALU work (~1/4 of the channel-sum time as a separate kernel) runs under the
// cube stream instead of after it, and the sum image never goes to memory.
//
// Decomposition: the image is cut into column strips of 128 output columns and row bands, one
// CTA per (strip, band), all resident at once (<= one per SM).  A CTA walks its band top to
// bottom with three warp roles:
//   producer (1 warp)   one lane keeps NS 1-D bulk copies (cp.async.bulk, the TMA engine) in
//                       flight: one image row of the strip's 144-pixel window = 144*C*4 bytes
//                       (16-byte aligned because windows start on multiples of 4 pixels).
//   summers  (5 warps)  thread t sums pixel t of the landed row out of shared memory (stride-C
//                       words: conflict-free for odd C) in float64 and stores it in a ring of 26
//                       sum rows; releases the stage; signals a row block when its last row is in.
//   stencil  (8 warps)  per block of 8 output rows: takes the 18 x 138 window of the ring, maps it
//                       affinely onto 31-bit integers using the WINDOW's own min/max (exact
//                       differences, see lne2d_q.cu; a local range only makes the grid finer),
//                       then runs the baked (11, 9) line table with LDS immediates and FMNMX3,
//                       4 pixels per thread, and writes the float32 scores.
// Neighbouring strips re-read 16 of 144 window columns; they run in lock step, so the second
// read is an L2 hit.  Bands re-read 10 halo rows each (4 % at 2048 rows / 9 bands).
#include "hipr_common.cuh"
#include "lne_math.cuh"
#include "lne_fixed.cuh"

namespace hipr {

constexpr int FU_WT = 128;                  // output columns per strip
constexpr int FU_WIN = 144;                 // loaded window: columns [x0 - 8, x0 + 136)
constexpr int FU_LEFT = 8;
constexpr int FU_RB = 8;                    // output rows per block
constexpr int FU_RING = 2 * FU_RB + 10;     // sum rows kept on chip
constexpr int FU_SUM_WARPS = 5, FU_ST_WARPS = 8;
constexpr int FU_THREADS = (FU_SUM_WARPS + FU_ST_WARPS + 1) * 32;   // 448
constexpr int FU_QW = FU_WT + 10, FU_QH = FU_RB + 10;               // 138 x 18 fixed-point tile
constexpr int FU_MAX_STAGES = 4;
constexpr int FU_SMEM_FIXED = 256 + FU_RING * FU_WIN * 8 + FU_QH * FU_QW * 4 + 256;
constexpr int FU_SMEM_BUDGET = 227 * 1024;

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

struct FusedGeom {
    int H, W, C;
    int strips, bands, band_rows;   // band_rows is a multiple of FU_RB
    int stages;
};

template <int FLAVOUR, bool WRITE_SUM>
__global__ void __launch_bounds__(FU_THREADS, 1)
fused2d_kernel(const float *__restrict__ cube, const FusedGeom g, float *__restrict__ score,
               double *__restrict__ sum_out, unsigned long long *__restrict__ range) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);           // [stages]
    uint64_t *empty = full + FU_MAX_STAGES;                        // [stages]
    uint64_t *blk_full = empty + FU_MAX_STAGES;                    // [2]
    uint64_t *blk_empty = blk_full + 2;                            // [2]
    double *ring = reinterpret_cast<double *>(smem + 256);         // [RING][WIN]
    float *qtile = reinterpret_cast<float *>(smem + 256 + FU_RING * FU_WIN * 8);
    double *red = reinterpret_cast<double *>(smem + 256 + FU_RING * FU_WIN * 8 + FU_QH * FU_QW * 4);
    unsigned char *stage0 = smem + FU_SMEM_FIXED;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int H = g.H, W = g.W, C = g.C, NS = g.stages;
    const uint32_t row_floats = (uint32_t)FU_WIN * (uint32_t)C;

    const int strip = blockIdx.x % g.strips, band = blockIdx.x / g.strips;
    const int x0 = strip * FU_WT;
    const int xa = x0 - FU_LEFT;                                    // window origin (may be < 0)
    const int lx0 = max(xa, 0), lx1 = min(xa + FU_WIN, W);          // loaded pixel range
    const int rb0 = band * g.band_rows, rb1 = min(rb0 + g.band_rows, H);
    if (rb0 >= rb1) return;
    const int ylo = max(rb0 - 5, 0), yhi = min(rb1 + 4, H - 1);
    const int nrow = yhi - ylo + 1;
    const int nblk = (rb1 - rb0 + FU_RB - 1) / FU_RB;

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], FU_SUM_WARPS);
        }
        for (int j = 0; j < 2; ++j) {
            mbar_init(&blk_full[j], FU_SUM_WARPS);
            mbar_init(&blk_empty[j], FU_ST_WARPS);
        }
        fence_barrier_init();
    }
    __syncthreads();

    if (warp == FU_SUM_WARPS + FU_ST_WARPS) {
        // ------------------------------------------------------------------ producer
        if (lane == 0) {
            const uint32_t bytes = (uint32_t)(lx1 - lx0) * (uint32_t)C * 4u;
            const uint32_t dst_off = (uint32_t)(lx0 - xa) * (uint32_t)C * 4u;
            for (int i = 0; i < nrow; ++i) {
                const int s = i % NS;
                if (i >= NS) mbar_wait(&empty[s], (uint32_t)((i / NS - 1) & 1));
                mbar_expect_tx(&full[s], bytes);
                const float *src = cube + ((int64_t)(ylo + i) * W + lx0) * C;
                asm volatile(
                    "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                        smem_u32(stage0 + (size_t)s * row_floats * 4 + dst_off)),
                    "l"(src), "r"(bytes), "r"(smem_u32(&full[s]))
                    : "memory");
            }
        }
        return;
    }

    if (warp < FU_SUM_WARPS) {
        // ------------------------------------------------------------------ summers
        const int t = tid;                       // window column 0..159 (144 used)
        const int px = xa + t;                   // image column
        const bool valid = (t < FU_WIN) && px >= lx0 && px < lx1;
        const bool owned_col = px >= x0 && px < min(x0 + FU_WT, W);
        double vmax = -__longlong_as_double(0x7ff0000000000000ll), vmin = -vmax;
        int kb = 0;                              // next block to signal
        for (int i = 0; i < nrow; ++i) {
            const int y = ylo + i;
            // the ring slot of row y last held row y - RING: wait until its last reader block is done
            const int yprev = y - FU_RING;
            if (yprev >= ylo) {
                const int kprev = min((yprev + 5 - rb0) / FU_RB, nblk - 1);
                const int first_row_of_kprev = max(kprev * FU_RB + rb0 - 5, ylo) ;
                (void)first_row_of_kprev;
                mbar_wait(&blk_empty[kprev & 1], (uint32_t)((kprev >> 1) & 1));
            }
            const int s = i % NS;
            mbar_wait(&full[s], (uint32_t)((i / NS) & 1));
            if (valid) {
                const float *p = reinterpret_cast<const float *>(stage0 + (size_t)s * row_floats * 4) + (size_t)t * C;
                const double sum = sum_channels<false>(p, C);
                ring[(y % FU_RING) * FU_WIN + t] = sum;
                if (WRITE_SUM && owned_col && y >= rb0 && y < rb1) {
                    sum_out[(int64_t)y * W + px] = sum;
                    vmax = fmax(vmax, sum);
                    vmin = fmin(vmin, sum);
                }
            }
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[s]);
                while (kb < nblk && y == min(rb0 + (kb + 1) * FU_RB + 4, yhi)) {
                    mbar_arrive(&blk_full[kb & 1]);
                    ++kb;
                }
            }
        }
        if (WRITE_SUM && range != nullptr) {
            vmax = warp_max(vmax);
            vmin = -warp_max(-vmin);
            if (lane == 0) {
                atomicMax(range, (unsigned long long)key_of_double(vmax));
                atomicMin(range + 1, (unsigned long long)key_of_double(vmin));
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- stencil
    const int sw = warp - FU_SUM_WARPS;          // 0..7 = row inside the block
    const int st = tid - FU_SUM_WARPS * 32;      // 0..255
    constexpr int NST = FU_ST_WARPS * 32;
    for (int kb = 0; kb < nblk; ++kb) {
        const int r = rb0 + kb * FU_RB;
        mbar_wait(&blk_full[kb & 1], (uint32_t)((kb >> 1) & 1));
        // 1. window range
        double wmax = -__longlong_as_double(0x7ff0000000000000ll), wmin = -wmax;
        for (int e = st; e < FU_QH * FU_QW; e += NST) {
            const int ty = e / FU_QW, tx = e - ty * FU_QW;
            const int wy = min(max(r - 5 + ty, 0), H - 1), wx = min(max(x0 - 5 + tx, 0), W - 1);
            const double v = ring[(wy % FU_RING) * FU_WIN + (wx - xa)];
            wmax = fmax(wmax, v);
            wmin = fmin(wmin, v);
        }
        wmax = warp_max(wmax);
        wmin = -warp_max(-wmin);
        if (lane == 0) {
            red[sw * 2] = wmax;
            red[sw * 2 + 1] = wmin;
        }
        named_bar_sync(1, NST);
#pragma unroll
        for (int j = 0; j < FU_ST_WARPS; ++j) {
            wmax = fmax(wmax, red[j * 2]);
            wmin = fmin(wmin, red[j * 2 + 1]);
        }
        const double K = q_scale(wmax, wmin);
        // 2. fixed-point tile
        for (int e = st; e < FU_QH * FU_QW; e += NST) {
            const int ty = e / FU_QW, tx = e - ty * FU_QW;
            const int wy = min(max(r - 5 + ty, 0), H - 1), wx = min(max(x0 - 5 + tx, 0), W - 1);
            double v = ring[(wy % FU_RING) * FU_WIN + (wx - xa)];
            if (v != v) v = 0.0;
            qtile[e] = q_encode(v, wmin, K);
        }
        named_bar_sync(1, NST);
        // the ring rows of this block are no longer needed
        if (lane == 0) mbar_arrive(&blk_empty[kb & 1]);
        // 3. line profiles + epilogue, 4 pixels per thread
        const int y = r + sw;
        if (y < rb1) {
#pragma unroll 1
            for (int j = 0; j < FU_WT / 32; ++j) {
                const int lx = lane + 32 * j;
                const int x = x0 + lx;
                if (x >= W) break;
                const float *base = qtile + sw * FU_QW + lx;
                float rr[9];
                static_for<0, 9>([&](auto tc) {
                    constexpr int t = decltype(tc)::value;
                    constexpr int o0 = baked2d_off<FU_QW>(t, 0);
                    float mn = base[o0], mx = mn;
                    static_for<1, 11>([&](auto lc) {
                        constexpr int off = baked2d_off<FU_QW>(t, decltype(lc)::value);
                        const float s = base[off];
                        mn = fminf(mn, s);
                        mx = fmaxf(mx, s);
                    });
                    constexpr int oc = baked2d_off<FU_QW>(t, 5);
                    rr[t] = q_line<FLAVOUR>(base[oc], mn, mx, 0.f);
                });
                float sum = 0.f;
#pragma unroll
                for (int q = 0; q < 9; ++q) sum += rr[q];
                const float mean = sum * (1.0f / 9.0f);
                sort_network<float, 9>(rr);
                float A, B;
                bool unit;
                score[(int64_t)y * W + x] = mean * q_factor<FLAVOUR>(rr[2], rr[6], A, B, unit);
            }
        }
        // all warps must be done with qtile / red before the next block rewrites them
        named_bar_sync(2, NST);
    }
}

}  // namespace hipr

using namespace hipr;

// Returns HIPR_E_UNSUPPORTED when the shape / parameters are outside what this kernel handles;
// callers then run hipr_chansum + hipr_lne2d_q (same results).
extern "C" int hipr_neighbor2d_fused(const float *cube_dev, int H, int W, int C, int patch_size, int n_dirs,
                                     const int32_t *table_host, int flavour, float *score_dev, double *sum_dev,
                                     uint64_t *range_dev, void *stream) {
    if (!cube_dev || !score_dev || !table_host || H < 1 || W < 1 || C < 1) return HIPR_E_ARG;
    if (patch_size != 11 || n_dirs != 9) return HIPR_E_UNSUPPORTED;
    if (flavour != HIPR_FLAVOUR_F1 && flavour != HIPR_FLAVOUR_F2) return HIPR_E_UNSUPPORTED;
    for (int i = 0; i < 198; ++i)
        if (table_host[i] != kBaked2D[i]) return HIPR_E_UNSUPPORTED;
    if ((W & 3) || (((uintptr_t)cube_dev) & 15u)) return HIPR_E_UNSUPPORTED;   // 16-byte row windows
    const int64_t stage_bytes = (int64_t)FU_WIN * C * 4;
    int stages = (int)((FU_SMEM_BUDGET - FU_SMEM_FIXED) / stage_bytes);
    if (stages > FU_MAX_STAGES) stages = FU_MAX_STAGES;
    if (stages < 2) return HIPR_E_UNSUPPORTED;
    if (const char *env = getenv("HIPR_FUSED_STAGES")) {   // tuning knob
        const int v = atoi(env);
        if (v >= 2 && v <= stages) stages = v;
    }
    FusedGeom g;
    g.H = H; g.W = W; g.C = C; g.stages = stages;
    g.strips = (W + FU_WT - 1) / FU_WT;
    const int sms = sm_count();
    int bands = sms / g.strips;
    if (bands < 1) bands = 1;
    const int nblk_total = (H + FU_RB - 1) / FU_RB;
    if (bands > nblk_total) bands = nblk_total;
    g.band_rows = ((nblk_total + bands - 1) / bands) * FU_RB;
    g.bands = (H + g.band_rows - 1) / g.band_rows;
    const size_t smem = (size_t)FU_SMEM_FIXED + (size_t)stages * stage_bytes;
    cudaStream_t st = (cudaStream_t)stream;
    const bool ws = (sum_dev != nullptr);
    if (ws && range_dev) {
        HIPR_CUDA(cudaMemsetAsync(range_dev, 0x00, 8, st));
        HIPR_CUDA(cudaMemsetAsync(range_dev + 1, 0xff, 8, st));
    }
    unsigned long long *rg = reinterpret_cast<unsigned long long *>(range_dev);
    const unsigned grid = (unsigned)(g.strips * g.bands);
#define HIPR_FUSED_LAUNCH(FL, WS)                                                                             \
    do {                                                                                                      \
        auto kern = fused2d_kernel<FL, WS>;                                                                   \
        static std::atomic<uint64_t> attr{0};                                                                 \
        if (first_use_on_device(attr))                                                                        \
            HIPR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FU_SMEM_BUDGET)); \
        kern<<<grid, FU_THREADS, smem, st>>>(cube_dev, g, score_dev, sum_dev, rg);                            \
    } while (0)
    if (flavour == HIPR_FLAVOUR_F1) {
        if (ws) HIPR_FUSED_LAUNCH(HIPR_FLAVOUR_F1, true); else HIPR_FUSED_LAUNCH(HIPR_FLAVOUR_F1, false);
    } else {
        if (ws) HIPR_FUSED_LAUNCH(HIPR_FLAVOUR_F2, true); else HIPR_FUSED_LAUNCH(HIPR_FLAVOUR_F2, false);
    }
#undef HIPR_FUSED_LAUNCH
    return after_launch();
}

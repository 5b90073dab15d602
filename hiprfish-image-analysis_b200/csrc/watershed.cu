// K11: the marker watershed, skimage.segmentation.watershed(image, markers, connectivity, mask) without compactness
// or watershed lines, as the fixpoint of a deterministic rule that equals scikit-image's heap flood wherever no pixel
// is tie-decided (DESIGN.md K11 states the rule and proves it).
//
// Every flooded pixel p gets a key K(p) = (L, d, l), compared lexicographically: L its level (the minimax path value
// from the markers, as an order-preserving key of the value with -0.0 taken as +0.0), d its hop count within the level
// group, l its label (signed).  A marker has K = (v, 0, its label); any other in-mask pixel K(p) = f(min_q K(q), p)
// over its in-mask neighbours q, f((L, d, l), p) = (L, d + 1, l) if v(p) <= L, else (v(p), 1, l).  f is not monotone
// in its argument, so the key is computed as three minimum relaxations, each over words that only ever decrease:
//   phase 1  L(p) = max(v(p), min_q L(q)), markers fixed at v                                     (64-bit keys)
//   phase 2  candidates of p: its neighbours of minimal L.  Markers d = 0, entry pixels (v(p) > min L) d = 1,
//            every other pixel d(p) = 1 + min d over its candidates                               (32-bit words)
//   phase 3  l(p) = min l over the candidates of minimal d (the parents)                           (64-bit words)
// Each phase is a Bellman-Ford style relaxation whose fixpoint is unique.  It runs in 64 x 64 (2-D) or 16^3 (3-D)
// tiles: a CTA loads a tile with a one-pixel halo into shared memory and sweeps it until it stops changing, writes
// back what fell, and marks the neighbouring tiles dirty for the next round; a round ends at a grid barrier, and a
// phase ends after a round in which nothing changed.  One persistent cooperative launch runs all three phases; each
// phase stops after npix + 1 rounds at the latest (never reached: a round moves every wavefront at least one pixel)
// and reports it in the status word.  Every workspace word is written before it is read, except the control block
// and the dirty flags, which the call zeroes.
#include "hipr_common.cuh"

namespace hipr {

constexpr int WS_THREADS = 512;
constexpr int WS_TILE = 4096;                       // pixels per tile, WS_PPT per thread
constexpr int WS_PPT = WS_TILE / WS_THREADS;
constexpr int WS_EDGE2 = 64, WS_EDGE3 = 16;         // tile edge in 2-D / 3-D
constexpr int WS_HALO_MAX = (WS_EDGE3 + 2) * (WS_EDGE3 + 2) * (WS_EDGE3 + 2);   // >= (64 + 2)^2 as well
constexpr int WS_MAXN = 26;
constexpr uint64_t WS_INF = ~0ull;                  // never the key of a non-NaN value
constexpr uint32_t WS_INF32 = ~0u;
constexpr uint32_t WS_FIXED = 0x80000000u;          // info bit: the pixel's word is not relaxed in this phase
constexpr uint64_t WS_SIGN = 0x8000000000000000ull;

struct WsGeom {
    int X, Y, Z;                  // volume (X, Y, Z), Z fastest; an image is (1, H, W)
    int TX, TY, TZ;               // tile
    int NTX, NTY, NTZ;            // tiles per axis
    int hx;                       // halo along X: 1 for volumes, 0 for images
    int nn;                       // neighbours
    signed char off[WS_MAXN][3];  // their offsets (dx, dy, dz)
    int64_t npix;
    int64_t cap;                  // rounds per phase at most
};

struct WsCtrl {                   // zeroed before the launch
    unsigned int barrier;
    unsigned int changed[3][3];   // per phase, round r writes slot r % 3
    unsigned int rounds[3];
    unsigned int status;
    unsigned long long visits[3]; // tile visits per phase
};

constexpr int64_t WS_CTRL_BYTES = 256;
static_assert(sizeof(WsCtrl) <= WS_CTRL_BYTES, "control block");

template <typename V>
__device__ __forceinline__ uint64_t level_key(V v) {
    const double d = (double)v;                     // exact for float32
    return key_of_double(d == 0.0 ? 0.0 : d);       // the heap compares with < and ==: -0.0 is +0.0
}

__device__ __forceinline__ bool in_image(const WsGeom &g, int x, int y, int z) {
    return x >= 0 && y >= 0 && z >= 0 && x < g.X && y < g.Y && z < g.Z;
}

template <typename Wt>
__device__ __forceinline__ uint64_t ws_inf() { return sizeof(Wt) == 4 ? (uint64_t)WS_INF32 : WS_INF; }

// One visit of `tile` in phase PH: load the halo'd tile of W, sweep to the local fixpoint, write back what fell.
// -> 0 nothing fell, 1 something fell, 2 something fell and the sweep cap (tile pixels + 1, never reached) cut it.
template <int PH, typename Wt, typename V, typename MT>
__device__ int ws_tile(const WsGeom &g, int tile, const V *__restrict__ img, const MT *__restrict__ markers,
                       const uint8_t *__restrict__ mask, Wt *W, const uint32_t *info_w, uint64_t *s_w,
                       const int *s_hoff) {
    const int tid = threadIdx.x;
    const int tz = tile % g.NTZ, ty = (tile / g.NTZ) % g.NTY, tx = tile / (g.NTZ * g.NTY);
    const int x0 = tx * g.TX, y0 = ty * g.TY, z0 = tz * g.TZ;
    const int HY = g.TY + 2, HZ = g.TZ + 2, HX = g.TX + 2 * g.hx;
    const int HN = HX * HY * HZ;
    for (int h = tid; h < HN; h += WS_THREADS) {
        const int hz = h % HZ, hy = (h / HZ) % HY, hxx = h / (HZ * HY);
        const int x = x0 + hxx - g.hx, y = y0 + hy - 1, z = z0 + hz - 1;
        s_w[h] = in_image(g, x, y, z) ? (uint64_t)__ldcg(W + ((int64_t)x * g.Y + y) * g.Z + z) : ws_inf<Wt>();
    }
    // per own pixel: halo index and what the sweep needs (phase 1: the value's key; 2, 3: the neighbour mask)
    const int tn = g.TX * g.TY * g.TZ;
    unsigned short hidx[WS_PPT];   // < WS_HALO_MAX
    uint64_t inf[WS_PPT];
    unsigned live = 0;
#pragma unroll
    for (int j = 0; j < WS_PPT; ++j) {
        const int i = tid + j * WS_THREADS;
        const int iz = i % g.TZ, iy = (i / g.TZ) % g.TY, ix = i / (g.TZ * g.TY);
        const int x = x0 + ix, y = y0 + iy, z = z0 + iz;
        hidx[j] = (unsigned short)(((ix + g.hx) * HY + iy + 1) * HZ + iz + 1);
        inf[j] = 0;
        if (i >= tn || !in_image(g, x, y, z)) continue;
        const int64_t p = ((int64_t)x * g.Y + y) * g.Z + z;
        if (PH == 1) {
            if ((mask && !mask[p]) || markers[p] != 0) continue;   // fixed: outside the mask (INF) or a marker
            inf[j] = level_key(img[p]);
        } else {
            const uint32_t m = __ldcg(info_w + p);
            if (m & WS_FIXED) continue;
            inf[j] = m;
        }
        live |= 1u << j;
    }
    __syncthreads();
    unsigned fell = 0;
    bool more = true;
    for (int sweep = 0; sweep <= tn && more; ++sweep) {
        bool any = false;
#pragma unroll
        for (int j = 0; j < WS_PPT; ++j) {
            if (!(live >> j & 1u)) continue;
            const int h = hidx[j];
            uint64_t m = WS_INF, nv;
            if (PH == 1) {
                for (int k = 0; k < g.nn; ++k) m = min(m, s_w[h + s_hoff[k]]);
                nv = max(m, inf[j]);
            } else {
                for (uint32_t b = (uint32_t)inf[j]; b; b &= b - 1) m = min(m, s_w[h + s_hoff[__ffs(b) - 1]]);
                nv = PH == 2 ? (m >= WS_INF32 ? (uint64_t)WS_INF32 : m + 1) : m;
            }
            if (nv < s_w[h]) {
                s_w[h] = nv;
                fell |= 1u << j;
                any = true;
            }
        }
        more = __syncthreads_or(any);
    }
#pragma unroll
    for (int j = 0; j < WS_PPT; ++j) {
        if (!(fell >> j & 1u)) continue;
        const int i = tid + j * WS_THREADS;
        const int iz = i % g.TZ, iy = (i / g.TZ) % g.TY, ix = i / (g.TZ * g.TY);
        W[((int64_t)(x0 + ix) * g.Y + y0 + iy) * g.Z + z0 + iz] = (Wt)s_w[hidx[j]];
    }
    const int changed = __syncthreads_or(fell != 0);
    return changed ? (more ? 2 : 1) : 0;
}

// Rounds of phase PH until one changes nothing.  dirty: 2 x ntiles flags of this phase (round r reads r & 1).
template <int PH, typename Wt, typename V, typename MT>
__device__ void ws_phase(const WsGeom &g, const V *img, const MT *markers, const uint8_t *mask, Wt *W,
                         const uint32_t *info_w, unsigned int *dirty, WsCtrl *ctrl, unsigned int &bar_target,
                         uint64_t *s_w, const int *s_hoff, unsigned int *s_flag) {
    const int tid = threadIdx.x;
    const int ntiles = g.NTX * g.NTY * g.NTZ;
    const int ph = PH - 1;
    for (int64_t r = 0; r < g.cap; ++r) {
        unsigned int *cur = dirty + (r & 1) * ntiles, *next = dirty + ((r + 1) & 1) * ntiles;
        const int slot = (int)(r % 3);
        unsigned long long visits = 0;
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
            if (r > 0 && !__ldcg(cur + t)) continue;   // uniform: only this CTA writes cur[t] in this round
            ++visits;
            const int res = ws_tile<PH, Wt>(g, t, img, markers, mask, W, info_w, s_w, s_hoff);
            if (tid == 0) cur[t] = 0;
            if (res && tid < 27) {
                const int dx = tid / 9 - 1, dy = tid / 3 % 3 - 1, dz = tid % 3 - 1;
                const int tz = t % g.NTZ + dz, ty = t / g.NTZ % g.NTY + dy, tx = t / (g.NTZ * g.NTY) + dx;
                const bool self = dx == 0 && dy == 0 && dz == 0;
                if ((!self || res == 2) && tx >= 0 && ty >= 0 && tz >= 0 && tx < g.NTX && ty < g.NTY && tz < g.NTZ)
                    next[(tx * g.NTY + ty) * g.NTZ + tz] = 1;
                if (self) *(volatile unsigned int *)&ctrl->changed[ph][slot] = 1;
            }
        }
        // slot (r + 1) % 3 was last read after barrier r - 2, which every CTA has left
        if (tid == 0 && blockIdx.x == 0) ctrl->changed[ph][(r + 1) % 3] = 0;
        if (tid == 0 && visits) atomicAdd(&ctrl->visits[ph], visits);
        grid_barrier(&ctrl->barrier, bar_target);
        if (tid == 0) *s_flag = *(volatile unsigned int *)&ctrl->changed[ph][slot];
        __syncthreads();
        if (!*s_flag) {
            if (tid == 0 && blockIdx.x == 0) ctrl->rounds[ph] = (unsigned int)(r + 1);
            return;
        }
    }
    if (tid == 0 && blockIdx.x == 0) {
        ctrl->rounds[ph] = (unsigned int)g.cap;
        if (!ctrl->status) ctrl->status = (unsigned int)PH;
    }
}

template <typename V, typename MT, typename OutT>
__global__ void __launch_bounds__(WS_THREADS, 1)
watershed_kernel(const V *__restrict__ img, const MT *__restrict__ markers, const uint8_t *__restrict__ mask,
                 const WsGeom g, WsCtrl *ctrl, unsigned int *dirty, uint64_t *lw, uint32_t *dw, uint32_t *iw,
                 OutT *__restrict__ out, int64_t *__restrict__ status) {
    __shared__ uint64_t s_w[WS_HALO_MAX];
    __shared__ int s_hoff[WS_MAXN];
    __shared__ unsigned int s_flag;
    const int tid = threadIdx.x;
    const int HY = g.TY + 2, HZ = g.TZ + 2;
    if (tid < g.nn) s_hoff[tid] = (g.off[tid][0] * HY + g.off[tid][1]) * HZ + g.off[tid][2];
    unsigned int bar_target = 0;
    const int ntiles = g.NTX * g.NTY * g.NTZ;
    const int64_t stride = (int64_t)gridDim.x * WS_THREADS;
    const int64_t first = (int64_t)blockIdx.x * WS_THREADS + tid;
    auto coords = [&](int64_t p, int &x, int &y, int &z) {
        z = (int)(p % g.Z);
        y = (int)(p / g.Z % g.Y);
        x = (int)(p / ((int64_t)g.Z * g.Y));
    };

    // phase 1: levels.  Markers outside the mask are dropped (scikit-image's markers * mask).
    for (int64_t p = first; p < g.npix; p += stride)
        lw[p] = (!mask || mask[p]) && markers[p] != 0 ? level_key(img[p]) : WS_INF;
    grid_barrier(&ctrl->barrier, bar_target);
    ws_phase<1, uint64_t>(g, img, markers, mask, lw, nullptr, dirty, ctrl, bar_target, s_w, s_hoff, &s_flag);

    // phase 2: candidates (neighbours of minimal level) and hops.  L == INF: outside the mask or unreached.
    for (int64_t p = first; p < g.npix; p += stride) {
        const uint64_t lp = __ldcg(lw + p);
        uint32_t info = WS_FIXED, d = WS_INF32;
        if (lp != WS_INF && markers[p] != 0) {
            d = 0;
        } else if (lp != WS_INF) {
            int x, y, z;
            coords(p, x, y, z);
            uint64_t ml = WS_INF;
            uint32_t cand = 0;
            for (int k = 0; k < g.nn; ++k) {
                const int qx = x + g.off[k][0], qy = y + g.off[k][1], qz = z + g.off[k][2];
                if (!in_image(g, qx, qy, qz)) continue;
                const uint64_t lq = __ldcg(lw + ((int64_t)qx * g.Y + qy) * g.Z + qz);
                if (lq < ml) { ml = lq; cand = 1u << k; }
                else if (lq == ml) cand |= 1u << k;
            }
            if (lp > ml) { info = WS_FIXED | cand; d = 1; }    // entry pixel: v(p) > min L
            else info = cand;
        }
        iw[p] = info;
        dw[p] = d;
    }
    grid_barrier(&ctrl->barrier, bar_target);
    ws_phase<2, uint32_t>(g, img, markers, mask, dw, iw, dirty + 2 * ntiles, ctrl, bar_target, s_w, s_hoff, &s_flag);

    // phase 3: parents (candidates of minimal d) and labels, stored sign-flipped so that unsigned order is signed
    // order.  The label words take the level array's place; d == 0 exactly at the markers.
    for (int64_t p = first; p < g.npix; p += stride) {
        const uint32_t dp = __ldcg(dw + p);
        uint32_t info = WS_FIXED;
        uint64_t lab = WS_INF;
        if (dp == 0) {
            lab = (uint64_t)(int64_t)markers[p] ^ WS_SIGN;
        } else if (dp != WS_INF32) {
            int x, y, z;
            coords(p, x, y, z);
            uint32_t md = WS_INF32, par = 0;
            for (uint32_t b = __ldcg(iw + p) & ~WS_FIXED; b; b &= b - 1) {
                const int k = __ffs(b) - 1;
                const uint32_t dq = __ldcg(dw + ((int64_t)(x + g.off[k][0]) * g.Y + y + g.off[k][1]) * g.Z + z + g.off[k][2]);
                if (dq < md) { md = dq; par = 1u << k; }
                else if (dq == md) par |= 1u << k;
            }
            info = par;
        }
        iw[p] = info;
        lw[p] = lab;
    }
    grid_barrier(&ctrl->barrier, bar_target);
    ws_phase<3, uint64_t>(g, img, markers, mask, lw, iw, dirty + 4 * ntiles, ctrl, bar_target, s_w, s_hoff, &s_flag);

    for (int64_t p = first; p < g.npix; p += stride)
        out[p] = __ldcg(dw + p) != WS_INF32 ? (OutT)(int64_t)(__ldcg(lw + p) ^ WS_SIGN) : (OutT)0;
    if (blockIdx.x == 0 && tid == 0) {
        const volatile WsCtrl *c = ctrl;
        status[0] = c->status;
        for (int k = 0; k < 3; ++k) {
            status[1 + k] = c->rounds[k];
            status[4 + k] = (int64_t)c->visits[k];
        }
        status[7] = gridDim.x;
    }
}

static bool ws_geom(int ndim, int d0, int d1, int d2, int connectivity, WsGeom &g) {
    if (ndim == 2) { g.X = 1; g.Y = d0; g.Z = d1; }
    else if (ndim == 3) { g.X = d0; g.Y = d1; g.Z = d2; }
    else return false;
    if (g.X < 1 || g.Y < 1 || g.Z < 1 || connectivity < 1 || connectivity > ndim) return false;
    auto edge = [](int n, int cap) { int p = 1; while (p < n && p < cap) p <<= 1; return p; };
    const int e = ndim == 2 ? WS_EDGE2 : WS_EDGE3;
    g.TX = ndim == 2 ? 1 : edge(g.X, e);
    g.TY = edge(g.Y, e);
    g.TZ = edge(g.Z, e);
    g.NTX = (g.X + g.TX - 1) / g.TX;
    g.NTY = (g.Y + g.TY - 1) / g.TY;
    g.NTZ = (g.Z + g.TZ - 1) / g.TZ;
    g.hx = ndim == 3 ? 1 : 0;
    // scipy's generate_binary_structure(ndim, connectivity): city-block distance <= connectivity, one step per axis
    g.nn = 0;
    for (int dx = -1; dx <= 1; ++dx)
        for (int dy = -1; dy <= 1; ++dy)
            for (int dz = -1; dz <= 1; ++dz) {
                const int dist = (dx != 0) + (dy != 0) + (dz != 0);
                if (dist == 0 || dist > connectivity || (ndim == 2 && dx != 0)) continue;
                g.off[g.nn][0] = (signed char)dx;
                g.off[g.nn][1] = (signed char)dy;
                g.off[g.nn][2] = (signed char)dz;
                ++g.nn;
            }
    g.npix = (int64_t)g.X * g.Y * g.Z;
    g.cap = g.npix + 1;
    return true;
}

static int64_t ws_align(int64_t b) { return (b + 255) / 256 * 256; }

}  // namespace hipr

using namespace hipr;

extern "C" int64_t hipr_watershed_workspace_bytes(int ndim, int d0, int d1, int d2, int image_dtype, int label_bytes) {
    if (image_dtype != HIPR_F32 && image_dtype != HIPR_F64) return HIPR_E_DTYPE;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    WsGeom g;
    if (!ws_geom(ndim, d0, d1, d2, 1, g)) return HIPR_E_ARG;
    if (g.npix > 0x7fffffffLL) return HIPR_E_RANGE;
    const int64_t ntiles = (int64_t)g.NTX * g.NTY * g.NTZ;
    return WS_CTRL_BYTES + ws_align(6 * ntiles * 4) + ws_align(g.npix * 8) + 2 * ws_align(g.npix * 4);
}

template <typename V, typename MT, typename OutT>
static int ws_launch(const void *image, const void *markers, const uint8_t *mask, const WsGeom &g, char *ws,
                     void *out, int64_t *status, cudaStream_t st) {
    auto kern = watershed_kernel<V, MT, OutT>;
    int dev = 0, sms = 0, per_sm = 0, coop = 0;
    HIPR_CUDA(cudaGetDevice(&dev));
    HIPR_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) return HIPR_E_UNSUPPORTED;
    HIPR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    HIPR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WS_THREADS, 0));
    if (per_sm < 1) return HIPR_E_UNSUPPORTED;
    const int64_t ntiles = (int64_t)g.NTX * g.NTY * g.NTZ;
    int64_t grid = (int64_t)sms * per_sm;
    if (grid > ntiles) grid = ntiles;
    WsCtrl *ctrl = (WsCtrl *)ws;
    unsigned int *dirty = (unsigned int *)(ws + WS_CTRL_BYTES);
    char *p = ws + WS_CTRL_BYTES + ws_align(6 * ntiles * 4);
    uint64_t *lw = (uint64_t *)p;
    uint32_t *dw = (uint32_t *)(p + ws_align(g.npix * 8));
    uint32_t *iw = (uint32_t *)(p + ws_align(g.npix * 8) + ws_align(g.npix * 4));
    HIPR_CUDA(cudaMemsetAsync(ws, 0, WS_CTRL_BYTES + 6 * ntiles * 4, st));
    const V *img = (const V *)image;
    const MT *mk = (const MT *)markers;
    OutT *o = (OutT *)out;
    void *args[] = {&img, &mk, &mask, (void *)&g, &ctrl, &dirty, &lw, &dw, &iw, &o, &status};
    HIPR_CUDA(cudaLaunchCooperativeKernel((const void *)kern, dim3((unsigned)grid), dim3(WS_THREADS), args, 0, st));
    return after_launch();
}

extern "C" int hipr_watershed(const void *image_dev, int image_dtype, const void *markers_dev, int label_bytes,
                              const uint8_t *mask_dev, int ndim, int d0, int d1, int d2, int connectivity,
                              void *workspace_dev, int64_t workspace_bytes, void *labels_out, int64_t *status_dev,
                              void *stream) {
    WsGeom g;
    if (!image_dev || !markers_dev || !workspace_dev || !labels_out || !status_dev) return HIPR_E_ARG;
    if (!ws_geom(ndim, d0, d1, d2, connectivity, g)) return HIPR_E_ARG;
    const int64_t need = hipr_watershed_workspace_bytes(ndim, d0, d1, d2, image_dtype, label_bytes);
    if (need < 0) return (int)need;
    if (workspace_bytes < need) return HIPR_E_RANGE;
    char *ws = (char *)workspace_dev;
    cudaStream_t st = (cudaStream_t)stream;
    const bool f32 = image_dtype == HIPR_F32;
    if (label_bytes == 4)
        return f32 ? ws_launch<float, int, int>(image_dev, markers_dev, mask_dev, g, ws, labels_out, status_dev, st)
                   : ws_launch<double, int, int>(image_dev, markers_dev, mask_dev, g, ws, labels_out, status_dev, st);
    return f32 ? ws_launch<float, long long, long long>(image_dev, markers_dev, mask_dev, g, ws, labels_out, status_dev, st)
               : ws_launch<double, long long, long long>(image_dev, markers_dev, mask_dev, g, ws, labels_out, status_dev, st);
}

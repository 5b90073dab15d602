// K10: connected-component labelling and the per-label passes built on it (remove_small_objects,
// binary_fill_holes, clear_border, relabel_sequential).
//
// Labelling is union-find on linear pixel indices (Playne & Hawick 2018; Allegretti et al. 2019), in five
// launches whatever the image holds:
//   1. tile_union_kernel   one CTA per tile: union-find in shared memory over the neighbours inside the tile, then
//                          every pixel's parent = its tile root (global index), background = BG.
//   2. border_union_kernel unions across tile faces in global memory.
//   3. flatten_kernel      every pixel points at its root.  A union always links the larger root under the smaller
//                          (atomicMin), so parent[p] <= p and the root of a component is its smallest linear index:
//                          its first pixel in raster order.  Per chunk of LB_CHUNK pixels the roots are ranked (the
//                          root's parent becomes -(rank + 1)) and counted.
//   4. chunk_scan_kernel   one CTA: exclusive scan of the chunk counts, total -> *n.
//   5. write_labels_kernel label = chunk offset of the root + rank + 1, 0 for the background.
// Nothing iterates until a fixed point, so a one-pixel serpentine costs what noise costs; the numbering depends only
// on the image (the root is the minimum, whatever order the unions ran in); every workspace word is written before
// it is read.
//
// A 2-D (H, W) image is the volume (1, H, W): the in-plane neighbours of 6- / 18-connectivity are the 4- / 8-
// neighbours.  Foreground: value != 0 (== 0 with `invert`, the background components of binary_fill_holes).  Two
// foreground neighbours are connected when the image is a uint8 mask, or when their values are equal (label image).
#include "hipr_common.cuh"

namespace hipr {

constexpr int LB_THREADS = 512;     // pixels per tile = threads of tile_union_kernel
constexpr int LB_CHUNK = 4096;      // pixels ranked by one CTA of flatten_kernel (512 threads x 8)
constexpr int LB_SCAN_ITEMS = 16;   // chunk counts per thread and round of chunk_scan_kernel
constexpr int BG = (int)0x80000000;

struct Dims {
    int X, Y, Z;      // volume (X, Y, Z), Z fastest
    int TX, TY, TZ;   // tile
    int NTY, NTZ;     // tiles along Y and Z
};

// Backward neighbour offsets (linear offset < 0) of scipy's generate_binary_structure(3, conn): a union for each
// pair is issued by the later pixel.  conn 1: 3 offsets, 2: 9, 3: 13.
__constant__ signed char c_off[13][3] = {
    {-1, 0, 0}, {0, -1, 0}, {0, 0, -1},                                        // faces
    {-1, -1, 0}, {-1, 1, 0}, {-1, 0, -1}, {-1, 0, 1}, {0, -1, -1}, {0, -1, 1},  // edges
    {-1, -1, -1}, {-1, -1, 1}, {-1, 1, -1}, {-1, 1, 1}};                        // corners
__host__ __device__ inline int n_offsets(int conn) { return conn == 1 ? 3 : conn == 2 ? 9 : 13; }

template <typename T>
__device__ __forceinline__ bool fg(T v, bool invert) { return (v != 0) != invert; }
// uint8 is a mask: any two foreground pixels connect.  Label images connect equal values.
template <typename T>
__device__ __forceinline__ bool same(T a, T b) { return sizeof(T) == 1 || a == b; }

// Find with path halving, on the shared-memory tile (pass 1) or the global parent array (pass 2).  A store replaces
// a parent by one of its ancestors, so it never changes which component a pixel belongs to and keeps
// parent[p] <= p; roots change only through the atomicMin of unite().
__device__ __forceinline__ int find_root(int *par, int a) {
    for (;;) {
        const int q = par[a];
        if (q == a) return a;
        const int r = par[q];
        if (r == q) return q;
        par[a] = r;
        a = r;
    }
}
__device__ void unite(int *par, int a, int b) {
    for (;;) {
        a = find_root(par, a);
        b = find_root(par, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(par + a, b);   // link the larger root under the smaller
        if (old == a) return;
        a = old;                                 // a was linked meanwhile: join its new parent instead
    }
}

template <typename T>
__global__ void __launch_bounds__(LB_THREADS)
tile_union_kernel(const T *__restrict__ img, Dims d, int conn, bool invert, int *__restrict__ par) {
    __shared__ int s_par[LB_THREADS];
    __shared__ T s_val[LB_THREADS];
    const int t = threadIdx.x;
    const int iz = t % d.TZ, iy = (t / d.TZ) % d.TY, ix = t / (d.TZ * d.TY);
    const int tile = blockIdx.x;
    const int tz = tile % d.NTZ, ty = (tile / d.NTZ) % d.NTY, tx = tile / (d.NTZ * d.NTY);
    const int x = tx * d.TX + ix, y = ty * d.TY + iy, z = tz * d.TZ + iz;
    const bool inside = x < d.X && y < d.Y && z < d.Z;
    const int64_t g = ((int64_t)x * d.Y + y) * d.Z + z;
    const T v = inside ? img[g] : T(0);
    const bool f = inside && fg(v, invert);
    s_val[t] = v;
    s_par[t] = f ? t : -1;
    __syncthreads();
    if (f) {
        const int no = n_offsets(conn);
        for (int k = 0; k < no; ++k) {
            const int jx = ix + c_off[k][0], jy = iy + c_off[k][1], jz = iz + c_off[k][2];
            if (jx < 0 || jy < 0 || jz < 0 || jy >= d.TY || jz >= d.TZ) continue;   // jx <= ix: never past the tile
            const int u = (jx * d.TY + jy) * d.TZ + jz;
            if (s_par[u] >= 0 && same(v, s_val[u])) unite(s_par, t, u);     // s_par[u] >= 0 iff foreground
        }
    }
    __syncthreads();
    if (!inside) return;
    int root = -1;
    if (f) root = find_root(s_par, t);
    // a tile's local raster order is the global one restricted to the tile, so the local minimum is the global one
    const int rz = root % d.TZ, ry = (root / d.TZ) % d.TY, rx = root / (d.TZ * d.TY);
    par[g] = f ? (int)(((int64_t)(tx * d.TX + rx) * d.Y + (ty * d.TY + ry)) * d.Z + (tz * d.TZ + rz)) : BG;
}

template <typename T>
__global__ void __launch_bounds__(LB_THREADS)
border_union_kernel(const T *__restrict__ img, Dims d, int conn, bool invert, int *__restrict__ par) {
    const int t = threadIdx.x;
    const int iz = t % d.TZ, iy = (t / d.TZ) % d.TY, ix = t / (d.TZ * d.TY);
    const int tile = blockIdx.x;
    const int tz = tile % d.NTZ, ty = (tile / d.NTZ) % d.NTY, tx = tile / (d.NTZ * d.NTY);
    const int x = tx * d.TX + ix, y = ty * d.TY + iy, z = tz * d.TZ + iz;
    if (x >= d.X || y >= d.Y || z >= d.Z) return;
    const bool face = ix == 0 || iy == 0 || iz == 0 || (conn > 1 && (iz == d.TZ - 1 || iy == d.TY - 1));
    if (!face) return;
    const int64_t g = ((int64_t)x * d.Y + y) * d.Z + z;
    const T v = img[g];
    if (!fg(v, invert)) return;
    const int no = n_offsets(conn);
    for (int k = 0; k < no; ++k) {
        const int jx = ix + c_off[k][0], jy = iy + c_off[k][1], jz = iz + c_off[k][2];
        if (jx >= 0 && jy >= 0 && jz >= 0 && jy < d.TY && jz < d.TZ) continue;   // inside the tile: done in pass 1
        const int nx = x + c_off[k][0], ny = y + c_off[k][1], nz = z + c_off[k][2];
        if (nx < 0 || ny < 0 || nz < 0 || ny >= d.Y || nz >= d.Z) continue;
        const int64_t h = ((int64_t)nx * d.Y + ny) * d.Z + nz;
        const T w = img[h];
        if (fg(w, invert) && same(v, w)) unite(par, (int)g, (int)h);
    }
}

// Per chunk of LB_CHUNK consecutive pixels: non-roots point at their root, roots take -(rank in chunk + 1).
// Roots are final after pass 2, so "is a root" is read once; a concurrent find stops at a root in either encoding.
__global__ void __launch_bounds__(LB_THREADS)
flatten_kernel(int *__restrict__ par, int64_t npix, int *__restrict__ chunk_count) {
    __shared__ int warp_tot[LB_THREADS / 32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int64_t base = (int64_t)blockIdx.x * LB_CHUNK;
    int carry = 0;   // roots in the earlier rounds, the same in every thread
    for (int r = 0; r < LB_CHUNK / LB_THREADS; ++r) {
        const int64_t p = base + r * LB_THREADS + t;
        const int q = p < npix ? par[p] : BG;
        bool root = false;
        if (q >= 0) {
            if (q == (int)p) {
                root = true;
            } else {
                int a = q, b;
                while ((b = par[a]) >= 0 && b != a) a = b;
                par[p] = a;
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, root);
        if (lane == 0) warp_tot[warp] = __popc(m);
        __syncthreads();
        int before = carry, total = 0;
#pragma unroll
        for (int w = 0; w < LB_THREADS / 32; ++w) {
            const int c = warp_tot[w];
            before += w < warp ? c : 0;
            total += c;
        }
        if (root) par[p] = -(before + __popc(m & ((1u << lane) - 1u)) + 1);
        carry += total;
        __syncthreads();
    }
    if (t == 0) chunk_count[blockIdx.x] = carry;
}

// One CTA: chunk counts -> exclusive offsets (in place), total -> *n.
__global__ void __launch_bounds__(1024)
chunk_scan_kernel(int *__restrict__ chunk, int64_t nchunks, long long *__restrict__ n) {
    __shared__ int warp_tot[32];
    __shared__ int carry;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nchunks; base += 1024 * LB_SCAN_ITEMS) {
        int v[LB_SCAN_ITEMS];
        int sum = 0;
#pragma unroll
        for (int i = 0; i < LB_SCAN_ITEMS; ++i) {
            const int64_t c = base + (int64_t)t * LB_SCAN_ITEMS + i;
            v[i] = c < nchunks ? chunk[c] : 0;
            sum += v[i];
        }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += u;
            }
            warp_tot[lane] = w;
        }
        __syncthreads();
        int run = carry + (warp > 0 ? warp_tot[warp - 1] : 0) + incl - sum;
#pragma unroll
        for (int i = 0; i < LB_SCAN_ITEMS; ++i) {
            const int64_t c = base + (int64_t)t * LB_SCAN_ITEMS + i;
            if (c < nchunks) chunk[c] = run;
            run += v[i];
        }
        __syncthreads();
        if (t == 0) carry += warp_tot[31];
        __syncthreads();
    }
    if (t == 0) *n = carry;
}

template <typename OutT>
__global__ void __launch_bounds__(256)
write_labels_kernel(const int *__restrict__ par, int64_t npix, const int *__restrict__ chunk_off, OutT *__restrict__ out) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
        int q = par[p];
        OutT lab = 0;
        if (q != BG) {
            int r = (int)p;
            while (q >= 0) { r = q; q = par[r]; }   // after pass 3: at most one step
            lab = (OutT)chunk_off[r / LB_CHUNK] + (OutT)(-q);
        }
        out[p] = lab;
    }
}

// Per-label pixel counts, as np.bincount: each thread walks LB_STRIP consecutive pixels and flushes runs of equal
// labels with one atomic; zeros are summed per warp.  border >= 0: only pixels within `border` of an edge of one of
// the image's axes count.  Labels < 0 or > max_label go to *overflow.
constexpr int LB_STRIP = 32;

__device__ __forceinline__ bool near_edge(int c, int n, int b) { return c <= b || c >= n - 1 - b; }

template <typename LabelT>
__global__ void __launch_bounds__(256)
label_counts_kernel(const LabelT *__restrict__ labels, Dims d, bool three_d, int border, int64_t max_label,
                    int *__restrict__ counts, int *__restrict__ overflow) {
    const int64_t npix = (int64_t)d.X * d.Y * d.Z;
    const int64_t p0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * LB_STRIP;
    int zeros = 0, over = 0;
    if (p0 < npix) {
        const int64_t p1 = p0 + LB_STRIP < npix ? p0 + LB_STRIP : npix;
        int z = (int)(p0 % d.Z);
        int64_t xy = p0 / d.Z;
        int y = (int)(xy % d.Y), x = (int)(xy / d.Y);
        long long cur = 0;
        int run = 0;
        for (int64_t p = p0; p < p1; ++p) {
            const bool take = border < 0 || near_edge(z, d.Z, border) || near_edge(y, d.Y, border) ||
                              (three_d && near_edge(x, d.X, border));
            if (take) {
                const long long lab = (long long)labels[p];
                if (lab == 0) {
                    ++zeros;
                } else if (lab < 0 || lab > max_label) {
                    ++over;
                } else {
                    if (lab != cur) {
                        if (run) atomicAdd(counts + cur, run);
                        cur = lab;
                        run = 0;
                    }
                    ++run;
                }
            }
            if (++z == d.Z) {
                z = 0;
                if (++y == d.Y) { y = 0; ++x; }
            }
        }
        if (run) atomicAdd(counts + cur, run);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        zeros += __shfl_xor_sync(0xffffffffu, zeros, o);
        over += __shfl_xor_sync(0xffffffffu, over, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (zeros) atomicAdd(counts, zeros);
        if (over && overflow) atomicAdd(overflow, over);
    }
}

// clear_border's write: out[p] = flagged[labels[p]] != 0 ? fill : image[p].
template <typename T>
__global__ void __launch_bounds__(256)
label_clear_kernel(const T *__restrict__ img, const int *__restrict__ labels, int64_t npix,
                   const int *__restrict__ flagged, T fill, T *__restrict__ out) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x)
        out[p] = flagged[labels[p]] ? fill : img[p];
}

// Tiles of up to 512 pixels, 32 along Z where the image allows it (coalesced rows); a volume splits the rest
// evenly between X and Y (4 x 4 x 32), an image takes 16 rows.
static void choose_tile(Dims &d) {
    d.TZ = pow2_at_least(d.Z, 32);
    const int rest = LB_THREADS / d.TZ;
    d.TY = pow2_at_least(d.Y, d.X > 1 ? (rest >= 16 ? rest / 4 : rest) : rest);
    d.TX = pow2_at_least(d.X, rest / d.TY);
    d.NTY = (d.Y + d.TY - 1) / d.TY;
    d.NTZ = (d.Z + d.TZ - 1) / d.TZ;
}

}  // namespace hipr

using namespace hipr;

extern "C" int64_t hipr_label_workspace_bytes(int ndim, int d0, int d1, int d2) {
    Dims d;
    const int e = volume_xyz(ndim, d0, d1, d2, d.X, d.Y, d.Z);
    if (e) return e;
    const int64_t npix = (int64_t)d.X * d.Y * d.Z;
    return align256(npix * 4) + align256((npix + LB_CHUNK - 1) / LB_CHUNK * 4);
}

extern "C" int hipr_label(const void *image_dev, int dtype, int invert, int ndim, int d0, int d1, int d2,
                          int connectivity, void *workspace_dev, int64_t workspace_bytes, void *labels_out,
                          int label_bytes, int64_t *n_dev, void *stream) {
    Dims d;
    if (!image_dev || !workspace_dev || !labels_out || volume_xyz(ndim, d0, d1, d2, d.X, d.Y, d.Z) == HIPR_E_ARG)
        return HIPR_E_ARG;
    if (connectivity < 1 || connectivity > ndim) return HIPR_E_ARG;
    if (dtype != HIPR_U8 && dtype != HIPR_I32 && dtype != HIPR_I64) return HIPR_E_DTYPE;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    const int64_t need = hipr_label_workspace_bytes(ndim, d0, d1, d2);
    if (need < 0) return (int)need;
    if (workspace_bytes < need) return HIPR_E_RANGE;
    choose_tile(d);
    const int conn = connectivity;   // ndim 2: the in-plane offsets of 6- / 18-connectivity are the 4- / 8-neighbours
    const int64_t npix = (int64_t)d.X * d.Y * d.Z;
    const int64_t tiles = (int64_t)((d.X + d.TX - 1) / d.TX) * d.NTY * d.NTZ;
    const int threads = d.TX * d.TY * d.TZ;
    const int64_t nchunks = (npix + LB_CHUNK - 1) / LB_CHUNK;
    int *par = (int *)workspace_dev;
    int *chunk = (int *)((char *)workspace_dev + align256(npix * 4));
    cudaStream_t st = (cudaStream_t)stream;
    const bool inv = invert != 0;
    int e;
#define HIPR_LABEL_PASSES(T)                                                                                       \
    tile_union_kernel<T><<<(unsigned)tiles, threads, 0, st>>>((const T *)image_dev, d, conn, inv, par);            \
    if ((e = after_launch())) return e;                                                                            \
    border_union_kernel<T><<<(unsigned)tiles, threads, 0, st>>>((const T *)image_dev, d, conn, inv, par);          \
    if ((e = after_launch())) return e
    if (dtype == HIPR_U8) { HIPR_LABEL_PASSES(uint8_t); }
    else if (dtype == HIPR_I32) { HIPR_LABEL_PASSES(int); }
    else { HIPR_LABEL_PASSES(long long); }
#undef HIPR_LABEL_PASSES
    flatten_kernel<<<(unsigned)nchunks, LB_THREADS, 0, st>>>(par, npix, chunk);
    if ((e = after_launch())) return e;
    chunk_scan_kernel<<<1, 1024, 0, st>>>(chunk, nchunks, (long long *)(n_dev));
    if ((e = after_launch())) return e;
    int64_t blocks = (npix + 2047) / 2048;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (label_bytes == 4)
        write_labels_kernel<int><<<(unsigned)blocks, 256, 0, st>>>(par, npix, chunk, (int *)labels_out);
    else
        write_labels_kernel<long long><<<(unsigned)blocks, 256, 0, st>>>(par, npix, chunk, (long long *)labels_out);
    return after_launch();
}

extern "C" int hipr_label_counts(const void *labels_dev, int label_bytes, int ndim, int d0, int d1, int d2,
                                 int border, int64_t max_label, int32_t *counts_dev, int32_t *overflow_dev,
                                 void *stream) {
    Dims d;
    const int vol = volume_xyz(ndim, d0, d1, d2, d.X, d.Y, d.Z);
    if (!labels_dev || !counts_dev || max_label < 0 || vol == HIPR_E_ARG) return HIPR_E_ARG;
    if (label_bytes != 4 && label_bytes != 8) return HIPR_E_DTYPE;
    if (vol) return vol;
    const int64_t npix = (int64_t)d.X * d.Y * d.Z;
    cudaStream_t st = (cudaStream_t)stream;
    HIPR_CUDA(cudaMemsetAsync(counts_dev, 0, (size_t)(max_label + 1) * sizeof(int32_t), st));
    if (overflow_dev) HIPR_CUDA(cudaMemsetAsync(overflow_dev, 0, sizeof(int32_t), st));
    const int64_t threads = (npix + LB_STRIP - 1) / LB_STRIP;
    const unsigned blocks = (unsigned)((threads + 255) / 256);
    if (label_bytes == 4)
        label_counts_kernel<int><<<blocks, 256, 0, st>>>((const int *)labels_dev, d, ndim == 3, border, max_label,
                                                         counts_dev, overflow_dev);
    else
        label_counts_kernel<long long><<<blocks, 256, 0, st>>>((const long long *)labels_dev, d, ndim == 3, border,
                                                               max_label, counts_dev, overflow_dev);
    return after_launch();
}

extern "C" int hipr_label_clear(const void *image_dev, int dtype, const int32_t *labels_dev, int64_t npix,
                                const int32_t *flagged_dev, int64_t fill, void *out_dev, void *stream) {
    if (!image_dev || !labels_dev || !flagged_dev || !out_dev || npix < 1) return HIPR_E_ARG;
    if (npix > 0x7fffffffLL) return HIPR_E_RANGE;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t blocks = (npix + 2047) / 2048;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (dtype == HIPR_U8)
        label_clear_kernel<uint8_t><<<(unsigned)blocks, 256, 0, st>>>((const uint8_t *)image_dev, labels_dev, npix,
                                                                       flagged_dev, (uint8_t)fill, (uint8_t *)out_dev);
    else if (dtype == HIPR_I32)
        label_clear_kernel<int><<<(unsigned)blocks, 256, 0, st>>>((const int *)image_dev, labels_dev, npix, flagged_dev,
                                                                   (int)fill, (int *)out_dev);
    else if (dtype == HIPR_I64)
        label_clear_kernel<long long><<<(unsigned)blocks, 256, 0, st>>>((const long long *)image_dev, labels_dev, npix,
                                                                         flagged_dev, (long long)fill, (long long *)out_dev);
    else
        return HIPR_E_DTYPE;
    return after_launch();
}

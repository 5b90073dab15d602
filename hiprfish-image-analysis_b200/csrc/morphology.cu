// K12: binary erosion and dilation (scipy.ndimage.binary_erosion / binary_dilation with an odd structure, origin 0),
// one launch per pass.
//
// Erosion by S with border b: out[p] = AND over o in S of in[p + o], in = b outside the image.  Dilation uses scipy's
// own identity: dilation by S with border b = NOT(erosion of NOT in by the reflected S with border NOT b).  So one
// kernel does both; `inv` complements the staged input, the border and the result.
//
// A 2-D (H, W) image is the volume (1, H, W).  The structure is a table of runs: for every (dx, dy) row of the
// structure, each maximal run [za, zb] of members along z (the fastest axis).  The host turns a run into a bit offset
// into the CTA's staged tile and a length, and passes the table by value in the kernel parameters.
//
// A CTA owns a tile of TX planes x TY rows x TW 32-pixel words along z.  It stages the tile plus a halo of the
// structure's radii (rx planes, ry rows, one word on each side along z, rz <= 15 < 32) in shared memory as bit words,
// one warp ballot per word; pixels outside the image take the border value.  Each output word is the AND over the runs
// of the 64-bit window at the run's offset, eroded along z by the run's length with doubling shifts (log2 L steps).
// The 32 results are written back as bytes.
#include "hipr_common.cuh"

namespace hipr {

constexpr int MO_THREADS = 256;
constexpr int MO_STAGE = 8;            // staged words per warp and round
constexpr int MO_SMEM_WORDS = 12288;   // 48 KB: the static limit, no opt-in needed

struct MorphArgs {
    int X, Y, Z;            // volume, Z fastest
    int TX, TY, TW;         // tile: planes, rows, 32-pixel words
    int NTY, NTW;           // tiles along Y and along the words of Z
    int rx, ry;             // halo planes and rows
    int inv;                // 1: dilation (complement in, border and out)
    int fill;               // the staged bit outside the image (border value, complemented when inv)
    int nruns;
    // run k: offset * 32 + (length - 1), offset = the bit of the run's first member in the staged tile minus the bit
    // of the output word's first pixel
    int run[HIPR_MORPH_MAX_RUNS];
};

__device__ __forceinline__ uint32_t erode_run(const uint32_t *s_in, int q, int len) {
    const int w = q >> 5, s = q & 31;
    const uint32_t w0 = s_in[w], w1 = s_in[w + 1], w2 = s_in[w + 2];
    uint64_t v = ((uint64_t)__funnelshift_r(w1, w2, s) << 32) | __funnelshift_r(w0, w1, s);
    // v[i] = AND of the window's bits i .. i + span - 1; bits 0..31 only ever read bits <= 31 + len - 1 <= 61
    int span = 1;
    while (2 * span <= len) {
        v &= v >> span;
        span *= 2;
    }
    if (span < len) v &= v >> (len - span);
    return (uint32_t)v;
}

__global__ void __launch_bounds__(MO_THREADS)
morphology_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, const MorphArgs a) {
    extern __shared__ uint32_t smem[];
    const int SY = a.TY + 2 * a.ry, SW = a.TW + 2;
    const int nstage = (a.TX + 2 * a.rx) * SY * SW;
    uint32_t *s_in = smem;                 // nstage words + 1 pad word (erode_run reads one word past a row)
    uint32_t *s_out = smem + nstage + 1;   // TX * TY * TW result words
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int tile = blockIdx.x;
    const int tw = tile % a.NTW, ty = (tile / a.NTW) % a.NTY, tx = tile / (a.NTW * a.NTY);
    const int x0 = tx * a.TX, y0 = ty * a.TY, z0 = tw * a.TW * 32;

    // MO_STAGE words per warp and round, their loads issued before the first ballot: the staging is bound by the
    // latency of these byte loads, not by their bandwidth
    const bool fill = a.fill != 0, inv = a.inv != 0;
    for (int w0 = warp * MO_STAGE; w0 < nstage; w0 += MO_THREADS / 32 * MO_STAGE) {
        uint8_t v[MO_STAGE];
        bool inside[MO_STAGE];
#pragma unroll
        for (int u = 0; u < MO_STAGE; ++u) {
            const int w = w0 + u;
            const int pw = w % SW, py = (w / SW) % SY, px = w / (SW * SY);
            const int x = x0 - a.rx + px, y = y0 - a.ry + py, z = z0 + (pw - 1) * 32 + lane;
            inside[u] = w < nstage && x >= 0 && x < a.X && y >= 0 && y < a.Y && z >= 0 && z < a.Z;
            v[u] = inside[u] ? in[((int64_t)x * a.Y + y) * a.Z + z] : 0;
        }
#pragma unroll
        for (int u = 0; u < MO_STAGE; ++u) {
            const uint32_t word = __ballot_sync(0xffffffffu, inside[u] ? (v[u] != 0) != inv : fill);
            if (lane == 0 && w0 + u < nstage) s_in[w0 + u] = word;
        }
    }
    if (t == 0) s_in[nstage] = 0u;
    __syncthreads();

    const int nout = a.TX * a.TY * a.TW;
    for (int k = t; k < nout; k += MO_THREADS) {
        const int ow = k % a.TW, oy = (k / a.TW) % a.TY, ox = k / (a.TW * a.TY);
        const int base = (((ox + a.rx) * SY + (oy + a.ry)) * SW + ow + 1) * 32;
        uint32_t r = 0xffffffffu;   // AND over no member: erosion by an empty structure is all True
        for (int j = 0; j < a.nruns; ++j) {
            const int run = a.run[j];
            r &= erode_run(s_in, base + (run >> 5), (run & 31) + 1);
        }
        s_out[k] = inv ? ~r : r;
    }
    __syncthreads();

    const int rowpix = a.TW * 32;
    for (int i = t; i < nout * 32; i += MO_THREADS) {
        const int oz = i % rowpix, oy = (i / rowpix) % a.TY, ox = i / (rowpix * a.TY);
        const int x = x0 + ox, y = y0 + oy, z = z0 + oz;
        if (x < a.X && y < a.Y && z < a.Z)
            out[((int64_t)x * a.Y + y) * a.Z + z] =
                (uint8_t)((s_out[(ox * a.TY + oy) * a.TW + (oz >> 5)] >> (oz & 31)) & 1u);
    }
}

static int stage_words(const MorphArgs &a) {
    return (a.TX + 2 * a.rx) * (a.TY + 2 * a.ry) * (a.TW + 2) + 1 + a.TX * a.TY * a.TW;
}

// 256 output words per tile: up to 8 words (256 pixels) along z, the rest rows (2-D) or split between planes and rows
// (3-D); then planes and rows are halved until the staged tile fits 48 KB (at radii 15 and 15 a 1 x 1 x 8 tile stages
// 31 x 31 x 10 words, so the loop ends).
static void choose_tile(MorphArgs &a) {
    const int nw = (a.Z + 31) / 32;
    a.TW = pow2_at_least(nw, 8);
    const int rest = MO_THREADS / a.TW;   // >= 32
    a.TY = pow2_at_least(a.Y, a.X > 1 ? rest / 8 : rest);
    a.TX = pow2_at_least(a.X, rest / a.TY);
    while (stage_words(a) > MO_SMEM_WORDS) {
        if (a.TX >= a.TY && a.TX > 1) a.TX >>= 1;
        else a.TY >>= 1;
    }
    a.NTY = (a.Y + a.TY - 1) / a.TY;
    a.NTW = (nw + a.TW - 1) / a.TW;
}

}  // namespace hipr

using namespace hipr;

extern "C" int hipr_morphology_runs(const uint8_t *structure_host, int s0, int s1, int s2, int32_t *runs_out,
                                    int capacity) {
    if (!structure_host || (capacity > 0 && !runs_out)) return HIPR_E_ARG;
    if (s0 < 1 || s1 < 1 || s2 < 1 || !(s0 & s1 & s2 & 1)) return HIPR_E_ARG;
    if (s0 > HIPR_MORPH_MAX_EXTENT || s1 > HIPR_MORPH_MAX_EXTENT || s2 > HIPR_MORPH_MAX_EXTENT) return HIPR_E_RANGE;
    int n = 0;
    for (int i = 0; i < s0; ++i)
        for (int j = 0; j < s1; ++j)
            for (int k = 0; k < s2; ++k) {
                const uint8_t *row = structure_host + ((int64_t)i * s1 + j) * s2;
                if (!row[k] || (k > 0 && row[k - 1])) continue;
                int e = k;
                while (e + 1 < s2 && row[e + 1]) ++e;
                if (n < capacity) {
                    int32_t *r = runs_out + 4 * n;
                    r[0] = i - s0 / 2; r[1] = j - s1 / 2; r[2] = k - s2 / 2; r[3] = e - s2 / 2;
                }
                ++n;
            }
    return n;
}

extern "C" int64_t hipr_morphology_workspace_bytes(int ndim, int d0, int d1, int d2, int iterations) {
    int X, Y, Z;
    const int e = volume_xyz(ndim, d0, d1, d2, X, Y, Z);
    if (e == HIPR_E_ARG || iterations < 1) return HIPR_E_ARG;
    if (e) return e;
    return iterations > 1 ? align256((int64_t)X * Y * Z) : 0;
}

extern "C" int hipr_binary_morphology(const uint8_t *mask_dev, int ndim, int d0, int d1, int d2,
                                      const uint8_t *structure_host, int s0, int s1, int s2, int dilate,
                                      int border_value, int iterations, void *workspace_dev, int64_t workspace_bytes,
                                      uint8_t *out_dev, void *stream) {
    MorphArgs a;
    if (!mask_dev || !out_dev || volume_xyz(ndim, d0, d1, d2, a.X, a.Y, a.Z) == HIPR_E_ARG) return HIPR_E_ARG;
    if (ndim == 2) { s2 = s1; s1 = s0; s0 = 1; }
    const int64_t need = hipr_morphology_workspace_bytes(ndim, d0, d1, d2, iterations);
    if (need < 0) return (int)need;
    if (workspace_bytes < need || (need > 0 && !workspace_dev)) return HIPR_E_RANGE;
    int32_t runs[4 * HIPR_MORPH_MAX_RUNS];
    const int nruns = hipr_morphology_runs(structure_host, s0, s1, s2, runs, HIPR_MORPH_MAX_RUNS);
    if (nruns < 0) return nruns;
    if (nruns > HIPR_MORPH_MAX_RUNS) return HIPR_E_RANGE;
    a.rx = s0 / 2;
    a.ry = s1 / 2;
    a.inv = dilate != 0;
    a.fill = (border_value != 0) != (dilate != 0);
    a.nruns = nruns;
    choose_tile(a);
    const int SY = a.TY + 2 * a.ry, SW = a.TW + 2;
    for (int k = 0; k < nruns; ++k) {
        int dx = runs[4 * k], dy = runs[4 * k + 1], za = runs[4 * k + 2], zb = runs[4 * k + 3];
        if (dilate) {   // the reflected structure: member o becomes -o
            const int t = za;
            dx = -dx; dy = -dy; za = -zb; zb = -t;
        }
        a.run[k] = ((dx * SY + dy) * SW * 32 + za) * 32 + (zb - za);
    }
    const int64_t tiles = (int64_t)((a.X + a.TX - 1) / a.TX) * a.NTY * a.NTW;
    if (tiles > 0x7fffffffLL) return HIPR_E_RANGE;
    const size_t smem = (size_t)stage_words(a) * sizeof(uint32_t);
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t *src = mask_dev;
    for (int it = 0; it < iterations; ++it) {
        // the last pass writes out_dev; earlier ones alternate with the workspace backwards from it
        uint8_t *dst = ((iterations - 1 - it) & 1) ? (uint8_t *)workspace_dev : out_dev;
        morphology_kernel<<<(unsigned)tiles, MO_THREADS, smem, st>>>(src, dst, a);
        const int e = after_launch();
        if (e) return e;
        src = dst;
    }
    return HIPR_OK;
}

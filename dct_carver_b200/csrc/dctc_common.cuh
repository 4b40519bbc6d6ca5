// Shared device helpers of the DCT-Carver energy kernels (sm_100a).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include "dctc_dct_gen.cuh"

// Arguments of every K1 variant.  Rows are "virtual": y in [-top_rows, h + bot_rows) maps to the top halo,
// the band itself or the bottom halo; outside that range the coordinate clamp of the reference
// (src/render.c:122-132) replicates the outermost row.  A plain image is a band with no halos.
struct DctcK1Args {
    const uint8_t* img;
    const uint8_t* top;
    const uint8_t* bot;
    size_t pitch, top_pitch, bot_pitch;
    size_t frame_stride;      // bytes between frames (batch launches, blockIdx.z)
    float* out;
    size_t out_pitch;         // floats
    size_t out_frame_stride;  // floats
    int w, h;                 // band size: outputs are produced for rows [0,h)
    int top_rows, bot_rows;
    int channels;
    float w_edges, w_textures;  // edges/255, textures/255 (luma is kept in 0..255 units inside the kernels)
    // band mode (K2, per-seam incremental update): when seam != nullptr only the pixels of row y with
    //   x in [min_{|y'-y|<=band_r} seam[y'] - band_r, max_{|y'-y|<=band_r} seam[y'] + band_r - 1] /\ [0, w-1]
    // are produced (liblqr update_emap), and also copied to band_vals[y*band_stride + x - xmin(y)].  Batch launches:
    // frame z reads its seam at seam + z * seam_frame_stride (band_vals is then left null).
    const int* seam;
    float* band_vals;
    int band_r, band_stride;
    int seam_frame_stride;
    // preview operator (dct_energy_preview_rows, src/render.c:31-60): window offsets -(C-1) .. b-C with C = (b-1)/2
    // (src/dct.h:8-9), BT.601 byte luminance (src/render.h:5), first transform index walks y (tile kernel only)
    int preview;
    // Global row of band row 0 (row bands of a taller image; 0 for whole images).  Only K1-TC16 uses it: its 16-row
    // steps are anchored to the global row grid, so a pixel's FP32 accumulation order does not depend on the band cut.
    int row_origin;
    // launch with programmatic stream serialization (device seam loop; tile kernel only)
    int pdl;
};

// Band mode of a biased carver session (tile kernel only, a kernel argument of its own so that DctcK1Args and the other
// kernels' parameters keep their layout): the stored value is e + bias[y][x] / ext, bias laid out like DctcK1Args::out.
struct DctcK1Bias {
    const float* bias;
    float ext;
};

// Band limits of row y for a removed seam (seam[] in the coordinates before removal, w = width after removal).
__host__ __device__ __forceinline__ void dctc_band_limits(const int* seam, int y, int h, int w, int r, int* xmin, int* xmax)
{
    int lo = seam[y], hi = seam[y];
    for (int d = -r; d <= r; d++) {
        const int yy = y + d;
        if (yy < 0 || yy >= h) continue;
        const int s = seam[yy];
        lo = s < lo ? s : lo;
        hi = s > hi ? s : hi;
    }
    lo -= r;
    hi += r - 1;
    *xmin = lo < 0 ? 0 : lo;
    *xmax = hi > w - 1 ? w - 1 : hi;
}

// Rec.709 luma in 0..255 units (the 1/255 normalisation of liblqr's reader is folded into the final weight,
// which is exact for the linear transform).  [liblqr LQR_ER_LUMA, see oracle/oracle_luma.h]
__device__ __forceinline__ float dctc_luma255(const uint8_t* __restrict__ p, int channels)
{
    float v;
    if (channels >= 3) {
        v = fmaf(0.2126f, (float) p[0], fmaf(0.7152f, (float) p[1], 0.0722f * (float) p[2]));
    } else {
        v = (float) p[0];
    }
    if (channels == 2 || channels == 4) v *= (float) p[channels - 1] * (1.0f / 255.0f);
    return v;
}

// Preview path luminance: RGB2LUMINANCE of src/render.h:5, (guchar)(16.0 + r*0.2568 + g*0.5041 + b*0.0979) evaluated in
// double in the reference's order and truncated; grey is passed through (src/render.c:62-79).
__device__ __forceinline__ float dctc_luma_preview(const uint8_t* __restrict__ p, int channels)
{
    if (channels < 3) return (float) p[0];
    const double v = __dadd_rn(__dadd_rn(__dadd_rn(16.0, __dmul_rn((double) p[0], 0.2568)), __dmul_rn((double) p[1], 0.5041)),
                               __dmul_rn((double) p[2], 0.0979));
    return (float) (uint8_t) v;
}

__device__ __forceinline__ const uint8_t* dctc_row_ptr(const DctcK1Args& a, const uint8_t* img, int vy)
{
    vy = max(-a.top_rows, min(vy, a.h + a.bot_rows - 1));
    if (vy < 0) return a.top + (size_t) (vy + a.top_rows) * a.top_pitch;
    if (vy >= a.h) return a.bot + (size_t) (vy - a.h) * a.bot_pitch;
    return img + (size_t) vy * a.pitch;
}

// Last-arg-max bookkeeping of weighted_max_dct_correlation (src/dct.c:96-110) without indices.
// Row-major index i = k1*B + k2; edge atoms are i=1 and i=B (src/dct.c:10-43).  With
//   A = |T[0][1]|, M = max|T[0][2..B-1]|, Bv = |T[1][0]|, Z = max over i > B
// the last maximal index is a texture atom iff  Z >= max(A,M,Bv)  or  (Bv < max(A,M) and M >= A).
template <bool UNIFORM>
struct DctcTracker;

template <>
struct DctcTracker<true> {   // edges == textures: only the maximum matters
    float m;
    __device__ __forceinline__ void init() { m = 0.0f; }
    template <int B>
    __device__ __forceinline__ void add(int k1, const float* X)
    {
#pragma unroll
        for (int k2 = 0; k2 < B; k2++)
            if (k1 != 0 || k2 != 0) m = fmaxf(m, fabsf(X[k2]));
    }
    template <int B>
    __device__ __forceinline__ void add_t(int k1, const float* X) { add<B>(k1, X); }
    __device__ __forceinline__ float result(float we, float wt) const { (void) we; return m * wt; }
};

template <>
struct DctcTracker<false> {
    float a, mm, bv, z;
    __device__ __forceinline__ void init() { a = 0.0f; mm = -1.0f; bv = 0.0f; z = 0.0f; }
    template <int B>
    __device__ __forceinline__ void add(int k1, const float* X)
    {
        if (k1 == 0) {
            a = fabsf(X[1]);
#pragma unroll
            for (int k2 = 2; k2 < B; k2++) mm = fmaxf(mm, fabsf(X[k2]));
        } else if (k1 == 1) {
            bv = fabsf(X[0]);
#pragma unroll
            for (int k2 = 1; k2 < B; k2++) z = fmaxf(z, fabsf(X[k2]));
        } else {
#pragma unroll
            for (int k2 = 0; k2 < B; k2++) z = fmaxf(z, fabsf(X[k2]));
        }
    }
    // transposed scan (preview path: the first transform index walks y): element (k1, k2) of the x-first layout is
    // T[k2][k1] of the reference's matrix, so the categories swap roles
    template <int B>
    __device__ __forceinline__ void add_t(int k1, const float* X)
    {
#pragma unroll
        for (int k2 = 0; k2 < B; k2++) {
            const float v = fabsf(X[k2]);
            if (k2 == 0) {
                if (k1 == 1) a = v;
                else if (k1 >= 2) mm = fmaxf(mm, v);
            } else if (k2 == 1 && k1 == 0) {
                bv = v;
            } else {
                z = fmaxf(z, v);
            }
        }
    }
    __device__ __forceinline__ float result(float we, float wt) const
    {
        const float am = fmaxf(a, mm);
        const float top = fmaxf(fmaxf(am, bv), z);
        const bool tex = (z >= fmaxf(am, bv)) || (!(bv >= am) && (mm >= a));
        return top * (tex ? wt : we);
    }
};

// Counter-based synthetic image generator (bench + tests), bit-identical to dctc_synth_byte() on the host.
__host__ __device__ __forceinline__ uint32_t dctc_mix32(uint32_t h)
{
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}

__host__ __device__ __forceinline__ uint8_t dctc_synth_px(uint32_t seed, uint32_t frame, uint32_t y, uint32_t x,
                                                          uint32_t c, int pattern)
{
    switch (pattern) {
    default:
    case 0: {  // P1 iid uniform noise
        uint32_t h = seed ^ (frame * 0x9E3779B1u);
        h = dctc_mix32(h ^ (y * 0x85EBCA77u));
        h = dctc_mix32(h ^ (x * 0xC2B2AE3Du));
        h = dctc_mix32(h ^ (c * 0x27D4EB2Fu));
        return (uint8_t) (h >> 24);
    }
    case 1: {  // P2 smooth gradient + slow triangle waves (near-zero AC, tie stress), integer-only
        uint32_t t = (x + 2u * y + 5u * frame + 3u * c) & 511u;
        uint32_t tri = t < 256u ? t : 511u - t;
        uint32_t g = ((x >> 3) + (y >> 4) + (seed & 15u)) & 255u;
        return (uint8_t) ((tri + g) >> 1);
    }
    case 2: {  // P3 8-px checkerboard with constant patches (exact ties, zero energy)
        uint32_t cell = ((x >> 3) + (y >> 3) + frame) & 1u;
        uint32_t flat = (((x >> 6) + (y >> 6)) % 3u) == 0u;
        return (uint8_t) (flat ? 128u : (cell ? 200u + 10u * c : 40u));
    }
    case 3: {  // P4 step edges at several orientations (edge-atom dominance)
        int xi = (int) (x & 63u) - 32, yi = (int) (y & 63u) - 32;
        uint32_t o = ((x >> 6) + 3u * (y >> 6) + frame) & 7u;
        int s;
        switch (o) {
        case 0: s = xi; break;
        case 1: s = yi; break;
        case 2: s = xi + yi; break;
        case 3: s = xi - yi; break;
        case 4: s = 2 * xi + yi; break;
        case 5: s = xi - 2 * yi; break;
        case 6: s = 3 * xi + yi; break;
        default: s = xi + 3 * yi; break;
        }
        return (uint8_t) (s >= 0 ? 220u - 20u * c : 30u + 5u * c);
    }
    }
}

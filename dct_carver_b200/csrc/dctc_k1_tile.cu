// K1 (generic): full DCT energy map, FP32 CUDA cores, any block size B in {2,4,8,16}.
//
// Replaces, for a whole image at once, the reference's per-pixel chain
//   dct_pixel_energy (src/render.c:134-157) -> dctNxN (src/dct.c:77-94) -> weighted_max_dct_correlation
//   (src/dct.c:96-110), with liblqr's LQR_ER_LUMA reader fused in.
//
// One CTA produces a TW x TH tile of energies:
//   phase 0  u8 interleaved pixels (+ B-1 halo, coordinate clamp = edge replication) -> luma tile in smem
//   phase 1  1-D DCT along x of every window start (x, y'): H[k1][y'][x]; computed ONCE per (x,y') and
//            shared by the B vertically overlapping windows (B+1 instead of 2B 1-D DCTs per pixel)
//   phase 2  each thread owns P vertically adjacent pixels of one column: per k1 it loads P+B-1 samples of H,
//            runs P 1-D DCTs along y in registers and folds |T[k1][k2]| into the arg-max tracker
//   store    one coalesced float per pixel
#include "dctc_common.cuh"
#include "dctc_launch.h"

// full-map tile shape for block size 16 (tile width, height, rows per thread).  Measured on 8 frames of 4K RGB:
// 32x32 tiles with 8 rows per thread (128 threads, 2 CTAs/SM: 8 warps per SM) 761 us per frame, 4 rows per thread
// (256 threads) 569 us, 2 rows per thread 722 us, 16x64 tiles with 4 rows per thread 608 us.
#ifndef DCTC_TILE16_TW
#define DCTC_TILE16_TW 32
#define DCTC_TILE16_TH 32
#define DCTC_TILE16_P 4
#endif

// BIAS (band mode of a biased carver session): the band store writes the seam energy e + bias.bias / bias.ext
template <int B, int TW, int TH, int P, bool UNIFORM, bool BIAS>
__global__ void __launch_bounds__(TW* TH / P) dctc_k1_tile_kernel(const DctcK1Args a, const DctcK1Bias bias)
{
    DCTC_PDL_PROLOGUE();
    constexpr int NT = TW * TH / P;
    // samples before the pixel: carver path window offsets -B/2+1 .. B/2 (src/render.c:146-147); preview path
    // -(C-1) .. B-C with C = (B-1)/2 (src/render.c:43-44, src/dct.h:8-9)
    const int R0 = a.preview ? (B - 1) / 2 - 1 : B / 2 - 1;
    constexpr int LW = TW + B - 1, LH = TH + B - 1;
    extern __shared__ float smem[];
    float* __restrict__ L = smem;            // [LH][LW] luma
    float* __restrict__ Hs = smem + LH * LW;  // [B][LH][TW] x-pass coefficients

    const int tid = threadIdx.x;
    const int ty0 = blockIdx.y * TH;
    int tx0 = blockIdx.x * TW;
    __shared__ int s_xmin[TH], s_xmax[TH], s_x0;
    if (a.seam) {  // band mode: the tile row starts at the leftmost band pixel of its rows
        const int* seam = a.seam + (size_t) blockIdx.z * a.seam_frame_stride;
        if (tid < TH) {
            int lo = a.w, hi = -1;
            if (ty0 + tid < a.h) dctc_band_limits(seam, ty0 + tid, a.h, a.w, a.band_r, &lo, &hi);
            s_xmin[tid] = lo;
            s_xmax[tid] = hi;
        }
        __syncthreads();
        if (tid == 0) {
            int lo = a.w;
            for (int i = 0; i < TH; i++) lo = min(lo, s_xmin[i]);
            s_x0 = lo;
        }
        __syncthreads();
        tx0 += s_x0;
        if (tx0 >= a.w) return;
    }
    const uint8_t* __restrict__ img = a.img + (size_t) blockIdx.z * a.frame_stride;
    float* __restrict__ out = a.out + (size_t) blockIdx.z * a.out_frame_stride;

    // phase 0
    for (int i = tid; i < LH * LW; i += NT) {
        const int ly = i / LW, lx = i - ly * LW;
        const int gx = max(0, min(tx0 + lx - R0, a.w - 1));
        const uint8_t* row = dctc_row_ptr(a, img, ty0 + ly - R0);
        const uint8_t* px = row + (size_t) gx * a.channels;
        L[i] = a.preview ? dctc_luma_preview(px, a.channels) : dctc_luma255(px, a.channels);
    }
    __syncthreads();

    // phase 1: x-pass
    for (int i = tid; i < LH * TW; i += NT) {
        const int ly = i / TW, x = i - ly * TW;
        float v[B], X[B];
#pragma unroll
        for (int j = 0; j < B; j++) v[j] = L[ly * LW + x + j];
        dctc_dct_fwd<B>(v, X);
#pragma unroll
        for (int k = 0; k < B; k++) Hs[(k * LH + ly) * TW + x] = X[k];
    }
    __syncthreads();

    // phase 2: y-pass + arg-max
    const int x = tid % TW, y0 = (tid / TW) * P;
    DctcTracker<UNIFORM> tr[P];
#pragma unroll
    for (int p = 0; p < P; p++) tr[p].init();
    if (B >= 8) {
        // two k1 planes per packed FP32x2 transform (same operations and rounding as the scalar transform, half the
        // instructions): X2[k2] = (T[k1][k2], T[k1+1][k2])
#pragma unroll
        for (int k1 = 0; k1 < B; k1 += 2) {
            float2 col2[P + B - 1];
#pragma unroll
            for (int j = 0; j < P + B - 1; j++)
                col2[j] = make_float2(Hs[(k1 * LH + y0 + j) * TW + x], Hs[((k1 + 1) * LH + y0 + j) * TW + x]);
#pragma unroll
            for (int p = 0; p < P; p++) {
                float2 X2[B];
                dctc_dct_fwd2<(B >= 8 ? B : 8)>(col2 + p, X2);
                float Xa[B], Xb[B];
#pragma unroll
                for (int k = 0; k < B; k++) { Xa[k] = X2[k].x; Xb[k] = X2[k].y; }
                if (a.preview) { tr[p].template add_t<B>(k1, Xa); tr[p].template add_t<B>(k1 + 1, Xb); }
                else { tr[p].template add<B>(k1, Xa); tr[p].template add<B>(k1 + 1, Xb); }
            }
        }
    } else {
#pragma unroll
        for (int k1 = 0; k1 < B; k1++) {
            float col[P + B - 1];
#pragma unroll
            for (int j = 0; j < P + B - 1; j++) col[j] = Hs[(k1 * LH + y0 + j) * TW + x];
#pragma unroll
            for (int p = 0; p < P; p++) {
                float X[B];
                dctc_dct_fwd<B>(col + p, X);
                if (a.preview) tr[p].template add_t<B>(k1, X); else tr[p].template add<B>(k1, X);
            }
        }
    }
    const int gx = tx0 + x;
    if (gx < a.w) {
#pragma unroll
        for (int p = 0; p < P; p++) {
            const int gy = ty0 + y0 + p;
            if (gy >= a.h) continue;
            const float e = tr[p].result(a.w_edges, a.w_textures);
            if (!a.seam) {
                out[(size_t) gy * a.out_pitch + gx] = e;
            } else if (gx >= s_xmin[y0 + p] && gx <= s_xmax[y0 + p]) {
                if constexpr (BIAS) {
                    const float b = bias.bias[(size_t) blockIdx.z * a.out_frame_stride + (size_t) gy * a.out_pitch + gx];
                    out[(size_t) gy * a.out_pitch + gx] = __fadd_rn(e, __fdiv_rn(b, bias.ext));
                    continue;   // (no band_vals: dctc_carve_and_update refuses biased sessions)
                }
                out[(size_t) gy * a.out_pitch + gx] = e;
                if (a.band_vals) a.band_vals[(size_t) gy * a.band_stride + (gx - s_xmin[y0 + p])] = e;
            }
        }
    }
}

template <int B, int TW, int TH, int P, bool BIAS = false>
static cudaError_t launch_tile(const DctcK1Args& a, int n_frames, bool uniform, cudaStream_t stream, DctcK1Bias bias = {}, int dx = 1)
{
    constexpr int LW = TW + B - 1, LH = TH + B - 1;
    constexpr size_t smem = sizeof(float) * (size_t) (LH * LW + B * LH * TW);
    // band mode: a tile row spans at most dx * (TH-1 + 2*band_r) + 2*band_r + 1 columns (seam drift of dx per row over
    // TH+2r rows plus 2r; TH + 4*band_r for connected seams)
    const int span = a.seam ? dx * (TH - 1 + 2 * a.band_r) + 2 * a.band_r + 1 : a.w;
    dim3 grid((span + TW - 1) / TW, (a.h + TH - 1) / TH, n_frames), block(TW * TH / P);
    return dctc_dispatch<0>(uniform, 0, [&](auto U, auto) {   // one kernel for every channel count
        const cudaError_t e = cudaFuncSetAttribute(dctc_k1_tile_kernel<B, TW, TH, P, U, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (e != cudaSuccess) return e;
        if (a.pdl) return dctc_launch_pdl(dctc_k1_tile_kernel<B, TW, TH, P, U, BIAS>, grid, block, smem, stream, true, a, bias);
        dctc_k1_tile_kernel<B, TW, TH, P, U, BIAS><<<grid, block, smem, stream>>>(a, bias);
        return cudaGetLastError();
    });
}

// band configuration (32 x 16 tiles, two pixels per thread), with the bias store for biased carver sessions
template <int B>
static cudaError_t launch_band(const DctcK1Args& a, int n_frames, bool uniform, cudaStream_t stream, const DctcK1Bias* bias, int dx)
{
    if (bias) return launch_tile<B, 32, 16, 2, true>(a, n_frames, uniform, stream, *bias, dx);
    return launch_tile<B, 32, 16, 2>(a, n_frames, uniform, stream, {}, dx);
}

cudaError_t dctc_launch_k1_tile(const DctcK1Args& a, int blocksize, int n_frames, bool uniform, cudaStream_t stream, const DctcK1Bias* bias,
                                int delta_x)
{
    if (a.w <= 0 || a.h <= 0 || n_frames <= 0) return cudaSuccess;
    if (n_frames > 65535 || (a.h + 31) / 32 > 65535) return cudaErrorInvalidConfiguration;
    if (a.seam) {
        // band mode (per-seam update): ~10 x 1080 pixels in all, so the launch is pure latency -- small tiles with two
        // pixels per thread keep the per-thread chain short (8 k1 x 2 instead of 8 k1 x 8 transforms for b = 8); the
        // arithmetic per pixel is the same as in the full-map configuration (bit-identical energies)
        switch (blocksize) {
        case 2: return launch_band<2>(a, n_frames, uniform, stream, bias, delta_x);
        case 4: return launch_band<4>(a, n_frames, uniform, stream, bias, delta_x);
        case 8: return launch_band<8>(a, n_frames, uniform, stream, bias, delta_x);
        case 16: return launch_band<16>(a, n_frames, uniform, stream, bias, delta_x);
        default: return cudaErrorInvalidValue;
        }
    }
    switch (blocksize) {
    case 2: return launch_tile<2, 64, 32, 8>(a, n_frames, uniform, stream);
    case 4: return launch_tile<4, 64, 32, 8>(a, n_frames, uniform, stream);
    case 8: return launch_tile<8, 64, 32, 8>(a, n_frames, uniform, stream);
    case 16: return launch_tile<16, DCTC_TILE16_TW, DCTC_TILE16_TH, DCTC_TILE16_P>(a, n_frames, uniform, stream);
    default: return cudaErrorInvalidValue;
    }
}

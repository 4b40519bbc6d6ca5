// K3: energy-image export (SURVEY section 8f rank 2).
//
// The plug-in's "output energy" option (src/render.c:175-202) asks liblqr for an 8-bit grey rendering of the energy
// map: lqr_carver_get_energy_image(carver, buf, orientation, LQR_COLDEPTH_8I, LQR_GREY_IMAGE) at src/render.c:191.
// liblqr compresses e -> 1/(1 + 1/e) (= e/(1+e); 0 for e = 0), min-max normalises to [0,1] in float and quantises by
// truncation, (guchar)(val * 255) as lqr_pixel_set_norm does for LQR_COLDEPTH_8I [liblqr 0.4.x lqr_energy.c /
// lqr_carver_rw.c, from memory: PARITY UNPINNED; restated in dct_carver_b200/host/dctc_lqr.c:
// dctc_lqr_carver_get_energy_image].  Two HBM-bound passes over the float plane:
// a min/max reduction of the compressed values (4 B/px read) and the scale + quantise pass (4 B/px read, 1 B/px
// written).  The FP32 operation order is the host's, so the bytes are identical.  When the map is sharded into row
// bands the (lo, hi) pair is what the ranks all-reduce (min, max) between the two passes.
#include <cstring>
#include "dctc_common.cuh"
#include "dctc_launch.h"

namespace {

// e >= 0 -> 1 / (1 + 1/e), IEEE divisions (1/0 = inf, 1/inf = 0): the same two roundings as the host carver
__device__ __forceinline__ float dctc_k3_compress(float e) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, __fdiv_rn(1.0f, e))); }

// compressed values are >= 0, so their bit patterns order like unsigned integers
__global__ void __launch_bounds__(256) dctc_minmax_kernel(const float* __restrict__ en, size_t pitch, int w, int h,
                                                          unsigned int* __restrict__ lo_hi)
{
    float lo = __int_as_float(0x7f800000), hi = 0.0f;
    for (int y = blockIdx.y; y < h; y += gridDim.y) {
        const float* row = en + (size_t) y * pitch;
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) {
            const float c = dctc_k3_compress(row[x]);
            lo = fminf(lo, c);
            hi = fmaxf(hi, c);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    __shared__ float slo[8], shi[8];
    if ((threadIdx.x & 31) == 0) { slo[threadIdx.x >> 5] = lo; shi[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x < 8) {
        lo = slo[threadIdx.x]; hi = shi[threadIdx.x];
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffu, hi, o));
        }
        if (threadIdx.x == 0) {
            atomicMin(lo_hi, __float_as_uint(lo));
            atomicMax(lo_hi + 1, __float_as_uint(hi));
        }
    }
}

__global__ void __launch_bounds__(256) dctc_energy_image_kernel(const float* __restrict__ en, size_t pitch, int w, int h,
                                                                const unsigned int* __restrict__ lo_hi_dev, float lo_arg, float hi_arg,
                                                                uint8_t* __restrict__ out, size_t out_pitch)
{
    const float lo = lo_hi_dev ? __uint_as_float(lo_hi_dev[0]) : lo_arg;
    const float hi = lo_hi_dev ? __uint_as_float(lo_hi_dev[1]) : hi_arg;
    const float span = hi - lo;
    for (int y = blockIdx.y; y < h; y += gridDim.y) {
        const float* row = en + (size_t) y * pitch;
        uint8_t* orow = out + (size_t) y * out_pitch;
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) {
            const float c = dctc_k3_compress(row[x]);
            // same FP32 operation order as the host carver: (c - lo) / span, then * 255, truncate
            orow[x] = hi > lo ? (uint8_t) __fmul_rn(__fdiv_rn(__fsub_rn(c, lo), span), 255.0f) : (uint8_t) 0;
        }
    }
}

dim3 plane_grid(int w, int h)
{
    int gx = (w + 255) / 256;
    if (gx > 64) gx = 64;
    int gy = h < 592 ? h : 592;
    return dim3((unsigned) gx, (unsigned) gy, 1);
}

}  // namespace

static int ensure_lohi(dctc_context* ctx)
{
    if (!ctx->k3_lohi) CK(ctx, cudaMalloc((void**) &ctx->k3_lohi, 2 * sizeof(unsigned int)));
    return DCTC_OK;
}

static int minmax_launch(dctc_context* ctx, const float* d_en, size_t pitch, int w, int h)
{
    const unsigned int init[2] = {0x7f800000u, 0u};
    CK(ctx, cudaMemcpyAsync(ctx->k3_lohi, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    dctc_minmax_kernel<<<plane_grid(w, h), 256, 0, ctx->stream>>>(d_en, pitch, w, h, ctx->k3_lohi);
    CK(ctx, cudaGetLastError());
    ctx->launches++;
    return DCTC_OK;
}

extern "C" {

int dctc_energy_minmax_dev(dctc_context* ctx, const float* d_en, size_t en_pitch, int w, int h, float* lo_hi)
{
    if (!ctx || !d_en || !lo_hi || w <= 0 || h <= 0 || en_pitch < (size_t) w) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_lohi(ctx);
    if (rc) return rc;
    rc = minmax_launch(ctx, d_en, en_pitch, w, h);
    if (rc) return rc;
    unsigned int v[2];
    CK(ctx, cudaMemcpyAsync(v, ctx->k3_lohi, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(lo_hi, v, sizeof(v));
    return DCTC_OK;
}

int dctc_energy_image_dev(dctc_context* ctx, const float* d_en, size_t en_pitch, int w, int h, const float* lo_hi,
                          uint8_t* d_out, size_t out_pitch, int sync)
{
    if (!ctx || !d_en || !d_out || w <= 0 || h <= 0 || en_pitch < (size_t) w || out_pitch < (size_t) w) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_lohi(ctx);
    if (rc) return rc;
    if (!lo_hi) {   // single device: both passes back to back, (lo, hi) never leave the GPU
        rc = minmax_launch(ctx, d_en, en_pitch, w, h);
        if (rc) return rc;
    }
    dctc_energy_image_kernel<<<plane_grid(w, h), 256, 0, ctx->stream>>>(d_en, en_pitch, w, h, lo_hi ? nullptr : ctx->k3_lohi,
                                                                       lo_hi ? lo_hi[0] : 0.0f, lo_hi ? lo_hi[1] : 0.0f, d_out, out_pitch);
    CK(ctx, cudaGetLastError());
    ctx->launches++;
    if (sync) CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_carver_energy_image(dctc_context* ctx, uint8_t* out)
{
    if (!ctx || !out) return DCTC_ERR_INVALID;
    if (!ctx->carver) return DCTC_ERR_STATE;
    CK(ctx, cudaSetDevice(ctx->device));
    const float* en;
    size_t en_pitch;
    int w, h;
    int rc = dctc_carver_energy_plane(ctx, &en, &en_pitch, &w, &h);   // in image orientation
    if (rc) return rc;
    const size_t need = (size_t) w * h;
    if (ctx->k3_img_cap < need) {
        if (ctx->k3_img) cudaFree(ctx->k3_img);
        ctx->k3_img = nullptr; ctx->k3_img_cap = 0;
        CK(ctx, cudaMalloc((void**) &ctx->k3_img, need));
        ctx->k3_img_cap = need;
    }
    rc = dctc_energy_image_dev(ctx, en, en_pitch, w, h, nullptr, ctx->k3_img, (size_t) w, 0);
    if (rc) return rc;
    CK(ctx, cudaMemcpyAsync(out, ctx->k3_img, need, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

}  // extern "C"

// ---- preview path (SURVEY section 8f rank 3) --------------------------------------------------------------------
// dct_energy_preview (src/render.c:421-501): the GIMP preview / "energy image" filter.  Per pixel the same operator
// with the preview window and BT.601 byte luminance (dct_energy_preview_rows, src/render.c:31-60; K1 tile kernel in
// preview mode), stored as gdouble (holding float values), then normalize_image (src/render.c:81-109):
// out = (guchar) ROUND(255 * ((e - min) / (max - min))) in double, replicated to every channel of the drawable.
namespace {

// energies are >= 0: float bit patterns order like unsigned integers
__global__ void __launch_bounds__(256) dctc_minmax_plain_kernel(const float* __restrict__ en, size_t pitch, int w, int h,
                                                                unsigned int* __restrict__ lo_hi)
{
    float lo = __int_as_float(0x7f800000), hi = 0.0f;
    for (int y = blockIdx.y; y < h; y += gridDim.y) {
        const float* row = en + (size_t) y * pitch;
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) {
            const float e = row[x];
            lo = fminf(lo, e);
            hi = fmaxf(hi, e);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(lo_hi, __float_as_uint(lo));
        atomicMax(lo_hi + 1, __float_as_uint(hi));
    }
}

__global__ void __launch_bounds__(256) dctc_preview_normalize_kernel(const float* __restrict__ en, size_t pitch, int w, int h,
                                                                     const unsigned int* __restrict__ lo_hi, int channels,
                                                                     uint8_t* __restrict__ out, size_t out_pitch)
{
    const double lo = (double) __uint_as_float(lo_hi[0]), hi = (double) __uint_as_float(lo_hi[1]);
    const double span = hi - lo;
    for (int y = blockIdx.y; y < h; y += gridDim.y) {
        const float* row = en + (size_t) y * pitch;
        uint8_t* orow = out + (size_t) y * out_pitch;
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < w; x += gridDim.x * blockDim.x) {
            // DOUBLE2GUCHAR (src/render.h:6) with ROUND(x) = (int)(x + 0.5); max == min gives 0/0 in the reference
            // (an undefined conversion that x86 turns into byte 0): we write 0
            const double t = __dadd_rn(__dmul_rn(255.0, __ddiv_rn(__dsub_rn((double) row[x], lo), span)), 0.5);
            const uint8_t v = span > 0.0 ? (uint8_t) (int) t : (uint8_t) 0;
            for (int c = 0; c < channels; c++) orow[(size_t) x * channels + c] = v;
        }
    }
}

}  // namespace

extern "C" int dctc_preview_energy(dctc_context* ctx, const uint8_t* img, int w, int h, int channels, size_t pitch,
                                   float* energy_out, uint8_t* image_out)
{
    if (!ctx || !img || w <= 0 || h <= 0 || pitch < (size_t) w * channels) return DCTC_ERR_INVALID;
    if (!(channels == 1 || channels == 3 || channels == 4)) return DCTC_ERR_INVALID;   // convert_row_to_luminance, src/render.c:62-79
    const int b = ctx->op.blocksize;
    if (!dctc_valid_blocksize(b)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_lohi(ctx);
    if (rc) return rc;
    const size_t d_pitch = ((size_t) w * channels + 15) & ~(size_t) 15;
    uint8_t *d_img = nullptr, *d_out = nullptr;
    float* d_en = nullptr;
    cudaError_t e = cudaMalloc((void**) &d_img, d_pitch * h);
    if (e == cudaSuccess) e = cudaMalloc((void**) &d_en, sizeof(float) * (size_t) w * h);
    if (e == cudaSuccess && image_out) e = cudaMalloc((void**) &d_out, (size_t) w * h * channels);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(d_img, d_pitch, img, pitch, (size_t) w * channels, h, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        DctcK1Args a;
        memset(&a, 0, sizeof(a));
        a.img = d_img; a.pitch = d_pitch; a.w = w; a.h = h; a.channels = channels;
        a.out = d_en; a.out_pitch = (size_t) w;
        a.preview = 1;
        // the preview operator works on 0..255 luminance bytes and applies the weights as they are (no 1/255)
        a.w_edges = ctx->op.edges; a.w_textures = ctx->op.textures;
        e = dctc_launch_k1_tile(a, b, 1, ctx->op.edges == ctx->op.textures, ctx->stream);
        if (e == cudaSuccess) ctx->launches++;
    }
    if (e == cudaSuccess && energy_out)
        e = cudaMemcpyAsync(energy_out, d_en, sizeof(float) * (size_t) w * h, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && image_out) {
        const unsigned int init[2] = {0x7f800000u, 0u};
        e = cudaMemcpyAsync(ctx->k3_lohi, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            dctc_minmax_plain_kernel<<<plane_grid(w, h), 256, 0, ctx->stream>>>(d_en, (size_t) w, w, h, ctx->k3_lohi);
            dctc_preview_normalize_kernel<<<plane_grid(w, h), 256, 0, ctx->stream>>>(d_en, (size_t) w, w, h, ctx->k3_lohi, channels, d_out,
                                                                                    (size_t) w * channels);
            e = cudaGetLastError();
            ctx->launches += 2;
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(image_out, d_out, (size_t) w * h * channels, cudaMemcpyDeviceToHost, ctx->stream);
    }
    cudaError_t es = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) e = es;
    if (d_img) cudaFree(d_img);
    if (d_en) cudaFree(d_en);
    if (d_out) cudaFree(d_out);
    if (e != cudaSuccess) return dctc_fail_cuda(ctx, e);
    return DCTC_OK;
}

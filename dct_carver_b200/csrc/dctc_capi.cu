// C ABI of the DCT-Carver energy hot path (see include/dctc.h for the reference interface each entry replaces).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include "dctc_common.cuh"
#include "dctc_launch.h"
#include "dctc_k1_select.h"

int dctc_fail_cuda(dctc_context* ctx, cudaError_t e)
{
    if (ctx) ctx->last_cuda = (int) e;
    if (e == cudaErrorMemoryAllocation) return DCTC_ERR_NOMEM;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return DCTC_ERR_NO_DEVICE;
    return DCTC_ERR_CUDA;
}

static int check_image(int w, int h, int channels, size_t pitch)
{
    if (w <= 0 || h <= 0) return DCTC_ERR_INVALID;
    if (channels < 1 || channels > 4) return DCTC_ERR_INVALID;
    if (pitch < (size_t) w * (size_t) channels) return DCTC_ERR_INVALID;
    return DCTC_OK;
}

extern "C" {

int dctc_version(void) { return DCTC_VERSION; }

const char* dctc_strerror(int status)
{
    switch (status) {
    case DCTC_OK: return "ok";
    case DCTC_ERR_INVALID: return "invalid argument";
    case DCTC_ERR_BLOCKSIZE: return "blocksize must be 2, 4, 8 or 16";
    case DCTC_ERR_NOMEM: return "out of device or pinned memory";
    case DCTC_ERR_CUDA: return "CUDA error (see dctc_last_cuda_error)";
    case DCTC_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case DCTC_ERR_STATE: return "carver session not loaded or seam out of range";
    case DCTC_ERR_UNSUPPORTED: return "kernel variant not available for this configuration";
    default: return "unknown status";
    }
}

int dctc_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return dctc_fail_cuda(nullptr, e);
    return n;
}

int dctc_create(dctc_context** out, int device)
{
    if (!out) return DCTC_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return DCTC_ERR_NO_DEVICE;
    if (device < 0 || device >= n) return DCTC_ERR_INVALID;
    dctc_context* ctx = new (std::nothrow) dctc_context();
    if (!ctx) return DCTC_ERR_NOMEM;
    ctx->device = device;
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc((void**) &ctx->tc_counters, DCTC_TC_COUNTERS * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(ctx->tc_counters, 0, DCTC_TC_COUNTERS * sizeof(int));   // the tensor-core kernel leaves its counter at 0
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_t0);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_t1);
    for (int i = 0; i < DCTC_SLOTS && e == cudaSuccess; i++) {
        e = cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_k[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_out[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        int rc = dctc_fail_cuda(nullptr, e);
        dctc_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return DCTC_OK;
}

void dctc_destroy(dctc_context* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->s_in) cudaStreamSynchronize(ctx->s_in);
    if (ctx->s_out) cudaStreamSynchronize(ctx->s_out);
    dctc_carver_release(ctx);
    for (int i = 0; i < DCTC_SLOTS; i++) {
        if (ctx->d_in[i]) cudaFree(ctx->d_in[i]);
        if (ctx->d_out[i]) cudaFree(ctx->d_out[i]);
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_k[i]) cudaEventDestroy(ctx->ev_k[i]);
        if (ctx->ev_out[i]) cudaEventDestroy(ctx->ev_out[i]);
    }
    if (ctx->tc_counters) cudaFree(ctx->tc_counters);
    if (ctx->k3_lohi) cudaFree(ctx->k3_lohi);
    if (ctx->k3_img) cudaFree(ctx->k3_img);
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    delete ctx;
}

int dctc_set_params(dctc_context* ctx, const DctcEnergyParameters* p)
{
    if (!ctx || !p) return DCTC_ERR_INVALID;
    if (!dctc_valid_blocksize(p->blocksize)) return DCTC_ERR_BLOCKSIZE;
    if (!(std::isfinite(p->edges) && std::isfinite(p->textures))) return DCTC_ERR_INVALID;
    const bool changed = ctx->op.edges != p->edges || ctx->op.textures != p->textures || ctx->op.blocksize != p->blocksize;
    ctx->op.edges = p->edges;
    ctx->op.textures = p->textures;
    ctx->op.blocksize = p->blocksize;
    ctx->mirror_valid = false;
    // a loaded carver session keeps its map in step with the operator (band radius, weights), like liblqr, whose
    // lqr_carver_set_energy_function (src/render.c:314-315) invalidates the energy map
    if (changed && ctx->carver) return dctc_carver_params_changed(ctx);
    return DCTC_OK;
}

int dctc_set_kernel(dctc_context* ctx, int kernel)
{
    if (!ctx) return DCTC_ERR_INVALID;
    if (kernel < DCTC_KERNEL_AUTO || kernel > DCTC_KERNEL_FP32_STREAM) return DCTC_ERR_INVALID;
    ctx->op.kernel = kernel;
    return DCTC_OK;
}

int dctc_last_cuda_error(const dctc_context* ctx) { return ctx ? ctx->last_cuda : 0; }
void* dctc_stream(dctc_context* ctx) { return ctx ? (void*) ctx->stream : nullptr; }
unsigned long long dctc_launch_count(const dctc_context* ctx) { return ctx ? ctx->launches : 0ull; }

}  // extern "C"

// ---- K1 dispatch ------------------------------------------------------------------------------------------

bool dctc_k1_fast_layout(const DctcK1Args& a)
{
    auto aligned16 = [](const void* p, size_t pitch) { return (((uintptr_t) p | pitch) & 15) == 0; };
    return (a.channels == 3 || a.channels == 1) && aligned16(a.img, a.pitch) && (a.frame_stride & 15) == 0 &&
           (!a.top || aligned16(a.top, a.top_pitch)) && (!a.bot || aligned16(a.bot, a.bot_pitch));
}

// The context supplies the device, the tensor-core counters and the launch counter; op the operator and kernel selection.
int dctc_run_k1(dctc_context* ctx, const DctcK1Op& op, DctcK1Args& a, int n_frames, cudaStream_t stream, const DctcK1Bias* bias,
                int delta_x)
{
    // E = max|T| * weight; the kernels keep luma in 0..255 units, so the 1/255 of liblqr's reader folds in here.
    a.w_edges = (float) ((double) op.edges / 255.0);
    a.w_textures = (float) ((double) op.textures / 255.0);
    const bool uniform = op.edges == op.textures;
    // every tensor-core launch takes its own work-item counter, so launches in flight on different streams never share one
    auto counter = [ctx] { return ctx->tc_counters + (ctx->tc_next++ % DCTC_TC_COUNTERS); };
    cudaError_t e = cudaSuccess;
    switch (dctc_k1_select(op.kernel, op.blocksize, a.seam != nullptr, a.preview != 0, dctc_k1_fast_layout(a))) {
    case DctcK1Variant::Tile: e = dctc_launch_k1_tile(a, op.blocksize, n_frames, uniform, stream, bias, delta_x); break;
    case DctcK1Variant::Small: e = dctc_launch_k1_small(a, op.blocksize, n_frames, uniform, ctx->sm_count, stream); break;
    case DctcK1Variant::March8: e = dctc_launch_k1_march8(a, n_frames, uniform, stream); break;
    case DctcK1Variant::Tc8: e = dctc_launch_k1_tc8(a, n_frames, uniform, counter(), ctx->sm_count, stream); break;
    case DctcK1Variant::Tc16: e = dctc_launch_k1_tc16(a, n_frames, uniform, counter(), ctx->sm_count, stream); break;
    }
    if (e != cudaSuccess) return dctc_fail_cuda(ctx, e);
    ctx->launches++;
    return DCTC_OK;
}

static void plain_args(DctcK1Args& a, const uint8_t* d_img, int w, int h, int channels, size_t pitch, float* d_out,
                       size_t out_pitch)
{
    memset(&a, 0, sizeof(a));
    a.img = d_img; a.pitch = pitch; a.w = w; a.h = h; a.channels = channels;
    a.out = d_out; a.out_pitch = out_pitch;
}

static int ensure_slot(dctc_context* ctx, int slot, size_t in_bytes, size_t out_bytes)
{
    if (ctx->d_in_cap[slot] < in_bytes) {
        if (ctx->d_in[slot]) cudaFree(ctx->d_in[slot]);
        ctx->d_in[slot] = nullptr; ctx->d_in_cap[slot] = 0;
        CK(ctx, cudaMalloc((void**) &ctx->d_in[slot], in_bytes));
        ctx->d_in_cap[slot] = in_bytes;
    }
    if (ctx->d_out_cap[slot] < out_bytes) {
        if (ctx->d_out[slot]) cudaFree(ctx->d_out[slot]);
        ctx->d_out[slot] = nullptr; ctx->d_out_cap[slot] = 0;
        CK(ctx, cudaMalloc((void**) &ctx->d_out[slot], out_bytes));
        ctx->d_out_cap[slot] = out_bytes;
    }
    return DCTC_OK;
}

extern "C" {

int dctc_energy_full_dev(dctc_context* ctx, const uint8_t* d_img, int w, int h, int channels, size_t pitch,
                         float* d_out, size_t out_pitch, int sync)
{
    return dctc_energy_batch_dev(ctx, d_img, 1, 0, w, h, channels, pitch, d_out, 0, out_pitch, sync);
}

int dctc_energy_batch_dev(dctc_context* ctx, const uint8_t* d_imgs, int n_frames, size_t frame_stride, int w, int h,
                          int channels, size_t pitch, float* d_out, size_t out_frame_stride, size_t out_pitch,
                          int sync)
{
    if (!ctx || !d_imgs || !d_out || n_frames <= 0) return DCTC_ERR_INVALID;
    int rc = check_image(w, h, channels, pitch);
    if (rc) return rc;
    if (out_pitch < (size_t) w) return DCTC_ERR_INVALID;
    if (!dctc_valid_blocksize(ctx->op.blocksize)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    // grid.z carries the frame index: split very large batches
    for (int f0 = 0; f0 < n_frames; f0 += 32768) {
        const int nf = n_frames - f0 < 32768 ? n_frames - f0 : 32768;
        DctcK1Args a;
        plain_args(a, d_imgs + (size_t) f0 * frame_stride, w, h, channels, pitch, d_out + (size_t) f0 * out_frame_stride,
                   out_pitch);
        a.frame_stride = frame_stride;
        a.out_frame_stride = out_frame_stride;
        rc = dctc_run_k1(ctx, ctx->op, a, nf, ctx->stream);
        if (rc) return rc;
    }
    if (sync) CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_energy_band_dev(dctc_context* ctx, const uint8_t* d_band, int w, int band_rows, int channels, size_t pitch,
                         const uint8_t* d_top, int top_rows, size_t top_pitch, const uint8_t* d_bot, int bot_rows,
                         size_t bot_pitch, float* d_out, size_t out_pitch, int sync)
{
    return dctc_energy_band_dev_at(ctx, d_band, w, band_rows, 0, channels, pitch, d_top, top_rows, top_pitch, d_bot, bot_rows, bot_pitch,
                                   d_out, out_pitch, sync);
}

int dctc_energy_band_dev_at(dctc_context* ctx, const uint8_t* d_band, int w, int band_rows, int band_y0, int channels, size_t pitch,
                            const uint8_t* d_top, int top_rows, size_t top_pitch, const uint8_t* d_bot, int bot_rows,
                            size_t bot_pitch, float* d_out, size_t out_pitch, int sync)
{
    if (!ctx || !d_band || !d_out || band_y0 < 0) return DCTC_ERR_INVALID;
    int rc = check_image(w, band_rows, channels, pitch);
    if (rc) return rc;
    if (out_pitch < (size_t) w || top_rows < 0 || bot_rows < 0) return DCTC_ERR_INVALID;
    if ((top_rows > 0 && (!d_top || top_pitch < (size_t) w * channels)) ||
        (bot_rows > 0 && (!d_bot || bot_pitch < (size_t) w * channels)))
        return DCTC_ERR_INVALID;
    if (!dctc_valid_blocksize(ctx->op.blocksize)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    DctcK1Args a;
    plain_args(a, d_band, w, band_rows, channels, pitch, d_out, out_pitch);
    a.top = d_top; a.top_rows = d_top ? top_rows : 0; a.top_pitch = top_pitch;
    a.bot = d_bot; a.bot_rows = d_bot ? bot_rows : 0; a.bot_pitch = bot_pitch;
    a.row_origin = band_y0;
    rc = dctc_run_k1(ctx, ctx->op, a, 1, ctx->stream);
    if (rc) return rc;
    if (sync) CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_energy_full(dctc_context* ctx, const uint8_t* img, int w, int h, int channels, size_t pitch, float* out)
{
    return dctc_energy_batch(ctx, img, 1, 0, w, h, channels, pitch, out, 0);
}

// Host buffers: frames stream through DCTC_SLOTS device slots; H2D, kernel and D2H of consecutive frames overlap
// on three streams (copies are truly asynchronous when the host buffers are pinned, e.g. dctc_host_alloc_pinned).
int dctc_energy_batch(dctc_context* ctx, const uint8_t* imgs, int n_frames, size_t frame_stride, int w, int h,
                      int channels, size_t pitch, float* out, size_t out_frame_stride)
{
    if (!ctx || !imgs || !out || n_frames <= 0) return DCTC_ERR_INVALID;
    int rc = check_image(w, h, channels, pitch);
    if (rc) return rc;
    if (n_frames > 1 && (frame_stride < pitch * (size_t) h || out_frame_stride < (size_t) w * h)) return DCTC_ERR_INVALID;
    if (!dctc_valid_blocksize(ctx->op.blocksize)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t row_bytes = (size_t) w * channels;
    const size_t d_pitch = (row_bytes + 15) & ~(size_t) 15;
    const size_t in_bytes = d_pitch * h, out_bytes = sizeof(float) * (size_t) w * h;
    const int slots = n_frames < DCTC_SLOTS ? n_frames : DCTC_SLOTS;
    for (int s = 0; s < slots; s++) {
        rc = ensure_slot(ctx, s, in_bytes, out_bytes);
        if (rc) return rc;
    }
    for (int f = 0; f < n_frames; f++) {
        const int s = f % DCTC_SLOTS;
        if (f >= DCTC_SLOTS) CK(ctx, cudaStreamWaitEvent(ctx->s_in, ctx->ev_k[s], 0));  // slot input consumed
        if (pitch == row_bytes && d_pitch == row_bytes)   // contiguous on both sides: one linear copy per frame
            CK(ctx, cudaMemcpyAsync(ctx->d_in[s], imgs + (size_t) f * frame_stride, row_bytes * (size_t) h, cudaMemcpyHostToDevice, ctx->s_in));
        else
            CK(ctx, cudaMemcpy2DAsync(ctx->d_in[s], d_pitch, imgs + (size_t) f * frame_stride, pitch, row_bytes, h,
                                      cudaMemcpyHostToDevice, ctx->s_in));
        CK(ctx, cudaEventRecord(ctx->ev_in[s], ctx->s_in));
        CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[s], 0));
        if (f >= DCTC_SLOTS) CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_out[s], 0));  // slot output drained
        DctcK1Args a;
        plain_args(a, ctx->d_in[s], w, h, channels, d_pitch, ctx->d_out[s], (size_t) w);
        rc = dctc_run_k1(ctx, ctx->op, a, 1, ctx->stream);
        if (rc) return rc;
        CK(ctx, cudaEventRecord(ctx->ev_k[s], ctx->stream));
        CK(ctx, cudaStreamWaitEvent(ctx->s_out, ctx->ev_k[s], 0));
        CK(ctx, cudaMemcpyAsync(out + (size_t) f * out_frame_stride, ctx->d_out[s], out_bytes, cudaMemcpyDeviceToHost,
                                ctx->s_out));
        CK(ctx, cudaEventRecord(ctx->ev_out[s], ctx->s_out));
    }
    CK(ctx, cudaStreamSynchronize(ctx->s_out));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

// ---- synthetic inputs, memory helpers, timing ----------------------------------------------------------------

int dctc_synth_fill_dev(dctc_context* ctx, uint8_t* d_img, int n_frames, size_t frame_stride, int w, int h,
                        int channels, size_t pitch, uint32_t seed, int pattern, int first_frame, int y_offset)
{
    if (!ctx || !d_img) return DCTC_ERR_INVALID;
    int rc = check_image(w, h, channels, pitch);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    for (int f0 = 0; f0 < n_frames; f0 += 32768) {
        const int nf = n_frames - f0 < 32768 ? n_frames - f0 : 32768;
        for (int y0 = 0; y0 < h; y0 += 32768) {
            const int nh = h - y0 < 32768 ? h - y0 : 32768;
            CK(ctx, dctc_launch_synth(d_img + (size_t) f0 * frame_stride + (size_t) y0 * pitch, nf, frame_stride, w, nh,
                                      channels, pitch, seed, pattern, first_frame + f0, y_offset + y0, ctx->stream));
            ctx->launches++;
        }
    }
    return DCTC_OK;
}

int dctc_ipc_export(dctc_context* ctx, void* d_ptr, unsigned char handle[DCTC_IPC_HANDLE_BYTES])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == DCTC_IPC_HANDLE_BYTES, "IPC handle size");
    if (!ctx || !d_ptr || !handle) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t hnd;
    CK(ctx, cudaIpcGetMemHandle(&hnd, d_ptr));
    memcpy(handle, &hnd, sizeof(hnd));
    return DCTC_OK;
}

int dctc_ipc_open(dctc_context* ctx, const unsigned char handle[DCTC_IPC_HANDLE_BYTES], void** d_peer_ptr)
{
    if (!ctx || !handle || !d_peer_ptr) return DCTC_ERR_INVALID;
    *d_peer_ptr = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, handle, sizeof(hnd));
    CK(ctx, cudaIpcOpenMemHandle(d_peer_ptr, hnd, cudaIpcMemLazyEnablePeerAccess));
    return DCTC_OK;
}

int dctc_ipc_close(dctc_context* ctx, void* d_peer_ptr)
{
    if (!ctx || !d_peer_ptr) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaIpcCloseMemHandle(d_peer_ptr));
    return DCTC_OK;
}

int dctc_dev_alloc(dctc_context* ctx, void** d_ptr, size_t bytes)
{
    if (!ctx || !d_ptr) return DCTC_ERR_INVALID;
    *d_ptr = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMalloc(d_ptr, bytes ? bytes : 1));
    return DCTC_OK;
}

int dctc_dev_free(dctc_context* ctx, void* d_ptr)
{
    if (!ctx) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaFree(d_ptr));
    return DCTC_OK;
}

int dctc_host_alloc_pinned(void** h_ptr, size_t bytes)
{
    if (!h_ptr) return DCTC_ERR_INVALID;
    *h_ptr = nullptr;
    cudaError_t e = cudaMallocHost(h_ptr, bytes ? bytes : 1);
    return e == cudaSuccess ? DCTC_OK : dctc_fail_cuda(nullptr, e);
}

int dctc_host_alloc_pinned_wc(void** h_ptr, size_t bytes)
{
    if (!h_ptr) return DCTC_ERR_INVALID;
    *h_ptr = nullptr;
    cudaError_t e = cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocWriteCombined);
    return e == cudaSuccess ? DCTC_OK : dctc_fail_cuda(nullptr, e);
}

int dctc_host_free_pinned(void* h_ptr)
{
    cudaError_t e = cudaFreeHost(h_ptr);
    return e == cudaSuccess ? DCTC_OK : dctc_fail_cuda(nullptr, e);
}

int dctc_memcpy_h2d(dctc_context* ctx, void* d_dst, const void* h_src, size_t bytes)
{
    if (!ctx || !d_dst || !h_src) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_memcpy_d2h(dctc_context* ctx, void* h_dst, const void* d_src, size_t bytes)
{
    if (!ctx || !h_dst || !d_src) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_memset_dev(dctc_context* ctx, void* d_ptr, int value, size_t bytes)
{
    if (!ctx || !d_ptr) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemsetAsync(d_ptr, value, bytes, ctx->stream));
    return DCTC_OK;
}

int dctc_sync(dctc_context* ctx)
{
    if (!ctx) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_timer_begin(dctc_context* ctx)
{
    if (!ctx) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaEventRecord(ctx->ev_t0, ctx->stream));
    return DCTC_OK;
}

int dctc_timer_end(dctc_context* ctx, float* ms)
{
    if (!ctx || !ms) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaEventRecord(ctx->ev_t1, ctx->stream));
    CK(ctx, cudaEventSynchronize(ctx->ev_t1));
    CK(ctx, cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return DCTC_OK;
}

}  // extern "C"

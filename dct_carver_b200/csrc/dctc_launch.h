// Internal: kernel launchers and the context layout shared by the C-ABI translation units.
#pragma once
#include <cuda.h>       // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, no libcuda link)
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <type_traits>
#include "../../include/dctc.h"

struct DctcK1Args;
struct DctcK1Bias;

#define CK(ctx, call)                                             \
    do {                                                          \
        cudaError_t e_ = (call);                                  \
        if (e_ != cudaSuccess) return dctc_fail_cuda((ctx), e_);  \
    } while (0)

inline bool dctc_valid_blocksize(int b) { return b == 2 || b == 4 || b == 8 || b == 16; }

// Runs f(std::integral_constant<bool, uniform>, std::integral_constant<int, C>) for the first C of the list equal to c
// (the last C when none is): one kernel instantiation per (uniform, C) pair, picked at run time.
template <int C, int... Cs, typename F>
static inline cudaError_t dctc_dispatch(bool uniform, int c, F&& f)
{
    if constexpr (sizeof...(Cs) > 0)
        if (c != C) return dctc_dispatch<Cs...>(uniform, c, f);
    if (uniform) return f(std::true_type(), std::integral_constant<int, C>());
    return f(std::false_type(), std::integral_constant<int, C>());
}

typedef CUresult (*DctcTensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                          const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                          CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// The driver's tensor-map encoder, or null when the driver has none.  Looked up once (thread-safe static initialisation:
// dctc_multi_* launches from one host thread per device).
inline DctcTensorMapEncodeFn dctc_tensor_map_encoder()
{
    static const DctcTensorMapEncodeFn encode = []() -> DctcTensorMapEncodeFn {
        void* fp = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qres) == cudaSuccess && fp &&
            qres == cudaDriverEntryPointSuccess)
            return (DctcTensorMapEncodeFn) fp;
        (void) cudaGetLastError();
        return nullptr;
    }();
    return encode;
}

// Programmatic dependent launch (the kernels of the device seam loop): a kernel launched with the attribute may be
// scheduled while its predecessor in the stream is still running; its CTAs then block in DCTC_PDL_PROLOGUE until the
// predecessor has completed and its memory operations are visible.  The macro is a no-op in a normal launch.
#ifdef DCTC_PDL_NO_EARLY
#define DCTC_PDL_PROLOGUE() asm volatile("griddepcontrol.wait;" ::: "memory")
#else
#define DCTC_PDL_PROLOGUE()                                                                                            \
    do {                                                                                                               \
        asm volatile("griddepcontrol.launch_dependents;");                                                            \
        asm volatile("griddepcontrol.wait;" ::: "memory");                                                            \
    } while (0)
#endif

template <typename... KArgs, typename... Args>
static inline cudaError_t dctc_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl,
                                          Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// bias (band mode only, may be null): the band store of a biased carver session.  delta_x (band mode only): the seam's
// largest step between two rows, which sets how many columns a tile row of the band can span.
cudaError_t dctc_launch_k1_tile(const DctcK1Args& a, int blocksize, int n_frames, bool uniform, cudaStream_t stream,
                                const DctcK1Bias* bias = nullptr, int delta_x = 1);
cudaError_t dctc_launch_k1_small(const DctcK1Args& a, int blocksize, int n_frames, bool uniform, int sm_count, cudaStream_t stream);
cudaError_t dctc_launch_k1_march8(const DctcK1Args& a, int n_frames, bool uniform, cudaStream_t stream);
cudaError_t dctc_launch_k1_tc8(const DctcK1Args& a, int n_frames, bool uniform, int* counter, int sm_count, cudaStream_t stream);
cudaError_t dctc_launch_k1_tc16(const DctcK1Args& a, int n_frames, bool uniform, int* counter, int sm_count, cudaStream_t stream);
cudaError_t dctc_launch_synth(uint8_t* d_img, int n_frames, size_t frame_stride, int w, int h, int channels,
                              size_t pitch, uint32_t seed, int pattern, int first_frame, int y_offset,
                              cudaStream_t stream);
// dst[frame][x][y] = src[frame][y][x] over cols x rows elements of esize (1..4) bytes per frame (dctc_transpose.cu)
cudaError_t dctc_launch_transpose(const void* src, size_t src_pitch, size_t src_fs, void* dst, size_t dst_pitch, size_t dst_fs,
                                  int cols, int rows, int n_frames, int esize, cudaStream_t stream);

constexpr int DCTC_SLOTS = 4;   // device staging slots of the host-buffer batch call (H2D, kernel and D2H of different frames overlap)
constexpr int DCTC_TC_COUNTERS = 64;
// Floats per row of dctc_carve_and_update's band buffers: the widest band, 2 r (delta_x + 1) with r = 16 / 2
constexpr int DCTC_BAND_ROW = 2 * 8 * (DCTC_MAX_DELTA_X + 1);

// The energy operator and the K1 kernel selection of a K1 launch (dctc_run_k1)
struct DctcK1Op {
    float edges = 0.5f, textures = 0.5f;  // defaults src/main.c:30-33
    int blocksize = 8;
    int kernel = DCTC_KERNEL_AUTO;
};

// A frame set of a carver session (dctc_carver_batch, dctc_k2_carver.cu): n frames of w x h pixels (w0 x h when filled),
// frame f of every plane at f times the plane's frame stride.  The session moves between its sets (the loaded frames,
// their transposes, the enlarged frames); the context's single session is a session with n = 1.
// transposed: the frames are the transposes of the images (a height operation runs the width seam loop on them), so w is
// the image height and h the image width.  Only the axis switch that fills such frames and the way out to the caller
// (frames_download, frames_oriented) look at the flag.
struct CarverFrames {
    int n = 0, w0 = 0, w = 0, h = 0, ch = 0;
    bool transposed = false;
    size_t pitch = 0, img_fs = 0;       // image: bytes per row, per frame
    size_t en_pitch = 0, m_pitch = 0;   // energy / cumulative planes: floats per row (multiple of 4: 16-byte aligned rows;
                                        // m_pitch >= DP_WIN), frames pitch * h floats apart
    uint8_t* img = nullptr;             // compacted in place per seam
    float* en = nullptr;
    float* m = nullptr;                 // cumulative map of the seam DP (rebuilt per seam, read back by the back-track)
    int8_t* dir = nullptr;              // jump planes of the parallel back-track: per 32-row block and bottom column, the
    size_t dir_fs = 0;                  // path's column offset at the block top
    int* seam = nullptr;                // n * h: the seam each frame is removing
    int* xlast = nullptr;               // n: last-row column of each frame's seam
    int* seam_log = nullptr;            // n * n_seams * h of the current seam loop, frame-major
    size_t seam_log_cap = 0;
    // visibility maps (lqr_carver_set_dump_vmaps, src/render.c:374): raw = original column of every current pixel,
    // vs = removal order of every original pixel (0 = never removed); vs_w x h ints per frame, only when requested
    int* raw = nullptr;
    int* vs = nullptr;
    int depth = 0;
    int vs_w = 0;                       // width of the frame the maps belong to (w0 when they were reset)
    void* scratch = nullptr;            // transposed frames: a plane in image orientation on its way out (4 * w0 * h bytes
                                        // per frame, allocated by the first use)
    // bias (dctc_carver_set_bias): one float per pixel, laid out like en and carved, transposed and inflated with the
    // pixels; null when the frames have none.  A biased set's en holds the seam energy en_op + bias / w0, and the
    // getters compute the operator map into en_op (allocated by their first use).
    float* bias = nullptr;
    float* en_op = nullptr;
};

struct dctc_context {
    int device = 0;
    cudaStream_t stream = nullptr;      // compute
    cudaStream_t s_in = nullptr;        // H2D
    cudaStream_t s_out = nullptr;       // D2H
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    cudaEvent_t ev_in[DCTC_SLOTS] = {}, ev_k[DCTC_SLOTS] = {}, ev_out[DCTC_SLOTS] = {};
    DctcK1Op op;                        // dctc_set_params, dctc_set_kernel
    int last_cuda = 0;
    unsigned long long launches = 0;
    int sm_count = 0;
    int* tc_counters = nullptr;         // work-item counters of the persistent tensor-core kernel (device)
    unsigned tc_next = 0;
    // staging slots of the host-buffer API
    uint8_t* d_in[DCTC_SLOTS] = {};
    float* d_out[DCTC_SLOTS] = {};
    size_t d_in_cap[DCTC_SLOTS] = {}, d_out_cap[DCTC_SLOTS] = {};
    // carver session (K2): a one-frame dctc_carver_batch, null when nothing is loaded; the state only the single session
    // has follows
    dctc_carver_batch* carver = nullptr;
    bool c_dump_vmaps = false;     // record the visibility map in the next seam loops (lqr_carver_set_dump_vmaps)
    int* c_band = nullptr;         // c_band[0]: 'rebuild the cumulative map from scratch' flag of the incremental seam DP, c_band[1]: rebuilds (device)
    bool c_incremental = false;    // device seam loop: update the cumulative map incrementally (dctc_carver_set_incremental)
    bool c_m_valid = false;        // the cumulative plane holds the map of the image before the last removal, compacted over that seam
    float c_rigidity = 0.0f;       // rigidity of the single session's seam loops (dctc_carver_set_rigidity); survives loads
    int c_delta_x = 1;             // seam step width of the single session's seam loops (dctc_carver_set_delta_x); survives loads
    float* c_band_vals = nullptr;  // packed band values of dctc_carve_and_update
    float* h_mirror = nullptr;     // host mirror of the energy map for dctc_pixel_energy (pinned, allocated by its first use)
    int* h_band = nullptr;         // pinned: band values (DCTC_BAND_ROW floats per row) and seam of dctc_carve_and_update
    bool mirror_valid = false;
    // K3 energy-image export
    unsigned int* k3_lohi = nullptr;   // device (min, max) of the compressed energies, as float bit patterns
    uint8_t* k3_img = nullptr;
    size_t k3_img_cap = 0;
};

int dctc_fail_cuda(dctc_context* ctx, cudaError_t e);
// Launches the one K1 kernel dctc_k1_select picks (dctc_k1_select.h); bias: band mode of a biased carver session (the
// tile kernel's bias store); delta_x: band mode, the seam's largest step (dctc_launch_k1_tile)
int dctc_run_k1(dctc_context* ctx, const DctcK1Op& op, DctcK1Args& a, int n_frames, cudaStream_t stream,
                const DctcK1Bias* bias = nullptr, int delta_x = 1);
// The layout the Small, Tc8 and Tc16 kernels (and the 1/3-channel variants of the march kernel) read: 1 or 3 channels,
// image rows, frames and halo rows 16-byte aligned
bool dctc_k1_fast_layout(const DctcK1Args& a);
void dctc_carver_release(dctc_context* ctx);
int dctc_carver_params_changed(dctc_context* ctx);   // rebuilds the resident energy map of a loaded carver session
// The single session's operator energy plane in image orientation (K3 energy image): device pointer, row pitch in floats, w x h
int dctc_carver_energy_plane(dctc_context* ctx, const float** en, size_t* en_pitch, int* w, int* h);

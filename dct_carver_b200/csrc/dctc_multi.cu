// Multi-GPU host layer of the energy path, in C++ behind the C ABI (include/dctc.h, section "multi-GPU").
//
// The path shards with a fixed halo and no data-path collective (SURVEY section 8e):
//   * frames (BASELINE config 4): frame f goes to device f mod G;
//   * row bands of one image (config 5): device g owns rows [h*g/G, h*(g+1)/G) and needs blocksize/2-1 rows from the
//     band above and blocksize/2 rows from the band below (window offsets -b/2+1 .. b/2, src/render.c:146-147; the
//     image's own edges replicate, src/render.c:122-132).  The halo rows are NOT exchanged: the K1 kernel of a band
//     reads them straight out of the neighbour's HBM over NVLink (d_top / d_bot of dctc_energy_band_dev point into
//     peer memory).
// Two deployments share the band code:
//   * one process drives all devices (dctc_multi_*): what a C caller like the plug-in's render() (src/render.c:310-315,
//     a single process) would use; peers are reached through cudaDeviceEnablePeerAccess, one host thread per device;
//   * one process per GPU (dctc_band_runner_*, bench.py under torchrun): the band buffers are exported as CUDA IPC
//     handles and exchanged through a POSIX shared-memory rendezvous implemented here (dctc_rendezvous_allgather), so
//     no framework is needed for the data path.
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <vector>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include "dctc_common.cuh"
#include "dctc_launch.h"

// ---- band geometry ----------------------------------------------------------------------------------------------

extern "C" int dctc_band_plan(int h, int world, int rank, int blocksize, int* y0, int* rows, int* top_need, int* bot_need)
{
    if (h <= 0 || world <= 0 || rank < 0 || rank >= world) return DCTC_ERR_INVALID;
    if (!dctc_valid_blocksize(blocksize)) return DCTC_ERR_BLOCKSIZE;
    const long long a = (long long) h * rank / world, z = (long long) h * (rank + 1) / world;
    const int tn = rank > 0 ? blocksize / 2 - 1 : 0, bn = rank < world - 1 ? blocksize / 2 : 0;
    if (y0) *y0 = (int) a;
    if (rows) *rows = (int) (z - a);
    if (top_need) *top_need = tn;
    if (bot_need) *bot_need = bn;
    // every band must be able to serve its neighbours' halos out of its own rows (a kernel reads at most one band away)
    const int need = blocksize / 2;
    for (int r = 0; r < world; r++) {
        const long long ra = (long long) h * r / world, rz = (long long) h * (r + 1) / world;
        if (world > 1 && rz - ra < need) return DCTC_ERR_INVALID;
    }
    return DCTC_OK;
}

// ---- rendezvous over POSIX shared memory ------------------------------------------------------------------------
// Segment layout: [u32 arrived[world]] [u32 left] [pad to 64] [world * bytes blobs].  A rank writes its blob, then
// publishes arrived[rank] = 1 (release); everybody waits for all flags (acquire) and copies the blobs.  The last rank
// to leave unlinks the name.  `name` must be unique per exchange (callers append a sequence number).

extern "C" int dctc_rendezvous_allgather(const char* name, int rank, int world, const void* mine, size_t bytes, void* all,
                                         int timeout_ms)
{
    if (!name || !*name || world <= 0 || rank < 0 || rank >= world || (bytes && (!mine || !all))) return DCTC_ERR_INVALID;
    if (world == 1) {
        if (bytes) memcpy(all, mine, bytes);
        return DCTC_OK;
    }
    char path[200];
    snprintf(path, sizeof(path), "/dctc_%.180s", name);
    for (char* p = path + 1; *p; p++)
        if (*p == '/') *p = '_';
    const size_t head = ((sizeof(uint32_t) * ((size_t) world + 1)) + 63) & ~(size_t) 63;
    const size_t total = head + bytes * (size_t) world;
    const int fd = shm_open(path, O_CREAT | O_RDWR, 0600);
    if (fd < 0) return DCTC_ERR_STATE;
    if (ftruncate(fd, (off_t) total) != 0) { close(fd); return DCTC_ERR_STATE; }   // same size from every rank; new pages are zero
    void* base = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (base == MAP_FAILED) return DCTC_ERR_STATE;
    auto* arrived = reinterpret_cast<std::atomic<uint32_t>*>(base);
    auto* left = arrived + world;
    uint8_t* blobs = reinterpret_cast<uint8_t*>(base) + head;
    if (bytes) memcpy(blobs + bytes * (size_t) rank, mine, bytes);
    arrived[rank].store(1u, std::memory_order_release);
    int rc = DCTC_OK;
    const auto t0 = std::chrono::steady_clock::now();
    for (int r = 0; r < world && rc == DCTC_OK; r++) {
        while (arrived[r].load(std::memory_order_acquire) == 0u) {
            if (timeout_ms > 0 && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(timeout_ms)) { rc = DCTC_ERR_STATE; break; }
            std::this_thread::sleep_for(std::chrono::microseconds(50));
        }
    }
    if (rc == DCTC_OK && bytes) memcpy(all, blobs, bytes * (size_t) world);
    if (left->fetch_add(1u, std::memory_order_acq_rel) + 1u == (uint32_t) world || rc != DCTC_OK) shm_unlink(path);
    munmap(base, total);
    return rc;
}

// ---- one band ----------------------------------------------------------------------------------------------------

struct DctcBand {
    dctc_context* ctx = nullptr;
    int w = 0, h = 0, ch = 0;            // whole image
    int y0 = 0, rows = 0, top_need = 0, bot_need = 0;
    size_t pitch = 0;                    // bytes, 16-byte multiple (same on every band so neighbours can address rows)
    uint8_t* d_band = nullptr;
    float* d_out = nullptr;
    uint8_t* d_img8 = nullptr;           // K3 output (lazy)
    const uint8_t* d_top = nullptr;      // first of the top_need rows above the band, in the neighbour's buffer
    const uint8_t* d_bot = nullptr;
    void* ipc_top = nullptr;             // IPC mappings to close (rank mode)
    void* ipc_bot = nullptr;
};

static size_t band_pitch(int w, int ch) { return ((size_t) w * ch + 15) & ~(size_t) 15; }

static int band_alloc(DctcBand& b, dctc_context* ctx, int w, int h, int ch, int rank, int world)
{
    b.ctx = ctx; b.w = w; b.h = h; b.ch = ch;
    int rc = dctc_band_plan(h, world, rank, ctx->op.blocksize, &b.y0, &b.rows, &b.top_need, &b.bot_need);
    if (rc) return rc;
    b.pitch = band_pitch(w, ch);
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMalloc((void**) &b.d_band, b.pitch * (size_t) b.rows));
    CK(ctx, cudaMalloc((void**) &b.d_out, sizeof(float) * (size_t) w * b.rows));
    return DCTC_OK;
}

static void band_free(DctcBand& b)
{
    if (!b.ctx) return;
    cudaSetDevice(b.ctx->device);
    cudaStreamSynchronize(b.ctx->stream);
    if (b.ipc_top) cudaIpcCloseMemHandle(b.ipc_top);
    if (b.ipc_bot) cudaIpcCloseMemHandle(b.ipc_bot);
    if (b.d_band) cudaFree(b.d_band);
    if (b.d_out) cudaFree(b.d_out);
    if (b.d_img8) cudaFree(b.d_img8);
    b = DctcBand();
}

static int band_synth(DctcBand& b, uint32_t seed, int pattern)
{
    // rows y0 .. y0+rows of the virtual image: y_offset keeps the bands consistent with a single-device fill
    int rc = dctc_synth_fill_dev(b.ctx, b.d_band, 1, 0, b.w, b.rows, b.ch, b.pitch, seed, pattern, 0, b.y0);
    if (rc) return rc;
    return dctc_sync(b.ctx);
}

static int band_upload(DctcBand& b, const uint8_t* rows_host, size_t host_pitch)
{
    CK(b.ctx, cudaSetDevice(b.ctx->device));
    CK(b.ctx, cudaMemcpy2DAsync(b.d_band, b.pitch, rows_host, host_pitch, (size_t) b.w * b.ch, b.rows, cudaMemcpyHostToDevice, b.ctx->stream));
    CK(b.ctx, cudaStreamSynchronize(b.ctx->stream));
    return DCTC_OK;
}

static int band_energy(DctcBand& b, int sync)
{
    return dctc_energy_band_dev_at(b.ctx, b.d_band, b.w, b.rows, b.y0, b.ch, b.pitch, b.d_top, b.d_top ? b.top_need : 0, b.pitch, b.d_bot,
                                   b.d_bot ? b.bot_need : 0, b.pitch, b.d_out, (size_t) b.w, sync);
}

static int band_download(DctcBand& b, float* out_rows)
{
    CK(b.ctx, cudaSetDevice(b.ctx->device));
    CK(b.ctx, cudaMemcpyAsync(out_rows, b.d_out, sizeof(float) * (size_t) b.w * b.rows, cudaMemcpyDeviceToHost, b.ctx->stream));
    CK(b.ctx, cudaStreamSynchronize(b.ctx->stream));
    return DCTC_OK;
}

static int band_image8(DctcBand& b, const float lo_hi[2], uint8_t* out_rows)
{
    CK(b.ctx, cudaSetDevice(b.ctx->device));
    if (!b.d_img8) CK(b.ctx, cudaMalloc((void**) &b.d_img8, (size_t) b.w * b.rows));
    int rc = dctc_energy_image_dev(b.ctx, b.d_out, (size_t) b.w, b.w, b.rows, lo_hi, b.d_img8, (size_t) b.w, 0);
    if (rc) return rc;
    CK(b.ctx, cudaMemcpyAsync(out_rows, b.d_img8, (size_t) b.w * b.rows, cudaMemcpyDeviceToHost, b.ctx->stream));
    CK(b.ctx, cudaStreamSynchronize(b.ctx->stream));
    return DCTC_OK;
}

// ---- one process per GPU: band runner ----------------------------------------------------------------------------

struct dctc_band_runner {
    DctcBand band;
    int rank = 0, world = 1;
    char name[160] = {0};
    unsigned seq = 0;
    bool connected = false;
};

struct BandBlob {
    unsigned char handle[DCTC_IPC_HANDLE_BYTES];
    int rows;
    int pad;
};

static int runner_exchange(dctc_band_runner* r, const void* mine, size_t bytes, void* all)
{
    char nm[200];
    snprintf(nm, sizeof(nm), "%s_%u", r->name, r->seq++);
    return dctc_rendezvous_allgather(nm, r->rank, r->world, mine, bytes, all, 120000);
}

extern "C" {

int dctc_band_runner_create(dctc_context* ctx, const char* rendezvous, int rank, int world, int w, int h, int channels,
                            dctc_band_runner** out)
{
    if (!ctx || !out || !rendezvous || w <= 0 || h <= 0 || channels < 1 || channels > 4) return DCTC_ERR_INVALID;
    *out = nullptr;
    dctc_band_runner* r = new (std::nothrow) dctc_band_runner();
    if (!r) return DCTC_ERR_NOMEM;
    r->rank = rank; r->world = world;
    snprintf(r->name, sizeof(r->name), "%.150s", rendezvous);
    int rc = band_alloc(r->band, ctx, w, h, channels, rank, world);
    if (rc) { band_free(r->band); delete r; return rc; }
    *out = r;
    return DCTC_OK;
}

int dctc_band_runner_geometry(const dctc_band_runner* r, int* y0, int* rows, size_t* pitch_bytes)
{
    if (!r) return DCTC_ERR_INVALID;
    if (y0) *y0 = r->band.y0;
    if (rows) *rows = r->band.rows;
    if (pitch_bytes) *pitch_bytes = r->band.pitch;
    return DCTC_OK;
}

void* dctc_band_runner_image_dev(dctc_band_runner* r) { return r ? r->band.d_band : nullptr; }
float* dctc_band_runner_energy_dev(dctc_band_runner* r) { return r ? r->band.d_out : nullptr; }

int dctc_band_runner_synth(dctc_band_runner* r, uint32_t seed, int pattern)
{
    if (!r) return DCTC_ERR_INVALID;
    return band_synth(r->band, seed, pattern);
}

int dctc_band_runner_upload(dctc_band_runner* r, const uint8_t* band_rows, size_t pitch_bytes)
{
    if (!r || !band_rows || pitch_bytes < (size_t) r->band.w * r->band.ch) return DCTC_ERR_INVALID;
    return band_upload(r->band, band_rows, pitch_bytes);
}

// Collective over the ranks of the rendezvous: publishes this rank's band buffer (which must hold its content by now:
// the exchange doubles as the barrier between "bands filled" and "neighbours may read") and maps the neighbours'.
int dctc_band_runner_connect(dctc_band_runner* r)
{
    if (!r) return DCTC_ERR_INVALID;
    DctcBand& b = r->band;
    if (r->connected) return DCTC_OK;
    BandBlob mine;
    memset(&mine, 0, sizeof(mine));
    mine.rows = b.rows;
    int rc = DCTC_OK;
    if (r->world > 1) rc = dctc_ipc_export(b.ctx, b.d_band, mine.handle);
    std::vector<BandBlob> all((size_t) r->world);
    // exchange even after a local failure (rows = -1) so that the other ranks do not wait for the timeout
    if (rc) mine.rows = -1;
    const int rx = runner_exchange(r, &mine, sizeof(mine), all.data());
    if (rc) return rc;
    if (rx) return rx;
    for (int i = 0; i < r->world; i++)
        if (all[(size_t) i].rows < 0) return DCTC_ERR_STATE;
    if (b.top_need > 0) {
        const BandBlob& nb = all[(size_t) r->rank - 1];
        if (nb.rows < b.top_need) return DCTC_ERR_INVALID;
        rc = dctc_ipc_open(b.ctx, nb.handle, &b.ipc_top);
        if (rc) return rc;
        b.d_top = (const uint8_t*) b.ipc_top + (size_t) (nb.rows - b.top_need) * b.pitch;
    }
    if (b.bot_need > 0) {
        const BandBlob& nb = all[(size_t) r->rank + 1];
        if (nb.rows < b.bot_need) return DCTC_ERR_INVALID;
        rc = dctc_ipc_open(b.ctx, nb.handle, &b.ipc_bot);
        if (rc) return rc;
        b.d_bot = (const uint8_t*) b.ipc_bot;
    }
    r->connected = true;
    return DCTC_OK;
}

// Barrier over the ranks (e.g. after re-filling the bands and before the next energy launch).
int dctc_band_runner_barrier(dctc_band_runner* r)
{
    if (!r) return DCTC_ERR_INVALID;
    int rc = dctc_sync(r->band.ctx);
    char z = 0;
    std::vector<char> all((size_t) r->world);
    const int rx = runner_exchange(r, &z, 1, all.data());
    return rc ? rc : rx;
}

int dctc_band_runner_energy(dctc_band_runner* r, int sync)
{
    if (!r) return DCTC_ERR_INVALID;
    if (r->world > 1 && !r->connected) return DCTC_ERR_STATE;
    return band_energy(r->band, sync);
}

int dctc_band_runner_download(dctc_band_runner* r, float* out_rows)
{
    if (!r || !out_rows) return DCTC_ERR_INVALID;
    return band_download(r->band, out_rows);
}

// K3 over a sharded map: per-band (min, max) of the compressed energies, all-gathered through the rendezvous and
// reduced on the host, then the 8-bit image of this rank's band.
int dctc_band_runner_energy_image(dctc_band_runner* r, uint8_t* out_rows)
{
    if (!r || !out_rows) return DCTC_ERR_INVALID;
    DctcBand& b = r->band;
    float lo_hi[2] = {0.0f, 0.0f};
    int rc = dctc_energy_minmax_dev(b.ctx, b.d_out, (size_t) b.w, b.w, b.rows, lo_hi);
    std::vector<float> all(2 * (size_t) r->world);
    if (rc) lo_hi[0] = lo_hi[1] = __builtin_nanf("");
    const int rx = runner_exchange(r, lo_hi, sizeof(lo_hi), all.data());
    if (rc) return rc;
    if (rx) return rx;
    for (int i = 0; i < r->world; i++) {
        if (all[2 * (size_t) i] != all[2 * (size_t) i]) return DCTC_ERR_STATE;
        lo_hi[0] = all[2 * (size_t) i] < lo_hi[0] ? all[2 * (size_t) i] : lo_hi[0];
        lo_hi[1] = all[2 * (size_t) i + 1] > lo_hi[1] ? all[2 * (size_t) i + 1] : lo_hi[1];
    }
    return band_image8(b, lo_hi, out_rows);
}

// Collective: no rank frees its band while a neighbour's kernel may still be reading it.
void dctc_band_runner_destroy(dctc_band_runner* r)
{
    if (!r) return;
    if (r->world > 1 && r->connected) dctc_band_runner_barrier(r);
    band_free(r->band);
    delete r;
}

}  // extern "C"

// ---- one process, all devices -----------------------------------------------------------------------------------

struct dctc_multi {
    std::vector<dctc_context*> ctx;
    std::vector<int> dev;
};

struct dctc_multi_bands {
    dctc_multi* m = nullptr;
    std::vector<DctcBand> bands;
};

template <typename F>
static int for_each_device(int n, F&& f)
{
    std::vector<int> rc((size_t) n, DCTC_OK);
    if (n == 1) {
        rc[0] = f(0);
    } else {
        std::vector<std::thread> th;
        th.reserve((size_t) n);
        for (int i = 0; i < n; i++) th.emplace_back([&rc, &f, i]() { rc[(size_t) i] = f(i); });
        for (auto& t : th) t.join();
    }
    for (int i = 0; i < n; i++)
        if (rc[(size_t) i]) return rc[(size_t) i];
    return DCTC_OK;
}

extern "C" {

int dctc_multi_create(dctc_multi** out, const int* devices, int n_devices)
{
    if (!out) return DCTC_ERR_INVALID;
    *out = nullptr;
    int visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible <= 0) return DCTC_ERR_NO_DEVICE;
    if (!devices) n_devices = visible;
    if (n_devices <= 0 || n_devices > 64) return DCTC_ERR_INVALID;
    dctc_multi* m = new (std::nothrow) dctc_multi();
    if (!m) return DCTC_ERR_NOMEM;
    for (int i = 0; i < n_devices; i++) {
        const int d = devices ? devices[i] : i;
        dctc_context* c = nullptr;
        const int rc = dctc_create(&c, d);
        if (rc) { dctc_multi_destroy(m); return rc; }
        m->ctx.push_back(c);
        m->dev.push_back(d);
    }
    // neighbours read each other's band buffers: enable peer access between every pair of distinct devices
    for (int i = 0; i < n_devices; i++) {
        for (int j = 0; j < n_devices; j++) {
            if (m->dev[(size_t) i] == m->dev[(size_t) j]) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, m->dev[(size_t) i], m->dev[(size_t) j]) != cudaSuccess || !can) { dctc_multi_destroy(m); return DCTC_ERR_UNSUPPORTED; }
            cudaSetDevice(m->dev[(size_t) i]);
            const cudaError_t e = cudaDeviceEnablePeerAccess(m->dev[(size_t) j], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { dctc_multi_destroy(m); return dctc_fail_cuda(nullptr, e); }
            (void) cudaGetLastError();
        }
    }
    *out = m;
    return DCTC_OK;
}

void dctc_multi_destroy(dctc_multi* m)
{
    if (!m) return;
    for (dctc_context* c : m->ctx) dctc_destroy(c);
    delete m;
}

int dctc_multi_device_count(const dctc_multi* m) { return m ? (int) m->ctx.size() : 0; }
dctc_context* dctc_multi_context(dctc_multi* m, int i) { return (m && i >= 0 && i < (int) m->ctx.size()) ? m->ctx[(size_t) i] : nullptr; }

int dctc_multi_set_params(dctc_multi* m, const DctcEnergyParameters* p)
{
    if (!m) return DCTC_ERR_INVALID;
    for (dctc_context* c : m->ctx) {
        const int rc = dctc_set_params(c, p);
        if (rc) return rc;
    }
    return DCTC_OK;
}

int dctc_multi_set_kernel(dctc_multi* m, int kernel)
{
    if (!m) return DCTC_ERR_INVALID;
    for (dctc_context* c : m->ctx) {
        const int rc = dctc_set_kernel(c, kernel);
        if (rc) return rc;
    }
    return DCTC_OK;
}

unsigned long long dctc_multi_launch_count(const dctc_multi* m)
{
    unsigned long long n = 0;
    if (m) for (dctc_context* c : m->ctx) n += dctc_launch_count(c);
    return n;
}

// Host buffers, frame f -> device f mod G (SURVEY section 8e, config 4); every device streams its frames through its
// own H2D / kernel / D2H pipeline (dctc_energy_batch), one host thread per device.
int dctc_multi_energy_batch(dctc_multi* m, const uint8_t* imgs, int n_frames, size_t frame_stride, int w, int h, int channels,
                            size_t pitch, float* out, size_t out_frame_stride)
{
    if (!m || !imgs || !out || n_frames <= 0) return DCTC_ERR_INVALID;
    if (n_frames > 1 && (frame_stride < pitch * (size_t) h || out_frame_stride < (size_t) w * h)) return DCTC_ERR_INVALID;
    const int G = (int) m->ctx.size();
    return for_each_device(G, [&](int g) -> int {
        const int mine = (n_frames - g + G - 1) / G;      // frames g, g+G, g+2G, ...
        if (mine <= 0) return DCTC_OK;
        return dctc_energy_batch(m->ctx[(size_t) g], imgs + (size_t) g * frame_stride, mine, frame_stride * (size_t) G, w, h, channels, pitch,
                                 out + (size_t) g * out_frame_stride, out_frame_stride * (size_t) G);
    });
}

int dctc_multi_bands_create(dctc_multi* m, int w, int h, int channels, dctc_multi_bands** out)
{
    if (!m || !out || w <= 0 || h <= 0 || channels < 1 || channels > 4) return DCTC_ERR_INVALID;
    *out = nullptr;
    dctc_multi_bands* b = new (std::nothrow) dctc_multi_bands();
    if (!b) return DCTC_ERR_NOMEM;
    b->m = m;
    const int G = (int) m->ctx.size();
    b->bands.resize((size_t) G);
    for (int g = 0; g < G; g++) {
        const int rc = band_alloc(b->bands[(size_t) g], m->ctx[(size_t) g], w, h, channels, g, G);
        if (rc) { dctc_multi_bands_destroy(b); return rc; }
    }
    // halo pointers straight into the neighbours' band buffers (peer access was enabled by dctc_multi_create)
    for (int g = 0; g < G; g++) {
        DctcBand& x = b->bands[(size_t) g];
        if (x.top_need > 0) {
            const DctcBand& up = b->bands[(size_t) g - 1];
            x.d_top = up.d_band + (size_t) (up.rows - x.top_need) * up.pitch;
        }
        if (x.bot_need > 0) x.d_bot = b->bands[(size_t) g + 1].d_band;
    }
    *out = b;
    return DCTC_OK;
}

void dctc_multi_bands_destroy(dctc_multi_bands* b)
{
    if (!b) return;
    for (DctcBand& x : b->bands)
        if (x.ctx) { cudaSetDevice(x.ctx->device); cudaStreamSynchronize(x.ctx->stream); }   // nobody reads a peer any more
    for (DctcBand& x : b->bands) band_free(x);
    delete b;
}

int dctc_multi_bands_geometry(const dctc_multi_bands* b, int g, int* y0, int* rows)
{
    if (!b || g < 0 || g >= (int) b->bands.size()) return DCTC_ERR_INVALID;
    if (y0) *y0 = b->bands[(size_t) g].y0;
    if (rows) *rows = b->bands[(size_t) g].rows;
    return DCTC_OK;
}

int dctc_multi_bands_synth(dctc_multi_bands* b, uint32_t seed, int pattern)
{
    if (!b) return DCTC_ERR_INVALID;
    return for_each_device((int) b->bands.size(), [&](int g) { return band_synth(b->bands[(size_t) g], seed, pattern); });
}

int dctc_multi_bands_upload(dctc_multi_bands* b, const uint8_t* img, size_t pitch)
{
    if (!b || !img || b->bands.empty() || pitch < (size_t) b->bands[0].w * b->bands[0].ch) return DCTC_ERR_INVALID;
    return for_each_device((int) b->bands.size(), [&](int g) {
        DctcBand& x = b->bands[(size_t) g];
        return band_upload(x, img + (size_t) x.y0 * pitch, pitch);
    });
}

// Launches K1 on every band (each on its own device and stream); with sync != 0 returns after all have finished.
// All bands must hold their content (upload / synth return synchronised).
int dctc_multi_bands_energy(dctc_multi_bands* b, int sync)
{
    if (!b) return DCTC_ERR_INVALID;
    for (DctcBand& x : b->bands) {
        const int rc = band_energy(x, 0);
        if (rc) return rc;
    }
    if (sync)
        for (DctcBand& x : b->bands) {
            const int rc = dctc_sync(x.ctx);
            if (rc) return rc;
        }
    return DCTC_OK;
}

int dctc_multi_bands_download(dctc_multi_bands* b, float* out)
{
    if (!b || !out) return DCTC_ERR_INVALID;
    return for_each_device((int) b->bands.size(), [&](int g) {
        DctcBand& x = b->bands[(size_t) g];
        return band_download(x, out + (size_t) x.y0 * x.w);
    });
}

// K3 over the sharded map: per-band min/max -> host reduction -> per-band scale + quantise (src/render.c:191).
int dctc_multi_bands_energy_image(dctc_multi_bands* b, uint8_t* out)
{
    if (!b || !out) return DCTC_ERR_INVALID;
    const int G = (int) b->bands.size();
    std::vector<float> mm(2 * (size_t) G);
    int rc = for_each_device(G, [&](int g) {
        DctcBand& x = b->bands[(size_t) g];
        return dctc_energy_minmax_dev(x.ctx, x.d_out, (size_t) x.w, x.w, x.rows, &mm[2 * (size_t) g]);
    });
    if (rc) return rc;
    float lo_hi[2] = {mm[0], mm[1]};
    for (int g = 1; g < G; g++) {
        lo_hi[0] = mm[2 * (size_t) g] < lo_hi[0] ? mm[2 * (size_t) g] : lo_hi[0];
        lo_hi[1] = mm[2 * (size_t) g + 1] > lo_hi[1] ? mm[2 * (size_t) g + 1] : lo_hi[1];
    }
    return for_each_device(G, [&](int g) {
        DctcBand& x = b->bands[(size_t) g];
        return band_image8(x, lo_hi, out + (size_t) x.y0 * x.w);
    });
}

// One host image -> row bands over the devices -> host energy map (and optionally the 8-bit energy image).
int dctc_multi_energy_bands(dctc_multi* m, const uint8_t* img, int w, int h, int channels, size_t pitch, float* out, uint8_t* image_out)
{
    if (!m || !img || (!out && !image_out)) return DCTC_ERR_INVALID;
    if (pitch < (size_t) w * channels) return DCTC_ERR_INVALID;
    dctc_multi_bands* b = nullptr;
    int rc = dctc_multi_bands_create(m, w, h, channels, &b);
    if (rc) return rc;
    rc = dctc_multi_bands_upload(b, img, pitch);
    if (!rc) rc = dctc_multi_bands_energy(b, 1);
    if (!rc && out) rc = dctc_multi_bands_download(b, out);
    if (!rc && image_out) rc = dctc_multi_bands_energy_image(b, image_out);
    dctc_multi_bands_destroy(b);
    return rc;
}

// ---- PCIe probe (bench.py: the ceiling of the host-buffer path) ------------------------------------------------
// Pinned host <-> device copies of `bytes` bytes, `iters` times: H2D alone, D2H alone, both directions at once on two
// streams.  Results in GB/s (10^9 bytes per second), the third one per direction.
int dctc_pcie_probe(dctc_context* ctx, size_t bytes, int iters, double* h2d_gbs, double* d2h_gbs, double* bidir_gbs_per_dir)
{
    if (!ctx || bytes == 0 || iters <= 0) return DCTC_ERR_INVALID;
    CK(ctx, cudaSetDevice(ctx->device));
    void *h0 = nullptr, *h1 = nullptr, *d0 = nullptr, *d1 = nullptr;
    cudaError_t e = cudaMallocHost(&h0, bytes);
    if (e == cudaSuccess) e = cudaMallocHost(&h1, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d0, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d1, bytes);
    if (e == cudaSuccess) { memset(h0, 1, bytes); memset(h1, 2, bytes); }
    auto run = [&](int mode, double* gbs) {
        if (e != cudaSuccess) return;
        for (int it = -1; it < iters; it++) {   // one warm-up round
            if (it == 0) {
                cudaStreamSynchronize(ctx->s_in); cudaStreamSynchronize(ctx->s_out);
            }
            if (it == 0) e = cudaEventRecord(ctx->ev_t0, ctx->s_in);
            if (it == 0 && e == cudaSuccess && mode == 2) e = cudaStreamWaitEvent(ctx->s_out, ctx->ev_t0, 0);
            if (e == cudaSuccess && (mode == 0 || mode == 2)) e = cudaMemcpyAsync(d0, h0, bytes, cudaMemcpyHostToDevice, ctx->s_in);
            if (e == cudaSuccess && (mode == 1 || mode == 2)) e = cudaMemcpyAsync(h1, d1, bytes, cudaMemcpyDeviceToHost, mode == 2 ? ctx->s_out : ctx->s_in);
            if (e != cudaSuccess) return;
        }
        if (mode == 2) {
            e = cudaEventRecord(ctx->ev_out[0], ctx->s_out);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->s_in, ctx->ev_out[0], 0);
        }
        if (e == cudaSuccess) e = cudaEventRecord(ctx->ev_t1, ctx->s_in);
        if (e == cudaSuccess) e = cudaEventSynchronize(ctx->ev_t1);
        float ms = 0.0f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1);
        if (e == cudaSuccess && gbs) *gbs = (double) bytes * iters / ((double) ms * 1e-3) / 1e9;
    };
    run(0, h2d_gbs);
    run(1, d2h_gbs);
    run(2, bidir_gbs_per_dir);
    if (h0) cudaFreeHost(h0);
    if (h1) cudaFreeHost(h1);
    if (d0) cudaFree(d0);
    if (d1) cudaFree(d1);
    if (e != cudaSuccess) return dctc_fail_cuda(ctx, e);
    return DCTC_OK;
}

}  // extern "C"

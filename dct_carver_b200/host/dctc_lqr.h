/* dctc_lqr.h — host-side carver: the subset of LiquidRescale (liblqr) that dct-carver's render.c drives,
 * with the energy coming from the GPU through batch hooks instead of one callback per pixel.
 *
 * liblqr itself (lqr-1, configure.in:64-67) is an external dependency that is neither in the reference tree nor
 * installed here, so this restates the behaviour the reference relies on [liblqr 0.4.x, from memory; SURVEY
 * Appendix A]: seams of width 1, delta_x = 1, rigidity 0 (src/render.c:313), cumulative map
 *   m[y][x] = en[y][x] + min(m[y-1][x-1], m[y-1][x], m[y-1][x+1])      (first strict minimum, left to right)
 * (dctc_lqr_carver_init also takes other delta_x and a rigidity: see dctc_render_ext)
 * seam end = leftmost minimum of the last row, energy update after each seam only within +-radius of it.
 * Call sites mirrored: src/render.c:312-316 (new/init/set_energy_function), :377 (resize), :264-269 (scan_line),
 * :214-231 (vmap), :413 (destroy).
 *
 * Two energy sources:
 *   - dctc_lqr_carver_attach_gpu(): build_emap -> dctc_carver_load + dctc_carver_energy,
 *                                   update_emap -> dctc_carve_and_update (K2).  This is the product path.
 *   - a per-pixel LqrEnergyFunc callback with a reading window, exactly liblqr's contract; used to plug the
 *     reference's own dct_pixel_energy in for seam-parity checks.
 * Define DCTC_LQR_COMPAT_NAMES before including to get the lqr_* names render.c uses.
 */
#ifndef DCTC_LQR_H
#define DCTC_LQR_H

#include <stdint.h>
#include "../../include/dctc.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct DctcLqrCarver_ DctcLqrCarver;

/* Reading window handed to the callback.  Only offsets within +-radius and inside the image are defined
 * (liblqr returns 0 outside); the reference clamps before reading (src/render.c:148-149). */
typedef struct DctcLqrReadingWindow_ {
    const double *luma; /* current w*h luma plane (LQR_ER_LUMA), row pitch = w */
    int w, h, x, y, radius;
} DctcLqrReadingWindow;

typedef float (*DctcLqrEnergyFunc)(int x, int y, int w, int h, DctcLqrReadingWindow *rw, void *extra_data);

enum { DCTC_LQR_OK = 0, DCTC_LQR_ERROR = 1, DCTC_LQR_NOMEM = 2 };
enum { DCTC_LQR_ER_BRIGHTNESS = 0, DCTC_LQR_ER_LUMA = 1 };

/* takes ownership of `buffer` (malloc'ed, w*h*channels bytes), like lqr_carver_new */
DctcLqrCarver *dctc_lqr_carver_new(uint8_t *buffer, int width, int height, int channels);
int dctc_lqr_carver_init(DctcLqrCarver *r, int delta_x, float rigidity);
int dctc_lqr_carver_set_energy_function(DctcLqrCarver *r, DctcLqrEnergyFunc f, int radius, int reader_type, void *extra);
int dctc_lqr_carver_attach_gpu(DctcLqrCarver *r, dctc_context *gpu);
void dctc_lqr_carver_set_dump_vmaps(DctcLqrCarver *r);
int dctc_lqr_carver_resize(DctcLqrCarver *r, int w1, int h1);
void dctc_lqr_carver_destroy(DctcLqrCarver *r);

int dctc_lqr_carver_get_width(const DctcLqrCarver *r);
int dctc_lqr_carver_get_height(const DctcLqrCarver *r);
int dctc_lqr_carver_get_channels(const DctcLqrCarver *r);
int dctc_lqr_carver_scan_by_row(const DctcLqrCarver *r);
void dctc_lqr_carver_scan_reset(DctcLqrCarver *r);
/* iterates the current image line by line (rows, or columns while transposed); returns 0 at the end */
int dctc_lqr_carver_scan_line(DctcLqrCarver *r, int *n, uint8_t **rgb);

/* current energy map (w*h floats, building it if needed) — lqr_carver_get_energy */
int dctc_lqr_carver_get_energy(DctcLqrCarver *r, float *buffer);
/* 8-bit grey energy image as lqr_carver_get_energy_image(.., LQR_COLDEPTH_8I, LQR_GREY_IMAGE) (src/render.c:191):
 * e -> 1/(1+1/e), min-max normalised, (uint8_t)(val*255) [liblqr, from memory] */
int dctc_lqr_carver_get_energy_image(DctcLqrCarver *r, uint8_t *buffer);
/* visibility map over the ORIGINAL w0*h0 frame: 0 = never carved, k = removed by the k-th seam (src/render.c:214-231) */
const int *dctc_lqr_carver_vmap(const DctcLqrCarver *r, int *w0, int *h0, int *depth);
/* removed column per row for every seam, in the coordinates at removal time: n_seams * h entries */
const int *dctc_lqr_carver_seams(const DctcLqrCarver *r, int *n_seams, int *seam_len);
/* per-phase wall time in seconds: [0] energy (build+update), [1] cumulative map, [2] seam search+carve */
const double *dctc_lqr_carver_timing(const DctcLqrCarver *r);

double dctc_lqr_rwindow_read(DctcLqrReadingWindow *rw, int x, int y, int channel);
int dctc_lqr_rwindow_get_radius(DctcLqrReadingWindow *rw);

/* ---- render.c-like glue (src/render.c:286-325 init_carver_from_vals, :327-419 render), GIMP-free ---- */
typedef struct DctcPlugInVals_ { /* src/main.h:12-22 */
    float edges;
    float textures;
    int blocksize;
    int seams_number; /* new size = old + seams_number along the chosen axis (src/render.c:357-363) */
    int new_layer, resize_canvas, output_energy, output_seams, vertically;
} DctcPlugInVals;

typedef struct DctcRenderResult_ {
    uint8_t *image;        /* malloc'ed, new_w*new_h*channels */
    int new_w, new_h, channels;
    uint8_t *energy_image; /* malloc'ed w*h grey, when output_energy */
    int *vmap;             /* malloc'ed w*h, when output_seams */
    int vmap_depth;
    int *seams;            /* malloc'ed n_seams*seam_len */
    int n_seams, seam_len;
    double t_energy, t_mmap, t_seam, t_total;
} DctcRenderResult;

/* gpu == NULL is refused (no CPU fallback in the product); cb != NULL selects the per-pixel callback source
 * instead (checker use: plug in the reference's dct_pixel_energy).  The plug-in's carver: delta_x 1, rigidity 0
 * (src/render.c:313), i.e. dctc_render_ext(.., 1, 0, ..). */
int dctc_render(const uint8_t *img, int w, int h, int channels, const DctcPlugInVals *vals, dctc_context *gpu,
                DctcLqrEnergyFunc cb, void *cb_extra, DctcRenderResult *res);
/* dctc_render with lqr_carver_init(carver, delta_x, rigidity): a seam step of |d| <= delta_x columns costs
 * fl(fl(rigidity * |d|^1.5) / h) more, h the seam length.  With a GPU attached, delta_x 1 .. DCTC_MAX_DELTA_X runs the
 * device seam loop (the context's dctc_carver_set_rigidity and dctc_carver_set_delta_x are set before each load); larger
 * delta_x run the host loop, whose band updates (dctc_carve_and_update) then refuse steps wider than 1.  Both context
 * options keep the render's values after it returns (delta_x 1 above DCTC_MAX_DELTA_X): a caller that shares the context
 * and relies on other values sets them again.
 * DCTC_ERR_INVALID also for delta_x < 1 and a negative or non-finite rigidity. */
int dctc_render_ext(const uint8_t *img, int w, int h, int channels, const DctcPlugInVals *vals, int delta_x, float rigidity,
                    dctc_context *gpu, DctcLqrEnergyFunc cb, void *cb_extra, DctcRenderResult *res);
void dctc_render_result_free(DctcRenderResult *res);

#ifdef DCTC_LQR_COMPAT_NAMES
typedef DctcLqrCarver LqrCarver;
typedef DctcLqrReadingWindow LqrReadingWindow;
typedef DctcLqrEnergyFunc LqrEnergyFunc;
#define LQR_ER_LUMA DCTC_LQR_ER_LUMA
#define lqr_carver_new dctc_lqr_carver_new
#define lqr_carver_init dctc_lqr_carver_init
#define lqr_carver_set_energy_function dctc_lqr_carver_set_energy_function
#define lqr_carver_set_dump_vmaps dctc_lqr_carver_set_dump_vmaps
#define lqr_carver_resize dctc_lqr_carver_resize
#define lqr_carver_destroy dctc_lqr_carver_destroy
#define lqr_carver_get_width dctc_lqr_carver_get_width
#define lqr_carver_get_height dctc_lqr_carver_get_height
#define lqr_carver_scan_by_row dctc_lqr_carver_scan_by_row
#define lqr_carver_scan_line dctc_lqr_carver_scan_line
#define lqr_rwindow_read dctc_lqr_rwindow_read
#define lqr_rwindow_get_radius dctc_lqr_rwindow_get_radius
#endif

#ifdef __cplusplus
}
#endif
/* Process-wide switch: hand the seam loop of dctc_lqr_carver_resize to the device (default) or keep the host loop
 * with GPU energy batches (cross-check, and automatic fallback for widths the device kernel does not cover). */
void dctc_host_set_device_seam_loop(int on);
int dctc_host_get_device_seam_loop(void);

#endif

/* dctc.h — C ABI of the B200-native DCT-Carver energy hot path.
 *
 * This is the drop-in boundary for ONE path of avivrosenberg/dct-carver: the per-pixel block-DCT energy
 * map that the plug-in registers with liblqr as a custom energy function.  Every entry point names the
 * reference interface it replaces (paths relative to the reference tree).  Plain C: pointers and sizes
 * only, no C++/torch types.  All compute runs in hand-written CUDA kernels for sm_100a
 * (dct_carver_b200/csrc); there is NO CPU fallback: without a CUDA device every compute call returns
 * DCTC_ERR_NO_DEVICE / DCTC_ERR_CUDA.
 *
 * Threading: one caller per context (the reference's callback is single-threaded and non re-entrant,
 * src/render.c:140,154).  Use one context per GPU / stream.
 */
#ifndef DCTC_H
#define DCTC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCTC_VERSION 1

/* status codes (the reference has no error channel: bad blocksize -> error()+untransformed data,
 * src/dct.c:89-92; OOM -> exit(1), src/fft2d/alloc.c:5-10.  Here every batch call returns int.) */
enum {
    DCTC_OK = 0,
    DCTC_ERR_INVALID = -1,    /* NULL pointer, non-positive size, channels not in 1..4, pitch too small */
    DCTC_ERR_BLOCKSIZE = -2,  /* blocksize not in {2,4,8,16}  (src/dct.c:77-93, UI combo src/interface.c:281) */
    DCTC_ERR_NOMEM = -3,      /* cudaMalloc / cudaMallocHost failed */
    DCTC_ERR_CUDA = -4,       /* a CUDA call failed; see dctc_last_cuda_error() */
    DCTC_ERR_NO_DEVICE = -5,  /* no usable CUDA device */
    DCTC_ERR_STATE = -6,      /* carver call without a loaded image / seam outside the current width */
    DCTC_ERR_UNSUPPORTED = -7 /* requested kernel variant does not exist for this block size */
};

/* The reference's operator state, src/render.h:9-18, filled at src/render.c:296-305.
 * Layout is kept bit-for-bit so a caller's existing struct can be passed as is.  ip / w / data are the
 * Ooura scratch areas of the CPU path; the GPU path ignores them (scratch lives in registers/shared memory)
 * and never frees caller memory (ownership: src/render.c:413-416). */
typedef struct DctcEnergyParameters_ {
    float edges;
    float textures;
    int blocksize;
    int *ip;
    double *w;
    double **data;
} DctcEnergyParameters;

typedef struct dctc_context dctc_context;

/* Superset handed to liblqr as extra_data (src/render.c:314-315): the prefix IS EnergyParameters, so the
 * reference's own dct_pixel_energy could still read it; the tail carries the GPU context. */
typedef struct DctcCarverEnergyParams_ {
    DctcEnergyParameters base;
    dctc_context *gpu;
} DctcCarverEnergyParams;

/* kernel selection for block size 8 (other block sizes always use the FP32 CUDA-core kernel) */
enum {
    DCTC_KERNEL_AUTO = 0,
    DCTC_KERNEL_FP32_TILE = 1,   /* generic shared-memory tile kernel, all block sizes */
    DCTC_KERNEL_FP32_MARCH = 2,  /* b=8 register-sliding column march */
    DCTC_KERNEL_TC_SPLIT = 3,    /* tcgen05 Toeplitz GEMM, fp16 hi/lo split operands, fp32 accumulate (b = 8; b = 16 by default) */
    DCTC_KERNEL_FP32_STREAM = 4  /* b=2, 4 streaming register-march kernel (what AUTO picks for them on aligned 1- or 3-channel rows) */
};

/* ---- lifetime -------------------------------------------------------------------------------------- */

/* Creates a context on CUDA device `device` with its own stream.  Replaces the scratch allocation of
 * src/render.c:296-305 (alloc_1d_int / alloc_1d_double / alloc_2d_double). */
int dctc_create(dctc_context **ctx, int device);
/* Frees device buffers, pinned staging and the stream.  Counterpart of the frees at src/render.c:413-416. */
void dctc_destroy(dctc_context *ctx);
/* edges / textures / blocksize as PlugInVals carries them (src/main.h:12-22, src/main.c:151-153).  With a carver
 * session loaded, a change of any of the three rebuilds the session's resident energy map with the new operator
 * (liblqr: lqr_carver_set_energy_function invalidates the map, src/render.c:314-315). */
int dctc_set_params(dctc_context *ctx, const DctcEnergyParameters *params);
int dctc_set_kernel(dctc_context *ctx, int kernel);
int dctc_last_cuda_error(const dctc_context *ctx);
const char *dctc_strerror(int status);
int dctc_version(void);
/* number of CUDA devices visible, or a negative status */
int dctc_device_count(void);
/* CUDA stream of the context as an opaque handle (cudaStream_t) */
void *dctc_stream(dctc_context *ctx);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
unsigned long long dctc_launch_count(const dctc_context *ctx);

/* ---- K1: full energy map ----------------------------------------------------------------------------
 * Replaces liblqr's build_emap loop "for y<h for x<w: en = dct_pixel_energy(x,y,w,h,rw,extra)"
 * (callback src/render.c:134-157; dctNxN src/dct.c:77-94; weighted_max_dct_correlation src/dct.c:96-110)
 * over the interleaved 8-bit buffer that lqr_carver_new() receives (src/render.c:310-312), with the
 * LQR_ER_LUMA reader fused in.  out[y*w+x] is the gfloat the callback would return.
 * Device-pointer variants: every row must be readable for its full pitch_bytes (the kernels stage rows in 16-byte
 * chunks up to the pitch), i.e. the buffer spans h*pitch_bytes; the host-buffer variants copy exactly w*channels
 * bytes per row into their own 16-byte-pitched staging. */
int dctc_energy_full(dctc_context *ctx, const uint8_t *img, int w, int h, int channels, size_t pitch_bytes,
                     float *out);

/* Same with device-resident input/output (no copies); out_pitch in floats.  Asynchronous on the context
 * stream unless `sync` is non-zero. */
int dctc_energy_full_dev(dctc_context *ctx, const uint8_t *d_img, int w, int h, int channels,
                         size_t pitch_bytes, float *d_out, size_t out_pitch, int sync);

/* Batch of n_frames equally sized frames (BASELINE config 4), one launch. */
int dctc_energy_batch_dev(dctc_context *ctx, const uint8_t *d_imgs, int n_frames, size_t frame_stride_bytes,
                          int w, int h, int channels, size_t pitch_bytes, float *d_out,
                          size_t out_frame_stride, size_t out_pitch, int sync);

/* Row band of a taller image (BASELINE config 5).  d_band holds `band_rows` rows; d_top points to the
 * top_rows image rows directly above the band (in image order, so its last row touches the band) and d_bot to
 * the bot_rows rows directly below.  Either may be NULL with 0 rows at the image edge, where
 * the reference's edge replication (src/render.c:122-132) applies.  d_top / d_bot may point into a peer
 * GPU's memory (NVLink P2P): the kernel then reads the halo straight from the neighbour, no exchange step.
 * Needs blocksize/2-1 rows above and blocksize/2 rows below for an exact result. */
int dctc_energy_band_dev(dctc_context *ctx, const uint8_t *d_band, int w, int band_rows, int channels,
                         size_t pitch_bytes, const uint8_t *d_top, int top_rows, size_t top_pitch_bytes,
                         const uint8_t *d_bot, int bot_rows, size_t bot_pitch_bytes, float *d_out,
                         size_t out_pitch, int sync);

/* Same for a caller that knows where the band sits in the whole image: band_y0 = image row of the band's first row.
 * The block-size-16 tensor-core kernel anchors its 16-row accumulation steps to the image's row grid, so with band_y0
 * given the band's map is bit-identical to the rows a single full-image call produces, however the image is cut
 * (dctc_energy_band_dev is band_y0 = 0; every other kernel ignores it).  The multi-GPU layer below passes it. */
int dctc_energy_band_dev_at(dctc_context *ctx, const uint8_t *d_band, int w, int band_rows, int band_y0, int channels,
                            size_t pitch_bytes, const uint8_t *d_top, int top_rows, size_t top_pitch_bytes,
                            const uint8_t *d_bot, int bot_rows, size_t bot_pitch_bytes, float *d_out,
                            size_t out_pitch, int sync);

/* Host-buffer batch through pinned staging with copy/compute overlap (what bench.py's e2e measures). */
int dctc_energy_batch(dctc_context *ctx, const uint8_t *imgs, int n_frames, size_t frame_stride_bytes, int w,
                      int h, int channels, size_t pitch_bytes, float *out, size_t out_frame_stride);

/* ---- K2: carver session, incremental per-seam energy ---------------------------------------------------
 * Replaces liblqr's update_emap, which re-invokes the callback for the pixels within +-radius of the removed
 * seam (radius = blocksize/2 as registered at src/render.c:314-315). */

/* Uploads the image, keeps it device-resident and builds the full map (K1). */
int dctc_carver_load(dctc_context *ctx, const uint8_t *img, int w, int h, int channels, size_t pitch_bytes);
/* Current carver width / height (of the image, also while height operations carve its transpose). */
int dctc_carver_width(const dctc_context *ctx);
int dctc_carver_height(const dctc_context *ctx);
/* Copies the current w*h energy map to the host (row pitch = current width). */
int dctc_carver_energy(dctc_context *ctx, float *out);
/* Removes one vertical seam (seam_x[y] = column removed in row y, h entries), compacts the device image and
 * energy planes and recomputes the energy only in the band the seam touched:
 *   row y: x in [min_{|y'-y|<=r} seam_x[y'] - r, max_{|y'-y|<=r} seam_x[y'] + r - 1] clipped to [0, w-2].
 * On return *xmin / *xmax (h entries each, may be NULL) hold that band and band_out (may be NULL) receives, row
 * by row, the xmax[y]-xmin[y]+1 recomputed values packed back to back (at most 2*(blocksize/2)*(delta_x+1) per row,
 * delta_x the context's dctc_carver_set_delta_x: band_out needs room for h*2*(blocksize/2)*(delta_x+1) floats, which
 * is h*4*(blocksize/2) for the default delta_x = 1).  A seam step must stay within the context's delta_x,
 * |seam_x[y]-seam_x[y-1]| <= delta_x, as liblqr's are (1 in the plug-in, src/render.c:313); anything else returns
 * DCTC_ERR_INVALID, a column outside [0, w) DCTC_ERR_STATE.
 * A vertical-seam call: DCTC_ERR_STATE after a height call since the load. */
int dctc_carve_and_update(dctc_context *ctx, const int *seam_x, float *band_out, int *xmin, int *xmax);
/* Copies the current (carved) interleaved image back to the host, pitch = w*channels. */
int dctc_carver_image(dctc_context *ctx, uint8_t *out);
/* Whole retarget loop on the device (energy -> seam DP -> back-track -> carve -> band update), `n_seams`
 * vertical seams; seams_out (may be NULL) receives n_seams*h removed columns in the coordinates of the image
 * at the time of removal.  Mirrors lqr_carver_resize(carver, w - n_seams, h) (src/render.c:377) with the delta_x of
 * dctc_carver_set_delta_x and the rigidity of dctc_carver_set_rigidity (1 and 0, the plug-in's values,
 * src/render.c:313, by default). */
int dctc_carver_resize_width(dctc_context *ctx, int n_seams, int *seams_out);
/* Enlarging: lqr_carver_resize(carver, w + n_seams, h) as the plug-in calls it for seams_number > 0
 * (src/render.c:357-363,377).  The n_seams seams a shrink would remove are computed on a freshly loaded session (same
 * energies, same order; seams_out as above), then every pixel of those seams is doubled on the device: the new pixel
 * sits on its left with the integer mean (a + b) / 2 of the pixel and its left neighbour in the original row (a copy in
 * column 0) [liblqr lqr_carver_inflate, from memory: parity unpinned].  The session continues on the enlarged image
 * (dctc_carver_image / _energy / _width reflect it); dctc_carver_vmap returns the start frame's visibility map. */
int dctc_carver_enlarge_width(dctc_context *ctx, int n_seams, int *seams_out);
/* Height retargeting: lqr_carver_resize(carver, w, h -/+ n_seams), the plug-in's PlugInVals.vertically
 * (src/render.c:357-363).  As liblqr does, the session transposes its image (on the device) and runs the width seam loop
 * on the transpose, whose energy map is computed afresh with the session's operator.  Every result is what
 * dctc_carver_load of the transposed image followed by the width call gives, turned back into image orientation.
 * seams_out (may be NULL): n_seams * w ints, seams_out[s*w + x] = the row removed from column x by seam s, in the
 * coordinates at removal time.  dctc_carver_width / _height / _image / _energy / _energy_image / _vmap / _paint_seams and
 * dctc_pixel_energy keep speaking image orientation: the visibility map covers the frame the first height call started
 * from (row pitch = image width) and holds the order of the horizontal seam that removed each pixel.  (The host carver's
 * vertically path returns its map transposed.)  Split resizes continue the loop, enlarge continues on the enlarged frame,
 * incremental mode and dctc_set_params work as for the width.
 * One axis per load: the first seam operation after dctc_carver_load (resize, enlarge or dctc_carve_and_update) fixes
 * the axis, and a call along the other axis returns DCTC_ERR_STATE until the next load.  n_seams == 0: DCTC_OK, nothing
 * happens.  DCTC_ERR_STATE also for n_seams >= the height; DCTC_ERR_UNSUPPORTED for images taller than the device
 * seam DP covers (the session stays loaded).  A CUDA failure in the first height call leaves the session unloaded. */
int dctc_carver_resize_height(dctc_context *ctx, int n_seams, int *seams_out);
int dctc_carver_enlarge_height(dctc_context *ctx, int n_seams, int *seams_out);

/* Both axes in one call: lqr_carver_resize(carver, new_w, new_h) (src/render.c:377) as a plan of passes.  The width
 * changes first, then the height.  Along each axis there is either one shrink pass of extent - new_extent seams, or
 * enlarge passes of min(new_extent - extent, extent - 1) seams each until the target is reached (an enlarge covers
 * fewer seams than the extent).  The host carver's dctc_lqr_carver_resize follows the same plan. */
enum { DCTC_RESIZE_WIDTH = 0, DCTC_RESIZE_HEIGHT = 1 };
typedef struct {
    int axis;              /* DCTC_RESIZE_WIDTH (vertical seams) or DCTC_RESIZE_HEIGHT (horizontal seams) */
    int enlarge;           /* 1: the pass inserts n_seams seams, 0: it removes them */
    int n_seams;
    int w, h;              /* image size at the start of the pass */
    size_t seams_offset;   /* ints before this pass's seams in one frame's seams_out block */
    size_t vmap_offset;    /* ints before this pass's map in one frame's vmaps_out block */
} DctcResizePass;
/* Plan of a resize from w x h to new_w x new_h.  Fills the first max_passes passes (passes may be NULL when max_passes
 * is 0) and returns the number of passes, 0 when nothing changes.  A frame's seams_out needs the last pass's
 * seams_offset + n_seams * len ints (len = h for a width pass, w for a height pass), its vmaps_out the last pass's
 * vmap_offset + w * h ints.  DCTC_ERR_INVALID for a non-positive size or max_passes < 0; DCTC_ERR_STATE when a pass
 * cannot make progress (an extent of 1 cannot grow). */
int dctc_resize_plan(int w, int h, int new_w, int new_h, DctcResizePass *passes, int max_passes);
/* Runs the plan on the session's frame, entirely on the device: the width passes as dctc_carver_resize_width /
 * _enlarge_width run them (an enlarge pass continues on the enlarged frame), then one transpose of the current frame
 * and one K1 launch on it (the energy rebuild a reload would do), then the height passes as the _height calls run them.
 * Each pass gives what the per-axis call gives on a session loaded with the image the previous pass left.
 * seams_out (may be NULL): the passes' seam logs back to back in plan order, pass p at its seams_offset, each in the
 * layout of the per-axis call (n_seams * h ints for a width pass, n_seams * w for a height pass, coordinates at removal
 * time).  vmaps_out (may be NULL): one visibility map per pass at its vmap_offset, over the pass's start frame in image
 * orientation (h * w ints), values 1..n_seams in removal order, 0 = never removed; recorded whenever vmaps_out is given,
 * whatever dctc_carver_set_dump_vmaps says.  Incremental mode applies to the shrink passes.
 * Needs a session loaded with no seam operation since the load (DCTC_ERR_STATE otherwise).  new_w == w && new_h == h:
 * DCTC_OK, nothing happens.  DCTC_ERR_INVALID: new_w <= 0 or new_h <= 0.  DCTC_ERR_STATE also when the plan refuses.
 * DCTC_ERR_UNSUPPORTED: some pass's extent along its axis is wider than the device seam DP covers (checked on the plan
 * before any work: the session stays loaded).  Afterwards dctc_carver_width / _height / _image / _energy /
 * _energy_image, dctc_pixel_energy and dctc_set_params work on the final frame; seam operations, another
 * dctc_carver_resize, dctc_carver_vmap and dctc_carver_paint_seams return DCTC_ERR_STATE until the next load.  A CUDA
 * failure leaves the session unloaded. */
int dctc_carver_resize(dctc_context *ctx, int new_w, int new_h, int *seams_out, int *vmaps_out);
/* ---- levels: interactive resizing (gui_interactive_dialog, src/interface.c:37-135, callback_resize_slider :647-670) --
 * One seam loop to depth n, then any extent within n of the start, each a gather over the start image and the visibility
 * map.  dctc_carver_levels_width / _height run what dctc_carver_resize_width / _height(depth) with visibility maps run
 * (maps recorded whatever dctc_carver_set_dump_vmaps says; incremental mode and a bias apply) and keep a device copy of
 * the start frame (for heights its transpose).  seams_out as for dctc_carver_resize_width / _height.  Needs a loaded
 * session with no seam operation since the load (DCTC_ERR_STATE otherwise).  DCTC_ERR_INVALID: depth < 0.
 * DCTC_ERR_STATE: depth >= the extent along the axis.  DCTC_ERR_UNSUPPORTED: an extent wider than the device seam DP
 * covers (before any work: the session stays loaded).  depth == 0: DCTC_OK, and only the start extent renders.
 * Afterwards dctc_carver_width / _height / _image / _energy / _energy_image and dctc_pixel_energy show the frame carved by
 * depth; dctc_carver_vmap and _paint_seams the depth-n map; dctc_set_params rebuilds the energy map and keeps the levels.
 * Seam operations, dctc_carver_resize, dctc_carver_set_bias and another build return DCTC_ERR_STATE until the next load,
 * which drops the levels.  A CUDA failure leaves the session unloaded. */
int dctc_carver_levels_width(dctc_context *ctx, int depth, int *seams_out);
int dctc_carver_levels_height(dctc_context *ctx, int depth, int *seams_out);
/* n_levels images along the built axis, level-major in the order of extents: level i is n_frames * H_i * W_i * channels
 * bytes in image orientation, rows packed (W_i = extents[i] for width levels, H_i = extents[i] for height levels, the
 * other side the start frame's).  With e0 the start extent, an extent e0 - k (k <= depth) is bit for bit the image that
 * dctc_carver_load + the resize by k gives, e0 + m (m <= depth) the image that dctc_carver_load + the enlarge by m gives.
 * Extents may come in any order and repeat; the session does not change.  DCTC_ERR_INVALID: n_levels <= 0, NULL extents
 * or out, an extent <= 0.  DCTC_ERR_STATE: no build since the load, an extent outside [e0 - depth, e0 + depth]. */
int dctc_carver_render_levels(dctc_context *ctx, int n_levels, const int *extents, uint8_t *out);

/* Optional: let the device loop update its cumulative map incrementally after each seam, like liblqr's update_mmap
 * (only the cells the removed seam can have changed are recomputed; a row whose changed range gets too wide falls
 * back to the full rebuild).  Same seams bit for bit; off by default because the full rebuild on an 8-CTA cluster is
 * currently the faster of the two (DESIGN.md section 4). */
int dctc_carver_set_incremental(dctc_context *ctx, int on);
/* Number of full cumulative-map rebuilds the incremental mode fell back to since dctc_carver_load (-1 on error). */
int dctc_carver_rebuild_count(dctc_context *ctx);

/* ---- bias: preserve and discard masks (liblqr's lqr_carver_bias_add) ----------------------------------------
 * A per-pixel float plane B that steers the seam search: every seam operation of the session (width and height resize
 * and enlarge, split resizes, incremental mode, dctc_carver_resize) runs on
 *     E_seam[y][x] = fl(en_op[y][x] + fl(B[y][x] / ext))      (FP32, IEEE division and add)
 * with en_op the operator energy and ext the start width of the frame the seam loop runs on: the loaded width for width
 * operations, the image height at the axis switch for height operations, the enlarged width for a pass after an enlarge
 * (liblqr's en = nrg + bias / w_start, with w_start and h_start swapped by the transpose [from memory: parity unpinned]).
 * The caller passes the value that is divided by ext.  Positive values keep pixels (a preserve mask), large negative
 * values remove them first (a discard mask: object removal).  The plane moves with the pixels: it is carved with them,
 * transposed at the axis switch, and an enlarge gives the inserted pixel the bias of the seam pixel it doubles.
 * Everything that shows energy (dctc_carver_energy, _energy_image, dctc_pixel_energy, dctc_carver_batch_energy) keeps
 * returning the operator map; on a biased session each such call computes it with one more K1 launch.
 * Launches: a biased seam loop launches per seam exactly what an unbiased one does.  Fixed extras of a biased session:
 * dctc_carver_set_bias one K1 and one bias-add launch; the axis switch one bias transpose and one bias add; an enlarge
 * one bias add (its inflate launch carries the bias).  A session without a bias launches what it launched before.
 * dctc_carver_set_bias: bias = w x h floats in image orientation, rows pitch_bytes apart, host or device memory (copied
 * with cudaMemcpyDefault like the loads); NULL clears the bias.  The values must be finite: this call does not check
 * them.  Needs a loaded session with no seam operation since the load (DCTC_ERR_STATE otherwise); dctc_carver_load clears
 * the bias.  DCTC_ERR_INVALID for a pitch below w floats.  dctc_carve_and_update returns DCTC_ERR_STATE on a biased
 * session.  A CUDA failure leaves the session unloaded. */
int dctc_carver_set_bias(dctc_context *ctx, const float *bias, size_t pitch_bytes);
/* The current bias plane (carved, transposed back, inflated): w * h floats, pitch w.  DCTC_ERR_STATE without a bias. */
int dctc_carver_bias(dctc_context *ctx, float *out);

/* ---- rigidity: straighter seams (liblqr's lqr_carver_init(carver, delta_x, rigidity)) -------------------------
 * A seam step to the left or right neighbour costs pen = fl(rigidity / h) more, h the length of the seams: the image
 * height for width operations, the image width at the axis switch for height operations (an enlarge uses the h of a
 * shrink along its axis).  Every seam loop of the session (width and height resize and enlarge, split resizes,
 * incremental mode, dctc_carver_resize, levels builds, with or without a bias) runs on
 *     m[y][x] = fl(E[y][x] + min(fl(m[y-1][x-1] + pen), m[y-1][x], fl(m[y-1][x+1] + pen)))
 * with the parent = the FIRST strict minimum of those three candidates scanning x-1, x, x+1, and the seam end the
 * leftmost minimum of the last row (liblqr's rigidity_map[dx] = rigidity * |dx|^1.5 / h for delta_x = 1, no rigidity
 * mask [from memory: parity unpinned]).  rigidity 0 (the default) gives the seams of a session that never set it, with
 * the same kernels.  A rigid seam loop launches per seam exactly what a loop of rigidity 0 launches.
 * dctc_carver_set_rigidity: an option of the context like dctc_carver_set_incremental; it survives loads and applies
 * from the next seam loop (so a value changed between two split resizes applies to the second one).  A levels build
 * that already ran and its renders are not affected.  A changed value drops the incremental map (the next seam rebuilds
 * it).  DCTC_ERR_INVALID: a negative or non-finite value. */
int dctc_carver_set_rigidity(dctc_context *ctx, float rigidity);

/* ---- seam step width (liblqr's lqr_carver_init(carver, delta_x, rigidity)) ----------------------------------
 * delta_x = dx, 1 .. DCTC_MAX_DELTA_X: a seam may move up to dx columns from one row to the next.  Every seam loop of the
 * session (the same list as for the rigidity) runs on
 *     pen[0] = 0,  pen[d] = fl(fl(rigidity * fl(d * fl(sqrt(d)))) / h)    d = 1 .. dx   (pen[1] is the rigidity's pen)
 *     m[y][x] = fl(E[y][x] + min over |d| <= dx of fl(m[y-1][x+d] + pen[|d|]))    (+inf outside the frame)
 * with the parent = the FIRST strict minimum scanning x-dx .. x+dx and the seam end the leftmost minimum of the last row
 * (liblqr's build_mmap with its rigidity_map [from memory: parity unpinned]).  delta_x = 1 (the default) is the plug-in's
 * value and runs exactly the kernels and launches of a session that never set it.  delta_x > 1 launches per seam what
 * delta_x = 1 launches, except for frames narrower than 261 columns or too tall for the parallel back-track's shared
 * memory at that delta_x, which walk the seam back inside the seam DP kernel (two launches fewer per seam); incremental
 * mode rebuilds the cumulative map for every seam (same seams: the incremental update is for delta_x = 1 only).  dctc_carve_and_update accepts steps up to delta_x.
 * dctc_carver_set_delta_x: an option of the context like dctc_carver_set_rigidity; it survives loads and applies from the
 * next seam loop, and a changed value drops the incremental map.  DCTC_ERR_INVALID: delta_x < 1.  DCTC_ERR_UNSUPPORTED:
 * delta_x > DCTC_MAX_DELTA_X. */
#define DCTC_MAX_DELTA_X 4
int dctc_carver_set_delta_x(dctc_context *ctx, int delta_x);

/* ---- visibility map and seam display ------------------------------------------------------------------------
 * lqr_carver_set_dump_vmaps (src/render.c:374): ask the session to record, for every ORIGINAL pixel, the order in
 * which dctc_carver_resize_width removed it (1-based, 0 = still visible).  Call before the first seam is removed. */
int dctc_carver_set_dump_vmaps(dctc_context *ctx, int on);
/* The map (w0*h ints, row pitch = original width; lqr_vmap_get_data / _get_depth, src/render.c:216-219). */
int dctc_carver_vmap(dctc_context *ctx, int *vmap_out, int *depth_out);
/* display_carver_seams (src/render.c:204-240) on a host image of the ORIGINAL size: every removed pixel with
 * x < w-1, y < h-1 becomes (0, (guchar)(255.0 * vis / depth), 0); painted on the device. */
int dctc_carver_paint_seams(dctc_context *ctx, uint8_t *img, int channels, size_t pitch_bytes);

/* ---- K2 batch: n equally sized frames through one device seam loop -----------------------------------------
 * A batch session, owned by the caller and tied to one context (destroy it before the context).  It has its own
 * device buffers and never touches the context's single-frame session.  Every phase of the seam loop is one launch
 * for all frames, and every frame's seam DP runs on its own cluster, so frames retarget side by side.  Each frame
 * gets exactly the seams, image, energy map and visibility map that dctc_carver_load + dctc_carver_resize_width
 * give it on its own, and dctc_carver_batch_enlarge_width gives every frame what dctc_carver_enlarge_width gives it;
 * the _height calls give every frame what the single session's _height calls give it.  The cumulative map is always
 * rebuilt: incremental mode is not batched.
 * Errors: DCTC_ERR_INVALID for NULL pointers, n_frames <= 0, a channel count outside 1..4, a pitch or frame stride
 * that is too small; DCTC_ERR_STATE for a resize before a load, after an enlarge, along the other axis than the first
 * seam operation since the load, or with n_seams >= the current width (height);
 * DCTC_ERR_UNSUPPORTED for widths the device seam DP does not cover (as dctc_carver_resize_width) and
 * n_frames > 65535. */
typedef struct dctc_carver_batch dctc_carver_batch;
/* n_frames frames of w x h, channels 1..4; uses the context's device, stream, blocksize / edges / textures and kernel
 * selection as they are at load time.  dump_vmaps: also keep a visibility map per frame. */
int dctc_carver_batch_create(dctc_context *ctx, int n_frames, int w, int h, int channels, int dump_vmaps,
                             dctc_carver_batch **batch);
void dctc_carver_batch_destroy(dctc_carver_batch *batch);
/* host frames (frame_stride_bytes apart, rows pitch_bytes apart) -> device, full energy map of every frame (one K1
 * batch launch).  A load restarts the session at the original width w, also after an enlarge. */
int dctc_carver_batch_load(dctc_carver_batch *batch, const uint8_t *imgs, size_t frame_stride_bytes, size_t pitch_bytes);
/* removes n_seams vertical seams from every frame; seams_out (may be NULL): n_frames * n_seams * h ints, frame-major,
 * in the coordinates at removal time (the layout dctc_carver_resize_width uses, per frame) */
int dctc_carver_batch_resize_width(dctc_carver_batch *batch, int n_seams, int *seams_out);
/* lqr_carver_resize to a larger width for every frame (the single session's dctc_carver_enlarge_width, per frame):
 * the n_seams seams a shrink would remove (seams_out as dctc_carver_batch_resize_width), then every pixel of those
 * seams is doubled.  Frames become w0 + n_seams wide; _images / _energy / _width reflect the enlarged frames (the energy
 * is the full map of the enlarged frame); _vmap (needs dump_vmaps) returns the start frames' maps over w0, depth
 * n_seams.  Each frame gets exactly the seams, enlarged image, energy map and start-frame visibility map that
 * dctc_carver_load + dctc_carver_enlarge_width give it alone on the same context.  A batch created without dump_vmaps
 * enlarges too (the removal order then lives in buffers the first enlarge allocates).
 * n_seams == 0: DCTC_OK, nothing happens.  DCTC_ERR_INVALID: NULL batch, n_seams < 0.  DCTC_ERR_STATE: not loaded, not
 * at the loaded width (a resize ran since the load), n_seams >= w.  DCTC_ERR_UNSUPPORTED: frames wider than the
 * device seam DP covers (checked before any work: the batch stays loaded).
 * After an enlarge, _resize_width and _enlarge_width return DCTC_ERR_STATE until the next dctc_carver_batch_load,
 * which restarts the batch at w x h.  A CUDA failure during the enlarge leaves the batch unloaded (DCTC_ERR_STATE until
 * the next load).  The buffers an enlarge allocates (a copy of the start frames, the enlarged frames, the removal
 * order) are reused by the next enlarge (the enlarged frames' when n_seams is the same) and freed by the destroy. */
int dctc_carver_batch_enlarge_width(dctc_carver_batch *batch, int n_seams, int *seams_out);
/* Height retargeting of every frame (the single session's dctc_carver_resize_height / _enlarge_height, per frame): the
 * first height call after a load transposes the frames on the device (one launch) into a transposed frame set the
 * batch keeps until the destroy, and computes their energy maps (one K1 launch); the width seam loop then runs on them.
 * seams_out: n_frames * n_seams * w ints, frame-major, seams_out[(f*n_seams + s)*w + x] = the row seam s removed from
 * column x of frame f.  One axis per load, as for the single session: after a width call the _height calls return
 * DCTC_ERR_STATE, and the other way round, until the next dctc_carver_batch_load.  _images / _energy / _vmap / _width /
 * _height speak image orientation; the visibility maps stay n_frames * h * w0 ints.  The enlarge rules of
 * dctc_carver_batch_enlarge_width apply (its buffers are reallocated when their size differs). */
int dctc_carver_batch_resize_height(dctc_carver_batch *batch, int n_seams, int *seams_out);
int dctc_carver_batch_enlarge_height(dctc_carver_batch *batch, int n_seams, int *seams_out);
/* dctc_carver_resize for every frame: each frame gets exactly the seams, maps, image and energy map that
 * dctc_carver_resize gives it alone on the same context.  Layout pass-major, then frame-major: pass p's block starts at
 * n_frames * its offset, and inside it is what the per-axis batch call writes (n_frames * n_seams * len seams,
 * n_frames * h * w map ints for the pass's start size).  The batch moves between frame sets: the transposed set is
 * filled from the current frames, an enlarge pass reads the previous pass's enlarged frames, and a set is reallocated
 * when its size differs (a batch that never calls this allocates nothing more).  Needs a loaded batch with no seam
 * operation since the load; the errors are those of dctc_carver_resize.  Afterwards _images / _energy / _width /
 * _height reflect the final frames; seam calls, another resize and _vmap return DCTC_ERR_STATE until
 * dctc_carver_batch_load, which restarts the batch at its created size.  A CUDA failure leaves the batch unloaded. */
int dctc_carver_batch_resize(dctc_carver_batch *batch, int new_w, int new_h, int *seams_out, int *vmaps_out);
/* dctc_carver_set_bias for every frame: n_frames planes of w x h floats (the created size), frame_stride_bytes apart,
 * rows pitch_bytes apart; NULL clears.  Every frame gets what dctc_carver_set_bias gives it on a single session.  Same
 * state rules: a loaded batch with no seam operation since the load, dctc_carver_batch_load clears the bias.  A batch
 * that never sets a bias allocates nothing more; its transposed and enlarged frame sets get bias planes only when the
 * set they come from has them.  A CUDA failure leaves the batch unloaded. */
int dctc_carver_batch_set_bias(dctc_carver_batch *batch, const float *bias, size_t frame_stride_bytes, size_t pitch_bytes);
/* current bias planes of every frame (n_frames * h * w floats, image orientation); DCTC_ERR_STATE without a bias */
int dctc_carver_batch_bias(dctc_carver_batch *batch, float *out);
/* dctc_carver_set_rigidity for the batch: every frame gets what the single session gives it with that rigidity.  A
 * setting of the batch, 0 at create; it survives loads and applies from the next seam loop.  DCTC_ERR_INVALID: NULL
 * batch, a negative or non-finite value. */
int dctc_carver_batch_set_rigidity(dctc_carver_batch *batch, float rigidity);
/* dctc_carver_set_delta_x for the batch: a setting of the batch, 1 at create; it survives loads and applies from the
 * next seam loop.  DCTC_ERR_INVALID: NULL batch, delta_x < 1.  DCTC_ERR_UNSUPPORTED: delta_x > DCTC_MAX_DELTA_X. */
int dctc_carver_batch_set_delta_x(dctc_carver_batch *batch, int delta_x);
/* current width / height of every frame */
int dctc_carver_batch_width(const dctc_carver_batch *batch);
int dctc_carver_batch_height(const dctc_carver_batch *batch);
/* current images (n_frames * h * w * channels, pitch w * channels) / energy maps (n_frames * h * w floats) */
int dctc_carver_batch_images(dctc_carver_batch *batch, uint8_t *out);
int dctc_carver_batch_energy(dctc_carver_batch *batch, float *out);
/* visibility map of every frame over the loaded size (n_frames * h * w0 ints) and the common depth; needs dump_vmaps
 * at create time */
int dctc_carver_batch_vmap(dctc_carver_batch *batch, int *vmap_out, int *depth_out);
/* dctc_carver_levels_width / _height and dctc_carver_render_levels for every frame: seams_out as the batch's
 * _resize_width / _resize_height; every frame's level is what the single session renders for it alone.  The rules are the
 * single session's; _vmap after a build needs dump_vmaps, as after an enlarge.  A CUDA failure in a build leaves the batch
 * unloaded. */
int dctc_carver_batch_levels_width(dctc_carver_batch *batch, int depth, int *seams_out);
int dctc_carver_batch_levels_height(dctc_carver_batch *batch, int depth, int *seams_out);
int dctc_carver_batch_render_levels(dctc_carver_batch *batch, int n_levels, const int *extents, uint8_t *out);
/* the same layout into device memory the caller owns (4-byte aligned), no host copy */
int dctc_carver_batch_render_levels_dev(dctc_carver_batch *batch, int n_levels, const int *extents, uint8_t *d_out);

/* ---- K3: energy-image export ------------------------------------------------------------------------------
 * Replaces lqr_carver_get_energy_image(carver, buf, orientation, LQR_COLDEPTH_8I, LQR_GREY_IMAGE) as called at
 * src/render.c:191 (the plug-in's "output energy" option, src/render.c:175-202): e -> 1/(1+1/e) (= e/(1+e)),
 * min-max normalise in float, 8-bit grey by truncation (guchar)(val*255) [liblqr, from memory: parity unpinned]. */

/* (min, max) of e/(1+e) over a device-resident w*h float plane; lo_hi receives two floats.  For a map sharded into
 * row bands each rank calls this on its band and the pairs are all-reduced (min, max) before dctc_energy_image_dev. */
int dctc_energy_minmax_dev(dctc_context *ctx, const float *d_en, size_t en_pitch, int w, int h, float *lo_hi);
/* Writes the 8-bit grey energy image of a device-resident plane.  lo_hi = the pair to normalise with (e.g. the
 * all-reduced one), or NULL to compute it from this plane on the device. */
int dctc_energy_image_dev(dctc_context *ctx, const float *d_en, size_t en_pitch, int w, int h, const float *lo_hi,
                          uint8_t *d_out, size_t out_pitch, int sync);
/* Energy image of the carver session's current map, copied to the host (w*h bytes, pitch w). */
int dctc_carver_energy_image(dctc_context *ctx, uint8_t *out);

/* ---- preview path --------------------------------------------------------------------------------------
 * Replaces dct_energy_preview (src/render.c:421-501), the GIMP preview / "energy image" filter: the same operator
 * with the preview window (offsets -(C-1) .. b-C, C = (b-1)/2, src/render.c:43-44 and src/dct.h:8-9), BT.601 byte
 * luminance (RGB2LUMINANCE, src/render.h:5; channels 1, 3 or 4 as convert_row_to_luminance accepts), weights applied
 * on the 0..255 scale, first transform index along y (src/render.c:47-51); then normalize_image
 * (src/render.c:81-109).  energy_out (w*h floats, may be NULL) receives the un-normalised map, image_out
 * (w*h*channels bytes, may be NULL) the normalised image replicated to every channel.  Uses the context's
 * blocksize / edges / textures (any block size). */
int dctc_preview_energy(dctc_context *ctx, const uint8_t *img, int w, int h, int channels, size_t pitch_bytes,
                        float *energy_out, uint8_t *image_out);

/* ---- per-pixel symbol, kept for ABI parity ---------------------------------------------------------------
 * Same signature as the reference's LqrEnergyFunc dct_pixel_energy (src/render.c:134).  `extra_data` must
 * point to a DctcCarverEnergyParams.  A per-pixel call cannot be GPU-backed, so it is served from the host
 * mirror of the device energy map of the context's carver session (valid when (w,h) match the session's
 * current size); otherwise it returns NaN and records DCTC_ERR_STATE.  `rw` is not dereferenced. */
struct DctcLqrReadingWindow_;
float dctc_pixel_energy(int x, int y, int w, int h, struct DctcLqrReadingWindow_ *rw, void *extra_data);

/* ---- synthetic inputs (bench / tests) ----------------------------------------------------------------- */

/* Counter-based generator, identical on CPU (tests) and GPU: byte = hash32(seed, frame, y, x, c) >> 24 for
 * pattern 0 (noise); patterns 1..3 are the gradient / checkerboard / step-edge stress images of SURVEY §8d. */
int dctc_synth_fill_dev(dctc_context *ctx, uint8_t *d_img, int n_frames, size_t frame_stride_bytes, int w, int h,
                        int channels, size_t pitch_bytes, uint32_t seed, int pattern, int first_frame, int y_offset);
uint8_t dctc_synth_byte(uint32_t seed, uint32_t frame, uint32_t y, uint32_t x, uint32_t c, int pattern);

/* ---- peer access for row-band sharding, one process per GPU (BASELINE config 5) ---------------------------
 * A rank exports its band buffer with dctc_ipc_export (64-byte CUDA IPC handle), sends the handle to its
 * neighbours over any channel, and they map it with dctc_ipc_open.  The mapped pointer is then passed as
 * d_top / d_bot of dctc_energy_band_dev, so the halo rows are loaded over NVLink by the energy kernel itself. */
#define DCTC_IPC_HANDLE_BYTES 64
int dctc_ipc_export(dctc_context *ctx, void *d_ptr, unsigned char handle[DCTC_IPC_HANDLE_BYTES]);
int dctc_ipc_open(dctc_context *ctx, const unsigned char handle[DCTC_IPC_HANDLE_BYTES], void **d_peer_ptr);
int dctc_ipc_close(dctc_context *ctx, void *d_peer_ptr);

/* ---- multi-GPU: frames and row bands over the GPUs of one box (SURVEY section 8e) ---------------------------
 * The reference runs in one process on one CPU thread (src/render.c:310-315 is the C caller of the energy path);
 * the path shards with a fixed halo and no collective: frame f -> device f mod G (BASELINE config 4), or one image
 * split into row bands, device g owning rows [h*g/G, h*(g+1)/G) (config 5).  A band needs blocksize/2-1 rows from
 * the band above and blocksize/2 rows from the band below (window offsets -b/2+1..b/2, src/render.c:146-147); the
 * image's own edges replicate (src/render.c:122-132).  Halo rows are not exchanged: the energy kernel of a band
 * loads them straight from the neighbour's HBM over NVLink (peer pointers). */

/* Band geometry of `rank` out of `world`: first row, row count, halo rows needed above / below.
 * DCTC_ERR_INVALID if some band would be thinner than blocksize/2 rows (it could not serve its neighbours' halos). */
int dctc_band_plan(int h, int world, int rank, int blocksize, int *y0, int *rows, int *top_need, int *bot_need);

/* -- one process drives all devices (what a C caller like render() would link against) -- */
typedef struct dctc_multi dctc_multi;
typedef struct dctc_multi_bands dctc_multi_bands;
/* One context (own streams) per entry of devices[] (NULL: every visible device); peer access is enabled between all
 * pairs.  The same device may be listed more than once (the bands then share one GPU; used by single-GPU tests). */
int dctc_multi_create(dctc_multi **m, const int *devices, int n_devices);
void dctc_multi_destroy(dctc_multi *m);
int dctc_multi_device_count(const dctc_multi *m);
dctc_context *dctc_multi_context(dctc_multi *m, int i);
int dctc_multi_set_params(dctc_multi *m, const DctcEnergyParameters *params);
int dctc_multi_set_kernel(dctc_multi *m, int kernel);
unsigned long long dctc_multi_launch_count(const dctc_multi *m);
/* dctc_energy_batch over all devices: frame f is processed by device f mod G, every device with its own
 * H2D / kernel / D2H pipeline, one host thread per device.  Same arguments and result as dctc_energy_batch. */
int dctc_multi_energy_batch(dctc_multi *m, const uint8_t *imgs, int n_frames, size_t frame_stride_bytes, int w, int h,
                            int channels, size_t pitch_bytes, float *out, size_t out_frame_stride);
/* One host image -> row bands over the devices -> the full energy map `out` (w*h floats, may be NULL) and / or the
 * 8-bit energy image `image_out` (w*h bytes, may be NULL; K3 with the (min, max) pair reduced over the bands).
 * Bit-identical to dctc_energy_full / dctc_carver_energy_image on one device. */
int dctc_multi_energy_bands(dctc_multi *m, const uint8_t *img, int w, int h, int channels, size_t pitch_bytes,
                            float *out, uint8_t *image_out);
/* The same in steps, bands resident on the devices (bench.py times dctc_multi_bands_energy). */
int dctc_multi_bands_create(dctc_multi *m, int w, int h, int channels, dctc_multi_bands **bands);
void dctc_multi_bands_destroy(dctc_multi_bands *bands);
int dctc_multi_bands_geometry(const dctc_multi_bands *bands, int g, int *y0, int *rows);
int dctc_multi_bands_upload(dctc_multi_bands *bands, const uint8_t *img, size_t pitch_bytes);
int dctc_multi_bands_synth(dctc_multi_bands *bands, uint32_t seed, int pattern);
int dctc_multi_bands_energy(dctc_multi_bands *bands, int sync);
int dctc_multi_bands_download(dctc_multi_bands *bands, float *out);
int dctc_multi_bands_energy_image(dctc_multi_bands *bands, uint8_t *out);

/* -- one process per GPU (bench.py under torchrun): each rank owns one band -- */
typedef struct dctc_band_runner dctc_band_runner;
/* All-gather of `bytes` bytes per rank through a POSIX shared-memory segment named after `name` (unique per
 * exchange); also a barrier.  DCTC_ERR_STATE on timeout (timeout_ms <= 0: wait forever). */
int dctc_rendezvous_allgather(const char *name, int rank, int world, const void *mine, size_t bytes, void *all,
                              int timeout_ms);
/* Allocates this rank's band of a w x h image on the context's device.  `rendezvous` names the job (e.g. the
 * launcher's port + run id); the collective calls below exchange through "<rendezvous>_<sequence number>". */
int dctc_band_runner_create(dctc_context *ctx, const char *rendezvous, int rank, int world, int w, int h, int channels,
                            dctc_band_runner **runner);
int dctc_band_runner_geometry(const dctc_band_runner *runner, int *y0, int *rows, size_t *pitch_bytes);
void *dctc_band_runner_image_dev(dctc_band_runner *runner);
float *dctc_band_runner_energy_dev(dctc_band_runner *runner);
int dctc_band_runner_synth(dctc_band_runner *runner, uint32_t seed, int pattern);
int dctc_band_runner_upload(dctc_band_runner *runner, const uint8_t *band_rows, size_t pitch_bytes);
/* COLLECTIVE: exports the band buffer as a CUDA IPC handle, all-gathers the handles and maps the neighbours' bands.
 * The band must hold its content: the exchange is the barrier between "filled" and "neighbours may read". */
int dctc_band_runner_connect(dctc_band_runner *runner);
/* COLLECTIVE: stream sync + barrier (e.g. between re-filling the bands and the next energy launch). */
int dctc_band_runner_barrier(dctc_band_runner *runner);
/* K1 on this rank's band, halo rows loaded from the neighbours' HBM by the kernel itself. */
int dctc_band_runner_energy(dctc_band_runner *runner, int sync);
int dctc_band_runner_download(dctc_band_runner *runner, float *out_rows);
/* COLLECTIVE: K3 over the sharded map ((min, max) all-gathered and reduced on the host), this rank's rows. */
int dctc_band_runner_energy_image(dctc_band_runner *runner, uint8_t *out_rows);
/* COLLECTIVE: barrier, then frees the band (no rank frees memory a neighbour's kernel may still be reading). */
void dctc_band_runner_destroy(dctc_band_runner *runner);

/* Pinned host <-> device copy bandwidth of this context's device in GB/s: H2D alone, D2H alone, and per direction
 * with both running (the ceiling of the host-buffer entry points; bench.py reports it next to `e2e`). */
int dctc_pcie_probe(dctc_context *ctx, size_t bytes, int iters, double *h2d_gbs, double *d2h_gbs,
                    double *bidir_gbs_per_dir);

/* ---- raw device memory helpers so that C / ctypes callers need no other CUDA binding -------------------- */
int dctc_dev_alloc(dctc_context *ctx, void **d_ptr, size_t bytes);
int dctc_dev_free(dctc_context *ctx, void *d_ptr);
int dctc_host_alloc_pinned(void **h_ptr, size_t bytes);
/* write-combined pinned memory for INPUT frames the host only writes (uploads do not snoop the CPU caches; CPU reads of
 * such memory are slow); freed with dctc_host_free_pinned */
int dctc_host_alloc_pinned_wc(void **h_ptr, size_t bytes);
int dctc_host_free_pinned(void *h_ptr);
int dctc_memcpy_h2d(dctc_context *ctx, void *d_dst, const void *h_src, size_t bytes);
int dctc_memcpy_d2h(dctc_context *ctx, void *h_dst, const void *d_src, size_t bytes);
int dctc_memset_dev(dctc_context *ctx, void *d_ptr, int value, size_t bytes);
int dctc_sync(dctc_context *ctx);
/* Event timing on the context stream: returns elapsed milliseconds between begin and end. */
int dctc_timer_begin(dctc_context *ctx);
int dctc_timer_end(dctc_context *ctx, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* DCTC_H */

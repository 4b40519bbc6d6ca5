/* dctc_lqr.c — host-side carver (liblqr subset) + render.c-like glue.  See dctc_lqr.h for what is restated
 * and from where.  Plain C; the only compute it delegates is the energy (GPU batch hooks or a callback). */
#include "dctc_lqr.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

struct DctcLqrCarver_ {
    uint8_t *rgb;          /* current image, row pitch = pitch*ch (rows are compacted in place per seam) */
    int pitch;             /* pixels per stored row (>= w) */
    int w, h, ch;
    int w_start, h_start;  /* size handed to lqr_carver_new */
    int transposed;
    int delta_x;
    float rigidity;
    DctcLqrEnergyFunc nrg;
    int radius, reader;
    void *extra;
    dctc_context *gpu;
    int dump_vmaps;
    int *vs;               /* visibility over the start frame of the first carve op */
    int vs_w, vs_h, vs_depth;
    int *seams;            /* all seams, concatenated */
    int n_seams, seam_len, seams_cap;
    uint8_t *line;         /* scan_line buffer */
    int scan_pos;
    double timing[3];
};

/* Whether carve_vertical hands the whole seam loop to the device (dctc_carver_resize_width) when a GPU context is
 * attached.  On by default; the host loop (energy batches on the GPU, cumulative map / seam search / carve here) stays
 * for widths the device kernel does not cover and as the cross-check the tests run against. */
static int g_device_seam_loop = 1;
void dctc_host_set_device_seam_loop(int on) { g_device_seam_loop = on != 0; }
int dctc_host_get_device_seam_loop(void) { return g_device_seam_loop; }

static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}

double dctc_lqr_rwindow_read(DctcLqrReadingWindow *rw, int dx, int dy, int channel)
{
    int xx = rw->x + dx, yy = rw->y + dy;
    (void) channel;
    if (dx < -rw->radius || dx > rw->radius || dy < -rw->radius || dy > rw->radius) return 0.0;
    if (xx < 0 || xx >= rw->w || yy < 0 || yy >= rw->h) return 0.0;
    return rw->luma[(size_t) yy * rw->w + xx];
}

int dctc_lqr_rwindow_get_radius(DctcLqrReadingWindow *rw) { return rw->radius; }

DctcLqrCarver *dctc_lqr_carver_new(uint8_t *buffer, int width, int height, int channels)
{
    DctcLqrCarver *r;
    if (!buffer || width <= 0 || height <= 0 || channels < 1 || channels > 4) return NULL;
    r = (DctcLqrCarver *) calloc(1, sizeof(*r));
    if (!r) return NULL;
    r->rgb = buffer;
    r->w = r->w_start = r->pitch = width;
    r->h = r->h_start = height;
    r->ch = channels;
    r->delta_x = 1;
    r->reader = DCTC_LQR_ER_LUMA;
    return r;
}

int dctc_lqr_carver_init(DctcLqrCarver *r, int delta_x, float rigidity)
{
    if (!r || delta_x < 0) return DCTC_LQR_ERROR;
    r->delta_x = delta_x;
    r->rigidity = rigidity;
    return DCTC_LQR_OK;
}

int dctc_lqr_carver_set_energy_function(DctcLqrCarver *r, DctcLqrEnergyFunc f, int radius, int reader_type, void *extra)
{
    if (!r || radius < 0) return DCTC_LQR_ERROR;
    r->nrg = f;
    r->radius = radius;
    r->reader = reader_type;
    r->extra = extra;
    return DCTC_LQR_OK;
}

int dctc_lqr_carver_attach_gpu(DctcLqrCarver *r, dctc_context *gpu)
{
    if (!r) return DCTC_LQR_ERROR;
    r->gpu = gpu;
    return DCTC_LQR_OK;
}

void dctc_lqr_carver_set_dump_vmaps(DctcLqrCarver *r) { if (r) r->dump_vmaps = 1; }
int dctc_lqr_carver_get_width(const DctcLqrCarver *r) { return r->transposed ? r->h : r->w; }
int dctc_lqr_carver_get_height(const DctcLqrCarver *r) { return r->transposed ? r->w : r->h; }
int dctc_lqr_carver_get_channels(const DctcLqrCarver *r) { return r->ch; }
int dctc_lqr_carver_scan_by_row(const DctcLqrCarver *r) { return !r->transposed; }
void dctc_lqr_carver_scan_reset(DctcLqrCarver *r) { r->scan_pos = 0; }
const double *dctc_lqr_carver_timing(const DctcLqrCarver *r) { return r->timing; }

int dctc_lqr_carver_scan_line(DctcLqrCarver *r, int *n, uint8_t **rgb)
{
    if (r->scan_pos >= r->h) { r->scan_pos = 0; return 0; }
    *n = r->scan_pos;
    *rgb = r->rgb + (size_t) r->scan_pos * r->pitch * r->ch;
    r->scan_pos++;
    return 1;
}

void dctc_lqr_carver_destroy(DctcLqrCarver *r)
{
    if (!r) return;
    free(r->rgb); free(r->vs); free(r->seams); free(r->line);
    free(r);
}

const int *dctc_lqr_carver_vmap(const DctcLqrCarver *r, int *w0, int *h0, int *depth)
{
    if (w0) *w0 = r->vs_w;
    if (h0) *h0 = r->vs_h;
    if (depth) *depth = r->vs_depth;
    return r->vs;
}

const int *dctc_lqr_carver_seams(const DctcLqrCarver *r, int *n_seams, int *seam_len)
{
    if (n_seams) *n_seams = r->n_seams;
    if (seam_len) *seam_len = r->seam_len;
    return r->seams;
}

/* liblqr LQR_ER_LUMA reader [from memory]: channels normalised to [0,1], Rec.709 weights, times alpha */
static double luma_px(const uint8_t *p, int ch)
{
    double v;
    if (ch >= 3) v = 0.2126 * ((double) p[0] / 255.0) + 0.7152 * ((double) p[1] / 255.0) + 0.0722 * ((double) p[2] / 255.0);
    else v = (double) p[0] / 255.0;
    if (ch == 2 || ch == 4) v *= (double) p[ch - 1] / 255.0;
    return v;
}

static void fill_luma(const DctcLqrCarver *r, double *luma)
{
    int x, y;
    for (y = 0; y < r->h; y++)
        for (x = 0; x < r->w; x++) luma[(size_t) y * r->w + x] = luma_px(r->rgb + ((size_t) y * r->pitch + x) * r->ch, r->ch);
}

static void band_limits(const int *seam, int y, int h, int w, int rad, int *xmin, int *xmax)
{
    int lo = seam[y], hi = seam[y], d;
    for (d = -rad; d <= rad; d++) {
        int yy = y + d;
        if (yy < 0 || yy >= h) continue;
        if (seam[yy] < lo) lo = seam[yy];
        if (seam[yy] > hi) hi = seam[yy];
    }
    lo -= rad; hi += rad - 1;
    *xmin = lo < 0 ? 0 : lo;
    *xmax = hi > w - 1 ? w - 1 : hi;
}

/* m[y][x] = en[y][x] + min over parents x1 = x-dx..x+dx (clipped) of m[y-1][x1] + rig[|x1-x|], first strict minimum
 * scanning left to right.  rig: liblqr's rigidity_map (rigidity_map_of), NULL for rigidity 0. */
static float parent_cost(const float *mrow_prev, int x1, int x, const float *rig)
{
    return rig ? mrow_prev[x1] + rig[x1 < x ? x - x1 : x1 - x] : mrow_prev[x1];
}

static float min_parent(const float *mrow_prev, int x, int w, int dx, const float *rig)
{
    int x1, lo = x - dx < 0 ? 0 : x - dx, hi = x + dx > w - 1 ? w - 1 : x + dx;
    float best = parent_cost(mrow_prev, lo, x, rig);
    for (x1 = lo + 1; x1 <= hi; x1++)
        if (parent_cost(mrow_prev, x1, x, rig) < best) best = parent_cost(mrow_prev, x1, x, rig);
    return best;
}

static int argmin_parent(const float *mrow_prev, int x, int w, int dx, const float *rig)
{
    int x1, lo = x - dx < 0 ? 0 : x - dx, hi = x + dx > w - 1 ? w - 1 : x + dx, arg = lo;
    float best = parent_cost(mrow_prev, lo, x, rig);
    for (x1 = lo + 1; x1 <= hi; x1++)
        if (parent_cost(mrow_prev, x1, x, rig) < best) { best = parent_cost(mrow_prev, x1, x, rig); arg = x1; }
    return arg;
}

/* liblqr's rigidity_map for seams h rows long [from memory: parity unpinned]: rig[d] = fl(fl(rigidity * |d|^1.5) / h),
 * d = 0..dx, with |d|^1.5 = fl(d * fl(sqrt(d))) (correctly rounded steps, so that other implementations can restate it
 * exactly; d = 1 gives the device's pen = fl(rigidity / h)).  Returns NULL for rigidity 0 (the plain seam search) or
 * when the allocation fails (*nomem is set). */
static float *rigidity_map_of(float rigidity, int dx, int h, int *nomem)
{
    float *rig;
    int d;
    *nomem = 0;
    if (rigidity == 0.0f) return NULL;
    rig = (float *) malloc(sizeof(float) * (size_t) (dx + 1));
    if (!rig) { *nomem = 1; return NULL; }
    for (d = 0; d <= dx; d++) rig[d] = (rigidity * ((float) d * sqrtf((float) d))) / (float) h;
    return rig;
}

/* removes k vertical seams from the current frame */
static int carve_vertical(DctcLqrCarver *r, int k, int record_vs)
{
    const int P = r->pitch, h = r->h, ch = r->ch, dx = r->delta_x;
    float *en = NULL, *m = NULL, *band = NULL, *rig = NULL;
    int *raw = NULL, *seam = NULL, *xmin = NULL, *xmax = NULL;
    double *luma = NULL;
    DctcLqrReadingWindow rw;
    int x, y, s, rc = DCTC_LQR_NOMEM, rig_nomem;
    double t0;

    if (k <= 0) return DCTC_LQR_OK;
    if (k >= r->w) return DCTC_LQR_ERROR;
    if (!r->gpu && !r->nrg) return DCTC_LQR_ERROR;
    if (r->gpu && g_device_seam_loop && dx >= 1 && dx <= DCTC_MAX_DELTA_X) {
        /* the whole lqr_carver_resize loop on the device: energy, seam DP, back-track, carve, band update */
        int drc, *dseams;
        t0 = now_s();
        if (r->n_seams + k > r->seams_cap || r->seam_len != h) {
            int *ns;
            if (r->seam_len != h) { r->n_seams = 0; r->seam_len = h; }
            ns = (int *) realloc(r->seams, sizeof(int) * (size_t) (r->n_seams + k) * h);
            if (!ns) return DCTC_LQR_NOMEM;
            r->seams = ns; r->seams_cap = r->n_seams + k;
        }
        dseams = r->seams + (size_t) r->n_seams * h;
        if (dctc_carver_set_rigidity(r->gpu, r->rigidity) != DCTC_OK || dctc_carver_set_delta_x(r->gpu, dx) != DCTC_OK)
            return DCTC_LQR_ERROR;
        if (dctc_carver_load(r->gpu, r->rgb, r->w, h, ch, (size_t) P * ch) != DCTC_OK) return DCTC_LQR_ERROR;
        r->timing[0] += now_s() - t0;
        t0 = now_s();
        dctc_carver_set_dump_vmaps(r->gpu, record_vs);
        drc = dctc_carver_resize_width(r->gpu, k, dseams);
        if (drc == DCTC_OK) {
            const int w1 = r->w - k;
            if (record_vs) {
                free(r->vs);
                r->vs = (int *) calloc((size_t) r->w * h, sizeof(int));
                if (!r->vs) return DCTC_LQR_NOMEM;
                r->vs_w = r->w; r->vs_h = h;
                if (dctc_carver_vmap(r->gpu, r->vs, &r->vs_depth) != DCTC_OK) return DCTC_LQR_ERROR;
                dctc_carver_set_dump_vmaps(r->gpu, 0);
            }
            if (dctc_carver_image(r->gpu, r->rgb) != DCTC_OK) return DCTC_LQR_ERROR;   /* compact rows, pitch = new width */
            r->n_seams += k;
            r->w = w1;
            r->pitch = w1;
            r->timing[2] += now_s() - t0;
            return DCTC_LQR_OK;
        }
        dctc_carver_set_dump_vmaps(r->gpu, 0);
        if (drc != DCTC_ERR_UNSUPPORTED) return DCTC_LQR_ERROR;
        /* wider than the device seam kernel covers: fall through to the host loop (energy still on the GPU) */
    }
    en = (float *) malloc(sizeof(float) * (size_t) P * h);
    m = (float *) malloc(sizeof(float) * (size_t) P * h);
    raw = (int *) malloc(sizeof(int) * (size_t) P * h);
    seam = (int *) malloc(sizeof(int) * h);
    xmin = (int *) malloc(sizeof(int) * h);
    xmax = (int *) malloc(sizeof(int) * h);
    /* dctc_carve_and_update's band: at most 2 r (delta_x + 1) values per row */
    band = (float *) malloc(sizeof(float) * (size_t) h * (2 * (r->radius > 0 ? r->radius : 1) * (dx + 1) + 2));
    if (!r->gpu) luma = (double *) malloc(sizeof(double) * (size_t) P * h);
    rig = rigidity_map_of(r->rigidity, dx, h, &rig_nomem);
    if (!en || !m || !raw || !seam || !xmin || !xmax || !band || (!r->gpu && !luma) || rig_nomem) goto done;
    if (r->n_seams + k > r->seams_cap || r->seam_len != h) {
        int *ns;
        if (r->seam_len != h) { r->n_seams = 0; r->seam_len = h; }
        ns = (int *) realloc(r->seams, sizeof(int) * (size_t) (r->n_seams + k) * h);
        if (!ns) goto done;
        r->seams = ns; r->seams_cap = r->n_seams + k;
    }
    if (record_vs) {
        free(r->vs);
        r->vs = (int *) calloc((size_t) P * h, sizeof(int));
        if (!r->vs) goto done;
        r->vs_w = r->w; r->vs_h = h; r->vs_depth = 0;
    }
    for (y = 0; y < h; y++)
        for (x = 0; x < P; x++) raw[(size_t) y * P + x] = x;

    /* build_emap (en rows are kept compact: pitch = current width) */
    t0 = now_s();
    rc = DCTC_LQR_ERROR;
    if (r->gpu) {
        float *tmp = (float *) malloc(sizeof(float) * (size_t) r->w * h);
        if (!tmp) { rc = DCTC_LQR_NOMEM; goto done; }
        /* dctc_carve_and_update takes steps up to the context's delta_x (1 above the device's bound: as before it existed) */
        if (dctc_carver_set_delta_x(r->gpu, dx >= 1 && dx <= DCTC_MAX_DELTA_X ? dx : 1) != DCTC_OK ||
            dctc_carver_load(r->gpu, r->rgb, r->w, h, ch, (size_t) P * ch) != DCTC_OK ||
            dctc_carver_energy(r->gpu, tmp) != DCTC_OK) { free(tmp); goto done; }
        for (y = 0; y < h; y++) memcpy(en + (size_t) y * P, tmp + (size_t) y * r->w, sizeof(float) * r->w);
        free(tmp);
    } else {
        fill_luma(r, luma);
        rw.luma = luma; rw.w = r->w; rw.h = h; rw.radius = r->radius;
        for (y = 0; y < h; y++)
            for (x = 0; x < r->w; x++) {
                rw.x = x; rw.y = y;
                en[(size_t) y * P + x] = r->nrg(x, y, r->w, h, &rw, r->extra);
            }
    }
    r->timing[0] += now_s() - t0;

    /* build_mmap */
    t0 = now_s();
    memcpy(m, en, sizeof(float) * r->w);
    for (y = 1; y < h; y++)
        for (x = 0; x < r->w; x++)
            m[(size_t) y * P + x] = en[(size_t) y * P + x] + min_parent(m + (size_t) (y - 1) * P, x, r->w, dx, rig);
    r->timing[1] += now_s() - t0;

    for (s = 0; s < k; s++) {
        const int w = r->w, w1 = w - 1;
        int clo = 0, chi = -1; /* changed interval of the previous row in update_mmap */
        /* build_vpath: leftmost minimum of the last row, then back-track */
        t0 = now_s();
        {
            const float *last = m + (size_t) (h - 1) * P;
            int best = 0;
            for (x = 1; x < w; x++)
                if (last[x] < last[best]) best = x;
            seam[h - 1] = best;
            for (y = h - 1; y > 0; y--) seam[y - 1] = argmin_parent(m + (size_t) (y - 1) * P, seam[y], w, dx, rig);
        }
        memcpy(r->seams + (size_t) r->n_seams * h, seam, sizeof(int) * h);
        r->n_seams++;
        /* update_vsmap + carve: shift the tail of every row one pixel to the left (pitch stays P) */
        for (y = 0; y < h; y++) {
            const int sx = seam[y], tail = w1 - sx;
            if (record_vs) r->vs[(size_t) y * r->vs_w + raw[(size_t) y * P + sx]] = r->vs_depth + 1;
            memmove(r->rgb + ((size_t) y * P + sx) * ch, r->rgb + ((size_t) y * P + sx + 1) * ch, (size_t) tail * ch);
            memmove(raw + (size_t) y * P + sx, raw + (size_t) y * P + sx + 1, sizeof(int) * tail);
            memmove(en + (size_t) y * P + sx, en + (size_t) y * P + sx + 1, sizeof(float) * tail);
            memmove(m + (size_t) y * P + sx, m + (size_t) y * P + sx + 1, sizeof(float) * tail);
        }
        if (record_vs) r->vs_depth++;
        r->w = w1;
        r->timing[2] += now_s() - t0;

        /* update_emap: only the band the seam touched */
        t0 = now_s();
        if (r->gpu) {
            size_t off = 0;
            if (dctc_carve_and_update(r->gpu, seam, band, xmin, xmax) != DCTC_OK) { rc = DCTC_LQR_ERROR; goto done; }
            for (y = 0; y < h; y++) {
                const int n = xmax[y] - xmin[y] + 1;
                if (n > 0) { memcpy(en + (size_t) y * P + xmin[y], band + off, sizeof(float) * n); off += n; }
            }
        } else {
            fill_luma(r, luma);
            rw.luma = luma; rw.w = w1; rw.h = h; rw.radius = r->radius;
            for (y = 0; y < h; y++) {
                band_limits(seam, y, h, w1, r->radius, &xmin[y], &xmax[y]);
                for (x = xmin[y]; x <= xmax[y]; x++) {
                    rw.x = x; rw.y = y;
                    en[(size_t) y * P + x] = r->nrg(x, y, w1, h, &rw, r->extra);
                }
            }
        }
        r->timing[0] += now_s() - t0;

        /* update_mmap: recompute only where en changed, where the seam disturbed the parent sets, and below
         * cells whose value actually changed (cone of delta_x per row); identical to a full rebuild */
        t0 = now_s();
        for (y = 0; y < h; y++) {
            float *mrow = m + (size_t) y * P;
            const float *erow = en + (size_t) y * P;
            int lo = xmin[y], hi = xmax[y], nlo = w1, nhi = -1;
            if (y > 0) {
                const int s0 = seam[y - 1] < seam[y] ? seam[y - 1] : seam[y];
                const int s1 = seam[y - 1] > seam[y] ? seam[y - 1] : seam[y];
                if (s0 - 2 < lo) lo = s0 - 2;
                if (s1 + 1 > hi) hi = s1 + 1;
                if (chi >= clo) {
                    if (clo - dx < lo) lo = clo - dx;
                    if (chi + dx > hi) hi = chi + dx;
                }
            }
            if (lo < 0) lo = 0;
            if (hi > w1 - 1) hi = w1 - 1;
            for (x = lo; x <= hi; x++) {
                const float v = y == 0 ? erow[x] : erow[x] + min_parent(mrow - P, x, w1, dx, rig);
                if (v != mrow[x]) {
                    mrow[x] = v;
                    if (x < nlo) nlo = x;
                    nhi = x;
                }
            }
            clo = nlo; chi = nhi;
        }
        r->timing[1] += now_s() - t0;
    }
    for (y = 1; y < h; y++) memmove(r->rgb + (size_t) y * r->w * ch, r->rgb + (size_t) y * P * ch, (size_t) r->w * ch);
    r->pitch = r->w;
    rc = DCTC_LQR_OK;
done:
    free(en); free(m); free(raw); free(seam); free(xmin); free(xmax); free(band); free(luma); free(rig);
    return rc;
}

static int transpose(DctcLqrCarver *r)
{
    const int w = r->w, h = r->h, ch = r->ch;
    int x, y;
    uint8_t *t = (uint8_t *) malloc((size_t) w * h * ch);
    if (!t) return DCTC_LQR_NOMEM;
    for (y = 0; y < h; y++)
        for (x = 0; x < w; x++) memcpy(t + ((size_t) x * h + y) * ch, r->rgb + ((size_t) y * r->pitch + x) * ch, ch);
    free(r->rgb);
    r->rgb = t; r->w = r->pitch = h; r->h = w;
    r->transposed = !r->transposed;
    return DCTC_LQR_OK;
}

/* Enlarging by k < w columns [liblqr lqr_carver_inflate, from memory: PARITY UNPINNED]: the k seams a shrink by k would
 * remove are computed (same energies, same order, recorded in the visibility map), then every pixel of those seams is
 * doubled: a new pixel is inserted on its left whose channels are the integer mean (a + b) / 2 of the pixel and its
 * left neighbour in the ORIGINAL row (a copy of the pixel in column 0).  The visibility map of the start frame and the
 * seam list are kept as for a shrink. */
static int enlarge_vertical(DctcLqrCarver *r, int k, int record_vs)
{
    const int w0 = r->w, h = r->h, ch = r->ch;
    uint8_t *orig, *out;
    int x, y, c, rc;
    (void) record_vs;
    if (k <= 0) return DCTC_LQR_OK;
    if (k >= w0) return DCTC_LQR_ERROR;
    orig = (uint8_t *) malloc((size_t) w0 * h * ch);
    if (!orig) return DCTC_LQR_NOMEM;
    for (y = 0; y < h; y++) memcpy(orig + (size_t) y * w0 * ch, r->rgb + (size_t) y * r->pitch * ch, (size_t) w0 * ch);
    if (r->gpu && g_device_seam_loop && r->delta_x >= 1 && r->delta_x <= DCTC_MAX_DELTA_X) {
        /* seams, visibility map and the pixel synthesis on the device */
        int *ns;
        if (r->seam_len != h) { r->n_seams = 0; r->seam_len = h; }
        ns = (int *) realloc(r->seams, sizeof(int) * (size_t) (r->n_seams + k) * h);
        if (!ns) { free(orig); return DCTC_LQR_NOMEM; }
        r->seams = ns; r->seams_cap = r->n_seams + k;
        rc = dctc_carver_set_rigidity(r->gpu, r->rigidity);
        if (rc == DCTC_OK) rc = dctc_carver_set_delta_x(r->gpu, r->delta_x);
        if (rc == DCTC_OK) rc = dctc_carver_load(r->gpu, orig, w0, h, ch, (size_t) w0 * ch);
        if (rc == DCTC_OK) rc = dctc_carver_enlarge_width(r->gpu, k, r->seams + (size_t) r->n_seams * h);
        if (rc == DCTC_OK) {
            out = (uint8_t *) malloc((size_t) (w0 + k) * h * ch);
            free(r->vs);
            r->vs = (int *) calloc((size_t) w0 * h, sizeof(int));
            if (!out || !r->vs) { free(out); free(orig); return DCTC_LQR_NOMEM; }
            r->vs_w = w0; r->vs_h = h;
            if (dctc_carver_vmap(r->gpu, r->vs, &r->vs_depth) != DCTC_OK || dctc_carver_image(r->gpu, out) != DCTC_OK) {
                free(out); free(orig);
                return DCTC_LQR_ERROR;
            }
            dctc_carver_set_dump_vmaps(r->gpu, 0);
            r->n_seams += k;
            free(r->rgb); free(orig);
            r->rgb = out; r->w = r->pitch = w0 + k;
            return DCTC_LQR_OK;
        }
        dctc_carver_set_dump_vmaps(r->gpu, 0);
        if (rc != DCTC_ERR_UNSUPPORTED) { free(orig); return DCTC_LQR_ERROR; }
        /* wider than the device seam kernel covers: host loop below */
    }
    rc = carve_vertical(r, k, 1);                      /* the seams: r->vs holds their order over the start frame */
    if (rc) { free(orig); return rc; }
    out = (uint8_t *) malloc((size_t) (w0 + k) * h * ch);
    if (!out) { free(orig); return DCTC_LQR_NOMEM; }
    for (y = 0; y < h; y++) {
        const uint8_t *src = orig + (size_t) y * w0 * ch;
        uint8_t *dst = out + (size_t) y * (w0 + k) * ch;
        int n = 0;
        for (x = 0; x < w0; x++) {
            const int vis = r->vs[(size_t) y * w0 + x];
            if (vis > 0 && vis <= k) {
                for (c = 0; c < ch; c++)
                    dst[(size_t) (x + n) * ch + c] = x > 0 ? (uint8_t) (((int) src[(size_t) (x - 1) * ch + c] + (int) src[(size_t) x * ch + c]) / 2)
                                                           : src[(size_t) x * ch + c];
                n++;
            }
            memcpy(dst + (size_t) (x + n) * ch, src + (size_t) x * ch, ch);
        }
    }
    free(r->rgb); free(orig);
    r->rgb = out; r->w = r->pitch = w0 + k;
    return DCTC_LQR_OK;
}

/* one axis of lqr_carver_resize: shrink, or enlarge in passes of fewer than w columns each */
static int resize_axis(DctcLqrCarver *r, int w1, int *first)
{
    int rc;
    if (w1 < r->w) {
        rc = carve_vertical(r, r->w - w1, *first);
        if (rc) return rc;
        *first = 0;
    }
    while (w1 > r->w) {
        const int k = w1 - r->w < r->w - 1 ? w1 - r->w : r->w - 1;
        if (k <= 0) return DCTC_LQR_ERROR;
        rc = enlarge_vertical(r, k, *first);
        if (rc) return rc;
        *first = 0;
    }
    return DCTC_LQR_OK;
}

/* lqr_carver_resize: width first, then height (through a transposed frame) [liblqr, from memory]. */
int dctc_lqr_carver_resize(DctcLqrCarver *r, int w1, int h1)
{
    int rc, first;
    if (!r || w1 <= 0 || h1 <= 0) return DCTC_LQR_ERROR;
    first = r->dump_vmaps;
    if (w1 != r->w) {
        rc = resize_axis(r, w1, &first);
        if (rc) return rc;
    }
    if (h1 != r->h) {
        rc = transpose(r);
        if (rc) return rc;
        rc = resize_axis(r, h1, &first);
        if (rc) { transpose(r); return rc; }
        rc = transpose(r);
        if (rc) return rc;
    }
    return DCTC_LQR_OK;
}

int dctc_lqr_carver_get_energy(DctcLqrCarver *r, float *buffer)
{
    int x, y;
    if (!r || !buffer) return DCTC_LQR_ERROR;
    if (r->gpu) {
        if (dctc_carver_load(r->gpu, r->rgb, r->w, r->h, r->ch, (size_t) r->pitch * r->ch) != DCTC_OK) return DCTC_LQR_ERROR;
        return dctc_carver_energy(r->gpu, buffer) == DCTC_OK ? DCTC_LQR_OK : DCTC_LQR_ERROR;
    }
    if (!r->nrg) return DCTC_LQR_ERROR;
    {
        DctcLqrReadingWindow rw;
        double *luma = (double *) malloc(sizeof(double) * (size_t) r->w * r->h);
        if (!luma) return DCTC_LQR_NOMEM;
        fill_luma(r, luma);
        rw.luma = luma; rw.w = r->w; rw.h = r->h; rw.radius = r->radius;
        for (y = 0; y < r->h; y++)
            for (x = 0; x < r->w; x++) {
                rw.x = x; rw.y = y;
                buffer[(size_t) y * r->w + x] = r->nrg(x, y, r->w, r->h, &rw, r->extra);
            }
        free(luma);
    }
    return DCTC_LQR_OK;
}

int dctc_lqr_carver_get_energy_image(DctcLqrCarver *r, uint8_t *buffer)
{
    size_t i, n = (size_t) r->w * r->h;
    float lo, hi, *e;
    int rc;
    if (r->gpu) {   /* K3: compression, min/max and quantisation on the device, same FP32 operation order */
        if (dctc_carver_load(r->gpu, r->rgb, r->w, r->h, r->ch, (size_t) r->pitch * r->ch) != DCTC_OK) return DCTC_LQR_ERROR;
        return dctc_carver_energy_image(r->gpu, buffer) == DCTC_OK ? DCTC_LQR_OK : DCTC_LQR_ERROR;
    }
    e = (float *) malloc(sizeof(float) * n);
    if (!e) return DCTC_LQR_NOMEM;
    rc = dctc_lqr_carver_get_energy(r, e);
    if (rc) { free(e); return rc; }
    for (i = 0; i < n; i++) e[i] = 1.0f / (1.0f + (1.0f / e[i]));   /* liblqr's soft compression; e = 0 -> 0 */
    lo = hi = e[0];
    for (i = 1; i < n; i++) { if (e[i] < lo) lo = e[i]; if (e[i] > hi) hi = e[i]; }
    for (i = 0; i < n; i++) buffer[i] = hi > lo ? (uint8_t) (((e[i] - lo) / (hi - lo)) * 255.0f) : 0;   /* lqr_pixel_set_norm truncates */
    free(e);
    return DCTC_LQR_OK;
}

/* ---- render.c-like glue --------------------------------------------------------------------------------- */

void dctc_render_result_free(DctcRenderResult *res)
{
    if (!res) return;
    free(res->image); free(res->energy_image); free(res->vmap); free(res->seams);
    memset(res, 0, sizeof(*res));
}

int dctc_render(const uint8_t *img, int w, int h, int channels, const DctcPlugInVals *vals, dctc_context *gpu,
                DctcLqrEnergyFunc cb, void *cb_extra, DctcRenderResult *res)
{
    return dctc_render_ext(img, w, h, channels, vals, 1, 0.0f, gpu, cb, cb_extra, res);   /* src/render.c:313 */
}

int dctc_render_ext(const uint8_t *img, int w, int h, int channels, const DctcPlugInVals *vals, int delta_x, float rigidity,
                    dctc_context *gpu, DctcLqrEnergyFunc cb, void *cb_extra, DctcRenderResult *res)
{
    DctcCarverEnergyParams ep;       /* superset of EnergyParameters: prefix layout of src/render.h:9-18 */
    DctcLqrCarver *carver;
    uint8_t *rgb_buffer, *line;
    int new_w, new_h, y, n, rc = DCTC_ERR_INVALID;
    const int *seams;
    double t0 = now_s();
    const double *tm;

    if (!img || !vals || !res || w <= 0 || h <= 0 || delta_x < 1 || !(rigidity >= 0.0f) || !isfinite(rigidity)) return DCTC_ERR_INVALID;
    if (!gpu && !cb) return DCTC_ERR_NO_DEVICE;     /* no CPU fallback in the product */
    memset(res, 0, sizeof(*res));

    /* init_carver_from_vals, src/render.c:296-316 */
    memset(&ep, 0, sizeof(ep));
    ep.base.edges = vals->edges;
    ep.base.textures = vals->textures;
    ep.base.blocksize = vals->blocksize;
    ep.gpu = gpu;
    if (gpu) {
        rc = dctc_set_params(gpu, &ep.base);
        if (rc != DCTC_OK) return rc;                /* bad blocksize: src/dct.c:89-92 would call error() */
    }
    rgb_buffer = (uint8_t *) malloc((size_t) w * h * channels);
    if (!rgb_buffer) return DCTC_ERR_NOMEM;
    memcpy(rgb_buffer, img, (size_t) w * h * channels);
    carver = dctc_lqr_carver_new(rgb_buffer, w, h, channels);
    if (!carver) { free(rgb_buffer); return DCTC_ERR_INVALID; }
    dctc_lqr_carver_init(carver, delta_x, rigidity);
    if (gpu) {
        dctc_lqr_carver_set_energy_function(carver, (DctcLqrEnergyFunc) dctc_pixel_energy, vals->blocksize / 2,
                                            DCTC_LQR_ER_LUMA, (void *) &ep);
        dctc_lqr_carver_attach_gpu(carver, gpu);
    } else {
        dctc_lqr_carver_set_energy_function(carver, cb, vals->blocksize / 2, DCTC_LQR_ER_LUMA, cb_extra);
    }

    /* render, src/render.c:357-377 */
    if (vals->vertically) { new_w = w; new_h = h + vals->seams_number; }
    else { new_w = w + vals->seams_number; new_h = h; }
    rc = DCTC_ERR_INVALID;
    if (new_w <= 0 || new_h <= 0) goto out;          /* seams_number > 0 enlarges (src/render.c:357-363) */
    if (vals->output_energy) {
        res->energy_image = (uint8_t *) malloc((size_t) w * h);
        if (!res->energy_image || dctc_lqr_carver_get_energy_image(carver, res->energy_image)) { rc = DCTC_ERR_CUDA; goto out; }
    }
    if (vals->output_seams && vals->seams_number != 0) dctc_lqr_carver_set_dump_vmaps(carver);
    if (dctc_lqr_carver_resize(carver, new_w, new_h) != DCTC_LQR_OK) { rc = DCTC_ERR_CUDA; goto out; }
    if (vals->output_seams && vals->seams_number != 0) {
        int vw, vh, depth;
        const int *vs = dctc_lqr_carver_vmap(carver, &vw, &vh, &depth);
        if (vs) {
            res->vmap = (int *) malloc(sizeof(int) * (size_t) vw * vh);
            if (res->vmap) memcpy(res->vmap, vs, sizeof(int) * (size_t) vw * vh);
            res->vmap_depth = depth;
        }
    }
    /* write_carver_to_layer, src/render.c:244-284 */
    res->new_w = new_w; res->new_h = new_h; res->channels = channels;
    res->image = (uint8_t *) malloc((size_t) new_w * new_h * channels);
    if (!res->image) { rc = DCTC_ERR_NOMEM; goto out; }
    dctc_lqr_carver_scan_reset(carver);
    while (dctc_lqr_carver_scan_line(carver, &y, &line))
        memcpy(res->image + (size_t) y * new_w * channels, line, (size_t) new_w * channels);
    seams = dctc_lqr_carver_seams(carver, &res->n_seams, &res->seam_len);
    n = res->n_seams * res->seam_len;
    if (n > 0) {
        res->seams = (int *) malloc(sizeof(int) * (size_t) n);
        if (res->seams) memcpy(res->seams, seams, sizeof(int) * (size_t) n);
    }
    tm = dctc_lqr_carver_timing(carver);
    res->t_energy = tm[0]; res->t_mmap = tm[1]; res->t_seam = tm[2];
    rc = DCTC_OK;
out:
    dctc_lqr_carver_destroy(carver);
    res->t_total = now_s() - t0;
    if (rc != DCTC_OK) { double t = res->t_total; dctc_render_result_free(res); res->t_total = t; }
    return rc;
}

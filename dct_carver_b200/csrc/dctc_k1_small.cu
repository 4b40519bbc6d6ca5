// K1 (block sizes 2 and 4, full maps): streaming register-march kernel.  These block sizes need only ~20 / ~55
// instructions per pixel, so the operator is bound by HBM traffic (7 B/px for RGB), not by the FP32 pipe
// (SURVEY 8d): the kernel is organised around keeping the image rows in flight, not around the arithmetic.
//
// Same operator as dctc_k1_tile.cu (reference chain src/render.c:134-157 -> dctNxN src/dct.c:77-94 -> ddct2d,
// src/fft2d/fftsg2d.c:566-627, unnormalised -> weighted_max_dct_correlation src/dct.c:96-110) with the same transform
// code (the packed twins of dctc_dct_fwd<B> along x and along y, last-arg-max fold).  RGB luma is the EXACT integer
// 2126 R + 7152 G + 722 B (two dp2a per pixel instead of three byte->float conversions and an FMA chain; the factor
// 1/10000 folds into the final weight), so RGB maps agree with the tile kernel within the stated tolerance, grey maps
// bit for bit.  Carver sessions never mix the two (they pin the FP32 tile / march kernels).
//
//   * a CTA of 128 threads owns a strip of 256 columns and marches down SEG rows; thread t owns the ADJACENT columns
//     x0+2t and x0+2t+1: both passes run packed (FP32x2) over the column pair -- the x-pass reads B+1 consecutive luma
//     values (one 32-bit and B/2 64-bit shared loads), the ring of the last B rows holds (column a, column b) pairs,
//     one 64-bit store per row
//   * raw interleaved rows are copied global -> shared with 16-byte cp.async, 8 rows per chunk, two chunks ahead; thread
//     (row = t >> 4, lane = t & 15) copies the chunks lane, lane+16, ... of its row: ONE source pointer per thread,
//     advanced by 8 pitches per chunk, the chunk offsets are immediates
//   * conversion: 4 pixels per task from three 32-bit shared loads (two PRMT, one shift, eight dp2a, four I2F); thread
//     (t >> 6, t & 63) converts quad t & 63 of the rows t >> 6, +2, +4, +6 (offsets are immediates again), sixteen
//     threads also convert the two halo quads of a row; luma rows double buffered in shared memory
#include "dctc_common.cuh"
#include "dctc_launch.h"

namespace {

constexpr int NT = 128;        // threads per CTA
constexpr int MW = 2 * NT;     // columns per CTA
constexpr int LWP = MW + 8;    // staged luma row: index i <-> column x0 - 4 + i
constexpr int NQM = MW / 4;    // quads of the strip itself; quads -1 and NQM are the halo columns

template <int CH>
struct RawGeom {
    static constexpr int CHUNKS = (16 + (MW + 4) * CH + 15) / 16;       // 16-byte chunks per staged raw row (quads up to x0+MW+3)
    static constexpr int ROW = CHUNKS * 16;
    static constexpr int PER = (CHUNKS + 15) / 16;                      // chunks per thread and 8-row block
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }

// packed twins of dctc_dct_fwd<2> / <4> (tools/gen_dct.py): the same operations in the same order on two lanes.
// A bare product is written as fma(c, t, +0): ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 despite the explicit
// rounding modifiers (and despite -fmad=false), which would fuse an x-pass product into the y-pass sum that reads it and
// break the bit-equality with the tile kernel; an FMA is never contracted further, and c * t + 0 rounds like c * t.
__device__ __forceinline__ float2 f2prod(float c, float2 a) { return __ffma2_rn(make_float2(c, c), a, make_float2(0.0f, 0.0f)); }
template <int N>
__device__ __forceinline__ void dct_fwd2(const float2* __restrict__ v, float2* __restrict__ X);

template <>
__device__ __forceinline__ void dct_fwd2<2>(const float2* __restrict__ v, float2* __restrict__ X)
{
    const float2 t1 = dctc_f2add(v[0], v[1]), t2 = dctc_f2sub(v[0], v[1]);
    X[1] = f2prod(7.071067691e-01f, t2);
    X[0] = t1;
}

template <>
__device__ __forceinline__ void dct_fwd2<4>(const float2* __restrict__ v, float2* __restrict__ X)
{
    const float2 t1 = dctc_f2add(v[0], v[3]), t2 = dctc_f2sub(v[0], v[3]);
    const float2 t3 = dctc_f2add(v[1], v[2]), t4 = dctc_f2sub(v[1], v[2]);
    X[1] = dctc_f2fma(3.826834261e-01f, t4, dctc_f2mul(9.238795042e-01f, t2));
    X[3] = dctc_f2fma(-9.238795042e-01f, t4, dctc_f2mul(3.826834261e-01f, t2));
    const float2 t5 = dctc_f2add(t1, t3), t6 = dctc_f2sub(t1, t3);
    X[2] = f2prod(7.071067691e-01f, t6);
    X[0] = t5;
}

__device__ __forceinline__ float2 f2absmax(float2 m, float2 a) { return make_float2(fmaxf(m.x, fabsf(a.x)), fmaxf(m.y, fabsf(a.y))); }
__device__ __forceinline__ float2 f2absmax3(float2 m, float2 a, float2 b)
{
    return make_float2(fmaxf(m.x, fmaxf(fabsf(a.x), fabsf(b.x))), fmaxf(m.y, fmaxf(fabsf(a.y), fabsf(b.y))));
}

// fold of the coefficients X[k2] = T[K1][k2] of the thread's two columns (.x / .y); same rule as DctcTracker
// (dctc_common.cuh), one tracker per lane
template <int B, bool UNIFORM>
struct Fold;

template <int B>
struct Fold<B, true> {
    float2 m;
    __device__ __forceinline__ void init() { m = make_float2(0.0f, 0.0f); }
    template <int K1>
    __device__ __forceinline__ void add(const float2* X)
    {
        if (K1 == 0) {                                           // (0,0) is skipped (src/dct.c:101)
            m = f2absmax(m, X[1]);
#pragma unroll
            for (int k2 = 2; k2 < B; k2 += 2) m = f2absmax3(m, X[k2], X[k2 + 1]);
        } else {
#pragma unroll
            for (int k2 = 0; k2 < B; k2 += 2) m = f2absmax3(m, X[k2], X[k2 + 1]);
        }
    }
    __device__ __forceinline__ float2 result(float we, float wt) const { (void) we; return make_float2(m.x * wt, m.y * wt); }
};

template <int B>
struct Fold<B, false> {
    float2 a, mm, bv, z;
    __device__ __forceinline__ void init()
    {
        a = make_float2(0.0f, 0.0f); mm = make_float2(-1.0f, -1.0f); bv = make_float2(0.0f, 0.0f); z = make_float2(0.0f, 0.0f);
    }
    template <int K1>
    __device__ __forceinline__ void add(const float2* X)
    {
        if (K1 == 0) {
            a = make_float2(fabsf(X[1].x), fabsf(X[1].y));
#pragma unroll
            for (int k2 = 2; k2 < B; k2++) mm = f2absmax(mm, X[k2]);
        } else if (K1 == 1) {
            bv = make_float2(fabsf(X[0].x), fabsf(X[0].y));
#pragma unroll
            for (int k2 = 1; k2 < B; k2++) z = f2absmax(z, X[k2]);
        } else {
#pragma unroll
            for (int k2 = 0; k2 < B; k2++) z = f2absmax(z, X[k2]);
        }
    }
    static __device__ __forceinline__ float one(float a, float mm, float bv, float z, float we, float wt)
    {
        const float am = fmaxf(a, mm);
        const float top = fmaxf(fmaxf(am, bv), z);
        const bool tex = (z >= fmaxf(am, bv)) || (!(bv >= am) && (mm >= a));
        return top * (tex ? wt : we);
    }
    __device__ __forceinline__ float2 result(float we, float wt) const
    {
        return make_float2(one(a.x, mm.x, bv.x, z.x, we, wt), one(a.y, mm.y, bv.y, z.y, we, wt));
    }
};

// ---- staging ---------------------------------------------------------------------------------------------------
// Raw bytes [x0*CH - 16, x0*CH - 16 + ROW) of 8 rows per block; chunks outside [0, pitch) are skipped (clamped pixel
// indices never read them).  Thread (r = t >> 4, l = t & 15) copies the chunks l + 16 i of row r: the mapping is the
// same for every block of a segment, and while consecutive blocks lie inside the band itself (no halo rows, no edge
// replication) the thread's one source pointer just advances by 8 pitches.
template <int CH>
struct StageMap {
    using G = RawGeom<CH>;
    const uint8_t* src;          // chunk l of row r in the block staged last
    unsigned mask;               // bit i: chunk l + 16 i exists and lies inside [0, pitch)
    int last_vy0;
    __device__ __forceinline__ void init(const DctcK1Args& a, int x0, int tid)
    {
        const int l = tid & 15;
        mask = 0u;
#pragma unroll
        for (int i = 0; i < G::PER; i++) {
            const int k = l + 16 * i;
            const long long gb = (long long) x0 * CH - 16 + 16 * k;
            if (k < G::CHUNKS && gb >= 0 && gb + 16 <= (long long) a.pitch) mask |= 1u << i;
        }
        src = nullptr;
        last_vy0 = (int) 0x80000000;
    }
    // rows vy0 .. vy0 + nrows - 1 -> R (nrows <= 8)
    __device__ __forceinline__ void stage(const DctcK1Args& a, const uint8_t* __restrict__ img, uint8_t* __restrict__ R, int vy0, int x0,
                                          int tid, int nrows = 8)
    {
        const int r = tid >> 4, l = tid & 15;
        const bool step8 = vy0 == last_vy0 + 8 && last_vy0 >= 0 && vy0 + 7 < a.h;
        if (step8) src += 8 * a.pitch;
        else src = dctc_row_ptr(a, img, vy0 + r) + ((long long) x0 * CH - 16 + 16 * l);
        const uint32_t dst = smem_u32(R + r * G::ROW + 16 * l);
        if (r < nrows) {
#pragma unroll
            for (int i = 0; i < G::PER; i++)
                if (mask & (1u << i))
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 256u * i), "l"(src + 256 * i) : "memory");
        }
        last_vy0 = vy0;
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
};

// RGB luma as the exact integer 2126 R + 7152 G + 722 B (< 2^22: exact as a float); grey stays the byte itself
constexpr float LUMA_INT_SCALE = 1.0f / 10000.0f;
constexpr uint32_t LUMA_RG = (7152u << 16) | 2126u;    // dp2a.lo: R * 2126 + G * 7152 from bytes 0, 1
constexpr uint32_t LUMA_B = 722u;                       // dp2a.hi: B * 722 (+ 0 * byte 3) from bytes 2, 3

template <int CH>
__device__ __forceinline__ float luma_raw(const uint8_t* __restrict__ p)
{
    if (CH == 3) return (float) (2126u * p[0] + 7152u * p[1] + 722u * p[2]);
    return (float) p[0];
}

// byte k (0..3) of w -> float, exactly: the byte becomes the low mantissa bits of 2^23 + byte
__device__ __forceinline__ float byte_to_float(uint32_t w, int k)
{
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u | (uint32_t) k)) - 8388608.0f;
}

// luma of four consecutive pixels from their CH*4 raw bytes (4-byte aligned); same values as luma_raw
template <int CH>
__device__ __forceinline__ float4 quad_luma(const uint8_t* __restrict__ p)
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    float4 l;
    if (CH == 3) {
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
        const uint32_t p1 = __byte_perm(w0, w1, 0x6543), p2 = __byte_perm(w1, w2, 0x5432), p3 = w2 >> 8;
        l.x = (float) __dp2a_lo(LUMA_RG, w0, __dp2a_hi(LUMA_B, w0, 0u));
        l.y = (float) __dp2a_lo(LUMA_RG, p1, __dp2a_hi(LUMA_B, p1, 0u));
        l.z = (float) __dp2a_lo(LUMA_RG, p2, __dp2a_hi(LUMA_B, p2, 0u));
        l.w = (float) __dp2a_lo(LUMA_RG, p3, __dp2a_hi(LUMA_B, p3, 0u));
    } else {
        const uint32_t w0 = w[0];
        l.x = byte_to_float(w0, 0);
        l.y = byte_to_float(w0, 1);
        l.z = byte_to_float(w0, 2);
        l.w = byte_to_float(w0, 3);
    }
    return l;
}

// Raw rows -> luma rows; staged index i <-> image column clamp(x0 - 4 + i) (src/render.c:122-132).
// A task is one 4-pixel group (quad) of one row.  Thread (rr = t >> 6, q = t & 63) converts quad q of the rows
// rr, rr + 2, rr + 4, rr + 6 (fixed offsets from one raw / one luma address); threads 0..15 also convert the halo quad
// (q = -1 or NQM) of row t >> 1.  Quads that touch the image border take the per-pixel clamped path.
template <int CH>
struct ConvMap {
    using G = RawGeom<CH>;
    int roff, loff;              // raw byte offset / luma float index of the thread's quad in row rr
    int hroff, hloff, hg;        // halo quad (threads 0..15); hg = image column of its first pixel
    bool border, hborder;
    __device__ __forceinline__ void init(const DctcK1Args& a, int x0, int tid)
    {
        const int rr = tid >> 6, q = tid & 63;
        roff = rr * G::ROW + 16 + 4 * CH * q;
        loff = rr * LWP + 4 * q + 4;
        border = x0 + 4 * q + 3 >= a.w;
        const int hr = (tid >> 1) & 7, hq = (tid & 1) ? NQM : -1;
        hroff = hr * G::ROW + 16 + 4 * CH * hq;
        hloff = hr * LWP + 4 * hq + 4;
        hg = x0 + 4 * hq;
        hborder = hg < 0 || hg + 3 >= a.w;
    }
    static __device__ __forceinline__ float4 clamped(const DctcK1Args& a, const uint8_t* __restrict__ r, int g)
    {
        float t[4];
#pragma unroll
        for (int k = 0; k < 4; k++) t[k] = luma_raw<CH>(r + (max(0, min(g + k, a.w - 1)) - g) * CH);
        return make_float4(t[0], t[1], t[2], t[3]);
    }
    template <int NROWS>
    __device__ __forceinline__ void convert(const DctcK1Args& a, const uint8_t* __restrict__ R, float* __restrict__ L, int x0, int tid) const
    {
        const int rr = tid >> 6;
        if (!border) {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (NROWS == 8 || rr + 2 * i < NROWS)
                    *reinterpret_cast<float4*>(L + loff + 2 * i * LWP) = quad_luma<CH>(R + roff + 2 * i * G::ROW);
        } else {
            const int g = x0 + 4 * (tid & 63);
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (NROWS == 8 || rr + 2 * i < NROWS)
                    *reinterpret_cast<float4*>(L + loff + 2 * i * LWP) = clamped(a, R + roff + 2 * i * G::ROW, g);
        }
        if (tid < 16 && (NROWS == 8 || (tid >> 1) < NROWS))
            *reinterpret_cast<float4*>(L + hloff) = hborder ? clamped(a, R + hroff, hg) : quad_luma<CH>(R + hroff);
    }
};

// ---- march -----------------------------------------------------------------------------------------------------
// H[slot][k1] = x-pass coefficient k1 of (column a, column b) in ring slot `slot`
template <int B, int SLOT>
__device__ __forceinline__ void xpass(float2 (&H)[B][B], const float* __restrict__ Lrow, int tid)
{
    constexpr int R0 = B / 2 - 1;
    const float* p = Lrow + 2 * tid + 4 - R0;                  // the B + 1 samples both windows read
    float f[B + 1];
    if (B == 4) {
        f[0] = p[0];
        const float2 a = *reinterpret_cast<const float2*>(p + 1), b = *reinterpret_cast<const float2*>(p + 3);
        f[1] = a.x; f[2] = a.y; f[3] = b.x; f[B] = b.y;
    } else {
        const float2 a = *reinterpret_cast<const float2*>(p);
        f[0] = a.x; f[1] = a.y; f[B] = p[2];
    }
    float2 v[B], X[B];
#pragma unroll
    for (int j = 0; j < B; j++) v[j] = make_float2(f[j], f[j + 1]);
    dct_fwd2<B>(v, X);
#pragma unroll
    for (int k = 0; k < B; k++) H[SLOT][k] = X[k];
}

// y-pass over the window whose oldest row sits in ring slot J
template <int B, int J, bool UNIFORM>
__device__ __forceinline__ float2 ypass(const float2 (&H)[B][B], float we, float wt)
{
    Fold<B, UNIFORM> f;
    f.init();
#define DCTC_YP(K1)                                                                                                    \
    if (K1 < B) {                                                                                                      \
        float2 v[B], X[B];                                                                                             \
        _Pragma("unroll") for (int i = 0; i < B; i++) v[i] = H[(J + i) % B][K1 < B ? K1 : 0];                          \
        dct_fwd2<B>(v, X);                                                                                             \
        f.template add<K1>(X);                                                                                         \
    }
    DCTC_YP(0) DCTC_YP(1) DCTC_YP(2) DCTC_YP(3)
#undef DCTC_YP
    return f.result(we, wt);
}

// row RW of the chunk: the new image row lands in ring slot (RW + B - 1) % B, the window of output row gy+RW starts in
// slot RW % B; `o` points at this thread's pixel pair of that output row.  VEC: one unpredicated 64-bit store (the
// strip lies inside the image and the rows are 8-byte aligned); otherwise two predicated scalar stores.
template <int B, int RW, bool UNIFORM, bool VEC>
__device__ __forceinline__ void step(float2 (&H)[B][B], const float* __restrict__ Lbuf, int tid, float we, float wt,
                                     float* __restrict__ o, bool ok0, bool ok1)
{
    xpass<B, (RW + B - 1) % B>(H, Lbuf + RW * LWP, tid);
    const float2 e = ypass<B, RW % B, UNIFORM>(H, we, wt);
    if (VEC) {
        *reinterpret_cast<float2*>(o) = e;
    } else {
        asm volatile("{\n.reg .pred p, q;\nsetp.ne.b32 p, %3, 0;\nsetp.ne.b32 q, %4, 0;\n@p st.global.f32 [%0], %1;\n@q st.global.f32 [%0+4], %2;\n}" ::"l"(o), "f"(e.x), "f"(e.y), "r"((int) ok0), "r"((int) ok1) : "memory");
    }
}

// six CTAs per SM for both block sizes (b=4: 80 registers, 19.0 -> 18.3 us per 4K frame against five CTAs at 96 registers)
template <int B, bool UNIFORM, int CH>
__global__ void __launch_bounds__(NT, 6) dctc_k1_small_kernel(const DctcK1Args a, int seg_rows, int vec_ok)
{
    // programmatic dependent launch: back-to-back launches hide each other's launch latency; nothing is read or written
    // before the predecessor in the stream has completed
    DCTC_PDL_PROLOGUE();
    using G = RawGeom<CH>;
    constexpr int R0 = B / 2 - 1, R1 = B / 2;
    __shared__ __align__(16) float L[2][8 * LWP];
    __shared__ __align__(16) uint8_t Raw[3][8 * G::ROW];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * MW;
    const int y0 = blockIdx.y * seg_rows;                       // first output row of this segment (multiple of 8)
    const int y1 = min(y0 + seg_rows, a.h);
    const uint8_t* __restrict__ img = a.img + (size_t) blockIdx.z * a.frame_stride;
    float* __restrict__ out = a.out + (size_t) blockIdx.z * a.out_frame_stride;
    const int gx = x0 + 2 * tid;
    const bool ok0 = gx < a.w, ok1 = gx + 1 < a.w;
    const bool vec = vec_ok && x0 + MW <= a.w;                  // CTA-uniform
    float2 H[B][B];
    const float lscale = CH == 3 ? LUMA_INT_SCALE : 1.0f;       // RGB luma is 10000 x the 0..255 luma
    const float we = a.w_edges * lscale, wt = a.w_textures * lscale;
    ConvMap<CH> cm;
    cm.init(a, x0, tid);

    // chunk 0 = virtual rows y0-R0 .. (only the first B-1 are used: prologue); chunk c >= 1 = rows y0+R1+8(c-1) .. +7,
    // which feed output rows y0+8(c-1) .. +7.  Raw buffers rotate over three slots (two chunks in flight).
    const int nchunks = 1 + (y1 - y0 + 7) / 8;
    StageMap<CH> sm;
    sm.init(a, x0, tid);
    sm.stage(a, img, Raw[0], y0 - R0, x0, tid, B - 1);           // the prologue needs B-1 rows only
    sm.stage(a, img, Raw[1], y0 + R1, x0, tid);
    if (nchunks > 2) sm.stage(a, img, Raw[2], y0 + R1 + 8, x0, tid);
    else asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    __syncthreads();
    cm.template convert<B - 1>(a, Raw[0], L[0], x0, tid);
    __syncthreads();
    if (B == 4) {
        xpass<B, 0>(H, L[0] + 0 * LWP, tid);
        xpass<B, 1 % B>(H, L[0] + 1 * LWP, tid);
        xpass<B, 2 % B>(H, L[0] + 2 * LWP, tid);
    } else {
        xpass<B, 0>(H, L[0] + 0 * LWP, tid);
    }
    int slot = 1;                                               // raw buffer of the chunk being converted next
    for (int c = 1; c < nchunks; c++) {
        const int gy = y0 + 8 * (c - 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");   // this thread's copies of chunk c have landed
        __syncthreads();                                        // ... everybody's; L[c&1] and the raw buffer of chunk c-1 are free
        // refill the raw buffer chunk c-1 sat in with chunk c+2
        const int fslot = slot == 0 ? 2 : slot - 1;
        if (c + 2 < nchunks) sm.stage(a, img, Raw[fslot], y0 + R1 + 8 * (c + 1), x0, tid);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        float* Lb = L[c & 1];
        cm.template convert<8>(a, Raw[slot], Lb, x0, tid);
        __syncthreads();
        // one pointer per chunk, advanced by the pitch: no 64-bit multiply and no divergent guard per pixel
        float* o = out + (size_t) gy * a.out_pitch + gx;
        const size_t op = a.out_pitch;
        if (vec && gy + 8 <= a.h) {
            step<B, 0, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 1, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 2, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 3, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 4, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 5, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 6, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true); o += op;
            step<B, 7, UNIFORM, true>(H, Lb, tid, we, wt, o, true, true);
        } else {
#define DCTC_ROW(RW) { const bool rok = gy + RW < a.h; step<B, RW, UNIFORM, false>(H, Lb, tid, we, wt, o, ok0 && rok, ok1 && rok); o += op; }
            DCTC_ROW(0) DCTC_ROW(1) DCTC_ROW(2) DCTC_ROW(3) DCTC_ROW(4) DCTC_ROW(5) DCTC_ROW(6) DCTC_ROW(7)
#undef DCTC_ROW
        }
        slot = slot == 2 ? 0 : slot + 1;
    }
}

template <int B>
cudaError_t launch_small(const DctcK1Args& a, int n_frames, bool uniform, int sm_count, cudaStream_t stream)
{
    const int strips = (a.w + MW - 1) / MW;
    // segment height: long segments amortise the prologue, short ones fill the machine for small inputs
    // (measured on 64 / 16 frames of 4K per launch: b=2 64 rows 9.2 / 9.6 us per frame, 128 rows 9.3 / 9.8, 256 rows 9.6 / 9.8;
    //  b=4 64 rows 18.5 / 19.0, 128 rows 18.3 / 19.2, 256 rows 18.6 / 19.2)
    int seg = B == 2 ? 64 : 128;
    while (seg > 16 && (long long) strips * ((a.h + seg - 1) / seg) * n_frames < 16LL * sm_count) seg >>= 1;
    const int segs = (a.h + seg - 1) / seg;
    if (segs > 65535 || n_frames > 65535) return cudaErrorInvalidConfiguration;
    // 64-bit stores need 8-byte aligned output rows
    const int vec_ok = (((uintptr_t) a.out & 7) == 0 && (a.out_pitch & 1) == 0 && (a.out_frame_stride & 1) == 0) ? 1 : 0;
    dim3 grid(strips, segs, n_frames), block(NT);
    const cudaError_t e = dctc_dispatch<3, 1>(uniform, a.channels, [&](auto U, auto C) {
        return dctc_launch_pdl(dctc_k1_small_kernel<B, U, C>, grid, block, 0, stream, true, a, seg, vec_ok);
    });
    return e != cudaSuccess ? e : cudaGetLastError();
}

}  // namespace

// Block size 2 or 4, full maps (no band / preview mode) in the fast layout (dctc_k1_fast_layout)
cudaError_t dctc_launch_k1_small(const DctcK1Args& a, int blocksize, int n_frames, bool uniform, int sm_count, cudaStream_t stream)
{
    if (a.w <= 0 || a.h <= 0 || n_frames <= 0) return cudaSuccess;
    return blocksize == 2 ? launch_small<2>(a, n_frames, uniform, sm_count, stream) : launch_small<4>(a, n_frames, uniform, sm_count, stream);
}

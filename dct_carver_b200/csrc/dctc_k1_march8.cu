// K1 (block size 8, fast path): register-marching column kernel, FP32 with packed FP32x2 math.
//
// Same operator as dctc_k1_tile.cu (reference chain src/render.c:134-157 -> src/dct.c:77-110), restructured so that
// the x-pass coefficients never touch shared memory:
//   * a CTA owns a strip of 128 columns and marches down SEG rows; thread t owns column x0+t
//   * per new image row the thread runs ONE 1-D DCT along x (8 luma taps from a small staged luma row block in
//     smem) and keeps the 8 coefficients of the last 8 rows in a register ring H2[slot][pair] (k1 pairs packed
//     as float2: 64 registers)
//   * the y-pass is 4 packed DCT-8 (FFMA2/FADD2/FMUL2, two k1 planes per instruction) straight from registers,
//     followed by the |.|-max fold (FMNMX3) and one coalesced float store
// Per pixel: 8 LDS + 36 FP32 + 144 FP32x2 + 32 FMNMX3 (+ staging) vs 516 lane instructions of the tile kernel.
// The luma rows are staged 8 at a time (double buffered) with the reference's coordinate clamp
// (src/render.c:122-132) applied while staging, so band halos / image borders cost nothing in the main loop.
#include "dctc_common.cuh"
#include "dctc_launch.h"

namespace {

constexpr int MW = 128;       // columns per CTA (= threads)
constexpr int LWP = MW + 8;   // staged luma row: columns x0-3 .. x0+MW+4, padded to 136

template <bool UNIFORM>
struct Fold;

template <>
struct Fold<true> {
    float m;
    __device__ __forceinline__ void init() { m = 0.0f; }
    // X = (T[2p][k2], T[2p+1][k2]) for k2 = 0..7
    template <int PAIR>
    __device__ __forceinline__ void add(const float2* X)
    {
#pragma unroll
        for (int k2 = 0; k2 < 8; k2++) {
            if (PAIR == 0 && k2 == 0) m = fmaxf(m, fabsf(X[0].y));  // skip the DC term T[0][0]
            else m = fmaxf(m, fmaxf(fabsf(X[k2].x), fabsf(X[k2].y)));
        }
    }
    __device__ __forceinline__ float result(float we, float wt) const { (void) we; return m * wt; }
};

template <>
struct Fold<false> {  // same last-arg-max rule as DctcTracker<false>
    float a, mm, bv, z;
    __device__ __forceinline__ void init() { a = 0.0f; mm = -1.0f; bv = 0.0f; z = 0.0f; }
    template <int PAIR>
    __device__ __forceinline__ void add(const float2* X)
    {
        if (PAIR == 0) {  // .x is k1 = 0, .y is k1 = 1
            a = fabsf(X[1].x);
            bv = fabsf(X[0].y);
#pragma unroll
            for (int k2 = 2; k2 < 8; k2++) mm = fmaxf(mm, fabsf(X[k2].x));
#pragma unroll
            for (int k2 = 1; k2 < 8; k2++) z = fmaxf(z, fabsf(X[k2].y));
        } else {
#pragma unroll
            for (int k2 = 0; k2 < 8; k2++) z = fmaxf(z, fmaxf(fabsf(X[k2].x), fabsf(X[k2].y)));
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

// stage 8 luma rows (virtual rows vy0 .. vy0+7) of the strip into L[8][LWP]
__device__ __forceinline__ void stage_rows(const DctcK1Args& a, const uint8_t* __restrict__ img, float* __restrict__ L,
                                           int vy0, int x0, int tid)
{
    for (int i = tid; i < 8 * (MW + 7); i += MW) {
        const int ly = i / (MW + 7), lx = i - ly * (MW + 7);
        const int gx = max(0, min(x0 + lx - 3, a.w - 1));
        const uint8_t* row = dctc_row_ptr(a, img, vy0 + ly);
        L[ly * LWP + lx] = dctc_luma255(row + (size_t) gx * a.channels, a.channels);
    }
}

// ---- asynchronous staging (fast path: CH = 1 or 3, every row pointer and pitch 16-byte aligned) --------------
// The raw interleaved bytes [x0*CH-16, x0*CH+(MW+4)*CH) of 8 rows are copied global -> shared with 16-byte cp.async
// one chunk ahead of their conversion, so no thread waits on HBM in the main loop (x0*CH is 16-byte aligned because
// x0 is a multiple of 128).  Chunks outside [0, pitch) are skipped: clamped pixel indices never read them.
template <int CH>
struct RawGeom {
    static constexpr int CHUNKS = (16 + (MW + 4) * CH + 15) / 16;   // 16-byte chunks per row (CH=3: 26, CH=1: 10)
    static constexpr int ROW = CHUNKS * 16;                         // bytes per staged raw row
};

template <int CH>
__device__ __forceinline__ void stage_raw_async(const DctcK1Args& a, const uint8_t* __restrict__ img, uint8_t* __restrict__ R,
                                                int vy0, int x0, int tid)
{
    const int warp = tid >> 5, lane = tid & 31;
    if (lane < RawGeom<CH>::CHUNKS) {
        const long long gb = (long long) x0 * CH - 16 + 16 * lane;   // byte offset of this chunk inside the row
        if (gb >= 0 && gb + 16 <= (long long) a.pitch) {
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const int ly = 2 * warp + r;
                const uint8_t* src = dctc_row_ptr(a, img, vy0 + ly) + gb;
                const uint32_t dst = (uint32_t) __cvta_generic_to_shared(R + ly * RawGeom<CH>::ROW + 16 * lane);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
            }
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int CH>
__device__ __forceinline__ float luma_raw(const uint8_t* __restrict__ p)
{
    if (CH == 3) return fmaf(0.2126f, (float) p[0], fmaf(0.7152f, (float) p[1], 0.0722f * (float) p[2]));
    return (float) p[0];
}

template <int CH>
__device__ __forceinline__ void convert_raw(const DctcK1Args& a, const uint8_t* __restrict__ R, float* __restrict__ L, int x0, int tid)
{
    // staged luma column lx <-> image column clamp(x0 + lx - 3); raw byte of pixel gx = (gx - x0)*CH + 16
    const int b0 = (max(0, min(x0 + tid - 3, a.w - 1)) - x0) * CH + 16;
#pragma unroll
    for (int ly = 0; ly < 8; ly++) L[ly * LWP + tid] = luma_raw<CH>(R + ly * RawGeom<CH>::ROW + b0);
    if (tid < 56) {
        const int ly = tid / 7, lx = MW + tid - ly * 7;
        const int b1 = (max(0, min(x0 + lx - 3, a.w - 1)) - x0) * CH + 16;
        L[ly * LWP + lx] = luma_raw<CH>(R + ly * RawGeom<CH>::ROW + b1);
    }
}

// L1 prefetch of the cache lines the staging of rows vy0..vy0+7 will touch (no registers held, no stall):
// issued one chunk ahead so that stage_rows' byte loads hit L1 instead of waiting on HBM.
__device__ __forceinline__ void prefetch_rows(const DctcK1Args& a, const uint8_t* __restrict__ img, int vy0, int x0, int tid)
{
    if (tid < 8 * 5) {
        const int ly = tid / 5, l = tid - ly * 5;
        const int b0 = max(0, x0 - 3) * a.channels, b1 = min(a.w, x0 + MW + 4) * a.channels - 1;
        const uint8_t* p = dctc_row_ptr(a, img, vy0 + ly) + min(b0 + l * 128, b1);
        asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
    }
}

// x-pass of one staged row into ring slot SLOT
template <int SLOT>
__device__ __forceinline__ void xpass(float2 (&H2)[8][4], const float* __restrict__ Lrow, int tid)
{
    float v[8], X[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = Lrow[tid + j];
    dctc_dct_fwd<8>(v, X);
#pragma unroll
    for (int p = 0; p < 4; p++) H2[SLOT][p] = make_float2(X[2 * p], X[2 * p + 1]);
}

// y-pass over the window whose oldest row sits in ring slot J (rows J, J+1, .., J+7 mod 8)
template <int J, bool UNIFORM>
__device__ __forceinline__ float ypass(const float2 (&H2)[8][4], float we, float wt)
{
    Fold<UNIFORM> f;
    f.init();
    {
        float2 v[8], X[8];
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = H2[(J + i) & 7][0];
        dctc_dct_fwd2<8>(v, X);
        f.template add<0>(X);
    }
#pragma unroll
    for (int p = 1; p < 4; p++) {
        float2 v[8], X[8];
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = H2[(J + i) & 7][p];
        dctc_dct_fwd2<8>(v, X);
        f.template add<1>(X);
    }
    return f.result(we, wt);
}

template <int J, bool UNIFORM>
__device__ __forceinline__ void step(float2 (&H2)[8][4], const float* __restrict__ Lbuf, int tid, const DctcK1Args& a,
                                     float* __restrict__ out, int gx, int gy)
{
    // new image row gy+4 arrives in ring slot (J+7)&7; the window for output row gy is slots J..J+7
    xpass<(J + 7) & 7>(H2, Lbuf + J * LWP, tid);
    const float e = ypass<J, UNIFORM>(H2, a.w_edges, a.w_textures);
    if (gx < a.w && gy < a.h) out[(size_t) gy * a.out_pitch + gx] = e;
}

template <bool UNIFORM, int CH>   // CH = 1 or 3: asynchronous fast path; CH = 0: generic staging (any channels / alignment)
__global__ void __launch_bounds__(MW, 4) dctc_k1_march8_kernel(const DctcK1Args a, int seg_rows)
{
    constexpr bool FAST = CH != 0;
    constexpr int CHX = FAST ? CH : 1;
    __shared__ float L[2][8 * LWP];
    __shared__ __align__(16) uint8_t Raw[FAST ? 2 : 1][FAST ? 8 * RawGeom<CHX>::ROW : 16];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * MW;
    const int y0 = blockIdx.y * seg_rows;                       // first output row of this segment (multiple of 8)
    const int y1 = min(y0 + seg_rows, a.h);
    const uint8_t* __restrict__ img = a.img + (size_t) blockIdx.z * a.frame_stride;
    float* __restrict__ out = a.out + (size_t) blockIdx.z * a.out_frame_stride;
    const int gx = x0 + tid;
    float2 H2[8][4];

    if (FAST) {
        // chunk k = virtual rows y0-3+8k .. ; chunk 0 is the prologue (7 rows used), chunk c+1 feeds output rows y0+8c..
        stage_raw_async<CHX>(a, img, Raw[0], y0 - 3, x0, tid);
        stage_raw_async<CHX>(a, img, Raw[1], y0 + 4, x0, tid);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        convert_raw<CHX>(a, Raw[0], L[0], x0, tid);
        __syncthreads();
        xpass<0>(H2, L[0] + 0 * LWP, tid);
        xpass<1>(H2, L[0] + 1 * LWP, tid);
        xpass<2>(H2, L[0] + 2 * LWP, tid);
        xpass<3>(H2, L[0] + 3 * LWP, tid);
        xpass<4>(H2, L[0] + 4 * LWP, tid);
        xpass<5>(H2, L[0] + 5 * LWP, tid);
        xpass<6>(H2, L[0] + 6 * LWP, tid);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                         // raw chunk 1 landed everywhere, L[0]/Raw[0] free
        if (y0 + 8 < y1) stage_raw_async<CHX>(a, img, Raw[0], y0 + 12, x0, tid);
        convert_raw<CHX>(a, Raw[1], L[1], x0, tid);
        __syncthreads();
        int buf = 1;                                             // L[buf] holds the rows for output chunk gy
        for (int gy = y0; gy < y1; gy += 8) {
            const float* Lb = L[buf];
            step<0, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 0);
            step<1, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 1);
            step<2, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 2);
            step<3, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 3);
            step<4, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 4);
            step<5, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 5);
            step<6, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 6);
            step<7, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 7);
            if (gy + 8 >= y1) break;
            // rows for the next output chunk were copied into Raw[buf ^ 1] during this chunk
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();                                     // copies visible, L[buf ^ 1] and Raw[buf] free
            if (gy + 16 < y1) stage_raw_async<CHX>(a, img, Raw[buf], gy + 20, x0, tid);
            convert_raw<CHX>(a, Raw[buf ^ 1], L[buf ^ 1], x0, tid);
            __syncthreads();
            buf ^= 1;
        }
        return;
    }

    // prologue: rows y0-3 .. y0+3 -> ring slots 0..6 (the 8th staged row is not used)
    stage_rows(a, img, L[0], y0 - 3, x0, tid);
    __syncthreads();
    xpass<0>(H2, L[0] + 0 * LWP, tid);
    xpass<1>(H2, L[0] + 1 * LWP, tid);
    xpass<2>(H2, L[0] + 2 * LWP, tid);
    xpass<3>(H2, L[0] + 3 * LWP, tid);
    xpass<4>(H2, L[0] + 4 * LWP, tid);
    xpass<5>(H2, L[0] + 5 * LWP, tid);
    xpass<6>(H2, L[0] + 6 * LWP, tid);
    stage_rows(a, img, L[1], y0 + 4, x0, tid);                  // rows y0+4 .. y0+11 feed output rows y0 .. y0+7
    prefetch_rows(a, img, y0 + 12, x0, tid);
    __syncthreads();

    int buf = 1;
    for (int gy = y0; gy < y1; gy += 8) {
        // stage the next 8 rows while this chunk is consumed (the other buffer is free since the last barrier)
        if (gy + 8 < y1) stage_rows(a, img, L[buf ^ 1], gy + 12, x0, tid);
        if (gy + 16 < y1) prefetch_rows(a, img, gy + 20, x0, tid);
        const float* Lb = L[buf];
        step<0, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 0);
        step<1, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 1);
        step<2, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 2);
        step<3, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 3);
        step<4, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 4);
        step<5, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 5);
        step<6, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 6);
        step<7, UNIFORM>(H2, Lb, tid, a, out, gx, gy + 7);
        __syncthreads();
        buf ^= 1;
    }
}

}  // namespace

// Full maps (no band / preview mode) in any layout
cudaError_t dctc_launch_k1_march8(const DctcK1Args& a, int n_frames, bool uniform, cudaStream_t stream)
{
    if (a.w <= 0 || a.h <= 0 || n_frames <= 0) return cudaSuccess;
    const int strips = (a.w + MW - 1) / MW;
    // segment height: long segments amortise the 7-row prologue, short ones fill the machine for small inputs
    int seg = 128;
    while (seg > 16 && (long long) strips * ((a.h + seg - 1) / seg) * n_frames < 4LL * 148 * 2) seg >>= 1;
    const int segs = (a.h + seg - 1) / seg;
    if (segs > 65535 || n_frames > 65535) return cudaErrorInvalidConfiguration;
    dim3 grid(strips, segs, n_frames), block(MW);
    // C = 3 / 1 in the fast layout (rows readable for `pitch` bytes, all row pointers 16-byte aligned), else generic C = 0
    return dctc_dispatch<3, 1, 0>(uniform, dctc_k1_fast_layout(a) ? a.channels : 0, [&](auto U, auto C) {
        dctc_k1_march8_kernel<U, C><<<grid, block, 0, stream>>>(a, seg);
        return cudaGetLastError();
    });
}

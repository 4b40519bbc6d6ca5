// K1-TC16 (block size 16, full maps and row bands): the y-pass of the 16x16 block DCT on the 5th-generation tensor
// cores (tcgen05, sm_100a).  Same operator as the b = 16 instance of dctc_k1_tile.cu (reference chain
// src/render.c:134-157 -> src/dct.c:77-110 -> ddct16x16s, src/fft2d/shrtdct.c:238-386).
//
// Block size 16 needs 1938 FP32 flop per pixel on the CUDA cores (FP32-pipe floor ~216 us per 4K frame); 15/16 of them
// are the y-pass, which is a sliding-window contraction and therefore a Toeplitz GEMM:
//     D[lane][(i, k2)] = sum_y' A_k1[lane][y'] * Tz[y'][(i, k2)],   Tz[y'][(i, k2)] = B16[k2][y' - i]  (0 <= y' - i < 16)
// for the 16 output rows i of a step and the 31 window rows y' they read (K = 32 = two K = 16 MMAs, one per 16-row
// group of the operand ring).  FP32-grade accuracy from fp16 operands as in K1-TC (dctc_k1_tc8.cu): H = hi + lo,
// B16 = Bh + Bl, D = hi*Bh + lo*Bh + hi*Bl accumulated in FP32 in TMEM.
//
// One CTA per SM owns all 512 TMEM columns and marches down a strip of 64 pixel columns 16 rows ("a group") at a time.
// The 128 TMEM lanes are 64 columns x 2 PARITIES of k1: lane l holds the x-pass coefficients k1 = 2m + (l >> 6) of
// column l & 63, m = 0..7 -- a DCT-16 splits into an even half (sums v[j] + v[15-j]) and an odd half (differences)
// with no shared work, so nothing is computed twice and the operands of a step fill exactly half of TMEM:
//     A ring  256 columns: [m][hi|lo][slot g&1][row pair]   (8 columns = 16 rows = one K = 16 operand)
//     D tiles 2 x 128 columns: tile h holds k2 = 8h .. 8h+7 of the 16 output rows, column n = tc16_col(i, k2 & 7):
//       ordered [k2 & 7 = 1..7, 0][row], because the basis rows k2 = 0 and 8 (all entries +-1/4) are exact in fp16, their
//       Bl term is zero and the hi*Bl MMAs only cover the first 112 columns
// Per (step, m): 2 tiles x 2 groups x 3 split terms = 12 MMAs M128 N128 K16 (68.3 clk each): 6560 clk per 1024 px,
// i.e. a tensor floor of ~183 us per 4K frame -- and, unlike block size 8, everything else (x-pass 60, split 32, fold
// 128 FMNMX3 per pixel) fits in that shadow, so the roles are built for slack, not for instruction count:
//   converter warps 13-15: global loads -> EXACT integer luma (2126 R + 7152 G + 722 B, dp2a) * 2^-13 -> shared memory
//   producer warps 0-3 (thread = lane): packed FP32x2 DCT-16 along x per row pair (only the lane's parity half
//       survives dead-code elimination), hi / -lo split, operands of the whole group parked in shared memory; the TMEM
//       stores of each m wait for that m's "operands consumed" commit of step g-2 and are announced per m, so the
//       next step's first MMAs never wait for a store phase
//   MMA warp 12 (one elected thread)
//   consumer warpgroups 4-7 (tile 0) and 8-11 (tile 1): tcgen05.ld 128 accumulators, release the tile, fold |.|-max;
//       the four partial maxima of a pixel (2 tiles x 2 parities) meet in shared memory once per step.
// Steps are anchored to the global 16-row grid (DctcK1Args::row_origin), so a map does not depend on how the image was
// cut into segments or row bands: the FP32 accumulation order of a pixel is fixed by its global row.
#include <cuda_fp16.h>
#include <cstdio>
#include "dctc_common.cuh"
#include "dctc_launch.h"
#include "dctc_tc_tables.cuh"

namespace {

// -DDCTC_TC16_TIMING: per-role cycle accounting (clock64 deltas between marks), printed by CTA 0 when it retires
#ifdef DCTC_TC16_TIMING
struct TT { long long acc[5]; long long last; };
#define TT_DECL() TT tt = {{0, 0, 0, 0, 0}, clock64()}; const long long tt_start = tt.last
#define TT_ACC(k) { const long long tt_now = clock64(); tt.acc[k] += tt_now - tt.last; tt.last = tt_now; }
#define TT_REPORT(role, cond)                                                                                          \
    if (blockIdx.x == 0 && (cond))                                                                                     \
        printf("role %d: total %lld clk, marks %lld %lld %lld %lld %lld\n", role, clock64() - tt_start, tt.acc[0], tt.acc[1], tt.acc[2], tt.acc[3], tt.acc[4])
#else
struct TT {};
#define TT_DECL() TT tt
#define TT_ACC(k)
#define TT_REPORT(role, cond)
#endif

constexpr int PW = 64;             // pixel columns per CTA
constexpr int LW = 80;             // staged luma row: index i <-> column x0 - 8 + i (1..79 are read)
constexpr int NQ = LW / 4;         // 4-pixel conversion tasks per row pair
constexpr int NTHREADS = 512;
constexpr int NCONV = 96;
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t TM_A = 0;       // (m*2 + part)*16 + slot*8 + pair
constexpr uint32_t TM_D = 256;     // two accumulator tiles of 128 columns
constexpr float LUMA_WEIGHT_SCALE = 8192.0f / 10000.0f;
// accumulator column of (output row i, k2 & 7): the k2 whose basis row is exact in fp16 (k2 & 7 == 0) comes last
__host__ __device__ constexpr int tc16_col(int i, int k2l) { return ((k2l + 7) & 7) * 16 + i; }

struct alignas(128) Tc16Smem {
    __half B[8][2048];               // Tz sub-operands [(v*2 + kh)*2 + h]: v = Bh/Bl, kh = K half (group), h = k2 half (tile)
    float2 L[2][8][LW];              // scaled luma of two groups: [buffer][row pair][column], .x = even row
    uint32_t stash[8][2][8][128];    // operands of one group: [m][hi|-lo][row pair][lane]
    float comb[2][8][16][PW];        // per-step partials: [step parity][plane][row][column]; planes 0-3: maxima of
                                     // (tile*2 + k1 parity); edges != textures also: 4 |T[0][1]|, 5/6 max|T[0][2..]| of
                                     // tile 0 / 1, 7 |T[1][0]| (the quantities of DctcTracker<false>)
    uint64_t bar_a_full[8], bar_a_free[8], bar_d_full[2];
    uint32_t tmem_base;
    int work;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_inval(uint32_t bar) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
// Bounded parity wait: a protocol error traps after ~2^22 failed attempts (seconds) instead of hanging the GPU.
#ifdef DCTC_TC16_DEBUG
__device__ __noinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag = 0)
{
    for (uint32_t n = 0;; n++) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        if (n > (1u << 18)) { printf("tc16 mbar timeout tag %d parity %u block %d thread %d\n", tag, parity, blockIdx.x, threadIdx.x); __trap(); }
    }
}
#else
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag = 0)
{
    (void) tag;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 n;\n"
        "mov.u32 n, 0;\n"
        "DCTC16_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC16_DONE;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC16_DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 p, n, 0x200000;\n"
        "@p bra DCTC16_WAIT;\n"
        "trap;\n"
        "DCTC16_DONE:\n"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
#endif
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// Named barriers: 2,3 accumulator tile released (128 consumers arrive, the MMA warp syncs); 5,6 luma buffer full
// (96 converters arrive, 128 producers sync); 7,8 luma buffer free; 11 partial maxima of a step written (256 consumers).
__device__ __forceinline__ void bar_tile_arrive(int t) { asm volatile("bar.arrive %0, 160;" ::"r"(2 + t) : "memory"); }
__device__ __forceinline__ void bar_tile_sync(int t) { asm volatile("bar.sync %0, 160;" ::"r"(2 + t) : "memory"); }
__device__ __forceinline__ void bar_lfull_arrive(int b) { asm volatile("bar.arrive %0, 224;" ::"r"(5 + b) : "memory"); }
__device__ __forceinline__ void bar_lfull_sync(int b) { asm volatile("bar.sync %0, 224;" ::"r"(5 + b) : "memory"); }
__device__ __forceinline__ void bar_lfree_arrive(int b) { asm volatile("bar.arrive %0, 224;" ::"r"(7 + b) : "memory"); }
__device__ __forceinline__ void bar_lfree_sync(int b) { asm volatile("bar.sync %0, 224;" ::"r"(7 + b) : "memory"); }
__device__ __forceinline__ void bar_comb_sync() { asm volatile("bar.sync 11, 256;" ::: "memory"); }

// shared-memory matrix descriptor, no swizzle, K-major (same layout as K1-TC: LBO = 128 B between the two K core
// matrices, SBO = 256 B between 8-row groups along N)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t) ((addr & 0x3FFFF) >> 4);
    d |= (uint64_t) ((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t) ((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t) 1 << 46;
    return d;
}
// kind::f16 instruction descriptor: D = F32, A = B = F16, both K-major, dense
__device__ __forceinline__ constexpr uint32_t make_idesc(int M, int N) { return (1u << 4) | ((uint32_t) (N >> 3) << 17) | ((uint32_t) (M >> 4) << 24); }
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void tmem_st_x4(uint32_t taddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
// 32 consecutive TMEM columns -> registers (no wait)
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t* v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}

// Luma: the EXACT integer 2126 R + 7152 G + 722 B (grey: 10000 v), below 2^22, times 2^-13 (exact) so that the x-pass
// coefficients stay inside the fp16 range of the hi/lo split; 8192 / 10000 is folded into the final weight.
template <int CH>
__device__ __forceinline__ float luma_px(const uint8_t* __restrict__ p)
{
    const uint32_t v = CH == 3 ? 2126u * p[0] + 7152u * p[1] + 722u * p[2] : 10000u * p[0];
    return (float) v * (1.0f / 8192.0f);
}
template <int CH>
__device__ __forceinline__ void luma_quad(const uint8_t* __restrict__ p, float (&l)[4])
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    if (CH == 3) {
        const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
        constexpr uint32_t CRG = (7152u << 16) | 2126u, CB = 722u;
        const uint32_t p1 = __byte_perm(w0, w1, 0x6543), p2 = __byte_perm(w1, w2, 0x5432), p3 = w2 >> 8;
        l[0] = (float) __dp2a_lo(CRG, w0, __dp2a_hi(CB, w0, 0u)) * (1.0f / 8192.0f);
        l[1] = (float) __dp2a_lo(CRG, p1, __dp2a_hi(CB, p1, 0u)) * (1.0f / 8192.0f);
        l[2] = (float) __dp2a_lo(CRG, p2, __dp2a_hi(CB, p2, 0u)) * (1.0f / 8192.0f);
        l[3] = (float) __dp2a_lo(CRG, p3, __dp2a_hi(CB, p3, 0u)) * (1.0f / 8192.0f);
    } else {
        const uint32_t w0 = __ldg(w);
#pragma unroll
        for (int i = 0; i < 4; i++) l[i] = (float) (10000u * ((w0 >> (8 * i)) & 255u)) * (1.0f / 8192.0f);
    }
}

// one group (16 virtual rows from vy0) -> luma row pairs; staged index i <-> image column clamp(x0 - 8 + i)
// (src/render.c:122-132); a task is one 4-pixel group of one row pair
template <int CH>
__device__ __forceinline__ void convert_group(const DctcK1Args& a, const uint8_t* __restrict__ img, int vy0, int x0, float2 (*__restrict__ L)[LW], int ct)
{
    for (int task = ct; task < 8 * NQ; task += NCONV) {
        const int p = task / NQ, q = task - p * NQ;
        const int gx = x0 - 8 + 4 * q;
        const uint8_t* r0 = dctc_row_ptr(a, img, vy0 + 2 * p);
        const uint8_t* r1 = dctc_row_ptr(a, img, vy0 + 2 * p + 1);
        float l0[4], l1[4];
        if (gx >= 0 && gx + 3 < a.w) {
            luma_quad<CH>(r0 + (size_t) gx * CH, l0);
            luma_quad<CH>(r1 + (size_t) gx * CH, l1);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const size_t off = (size_t) max(0, min(gx + k, a.w - 1)) * CH;
                l0[k] = luma_px<CH>(r0 + off);
                l1[k] = luma_px<CH>(r1 + off);
            }
        }
        float4* dst = reinterpret_cast<float4*>(&L[p][4 * q]);
        dst[0] = make_float4(l0[0], l1[0], l0[1], l1[1]);
        dst[1] = make_float4(l0[2], l1[2], l0[3], l1[3]);
    }
}

// H -> fp16 hi and fp16 MINUS lo for two vertically adjacent rows (low half = even row = even K index); see K1-TC
__device__ __forceinline__ void split_pair(float2 x, uint32_t& hi, uint32_t& nlo)
{
    const __half2 h = __floats2half2_rn(x.x, x.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const uint16_t h0 = (uint16_t) (hi & 0xffffu), h1 = (uint16_t) (hi >> 16);
    float r0, r1;
    asm("sub.rn.f32.f16 %0, %1, %2;" : "=f"(r0) : "h"(h0), "f"(x.x));
    asm("sub.rn.f32.f16 %0, %1, %2;" : "=f"(r1) : "h"(h1), "f"(x.y));
    const __half2 l = __floats2half2_rn(r0, r1);
    nlo = *reinterpret_cast<const uint32_t*>(&l);
}

// x-pass + split of group g (rows staged in s.L[g&1]) for this lane's parity, parked in s.stash; then, m by m, the
// TMEM stores into ring slot g&1 as soon as the MMAs of step g-2 have consumed that m
template <int PARITY>
__device__ __forceinline__ void produce_group(Tc16Smem& s, int g, int lane128, uint32_t tmem_lane, TT& tt)
{
    (void) tt;
    const int px = lane128 & (PW - 1);
    const float2 (*Lg)[LW] = s.L[g & 1];
#pragma unroll 2
    for (int p = 0; p < 8; p++) {
        float2 v[16], X[16];
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = Lg[p][px + 1 + j];
        if (p == 7) bar_lfree_arrive(g & 1);   // last read of this luma buffer
        dctc_dct_fwd2<16>(v, X);               // the other parity's outputs are dead code
#pragma unroll
        for (int m = 0; m < 8; m++) {
            uint32_t hi, nlo;
            split_pair(X[2 * m + PARITY], hi, nlo);
            s.stash[m][0][p][lane128] = hi;
            s.stash[m][1][p][lane128] = nlo;
        }
    }
    TT_ACC(2);
    const uint32_t ta = tmem_lane + TM_A + (uint32_t) (g & 1) * 8u;
    // the parked operands of m+1 are fetched while the stores of m complete
    uint32_t o[2][8], on[2][8];
#pragma unroll
    for (int part = 0; part < 2; part++)
#pragma unroll
        for (int p = 0; p < 8; p++) o[part][p] = s.stash[0][part][p][lane128];
#pragma unroll
    for (int m = 0; m < 8; m++) {
        if (g >= 2) {
            TT_ACC(3);
            mbar_wait(smem_u32(&s.bar_a_free[m]), (uint32_t) (g & 1), 100 + m);   // completion g-2 of this barrier
            TT_ACC(4);
            tc_fence_after();
        }
#pragma unroll
        for (int part = 0; part < 2; part++) {
            const uint32_t t = ta + (uint32_t) ((m * 2 + part) * 16);
            tmem_st_x4(t, o[part][0], o[part][1], o[part][2], o[part][3]);
            tmem_st_x4(t + 4u, o[part][4], o[part][5], o[part][6], o[part][7]);
        }
        if (m < 7) {
#pragma unroll
            for (int part = 0; part < 2; part++)
#pragma unroll
                for (int p = 0; p < 8; p++) on[part][p] = s.stash[m + 1][part][p][lane128];
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        // Group 0 is not announced on its own: the arrival of group 1 covers both (same thread, program order; wait::st
        // covers all earlier stores).  Completion j of this barrier is group j+1, which needs the "consumed" commit of
        // step j-1, issued after the MMA warp's wait for completion j-1: never more than one completion ahead.
        if (g >= 1 && (lane128 & 31) == 0) mbar_arrive(smem_u32(&s.bar_a_full[m]));   // 4 arrivals (one per producer warp)
#pragma unroll
        for (int part = 0; part < 2; part++)
#pragma unroll
            for (int p = 0; p < 8; p++) o[part][p] = on[part][p];
    }
}

// |.|-max of one accumulator tile into the 16 row maxima; DC: this lane holds k1 = 0 and the tile k2 = 0, whose
// product (0,0) is skipped (src/dct.c:101)
template <bool DC>
__device__ __forceinline__ void fold_tile(const uint32_t (&v)[128], float (&mx)[16])
{
#pragma unroll
    for (int i = 0; i < 16; i++) {
        float t = mx[i];
        if (DC) t = fmaxf(t, fabsf(__uint_as_float(v[tc16_col(i, 1)])));
        else t = fmaxf(t, fmaxf(fabsf(__uint_as_float(v[tc16_col(i, 0)])), fabsf(__uint_as_float(v[tc16_col(i, 1)]))));
#pragma unroll
        for (int k = 2; k < 8; k += 2)
            t = fmaxf(t, fmaxf(fabsf(__uint_as_float(v[tc16_col(i, k)])), fabsf(__uint_as_float(v[tc16_col(i, k + 1)]))));
        mx[i] = t;
    }
}

// edges != textures (last-arg-max class rule, DctcTracker<false>): the m = 0 tiles hold the row k1 = 0 (parity 0) and
// k1 = 1 (parity 1) of the coefficient matrix, whose entries the rule treats separately.  They are parked in shared
// memory right away (planes 4-7 of the step's comb buffer); everything else folds into the plain maximum Z.
//   KIND 0: k1 = 0, k2 = 0..7:  A = |T[0][1]| -> plane 4, max|T[0][2..7]| -> plane 5, (0,0) skipped
//   KIND 1: k1 = 0, k2 = 8..15: max -> plane 6
//   KIND 2: k1 = 1, k2 = 0..7:  Bv = |T[1][0]| -> plane 7, the rest -> Z
template <int KIND>
__device__ __forceinline__ void fold_tile_class(const uint32_t (&v)[128], float (&mx)[16], float (*__restrict__ cb)[16][PW], int px)
{
#pragma unroll
    for (int i = 0; i < 16; i++) {
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; k++) f[k] = fabsf(__uint_as_float(v[tc16_col(i, k)]));
        const float m27 = fmaxf(fmaxf(f[2], fmaxf(f[3], f[4])), fmaxf(f[5], fmaxf(f[6], f[7])));
        if (KIND == 0) {
            cb[4][i][px] = f[1];
            cb[5][i][px] = m27;
        } else if (KIND == 1) {
            cb[6][i][px] = fmaxf(m27, fmaxf(f[0], f[1]));
        } else {
            cb[7][i][px] = f[0];
            mx[i] = fmaxf(mx[i], fmaxf(m27, f[1]));
        }
    }
}

template <bool UNIFORM, int CH>
__global__ void __launch_bounds__(NTHREADS, 1) dctc_k1_tc16_kernel(const DctcK1Args a, int seg_rows, int strips, int segs, int n_items,
                                                                     int phase, int* __restrict__ counter)
{
    extern __shared__ __align__(128) uint8_t dctc_tc16_smem[];
    Tc16Smem& s = *reinterpret_cast<Tc16Smem*>(dctc_tc16_smem);
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler

    // programmatic dependent launch, as in dctc_k1_tc8.cu: this launch's ramp (TMEM allocation, Toeplitz operands from
    // immutable tables) overlaps the tail of the grid before it in the stream
    asm volatile("griddepcontrol.launch_dependents;");
    if (warp == 12) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // Toeplitz sub-operands as UMMA K-major no-swizzle tiles: element (n = tc16_col(i, k2l), k) of sub-operand (v, kh, h) is
    // B16[8h + k2l][16 kh + k - i] (zero outside the basis)
    {
        uint16_t* Bq = reinterpret_cast<uint16_t*>(&s.B[0][0]);
        for (int idx = tid; idx < 8 * 2048; idx += NTHREADS) {
            const int sub = idx >> 11, n = (idx >> 4) & 127, k = idx & 15;
            const int v = sub >> 2, kh = (sub >> 1) & 1, h = sub & 1;
            const int i = n & 15, k2 = 8 * h + (((n >> 4) + 1) & 7);
            const int c = 16 * kh + k - i;
            const uint16_t val = (c >= 0 && c < 16) ? DCTC_TC_BASIS16[v][k2 * 16 + c] : (uint16_t) 0;
            Bq[sub * 2048 + (n >> 3) * 128 + (k >> 3) * 64 + (n & 7) * 8 + (k & 7)] = val;
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");     // everything before this grid in the stream is complete and visible
    const uint32_t lane_off = (uint32_t) ((warp & 3) * 32) << 16;

    auto begin_item = [&](bool first) -> int {
        if (tid == 0) {
            // n_items + gridDim.x fetches in all: the wrapping increment leaves the counter at 0 for the next launch
            s.work = (int) atomicInc(reinterpret_cast<unsigned int*>(counter), (unsigned int) n_items + gridDim.x - 1u);
            for (int m = 0; m < 8; m++) {
                if (!first) { mbar_inval(smem_u32(&s.bar_a_full[m])); mbar_inval(smem_u32(&s.bar_a_free[m])); }
                mbar_init(smem_u32(&s.bar_a_full[m]), 4);
                mbar_init(smem_u32(&s.bar_a_free[m]), 1);
            }
            for (int h = 0; h < 2; h++) {
                if (!first) mbar_inval(smem_u32(&s.bar_d_full[h]));
                mbar_init(smem_u32(&s.bar_d_full[h]), 1);
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        return s.work;
    };
    auto end_item = [&]() {
        tc_fence_before();
        __syncthreads();    // every role is done with the barriers, TMEM and staging buffers of this item
    };
    // item -> (frame, segment, strip); rows Y0 .. Y0 + seg_rows of the band, Y0 + row_origin a multiple of 16
#define DCTC16_ITEM_LOOP                                                                                               \
    for (bool first = true;; first = false) {                                                                          \
        const int item = begin_item(first);                                                                            \
        if (item >= n_items) break;                                                                                    \
        const uint32_t tmem = s.tmem_base;                                                                             \
        const uint32_t tmem_lane = tmem + lane_off;                                                                    \
        const int strip = item % strips;                                                                               \
        const int rest = item / strips;                                                                                \
        const int seg = rest % segs, frame = rest / segs;                                                              \
        const int x0 = strip * PW;                                                                                     \
        const int Y0 = seg * seg_rows - phase;                                                                         \
        const int y1 = min(Y0 + seg_rows, a.h);                                                                        \
        const int nsteps = (y1 - Y0 + 15) >> 4;                                                                        \
        const uint8_t* __restrict__ img = a.img + (size_t) frame * a.frame_stride;                                     \
        float* __restrict__ out = a.out + (size_t) frame * a.out_frame_stride;                                         \
        (void) tmem; (void) tmem_lane; (void) x0; (void) y1; (void) img; (void) out;

    TT_DECL();
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 104;");
        DCTC16_ITEM_LOOP
        // ===== producers: group g = virtual rows Y0-7+16g .. Y0+8+16g; step j consumes groups j and j+1 =====
        for (int g = 0; g <= nsteps; g++) {
            TT_ACC(0);
            bar_lfull_sync(g & 1);
            TT_ACC(1);
            if (warp < 2) produce_group<0>(s, g, tid, tmem_lane, tt);
            else produce_group<1>(s, g, tid, tmem_lane, tt);
            TT_ACC(3);
        }
        end_item();
        }
        TT_REPORT(0, tid == 0);
    } else if (warp < 12) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
        DCTC16_ITEM_LOOP
        // ===== consumers: warpgroup h folds tile h =====
        const int h = (warp - 4) >> 2;
        const int lane128 = tid & 127;
        const int px = lane128 & (PW - 1), parity = lane128 >> 6;
        const int ctid = tid - 128;                            // 0..255
        const float wgt = a.w_textures * LUMA_WEIGHT_SCALE, wge = a.w_edges * LUMA_WEIGHT_SCALE;
        (void) wge;
        for (int st = 0; st < nsteps; st++) {
            float mx[16];
#pragma unroll
            for (int i = 0; i < 16; i++) mx[i] = 0.0f;
#pragma unroll 1
            for (int m = 0; m < 8; m++) {
                TT_ACC(0);
                mbar_wait(smem_u32(&s.bar_d_full[h]), (uint32_t) (m & 1), 200 + 10 * h + m);   // completion 8 st + m
                TT_ACC(1);
                tc_fence_after();
                uint32_t v[128];
                const uint32_t td = tmem_lane + TM_D + 128u * (uint32_t) h;
                tmem_ld_x32(td, v);
                tmem_ld_x32(td + 32u, v + 32);
                tmem_ld_x32(td + 64u, v + 64);
                tmem_ld_x32(td + 96u, v + 96);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                tc_fence_before();
                TT_ACC(2);
                bar_tile_arrive(h);
                if (UNIFORM) {
                    if (m == 0 && h == 0 && parity == 0) fold_tile<true>(v, mx);
                    else fold_tile<false>(v, mx);
                } else {
                    if (m == 0 && parity == 0) {
                        if (h == 0) fold_tile_class<0>(v, mx, s.comb[st & 1], px);
                        else fold_tile_class<1>(v, mx, s.comb[st & 1], px);
                    } else if (m == 0 && h == 0) {
                        fold_tile_class<2>(v, mx, s.comb[st & 1], px);
                    } else {
                        fold_tile<false>(v, mx);
                    }
                }
                TT_ACC(3);
            }
            float (*cb)[16][PW] = s.comb[st & 1];
#pragma unroll
            for (int i = 0; i < 16; i++) cb[h * 2 + parity][i][px] = mx[i];
            bar_comb_sync();
            const int gy0 = Y0 + 16 * st;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int idx = ctid + 256 * q;
                const int i = idx >> 6, c = idx & (PW - 1);
                const float z = fmaxf(fmaxf(cb[0][i][c], cb[1][i][c]), fmaxf(cb[2][i][c], cb[3][i][c]));
                float e;
                if (UNIFORM) {
                    e = z * wgt;
                } else {   // DctcTracker<false>::result
                    const float av = cb[4][i][c], mm = fmaxf(cb[5][i][c], cb[6][i][c]), bv = cb[7][i][c];
                    const float am = fmaxf(av, mm);
                    const float top = fmaxf(fmaxf(am, bv), z);
                    const bool tex = (z >= fmaxf(am, bv)) || (!(bv >= am) && (mm >= av));
                    e = top * (tex ? wgt : wge);
                }
                const int gy = gy0 + i, gx = x0 + c;
                if (gy >= 0 && gy < y1 && gx < a.w) out[(size_t) gy * a.out_pitch + gx] = e;
            }
        }
        end_item();
        }
        TT_REPORT(1, tid == 128 || tid == 256);
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 12) {
        DCTC16_ITEM_LOOP
        // ===== MMA issuer =====
        const uint32_t idesc = make_idesc(128, 128);
        const uint32_t idesc_bl = make_idesc(128, 112);          // hi*Bl: the columns of k2 & 7 == 0 (Bl = 0) are skipped
        const uint64_t bd0 = make_smem_desc(smem_u32(&s.B[0][0]), 128, 256);   // sub-operand stride: 4096 B = 256 address units
        for (int st = 0; st < nsteps; st++) {
            const uint32_t so = (uint32_t) (st & 1) * 8u, sn = so ^ 8u;   // ring slots of the older / newer group
#pragma unroll 1
            for (int m = 0; m < 8; m++) {
                TT_ACC(0);
                mbar_wait(smem_u32(&s.bar_a_full[m]), (uint32_t) (st & 1), 400 + m);    // completion st: groups <= st+1 stored
                TT_ACC(1);
                tc_fence_after();
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    TT_ACC(1);
                    if (st > 0 || m > 0) bar_tile_sync(h);     // the consumers have loaded the previous contents of tile h
                    TT_ACC(2);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t d = tmem + TM_D + 128u * (uint32_t) h;
                        const uint32_t ah = tmem + TM_A + (uint32_t) (m * 32), al = ah + 16u;
                        const uint64_t bh0 = bd0 + (uint64_t) (256 * ((0 * 2 + 0) * 2 + h)), bh1 = bd0 + (uint64_t) (256 * ((0 * 2 + 1) * 2 + h));
                        const uint64_t bl0 = bd0 + (uint64_t) (256 * ((1 * 2 + 0) * 2 + h)), bl1 = bd0 + (uint64_t) (256 * ((1 * 2 + 1) * 2 + h));
                        mma_ts(d, ah + so, bh0, idesc, 0u);
                        mma_ts(d, al + so, bh0, idesc | (1u << 13), 1u);   // A negated: the ring holds -lo
                        mma_ts(d, ah + so, bl0, idesc_bl, 1u);
                        mma_ts(d, ah + sn, bh1, idesc, 1u);
                        mma_ts(d, al + sn, bh1, idesc | (1u << 13), 1u);
                        mma_ts(d, ah + sn, bl1, idesc_bl, 1u);
                        mma_commit(smem_u32(&s.bar_d_full[h]));
                        if (h == 1 && st + 2 <= nsteps) mma_commit(smem_u32(&s.bar_a_free[m]));   // waited on by the producers of group st+2
                    }
                    __syncwarp();
                    TT_ACC(3);
                }
            }
        }
        // the last use of each tile was arrived on but never waited for: drain both named barriers
        bar_tile_sync(0);
        bar_tile_sync(1);
        end_item();
        }
        TT_REPORT(2, tid == 384);
        } else {
        DCTC16_ITEM_LOOP
        // ===== converters =====
        const int ct = tid - (NTHREADS - NCONV);
        for (int g = 0; g <= nsteps; g++) {
            if (g >= 2) bar_lfree_sync(g & 1);                 // the producers have read group g-2 out of this buffer
            convert_group<CH>(a, img, Y0 - 7 + 16 * g, x0, s.L[g & 1], ct);
            bar_lfull_arrive(g & 1);
        }
        // the last two groups' "free" arrivals were never waited for: drain them so the next item starts clean
        if (nsteps >= 1) bar_lfree_sync((nsteps - 1) & 1);
        bar_lfree_sync(nsteps & 1);
        end_item();
        }
        }
    }
#undef DCTC16_ITEM_LOOP

    if (warp == 12) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s.tmem_base), "r"(TMEM_COLS));
}

}  // namespace

// Full maps (no band / preview mode) in the fast layout (dctc_k1_fast_layout); `counter` as for dctc_launch_k1_tc8.
cudaError_t dctc_launch_k1_tc16(const DctcK1Args& a, int n_frames, bool uniform, int* counter, int sm_count, cudaStream_t stream)
{
    if (a.w <= 0 || a.h <= 0 || n_frames <= 0) return cudaSuccess;
    const int strips = (a.w + PW - 1) / PW;
    const int phase = a.row_origin & 15;
    const int rows = a.h + phase;
    // Segment height: an item of S rows costs S/16 + 2 groups of producer work and S/16 tensor steps; one CTA per SM
    // takes items from a counter.  Few items: minimise rounds x steps; many: ~432-row segments (7 % prologue).
    const long long ctas = sm_count;
    auto even_seg = [&](int nseg) { return (((rows + nseg - 1) / nseg) + 15) & ~15; };
    int best_rows = even_seg(1);
    long long best_cost = -1;
    const int max_segs = (rows + 31) / 32;
    for (int nseg = 1; nseg <= max_segs && nseg <= 64; nseg++) {
        const int sr = even_seg(nseg);
        const long long sg = (rows + sr - 1) / sr, it = (long long) strips * sg * n_frames;
        const long long per = sr / 16 + 2;   // the two prologue groups of an item cost about two steps
        const long long rounds = (it + ctas - 1) / ctas;
        const long long cost = it <= 8 * ctas ? rounds * per : (it * per + ctas - 1) / ctas + per / 2;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_rows = sr; }
    }
    const int seg = best_rows;
    const int segs = (rows + seg - 1) / seg;
    const long long items = (long long) strips * segs * n_frames;
    if (items > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
    const int grid = (int) (items < ctas ? items : ctas);
    const int smem = (int) sizeof(Tc16Smem);
    const cudaError_t e = dctc_dispatch<3, 1>(uniform, a.channels, [&](auto U, auto C) {
        const cudaError_t ea = cudaFuncSetAttribute(dctc_k1_tc16_kernel<U, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (ea != cudaSuccess) return ea;
        return dctc_launch_pdl(dctc_k1_tc16_kernel<U, C>, dim3(grid), dim3(NTHREADS), (size_t) smem, stream, true, a, seg, strips, segs,
                               (int) items, phase, counter);
    });
    return e != cudaSuccess ? e : cudaGetLastError();
}

// K1-TC (block size 8, full maps): the y-pass of the block DCT on the 5th-generation tensor cores (tcgen05, sm_100a).
//
// Same operator as dctc_k1_march8.cu / dctc_k1_tile.cu (reference chain src/render.c:134-157 -> src/dct.c:77-110 ->
// ddct8x8s, src/fft2d/shrtdct.c:61-117).  A CTA owns a strip of 128 columns and marches down its segment 8 rows
// ("a group") at a time; pixel column x0+m is row m of every MMA (TMEM lane m).
//
//   converter warps 9-11: stage the raw rows two groups ahead (triple-buffered): the 8 x 416-byte tile of a group that
//       lies inside the image is ONE 3-D tensor copy (TMA, cp.async.bulk.tensor.3d over (row bytes / 4, rows, frames),
//       completion on the buffer's mbarrier); groups that touch the top / bottom edge or the halo rows of a band (edge
//       replication, src/render.c:122-132) are gathered row by row with 16-byte cp.async.  Then convert one group to luma
//       (four pixels x two rows per task: 32-bit shared loads, exact integer luma by dp2a, four I2F) and
//       hand the luma row pairs to the producers through hardware named barriers (double-buffered)
//   producer warps 0-3 (thread = column): run the
//       x-pass (one packed FP32x2 DCT-8 per row pair), split each coefficient H[k1] into fp16 hi + fp16 lo
//       (hi = rn16(H), lo = rn16(H - hi): 22 significant bits) and store the group into the TMEM A operand ring
//       with tcgen05.st: columns [k1][hi|lo][slot g&1][row pair], two consecutive rows per 32-bit column
//   MMA warp 8 (one elected thread): for every k1, D[128 x 64] = A_k1[128 x 16] * Tz[16 x 64] with
//       Tz[y'][(i,k2)] = B8[k2][y'-i] (Toeplitz expansion of the DCT basis: output row i of the group reads window
//       rows i..i+7 of the 16 staged rows), as three kind::f16 MMAs with FP32 accumulation in TMEM:
//       hi*Bh + lo*Bh + hi*Bl (the dropped lo*Bl term is 2^-22 relative).  Odd steps use the K-swapped copy of Tz
//       because the older group then sits in ring slot 1.
//       The basis is stored times 2*sqrt(2) (dctc_tc_tables.cuh): its rows k2 = 0 and 4 are then +-1 exactly, their Bl
//       term is zero, and the accumulator columns are ordered [k2 = 1,2,3,5,6,7,0,4][row] so that the hi*Bl MMA only
//       covers the first 48 columns (N = 48).
//   consumer warps 4-7 (thread = column): tcgen05.ld the 64 accumulators of (8 rows x 8 k2), fold |.|-max over k2
//       and k1 with FMNMX3 (or the last-arg-max class tracker when edges != textures), scale, coalesced store.
//
// Per pixel the CUDA cores execute ~120 instructions instead of the ~264 of the FP32 march kernel; the tensor pipe
// does 24 M128 K16 MMAs per 1024 pixels (16 with N = 64: 36.3 clk each measured, profiles/r01_tcgen05_probe2.txt; 8 with
// N = 48).  The operands of a group are announced in two halves (k1 = 0..3, 4..7).
#include <cuda_fp16.h>
#include <cstdio>
#include <cstring>
#include "dctc_common.cuh"
#include "dctc_launch.h"
#include "dctc_tc_tables.cuh"

#ifndef DCTC_TC_ABL
#define DCTC_TC_ABL 0   // timing ablations only (wrong results): 1 fold one row of eight, 2 no x-pass / split
#endif
namespace {

// -DDCTC_TC_TIMING: per-role wait-cycle accounting (clock64), printed by CTA 0 when it retires (tools/time_tc.py)
#ifdef DCTC_TC_TIMING
#define TT_T0() const long long tt_b = clock64()
#define TT_ACC(role, k) g_tt_acc[k] += clock64() - tt_b
#define TT_DECL() long long g_tt_acc[4] = {0, 0, 0, 0}; const long long tt_start = clock64()
#define TT_REPORT(role, cond)                                                                                          \
    if (blockIdx.x == 0 && (cond))                                                                                     \
        printf("role %d: total %lld clk, waits %lld %lld %lld %lld\n", role, clock64() - tt_start, g_tt_acc[0], g_tt_acc[1], g_tt_acc[2], g_tt_acc[3])
#else
#define TT_T0()
#define TT_ACC(role, k)
#define TT_DECL() long long* const g_tt_acc = nullptr
#define TT_REPORT(role, cond)
#endif

constexpr int MW = 128;            // columns per CTA = MMA M
constexpr int LWP = MW + 8;        // staged luma row: index i <-> column x0-4+i (index 0 is a pad, 1..135 are read)
constexpr int NTHREADS = 384;      // 4 producer warps, 4 consumer warps, 1 MMA warp, 3 converter warps
constexpr int NCONV = 96;          // converter threads
constexpr int NQUAD = 34;          // 4-pixel groups per staged row: columns x0-4 .. x0+131
constexpr uint32_t TMEM_COLS = 256;
constexpr uint32_t TM_A = 0;       // A ring: (k1*2 + part)*8 + slot*4 + pair
constexpr uint32_t TM_D = 128;     // two accumulator tiles of 64 columns
constexpr int PAD_SMEM = 64 * 1024;  // dynamic shared memory requested only to cap residency at 2 CTAs/SM (2 x 256 TMEM columns)

template <int CH>
struct RawGeom {
    static constexpr int CHUNKS = (16 + (MW + 4) * CH + 15) / 16;   // 16-byte chunks per staged raw row
    static constexpr int ROW = CHUNKS * 16;
};

struct alignas(128) TcSmem {
    __half B[4][64 * 16];            // Tz as UMMA K-major no-swizzle operands: [0] Bh, [1] Bl, [2]/[3] the K-swapped copies
    float2 L[2][4][LWP];             // luma of two groups: [buffer][row pair][column], .x = even row
    uint8_t Raw[3][8 * RawGeom<3>::ROW];
    uint64_t bar_a_free, bar_a_free_lo, bar_d_full[2];
    uint64_t bar_raw[3];             // raw buffer filled: NCONV arrivals (+ the bytes of a tensor copy)
    uint32_t tmem_base;
    int work;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_inval(uint32_t bar) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
// Tight parity wait (labels are local to the braces).  try_wait suspends the warp in hardware for a bounded time per
// attempt; after 2^22 failed attempts (seconds) a protocol error traps, so the launch fails instead of hanging.
#ifdef DCTC_TC_DEBUG
__device__ __noinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag = 0)
{
    for (uint32_t n = 0;; n++) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        if (n > (1u << 20)) { printf("mbar timeout tag %d parity %u block %d thread %d\n", tag, parity, blockIdx.x, threadIdx.x); __trap(); }
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
        "DCTC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC_DONE;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC_DONE;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC_DONE;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCTC_DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 p, n, 0x100000;\n"
        "@p bra DCTC_WAIT;\n"
        "trap;\n"
        "DCTC_DONE:\n"
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
// Named barriers: 2,3 accumulator tiles; 4 converter threads; 5,6 luma buffer full; 7,8 luma buffer free; 9 step started
// (MMA warp -> consumers: they block here instead of polling bar_d_full during the producers' phase); 10 operands of a
// group stored (producers -> MMA warp).  A blocked bar.sync costs no issue slots, unlike an mbarrier poll loop.
__device__ __forceinline__ void bar_step_arrive() { asm volatile("bar.arrive 9, 160;" ::: "memory"); }
__device__ __forceinline__ void bar_step_sync() { asm volatile("bar.sync 9, 160;" ::: "memory"); }
// "operands stored" comes in two halves (k1 = 0..3 -> barrier 10, k1 = 4..7 -> barrier 11): the first four tiles of a step
// start while the producers still store the second half behind the previous step's last MMAs
__device__ __forceinline__ void bar_afull_arrive(int half) { asm volatile("bar.arrive %0, 160;" ::"r"(10 + half) : "memory"); }
__device__ __forceinline__ void bar_afull_sync(int half) { asm volatile("bar.sync %0, 160;" ::"r"(10 + half) : "memory"); }
__device__ __forceinline__ void bar_converters() { asm volatile("bar.sync 4, 96;" ::: "memory"); }
__device__ __forceinline__ void bar_lfull_arrive(int b) { asm volatile("bar.arrive %0, 224;" ::"r"(5 + b) : "memory"); }
__device__ __forceinline__ void bar_lfull_sync(int b) { asm volatile("bar.sync %0, 224;" ::"r"(5 + b) : "memory"); }
__device__ __forceinline__ void bar_lfree_arrive(int b) { asm volatile("bar.arrive %0, 224;" ::"r"(7 + b) : "memory"); }
__device__ __forceinline__ void bar_lfree_sync(int b) { asm volatile("bar.sync %0, 224;" ::"r"(7 + b) : "memory"); }
// Accumulator tile t is handed back to the MMA warp through hardware named barrier 2+t (4 consumer warps arrive, the
// MMA warp syncs: 160 threads): the wake-up is immediate, unlike polling an mbarrier from the issuing thread.
__device__ __forceinline__ void bar_tile_arrive(int t) { asm volatile("bar.arrive %0, 160;" ::"r"(2 + t) : "memory"); }
__device__ __forceinline__ void bar_tile_sync(int t) { asm volatile("bar.sync %0, 160;" ::"r"(2 + t) : "memory"); }

// shared-memory matrix descriptor, no swizzle, K-major: LBO = byte stride between core matrices along K,
// SBO = byte stride between 8-row groups along N (validated by tools/tc_probe.cu)
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

// 64 consecutive TMEM columns -> registers as two 32-column loads and one wait (a single .x64 needs 82 registers at its
// point of issue, which ptxas checks against the launch-time register target, not the setmaxnreg value of the region)
__device__ __forceinline__ void tmem_st_x4(uint32_t taddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void tmem_ld_x64(uint32_t taddr, uint32_t (&v)[64])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
                 : "r"(taddr + 32u));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- staging + conversion (converter warps) ----------------------------------------------------------------------
// The raw interleaved bytes [x0*CH-16, x0*CH-16+ROW) of the 8 rows of a group are staged global -> shared two groups ahead
// of their conversion (x0*CH is 16-byte aligned: x0 is a multiple of 128).  Every converter thread arrives once per group
// on the raw buffer's mbarrier:
//   * group inside the image (no halo rows, no edge replication): thread 0 issues one 3-D tensor copy (box = ROW/4 x 8 x 1
//     32-bit elements at (x0*CH/4 - 4, vy0, frame); bytes left of the row start / beyond the pitch are zero-filled and
//     never read) and arrives with the expected byte count, the others just arrive;
//   * otherwise each thread gathers its 16-byte chunks with cp.async from the clamped / halo row pointers (chunks
//     outside [0, pitch) are skipped) and arrives through cp.async.mbarrier.arrive.noinc.
template <int CH>
struct StageMap {
    static constexpr int CHUNKS = RawGeom<CH>::CHUNKS;
    static constexpr int PER = (8 * CHUNKS + NCONV - 1) / NCONV;   // chunks per thread (CH=3: 3, CH=1: 1)
    __device__ __forceinline__ static void gather(const DctcK1Args& a, const uint8_t* __restrict__ img, uint8_t* __restrict__ R, int vy0, int x0, int ct)
    {
#pragma unroll
        for (int i = 0; i < PER; i++) {
            const int c = ct + i * NCONV;
            const int r = c / CHUNKS, k = c - r * CHUNKS;
            const long long gb = (long long) x0 * CH - 16 + 16 * k;
            if (c < 8 * CHUNKS && gb >= 0 && gb + 16 <= (long long) a.pitch) {
                const uint8_t* src = dctc_row_ptr(a, img, vy0 + r) + gb;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(R + r * RawGeom<CH>::ROW + 16 * k)), "l"(src) : "memory");
            }
        }
    }
    __device__ __forceinline__ static void stage(const DctcK1Args& a, const CUtensorMap* tmap, int use_tmap, const uint8_t* __restrict__ img,
                                                 int frame, uint8_t* __restrict__ R, uint32_t bar, int vy0, int x0, int ct)
    {
        if (use_tmap && vy0 >= 0 && vy0 + 7 < a.h) {
            if (ct == 0) {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t) (8 * RawGeom<CH>::ROW)) : "memory");
                asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                             ::"r"(smem_u32(R)), "l"(tmap), "r"(x0 * CH / 4 - 4), "r"(vy0), "r"(frame), "r"(bar) : "memory");
            } else {
                mbar_arrive(bar);
            }
        } else {
            gather(a, img, R, vy0, x0, ct);
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
        }
    }
};


// Luma in this kernel is the EXACT integer 2126 R + 7152 G + 722 B (= 10000 * 255 * liblqr's LQR_ER_LUMA value, below
// 2^22, so its float is exact too); grey is 10000 * v.  Two dp2a per pixel (16-bit coefficients times the pixel's bytes)
// replace three byte->float conversions and an FMA chain.  The factor 2^-13 of the scaled x-pass
// (fp16 range of the hi/lo operands) and the 1/10000 are folded into the final weight.
// ... and so is the factor 2*sqrt(2) the stored DCT basis carries (dctc_tc_tables.cuh).
constexpr float LUMA_WEIGHT_SCALE = (float) (8192.0 / 10000.0 / 2.8284271247461903);
// accumulator column of (output row i, coefficient k2): the two k2 whose basis rows are exact in fp16 come last
__host__ __device__ constexpr int tc_cls(int k2) { return k2 == 0 ? 6 : k2 == 4 ? 7 : k2 < 4 ? k2 - 1 : k2 - 2; }
__host__ __device__ constexpr int tc_k2(int cls) { return cls == 6 ? 0 : cls == 7 ? 4 : cls < 3 ? cls + 1 : cls + 2; }
__host__ __device__ constexpr int tc_col(int i, int k2) { return tc_cls(k2) * 8 + i; }

template <int CH>
__device__ __forceinline__ float luma_raw(const uint8_t* __restrict__ p)
{
    if (CH == 3) return (float) (2126u * p[0] + 7152u * p[1] + 722u * p[2]);
    return (float) (10000u * p[0]);
}

// luma of four consecutive pixels from their CH*4 raw bytes (4-byte aligned); same values as luma_raw
template <int CH>
__device__ __forceinline__ void quad_luma(const uint8_t* __restrict__ p, float (&l)[4])
{
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    if (CH == 3) {
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
        // dp2a.lo: R * 2126 + G * 7152 from bytes 0, 1; dp2a.hi: B * 722 (+ 0 * byte 3) from bytes 2, 3
        constexpr uint32_t CRG = (7152u << 16) | 2126u, CB = 722u;
        const uint32_t p1 = __byte_perm(w0, w1, 0x6543), p2 = __byte_perm(w1, w2, 0x5432), p3 = w2 >> 8;
        l[0] = (float) __dp2a_lo(CRG, w0, __dp2a_hi(CB, w0, 0u));
        l[1] = (float) __dp2a_lo(CRG, p1, __dp2a_hi(CB, p1, 0u));
        l[2] = (float) __dp2a_lo(CRG, p2, __dp2a_hi(CB, p2, 0u));
        l[3] = (float) __dp2a_lo(CRG, p3, __dp2a_hi(CB, p3, 0u));
    } else {
        const uint32_t w0 = w[0];
#pragma unroll
        for (int i = 0; i < 4; i++) l[i] = (float) (10000u * ((w0 >> (8 * i)) & 255u));
    }
}

// dctc_dct_fwd2<8> (tools/gen_dct.py) with every constant scaled by 2^-13 (exact), so that the x-pass coefficients of
// integer luma values up to 2.55e6 stay inside the fp16 range of the hi/lo operand split
__device__ __forceinline__ void dct8_fwd2_scaled(const float2* __restrict__ v, float2* __restrict__ X)
{
    constexpr float S = 1.0f / 8192.0f;
    const float2 t1 = dctc_f2add(v[0], v[7]), t2 = dctc_f2sub(v[0], v[7]);
    const float2 t3 = dctc_f2add(v[1], v[6]), t4 = dctc_f2sub(v[1], v[6]);
    const float2 t5 = dctc_f2add(v[2], v[5]), t6 = dctc_f2sub(v[2], v[5]);
    const float2 t7 = dctc_f2add(v[3], v[4]), t8 = dctc_f2sub(v[3], v[4]);
    X[1] = dctc_f2fma(S * 9.754516184e-02f, t8, dctc_f2fma(S * 2.777851224e-01f, t6, dctc_f2fma(S * 4.157347977e-01f, t4, dctc_f2mul(S * 4.903926253e-01f, t2))));
    X[3] = dctc_f2fma(S * -2.777851224e-01f, t8, dctc_f2fma(S * -4.903926253e-01f, t6, dctc_f2fma(S * -9.754516184e-02f, t4, dctc_f2mul(S * 4.157347977e-01f, t2))));
    X[5] = dctc_f2fma(S * 4.157347977e-01f, t8, dctc_f2fma(S * 9.754516184e-02f, t6, dctc_f2fma(S * -4.903926253e-01f, t4, dctc_f2mul(S * 2.777851224e-01f, t2))));
    X[7] = dctc_f2fma(S * -4.903926253e-01f, t8, dctc_f2fma(S * 4.157347977e-01f, t6, dctc_f2fma(S * -2.777851224e-01f, t4, dctc_f2mul(S * 9.754516184e-02f, t2))));
    const float2 t9 = dctc_f2add(t1, t7), t10 = dctc_f2sub(t1, t7);
    const float2 t11 = dctc_f2add(t3, t5), t12 = dctc_f2sub(t3, t5);
    X[2] = dctc_f2fma(S * 1.913417131e-01f, t12, dctc_f2mul(S * 4.619397521e-01f, t10));
    X[6] = dctc_f2fma(S * -4.619397521e-01f, t12, dctc_f2mul(S * 1.913417131e-01f, t10));
    const float2 t13 = dctc_f2add(t9, t11), t14 = dctc_f2sub(t9, t11);
    X[4] = dctc_f2mul(S * 3.535533845e-01f, t14);
    X[0] = dctc_f2mul(S * 3.535533845e-01f, t13);
}

// raw rows -> luma row pairs; staged index i <-> image column clamp(x0 - 4 + i) (src/render.c:122-132).
// A task is one 4-pixel group of one row pair (4 x 34 tasks per group of rows); a converter thread owns the same one or
// two tasks for every group of an item, so their offsets and the border test are computed once per item (ConvMap).
// Groups that touch the image border take the per-pixel clamped path.
template <int CH>
struct ConvMap {
    static constexpr int ROW = RawGeom<CH>::ROW;
    static constexpr int PER = (4 * NQUAD + NCONV - 1) / NCONV;   // 2
    int roff[PER];     // byte offset of the task's first raw row inside a raw buffer, -1: no task
    int loff[PER];     // float2 index inside a luma buffer
    int gx[PER];       // image column of the first pixel; INT_MIN when the four pixels are all inside the image
    __device__ __forceinline__ void init(const DctcK1Args& a, int x0, int ct)
    {
#pragma unroll
        for (int i = 0; i < PER; i++) {
            const int task = ct + i * NCONV;
            const int p = task / NQUAD, q = task - p * NQUAD - 1;   // row pair 0..3, quad -1..32
            const int g = x0 + 4 * q;
            roff[i] = task < 4 * NQUAD ? (2 * p) * ROW + 16 + 4 * CH * q : -1;
            loff[i] = p * LWP + 4 * q + 4;
            gx[i] = (g >= 0 && g + 3 < a.w) ? (int) 0x80000000 : g;
        }
    }
    __device__ __forceinline__ void convert(const DctcK1Args& a, const uint8_t* __restrict__ R, float2* __restrict__ L) const
    {
#pragma unroll
        for (int i = 0; i < PER; i++) {
            if (roff[i] < 0) continue;
            const uint8_t* r0 = R + roff[i];
            const uint8_t* r1 = r0 + ROW;
            float l0[4], l1[4];
            if (gx[i] == (int) 0x80000000) {
                quad_luma<CH>(r0, l0);
                quad_luma<CH>(r1, l1);
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int off = (max(0, min(gx[i] + k, a.w - 1)) - gx[i]) * CH;
                    l0[k] = luma_raw<CH>(r0 + off);
                    l1[k] = luma_raw<CH>(r1 + off);
                }
            }
            float4* dst = reinterpret_cast<float4*>(L + loff[i]);
            dst[0] = make_float4(l0[0], l1[0], l0[1], l1[1]);
            dst[1] = make_float4(l0[2], l1[2], l0[3], l1[3]);
        }
    }
};

// H -> fp16 hi and fp16 MINUS lo for two vertically adjacent rows (low half = even row = even K index).
// hi = rn16(H); the residual comes from one mixed-precision subtract per value (sub.f32.f16 = FHADD: hi - H, exact),
// so no half->float conversion is needed; the sign is undone by the negate-A bit of the lo*Bh MMA's descriptor.
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

// x-pass + split + tcgen05.st of group g (rows staged in s.L) into ring slot g&1; arrives on the "operands stored" barrier
__device__ __forceinline__ void produce_group(TcSmem& s, int g, int tid, uint32_t tmem_lane, long long* g_tt_acc)
{
    (void) g_tt_acc;
    const uint32_t ta = tmem_lane + TM_A + (uint32_t) (g & 1) * 4u;
    const float2 (*Lg)[LWP] = s.L[g & 1];
    // the whole x-pass and hi/lo split of the group happens before the ring-slot wait (64 operand registers: the
    // producer warpgroup runs with 112 registers), so that only the TMEM stores sit between two MMA phases
    uint32_t hi[8][4], lo[8][4];
#pragma unroll
    for (int p = 0; p < 4; p++) {
        float2 v[8], X[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = Lg[p][tid + j + 1];
        if (p == 3) bar_lfree_arrive(g & 1);   // last read of this luma buffer
#if DCTC_TC_ABL & 2
#pragma unroll
        for (int k1 = 0; k1 < 8; k1++) { hi[k1][p] = __float_as_uint(v[k1].x); lo[k1][p] = __float_as_uint(v[k1].y); }
#else
        dct8_fwd2_scaled(v, X);
#pragma unroll
        for (int k1 = 0; k1 < 8; k1++) split_pair(X[k1], hi[k1][p], lo[k1][p]);
#endif
    }
    // slot g&1 still holds group g-2, read by the MMAs of step g-2: the k1 = 0..3 operands are released when the first
    // half of those MMAs has completed, the rest at the end of the step
#pragma unroll
    for (int hk = 0; hk < 2; hk++) {
        if (g >= 2) {
            TT_T0();
            mbar_wait(smem_u32(hk ? &s.bar_a_free : &s.bar_a_free_lo), (uint32_t) (g & 1));
            TT_ACC(0, 1);
            tc_fence_after();
        }
#pragma unroll
        for (int k1 = 4 * hk; k1 < 4 * hk + 4; k1++) {
            tmem_st_x4(ta + (uint32_t) (k1 * 16), hi[k1][0], hi[k1][1], hi[k1][2], hi[k1][3]);
            tmem_st_x4(ta + (uint32_t) (k1 * 16 + 8), lo[k1][0], lo[k1][1], lo[k1][2], lo[k1][3]);
        }
        {
            TT_T0();
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");   // warp-wide: every lane's stores have completed
            TT_ACC(0, 2);
        }
        tc_fence_before();
        // Group 0 is not announced on its own: the arrivals of group 1 cover both (same warp, program order).  The
        // arrival of half hk of group g+1 needs the completion of the MMAs k1 <= 4 hk + 3 of step g-1, which the MMA warp
        // issues after its sync on this half for step g-1: there is never more than one pending arrival per barrier.
        if (g >= 1) bar_afull_arrive(hk);
    }
}

// ---- consumer fold -------------------------------------------------------------------------------------------
template <bool UNIFORM>
struct TcFold;

template <>
struct TcFold<true> {   // edges == textures: only the maximum matters
    float m[8];
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = 0.0f;
    }
    template <int K1>
    __device__ __forceinline__ void add(const uint32_t (&v)[64])
    {
#pragma unroll
#if DCTC_TC_ABL & 1
        for (int i = 0; i < 1; i++) {
#else
        for (int i = 0; i < 8; i++) {
#endif
            float t = m[i];
            if (K1 != 0) t = fmaxf(t, fabsf(__uint_as_float(v[tc_col(i, 0)])));   // (0,0) is skipped (src/dct.c:101)
            t = fmaxf(t, fabsf(__uint_as_float(v[tc_col(i, 1)])));
#pragma unroll
            for (int k2 = 2; k2 < 8; k2 += 2)
                t = fmaxf(t, fmaxf(fabsf(__uint_as_float(v[tc_col(i, k2)])), fabsf(__uint_as_float(v[tc_col(i, k2 + 1)]))));
            m[i] = t;
        }
    }
    __device__ __forceinline__ float result(int i, float we, float wt) const { (void) we; return m[i] * wt; }
};

template <>
struct TcFold<false> {  // last-arg-max class rule of DctcTracker<false>
    // With A = |T[0][1]|, M = max|T[0][2..]|, Bv = |T[1][0]|, Z = max of the rest, the winner is a texture atom iff
    //   Z >= max(A, M, Bv)  or  (Bv < max(A, M) and M >= A).
    // A and M are final after the k1 = 0 tile, Bv arrives first in the k1 = 1 tile; from then on only
    //   pre = max(A, M, Bv)  and the bit  tex_pre = (Bv < max(A, M) and M >= A)
    // are needed next to the running Z:  texture iff  Z >= pre  or  tex_pre.
    float z[8], pre[8];
    unsigned flags;          // bit i: M >= A (after the k1 = 0 tile), then tex_pre (after the k1 = 1 tile) of row i
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int i = 0; i < 8; i++) z[i] = 0.0f;
        flags = 0u;
    }
    template <int K1>
    __device__ __forceinline__ void add(const uint32_t (&v)[64])
    {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            if (K1 == 0) {
                const float a = fabsf(__uint_as_float(v[tc_col(i, 1)]));
                float mm = -1.0f;
#pragma unroll
                for (int k2 = 2; k2 < 8; k2++) mm = fmaxf(mm, fabsf(__uint_as_float(v[tc_col(i, k2)])));
                pre[i] = fmaxf(a, mm);
                if (mm >= a) flags |= 1u << i;
            } else {
                if (K1 == 1) {
                    const float bv = fabsf(__uint_as_float(v[tc_col(i, 0)]));
                    if (bv >= pre[i]) flags &= ~(1u << i);      // Bv is the last maximal index among A, M, Bv: an edge atom
                    pre[i] = fmaxf(pre[i], bv);
                } else {
                    z[i] = fmaxf(z[i], fabsf(__uint_as_float(v[tc_col(i, 0)])));
                }
#pragma unroll
                for (int k2 = 1; k2 < 8; k2++) z[i] = fmaxf(z[i], fabsf(__uint_as_float(v[tc_col(i, k2)])));
            }
        }
    }
    __device__ __forceinline__ float result(int i, float we, float wt) const
    {
        const float top = fmaxf(pre[i], z[i]);
        const bool tex = (z[i] >= pre[i]) || ((flags >> i) & 1u);
        return top * (tex ? wt : we);
    }
};

template <int K1, bool UNIFORM>
__device__ __forceinline__ void consume_k1(TcSmem& s, TcFold<UNIFORM>& f, uint32_t tmem_lane, bool lane0, long long* g_tt_acc)
{
    (void) g_tt_acc;
    constexpr int b = K1 & 1, q = K1 >> 1;
    {
        TT_T0();
        mbar_wait(smem_u32(&s.bar_d_full[b]), (uint32_t) (q & 1));
        TT_ACC(1, K1 == 0 ? 0 : 1);
    }
    tc_fence_after();
    uint32_t v[64];
    {
        TT_T0();
        tmem_ld_x64(tmem_lane + TM_D + 64u * b, v);
        TT_ACC(1, 2);
    }
    tc_fence_before();
    (void) lane0;
    bar_tile_arrive(b);
    f.template add<K1>(v);
}

// Persistent kernel: two CTAs per SM (256 TMEM columns each), work items = (frame, segment, strip) handed out by an
// atomic counter.
template <bool UNIFORM, int CH>
__global__ void __launch_bounds__(NTHREADS, 2) dctc_k1_tc8_kernel(const DctcK1Args a, int seg_rows, int strips, int segs, int n_items,
                                                                    int* __restrict__ counter, const __grid_constant__ CUtensorMap tmap,
                                                                    int use_tmap)
{
    __shared__ TcSmem s;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler

    // Programmatic dependent launch: the next launch in the stream may start its CTAs as soon as this grid's CTAs retire;
    // what follows up to griddepcontrol.wait (TMEM allocation, the Toeplitz operands from immutable tables) touches no
    // memory an earlier grid writes, so a launch's ramp overlaps its predecessor's tail.
    asm volatile("griddepcontrol.launch_dependents;");
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // Toeplitz operands: Tz[n = tc_col(i, k2)][k] = B8[k2][r - i] with window row r = k (normal) or k ^ 8 (K-swapped)
    {
        uint16_t* Bq = reinterpret_cast<uint16_t*>(&s.B[0][0]);
        for (int idx = tid; idx < 4 * 1024; idx += NTHREADS) {
            const int v = idx >> 10, n = (idx >> 4) & 63, k = idx & 15;
            const int i = n & 7, k2 = tc_k2(n >> 3);
            const int c = ((v & 2) ? (k ^ 8) : k) - i;
            const uint16_t val = (c >= 0 && c < 8) ? DCTC_TC_BASIS8[v & 1][k2 * 8 + c] : (uint16_t) 0;
            Bq[v * 1024 + (n >> 3) * 128 + (k >> 3) * 64 + (n & 7) * 8 + (k & 7)] = val;
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");     // everything before this grid in the stream is complete and visible
    const uint32_t lane_off = (uint32_t) ((warp & 3) * 32) << 16;

    // Every role runs its own copy of the persistent item loop (begin_item / end_item contain the CTA-wide barriers), so
    // that each warpgroup's whole body follows its setmaxnreg: the 384 threads are launched with 80 registers; the
    // producers (64 operand registers per group) grow to 104, the consumers to 96, the MMA + converter warpgroup
    // shrinks to 40.
    auto begin_item = [&](bool first) -> int {
        if (tid == 0) {
            // Every CTA fetches until its first item >= n_items: n_items + gridDim.x fetches in all, so the wrapping
            // increment leaves the counter at 0 for the next launch that uses it (no memset between launches).
            s.work = (int) atomicInc(reinterpret_cast<unsigned int*>(counter), (unsigned int) n_items + gridDim.x - 1u);
            if (!first) {
                mbar_inval(smem_u32(&s.bar_a_free));
                mbar_inval(smem_u32(&s.bar_a_free_lo));
                mbar_inval(smem_u32(&s.bar_d_full[0]));
                mbar_inval(smem_u32(&s.bar_d_full[1]));
                for (int i = 0; i < 3; i++) mbar_inval(smem_u32(&s.bar_raw[i]));
            }
            mbar_init(smem_u32(&s.bar_a_free), 1);
            mbar_init(smem_u32(&s.bar_a_free_lo), 1);
            mbar_init(smem_u32(&s.bar_d_full[0]), 1);
            mbar_init(smem_u32(&s.bar_d_full[1]), 1);
            for (int i = 0; i < 3; i++) mbar_init(smem_u32(&s.bar_raw[i]), NCONV);
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
#define DCTC_ITEM_LOOP                                                                                                 \
    for (bool first = true;; first = false) {                                                                          \
        const int item = begin_item(first);                                                                            \
        if (item >= n_items) break;                                                                                    \
        const uint32_t tmem = s.tmem_base;                                                                             \
        const uint32_t tmem_lane = tmem + lane_off;                                                                    \
        const int strip = item % strips;                                                                               \
        const int rest = item / strips;                                                                                \
        const int seg = rest % segs, frame = rest / segs;                                                              \
        (void) frame;                                                                                                  \
        const int x0 = strip * MW;                                                                                     \
        const int y0 = seg * seg_rows;                                                                                 \
        const int y1 = min(y0 + seg_rows, a.h);                                                                        \
        const int nsteps = (y1 - y0 + 7) >> 3;                                                                         \
        const uint8_t* __restrict__ img = a.img + (size_t) frame * a.frame_stride;                                     \
        float* __restrict__ out = a.out + (size_t) frame * a.out_frame_stride;                                         \
        (void) tmem; (void) tmem_lane; (void) x0; (void) y1; (void) img; (void) out;

    TT_DECL();
    if (warp < 4) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
        DCTC_ITEM_LOOP
        // ===== producers: group g = virtual rows y0-3+8g .. y0+4+8g; step j consumes groups j and j+1 =====
        for (int g = 0; g <= nsteps; g++) {
            {
                TT_T0();
                bar_lfull_sync(g & 1);                        // the converters have written luma buffer g&1
                TT_ACC(0, 0);
            }
            produce_group(s, g, tid, tmem_lane, g_tt_acc);    // arrives on "luma buffer free" after its last read
        }
        end_item();
        }
        TT_REPORT(0, tid == 0);
    } else if (warp < 8) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 96;");
        DCTC_ITEM_LOOP
        // ===== consumers =====
        const int px = tid - 128;
        const int gx = x0 + px;
        const bool lane0 = (tid & 31) == 0;
        // one running output pointer per item (advanced by 8 rows per step) instead of a 64-bit row address per store
        const size_t op = a.out_pitch;
        float* __restrict__ orow = out + (size_t) y0 * op + gx;
        const float we = a.w_edges * LUMA_WEIGHT_SCALE, wt = a.w_textures * LUMA_WEIGHT_SCALE;
        for (int st = 0; st < nsteps; st++) {
            TcFold<UNIFORM> f;
            f.init();
            bar_step_sync();                                  // the MMA warp has started this step
            consume_k1<0, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<1, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<2, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<3, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<4, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<5, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<6, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            consume_k1<7, UNIFORM>(s, f, tmem_lane, lane0, g_tt_acc);
            const int gy = y0 + 8 * st;
            if (gx < a.w) {
                float* __restrict__ o = orow;
                if (gy + 8 <= y1) {
#pragma unroll
                    for (int i = 0; i < 8; i++) { *o = f.result(i, we, wt); o += op; }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        if (gy + i < y1) *o = f.result(i, we, wt);
                        o += op;
                    }
                }
            }
            orow += 8 * op;
        }
        end_item();
        }
        TT_REPORT(1, tid == 128);
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp == 8) {
        DCTC_ITEM_LOOP
        // ===== MMA issuer =====
        const uint32_t idesc = make_idesc(128, 64);
        const uint32_t idesc_bl = make_idesc(128, 48);           // hi*Bl: the columns of k2 = 0, 4 (Bl = 0) are skipped
        const uint64_t bd0 = make_smem_desc(smem_u32(&s.B[0][0]), 128, 256);
        for (int st = 0; st < nsteps; st++) {
            {
                TT_T0();
                bar_afull_sync(0);                            // the k1 = 0..3 operands of groups st and st+1 are in TMEM
                TT_ACC(2, 0);
            }
            tc_fence_after();
            bar_step_arrive();                                // wakes the consumers of this step
            // each operand copy is 2048 bytes = 128 descriptor address units
            const uint64_t bh = bd0 + (uint64_t) ((st & 1) ? 256 : 0);
            const uint64_t bl = bh + 128;
#pragma unroll
            for (int k1 = 0; k1 < 8; k1++) {
                const int b = k1 & 1;
                if (k1 == 4) {
                    bar_afull_sync(1);                        // ... and the k1 = 4..7 operands
                    tc_fence_after();
                }
                if (st > 0 || k1 >= 2) {
                    TT_T0();
                    bar_tile_sync(b);                         // the consumers have loaded the previous contents of tile b
                    TT_ACC(2, 1);
                }
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t d = tmem + TM_D + 64u * b;
                    const uint32_t ah = tmem + TM_A + (uint32_t) k1 * 16u, al = ah + 8u;
                    mma_ts(d, ah, bh, idesc, 0u);
                    mma_ts(d, al, bh, idesc | (1u << 13), 1u);   // A negated: the ring holds -lo
                    mma_ts(d, ah, bl, idesc_bl, 1u);
                    mma_commit(smem_u32(&s.bar_d_full[b]));
                    if (k1 == 3 && st + 2 <= nsteps) mma_commit(smem_u32(&s.bar_a_free_lo));
                    if (k1 == 7 && st + 2 <= nsteps) mma_commit(smem_u32(&s.bar_a_free));   // waited on by the producers of group st+2
                }
                __syncwarp();
            }
        }
        // the last use of each tile was arrived on but never waited for: drain both named barriers so that their
        // generations start clean for the next work item
        bar_tile_sync(0);
        bar_tile_sync(1);
        end_item();
        }
        TT_REPORT(2, tid == 256);
        } else {
        DCTC_ITEM_LOOP
        // ===== converters: raw rows of group g+2 in flight while group g is converted =====
        const int ct = tid - (NTHREADS - NCONV);
        ConvMap<CH> cm;
        cm.init(a, x0, ct);
        StageMap<CH>::stage(a, &tmap, use_tmap, img, frame, s.Raw[0], smem_u32(&s.bar_raw[0]), y0 - 3, x0, ct);
        StageMap<CH>::stage(a, &tmap, use_tmap, img, frame, s.Raw[1], smem_u32(&s.bar_raw[1]), y0 + 5, x0, ct);
        int slot = 0;                                         // raw buffer of group g (g % 3)
        uint32_t par = 0u;                                    // bit i: parity of the next completion of raw buffer i
        for (int g = 0; g <= nsteps; g++) {
            {
                TT_T0();
                mbar_wait(smem_u32(&s.bar_raw[slot]), (par >> slot) & 1u);   // the copies of group g have landed
                par ^= 1u << slot;
                TT_ACC(3, 0);
            }
            {
                TT_T0();
                bar_converters();                             // every converter has left group g-1: raw buffer (g+2)%3 = (g-1)%3 is free
                TT_ACC(3, 1);
            }
            if (g >= 2) {
                TT_T0();
                bar_lfree_sync(g & 1);                        // the producers have read group g-2 out of this buffer
                TT_ACC(3, 2);
            }
            cm.convert(a, s.Raw[slot], &s.L[g & 1][0][0]);
            bar_lfull_arrive(g & 1);
            const int nslot = slot == 0 ? 2 : slot - 1;       // (g + 2) % 3
            if (g + 2 <= nsteps)
                StageMap<CH>::stage(a, &tmap, use_tmap, img, frame, s.Raw[nslot], smem_u32(&s.bar_raw[nslot]), y0 - 3 + 8 * (g + 2), x0, ct);
            slot = slot == 2 ? 0 : slot + 1;
        }
        // the last two groups' "free" arrivals were never waited for: drain them so the next item starts clean
        bar_lfree_sync((nsteps - 1) & 1);
        bar_lfree_sync(nsteps & 1);
        end_item();
        }
        TT_REPORT(3, tid == 288);
        }
    }
#undef DCTC_ITEM_LOOP

    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s.tmem_base), "r"(TMEM_COLS));
}

}  // namespace

// Full maps (no band / preview mode) in the fast layout (dctc_k1_fast_layout).
// `counter` is a device int owned by the context (work-item counter of the persistent kernel), zero before the launch;
// the kernel leaves it at zero again.
cudaError_t dctc_launch_k1_tc8(const DctcK1Args& a, int n_frames, bool uniform, int* counter, int sm_count, cudaStream_t stream)
{
    if (a.w <= 0 || a.h <= 0 || n_frames <= 0) return cudaSuccess;
    const int strips = (a.w + MW - 1) / MW;
    // Segment height.  An item of S rows costs S/8 + 2 steps (two prologue groups); the 2 x sm_count resident CTAs take
    // items from a counter, so a launch lasts about ceil(items / CTAs) x (S/8 + 2) steps when the items are few, and
    // (total steps + 2 x items) / CTAs when they are many.  Candidates: 256 / 128 / 64 / 32 rows (evened out over the
    // image height) and the "one round" split that gives every CTA at most one item (one 4K frame: 9 segments of 240
    // rows = 270 items on 296 CTAs, 32 steps, instead of 1020 items of 64 rows, 4 rounds of 10 steps).
    // (measured on 16 frames of 4K: 1024/512 rows 50.5 us per frame, 256 rows 49.3, 128 rows 50.5, 64 rows 54.7)
    const long long ctas = 2LL * sm_count;
    auto even_seg = [&](int want) {
        int sg = (a.h + want - 1) / want;
        int sr = (((a.h + sg - 1) / sg) + 7) & ~7;          // even segments (1080 rows: 5 x 216 instead of 4 x 256 + 56)
        return sr < 8 ? 8 : sr;
    };
    auto cost = [&](int sr) {
        const long long sg = (a.h + sr - 1) / sr, it = (long long) strips * sg * n_frames;
        const long long per = sr / 8 + 2;
        const long long rounds = (it + ctas - 1) / ctas;
        const long long balanced = (it * per + ctas - 1) / ctas + per / 2;   // many items: the tail is about half an item
        return it <= 4 * ctas ? rounds * per : balanced;
    };
    int seg = even_seg(256);
    for (int want : {128, 64, 32}) {
        const int sr = even_seg(want);
        if (cost(sr) < cost(seg)) seg = sr;
    }
    {
        const long long per_col = ctas / ((long long) strips * n_frames);      // segments per strip that still fit one round
        if (per_col >= 1) {
            const int sr = even_seg((int) ((a.h + per_col - 1) / per_col));
            if ((long long) strips * ((a.h + sr - 1) / sr) * n_frames <= ctas && cost(sr) < cost(seg)) seg = sr;
        }
    }
    // Large batches (every CTA gets eight or more items even at ~544 rows): taller items, i.e. fewer prologue groups; the tail
    // of the item loop no longer matters (measured on 512 / 64 / 16 frames of 4K per launch: 240-row items 51.4 / 44.2 /
    // 45.8 us per frame, 544-row items 50.3 / 43.7 / 45.6, 1080-row items 50.2 / 44.2 / 48.4)
    {
        const int tall = even_seg(544);
        if (tall > seg && (long long) strips * ((a.h + tall - 1) / tall) * n_frames >= 8 * ctas) seg = tall;
    }
    const int segs = (a.h + seg - 1) / seg;
    const long long items = (long long) strips * segs * n_frames;
    if (items > 0x7fffffffLL) return cudaErrorInvalidConfiguration;
    const int grid = (int) (items < 2LL * sm_count ? items : 2LL * sm_count);
    // tensor map of the frames as 32-bit elements: (pitch / 4, h, frames); box = one staged raw tile (ROW / 4 x 8 x 1)
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    int use_tmap = 0;
    {
        const DctcTensorMapEncodeFn encode = dctc_tensor_map_encoder();
        const size_t fstride = n_frames > 1 ? a.frame_stride : a.pitch * (size_t) a.h;
        const int row = a.channels == 3 ? RawGeom<3>::ROW : RawGeom<1>::ROW;
        if (encode && a.h >= 8 && (fstride & 15) == 0 && fstride >= a.pitch && a.pitch < (1ull << 40) && fstride < (1ull << 40)) {
            const cuuint64_t gdim[3] = {(cuuint64_t) (a.pitch / 4), (cuuint64_t) a.h, (cuuint64_t) n_frames};
            const cuuint64_t gstr[2] = {(cuuint64_t) a.pitch, (cuuint64_t) fstride};
            const cuuint32_t box[3] = {(cuuint32_t) (row / 4), 8u, 1u};
            const cuuint32_t estr[3] = {1, 1, 1};
            if (encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(a.img), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
                use_tmap = 1;
        }
    }
    const cudaError_t e = dctc_dispatch<3, 1>(uniform, a.channels, [&](auto U, auto C) {
        const cudaError_t ea = cudaFuncSetAttribute(dctc_k1_tc8_kernel<U, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, PAD_SMEM);
        if (ea != cudaSuccess) return ea;
        return dctc_launch_pdl(dctc_k1_tc8_kernel<U, C>, dim3(grid), dim3(NTHREADS), PAD_SMEM, stream, true, a, seg, strips, segs,
                               (int) items, counter, tmap, use_tmap);
    });
    return e != cudaSuccess ? e : cudaGetLastError();
}

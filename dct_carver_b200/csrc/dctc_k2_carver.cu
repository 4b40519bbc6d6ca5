// K2: carver session with incremental per-seam energy.
//
// Replaces liblqr's per-seam "carve + update_emap" pair as driven by lqr_carver_resize (src/render.c:377):
// after a vertical seam is removed, liblqr re-invokes the energy callback (src/render.c:134-157) for the pixels
// within +-radius of the seam (radius = blocksize/2, registered at src/render.c:314-315).  Here the image and the
// energy plane stay resident in HBM; one kernel compacts both over the seam, then the K1 tile kernel runs in band
// mode over just the touched pixels, with arithmetic identical to a full recompute (bit-identical results).
#include <cmath>
#include <cstdio>
#include <type_traits>
#include <cstring>
#include <new>
#include <utility>
#include "dctc_common.cuh"
#include "dctc_launch.h"
#include "dctc_resize_plan.h"

// One CTA per row: shift image bytes and energy floats right of the seam one pixel to the left.
// Chunks are processed left to right; the barrier between a chunk's loads and its stores also orders them
// after the previous chunk's loads, so the one-element overlap between neighbouring chunks is safe.
// Batch sessions: blockIdx.y = frame, whose planes start img_fs bytes / en_fs, m_fs floats after the previous frame's
// and whose seam is seam[h * frame ...] (h = gridDim.x).
// BIAS: the bias plane of a biased session (laid out like the energy plane) is compacted too.
template <int NT, int K, bool BIAS>
__global__ void __launch_bounds__(NT) dctc_carve_rows_kernel(uint8_t* __restrict__ img, size_t pitch, int channels,
                                                             float* __restrict__ en, size_t en_pitch,
                                                             const int* __restrict__ seam, int w_old,
                                                             float* __restrict__ mplane, size_t m_pitch,
                                                             size_t img_fs, size_t en_fs, size_t m_fs, float* __restrict__ bias)
{
    DCTC_PDL_PROLOGUE();
    const int y = blockIdx.x, z = blockIdx.y;
    const int s = seam[(size_t) z * gridDim.x + y];
    uint8_t* row = img + z * img_fs + (size_t) y * pitch;
    float* erow = en + z * en_fs + (size_t) y * en_pitch;
    if constexpr (BIAS) {
        float* brow = bias + z * en_fs + (size_t) y * en_pitch;
        for (int base = s; base < w_old - 1; base += NT * K) {
            float v[K];
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int x = base + k * NT + threadIdx.x;
                v[k] = x < w_old - 1 ? brow[x + 1] : 0.0f;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int x = base + k * NT + threadIdx.x;
                if (x < w_old - 1) brow[x] = v[k];
            }
        }
    }
    // cumulative map of the seam DP (liblqr keeps it per pixel, so it moves with the pixels): dst x in [s, w_old-1)
    if (mplane) {
        float* mrow = mplane + z * m_fs + (size_t) y * m_pitch;
        for (int base = s; base < w_old - 1; base += NT * K) {
            float v[K];
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int x = base + k * NT + threadIdx.x;
                v[k] = x < w_old - 1 ? mrow[x + 1] : 0.0f;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int x = base + k * NT + threadIdx.x;
                if (x < w_old - 1) mrow[x] = v[k];
            }
        }
    }
    // energy floats: dst x in [s, w_old-1)
    for (int base = s; base < w_old - 1; base += NT * K) {
        float v[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int x = base + k * NT + threadIdx.x;
            v[k] = x < w_old - 1 ? erow[x + 1] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int x = base + k * NT + threadIdx.x;
            if (x < w_old - 1) erow[x] = v[k];
        }
    }
    // image bytes: dst byte in [s*ch, (w_old-1)*ch)
    const int b0 = s * channels, b1 = (w_old - 1) * channels;
    for (int base = b0; base < b1; base += NT * K) {
        uint8_t v[K];
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int i = base + k * NT + threadIdx.x;
            v[k] = i < b1 ? row[i + channels] : (uint8_t) 0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int i = base + k * NT + threadIdx.x;
            if (i < b1) row[i] = v[k];
        }
    }
}


// ---- seam DP + back-track on the device (SURVEY section 8f rank 1) ---------------------------------------------
// liblqr's build_mmap / build_vpath for delta_x = 1 (src/render.c:313,377; restated in dct_carver_b200/host/dctc_lqr.c
// and oracle/oracle_carver.c):
//   m[0][x] = en[0][x];  m[y][x] = en[y][x] + min(m[y-1][x-1], m[y-1][x], m[y-1][x+1])   (FP32, range clipped)
//   parent of (y, x) = FIRST strict minimum scanning x-1, x, x+1;  seam end = LEFTMOST minimum of the last row.
// Rigidity (the DpStep1<true> instantiations of the DP, jump, trace and incremental kernels): a diagonal step costs
// pen = fl(rigidity / h) more, i.e. the candidates are fl(m[y-1][x-1] + pen), m[y-1][x], fl(m[y-1][x+1] + pen) in the
// map and in the parent choice (liblqr's rigidity_map[1] = rigidity / h [from memory: parity unpinned]).  The host
// passes pen as the trailing kernel argument; DpStep1<false> never reads it and makes the kernels of rigidity 0.  Wider
// steps (delta_x > 1) take the DpSteps rule below.
// The map is rebuilt from scratch for every seam (same values as liblqr's incremental update_mmap).  Row y depends on
// the whole row y-1: a chain of h steps.  Versions with one CTA-wide barrier per row cost ~600-950 clk per row
// (shared-memory bandwidth, then the latency of a 16-warp barrier round); this one removes the per-row barrier with
// warp-private trapezoids: a warp owns a strip of 128*P columns, keeps the cells of the previous row in registers
// (4*P adjacent cells per lane) and exchanges neighbours with warp shuffles only.  What the strip's edge lanes
// cannot see contaminates one more column per row, so after DP_R rows the outer DP_R columns on each side are
// garbage and the warp publishes only its central 128*P - 2*DP_R columns; every DP_R rows the warps exchange the
// last row through shared memory (one barrier per DP_R rows) and restart with fresh halos.  Energies are staged
// a few chunks ahead by tensor copies (TMA variants) or prefetched into a register ring; the cumulative rows go to a global float plane from which warp 0 re-derives
// the parent choices during the back-track (dp_backtrack: 32-row batches through double-buffered shared-memory windows).
// Cells outside the image hold +inf, which reproduces the range clipping.
constexpr int DP_R = 32;          // rows between two exchanges = halo columns on each side of a strip
constexpr int DP_MAXW = 8;        // warps per CTA of the DP cluster (256 threads: room for a deep register prefetch ring)

constexpr int DP_CL = 8;          // CTAs of the cluster the strips are spread over (a lone SM can only pull ~35 GB/s from L2:
                                  // measured 425 clk per 1920-px row for the energy loads alone, against ~40 clk of math)

__device__ __forceinline__ uint32_t dp_cta_rank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void dp_cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a shared-memory location of this CTA's layout) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dp_map(const void* p, uint32_t rank)
{
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"((uint32_t) __cvta_generic_to_shared(p)), "r"(rank));
    return ra;
}
__device__ __forceinline__ float4 dp_ld_cluster_v4(uint32_t ra)
{
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ra) : "memory");
    return v;
}
// 16 bytes into a peer CTA's shared memory; their arrival is counted on the peer's mbarrier (complete_tx), so the
// receiver needs no fence and no cluster barrier: it waits on its own mbarrier for the bytes it expects
__device__ __forceinline__ void dp_st_async_v4(uint32_t remote_addr, float4 v, uint32_t remote_mbar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(remote_addr), "r"(__float_as_uint(v.x)), "r"(__float_as_uint(v.y)), "r"(__float_as_uint(v.z)), "r"(__float_as_uint(v.w)), "r"(remote_mbar) : "memory");
}
__device__ __forceinline__ void dp_st_cluster_f32(uint32_t ra, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory"); }
__device__ __forceinline__ void dp_st_cluster_s32(uint32_t ra, int v) { asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(ra), "r"(v) : "memory"); }

// ---- seam step rules ------------------------------------------------------------------------------------------------
// With delta_x = dx in 2 .. DCTC_MAX_DELTA_X a seam may move up to dx columns from one row to the next:
//   m[y][x] = en[y][x] + min_{|d| <= dx} fl(m[y-1][x+d] + pen[|d|]),   parent = FIRST strict minimum scanning x-dx .. x+dx,
// pen[0] = 0, pen[d] = fl(fl(rigidity * fl(d * fl(sqrt(d)))) / h) (liblqr's rigidity_map [from memory: parity unpinned]).
// Every seam-search kernel takes its step rule as a template parameter, and the rule's Arg as its trailing argument (a
// float for DpStep1, so that the dx = 1 kernels keep the parameter a plain float has; the table for DpSteps); the kernel
// rebuilds the rule from it.  A rule has D, the largest step it can take at compile time, dx, its step width, and
// pick(v, q): q(d) of the parent, the first strict minimum of the candidates d = -D .. D, where v(d) is the cumulative
// value at column x+d of the row above (+inf outside the image).  The serial walk, the jump and the trace kernels all
// choose the parent through pick; the seam DP needs only the minimum and forms it in its own row arithmetic.
template <bool RIG>
struct DpStep1 {                  // dx = 1; RIG: rigidity pen on the two diagonal candidates, else pen is never read
    using Arg = float;            // the kernel argument: pen
    static constexpr int D = 1, dx = 1;
    float pen;
    __device__ __forceinline__ float diag(float v) const { return RIG ? v + pen : v; }   // a diagonal candidate's cost
    template <typename V, typename Q>
    __device__ __forceinline__ auto pick(V v, Q q) const
    {
        const float a = diag(v(-1)), b = v(0), c = diag(v(1));
        const bool p1 = b < a;
        const float best = p1 ? b : a;
        const bool p2 = c < best;
        return p2 ? q(1) : (p1 ? q(0) : q(-1));
    }
};
// dx = 2 .. DCTC_MAX_DELTA_X at run time: pen[d] = +inf for dx < d <= D, so one kernel serves every dx: a candidate
// beyond the step bound costs +inf and never wins (best starts at +inf and the d = 0 candidate is finite).
struct DpSteps {
    using Arg = DpSteps;
    static constexpr int D = DCTC_MAX_DELTA_X;
    float pen[D + 1];
    int dx;
    template <typename V, typename Q>
    __device__ __forceinline__ auto pick(V v, Q q) const
    {
        float best = __int_as_float(0x7f800000);
        auto qb = q(0);
#pragma unroll
        for (int d = -D; d <= D; d++) {
            const float c = d == 0 ? v(0) : v(d) + pen[d < 0 ? -d : d];
            if (c < best) { best = c; qb = q(d); }
        }
        return qb;
    }
};

// ---- back-track (build_vpath) ------------------------------------------------------------------------------------
// One warp walks up from the last row: parent of (y, x) = the step rule's pick.  Every lane follows the same path,
// lane 0 records it.  The cumulative rows are read in batches of wb rows through shared-memory windows of DP_WIN
// columns, double buffered: with 2 wb dx + dx <= 66 (wb = 32 for dx = 1) the window of the NEXT batch (columns
// xs-66 .. xs+66 around the column xs at which the current batch starts) is known before the current batch is walked,
// and its cp.async copies land while the walk (a chain of dependent shared-memory reads) is running.
constexpr int DP_WIN = 144;       // back-track window (floats); the cumulative plane's pitch is at least this
constexpr int DP_WINP = DP_WIN + 8;   // window row in shared memory: 4 - D pad floats, D left sentinels, DP_WIN columns,
                                      // D right sentinels (needed when the window ends at column w) and 4 - D pad floats

template <typename Step>
__device__ __forceinline__ void dp_backtrack(const float* __restrict__ mplane, size_t m_pitch, int w, int h, int x,
                                             int* __restrict__ seam, int* __restrict__ seam_log,
                                             float (*win)[32][DP_WINP], int lane, const Step& st)
{
    const float INF = __int_as_float(0x7f800000);
    const int wb = (66 - st.dx) / (2 * st.dx);
    if (lane == 0) { seam[h - 1] = x; if (seam_log) seam_log[h - 1] = x; }
    const int max_base = (int) m_pitch - DP_WIN;
    // window rows of the batch that starts below image row ytop: window row i = image row ytop-1-i, column c of the
    // plane at win[buf][i][4 + c - base]
    auto stage = [&](int ytop, int xs, int buf) -> int {
        int base = (xs - 66) & ~3;
        base = base < 0 ? 0 : (base > max_base ? max_base : base);
        if (ytop >= 1) {
            for (int idx = lane; idx < wb * (DP_WIN / 4); idx += 32) {
                const int i = idx / (DP_WIN / 4), c = idx - i * (DP_WIN / 4);
                const int yy = ytop - 1 - i;
                if (yy >= 0) {
                    const float* src = mplane + (size_t) yy * m_pitch + base + 4 * c;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t) __cvta_generic_to_shared(&win[buf][i][4 + 4 * c])), "l"(src) : "memory");
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        return base;
    };
    int buf = 0;
    int base = stage(h - 1, x, 0);
    for (int ytop = h - 1; ytop >= 1; ytop -= wb) {
        const int base_next = stage(ytop - wb, x, buf ^ 1);     // lands while this batch is walked
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncwarp();
        // D +inf sentinels left of column 0 and from column w on (range clipping), so that the walk needs no bounds checks
        if (lane < wb) {
            if (base == 0)
                for (int j = 0; j < Step::D; j++) win[buf][lane][4 - Step::D + j] = INF;
            if (w - base >= 0 && w - base <= DP_WIN)   // <=: w == base + DP_WIN lands in the row's tail pad
                for (int j = 0; j < Step::D; j++) win[buf][lane][4 + w - base + j] = INF;
        }
        __syncwarp();
        const int steps = ytop < wb ? ytop : wb;
        // the walk: a chain of shared-memory reads at immediate offsets and the pick per row; lane i remembers the column
        // of step i and the batch's columns are written with one coalesced store at its end
        int mine = 0;
        const float* wp = &win[buf][0][4] + (x - base);        // wp[0] = cumulative value at (window row, column x)
        auto walk = [&](int i) {
            const int d = st.pick([&](int c) { return wp[c]; }, [](int c) { return c; });
            x += d;
            wp += DP_WINP + d;
            if (lane == i) mine = x;
        };
        if (Step::D == 1 && steps == 32) {
#pragma unroll
            for (int i = 0; i < 32; i++) walk(i);
        } else {
            for (int i = 0; i < steps; i++) walk(i);
        }
        if (lane < steps) { seam[ytop - 1 - lane] = mine; if (seam_log) seam_log[ytop - 1 - lane] = mine; }
        __syncwarp();
        base = base_next;
        buf ^= 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// TMA = true: the energies of a strip are staged nst chunks of DP_SR rows ahead into shared memory, one tensor copy per
// chunk (cp.async.bulk.tensor.3d, completion on an mbarrier per warp and stage) instead of a register ring of plain
// loads: nothing the cluster barrier's memory fence has to wait for, and up to 64 rows in flight per warp.
constexpr int DP_NST_MAX = 4;     // stages per warp: as many (2..4) as fit into shared memory, chosen by the host

__device__ __forceinline__ uint32_t dp_smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
// bounded parity wait: a protocol error traps after ~2^24 polls instead of hanging the GPU
__device__ __forceinline__ void dp_mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .u32 n;\n"
        "mov.u32 n, 0;\n"
        "DP_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DP_DONE;\n"
        "add.u32 n, n, 1;\n"
        "setp.lt.u32 p, n, 0x1000000;\n"
        "@p bra DP_WAIT;\n"
        "trap;\n"
        "DP_DONE:\n"
        "}" ::"r"(bar), "r"(parity) : "memory");
}

// compile-time loop: f(std::integral_constant<int, 0>) ... f(std::integral_constant<int, N - 1>)
template <int N, int I = 0, typename F>
__device__ __forceinline__ void dp_unroll(F&& f)
{
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        dp_unroll<N, I + 1>(f);
    }
}

// DP_P float4 groups per lane: strip = 128 * DP_P columns, 128 * DP_P - 2 * DP_R of them published.
// DP_SR: rows per staged chunk (32 when two stages per warp fit, else 16), 0 = register ring.  dp_plan instantiates the
// (DP_P, DP_SR) pairs a width can select: (1, 32), (1, 16), (2, 16), (2, 0), (4, 0).
// One cluster per frame: blockIdx.y = frame of a batch session, whose energy / cumulative planes start en_fs / m_fs
// floats after the previous frame's, whose seam is seam[h * frame ...], its log seam_log[log_fs * frame ...] and its
// last-row column xlast[frame].  The tensor map is 3-D (columns, rows, frames) with a box depth of one frame.
// Step: the step rule (see DpStep1, DpSteps), the trailing argument.  Every cell takes the minimum over the rule's
// candidates.  A DpSteps strip exchanges halos every DP_R / dx rows instead of every DP_R (its edge contaminates dx
// columns per row, still at most DP_R after a block); with at least 4 cells per lane every candidate comes from the lane
// or its two neighbours.  The incremental map (run_flag) is DpStep1 only.  Without xlast warp 0 of CTA 0 walks the seam
// back itself (dp_backtrack), with it the jump and trace kernels follow.
template <int DP_P, int DP_SR, typename Step>
__global__ void __cluster_dims__(DP_CL, 1, 1) __launch_bounds__(DP_MAXW * 32) dctc_seam_dp_kernel(const float* __restrict__ en, size_t en_pitch, int w, int h,
                                                                    float* __restrict__ mplane, size_t m_pitch,
                                                                    int* __restrict__ seam, int* __restrict__ seam_log,
                                                                    int* __restrict__ run_flag, int nst,
                                                                    const __grid_constant__ CUtensorMap tmap,
                                                                    int* __restrict__ xlast, size_t en_fs, size_t m_fs, size_t log_fs,
                                                                    typename Step::Arg arg)
{
    const Step st{arg};
    DCTC_PDL_PROLOGUE();
    // (the frame's seam, log and xlast offsets are applied after the row loop, so they occupy no registers in it)
    en += blockIdx.y * en_fs;
    // fallback of the incremental update (dctc_seam_incr_kernel): runs only when that kernel asked for a rebuild
    if (run_flag && *run_flag == 0) return;       // uniform over the cluster, before any cluster barrier
    if (run_flag && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(run_flag + 1, 1);   // rebuilds since the session was loaded
    constexpr bool TMA = DP_SR > 0;
    constexpr int SRD = TMA ? DP_SR : DP_R;       // (divisor that is never zero)
    constexpr int CPL = 4 * DP_P;                 // cells per lane
    constexpr int STRIP = 32 * CPL;               // columns a warp computes
    constexpr int WOUT = STRIP - 2 * DP_R;        // columns a warp publishes
    constexpr int HL = DP_R / CPL;                // halo lanes on each side (DP_R is a multiple of CPL)
    constexpr int PF = TMA ? 1 : 16 / DP_P;       // energy rows in flight per lane (register ring of the non-TMA variant)
    extern __shared__ __align__(128) float xrow[]; // two exchange rows of (warps per CTA * WOUT) floats, double buffered;
                                                  // TMA: followed by warps x nst stages x DP_SR rows x STRIP energies
    __shared__ __align__(8) unsigned long long ebar[DP_MAXW][DP_NST_MAX];
    __shared__ __align__(8) unsigned long long hbar[DP_MAXW][2];   // halo exchange: per warp and slot, counts the neighbours' bytes
    __shared__ __align__(8) unsigned long long rbar;               // CTA 0: counts the strips' last-row minima (8 bytes each)
    __shared__ __align__(8) int2 red_p[DP_CL * DP_MAXW];           // CTA 0: (value bits, column) per strip
    __shared__ float red_v[DP_CL * DP_MAXW];      // per-strip minima, gathered in CTA 0 through distributed shared memory
    __shared__ int red_i[DP_CL * DP_MAXW];
    __shared__ __align__(16) float win[2][32][DP_WINP];
    const int tid = threadIdx.x, lane = tid & 31;
    const int wpc = blockDim.x >> 5;                        // warps (strips) per CTA
    const uint32_t rank = dp_cta_rank();
    const int warp = (int) rank * wpc + (tid >> 5);         // strip index across the cluster
    const int nwarps = DP_CL * wpc;
    const int xlen = wpc * WOUT;
    const float INF = __int_as_float(0x7f800000);
    const int c0 = warp * WOUT - DP_R + lane * CPL;   // first column of this lane (may be < 0 or >= w)
    const bool central = lane >= HL && lane < 32 - HL;

    // Per-lane constants of the strip geometry: which groups start inside the image, which of their cells lie right of
    // it.  Cells outside the image must stay +inf in every row (range clipping); the patch is applied to the computed
    // row, never to a freshly loaded value -- touching the loaded registers right after the load would turn the
    // 8-rows-ahead prefetch into a synchronous load (measured: 425 clk per row instead of ~40).
    bool ld_ok[DP_P];
    unsigned inf_mask[DP_P];
#pragma unroll
    for (int g = 0; g < DP_P; g++) {
        const int x = c0 + 4 * g;
        ld_ok[g] = x >= 0 && x < w;              // x is a multiple of 4 and the row pitch covers round_up(w, 4)
        inf_mask[g] = !ld_ok[g] ? 15u : ((x + 1 >= w ? 2u : 0u) | (x + 2 >= w ? 4u : 0u) | (x + 3 >= w ? 8u : 0u));
    }
    auto patch = [&](float4& v, unsigned m) {
        if (m & 1u) v.x = INF;
        if (m & 2u) v.y = INF;
        if (m & 4u) v.z = INF;
        if (m & 8u) v.w = INF;
    };
    // Every lane loads unconditionally (lanes / rows outside the image re-read a valid address and their cells are
    // patched to +inf): a predicated load is compiled into "load to a temporary + predicated move", i.e. a wait for the
    // data right after the issue, which again serialises the prefetch.
    const float* en_g[DP_P];
#pragma unroll
    for (int g = 0; g < DP_P; g++) en_g[g] = en + (ld_ok[g] ? c0 + 4 * g : 0);
    float* const mframe = mplane + blockIdx.y * m_fs;
    const int hm1 = h - 1;

    // TMA staging of this warp's strip: columns [cs, cs + STRIP), DP_SR rows per stage
    const int cs = warp * WOUT - DP_R;
    float* estage = xrow + 2 * xlen + (size_t) (tid >> 5) * nst * SRD * STRIP;
    const int nchunks = (h - 1 + SRD - 1) / SRD;
    auto issue_chunk = [&](int ch, int st) {   // rows [1 + ch * DP_SR, 1 + (ch + 1) * DP_SR) -> stage st = ch % nst
        // one tensor copy: box = STRIP columns x DP_SR rows x 1 frame; columns left of the image and rows below it are
        // zero-filled by the TMA unit, never read from the next frame
        const uint32_t bar = dp_smem_u32(&ebar[tid >> 5][st]);
        if (lane == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t) (SRD * STRIP * 4)) : "memory");
            asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                         ::"r"(dp_smem_u32(estage + st * SRD * STRIP)), "l"(&tmap), "r"(cs), "r"(1 + ch * SRD), "r"(blockIdx.y), "r"(bar) : "memory");
        }
        __syncwarp();
    };
    if (lane == 0) {
        if (TMA) {
#pragma unroll
            for (int st = 0; st < DP_NST_MAX; st++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&ebar[tid >> 5][st])) : "memory");
        }
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&hbar[tid >> 5][0])) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&hbar[tid >> 5][1])) : "memory");
        if (tid == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dp_smem_u32(&rbar)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (TMA) {
        for (int ch = 0; ch < nst && ch < nchunks; ch++) issue_chunk(ch, ch);
    }
    dp_cluster_sync();   // once: every CTA's halo mbarriers exist before a neighbour's first st.async can arrive

    float4 cur[DP_P], e[PF][DP_P];
#pragma unroll
    for (int g = 0; g < DP_P; g++) {
        cur[g] = __ldg(reinterpret_cast<const float4*>(en_g[g]));
        const int x = c0 + 4 * g;
        if (central && ld_ok[g]) *reinterpret_cast<float4*>(mframe + x) = cur[g];
        patch(cur[g], inf_mask[g]);
        if (!TMA) {
#pragma unroll
            for (int k = 0; k < PF; k++)               // e[k] holds row y with (y - 1) % PF == k
                e[k][g] = __ldg(reinterpret_cast<const float4*>(en_g[g] + (size_t) min(1 + k, hm1) * en_pitch));
        }
    }
#ifdef DCTC_SYNC_DEBUG
    const long long dbg_t0 = clock64();
#endif
    // The row chain is bound by the number of instructions a lone warp per scheduler has to issue (the ncu source view
    // shows ~6 clk per instruction, mostly fixed-latency "wait" stalls), so the loop body is kept minimal: staged
    // energies are read with immediate offsets from a shared-space base register, cells outside the image are made
    // +inf once per chunk in the staged copy (inf + min = inf, no per-row patch), the cumulative plane is written
    // through one running pointer, and whole blocks run without per-row bounds checks.
    float* mptr = mframe + m_pitch + c0;             // this lane's first cell of row y
    unsigned any_mask = 0;
#pragma unroll
    for (int g = 0; g < DP_P; g++) any_mask |= inf_mask[g];
    int xb = 0;
    int hround = 0;                                  // halo exchanges done: slot = hround & 1, mbarrier parity = (hround >> 1) & 1
    int c_ch = 0, c_st = 0;                          // chunk being consumed, its stage and mbarrier parity
    uint32_t c_par = 0;
    uint32_t stg_s = 0;                              // shared-space address of this lane's cells in the current chunk
    auto chunk_begin = [&]() {                       // a new chunk of staged rows starts: wait for it, patch its +inf cells
        dp_mbar_wait(dp_smem_u32(&ebar[tid >> 5][c_st]), c_par);
        float* sp = estage + (size_t) c_st * SRD * STRIP + lane * CPL;
        stg_s = dp_smem_u32(sp);
        if (any_mask) {
            for (int rr = 0; rr < SRD; rr++) {
#pragma unroll
                for (int g = 0; g < DP_P; g++) {
                    float* q = sp + rr * STRIP + 4 * g;
                    if (inf_mask[g] & 1u) q[0] = INF;
                    if (inf_mask[g] & 2u) q[1] = INF;
                    if (inf_mask[g] & 4u) q[2] = INF;
                    if (inf_mask[g] & 8u) q[3] = INF;
                }
            }
        }
    };
    auto chunk_end = [&]() {                         // this warp is done with the chunk: refill its stage nst chunks ahead
        __syncwarp();
        if (c_ch + nst < nchunks) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue_chunk(c_ch + nst, c_st);
        }
        c_ch++;
        if (++c_st == nst) { c_st = 0; c_par ^= 1u; }
    };
    auto row = [&](auto kk_c, int y) {
        constexpr int kk = decltype(kk_c)::value;
        constexpr int k = kk % PF;
        if (TMA) {
#pragma unroll
            for (int g = 0; g < DP_P; g++)
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(e[0][g].x), "=f"(e[0][g].y), "=f"(e[0][g].z), "=f"(e[0][g].w)
                             : "r"(stg_s + (uint32_t) (((kk % SRD) * STRIP + 4 * g) * 4)));   // base register + immediate
        }
        if constexpr (Step::D > 1) {
            // the 4 cells on each side of the lane's cells (neighbour lanes; +inf beyond the strip), then per cell the
            // minimum of cur and fl(neighbour + pen[|d|]) over d = -4 .. 4 (min is exact: the order does not matter)
            constexpr int CW = 4 * DP_P;
            float c[CW + 8];
#pragma unroll
            for (int g = 0; g < DP_P; g++) {
                c[4 + 4 * g] = cur[g].x; c[5 + 4 * g] = cur[g].y; c[6 + 4 * g] = cur[g].z; c[7 + 4 * g] = cur[g].w;
            }
            const float lsrc[4] = {cur[DP_P - 1].x, cur[DP_P - 1].y, cur[DP_P - 1].z, cur[DP_P - 1].w};
            const float rsrc[4] = {cur[0].x, cur[0].y, cur[0].z, cur[0].w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float lv = __shfl_up_sync(0xffffffffu, lsrc[j], 1), rv = __shfl_down_sync(0xffffffffu, rsrc[j], 1);
                c[j] = lane == 0 ? INF : lv;
                c[CW + 4 + j] = lane == 31 ? INF : rv;
            }
            float mn[CW];
#pragma unroll
            for (int i = 0; i < CW; i++) mn[i] = c[4 + i];
#pragma unroll
            for (int d = 1; d <= 4; d++) {
                const float pd = st.pen[d];
                float qd[CW + 8];
#pragma unroll
                for (int i = 4 - d; i < CW + 4 + d; i++) qd[i] = c[i] + pd;
#pragma unroll
                for (int i = 0; i < CW; i++) mn[i] = fminf(mn[i], fminf(qd[4 + i - d], qd[4 + i + d]));
            }
            float4 o[DP_P];
#pragma unroll
            for (int g = 0; g < DP_P; g++) {
                o[g].x = e[k][g].x + mn[4 * g]; o[g].y = e[k][g].y + mn[4 * g + 1];
                o[g].z = e[k][g].z + mn[4 * g + 2]; o[g].w = e[k][g].w + mn[4 * g + 3];
            }
            if (!TMA) {
#pragma unroll
                for (int g = 0; g < DP_P; g++)
                    e[k][g] = __ldg(reinterpret_cast<const float4*>(en_g[g] + (size_t) min(y + PF, hm1) * en_pitch));
            }
#pragma unroll
            for (int g = 0; g < DP_P; g++) {
                if (central && ld_ok[g]) *reinterpret_cast<float4*>(mptr + 4 * g) = o[g];
                if (!TMA) patch(o[g], inf_mask[g]);
                cur[g] = o[g];
            }
            mptr += m_pitch;
        } else {
        // q: the previous row as a diagonal parent sees it (rigidity: cur + pen, one add per cell; else cur itself)
        float4 q[DP_P];
#pragma unroll
        for (int g = 0; g < DP_P; g++)
            q[g] = make_float4(st.diag(cur[g].x), st.diag(cur[g].y), st.diag(cur[g].z), st.diag(cur[g].w));
        // neighbours across lanes; the strip's outermost lanes see +inf (their cells are never published)
        float l = __shfl_up_sync(0xffffffffu, q[DP_P - 1].w, 1);
        float r = __shfl_down_sync(0xffffffffu, q[0].x, 1);
        if (lane == 0) l = INF;
        if (lane == 31) r = INF;
        float4 o[DP_P];
#pragma unroll
        for (int g = 0; g < DP_P; g++) {
            const float lg = g == 0 ? l : q[g > 0 ? g - 1 : 0].w;
            const float rg = g == DP_P - 1 ? r : q[g < DP_P - 1 ? g + 1 : g].x;
            o[g].x = e[k][g].x + fminf(fminf(lg, cur[g].x), q[g].y);
            o[g].y = e[k][g].y + fminf(fminf(q[g].x, cur[g].y), q[g].z);
            o[g].z = e[k][g].z + fminf(fminf(q[g].y, cur[g].z), q[g].w);
            o[g].w = e[k][g].w + fminf(fminf(q[g].z, cur[g].w), rg);
        }
        // register-ring variant: refill the slot just consumed with the row PF ahead (issued after the last use of the
        // slot, so the load targets the slot's registers directly; they are not touched again for PF rows)
        if (!TMA) {
#pragma unroll
            for (int g = 0; g < DP_P; g++)
                e[k][g] = __ldg(reinterpret_cast<const float4*>(en_g[g] + (size_t) min(y + PF, hm1) * en_pitch));
        }
#pragma unroll
        for (int g = 0; g < DP_P; g++) {
            if (central && ld_ok[g]) *reinterpret_cast<float4*>(mptr + 4 * g) = o[g];
            if (!TMA) patch(o[g], inf_mask[g]);      // cells outside the image stay +inf (TMA: their staged energy is +inf)
            cur[g] = o[g];
        }
        mptr += m_pitch;
        }
    };
    // Exchange the last row of a block with the two neighbouring strips only: the outer 32 published cells on each side
    // go straight into the neighbour warp's halo slot (st.async into its CTA's shared memory, completion counted on ITS
    // mbarrier), then this warp waits for the 2 x 128 bytes it expects itself.  No cluster-wide barrier and no memory
    // fence: the release/acquire cluster barrier used before carried MEMBAR.ALL.GPU + CCTL.IVALL, i.e. it also waited
    // for the block's global stores of the cumulative plane (40 % of the kernel's stall samples).
    // Slot xb = block parity: a neighbour can be at most one block ahead, it needs this warp's row to go further.  The
    // slot and the exchange count hround (mbarrier parity (hround >> 1) & 1) are advanced by the caller.
    auto exchange = [&](int xb, int hround) {
        const int wl = tid >> 5;                          // warp inside the CTA
        float* halo = xrow + (wl * 2 + xb) * 64;          // [0,32): cells left of the published range, [32,64): right
        const uint32_t my_bar = dp_smem_u32(&hbar[wl][xb]);
        if (lane == 0) {
            const uint32_t expect = (warp > 0 ? 128u : 0u) + (warp < nwarps - 1 ? 128u : 0u);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(my_bar), "r"(expect) : "memory");
        }
        if (lane >= HL && lane < 2 * HL && warp > 0) {                        // my leftmost 32 published cells
            const int nw = warp - 1;
            const uint32_t nrank = (uint32_t) (nw / wpc);
            const int nwl = nw - (int) nrank * wpc;
            const uint32_t dst = dp_map(xrow + (nwl * 2 + xb) * 64 + 32 + (lane - HL) * CPL, nrank);
            const uint32_t bar = dp_map(&hbar[nwl][xb], nrank);
#pragma unroll
            for (int g = 0; g < DP_P; g++) dp_st_async_v4(dst + 16u * g, cur[g], bar);
        }
        if (lane >= 32 - 2 * HL && lane < 32 - HL && warp < nwarps - 1) {     // my rightmost 32 published cells
            const int nw = warp + 1;
            const uint32_t nrank = (uint32_t) (nw / wpc);
            const int nwl = nw - (int) nrank * wpc;
            const uint32_t dst = dp_map(xrow + (nwl * 2 + xb) * 64 + (lane - (32 - 2 * HL)) * CPL, nrank);
            const uint32_t bar = dp_map(&hbar[nwl][xb], nrank);
#pragma unroll
            for (int g = 0; g < DP_P; g++) dp_st_async_v4(dst + 16u * g, cur[g], bar);
        }
        dp_mbar_wait(my_bar, (uint32_t) ((hround >> 1) & 1));
        if (!central) {
            const float* hp = halo + (lane < HL ? lane * CPL : 32 + (lane - (32 - HL)) * CPL);
#pragma unroll
            for (int g = 0; g < DP_P; g++) {
                const int x = c0 + 4 * g;
                if (x >= 0 && x < w) cur[g] = *reinterpret_cast<const float4*>(hp + 4 * g);   // cells right of the image arrive as +inf
                else cur[g] = make_float4(INF, INF, INF, INF);
            }
        }
    };
    // Two block loops: one for DpStep1 (exchange after every DP_R rows) and one for DpSteps (after every DP_R / dx rows
    // counted from row 0); merged into one, the DpStep1 kernels got another register allocation.  Never after the last row.
    if constexpr (Step::D == 1) {
        for (int yb = 1; yb < h; yb += DP_R) {
            if (yb + DP_R <= h) {                         // whole block: no per-row bounds checks
                dp_unroll<DP_R>([&](auto kk_c) {
                    constexpr int kk = decltype(kk_c)::value;
                    if (TMA && kk % SRD == 0) chunk_begin();
                    row(kk_c, yb + kk);
                    if (TMA && kk % SRD == SRD - 1) chunk_end();
                });
            } else {
                dp_unroll<DP_R>([&](auto kk_c) {
                    constexpr int kk = decltype(kk_c)::value;
                    const int y = yb + kk;
                    if (TMA && kk % SRD == 0 && y < h) chunk_begin();
                    if (y < h) row(kk_c, y);              // uniform across the CTA
                    if (TMA && kk % SRD == SRD - 1) chunk_end();
                });
            }
            if (yb + DP_R < h) {
                exchange(xb, hround);
                xb ^= 1;
                hround++;
            }
        }
    } else {
        const int rb = DP_R / st.dx;
        int since = 0;
        for (int yb = 1; yb < h; yb += DP_R) {
            dp_unroll<DP_R>([&](auto kk_c) {
                constexpr int kk = decltype(kk_c)::value;
                const int y = yb + kk;
                if (TMA && kk % SRD == 0 && y < h) chunk_begin();
                if (y < h) row(kk_c, y);
                if (++since == rb && y + 1 < h) {
                    exchange(xb, hround);
                    xb ^= 1;
                    hround++;
                    since = 0;
                }
                if (TMA && kk % SRD == SRD - 1) chunk_end();
            });
        }
    }
#ifdef DCTC_SYNC_DEBUG
    const long long dbg_t1 = clock64();
#endif
    // leftmost minimum of the last row (central cells only: the others are either duplicates or contaminated)
    float bv = INF;
    int bi = 0x7fffffff;
    if (central) {
#pragma unroll
        for (int g = 0; g < DP_P; g++) {
            const float c4[4] = {cur[g].x, cur[g].y, cur[g].z, cur[g].w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int x = c0 + 4 * g + k;
                if (x >= 0 && x < w && (c4[k] < bv || bi == 0x7fffffff)) { bv = c4[k]; bi = x; }   // ascending x: strict < keeps the leftmost
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if (xlast) {
        // parallel back-track follows in other kernels (the launch boundary publishes the cumulative plane): the strips'
        // minima travel to CTA 0 like the halos (st.async + mbarrier), no cluster barrier and no memory fence at the end
        if (lane == 0)
            asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];"
                         ::"r"(dp_map(&red_p[warp], 0u)), "r"(__float_as_uint(bv)), "r"(bi), "r"(dp_map(&rbar, 0u)) : "memory");
        if (rank == 0 && tid < 32) {
            if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dp_smem_u32(&rbar)), "r"((uint32_t) nwarps * 8u) : "memory");
            dp_mbar_wait(dp_smem_u32(&rbar), 0u);
        }
    } else {
        if (lane == 0) { dp_st_cluster_f32(dp_map(&red_v[warp], 0u), bv); dp_st_cluster_s32(dp_map(&red_i[warp], 0u), bi); }
        dp_cluster_sync();   // release/acquire at cluster scope: also orders every CTA's global writes of the cumulative plane
    }
    if (rank == 0 && tid < 32) {
        const int fz = blockIdx.y;
        seam += (size_t) fz * h;
        if (seam_log) seam_log += fz * log_fs;
        if (xlast) xlast += fz;
        bv = INF;
        bi = 0x7fffffff;
        for (int i = tid; i < nwarps; i += 32) {   // strips in ascending column order: strict < keeps the leftmost
            const float rv = xlast ? __int_as_float(red_p[i].x) : red_v[i];
            const int ri = xlast ? red_p[i].y : red_i[i];
            if (ri != 0x7fffffff && (bi == 0x7fffffff || rv < bv)) { bv = rv; bi = ri; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi != 0x7fffffff && (bi == 0x7fffffff || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
        }
        if (xlast) {
            // parallel back-track: the jump and trace kernels below take over from the seam's last-row column
            if (lane == 0) { *xlast = bi; seam[h - 1] = bi; if (seam_log) seam_log[h - 1] = bi; }
        } else {
            dp_backtrack(mplane + fz * m_fs, m_pitch, w, h, bi, seam, seam_log, win, lane, st);   // serial walk by warp 0 of CTA 0
        }
#ifdef DCTC_SYNC_DEBUG
        if (tid == 0) {
            unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
            printf("dp kernel w %d h %d: chain %lld clk, reduce+backtrack %lld clk, globaltimer %llu ns\n", w, h, dbg_t1 - dbg_t0, clock64() - dbg_t1, gt);
        }
#endif
    }
}

// ---- parallel back-track (build_vpath without the h-step dependent chain) ---------------------------------------
// The serial walk above is a chain of h dependent shared-memory reads (133 clk per row: 73 us of a 1080-row seam).  The
// parent choice of a cell depends only on the cumulative map, not on the path, so the rows are cut into blocks of jb
// rows (counted upwards from the last row) and, for EVERY column x of a block's bottom row, the column its path has at
// the block's top row is computed in parallel: top-down, P_top[x] = x, P_y[x] = P_{y-1}[x + d_y(x)] with d_y(x) the
// parent step of (y, x) -- at most D columns, so a warp keeps a strip of 32 jc columns in registers and exchanges the
// outer cells by shuffles, like the seam DP (jb * D <= 8 jc contaminated columns on each side, 16 jc published).
// dctc_seam_jump_kernel: one warp per (strip, block), the whole grid busy for ~1 us; it stores the jump as an int8
// offset (at most jb * D = 124 columns).  dctc_seam_trace_kernel: one CTA per block; it follows the ceil((h-1)/jb)
// jumps from the seam's last-row column down to its own block (the jump entries a path can reach form a cone of
// 2 jb dx j + 1 columns in block j, staged into shared memory first), then walks its jb rows like dp_backtrack does.
// ~100 dependent steps instead of h.
// The geometry of a rule whose steps reach D columns (DpStep1: D = 1, DpSteps: D = DCTC_MAX_DELTA_X), in one place:
//   jb        jump block rows
//   jc        jump cells per lane: strips of 32 jc columns, the central 16 jc published
//   jr        jump rows of loads in flight
//   win, wl   trace window: columns, of which wl lie left of the block's bottom column
//   cone_max  largest cone (bytes of the trace kernel's dynamic shared memory) of the parallel back-track: D > 1 has less
//             room next to its window's 34 KB of static shared memory
template <int D>
struct BtGeom;
template <>
struct BtGeom<1> { static constexpr int jb = 32, jc = 4, jr = 8, win = 72, wl = 34, cone_max = 200 * 1024; };
template <>
struct BtGeom<DCTC_MAX_DELTA_X> { static constexpr int jb = 31, jc = 16, jr = 4, win = 264, wl = 132, cone_max = 180 * 1024; };
constexpr int JH = 8;             // jump halo lanes on each side of a strip (8 jc >= jb * D)

// Batch sessions: blockIdx.z = frame (planes m_fs floats / j_fs bytes apart).
template <typename Step>
__global__ void __launch_bounds__(128) dctc_seam_jump_kernel(const float* __restrict__ mplane, size_t m_pitch, int w, int h,
                                                             int8_t* __restrict__ jump, size_t j_pitch, int strips,
                                                             size_t m_fs, size_t j_fs, typename Step::Arg arg)
{
    constexpr int D = Step::D;
    using G = BtGeom<D>;
    constexpr int JC = G::jc, NG = JC / 4;         // cells and float4 groups per lane
    const Step st{arg};
    DCTC_PDL_PROLOGUE();
    const int lane = threadIdx.x & 31;
    const int strip = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (strip >= strips) return;
    const int k = blockIdx.y;
    mplane += blockIdx.z * m_fs;
    jump += blockIdx.z * j_fs;
    const int yb = h - 1 - G::jb * k;                  // bottom row of the block
    const int yt = max(yb - G::jb, 0);                 // top row
    const int steps = yb - yt;
    const float INF = __int_as_float(0x7f800000);
    const int c0 = strip * 16 * JC - JH * JC + JC * lane;   // this lane's JC columns
    bool ok[NG];
#pragma unroll
    for (int g = 0; g < NG; g++) ok[g] = c0 + 4 * g >= 0 && c0 + 4 * g < w;     // (multiples of 4: the pitch covers round_up(w, 4))
    const float* const src = mplane + (size_t) yt * m_pitch;
    int P[JC];
#pragma unroll
    for (int i = 0; i < JC; i++) P[i] = c0 + i;
    auto row = [&](const float4 (&v)[NG]) {           // cumulative values of row y-1 -> P of row y
        float e[JC + 2 * D];                          // e[D + i]: column c0 + i, D neighbour cells on each side
        int pe[JC + 2 * D];
#pragma unroll
        for (int g = 0; g < NG; g++) {
            const float c4[4] = {v[g].x, v[g].y, v[g].z, v[g].w};
#pragma unroll
            for (int j = 0; j < 4; j++) e[D + 4 * g + j] = ok[g] && c0 + 4 * g + j < w ? c4[j] : INF;   // range clipping
        }
#pragma unroll
        for (int i = 0; i < JC; i++) pe[D + i] = P[i];
#pragma unroll
        for (int j = 0; j < D; j++) {                 // neighbours across lanes; the strip's outermost lanes see +inf
            const float l = __shfl_up_sync(0xffffffffu, e[JC + j], 1), r = __shfl_down_sync(0xffffffffu, e[D + j], 1);
            pe[j] = __shfl_up_sync(0xffffffffu, P[JC - D + j], 1);
            pe[JC + D + j] = __shfl_down_sync(0xffffffffu, P[j], 1);
            e[j] = lane == 0 ? INF : l;
            e[JC + D + j] = lane == 31 ? INF : r;
        }
#pragma unroll
        for (int i = 0; i < JC; i++) P[i] = st.pick([&](int d) { return e[D + i + d]; }, [&](int d) { return pe[D + i + d]; });
    };
    for (int i0 = 0; i0 < steps; i0 += G::jr) {       // jr rows of independent loads in flight, then jr dependent steps
        float4 pv[G::jr][NG];
#pragma unroll
        for (int j = 0; j < G::jr; j++)
#pragma unroll
            for (int g = 0; g < NG; g++)
                pv[j][g] = __ldcg(reinterpret_cast<const float4*>(src + (ok[g] ? c0 + 4 * g : 0) + (size_t) min(i0 + j, steps - 1) * m_pitch));
#pragma unroll
        for (int j = 0; j < G::jr; j++)
            if (i0 + j < steps) row(pv[j]);
    }
    dp_unroll<NG>([&](auto g_c) {                    // (expanded at compile time: as an unrolled loop, D > 1 takes one register more)
        constexpr int g = decltype(g_c)::value;
        if (lane >= JH && lane < 32 - JH && ok[g]) {
            int8_t* dst = jump + (size_t) k * j_pitch + c0 + 4 * g;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (c0 + 4 * g + j < w) dst[j] = (int8_t) (P[4 * g + j] - (c0 + 4 * g + j));
        }
    });
}

constexpr int TR_THREADS = 256;

// Batch sessions: blockIdx.y = frame (planes m_fs floats / j_fs bytes apart, seam[h * frame ...],
// seam_log[log_fs * frame ...], xlast[frame]).
template <typename Step>
__global__ void __launch_bounds__(TR_THREADS) dctc_seam_trace_kernel(const float* __restrict__ mplane, size_t m_pitch, int w, int h,
                                                              const int8_t* __restrict__ jump, size_t j_pitch,
                                                              const int* __restrict__ xlast, int* __restrict__ seam,
                                                              int* __restrict__ seam_log, size_t m_fs, size_t j_fs, size_t log_fs,
                                                              typename Step::Arg arg)
{
    constexpr int D = Step::D;
    using G = BtGeom<D>;
    const Step st{arg};
    extern __shared__ __align__(16) unsigned char tr_smem[];
    __shared__ __align__(16) float win[G::jb][G::win + 8];
    __shared__ int xb_s;
    DCTC_PDL_PROLOGUE();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int k = blockIdx.x, fz = blockIdx.y;
    mplane += fz * m_fs;
    jump += fz * j_fs;
    seam += (size_t) fz * h;
    if (seam_log) seam_log += fz * log_fs;
    const int x0 = xlast[fz];
    // Cone of block j: its bottom column can be x0 - R j .. x0 + R j, R = jb dx.  The entries are staged as aligned
    // 16-byte chunks (at most (R8 / 8) j + 3 per row, R8 = R rounded up to 8, at byte offset R8 j (j - 1) + 48 j of the
    // cone buffer); warp w takes the rows j = w, w + 8, ... and issues all chunks of a row before it stores any of them,
    // so the loads of a row (and of the other warps' rows) are in flight together instead of one L2 round trip per
    // iteration.
    const int R = G::jb * st.dx, R8 = (R + 7) & ~7;
    for (int j = wid; j < k; j += TR_THREADS / 32) {
        const int a0 = max(0, x0 - R * j) & ~15;
        const int last = min(w - 1, x0 + R * j);
        const int nchunk = ((last - a0) >> 4) + 1;                          // <= (R8 / 8) j + 3
        const uint4* srcj = reinterpret_cast<const uint4*>(jump + (size_t) j * j_pitch + a0);
        uint4* dstj = reinterpret_cast<uint4*>(tr_smem + R8 * j * j + (48 - R8) * j);
        for (int c0 = 0; c0 < nchunk; c0 += 160) {                          // (one pass up to 1080 rows at dx = 1, two beyond)
            uint4 v[5];
#pragma unroll
            for (int i = 0; i < 5; i++)
                if (c0 + lane + 32 * i < nchunk) v[i] = __ldcg(srcj + c0 + lane + 32 * i);
#pragma unroll
            for (int i = 0; i < 5; i++)
                if (c0 + lane + 32 * i < nchunk) dstj[c0 + lane + 32 * i] = v[i];
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int8_t* cone = reinterpret_cast<const int8_t*>(tr_smem);
        int x = x0;
        for (int j = 0; j < k; j++) x += cone[R8 * j * j + (48 - R8) * j + (x - (max(0, x0 - R * j) & ~15))];
        xb_s = x;
    }
    __syncthreads();
    int x = xb_s;
    const int yb = h - 1 - G::jb * k, yt = max(yb - G::jb, 0), steps = yb - yt;
    // window rows: win[i] = cumulative row yb-1-i, columns base .. base+win-1 at win[i][4 + c - base]
    const int max_base = (int) m_pitch - G::win;                   // >= 0: bt_plan asks for m_pitch >= win
    int base = (x - G::wl) & ~3;
    base = base < 0 ? 0 : (base > max_base ? max_base : base);
    for (int idx = tid; idx < steps * (G::win / 4); idx += TR_THREADS) {
        const int i = idx / (G::win / 4), c = idx - i * (G::win / 4);
        const float* src = mplane + (size_t) (yb - 1 - i) * m_pitch + base + 4 * c;
        *reinterpret_cast<float4*>(&win[i][4 + 4 * c]) = __ldcg(reinterpret_cast<const float4*>(src));
    }
    __syncthreads();
    if (tid >= 32) return;
    const float INF = __int_as_float(0x7f800000);
    // D +inf sentinels left of column 0 and from column w on (range clipping), so that the walk needs no bounds checks
    if (lane < steps) {
        if (base == 0)
            for (int j = 0; j < D; j++) win[lane][4 - D + j] = INF;
        if (w - base >= 0 && w - base <= G::win)
            for (int j = 0; j < D; j++) win[lane][4 + w - base + j] = INF;
    }
    __syncwarp();
    int mine = 0;
    const float* wp = &win[0][4] + (x - base);
    for (int i = 0; i < steps; i++) {
        const int d = st.pick([&](int c) { return wp[c]; }, [](int c) { return c; });
        x += d;
        wp += G::win + 8 + d;
        if (lane == i) mine = x;
    }
    if (lane < steps) { seam[yb - 1 - lane] = mine; if (seam_log) seam_log[yb - 1 - lane] = mine; }
}

// ---- incremental cumulative map (liblqr's update_mmap) -----------------------------------------------------------
// After a seam is removed only part of the cumulative map changes: the cells inside the energy band of the removed seam
// (their energy, or the identity of their parents, changed) and, row after row, the cells below a cell whose value
// changed.  liblqr's update_mmap walks the rows with exactly that shrinking / growing column range instead of
// rebuilding the map (lqr_carver_resize, src/render.c:377).  Here one warp does the walk: the cumulative plane was
// compacted over the seam by the carve kernel, row y is recomputed for x in
//     R(y) = band(y)  U  [first changed cell of row y-1  - 1,  last changed cell of row y-1  + 1]
// with the same FP32 formula as the full rebuild, so the plane (and every later seam) is bit-identical to it.
// R(y) grows by at most one column per side and row, so the energies and old map values a row can need are known
// INCR_D rows ahead: they are staged with cp.async into a shared-memory ring, and the walk itself touches shared memory
// only (lane l owns the columns lo + l + 32k; the recomputed row is handed to the next one through a double buffer with
// two unchanged cells on each side).  R(y) wider than INCR_CAP columns raises the rebuild flag and the full DP kernel
// takes over for this seam.  The walk ends with the leftmost minimum of the last row and the same back-track as the
// full kernel.
// MEASURED (1920x1080 noise, 480 seams): the walk recomputes ~150 columns per row on average and needs the full rebuild
// for 2 of 480 seams, but ONE warp spends ~900 clk per row on it (phases per row: 250-470 clk row arithmetic, ~180 clk
// side cells + next range, ~340 clk staging; a lone warp has no other warp to hide its 4-6 clk dependent-issue
// latencies behind), i.e. 918 us per seam against 199 us for the cluster-wide rebuild.  It is therefore OFF by default
// (dctc_carver_set_incremental) and kept as the bit-identical reference point for a multi-warp block version.
#ifndef DCTC_INCR_ABL
#define DCTC_INCR_ABL 0   // timing ablations only
#endif
constexpr int INCR_CAP = 512;                           // widest recomputed range per row
constexpr int INCR_D = 8;                               // rows staged ahead
constexpr int INCR_T = 8;                               // rows between two tightenings of the recomputed range
constexpr int INCR_SW = INCR_CAP + 2 * INCR_D + 16;     // floats per staged row and plane

// one row of the walk with NK columns per lane: every shared-memory load first, then the arithmetic and the stores
template <int NK, typename Step>
__device__ __forceinline__ void incr_row(int y, int lane, int lo, int hi, int w, int plo, const float* __restrict__ re,
                                         const float* __restrict__ rm, int xs, const float* __restrict__ prev,
                                         float* __restrict__ next, float* __restrict__ mrow, int& clo, int& chi, const Step& st)
{
    const float INF = __int_as_float(0x7f800000);
    float e[NK], mo[NK], pl[NK], pc[NK], pr[NK];
#pragma unroll
    for (int k = 0; k < NK; k++) {
        const int xc = min(lo + lane + 32 * k, hi);
        e[k] = re[xc - xs];
        mo[k] = rm[xc - xs];
        const int i = y > 0 ? xc - plo + 2 : 1;
        pl[k] = prev[i - 1];
        pc[k] = prev[i];
        pr[k] = prev[i + 1];
    }
#pragma unroll
    for (int k = 0; k < NK; k++) {
        const int x = lo + lane + 32 * k;
        if (x <= hi) {
            float mn = e[k];
            if (y > 0) mn = e[k] + fminf(fminf(x > 0 ? st.diag(pl[k]) : INF, pc[k]), x < w - 1 ? st.diag(pr[k]) : INF);
            next[x - lo + 2] = mn;
            if (__float_as_uint(mn) != __float_as_uint(mo[k])) {
#if DCTC_INCR_ABL != 1
                mrow[x] = mn;
#endif
                clo = min(clo, x);
                chi = max(chi, x);
            }
        }
    }
}

// Step: DpStep1, as in the DP (the changed cells spread by one column per row).
template <typename Step>
__global__ void __launch_bounds__(32) dctc_seam_incr_kernel(const float* __restrict__ en, size_t en_pitch, int w, int h,
                                                            float* __restrict__ mplane, size_t m_pitch, int r,
                                                            int* __restrict__ seam, int* __restrict__ seam_log,
                                                            int* __restrict__ rebuild_flag, typename Step::Arg arg)
{
    const Step st{arg};
    extern __shared__ __align__(16) int incr_sm[];
    float* ring = reinterpret_cast<float*>(incr_sm);                       // INCR_D slots x (energy row, map row) x INCR_SW
    float* buf = ring + INCR_D * 2 * INCR_SW;                              // two hand-over rows of INCR_CAP + 4 cells
    int* xsb = reinterpret_cast<int*>(buf + 2 * (INCR_CAP + 4));           // first staged column per slot
    int* bmin = xsb + INCR_D;                                              // band of the removed seam per row
    int* bmax = bmin + h;
    __shared__ __align__(16) float win[2][32][DP_WINP];
    const int lane = threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    if (lane == 0) *rebuild_flag = 0;
    for (int y = lane; y < h; y += 32) {
        int lo, hi;
        dctc_band_limits(seam, y, h, w, r, &lo, &hi);
        bmin[y] = lo;
        bmax[y] = hi;
    }
    __syncwarp();
    const int xmax4 = ((w + 3) & ~3) - 1;             // last column of the 16-byte chunk that holds column w-1
    // stage row ys (columns that R(ys) and its two neighbours on each side can reach from the range [lo, hi] of a row
    // at most INCR_D above it) into ring slot ys % INCR_D
    auto stage = [&](int ys, int lo, int hi) {
        if (ys < h) {
            const int slot = ys % INCR_D;
            const int s0 = max(0, lo - INCR_D - 2) & ~3, s1 = min(xmax4, (hi + INCR_D + 2) | 3);
            if (lane == 0) xsb[slot] = s0;
            const float* ge = en + (size_t) ys * en_pitch + s0;
            const float* gm = mplane + (size_t) ys * m_pitch + s0;
            float* de = ring + slot * 2 * INCR_SW;
            float* dm = de + INCR_SW;
            const int nch = (s1 - s0 + 1) >> 2;
            for (int c = lane; c < nch; c += 32) {
                asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t) __cvta_generic_to_shared(de + 4 * c)), "l"(ge + 4 * c) : "memory");
                asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t) __cvta_generic_to_shared(dm + 4 * c)), "l"(gm + 4 * c) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    int lo = bmin[0], hi = bmax[0];
    if (hi - lo + 1 > INCR_CAP) {
        if (lane == 0) *rebuild_flag = 1;
        return;
    }
    for (int ys = 0; ys < INCR_D; ys++) stage(ys, lo, hi);
    float* prev = buf;
    float* next = buf + INCR_CAP + 4;
    int plo = 0;                                      // prev[i] holds the cell x = plo - 2 + i of row y-1
#ifdef DCTC_INCR_STATS
    int stat_w = 0;
    long long st[5] = {0, 0, 0, 0, 0};
    const long long stat_t0 = clock64();
#endif
    for (int y = 0; y < h; y++) {
        const int width = hi - lo + 1;
#ifdef DCTC_INCR_STATS
        stat_w += width;
#endif
        if (width > INCR_CAP) {                       // uniform
            if (lane == 0) *rebuild_flag = 1;
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            return;
        }
#ifdef DCTC_INCR_STATS
        const long long c0 = clock64();
#endif
        asm volatile("cp.async.wait_group %0;" ::"n"(INCR_D - 1) : "memory");   // row y has landed (own copies)
        __syncwarp();                                                            // ... and everybody's
#ifdef DCTC_INCR_STATS
        const long long c1 = clock64();
#endif
        const int slot = y % INCR_D;
        const float* re = ring + slot * 2 * INCR_SW;
        const float* rm = re + INCR_SW;
        const int xs = xsb[slot];
        float* mrow = mplane + (size_t) y * m_pitch;
        int clo = 0x7fffffff, chi = -1;
        if (width <= 32) incr_row<1>(y, lane, lo, hi, w, plo, re, rm, xs, prev, next, mrow, clo, chi, st);
        else if (width <= 64) incr_row<2>(y, lane, lo, hi, w, plo, re, rm, xs, prev, next, mrow, clo, chi, st);
        else if (width <= 128) incr_row<4>(y, lane, lo, hi, w, plo, re, rm, xs, prev, next, mrow, clo, chi, st);
        else if (width <= 256) incr_row<8>(y, lane, lo, hi, w, plo, re, rm, xs, prev, next, mrow, clo, chi, st);
        else incr_row<16>(y, lane, lo, hi, w, plo, re, rm, xs, prev, next, mrow, clo, chi, st);
#ifdef DCTC_INCR_STATS
        const long long c2 = clock64();
#endif
        if (lane < 4) {   // two unchanged cells on each side of the range, from the staged (old) map row
            const int xe = lane < 2 ? lo - 2 + lane : hi + lane - 1;
            const int idx = lane < 2 ? lane : width + lane;
            next[idx] = (xe >= 0 && xe < w) ? rm[xe - xs] : INF;
        }
        // Next range.  Finding the changed cells is a warp-wide reduction on the row-to-row critical path, so it is done
        // only every INCR_T rows; in between the range simply grows by one column per side (a superset of R(y+1):
        // cells recomputed without need come out bit-identical, and band(y+1) lies inside band(y) +- 1).
        int nlo = max(lo - 1, 0), nhi = min(hi + 1, w - 1);
        if ((y & (INCR_T - 1)) == INCR_T - 1 && y + 1 < h) {
            clo = __reduce_min_sync(0xffffffffu, clo);
            chi = __reduce_max_sync(0xffffffffu, chi);
            nlo = bmin[y + 1];
            nhi = bmax[y + 1];
            if (chi >= 0) { nlo = min(nlo, clo - 1); nhi = max(nhi, chi + 1); }
            nlo = max(nlo, 0);
            nhi = min(nhi, w - 1);
        }
        plo = lo;
        float* t = prev; prev = next; next = t;
        lo = nlo;
        hi = nhi;
#ifdef DCTC_INCR_STATS
        const long long c3 = clock64();
#endif
        __syncwarp();                                 // hand-over row written, ring slot of row y read by everybody
#ifdef DCTC_INCR_STATS
        const long long c4 = clock64();
#endif
#if DCTC_INCR_ABL == 2
        asm volatile("cp.async.commit_group;" ::: "memory");
#else
        if (hi - lo + 1 <= INCR_CAP) stage(y + INCR_D, lo, hi);                  // refills the slot row y sat in
        else asm volatile("cp.async.commit_group;" ::: "memory");
#endif
#ifdef DCTC_INCR_STATS
        st[0] += c1 - c0; st[1] += c2 - c1; st[2] += c3 - c2; st[3] += c4 - c3; st[4] += clock64() - c4;
#endif
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#ifdef DCTC_INCR_STATS
    if (lane == 0) { atomicAdd(rebuild_flag + 2, stat_w / 16); atomicAdd(rebuild_flag + 3, (int) ((clock64() - stat_t0) >> 10));
        if (w == 1900) printf("walk phases (clk per row): wait %lld, row %lld, ext+range %lld, syncwarp %lld, stage %lld\n", st[0] / h, st[1] / h, st[2] / h, st[3] / h, st[4] / h); }
#endif
    __threadfence();
    __syncwarp();
    // leftmost minimum of the last row (from L2: part of it was just rewritten)
    const float* last = mplane + (size_t) (h - 1) * m_pitch;
    float bv = INF;
    int bi = 0x7fffffff;
    for (int x = lane; x < w; x += 32) {
        const float v = __ldcg(last + x);
        if (v < bv || bi == 0x7fffffff) { bv = v; bi = x; }     // ascending x per lane: strict < keeps the leftmost
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    dp_backtrack(mplane, m_pitch, w, h, bi, seam, seam_log, win, lane, st);
}

// Instantiated here, ahead of the DP kernels: the module then declares the dynamic shared arrays of the trace and
// incremental kernels before the DP's 128-byte aligned one, which keeps the trace kernel's dynamic shared memory at the
// 16-byte aligned offset its static arrays end at.
template __global__ void dctc_seam_jump_kernel<DpStep1<false>>(const float*, size_t, int, int, int8_t*, size_t, int, size_t, size_t, float);
template __global__ void dctc_seam_jump_kernel<DpStep1<true>>(const float*, size_t, int, int, int8_t*, size_t, int, size_t, size_t, float);
template __global__ void dctc_seam_trace_kernel<DpStep1<false>>(const float*, size_t, int, int, const int8_t*, size_t, const int*, int*,
                                                                int*, size_t, size_t, size_t, float);
template __global__ void dctc_seam_trace_kernel<DpStep1<true>>(const float*, size_t, int, int, const int8_t*, size_t, const int*, int*,
                                                               int*, size_t, size_t, size_t, float);
template __global__ void dctc_seam_incr_kernel<DpStep1<false>>(const float*, size_t, int, int, float*, size_t, int, int*, int*, int*, float);
template __global__ void dctc_seam_incr_kernel<DpStep1<true>>(const float*, size_t, int, int, float*, size_t, int, int*, int*, int*, float);
template __global__ void dctc_seam_jump_kernel<DpSteps>(const float*, size_t, int, int, int8_t*, size_t, int, size_t, size_t, DpSteps);
template __global__ void dctc_seam_trace_kernel<DpSteps>(const float*, size_t, int, int, const int8_t*, size_t, const int*, int*, int*,
                                                         size_t, size_t, size_t, DpSteps);

// ---- visibility map + seam display (SURVEY section 8f rank 4) ---------------------------------------------------
// liblqr's update_vsmap: the pixel removed from row y by the k-th seam is original column raw[y][s]; its entry of the
// visibility map becomes k (1-based).  raw is compacted over the seam like the image (one CTA per row).  Batch sessions:
// blockIdx.y = frame, whose maps follow the previous frame's (w0 x h ints each) and whose seam is seam[h * frame ...].
__global__ void __launch_bounds__(256) dctc_vs_update_kernel(int* __restrict__ raw, int* __restrict__ vs, int w0,
                                                             const int* __restrict__ seam, int w_old, int order)
{
    DCTC_PDL_PROLOGUE();
    const int y = blockIdx.x;
    const size_t f0 = (size_t) blockIdx.y * gridDim.x;       // first row of this frame
    int* rrow = raw + (f0 + y) * w0;
    const int s = seam[f0 + y];
    if (threadIdx.x == 0) vs[(f0 + y) * w0 + rrow[s]] = order;
    for (int base = s; base < w_old - 1; base += 256 * 4) {
        int v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int x = base + k * 256 + threadIdx.x;
            v[k] = x < w_old - 1 ? rrow[x + 1] : 0;
        }
        __syncthreads();   // all loads of this chunk (incl. rrow[s] above) before any store; also orders chunk after chunk
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int x = base + k * 256 + threadIdx.x;
            if (x < w_old - 1) rrow[x] = v[k];
        }
    }
}

__global__ void __launch_bounds__(256) dctc_iota_rows_kernel(int* __restrict__ raw, int w0, int h)
{
    const size_t i = (size_t) blockIdx.x * 256 + threadIdx.x;
    if (i < (size_t) w0 * h) raw[i] = (int) (i % (size_t) w0);
}

// display_carver_seams (src/render.c:204-240): for x < w-1, y < h-1, every removed pixel becomes (0, 255*vis/depth, 0)
__global__ void __launch_bounds__(256) dctc_paint_seams_kernel(uint8_t* __restrict__ img, size_t pitch, int channels, int w, int h,
                                                               const int* __restrict__ vs, int depth)
{
    const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
    if (x >= w - 1 || y >= h - 1) return;
    const int vis = vs[(size_t) y * w + x];
    if (vis == 0) return;
    uint8_t* p = img + (size_t) y * pitch + (size_t) x * channels;
    p[0] = 0;
    if (channels > 1) p[1] = (uint8_t) (255.0 * ((double) vis) / ((double) depth));
    if (channels > 2) p[2] = 0;
}

// ---- seam enlarging (lqr_carver_resize to a larger size, src/render.c:357-363,377) ----------------------------------
// liblqr's lqr_carver_inflate [from memory: PARITY UNPINNED]: every pixel the first n seams went through is doubled;
// the new pixel sits on its left and holds the integer mean (a + b) / 2 of the pixel and its left neighbour in the
// original row (a copy in column 0).  One CTA per row: block-wide prefix sum of the "seam pixel" flags gives every
// original pixel its output column.  Batch sessions: blockIdx.y = frame, whose source image, visibility map and output
// image start orig_fs bytes, vs_fs ints and out_fs bytes after the previous frame's.
// BIAS: the bias planes of a biased session are inflated in the same pass with the copy rule (both copies of a doubled
// pixel carry its bias): borig rows bpitch floats and frames bfs floats apart, bout rows bout_pitch and frames bout_fs.
template <bool BIAS>
__global__ void __launch_bounds__(256) dctc_inflate_rows_kernel(const uint8_t* __restrict__ orig, size_t pitch, int channels, int w0,
                                                                const int* __restrict__ vs, int n, uint8_t* __restrict__ out, size_t out_pitch,
                                                                size_t orig_fs, size_t vs_fs, size_t out_fs,
                                                                const float* __restrict__ borig, size_t bpitch, size_t bfs,
                                                                float* __restrict__ bout, size_t bout_pitch, size_t bout_fs)
{
    __shared__ int wsum[8];
    __shared__ int running;
    const int y = blockIdx.x, z = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint8_t* src = orig + z * orig_fs + (size_t) y * pitch;
    uint8_t* dst = out + z * out_fs + (size_t) y * out_pitch;
    const int* vrow = vs + z * vs_fs + (size_t) y * w0;
    if (tid == 0) running = 0;
    __syncthreads();
    for (int base = 0; base < w0; base += 256) {
        const int x = base + tid;
        const int v = x < w0 ? vrow[x] : 0;
        const int flag = (v > 0 && v <= n) ? 1 : 0;
        int inc = flag;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        int before = running;
        for (int k = 0; k < wid; k++) before += wsum[k];
        const int pos = x + before + inc - flag;          // output column of the (possibly inserted) first pixel
        if (x < w0) {
            const uint8_t* p = src + (size_t) x * channels;
            uint8_t* q = dst + (size_t) pos * channels;
            if (flag) {
                for (int c = 0; c < channels; c++) q[c] = x > 0 ? (uint8_t) (((int) p[c - channels] + (int) p[c]) / 2) : p[c];
                q += channels;
            }
            for (int c = 0; c < channels; c++) q[c] = p[c];
            if constexpr (BIAS) {
                const float b = borig[z * bfs + (size_t) y * bpitch + x];
                float* bq = bout + z * bout_fs + (size_t) y * bout_pitch + pos;
                bq[0] = b;
                if (flag) bq[1] = b;
            }
        }
        __syncthreads();
        if (tid == 255) running = before + inc;
        __syncthreads();
    }
}

// ---- levels: every extent within the depth of one seam loop (liblqr's interactive resize) ------------------------------
// After a seam loop to depth n with visibility maps, the start image shrunk by k <= n seams is the row's pixels with
// vs == 0 || vs > k in their original order.  One CTA per row reads the row's map and pixels once and writes that row of
// every level of the table: a kept pixel's output column is x minus the pixels before it with 1 <= vs <= k, from one
// ballot per warp and level and the warps' counts in shared memory.  Chunks of 256 columns with a running count per level,
// as in dctc_inflate_rows_kernel, so any width the seam DP covers fits.  blockIdx.y = frame (source image, map orig_fs
// bytes and vs_fs ints after the previous frame's).  Level l is w0 - k[l] wide; its frames start at out + off[l], rows
// packed ((w0 - k) * channels bytes), frames h rows apart.
constexpr int LV_MAX = 32;   // levels per launch (the 256 threads hold one (level, warp) prefix each)
struct LevelTable {
    int n;
    int k[LV_MAX];
    size_t off[LV_MAX];
};

__global__ void __launch_bounds__(256) dctc_levels_gather_kernel(const uint8_t* __restrict__ orig, size_t pitch, int channels, int w0,
                                                                 const int* __restrict__ vs, size_t orig_fs, size_t vs_fs,
                                                                 const LevelTable lv, uint8_t* __restrict__ out)
{
    __shared__ int wsum[LV_MAX][8];      // removed pixels of the chunk in each warp
    __shared__ int wpre[LV_MAX][8];      // removed pixels of the row before each warp's part of the chunk
    __shared__ int running[LV_MAX];
    __shared__ int ks[LV_MAX];
    __shared__ size_t offs[LV_MAX];
    const int y = blockIdx.x, z = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nl = lv.n;
    const uint8_t* src = orig + z * orig_fs + (size_t) y * pitch;
    const int* vrow = vs + z * vs_fs + (size_t) y * w0;
    const size_t row0 = (size_t) z * gridDim.x + y;   // row index of this row in a level's frames
    const unsigned below = (1u << lane) - 1u;
    if (tid < nl) {
        running[tid] = 0;
        ks[tid] = lv.k[tid];
        offs[tid] = lv.off[tid];
    }
    __syncthreads();
    for (int base = 0; base < w0; base += 256) {
        const int x = base + tid;
        const bool in = x < w0;
        const int v = in ? vrow[x] : 0;
        uint8_t px[4];
#pragma unroll
        for (int c = 0; c < 4; c++)
            if (c < channels && in) px[c] = src[(size_t) x * channels + c];
        for (int l = 0; l < nl; l++) {
            const unsigned m = __ballot_sync(0xffffffffu, v >= 1 && v <= ks[l]);
            if (lane == 0) wsum[l][wid] = __popc(m);
        }
        __syncthreads();
        {
            const int l = tid >> 3, w = tid & 7;
            if (l < nl) {
                int s = running[l];
                for (int j = 0; j < w; j++) s += wsum[l][j];
                wpre[l][w] = s;
            }
        }
        __syncthreads();
        if (tid < nl) running[tid] = wpre[tid][7] + wsum[tid][7];
        for (int l = 0; l < nl; l++) {
            const int k = ks[l];
            const bool gone = v >= 1 && v <= k;
            const unsigned m = __ballot_sync(0xffffffffu, gone);
            if (in && !gone) {
                const int e = w0 - k, col = x - wpre[l][wid] - __popc(m & below);
                uint8_t* q = out + offs[l] + (row0 * e + col) * channels;
#pragma unroll
                for (int c = 0; c < 4; c++)
                    if (c < channels) q[c] = px[c];
            }
        }
        __syncthreads();
    }
}

// ---- bias (lqr_carver_bias_add: preserve / discard masks) ------------------------------------------------------------
// The seam energy of a biased session, after a full K1 of its frames: en = fl(en + fl(bias / ext)), ext = the frames'
// start width.  __fdiv_rn / __fadd_rn: IEEE division and add whatever the compiler flags (the band K1's bias store
// computes the same).  blockIdx.y = row, blockIdx.z = frame (planes fs floats apart).
__global__ void __launch_bounds__(256) dctc_bias_add_kernel(float* __restrict__ en, const float* __restrict__ bias, size_t pitch,
                                                            size_t fs, int w, float ext)
{
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= w) return;
    const size_t i = blockIdx.z * fs + (size_t) blockIdx.y * pitch + x;
    en[i] = __fadd_rn(en[i], __fdiv_rn(bias[i], ext));
}

// ---- carver sessions: host side -------------------------------------------------------------------------------------
// A session keeps its device state in CarverFrames sets (dctc_launch.h) of n equally sized frames (one for the context's
// single session).  The kernels above take the frame from a spare grid dimension, so one launch per phase serves every
// frame and each frame's seam DP runs on its own cluster of DP_CL CTAs; a frame gets exactly the seams, image, energy
// plane and visibility map whatever the number of frames around it.

constexpr int DP_MAX_W = DP_CL * DP_MAXW * (512 - 2 * DP_R);   // widest frame the seam DP's strips cover

// Geometry of n frames of w x h pixels: image rows 16-byte aligned, energy rows a multiple of 4 floats, cumulative rows
// at least one back-track window (DP_WIN floats) wide, so that the windows stay inside the plane.
static void frames_init(CarverFrames& f, int n, int w, int h, int ch)
{
    f.n = n; f.w0 = f.w = w; f.h = h; f.ch = ch;
    f.pitch = ((size_t) w * ch + 15) & ~(size_t) 15;
    f.img_fs = f.pitch * h;
    f.en_pitch = ((size_t) w + 3) & ~(size_t) 3;
    f.m_pitch = f.en_pitch < (size_t) DP_WIN ? (size_t) DP_WIN : f.en_pitch;
}

static void frames_free(CarverFrames& f)
{
    cudaFree(f.img); cudaFree(f.en); cudaFree(f.m); cudaFree(f.dir); cudaFree(f.seam); cudaFree(f.xlast);
    cudaFree(f.seam_log); cudaFree(f.raw); cudaFree(f.vs); cudaFree(f.scratch); cudaFree(f.bias); cudaFree(f.en_op);
    f = CarverFrames();
}

// Images, energy planes and seams; the seam loop adds its planes on first use (frames_loop_buffers), visibility maps are
// added by frames_vmaps.
static int frames_alloc(dctc_context* ctx, CarverFrames& f)
{
    const size_t n = (size_t) f.n, h = (size_t) f.h;
    CK(ctx, cudaMalloc((void**) &f.img, f.img_fs * n));
    CK(ctx, cudaMalloc((void**) &f.en, sizeof(float) * f.en_pitch * h * n));
    CK(ctx, cudaMemsetAsync(f.en, 0, sizeof(float) * f.en_pitch * h * n, ctx->stream));
    CK(ctx, cudaMalloc((void**) &f.seam, sizeof(int) * h * n));
    CK(ctx, cudaMalloc((void**) &f.xlast, sizeof(int) * n));
    CK(ctx, cudaMemsetAsync(f.xlast, 0, sizeof(int) * n, ctx->stream));
    return DCTC_OK;
}

// Empty visibility maps (w0 x h ints per frame) and the identity column map raw[frame][y][x] = x, allocated when the frames
// have none.
static int frames_vmaps(dctc_context* ctx, CarverFrames& f)
{
    const size_t nv = (size_t) f.w0 * f.h * f.n;
    if (!f.raw) {
        cudaFree(f.vs);
        f.vs = nullptr;
        CK(ctx, cudaMalloc((void**) &f.vs, sizeof(int) * nv));
        CK(ctx, cudaMalloc((void**) &f.raw, sizeof(int) * nv));
    }
    CK(ctx, cudaMemsetAsync(f.vs, 0, sizeof(int) * nv, ctx->stream));
    dctc_iota_rows_kernel<<<(unsigned) ((nv + 255) / 256), 256, 0, ctx->stream>>>(f.raw, f.w0, f.h * f.n);
    CK(ctx, cudaGetLastError());
    ctx->launches++;
    f.depth = 0;
    f.vs_w = f.w0;
    return DCTC_OK;
}

// frames_vmaps unless the maps are as it left them (only the seam loop's map update changes them, and it counts depth)
static int frames_fresh_vmaps(dctc_context* ctx, CarverFrames& f)
{
    if (f.raw && f.depth == 0 && f.vs_w == f.w0 && f.w == f.w0) return DCTC_OK;
    return frames_vmaps(ctx, f);
}

// A carver session keeps one arithmetic for the whole seam loop: the per-seam band updates run in the FP32 tile kernel, so
// full maps use the bit-identical FP32 march kernel rather than the tensor-core kernel (liblqr: update_emap must reproduce
// what build_emap would give on the carved image).
static DctcK1Op carver_op(DctcK1Op op)
{
    if (op.kernel == DCTC_KERNEL_AUTO || op.kernel == DCTC_KERNEL_TC_SPLIT || op.kernel == DCTC_KERNEL_FP32_STREAM)
        op.kernel = DCTC_KERNEL_FP32_MARCH;
    return op;
}

// K1 over the frames' current images into their energy planes; with a seam (h per frame), band mode around it with the
// operator's band radius
static DctcK1Args frames_k1_args(const CarverFrames& f, const DctcK1Op& op, const int* seam)
{
    DctcK1Args a;
    memset(&a, 0, sizeof(a));
    a.img = f.img; a.pitch = f.pitch; a.w = f.w; a.h = f.h; a.channels = f.ch;
    a.out = f.en; a.out_pitch = f.en_pitch;
    a.frame_stride = f.img_fs; a.out_frame_stride = f.en_pitch * f.h;
    if (seam) {
        a.seam = seam; a.seam_frame_stride = f.h;
        a.band_r = op.blocksize / 2; a.band_stride = 4 * (op.blocksize / 2);
    }
    return a;
}

// The frames' energy planes from scratch: one K1 launch, and for biased frames one bias-add launch that turns the
// operator map into the seam energy
static int frames_full_energy(dctc_context* ctx, const CarverFrames& f, const DctcK1Op& op)
{
    DctcK1Args a = frames_k1_args(f, op, nullptr);
    const int rc = dctc_run_k1(ctx, op, a, f.n, ctx->stream);
    if (rc || !f.bias) return rc;
    dctc_bias_add_kernel<<<dim3((f.w + 255) / 256, f.h, f.n), 256, 0, ctx->stream>>>(f.en, f.bias, f.en_pitch, f.en_pitch * f.h, f.w,
                                                                                     (float) f.w0);
    CK(ctx, cudaGetLastError());
    ctx->launches++;
    return DCTC_OK;
}

// The operator energy maps of the frames: their energy planes, or for biased frames (whose planes hold the seam energy)
// one full K1 of the current images into en_op.  Band updates equal a full recompute bit for bit, so this is the map the
// frames would hold without a bias.
static int frames_op_energy(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, const float** plane)
{
    *plane = f.en;
    if (!f.bias) return DCTC_OK;
    if (!f.en_op) CK(ctx, cudaMalloc((void**) &f.en_op, sizeof(float) * f.en_pitch * f.h * f.n));
    DctcK1Args a = frames_k1_args(f, op, nullptr);
    a.out = f.en_op;
    const int rc = dctc_run_k1(ctx, op, a, f.n, ctx->stream);
    if (rc) return rc;
    *plane = f.en_op;
    return DCTC_OK;
}

// Gives `to` a bias plane (laid out like its energy planes) when `from` has one, and none otherwise
static int frames_bias_like(dctc_context* ctx, const CarverFrames& from, CarverFrames& to)
{
    if (!from.bias) {
        cudaFree(to.bias);
        to.bias = nullptr;
    } else if (!to.bias) {
        CK(ctx, cudaMalloc((void**) &to.bias, sizeof(float) * to.en_pitch * to.h * to.n));
    }
    return DCTC_OK;
}

// ---- the way out: everything the caller sees is in image orientation --------------------------------------------------
// Transposed frames (a height operation's, frames_transpose) hold the images' transposes; these helpers are the only
// readers of the flag besides the axis switch.

static int frames_image_w(const CarverFrames& f) { return f.transposed ? f.h : f.w; }
static int frames_image_h(const CarverFrames& f) { return f.transposed ? f.w : f.h; }

// A plane of every frame in image orientation: cols x rows elements of esize bytes per frame, rows pitch bytes apart,
// frames rows * pitch bytes apart
struct Plane {
    const void* p;
    size_t pitch;
    int cols, rows;
};

// A plane of the frames (cols x f.h elements of esize bytes per frame, rows pitch bytes apart, frames f.h rows apart) in
// image orientation: the plane itself, or for transposed frames its transpose in the scratch plane (one launch).
static int frames_oriented(dctc_context* ctx, CarverFrames& f, const void* plane, size_t pitch, int cols, int esize, Plane& out)
{
    out = Plane{plane, pitch, cols, f.h};
    if (!f.transposed) return DCTC_OK;
    if (!f.scratch) CK(ctx, cudaMalloc(&f.scratch, sizeof(float) * (size_t) f.w0 * f.h * f.n));   // cols <= w0, esize <= 4
    const size_t spitch = (size_t) esize * f.h;
    CK(ctx, dctc_launch_transpose(plane, pitch, pitch * f.h, f.scratch, spitch, spitch * cols, cols, f.h, f.n, esize, ctx->stream));
    ctx->launches++;
    out = Plane{f.scratch, spitch, f.h, cols};
    return DCTC_OK;
}

// Images (w * ch bytes per row), operator energy maps (w floats per row, frames_op_energy with op), visibility maps (vs_w
// ints per row) and bias planes (w floats per row) of all frames, in image orientation, to the host
static int frames_download(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, uint8_t* img, float* en, int* vs,
                           float* bias = nullptr)
{
    CK(ctx, cudaSetDevice(ctx->device));
    const float* en_src = f.en;
    if (en) {
        const int rc = frames_op_energy(ctx, f, op, &en_src);
        if (rc) return rc;
    }
    struct { void* dst; const void* src; size_t pitch; int cols, esize; } planes[4] = {
        {img, f.img, f.pitch, f.w, f.ch}, {en, en_src, sizeof(float) * f.en_pitch, f.w, 4}, {vs, f.vs, sizeof(int) * f.vs_w, f.vs_w, 4},
        {bias, f.bias, sizeof(float) * f.en_pitch, f.w, 4}};
    for (const auto& q : planes) {
        if (!q.dst) continue;
        Plane p;
        const int rc = frames_oriented(ctx, f, q.src, q.pitch, q.cols, q.esize, p);
        if (rc) return rc;
        const size_t rb = (size_t) p.cols * q.esize;   // frames are p.rows rows apart
        CK(ctx, cudaMemcpy2DAsync(q.dst, rb, p.p, p.pitch, rb, (size_t) p.rows * f.n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

// ---- the axis switch: the first height operation since a load ------------------------------------------------------------
// liblqr changes the height by transposing the carver (lqr_carver_resize), and so does a carver session: t becomes the
// transposes of f's frames (one launch), with the full energy maps of the transposed images (one K1 launch with the
// session's operator, not a transpose of f's maps: the operator's window is not symmetric) and, with vmaps, fresh visibility
// maps.  The width seam loop then runs on t unchanged.  f may be carved or enlarged (dctc_carver_resize switches the
// axis on the frame its width passes left).  t is allocated when it has no frames of f's transposed size yet (the
// session keeps it).  Biased frames: the bias planes are transposed too (one more launch) and t's seam energy uses ext = t.w0,
// the image height (one bias-add launch after the K1).
static int frames_transpose(dctc_context* ctx, const CarverFrames& f, CarverFrames& t, const DctcK1Op& op, bool vmaps)
{
    if (!t.img || t.w0 != f.h || t.h != f.w) {
        frames_free(t);
        frames_init(t, f.n, f.h, f.w, f.ch);
        t.transposed = true;
        const int rc = frames_alloc(ctx, t);
        if (rc) return rc;
    }
    t.w = t.w0;
    CK(ctx, dctc_launch_transpose(f.img, f.pitch, f.img_fs, t.img, t.pitch, t.img_fs, f.w, f.h, f.n, f.ch, ctx->stream));
    ctx->launches++;
    int rc = frames_bias_like(ctx, f, t);
    if (rc) return rc;
    if (f.bias) {
        const size_t fp = sizeof(float) * f.en_pitch, tp = sizeof(float) * t.en_pitch;
        CK(ctx, dctc_launch_transpose(f.bias, fp, fp * f.h, t.bias, tp, tp * t.h, f.w, f.h, f.n, sizeof(float), ctx->stream));
        ctx->launches++;
    }
    rc = frames_full_energy(ctx, t, op);
    if (rc == DCTC_OK && vmaps) rc = frames_vmaps(ctx, t);
    return rc;
}

// Launch plan of the seam DP for frames of wcur x h (energy planes at en, row pitch en_pitch floats, n_frames of them
// en_pitch * h floats apart) with the step rule Step: strip width, CTA size, energy staging and the tensor map.
template <typename Step>
using dp_fn = void (*)(const float*, size_t, int, int, float*, size_t, int*, int*, int*, int, const CUtensorMap, int*, size_t, size_t, size_t,
                       typename Step::Arg);
template <typename Step>
struct DpPlan {
    dp_fn<Step> dp = nullptr;
    int wpc = 0, nst = 0;
    size_t smem = 0;
    CUtensorMap tmap;
};

template <typename Step>
static cudaError_t dp_plan(int wcur, int h, const float* en, size_t en_pitch, int n_frames, DpPlan<Step>& p)
{
    // strip geometry: 128*P columns per warp, 128*P - 2*DP_R published; the strips are spread over a cluster of DP_CL CTAs
    const int cap = DP_CL * DP_MAXW;
    const int P = wcur <= cap * (128 - 2 * DP_R) ? 1 : wcur <= cap * (256 - 2 * DP_R) ? 2 : 4;
    const int wout = 128 * P - 2 * DP_R;
    const int strips = (wcur + wout - 1) / wout;
    const int wpc = (strips + DP_CL - 1) / DP_CL;
    // energies staged by tensor copies when at least two stages (DP_SR rows each) per warp fit into shared memory
    // (the kernel also has ~38 KB of static shared memory: back-track windows, reduction scratch, mbarriers)
    const size_t xrow_smem = sizeof(float) * 2 * (size_t) wpc * wout;
    const size_t row_smem = sizeof(float) * ((size_t) wpc * 128 * P);      // one staged row of every warp
    const size_t budget = 180 * 1024 - xrow_smem;
    int nst, sr;
    if (2 * 32 * row_smem <= budget) { sr = 32; nst = 2; }                 // whole 32-row blocks, two in flight
    else {
        sr = 16;
        for (nst = DP_NST_MAX; nst >= 2 && (size_t) nst * 16 * row_smem > budget; nst--) {}
        if (nst < 2) { sr = 0; nst = 0; }
    }
    p.wpc = wpc;
    p.nst = nst;
    p.smem = xrow_smem + sizeof(float) * ((size_t) nst * sr * wpc * 128 * P);
    // the (P, SR) pairs the lines above select for widths 1 .. DP_MAX_W, for each of the three step rules:
    //   1-2560: (1, 32)   2561-4096: (1, 16)   4097-7680: (2, 16)   7681-12288: (2, 0)   12289-DP_MAX_W: (4, 0)
    static const struct { int P, sr; dp_fn<Step> fn; } variants[] = {
        {1, 32, dctc_seam_dp_kernel<1, 32, Step>}, {1, 16, dctc_seam_dp_kernel<1, 16, Step>}, {2, 16, dctc_seam_dp_kernel<2, 16, Step>},
        {2, 0, dctc_seam_dp_kernel<2, 0, Step>}, {4, 0, dctc_seam_dp_kernel<4, 0, Step>}};
    p.dp = nullptr;
    for (const auto& v : variants)
        if (v.P == P && v.sr == sr) p.dp = v.fn;
    if (!p.dp) return cudaErrorInvalidConfiguration;   // a pair without a kernel: the table and the plan disagree
    // tensor map of the energy planes for the staged variants (strips of up to 256 columns: the TMA box limit); frames
    // are its third dimension, so that a box never reaches into the next frame's rows
    memset(&p.tmap, 0, sizeof(p.tmap));
    if (sr > 0) {
        const DctcTensorMapEncodeFn encode = dctc_tensor_map_encoder();
        if (!encode) return cudaErrorNotSupported;
        const cuuint64_t gdim[3] = {(cuuint64_t) en_pitch, (cuuint64_t) h, (cuuint64_t) n_frames};
        const cuuint64_t gstr[2] = {(cuuint64_t) en_pitch * sizeof(float), (cuuint64_t) en_pitch * h * sizeof(float)};
        const cuuint32_t box[3] = {(cuuint32_t) (128 * P), (cuuint32_t) sr, 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        if (encode(&p.tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*) en, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    // always opt in: the kernel's static shared memory (back-track windows) plus the dynamic part can exceed 48 KB
    return cudaFuncSetAttribute(p.dp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (p.smem > 1024 ? p.smem : 1024));
}

// Back-track plan for frames of h rows and a step rule whose steps reach D columns, dx at most.  The parallel back-track
// (jump + trace kernels) needs the jump plane and a cone of jump entries in shared memory that grows with the square of
// the number of row blocks; very tall frames keep the serial walk of the DP kernel, and so do frames whose cumulative
// rows are narrower than the trace window (only possible for D > 1: the rows are at least DP_WIN floats).
struct BtPlan {
    int nb;             // row blocks of BtGeom<D>::jb rows
    size_t cone_smem;   // trace kernel's dynamic shared memory
    size_t j_pitch;     // bytes per row of the jump plane (nb rows per frame)
    bool par;           // parallel back-track
};

template <int D>
static BtPlan bt_plan(int h, size_t m_pitch, int dx)
{
    using G = BtGeom<D>;
    BtPlan b;
    b.nb = (h - 1 + G::jb - 1) / G::jb;
    const size_t r8 = (size_t) ((G::jb * dx + 7) & ~7), j = b.nb > 0 ? (size_t) (b.nb - 1) : 0;
    b.cone_smem = r8 * j * (j > 0 ? j - 1 : 0) + 48 * j + 16;   // rows j < nb-1: 16 ((R8 / 8) j + 3) bytes each
    b.j_pitch = (m_pitch + 15) & ~(size_t) 15;    // jump rows start 16-byte aligned (staged in 16-byte chunks)
    b.par = b.nb > 0 && b.cone_smem <= (size_t) G::cone_max && m_pitch >= (size_t) G::win;
    return b;
}

// Planes of the seam loop, allocated by its first call: cumulative planes, jump planes (parallel back-track only) and a
// seam log of log_fs ints per frame.
static int frames_loop_buffers(dctc_context* ctx, CarverFrames& f, const BtPlan& bt, size_t log_fs)
{
    const size_t n = (size_t) f.n;
    if (!f.m) {
        CK(ctx, cudaMalloc((void**) &f.m, sizeof(float) * f.m_pitch * f.h * n));
        CK(ctx, cudaMemsetAsync(f.m, 0, sizeof(float) * f.m_pitch * f.h * n, ctx->stream));
    }
    if (bt.par && (!f.dir || f.dir_fs < (size_t) bt.nb * bt.j_pitch)) {   // (delta_x > 1 has more, shorter blocks)
        cudaFree(f.dir);
        f.dir = nullptr;
        f.dir_fs = (size_t) bt.nb * bt.j_pitch;
        CK(ctx, cudaMalloc((void**) &f.dir, f.dir_fs * n));
    }
    if (f.seam_log_cap < log_fs * n) {
        cudaFree(f.seam_log);
        f.seam_log = nullptr; f.seam_log_cap = 0;
        CK(ctx, cudaMalloc((void**) &f.seam_log, sizeof(int) * log_fs * n));
        f.seam_log_cap = log_fs * n;
    }
    return DCTC_OK;
}

// What the caller of a seam operation brings besides the session: whether its seam loops record the visibility maps, the
// rigidity (dctc_carver_set_rigidity, dctc_carver_batch_set_rigidity), the seam step width (dctc_carver_set_delta_x,
// dctc_carver_batch_set_delta_x) and the context's incremental cumulative map (dctc_carver_set_incremental), which only
// the single session has.
struct SeamCall {
    bool vmaps = false;
    float rigidity = 0.0f;
    int delta_x = 1;
    bool incremental = false;
    bool* m_valid = nullptr;   // &ctx->c_m_valid (single session), null for a batch
};

// The device seam loop of every frame: removes n_seams seams from the images and energy planes (f.w shrinks by n_seams).
// Per seam: build_mmap + build_vpath (seam DP, then jump + trace or the DP's serial walk), update_vsmap when c.vmaps (maps
// as frames_vmaps leaves them), the carve, and update_emap (band K1 around each removed seam).  The caller has checked the
// width.
// c.incremental (one frame only, its flag buffer is ctx->c_band): *c.m_valid says whether f.m holds the map of the image
// before the last removal, compacted over that seam.  The walk then replaces DP + jump + trace, the DP only runs when the
// walk gave up, and the carve also compacts f.m.  A loop that does not keep the map up to date clears *c.m_valid.
// Step: the step rule (DpStep1 or DpSteps, chosen by seam_loop below) of every seam-search kernel of the loop, arg its
// kernel argument.  The incremental walk is DpStep1 only: with DpSteps the DP rebuilds the map every seam.
template <typename Step>
static int seam_loop_rule(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, int n_seams, int* seams_out, const SeamCall& c,
                          const typename Step::Arg arg)
{
    using G = BtGeom<Step::D>;
    const int n = f.n, h = f.h, dx = Step{arg}.dx;
    const size_t log_fs = (size_t) n_seams * h, en_fs = f.en_pitch * h, m_fs = f.m_pitch * h;
    const BtPlan bt = bt_plan<Step::D>(h, f.m_pitch, dx);
    int rc = frames_loop_buffers(ctx, f, bt, log_fs);
    if (rc) return rc;
    DpPlan<Step> plan;
    CK(ctx, dp_plan(f.w, h, f.en, f.en_pitch, n, plan));
    if (bt.par)   // the window's static shared memory plus the cone can exceed the 48 KB default
        CK(ctx, cudaFuncSetAttribute(dctc_seam_trace_kernel<Step>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bt.cone_smem));
    int* const xlast = bt.par ? f.xlast : nullptr;
    // incremental update (update_mmap): one warp; needs the band table of h rows twice in shared memory
    const size_t incr_smem = sizeof(float) * (INCR_D * 2 * INCR_SW + 2 * (INCR_CAP + 4)) + sizeof(int) * (INCR_D + 2 * (size_t) h);
    const bool incr = Step::D == 1 && c.incremental && n == 1 && incr_smem <= 160 * 1024;
    if constexpr (Step::D == 1) {
        if (incr) {   // dynamic + static shared memory can exceed the 48 KB default
            CK(ctx, cudaFuncSetAttribute(dctc_seam_incr_kernel<Step>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) incr_smem));
            if (!ctx->c_band) {
                CK(ctx, cudaMalloc((void**) &ctx->c_band, sizeof(int) * 4));
                CK(ctx, cudaMemsetAsync(ctx->c_band, 0, sizeof(int) * 4, ctx->stream));
            }
        }
    }
    for (int s = 0; s < n_seams; s++) {
        const int w_old = f.w;
        int* log_s = f.seam_log + (size_t) s * h;
        const bool walk = incr && *c.m_valid;
        if constexpr (Step::D == 1) {
            if (walk) {
                // update_mmap + build_vpath: walk the changed cells only; the DP below rebuilds the map only if the walk gave up
                dctc_seam_incr_kernel<Step><<<1, 32, incr_smem, ctx->stream>>>(f.en, f.en_pitch, w_old, h, f.m, f.m_pitch, op.blocksize / 2,
                                                                               f.seam, log_s, ctx->c_band, arg);
                CK(ctx, cudaGetLastError());
                ctx->launches++;
            }
        }
        // build_mmap, one cluster per frame, then build_vpath: jump maps of all row blocks in parallel, one trace CTA per
        // block and frame (programmatic dependent launches: each kernel of the loop is scheduled while its predecessor
        // drains and blocks in DCTC_PDL_PROLOGUE until that one's results are visible)
        CK(ctx, dctc_launch_pdl(plan.dp, dim3(DP_CL, n), dim3(plan.wpc * 32), plan.smem, ctx->stream, !walk, f.en, f.en_pitch, w_old, h,
                                f.m, f.m_pitch, f.seam, log_s, walk ? ctx->c_band : (int*) nullptr, plan.nst, plan.tmap,
                                walk ? (int*) nullptr : xlast, en_fs, m_fs, log_fs, arg));
        if (bt.par && !walk) {   // strips of 16 jc published columns
            const int js = (w_old + 16 * G::jc - 1) / (16 * G::jc);
            CK(ctx, dctc_launch_pdl(dctc_seam_jump_kernel<Step>, dim3((js + 3) / 4, bt.nb, n), dim3(128), 0, ctx->stream, true, f.m,
                                    f.m_pitch, w_old, h, f.dir, bt.j_pitch, js, m_fs, f.dir_fs, arg));
            CK(ctx, dctc_launch_pdl(dctc_seam_trace_kernel<Step>, dim3(bt.nb, n), dim3(TR_THREADS), bt.cone_smem, ctx->stream, true, f.m,
                                    f.m_pitch, w_old, h, f.dir, bt.j_pitch, f.xlast, f.seam, log_s, m_fs, f.dir_fs, log_fs, arg));
            ctx->launches += 2;
        }
#ifdef DCTC_SYNC_DEBUG
        { cudaError_t e_ = cudaStreamSynchronize(ctx->stream); if (e_ != cudaSuccess) { printf("seam %d: dp kernel failed: %s (w %d)\n", s, cudaGetErrorString(e_), w_old); return dctc_fail_cuda(ctx, e_); } }
#endif
        if (c.vmaps) {   // update_vsmap
            CK(ctx, dctc_launch_pdl(dctc_vs_update_kernel, dim3(h, n), dim3(256), 0, ctx->stream, true, f.raw, f.vs, f.w0, f.seam, w_old,
                                    ++f.depth));
            ctx->launches++;
        }
        // carve: compact image and energy rows (and the cumulative rows of the incremental map) over the seam
        CK(ctx, dctc_launch_pdl(f.bias ? dctc_carve_rows_kernel<256, 4, true> : dctc_carve_rows_kernel<256, 4, false>, dim3(h, n), dim3(256),
                                0, ctx->stream, true, f.img, f.pitch, f.ch, f.en, f.en_pitch, f.seam, w_old, incr ? f.m : (float*) nullptr,
                                f.m_pitch, f.img_fs, en_fs, m_fs, f.bias));
        ctx->launches += 2;
        f.w = w_old - 1;
        if (c.m_valid) *c.m_valid = incr;   // the plane now holds the map of the image before this removal, moved with the pixels
#ifdef DCTC_SYNC_DEBUG
        { cudaError_t e_ = cudaStreamSynchronize(ctx->stream); if (e_ != cudaSuccess) { printf("seam %d: carve kernel failed: %s (w %d)\n", s, cudaGetErrorString(e_), w_old); return dctc_fail_cuda(ctx, e_); } }
#endif
        // update_emap: K1 in band mode around every frame's removed seam
        DctcK1Args a = frames_k1_args(f, op, f.seam);
        a.pdl = 1;
        const DctcK1Bias bias{f.bias, (float) f.w0};   // biased frames: the band store writes the seam energy
        rc = dctc_run_k1(ctx, op, a, n, ctx->stream, f.bias ? &bias : nullptr, dx);
        if (rc) return rc;
#ifdef DCTC_SYNC_DEBUG
        { cudaError_t e_ = cudaStreamSynchronize(ctx->stream); if (e_ != cudaSuccess) { printf("seam %d: band kernel failed: %s (w %d)\n", s, cudaGetErrorString(e_), w_old); return dctc_fail_cuda(ctx, e_); } }
#endif
    }
    if (seams_out)
        CK(ctx, cudaMemcpyAsync(seams_out, f.seam_log, sizeof(int) * log_fs * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

// c.rigidity: the seams are f.h rows long (the image width at the axis switch for height operations), so the step rule
// gets pen = fl(rigidity / f.h) (DpStep1<true>; pen == 0 runs the kernels of rigidity 0, DpStep1<false>) or, for
// c.delta_x > 1, the table of pen[d] (DpSteps).  The band K1 covers a seam drift of delta_x per row.
static int seam_loop(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, int n_seams, int* seams_out, const SeamCall& c)
{
    const int h = f.h, dx = c.delta_x;
    if (dx > 1) {
        DpSteps steps;
        steps.dx = dx;
        for (int d = 0; d <= DCTC_MAX_DELTA_X; d++)   // the host carver's rigidity_map_of, +inf beyond the step bound
            steps.pen[d] = d > dx ? INFINITY : (c.rigidity * ((float) d * sqrtf((float) d))) / (float) h;
        return seam_loop_rule<DpSteps>(ctx, f, op, n_seams, seams_out, c, steps);
    }
    const float pen = c.rigidity / (float) h;
    return pen != 0.0f ? seam_loop_rule<DpStep1<true>>(ctx, f, op, n_seams, seams_out, c, pen)
                       : seam_loop_rule<DpStep1<false>>(ctx, f, op, n_seams, seams_out, c, pen);
}

// Enlarge core (lqr_carver_resize to a larger width, seams_number > 0, src/render.c:357-363): start_img holds a copy of
// f's images (session_copy_start), the seam loop removes n_seams seams and records their order in the visibility maps (as
// frames_vmaps leaves them), one inflate launch doubles every pixel of those seams in all frames into wide's images
// (w0 + n_seams wide) and one K1 launch computes their full energy maps.  f is left carved by n_seams.
// Biased frames: a copy of the start bias planes is inflated in the same launch (copy rule) into wide's bias planes, and
// one bias-add launch gives wide's seam energy with ext = wide.w0.
static int frames_enlarge(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, int n_seams, int* seams_out, SeamCall c,
                          const uint8_t* start_img, CarverFrames& wide)
{
    c.vmaps = true;
    const size_t en_fs = f.en_pitch * f.h;
    float* start_bias = nullptr;
    int rc = frames_bias_like(ctx, f, wide);
    if (rc == DCTC_OK && f.bias) {
        cudaError_t e = cudaMalloc((void**) &start_bias, sizeof(float) * en_fs * f.n);
        if (e == cudaSuccess) e = cudaMemcpyAsync(start_bias, f.bias, sizeof(float) * en_fs * f.n, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e != cudaSuccess) rc = dctc_fail_cuda(ctx, e);
    }
    if (rc == DCTC_OK) rc = seam_loop(ctx, f, op, n_seams, seams_out, c);
    if (rc == DCTC_OK) {
        auto inflate = f.bias ? dctc_inflate_rows_kernel<true> : dctc_inflate_rows_kernel<false>;
        inflate<<<dim3(f.h, f.n), 256, 0, ctx->stream>>>(start_img, f.pitch, f.ch, f.w0, f.vs, n_seams, wide.img, wide.pitch, f.img_fs,
                                                         (size_t) f.w0 * f.h, wide.img_fs, start_bias, f.en_pitch, en_fs, wide.bias,
                                                         wide.en_pitch, wide.en_pitch * wide.h);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = dctc_fail_cuda(ctx, e);
        ctx->launches++;
    }
    if (rc == DCTC_OK) rc = frames_full_energy(ctx, wide, op);
    const cudaError_t es = cudaStreamSynchronize(ctx->stream);
    cudaFree(start_bias);
    if (rc) return rc;
    if (es != cudaSuccess) return dctc_fail_cuda(ctx, es);
    return DCTC_OK;
}

// dctc_carver_set_bias / dctc_carver_batch_set_bias on frames as loaded: the caller's planes (w x h floats per frame, rows
// pitch bytes and frames fs bytes apart, any memory cudaMemcpyDefault reaches) become the bias planes and the energy
// planes are rebuilt (frames_full_energy); null clears the bias (the planes are rebuilt when there was one).
static int frames_set_bias(dctc_context* ctx, CarverFrames& f, const DctcK1Op& op, const float* bias, size_t fs, size_t pitch)
{
    if (!bias) {
        if (!f.bias) return DCTC_OK;
        cudaFree(f.bias);
        f.bias = nullptr;
    } else {
        if (!f.bias) CK(ctx, cudaMalloc((void**) &f.bias, sizeof(float) * f.en_pitch * f.h * f.n));
        for (int i = 0; i < f.n; i++)
            CK(ctx, cudaMemcpy2DAsync(f.bias + (size_t) i * f.en_pitch * f.h, sizeof(float) * f.en_pitch, (const char*) bias + i * fs, pitch,
                                      sizeof(float) * f.w, f.h, cudaMemcpyDefault, ctx->stream));
    }
    const int rc = frames_full_energy(ctx, f, op);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

// ---- the session: one type for the context's single session and for batch sessions ------------------------------------
// A batch session (dctc_carver_batch_*) is a dctc_carver_batch of n frames, the context's single session (dctc_carver_*,
// ctx->carver) one of one frame that each dctc_carver_load replaces.  The state machine below serves both.  The ways the
// two APIs differ are fields set at create (dump_vmaps, ends_at_enlarge) or what a call passes (SeamCall); the single
// session's wrappers also take the operator from the context at every call and release the session where a batch is
// left unloaded.

// The axis the seam operations work along since the load: the first one fixes it, a call for the other axis returns
// DCTC_ERR_STATE until the next load.  RESIZED: a combined resize ran since the load, which fixes both axes.  LEVELS: a
// levels build ran since the load (session_levels); it ends the seam operations until the next load, and the renders
// read cur's maps and the start frames' copy (cur->transposed: height levels).
enum { DCTC_AXIS_NONE = 0, DCTC_AXIS_WIDTH = 1, DCTC_AXIS_HEIGHT = 2, DCTC_AXIS_RESIZED = 3, DCTC_AXIS_LEVELS = 4 };

// Frame sets are allocated by their first use, reallocated when their size differs and freed with the session: the
// loaded frames f next to their transposes t, and the start frames' copy next to the enlarged sets.
struct dctc_carver_batch {
    dctc_context* ctx = nullptr;        // device, stream and launch counter
    DctcK1Op op;                        // the context's operator at load, with the carver's kernel rule (carver_op)
    bool dump_vmaps = false;            // every seam loop records the visibility maps (a batch's create flag; the maps
                                        // are reset at the load and at the axis switch).  The single session asks per call.
    bool ends_at_enlarge = false;       // an enlarge or a combined resize is the last seam operation until the next load,
                                        // n_seams = 0 included (a batch); otherwise the session continues on the enlarged frames
    int axis = DCTC_AXIS_NONE;
    CarverFrames* cur = nullptr;        // the frames the getters read and the next seam operation carves; null: not loaded
    CarverFrames* maps = nullptr;       // the set whose visibility maps _vmap and _paint_seams read: the one the last
                                        // map-recording seam loop ran on (null: none since the load or the axis switch)
    CarverFrames f;                     // the loaded frames
    CarverFrames t;                     // their transposes (height operations)
    CarverFrames wide, wide2;           // enlarged frames: an enlarge writes into the one that is not cur
    uint8_t* start_img = nullptr;       // an enlarge's or a levels build's copy of its start images
    size_t start_bytes = 0;
    uint8_t* lv_scratch = nullptr;      // height levels in the transposed orientation on their way out (session_render)
    size_t lv_scratch_bytes = 0;
    float rigidity = 0.0f;              // dctc_carver_batch_set_rigidity (the single session takes the context's instead)
    int delta_x = 1;                    // dctc_carver_batch_set_delta_x (likewise)
};

namespace {

void session_destroy(dctc_carver_batch* b)
{
    frames_free(b->f);
    frames_free(b->t);
    frames_free(b->wide);
    frames_free(b->wide2);
    cudaFree(b->start_img);
    cudaFree(b->lv_scratch);
    delete b;
}

int session_create(dctc_context* ctx, int n_frames, int w, int h, int channels, bool dump_vmaps, bool ends_at_enlarge,
                   dctc_carver_batch** out)
{
    dctc_carver_batch* b = new (std::nothrow) dctc_carver_batch;
    if (!b) return DCTC_ERR_NOMEM;
    b->ctx = ctx;
    b->dump_vmaps = dump_vmaps;
    b->ends_at_enlarge = ends_at_enlarge;
    frames_init(b->f, n_frames, w, h, channels);
    int rc = frames_alloc(ctx, b->f);
    if (rc == DCTC_OK) {
        const cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = dctc_fail_cuda(ctx, e);
    }
    if (rc) {
        session_destroy(b);
        return rc;
    }
    *out = b;
    return DCTC_OK;
}

// The size the getters report: the current frames', or while unloaded the loaded frames'
const CarverFrames& session_frames(const dctc_carver_batch* b) { return b->cur ? *b->cur : b->f; }

// Host frames (frame_stride bytes apart, rows pitch bytes apart) into f, which becomes cur: no bias, the axis free, maps
// reset with dump_vmaps, the full energy maps with the context's operator.  A failure leaves the session unloaded.
int session_load(dctc_carver_batch* b, const uint8_t* imgs, size_t frame_stride, size_t pitch)
{
    dctc_context* ctx = b->ctx;
    CarverFrames& f = b->f;
    b->cur = b->maps = nullptr;
    b->axis = DCTC_AXIS_NONE;
    b->op = carver_op(ctx->op);
    f.w = f.w0;
    cudaFree(f.bias);
    f.bias = nullptr;
    for (int i = 0; i < f.n; i++)
        CK(ctx, cudaMemcpy2DAsync(f.img + (size_t) i * f.img_fs, f.pitch, imgs + (size_t) i * frame_stride, pitch, (size_t) f.w0 * f.ch,
                                  f.h, cudaMemcpyDefault, ctx->stream));
    int rc = b->dump_vmaps ? frames_vmaps(ctx, f) : DCTC_OK;
    if (rc == DCTC_OK) rc = frames_full_energy(ctx, f, b->op);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    b->cur = &f;
    b->maps = b->dump_vmaps ? &f : nullptr;
    return DCTC_OK;
}

// frames_set_bias on the loaded frames, before any seam operation.  A failure leaves the session unloaded.
int session_set_bias(dctc_carver_batch* b, const float* bias, size_t frame_stride, size_t pitch)
{
    if (!b->cur || b->axis != DCTC_AXIS_NONE) return DCTC_ERR_STATE;   // loaded, no seam operation since
    CarverFrames& f = b->f;
    if (bias && (pitch < sizeof(float) * f.w0 || (f.n > 1 && frame_stride < pitch * f.h))) return DCTC_ERR_INVALID;
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    b->cur = nullptr;
    const int rc = frames_set_bias(ctx, f, b->op, bias, frame_stride, pitch);
    if (rc) return rc;
    b->cur = &f;
    return DCTC_OK;
}

// The axis switch: cur becomes its transposes in t (frames_transpose), with fresh maps when vmaps.  A failure leaves the
// session unloaded.
int session_transpose(dctc_carver_batch* b, bool vmaps, const SeamCall& c)
{
    CarverFrames* src = b->cur;
    b->cur = nullptr;
    if (c.m_valid) *c.m_valid = false;
    const int rc = frames_transpose(b->ctx, *src, b->t, b->op, vmaps);
    if (rc) return rc;
    b->cur = &b->t;
    b->maps = vmaps ? &b->t : nullptr;
    return DCTC_OK;
}

// A resize: the seam loop on cur.  Maps a call asks for start at its first recording loop on these frames (the caller
// checked that no seam was removed from them before).
int session_carve(dctc_carver_batch* b, int n_seams, int* seams_out, const SeamCall& c)
{
    CarverFrames& f = *b->cur;
    if (c.vmaps && b->maps != &f) {
        const int rc = frames_fresh_vmaps(b->ctx, f);
        if (rc) return rc;
        b->maps = &f;
    }
    return seam_loop(b->ctx, f, b->op, n_seams, seams_out, c);
}

// The start frames' copy of an enlarge or a levels build: f's images into start_img (reallocated when its size differs,
// kept until the destroy), one device copy on the stream
int session_copy_start(dctc_carver_batch* b, const CarverFrames& f)
{
    dctc_context* ctx = b->ctx;
    if (b->start_bytes != f.img_fs * f.n) {
        cudaFree(b->start_img);
        b->start_img = nullptr; b->start_bytes = 0;
        CK(ctx, cudaMalloc((void**) &b->start_img, f.img_fs * f.n));
        b->start_bytes = f.img_fs * f.n;
    }
    CK(ctx, cudaMemcpyAsync(b->start_img, f.img, f.img_fs * f.n, cudaMemcpyDeviceToDevice, ctx->stream));
    return DCTC_OK;
}

// An enlarge: frames_enlarge from cur (as loaded or enlarged) into the enlarged set that is not cur, which becomes cur;
// the maps stay those of the start frames.  cur is carved in place, so a failure leaves the session unloaded.
int session_enlarge(dctc_carver_batch* b, int n_seams, int* seams_out, const SeamCall& c)
{
    dctc_context* ctx = b->ctx;
    CarverFrames& f = *b->cur;
    CarverFrames& wide = b->cur == &b->wide ? b->wide2 : b->wide;
    b->cur = nullptr;
    const int w1 = f.w0 + n_seams;
    const int rs = session_copy_start(b, f);
    if (rs) return rs;
    if (wide.w0 != w1 || wide.h != f.h) {
        frames_free(wide);
        frames_init(wide, f.n, w1, f.h, f.ch);
        const int rc = frames_alloc(ctx, wide);
        if (rc) {
            frames_free(wide);
            return rc;
        }
    }
    wide.w = wide.w0;   // (a set an earlier pass carved)
    wide.transposed = f.transposed;
    int rc = frames_fresh_vmaps(ctx, f);
    if (rc == DCTC_OK) rc = frames_enlarge(ctx, f, b->op, n_seams, seams_out, c, b->start_img, wide);
    if (rc) return rc;
    b->cur = &wide;
    b->maps = &f;
    if (c.m_valid) {   // as after a load: no incremental map, its rebuild count from zero
        *c.m_valid = false;
        cudaFree(ctx->c_band);
        ctx->c_band = nullptr;
    }
    return DCTC_OK;
}

// dctc_carver_resize_width / _height, dctc_carver_enlarge_width / _height and the batch's: the checks (the axis fixed
// since the load, n_seams >= the image's extent along the axis, an extent wider than the seam DP covers), then the first
// height operation since the load switches the axis.
int session_seams(dctc_carver_batch* b, int axis, bool enlarge, int n_seams, int* seams_out, const SeamCall& c)
{
    const bool enlarged = b->cur == &b->wide || b->cur == &b->wide2;
    if (!b->cur || b->axis == DCTC_AXIS_LEVELS || (b->ends_at_enlarge && (enlarged || b->axis == DCTC_AXIS_RESIZED)))
        return DCTC_ERR_STATE;
    if (n_seams == 0) return DCTC_OK;
    const CarverFrames& f = *b->cur;
    if (enlarge && f.w != f.w0) return DCTC_ERR_STATE;   // an enlarge starts from frames as loaded (or enlarged)
    if (b->axis != DCTC_AXIS_NONE && b->axis != axis) return DCTC_ERR_STATE;
    const int extent = axis == DCTC_AXIS_WIDTH ? frames_image_w(f) : frames_image_h(f);
    if (n_seams >= extent) return DCTC_ERR_STATE;
    if (extent > DP_MAX_W) return DCTC_ERR_UNSUPPORTED;   // wider than the cluster's strips: use the host seam loop
    if (!enlarge && c.vmaps && b->maps != &f && f.w != f.w0) return DCTC_ERR_STATE;   // maps: before the first seam
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (axis == DCTC_AXIS_HEIGHT && b->axis == DCTC_AXIS_NONE) {
        const int rc = session_transpose(b, c.vmaps, c);
        if (rc) return rc;
    }
    b->axis = axis;
    return enlarge ? session_enlarge(b, n_seams, seams_out, c) : session_carve(b, n_seams, seams_out, c);
}

// dctc_carver_resize / dctc_carver_batch_resize: the plan (checked against the seam DP's reach before any work) as its
// per-axis calls run it, maps recorded whenever vmaps_out is given and each pass's map read back before the next pass
// reuses its set.  A failure leaves the session unloaded.
int session_resize(dctc_carver_batch* b, int new_w, int new_h, int* seams_out, int* vmaps_out, const SeamCall& c)
{
    if (!b->cur || b->axis != DCTC_AXIS_NONE) return DCTC_ERR_STATE;
    DctcResizePass plan[DCTC_RESIZE_MAX_PASSES];
    const int n = dctc_resize_passes(b->f.w, b->f.h, new_w, new_h, plan, DCTC_RESIZE_MAX_PASSES);
    if (n <= 0) return n;
    for (int i = 0; i < n; i++)
        if ((plan[i].axis == DCTC_RESIZE_WIDTH ? plan[i].w : plan[i].h) > DP_MAX_W) return DCTC_ERR_UNSUPPORTED;
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    SeamCall pc = c;
    pc.vmaps = vmaps_out != nullptr;
    const size_t nf = (size_t) b->f.n;
    for (int i = 0; i < n; i++) {
        const DctcResizePass& p = plan[i];
        int* seams = seams_out ? seams_out + nf * p.seams_offset : nullptr;
        int rc = DCTC_OK;
        if (p.axis == DCTC_RESIZE_HEIGHT && !b->cur->transposed) rc = session_transpose(b, false, c);
        if (rc == DCTC_OK) rc = p.enlarge ? session_enlarge(b, p.n_seams, seams, pc) : session_carve(b, p.n_seams, seams, pc);
        if (rc == DCTC_OK && vmaps_out) rc = frames_download(ctx, *b->maps, b->op, nullptr, nullptr, vmaps_out + nf * p.vmap_offset);
        if (rc) {
            b->cur = nullptr;
            return rc;
        }
    }
    b->axis = DCTC_AXIS_RESIZED;
    return DCTC_OK;
}

// dctc_carver_levels_width / _height and the batch's (lqr_carver_resize to the extreme size of the interactive dialog):
// on frames as loaded, the start frames' copy (session_copy_start) and what resize_width / resize_height with maps runs
// (the axis switch for heights, fresh maps, the seam loop to depth).  cur is left carved by depth with its maps recorded,
// and the axis becomes LEVELS.  A failure leaves the session unloaded.
int session_levels(dctc_carver_batch* b, int axis, int depth, int* seams_out, const SeamCall& c)
{
    if (!b->cur || b->axis != DCTC_AXIS_NONE) return DCTC_ERR_STATE;   // loaded, no seam operation since
    const int extent = axis == DCTC_AXIS_WIDTH ? frames_image_w(*b->cur) : frames_image_h(*b->cur);
    if (depth >= extent) return DCTC_ERR_STATE;
    if (extent > DP_MAX_W) return DCTC_ERR_UNSUPPORTED;
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    SeamCall lc = c;
    lc.vmaps = true;
    if (axis == DCTC_AXIS_HEIGHT) {
        const int rc = session_transpose(b, true, lc);
        if (rc) return rc;
    }
    b->axis = DCTC_AXIS_LEVELS;
    CarverFrames& f = *b->cur;
    b->cur = nullptr;
    int rc = session_copy_start(b, f);
    if (rc == DCTC_OK && b->maps != &f) {
        rc = frames_fresh_vmaps(ctx, f);
        b->maps = &f;
    }
    if (rc == DCTC_OK && depth > 0) rc = seam_loop(ctx, f, b->op, depth, seams_out, lc);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    b->cur = &f;
    return DCTC_OK;
}

// dctc_carver_render_levels_dev / dctc_carver_batch_render_levels_dev: the levels of a build since the load into d_out
// (device memory), level-major in the order of extents, each n frames of rows packed in image orientation.  Extents up
// to the start extent e0 are shrinks (one gather launch per LV_MAX of them), wider ones enlarges (one inflate launch each,
// level e - e0: what an enlarge by e - e0 writes).  Height levels are built in the transposed orientation in lv_scratch
// and turned into image orientation by one transpose launch each.  The session does not change.
int session_render(dctc_carver_batch* b, int n_levels, const int* extents, uint8_t* d_out)
{
    if (!b->cur || b->axis != DCTC_AXIS_LEVELS) return DCTC_ERR_STATE;
    const CarverFrames& f = *b->cur;
    const int e0 = f.w0;
    for (int i = 0; i < n_levels; i++)
        if (extents[i] < e0 - f.depth || extents[i] > e0 + f.depth) return DCTC_ERR_STATE;
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t unit = (size_t) f.n * f.h * f.ch;   // bytes of a level per column of extent (rows f.h in f's orientation)
    size_t total = 0;
    for (int i = 0; i < n_levels; i++) total += unit * extents[i];
    uint8_t* dst = d_out;
    if (f.transposed) {
        if (b->lv_scratch_bytes < total) {
            cudaFree(b->lv_scratch);
            b->lv_scratch = nullptr; b->lv_scratch_bytes = 0;
            CK(ctx, cudaMalloc((void**) &b->lv_scratch, total));
            b->lv_scratch_bytes = total;
        }
        dst = b->lv_scratch;
    }
    const size_t vs_fs = (size_t) f.w0 * f.h;
    LevelTable lt;
    lt.n = 0;
    auto gather = [&]() {
        dctc_levels_gather_kernel<<<dim3(f.h, f.n), 256, 0, ctx->stream>>>(b->start_img, f.pitch, f.ch, f.w0, f.vs, f.img_fs, vs_fs, lt, dst);
        ctx->launches++;
        lt.n = 0;
        return cudaGetLastError();
    };
    size_t off = 0;
    for (int i = 0; i < n_levels; i++) {
        const int e = extents[i];
        const size_t row = (size_t) e * f.ch;
        if (e <= e0) {
            lt.k[lt.n] = e0 - e;
            lt.off[lt.n] = off;
            if (++lt.n == LV_MAX) CK(ctx, gather());
        } else {
            dctc_inflate_rows_kernel<false><<<dim3(f.h, f.n), 256, 0, ctx->stream>>>(b->start_img, f.pitch, f.ch, f.w0, f.vs, e - e0,
                                                                                    dst + off, row, f.img_fs, vs_fs, row * f.h, nullptr,
                                                                                    0, 0, nullptr, 0, 0);
            ctx->launches++;
            CK(ctx, cudaGetLastError());
        }
        off += unit * e;
    }
    if (lt.n) CK(ctx, gather());
    if (f.transposed) {
        off = 0;
        for (int i = 0; i < n_levels; i++) {
            const int e = extents[i];
            const size_t row = (size_t) e * f.ch, orow = (size_t) f.h * f.ch;
            CK(ctx, dctc_launch_transpose(dst + off, row, row * f.h, d_out + off, orow, orow * e, e, f.h, f.n, f.ch, ctx->stream));
            ctx->launches++;
            off += unit * e;
        }
    }
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

// session_render into a device buffer of the call's size, then to the host
int session_render_host(dctc_carver_batch* b, int n_levels, const int* extents, uint8_t* out)
{
    if (!b->cur || b->axis != DCTC_AXIS_LEVELS) return DCTC_ERR_STATE;
    const CarverFrames& f = *b->cur;
    size_t total = 0;
    for (int i = 0; i < n_levels; i++) total += (size_t) f.n * f.h * f.ch * (size_t) (extents[i] > 0 ? extents[i] : 0);
    dctc_context* ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    uint8_t* d = nullptr;
    CK(ctx, cudaMalloc((void**) &d, total));
    int rc = session_render(b, n_levels, extents, d);
    if (rc == DCTC_OK) {
        cudaError_t e = cudaMemcpyAsync(out, d, total, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = dctc_fail_cuda(ctx, e);
    }
    cudaFree(d);
    return rc;
}

// Images, operator energy maps or bias planes of the current frames
int session_download(dctc_carver_batch* b, uint8_t* img, float* en, float* bias)
{
    if (!b->cur || (bias && !b->cur->bias)) return DCTC_ERR_STATE;
    return frames_download(b->ctx, *b->cur, b->op, img, en, nullptr, bias);
}

int session_vmap(dctc_carver_batch* b, int* vmap_out, int* depth_out)
{
    if (!b->cur || !b->maps || b->axis == DCTC_AXIS_RESIZED) return DCTC_ERR_STATE;   // a combined resize returned its maps
    const int rc = frames_download(b->ctx, *b->maps, b->op, nullptr, nullptr, vmap_out);
    if (rc == DCTC_OK && depth_out) *depth_out = b->maps->depth;
    return rc;
}

}  // namespace

// ---- the context's single session ----------------------------------------------------------------------------------------

void dctc_carver_release(dctc_context* ctx)
{
    if (ctx->carver) session_destroy(ctx->carver);
    ctx->carver = nullptr;
    cudaFree(ctx->c_band); cudaFree(ctx->c_band_vals);
    cudaFreeHost(ctx->h_mirror); cudaFreeHost(ctx->h_band);
    ctx->c_band = nullptr; ctx->c_band_vals = nullptr; ctx->h_mirror = nullptr; ctx->h_band = nullptr;
    ctx->c_m_valid = false;
    ctx->mirror_valid = false;
}

// dctc_set_params with a session loaded (liblqr: lqr_carver_set_energy_function invalidates the energy map): the
// resident map is rebuilt with the new operator and the cumulative plane of the seam DP is dropped.
int dctc_carver_params_changed(dctc_context* ctx)
{
    if (!ctx->carver) return DCTC_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    ctx->mirror_valid = false;
    ctx->c_m_valid = false;
    dctc_carver_batch* b = ctx->carver;
    b->op = carver_op(ctx->op);
    const int rc = frames_full_energy(ctx, *b->cur, b->op);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DCTC_OK;
}

int dctc_carver_energy_plane(dctc_context* ctx, const float** en, size_t* en_pitch, int* w, int* h)
{
    dctc_carver_batch* b = ctx->carver;
    CarverFrames& f = *b->cur;
    b->op = carver_op(ctx->op);
    const float* op_en;
    int rc = frames_op_energy(ctx, f, b->op, &op_en);
    if (rc) return rc;
    Plane p;
    rc = frames_oriented(ctx, f, op_en, sizeof(float) * f.en_pitch, f.w, sizeof(float), p);
    if (rc) return rc;
    *en = (const float*) p.p;
    *en_pitch = p.pitch / sizeof(float);
    *w = p.cols;
    *h = p.rows;
    return DCTC_OK;
}

// A call on the loaded single session with the context's operator, maps request and incremental map.  A call that leaves
// the session unloaded releases it; frames that changed invalidate the dctc_pixel_energy mirror, and frames that grew
// drop its allocation (sized by its first use).
template <typename Op>
static int carver_call(dctc_context* ctx, Op&& op)
{
    dctc_carver_batch* b = ctx->carver;
    if (!b) return DCTC_ERR_STATE;
    b->op = carver_op(ctx->op);
    const CarverFrames* f = b->cur;
    const int w = f->w, iw = frames_image_w(*f), ih = frames_image_h(*f);
    SeamCall c;
    c.vmaps = ctx->c_dump_vmaps;
    c.rigidity = ctx->c_rigidity;
    c.delta_x = ctx->c_delta_x;
    c.incremental = ctx->c_incremental;
    c.m_valid = &ctx->c_m_valid;
    const int rc = op(b, c);
    if (!b->cur) {
        dctc_carver_release(ctx);
        return rc;
    }
    if (b->cur != f || b->cur->w != w) ctx->mirror_valid = false;
    if (frames_image_w(*b->cur) > iw || frames_image_h(*b->cur) > ih) {
        cudaFreeHost(ctx->h_mirror);
        ctx->h_mirror = nullptr;
    }
    return rc;
}

static int carver_load_impl(dctc_context* ctx, const uint8_t* img, int w, int h, int channels, size_t pitch)
{
    const int rc = session_create(ctx, 1, w, h, channels, false, false, &ctx->carver);
    if (rc) return rc;
    CK(ctx, cudaMalloc((void**) &ctx->c_band_vals, sizeof(float) * (size_t) h * DCTC_BAND_ROW));
    CK(ctx, cudaMallocHost((void**) &ctx->h_band, sizeof(float) * (size_t) h * DCTC_BAND_ROW + sizeof(int) * h));
    return session_load(ctx->carver, img, 0, pitch);
}

static int carver_seams(dctc_context* ctx, int axis, bool enlarge, int n_seams, int* seams_out)
{
    if (!ctx || n_seams < 0) return DCTC_ERR_INVALID;
    return carver_call(ctx, [&](dctc_carver_batch* b, const SeamCall& c) { return session_seams(b, axis, enlarge, n_seams, seams_out, c); });
}

static int carver_download(dctc_context* ctx, uint8_t* img, float* en, float* bias)
{
    if (!ctx->carver) return DCTC_ERR_STATE;
    ctx->carver->op = carver_op(ctx->op);
    return session_download(ctx->carver, img, en, bias);
}

static int carver_levels(dctc_context* ctx, int axis, int depth, int* seams_out)
{
    if (!ctx || depth < 0) return DCTC_ERR_INVALID;
    return carver_call(ctx, [&](dctc_carver_batch* b, const SeamCall& c) { return session_levels(b, axis, depth, seams_out, c); });
}

// The argument checks of the render calls
static bool levels_args(int n_levels, const int* extents, const void* out)
{
    if (n_levels <= 0 || !extents || !out) return false;
    for (int i = 0; i < n_levels; i++)
        if (extents[i] <= 0) return false;
    return true;
}

extern "C" {

int dctc_carver_load(dctc_context* ctx, const uint8_t* img, int w, int h, int channels, size_t pitch)
{
    if (!ctx || !img || w <= 0 || h <= 0 || channels < 1 || channels > 4 || pitch < (size_t) w * channels)
        return DCTC_ERR_INVALID;
    const int b = ctx->op.blocksize;
    if (!dctc_valid_blocksize(b)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    dctc_carver_release(ctx);
    // a half-built session (an allocation or the upload failed) must not look loaded to the next call
    const int rc = carver_load_impl(ctx, img, w, h, channels, pitch);
    if (rc) dctc_carver_release(ctx);
    return rc;
}

int dctc_carver_set_bias(dctc_context* ctx, const float* bias, size_t pitch)
{
    if (!ctx) return DCTC_ERR_INVALID;
    dctc_carver_batch* b = ctx->carver;
    if (!b) return DCTC_ERR_STATE;
    b->op = carver_op(ctx->op);
    const int rc = session_set_bias(b, bias, 0, pitch);
    if (!b->cur) dctc_carver_release(ctx);
    else if (rc == DCTC_OK) ctx->mirror_valid = false;
    return rc;
}

int dctc_carver_bias(dctc_context* ctx, float* out)
{
    if (!ctx || !out) return DCTC_ERR_INVALID;
    return carver_download(ctx, nullptr, nullptr, out);
}

int dctc_carver_width(const dctc_context* ctx) { return ctx && ctx->carver ? frames_image_w(session_frames(ctx->carver)) : 0; }
int dctc_carver_height(const dctc_context* ctx) { return ctx && ctx->carver ? frames_image_h(session_frames(ctx->carver)) : 0; }

int dctc_carver_energy(dctc_context* ctx, float* out)
{
    if (!ctx || !out) return DCTC_ERR_INVALID;
    return carver_download(ctx, nullptr, out, nullptr);
}

int dctc_carver_image(dctc_context* ctx, uint8_t* out)
{
    if (!ctx || !out) return DCTC_ERR_INVALID;
    return carver_download(ctx, out, nullptr, nullptr);
}

int dctc_carve_and_update(dctc_context* ctx, const int* seam_x, float* band_out, int* xmin, int* xmax)
{
    if (!ctx || !seam_x) return DCTC_ERR_INVALID;
    dctc_carver_batch* s = ctx->carver;
    if (!s || (s->axis != DCTC_AXIS_NONE && s->axis != DCTC_AXIS_WIDTH)) return DCTC_ERR_STATE;   // vertical seams only
    CarverFrames* f = s->cur;
    if (f->w <= 1) return DCTC_ERR_STATE;
    if (f->bias) return DCTC_ERR_STATE;   // the caller's seam and the operator's band values: no place for a bias
    const DctcK1Op op = carver_op(ctx->op);
    const int dx = ctx->c_delta_x, h = f->h, w_old = f->w, r = op.blocksize / 2, bs = 2 * r * (dx + 1);
    int* h_seam = (int*) ((char*) ctx->h_band + sizeof(float) * (size_t) h * DCTC_BAND_ROW);
    for (int y = 0; y < h; y++) {
        if (seam_x[y] < 0 || seam_x[y] >= w_old) return DCTC_ERR_STATE;
        // steps of at most delta_x (1 in the plug-in, src/render.c:313): the band width 2r(dx+1) and the band tiles rely on it
        if (y > 0 && (seam_x[y] - seam_x[y - 1] > dx || seam_x[y - 1] - seam_x[y] > dx)) return DCTC_ERR_INVALID;
        h_seam[y] = seam_x[y];
    }
    s->axis = DCTC_AXIS_WIDTH;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(f->seam, h_seam, sizeof(int) * h, cudaMemcpyHostToDevice, ctx->stream));
    dctc_carve_rows_kernel<256, 4, false><<<h, 256, 0, ctx->stream>>>(f->img, f->pitch, f->ch, f->en, f->en_pitch, f->seam, w_old, nullptr,
                                                                      0, 0, 0, 0, nullptr);
    CK(ctx, cudaGetLastError());
    ctx->launches++;
    f->w = w_old - 1;
    ctx->mirror_valid = false;
    ctx->c_m_valid = false;     // the host picked this seam: the device's cumulative plane no longer matches
    DctcK1Args a = frames_k1_args(*f, op, f->seam);
    a.band_vals = ctx->c_band_vals;
    a.band_stride = bs;
    int rc = dctc_run_k1(ctx, op, a, 1, ctx->stream, nullptr, dx);
    if (rc) return rc;
    if (band_out) {
        CK(ctx, cudaMemcpyAsync(ctx->h_band, ctx->c_band_vals, sizeof(float) * (size_t) h * bs, cudaMemcpyDeviceToHost,
                                ctx->stream));
    }
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    size_t k = 0;
    for (int y = 0; y < h; y++) {
        int lo, hi;
        dctc_band_limits(h_seam, y, h, f->w, r, &lo, &hi);
        if (xmin) xmin[y] = lo;
        if (xmax) xmax[y] = hi;
        if (band_out && hi >= lo) {
            memcpy(band_out + k, ctx->h_band + (size_t) y * bs, sizeof(float) * (size_t) (hi - lo + 1));
            k += (size_t) (hi - lo + 1);
        }
    }
    return DCTC_OK;
}

int dctc_carver_resize_width(dctc_context* ctx, int n_seams, int* seams_out)
{
    return carver_seams(ctx, DCTC_AXIS_WIDTH, false, n_seams, seams_out);
}

int dctc_carver_resize_height(dctc_context* ctx, int n_seams, int* seams_out)
{
    return carver_seams(ctx, DCTC_AXIS_HEIGHT, false, n_seams, seams_out);
}

int dctc_carver_enlarge_width(dctc_context* ctx, int n_seams, int* seams_out)
{
    return carver_seams(ctx, DCTC_AXIS_WIDTH, true, n_seams, seams_out);
}

int dctc_carver_enlarge_height(dctc_context* ctx, int n_seams, int* seams_out)
{
    return carver_seams(ctx, DCTC_AXIS_HEIGHT, true, n_seams, seams_out);
}

int dctc_carver_levels_width(dctc_context* ctx, int depth, int* seams_out)
{
    return carver_levels(ctx, DCTC_AXIS_WIDTH, depth, seams_out);
}

int dctc_carver_levels_height(dctc_context* ctx, int depth, int* seams_out)
{
    return carver_levels(ctx, DCTC_AXIS_HEIGHT, depth, seams_out);
}

int dctc_carver_render_levels(dctc_context* ctx, int n_levels, const int* extents, uint8_t* out)
{
    if (!ctx || !levels_args(n_levels, extents, out)) return DCTC_ERR_INVALID;
    if (!ctx->carver) return DCTC_ERR_STATE;
    return session_render_host(ctx->carver, n_levels, extents, out);
}

int dctc_resize_plan(int w, int h, int new_w, int new_h, DctcResizePass* passes, int max_passes)
{
    return dctc_resize_passes(w, h, new_w, new_h, passes, max_passes);
}

int dctc_carver_resize(dctc_context* ctx, int new_w, int new_h, int* seams_out, int* vmaps_out)
{
    if (!ctx || new_w <= 0 || new_h <= 0) return DCTC_ERR_INVALID;
    return carver_call(ctx, [&](dctc_carver_batch* b, const SeamCall& c) { return session_resize(b, new_w, new_h, seams_out, vmaps_out, c); });
}

int dctc_carver_set_incremental(dctc_context* ctx, int on)
{
    if (!ctx) return DCTC_ERR_INVALID;
    ctx->c_incremental = on != 0;
    return DCTC_OK;
}

int dctc_carver_set_rigidity(dctc_context* ctx, float rigidity)
{
    if (!ctx || !(rigidity >= 0.0f) || !std::isfinite(rigidity)) return DCTC_ERR_INVALID;
    if (rigidity != ctx->c_rigidity) {
        ctx->c_rigidity = rigidity;
        ctx->c_m_valid = false;   // the incremental map was built with the old pen
    }
    return DCTC_OK;
}

int dctc_carver_set_delta_x(dctc_context* ctx, int delta_x)
{
    if (!ctx || delta_x < 1) return DCTC_ERR_INVALID;
    if (delta_x > DCTC_MAX_DELTA_X) return DCTC_ERR_UNSUPPORTED;
    if (delta_x != ctx->c_delta_x) {
        ctx->c_delta_x = delta_x;
        ctx->c_m_valid = false;   // the incremental map was built for the old step width
    }
    return DCTC_OK;
}

int dctc_carver_rebuild_count(dctc_context* ctx)
{
    if (!ctx || !ctx->carver) return -1;
    if (!ctx->c_band) return 0;
    int v[4] = {0, 0, 0, 0};
    if (cudaSetDevice(ctx->device) != cudaSuccess) return -1;
    if (cudaMemcpyAsync(v, ctx->c_band, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
#ifdef DCTC_INCR_STATS
    fprintf(stderr, "incremental map: rebuilds %d, sum of range widths / 16 = %d, walk kclk = %d\n", v[1], v[2], v[3]);
#endif
    return v[1];
}

int dctc_carver_set_dump_vmaps(dctc_context* ctx, int on)
{
    if (!ctx) return DCTC_ERR_INVALID;
    ctx->c_dump_vmaps = on != 0;
    return DCTC_OK;
}

int dctc_carver_vmap(dctc_context* ctx, int* vmap_out, int* depth_out)
{
    if (!ctx) return DCTC_ERR_INVALID;
    if (!ctx->carver) return DCTC_ERR_STATE;
    ctx->carver->op = carver_op(ctx->op);
    return session_vmap(ctx->carver, vmap_out, depth_out);
}

int dctc_carver_paint_seams(dctc_context* ctx, uint8_t* img, int channels, size_t pitch)
{
    if (!ctx || !img || channels < 1 || channels > 4) return DCTC_ERR_INVALID;
    const dctc_carver_batch* s = ctx->carver;
    if (!s || !s->maps || s->maps->depth <= 0 || s->axis == DCTC_AXIS_RESIZED) return DCTC_ERR_STATE;
    CarverFrames* f = s->maps;
    CK(ctx, cudaSetDevice(ctx->device));
    Plane vs;   // the map in image orientation, row pitch = its width
    const int rc = frames_oriented(ctx, *f, f->vs, sizeof(int) * f->vs_w, f->vs_w, sizeof(int), vs);
    if (rc) return rc;
    const int w = vs.cols, h = vs.rows;
    if (pitch < (size_t) w * channels) return DCTC_ERR_INVALID;
    uint8_t* d = nullptr;
    const size_t dp = ((size_t) w * channels + 15) & ~(size_t) 15;
    CK(ctx, cudaMalloc((void**) &d, dp * h));
    cudaError_t e = cudaMemcpy2DAsync(d, dp, img, pitch, (size_t) w * channels, h, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        dctc_paint_seams_kernel<<<dim3((w + 255) / 256, h), 256, 0, ctx->stream>>>(d, dp, channels, w, h, (const int*) vs.p, f->depth);
        e = cudaGetLastError();
        ctx->launches++;
    }
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(img, pitch, d, dp, (size_t) w * channels, h, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t es = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) return dctc_fail_cuda(ctx, e);
    return DCTC_OK;
}

float dctc_pixel_energy(int x, int y, int w, int h, struct DctcLqrReadingWindow_* rw, void* extra_data)
{
    (void) rw;
    DctcCarverEnergyParams* p = (DctcCarverEnergyParams*) extra_data;
    dctc_context* ctx = p ? p->gpu : nullptr;
    if (!ctx || !ctx->carver || w != dctc_carver_width(ctx) || h != dctc_carver_height(ctx) || x < 0 || y < 0 || x >= w || y >= h) {
        if (ctx) ctx->last_cuda = 0;
        return __builtin_nanf("");
    }
    if (!ctx->mirror_valid) {
        // (sized at the first use: the session only gets narrower until the next load or enlarge, which free it)
        if (!ctx->h_mirror) {
            const cudaError_t e = cudaMallocHost((void**) &ctx->h_mirror, sizeof(float) * (size_t) w * h);
            if (e != cudaSuccess) { ctx->h_mirror = nullptr; dctc_fail_cuda(ctx, e); return __builtin_nanf(""); }
        }
        if (dctc_carver_energy(ctx, ctx->h_mirror) != DCTC_OK) return __builtin_nanf("");
        ctx->mirror_valid = true;
    }
    return ctx->h_mirror[(size_t) y * w + x];
}

}  // extern "C"

// ---- batch session: n equally sized frames through one device seam loop ---------------------------------------------
// The batch never touches the context's single session; it uses the context's device, stream and launch counter.

// A batch call brings the batch's rigidity; the per-axis calls also its maps rule
static SeamCall batch_call(const dctc_carver_batch* b)
{
    SeamCall c;
    c.rigidity = b->rigidity;
    c.delta_x = b->delta_x;
    return c;
}

static int batch_seams(dctc_carver_batch* b, int axis, bool enlarge, int n_seams, int* seams_out)
{
    if (!b || n_seams < 0) return DCTC_ERR_INVALID;
    SeamCall c = batch_call(b);
    c.vmaps = b->dump_vmaps;
    return session_seams(b, axis, enlarge, n_seams, seams_out, c);
}

extern "C" {

int dctc_carver_batch_create(dctc_context* ctx, int n_frames, int w, int h, int channels, int dump_vmaps, dctc_carver_batch** batch)
{
    if (!ctx || !batch) return DCTC_ERR_INVALID;
    *batch = nullptr;
    if (n_frames <= 0 || w <= 0 || h <= 0 || channels < 1 || channels > 4) return DCTC_ERR_INVALID;
    if (n_frames > 65535) return DCTC_ERR_UNSUPPORTED;   // the frame is a grid dimension of every launch
    CK(ctx, cudaSetDevice(ctx->device));
    return session_create(ctx, n_frames, w, h, channels, dump_vmaps != 0, true, batch);
}

void dctc_carver_batch_destroy(dctc_carver_batch* b)
{
    if (!b) return;
    if (cudaSetDevice(b->ctx->device) == cudaSuccess) cudaStreamSynchronize(b->ctx->stream);
    session_destroy(b);
}

int dctc_carver_batch_load(dctc_carver_batch* b, const uint8_t* imgs, size_t frame_stride, size_t pitch)
{
    if (!b || !imgs) return DCTC_ERR_INVALID;
    const CarverFrames& f = b->f;
    if (pitch < (size_t) f.w0 * f.ch || (f.n > 1 && frame_stride < pitch * f.h)) return DCTC_ERR_INVALID;
    dctc_context* ctx = b->ctx;
    if (!dctc_valid_blocksize(ctx->op.blocksize)) return DCTC_ERR_BLOCKSIZE;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return session_load(b, imgs, frame_stride, pitch);
}

int dctc_carver_batch_set_bias(dctc_carver_batch* b, const float* bias, size_t frame_stride, size_t pitch)
{
    if (!b) return DCTC_ERR_INVALID;
    return session_set_bias(b, bias, frame_stride, pitch);
}

int dctc_carver_batch_bias(dctc_carver_batch* b, float* out)
{
    if (!b || !out) return DCTC_ERR_INVALID;
    return session_download(b, nullptr, nullptr, out);
}

int dctc_carver_batch_set_rigidity(dctc_carver_batch* b, float rigidity)
{
    if (!b || !(rigidity >= 0.0f) || !std::isfinite(rigidity)) return DCTC_ERR_INVALID;
    b->rigidity = rigidity;
    return DCTC_OK;
}

int dctc_carver_batch_set_delta_x(dctc_carver_batch* b, int delta_x)
{
    if (!b || delta_x < 1) return DCTC_ERR_INVALID;
    if (delta_x > DCTC_MAX_DELTA_X) return DCTC_ERR_UNSUPPORTED;
    b->delta_x = delta_x;
    return DCTC_OK;
}

int dctc_carver_batch_width(const dctc_carver_batch* b) { return b ? frames_image_w(session_frames(b)) : 0; }
int dctc_carver_batch_height(const dctc_carver_batch* b) { return b ? frames_image_h(session_frames(b)) : 0; }

int dctc_carver_batch_resize_width(dctc_carver_batch* b, int n_seams, int* seams_out)
{
    return batch_seams(b, DCTC_AXIS_WIDTH, false, n_seams, seams_out);
}

int dctc_carver_batch_resize_height(dctc_carver_batch* b, int n_seams, int* seams_out)
{
    return batch_seams(b, DCTC_AXIS_HEIGHT, false, n_seams, seams_out);
}

int dctc_carver_batch_enlarge_width(dctc_carver_batch* b, int n_seams, int* seams_out)
{
    return batch_seams(b, DCTC_AXIS_WIDTH, true, n_seams, seams_out);
}

int dctc_carver_batch_enlarge_height(dctc_carver_batch* b, int n_seams, int* seams_out)
{
    return batch_seams(b, DCTC_AXIS_HEIGHT, true, n_seams, seams_out);
}

int dctc_carver_batch_resize(dctc_carver_batch* b, int new_w, int new_h, int* seams_out, int* vmaps_out)
{
    if (!b || new_w <= 0 || new_h <= 0) return DCTC_ERR_INVALID;
    return session_resize(b, new_w, new_h, seams_out, vmaps_out, batch_call(b));
}

int dctc_carver_batch_images(dctc_carver_batch* b, uint8_t* out)
{
    if (!b || !out) return DCTC_ERR_INVALID;
    return session_download(b, out, nullptr, nullptr);
}

int dctc_carver_batch_energy(dctc_carver_batch* b, float* out)
{
    if (!b || !out) return DCTC_ERR_INVALID;
    return session_download(b, nullptr, out, nullptr);
}

int dctc_carver_batch_vmap(dctc_carver_batch* b, int* vmap_out, int* depth_out)
{
    if (!b) return DCTC_ERR_INVALID;
    if (!b->dump_vmaps) return DCTC_ERR_STATE;   // maps were not asked for at create (an enlarge records them anyway)
    return session_vmap(b, vmap_out, depth_out);
}

int dctc_carver_batch_levels_width(dctc_carver_batch* b, int depth, int* seams_out)
{
    if (!b || depth < 0) return DCTC_ERR_INVALID;
    return session_levels(b, DCTC_AXIS_WIDTH, depth, seams_out, batch_call(b));
}

int dctc_carver_batch_levels_height(dctc_carver_batch* b, int depth, int* seams_out)
{
    if (!b || depth < 0) return DCTC_ERR_INVALID;
    return session_levels(b, DCTC_AXIS_HEIGHT, depth, seams_out, batch_call(b));
}

int dctc_carver_batch_render_levels(dctc_carver_batch* b, int n_levels, const int* extents, uint8_t* out)
{
    if (!b || !levels_args(n_levels, extents, out)) return DCTC_ERR_INVALID;
    return session_render_host(b, n_levels, extents, out);
}

int dctc_carver_batch_render_levels_dev(dctc_carver_batch* b, int n_levels, const int* extents, uint8_t* d_out)
{
    if (!b || !levels_args(n_levels, extents, d_out)) return DCTC_ERR_INVALID;
    return session_render(b, n_levels, extents, d_out);
}

}  // extern "C"

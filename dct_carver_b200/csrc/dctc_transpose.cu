// Frame transpose of the height operations of the carver sessions (dctc_k2_carver.cu).  A height operation runs the width
// seam loop on the transposed frames, as liblqr's lqr_carver_resize changes the height by transposing the carver: one
// launch turns every loaded frame into its transpose, and one launch per plane turns a result back into image
// orientation on its way to the host.  It runs once per call, never per seam, and is bound by HBM bandwidth.
#include "dctc_launch.h"

namespace {

constexpr int TT = 32;        // tile edge
constexpr int TROWS = 8;      // rows of the tile each thread row walks

template <int E>
struct Elem { uint8_t b[E]; };
template <> struct Elem<2> { uint16_t v; };
template <> struct Elem<4> { uint32_t v; };

// dst[z][x][y] = src[z][y][x] for a cols x rows plane per frame (elements of E bytes).  One CTA moves one 32 x 32 tile
// through shared memory, so that reads and writes both walk along rows; blockIdx.z = frame, tile rows beyond the grid's
// y extent in a grid-stride loop.
template <int E>
__global__ void __launch_bounds__(TT * TROWS) dctc_transpose_kernel(const uint8_t* __restrict__ src, size_t src_pitch, size_t src_fs,
                                                                    uint8_t* __restrict__ dst, size_t dst_pitch, size_t dst_fs,
                                                                    int cols, int rows)
{
    __shared__ Elem<E> tile[TT][TT + 1];
    const uint8_t* s = src + blockIdx.z * src_fs;
    uint8_t* d = dst + blockIdx.z * dst_fs;
    const int x0 = blockIdx.x * TT;
    for (int y0 = blockIdx.y * TT; y0 < rows; y0 += gridDim.y * TT) {
        for (int j = threadIdx.y; j < TT; j += TROWS) {
            const int x = x0 + threadIdx.x, y = y0 + j;
            if (x < cols && y < rows) tile[j][threadIdx.x] = *(const Elem<E>*) (s + (size_t) y * src_pitch + (size_t) x * E);
        }
        __syncthreads();
        for (int j = threadIdx.y; j < TT; j += TROWS) {
            const int y = y0 + threadIdx.x, x = x0 + j;   // output row x, column y
            if (x < cols && y < rows) *(Elem<E>*) (d + (size_t) x * dst_pitch + (size_t) y * E) = tile[threadIdx.x][j];
        }
        __syncthreads();
    }
}

}  // namespace

cudaError_t dctc_launch_transpose(const void* src, size_t src_pitch, size_t src_fs, void* dst, size_t dst_pitch, size_t dst_fs,
                                  int cols, int rows, int n_frames, int esize, cudaStream_t stream)
{
    if (cols <= 0 || rows <= 0 || n_frames <= 0) return cudaSuccess;
    const unsigned ty = (unsigned) ((rows + TT - 1) / TT);
    const dim3 grid((unsigned) ((cols + TT - 1) / TT), ty < 65535u ? ty : 65535u, (unsigned) n_frames);
    const dim3 block(TT, TROWS);
    const uint8_t* s = (const uint8_t*) src;
    uint8_t* d = (uint8_t*) dst;
    switch (esize) {
    case 1: dctc_transpose_kernel<1><<<grid, block, 0, stream>>>(s, src_pitch, src_fs, d, dst_pitch, dst_fs, cols, rows); break;
    case 2: dctc_transpose_kernel<2><<<grid, block, 0, stream>>>(s, src_pitch, src_fs, d, dst_pitch, dst_fs, cols, rows); break;
    case 3: dctc_transpose_kernel<3><<<grid, block, 0, stream>>>(s, src_pitch, src_fs, d, dst_pitch, dst_fs, cols, rows); break;
    case 4: dctc_transpose_kernel<4><<<grid, block, 0, stream>>>(s, src_pitch, src_fs, d, dst_pitch, dst_fs, cols, rows); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

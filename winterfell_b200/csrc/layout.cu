// layout.cu — see layout.cuh.
#include "layout.cuh"

__global__ void __launch_bounds__(256) cols_to_seg_kernel(const u64* __restrict__ src, size_t nrows, int d, int q0, int mont,
                                                          SegMatrix dst) {
    // thread = (row, segment); reads W columns at `row` (coalesced per column across the warp),
    // writes one W*8-byte segment row. All W loads are issued before the first use: the kernel is a pure
    // transpose and ran latency-bound (56 long-scoreboard stalls per issue) with one load in flight per thread.
    size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = blockIdx.y;
    if (row >= nrows) return;
    u64* o = dst.base + (size_t)g * dst.seg_stride + row * dst.W;
    u64 v[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        u32 col = g * dst.W + q, sc = col + (u32)q0;   // base column `col` = component sc % d of source column sc / d
        v[q] = (q < dst.W && col < dst.cols) ? __ldg(src + (size_t)(sc / d) * nrows * d + row * d + (sc % d)) : 0;
    }
    if (mont) {
#pragma unroll
        for (int q = 0; q < 8; q++) v[q] = gl_from_mont(v[q]);
    }
    if (dst.W == 8) {
        ulonglong2* o2 = reinterpret_cast<ulonglong2*>(o);
#pragma unroll
        for (int k = 0; k < 4; k++) o2[k] = make_ulonglong2(v[2 * k], v[2 * k + 1]);
    } else {
#pragma unroll
        for (int q = 0; q < 8; q++) if (q < dst.W) o[q] = v[q];
    }
}
__global__ void __launch_bounds__(256) rows_to_seg_kernel(const u64* __restrict__ src, SegMatrix dst) {
    size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = blockIdx.y;
    if (row >= dst.rows) return;
    u64* o = dst.base + (size_t)g * dst.seg_stride + row * dst.W;
    for (int q = 0; q < dst.W; q++) {
        u32 col = g * dst.W + q;
        o[q] = col < dst.cols ? src[row * dst.cols + col] : 0;
    }
}
__global__ void __launch_bounds__(256) seg_to_flat_kernel(SegMatrix src, u64* __restrict__ dst, int row_major, int mont) {
    size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = blockIdx.y;
    if (row >= src.rows) return;
    const u64* in = src.base + (size_t)g * src.seg_stride + row * src.W;
    for (int q = 0; q < src.W; q++) {
        u32 col = g * src.W + q;
        if (col >= src.cols) break;
        u64 v = in[q];
        if (mont) v = gl_to_mont(v);
        if (row_major) dst[row * src.cols + col] = v;
        else dst[(size_t)col * src.rows + row] = v;
    }
}
__global__ void gather_rows_kernel(SegMatrix src, const u64* __restrict__ pos, size_t k, u64* __restrict__ dst, int mont) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= k * src.cols) return;
    size_t i = idx / src.cols;
    u32 col = (u32)(idx % src.cols);
    size_t row = pos[i];
    if (row == ~(size_t)0) { dst[idx] = 0; return; }  // not held by this rank (sharded proof): another rank's words are summed in
    u64 v = src.base[(size_t)(col / src.W) * src.seg_stride + row * src.W + (col % src.W)];
    dst[idx] = mont ? gl_to_mont(v) : v;
}
__global__ void gather_digests_kernel(const u64* __restrict__ nodes, const u64* __restrict__ leaves, size_t n,
                                      const u64* __restrict__ want, size_t k, u64* __restrict__ dst) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= k * 4) return;
    size_t i = idx >> 2, w = idx & 3;
    u64 e = want[i];
    if (e == ~(u64)0) { dst[idx] = 0; return; }       // not held by this rank
    dst[idx] = e < n ? nodes[e * 4 + w] : leaves[(e - n) * 4 + w];
}
// row r *= base^r. Each thread walks SCALE_ROWS rows spaced one block apart (coalesced), computing
// base^r once by square-and-multiply and stepping with base^256 afterwards (the one-power-per-element
// form was 104 us on the 2^21-row composition polynomial: 40 multiplications per element).
#define SCALE_ROWS 16
__global__ void __launch_bounds__(256) scale_rows_kernel(SegMatrix m, u64 base, u64 step /* base^256 */) {
    size_t row = (size_t)blockIdx.x * (256 * SCALE_ROWS) + threadIdx.x;
    u32 g = blockIdx.y;
    if (row >= m.rows) return;
    u64 f = gl_pow(base, row);
    u64* p = m.base + (size_t)g * m.seg_stride;
#pragma unroll 4
    for (int k = 0; k < SCALE_ROWS && row < m.rows; k++, row += 256) {
        u64* pr = p + row * m.W;
        for (int q = 0; q < m.W; q++) pr[q] = gl_mul(pr[q], f);
        f = gl_mul(f, step);
    }
}

__global__ void __launch_bounds__(256) select_cols_kernel(SegMatrix src, u32 first, SegMatrix dst) {
    size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 g = blockIdx.y;
    if (row >= dst.rows) return;
    u64* o = dst.base + (size_t)g * dst.seg_stride + row * dst.W;
    for (int q = 0; q < dst.W; q++) {
        u32 col = g * dst.W + q;
        u64 v = 0;
        if (col < dst.cols) {
            u32 sc = first + col;
            v = src.base[(size_t)(sc / src.W) * src.seg_stride + row * src.W + (sc % src.W)];
        }
        o[q] = v;
    }
}

static dim3 row_grid(size_t rows, u32 nseg) { return dim3((unsigned)((rows + 255) / 256), nseg); }

cudaError_t layout_cols_to_seg(const u64* src, size_t nrows, int d, int mont, const SegMatrix& dst, cudaStream_t st, int q0) {
    cols_to_seg_kernel<<<row_grid(nrows, dst.nseg()), 256, 0, st>>>(src, nrows, d, q0, mont, dst);
    return cudaGetLastError();
}
cudaError_t layout_rows_to_seg(const u64* src, const SegMatrix& dst, cudaStream_t st) {
    rows_to_seg_kernel<<<row_grid(dst.rows, dst.nseg()), 256, 0, st>>>(src, dst);
    return cudaGetLastError();
}
cudaError_t layout_seg_to_flat(const SegMatrix& src, u64* dst, int row_major, int mont, cudaStream_t st) {
    seg_to_flat_kernel<<<row_grid(src.rows, src.nseg()), 256, 0, st>>>(src, dst, row_major, mont);
    return cudaGetLastError();
}
cudaError_t layout_gather_rows(const SegMatrix& src, const u64* pos, size_t k, u64* dst, int mont, cudaStream_t st) {
    size_t total = k * src.cols;
    gather_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, pos, k, dst, mont);
    return cudaGetLastError();
}
cudaError_t layout_gather_digests(const u64* nodes, const u64* leaves, size_t n, const u64* want, size_t k, u64* dst,
                                  cudaStream_t st) {
    gather_digests_kernel<<<(unsigned)((k * 4 + 255) / 256), 256, 0, st>>>(nodes, leaves, n, want, k, dst);
    return cudaGetLastError();
}
cudaError_t layout_scale_rows_by_powers(const SegMatrix& m, u64 base, cudaStream_t st) {
    dim3 grid((unsigned)((m.rows + 256 * SCALE_ROWS - 1) / (256 * SCALE_ROWS)), m.nseg());
    scale_rows_kernel<<<grid, 256, 0, st>>>(m, base, gl_pow(base, 256));
    return cudaGetLastError();
}
cudaError_t layout_select_cols(const SegMatrix& src, u32 first, const SegMatrix& dst, cudaStream_t st) {
    select_cols_kernel<<<row_grid(dst.rows, dst.nseg()), 256, 0, st>>>(src, first, dst);
    return cudaGetLastError();
}

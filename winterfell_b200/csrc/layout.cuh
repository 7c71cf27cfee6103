// layout.cuh — conversions between host-facing layouts (column-major ColMatrix columns, row-major
// RowMatrix rows) and the device segment layout, plus small gathers for query openings.
#pragma once
#include <cuda_runtime.h>

#include "commit.cuh"

// src: columns of `d`-degree elements, column j at src[j * nrows * d ...], element (row, comp) at
// row * d + comp. Base column q = component (q0 + q) % d of column (q0 + q) / d: q0 < d skips the first components of
// column 0 (a block of base columns that starts inside an element). mont: words are Montgomery form.
cudaError_t layout_cols_to_seg(const u64* src, size_t nrows, int d, int mont, const SegMatrix& dst, cudaStream_t st, int q0 = 0);
// src: row-major [rows][cols]
cudaError_t layout_rows_to_seg(const u64* src, const SegMatrix& dst, cudaStream_t st);
// dst: column-major [cols][rows] (row_major = 0) or row-major [rows][cols] (row_major = 1)
cudaError_t layout_seg_to_flat(const SegMatrix& src, u64* dst, int row_major, int mont, cudaStream_t st);
// dst[i][0..cols) = row positions[i]
cudaError_t layout_gather_rows(const SegMatrix& src, const u64* d_positions, size_t k, u64* dst, int mont, cudaStream_t st);
// want[i] < n: nodes[want[i]]; else leaves[want[i] - n]; 4 words each
cudaError_t layout_gather_digests(const u64* nodes, const u64* leaves, size_t n, const u64* d_want, size_t k, u64* dst,
                                  cudaStream_t st);
// row i of every column *= base^i
cudaError_t layout_scale_rows_by_powers(const SegMatrix& m, u64 base, cudaStream_t st);
// dst(row, j) = src(row, first + j) for j < dst.cols
cudaError_t layout_select_cols(const SegMatrix& src, u32 first, const SegMatrix& dst, cudaStream_t st);

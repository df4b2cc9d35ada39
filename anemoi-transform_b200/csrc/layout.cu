// layout.cu — layout changes around the SpMM: field-major <-> point-major transposes, the
// row gather of the nearest-neighbour / masked regrid, and mask construction by comparison.
//
// Reference call sites (src/anemoi/transform/filters/fields/):
//   regrid.py:309  `field.to_numpy(flatten=True)` delivers one array per field (field-major);
//   regrid.py:380  `data[..., self.nearest_grid_points]`  (ScipyKDTreeNearestNeighbours)
//   regrid.py:420  `data[..., self.mask]`                  (MaskedRegrid)
//   apply_mask.py:160-163  `OPERATORS[op](mask_values, threshold)` / `mask_values == mask_value`
#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace at {

constexpr int kTile = 64;  // transpose tile edge (elements)

// dst[c, r] = src[r, c].  64x64 tile through shared memory; 256 threads, each moves 16
// elements.  Reads and writes are both coalesced along their contiguous dimension.
template <typename T>
__global__ void __launch_bounds__(256)
    transpose_kernel(const T* __restrict__ src, long long rows, long long cols, size_t ld_src,
                     T* __restrict__ dst, size_t ld_dst, long long tiles_c) {
    __shared__ T tile[kTile][kTile + 1];
    const long long tr = blockIdx.x / tiles_c, tc = blockIdx.x % tiles_c;
    const long long r0 = tr * kTile, c0 = tc * kTile;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
#pragma unroll 4
    for (int i = ty; i < kTile; i += 4) {
        const long long r = r0 + i, c = c0 + tx;
        if (r < rows && c < cols) tile[i][tx] = __ldg(src + static_cast<size_t>(r) * ld_src + c);
    }
    __syncthreads();
#pragma unroll 4
    for (int i = ty; i < kTile; i += 4) {
        const long long c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) dst[static_cast<size_t>(c) * ld_dst + r] = tile[tx][i];
    }
}

// The same transpose with 16-byte global accesses on both sides (float4 / double2): a thread
// loads PER consecutive elements of a source row, and writes PER consecutive elements of a
// destination row gathered from a shared-memory column.  Used whenever both arrays allow
// aligned 16-byte accesses (what the field I/O engine and DeviceBatch provide); ragged edges
// of the array fall back to scalar accesses inside the kernel.
template <typename T>
__global__ void __launch_bounds__(256)
    transpose_vec_kernel(const T* __restrict__ src, long long rows, long long cols, size_t ld_src,
                         T* __restrict__ dst, size_t ld_dst, long long tiles_c) {
    constexpr int PER = 16 / sizeof(T);       // elements per 16-byte access
    constexpr int VPR = kTile / PER;          // 16-byte accesses per tile row
    constexpr int STEP = 256 / VPR;           // tile rows covered per pass
    using Vec = typename std::conditional<sizeof(T) == 4, float4, double2>::type;
    __shared__ T tile[kTile][kTile + 1];
    const long long tr = blockIdx.x / tiles_c, tc = blockIdx.x % tiles_c;
    const long long r0 = tr * kTile, c0 = tc * kTile;
    const int v = threadIdx.x % VPR, line = threadIdx.x / VPR;
#pragma unroll 4
    for (int i = line; i < kTile; i += STEP) {
        const long long r = r0 + i, c = c0 + v * PER;
        if (r >= rows || c >= cols) continue;
        const T* p = src + static_cast<size_t>(r) * ld_src + c;
        if (c + PER <= cols) {
            const Vec x = __ldg(reinterpret_cast<const Vec*>(p));
            const T* e = reinterpret_cast<const T*>(&x);
#pragma unroll
            for (int k = 0; k < PER; ++k) tile[i][v * PER + k] = e[k];
        } else {
            for (int k = 0; c + k < cols; ++k) tile[i][v * PER + k] = __ldg(p + k);
        }
    }
    __syncthreads();
#pragma unroll 4
    for (int j = line; j < kTile; j += STEP) {
        const long long c = c0 + j, r = r0 + v * PER;
        if (c >= cols || r >= rows) continue;
        T* p = dst + static_cast<size_t>(c) * ld_dst + r;
        if (r + PER <= rows) {
            Vec x;
            T* e = reinterpret_cast<T*>(&x);
#pragma unroll
            for (int k = 0; k < PER; ++k) e[k] = tile[v * PER + k][j];
            *reinterpret_cast<Vec*>(p) = x;
        } else {
            for (int k = 0; r + k < rows; ++k) p[k] = tile[v * PER + k][j];
        }
    }
}

// One warp per output row and 16-byte chunk tile.  blockIdx.x = row_block * tiles + tile: CTAs
// that run together cover adjacent column tiles of the same rows, i.e. long contiguous spans
// of each source row (DRAM page locality, as in spmm_f32_kernel's super-tiles).
template <typename V>
__global__ void __launch_bounds__(256)
    gather_rows_kernel(const long long* __restrict__ idx, long long n_out, long long n_src,
                       const V* __restrict__ X, size_t ldx, V* __restrict__ Y, size_t ldy,
                       int n_vec, int tiles, int* __restrict__ err_flag) {
    const long long row = static_cast<long long>(blockIdx.x / tiles) * 8 + (threadIdx.x >> 5);
    const int tile = static_cast<int>(blockIdx.x % tiles);
    if (row >= n_out) return;
    const int lane = threadIdx.x & 31;
    const long long s = idx[row];
    if (s < 0 || s >= n_src) {
        if (lane == 0 && err_flag != nullptr) *err_flag = 1;
        return;
    }
    const V* xr = X + static_cast<size_t>(s) * ldx;
    V* yr = Y + static_cast<size_t>(row) * ldy;
    const int v0 = tile * 128;
    V tmp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int v = v0 + j * 32 + lane;
        if (v < n_vec) tmp[j] = __ldg(xr + v);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int v = v0 + j * 32 + lane;
        if (v < n_vec) __stcs(yr + v, tmp[j]);
    }
}

// Y[r, j] = X[r, cols[j]]: regroup the columns (fields) of a resident batch, e.g. to lay
// (u, v) / (q, t) partners next to each other.  One warp per row; writes are coalesced,
// reads stay inside one row (at most a few KB apart).
template <typename T>
__global__ void __launch_bounds__(256)
    gather_cols_kernel(const int* __restrict__ cols, int n_out, const T* __restrict__ X, size_t ldx,
                       T* __restrict__ Y, size_t ldy, long long n_rows) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const T* xr = X + static_cast<size_t>(row) * ldx;
    T* yr = Y + static_cast<size_t>(row) * ldy;
    for (int j = threadIdx.x & 31; j < n_out; j += 32) yr[j] = __ldg(xr + __ldg(cols + j));
}

template <typename T>
__global__ void compare_mask_kernel(const T* __restrict__ values, size_t stride, long long n,
                                    int op, T thr, uint8_t* __restrict__ mask) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const T v = values[static_cast<size_t>(i) * stride];
    bool m;
    switch (op) {
        case 0: m = v == thr; break;
        case 1: m = v != thr; break;
        case 2: m = v > thr; break;
        case 3: m = v >= thr; break;
        case 4: m = v < thr; break;
        case 5: m = v <= thr; break;
        default: m = v == v; break;  // 6: not NaN
    }
    mask[i] = m ? 1 : 0;
}

// Y[r, g] = sum over the group's columns in order, starting from the first term (numpy's
// `s = c0; s += c1; ...`, sum.py:109-115).  One warp per row, lanes over groups.
template <typename T>
__global__ void __launch_bounds__(256)
    sum_cols_kernel(const int* __restrict__ cols, int n_groups, int n_terms, const T* __restrict__ X, size_t ldx,
                    T* __restrict__ Y, size_t ldy, long long n_rows) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const T* xr = X + static_cast<size_t>(row) * ldx;
    T* yr = Y + static_cast<size_t>(row) * ldy;
    for (int g = threadIdx.x & 31; g < n_groups; g += 32) {
        T s = __ldg(xr + __ldg(cols + g * n_terms));
        for (int k = 1; k < n_terms; ++k) s = s + __ldg(xr + __ldg(cols + g * n_terms + k));
        yr[g] = s;
    }
}

// flags[j] |= 1 (any < lo) | 2 (any > hi) | 4 (any NaN) over the rows of column first_col + j.
// One warp per row chunk; lanes over columns; a warp ORs its findings once at the end.
template <typename T>
__global__ void __launch_bounds__(256)
    range_flags_kernel(const T* __restrict__ X, size_t ldx, long long n_rows, int first_col, int n_cols, T lo, T hi,
                       unsigned* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const long long warp = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    const long long n_warps = static_cast<long long>(gridDim.x) * 8;
    for (int c0 = 0; c0 < n_cols; c0 += 32) {
        const int c = c0 + lane;
        unsigned f = 0;
        if (c < n_cols)
            for (long long r = warp; r < n_rows; r += n_warps) {
                const T v = __ldg(X + static_cast<size_t>(r) * ldx + first_col + c);
                f |= (v < lo ? 1u : 0u) | (v > hi ? 2u : 0u) | (v != v ? 4u : 0u);
            }
        if (f != 0) atomicOr(flags + c, f);
    }
}

template <typename T>
static int launch_transpose(const void* src, int64_t rows, int64_t cols, int64_t ld_src, void* dst,
                            int64_t ld_dst, cudaStream_t st) {
    const long long tiles_r = (rows + kTile - 1) / kTile, tiles_c = (cols + kTile - 1) / kTile;
    const long long n_tiles = tiles_r * tiles_c;
    if (n_tiles >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "at_transpose: array too large");
    constexpr int64_t per16 = 16 / sizeof(T);
    const bool vec16 = ld_src % per16 == 0 && ld_dst % per16 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
    if (vec16) {
        transpose_vec_kernel<T><<<static_cast<unsigned>(n_tiles), 256, 0, st>>>(
            static_cast<const T*>(src), rows, cols, static_cast<size_t>(ld_src), static_cast<T*>(dst),
            static_cast<size_t>(ld_dst), tiles_c);
        AT_LAUNCH_CHECK("transpose_vec_kernel");
        return AT_OK;
    }
    transpose_kernel<T><<<static_cast<unsigned>(n_tiles), 256, 0, st>>>(
        static_cast<const T*>(src), rows, cols, static_cast<size_t>(ld_src), static_cast<T*>(dst),
        static_cast<size_t>(ld_dst), tiles_c);
    AT_LAUNCH_CHECK("transpose_kernel");
    return AT_OK;
}

template <typename V>
static int launch_gather(const int64_t* idx, int64_t n_out, int64_t n_src, const void* X, int64_t ldx_v,
                         void* Y, int64_t ldy_v, int64_t n_vec, int32_t* err_flag, cudaStream_t st) {
    const int64_t tiles = (n_vec + 127) / 128, gx = (n_out + 7) / 8 * tiles;
    if (gx >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "at_gather_rows: too large");
    gather_rows_kernel<V><<<static_cast<unsigned>(gx), 256, 0, st>>>(
        reinterpret_cast<const long long*>(idx), n_out, n_src, static_cast<const V*>(X), static_cast<size_t>(ldx_v),
        static_cast<V*>(Y), static_cast<size_t>(ldy_v), static_cast<int>(n_vec), static_cast<int>(tiles), err_flag);
    AT_LAUNCH_CHECK("gather_rows_kernel");
    return AT_OK;
}

}  // namespace at

using namespace at;

extern "C" int at_transpose(const void* src, int64_t rows, int64_t cols, int64_t ld_src, void* dst,
                            int64_t ld_dst, int elem_size, void* stream) {
    AT_REQUIRE(src != nullptr && dst != nullptr, "at_transpose: null argument");
    AT_REQUIRE(rows >= 0 && cols >= 0 && ld_src >= cols && ld_dst >= rows,
               "at_transpose: bad shape rows=%lld cols=%lld ld_src=%lld ld_dst=%lld", (long long)rows,
               (long long)cols, (long long)ld_src, (long long)ld_dst);
    if (rows == 0 || cols == 0) return AT_OK;
    if (elem_size == 4) return launch_transpose<float>(src, rows, cols, ld_src, dst, ld_dst, as_stream(stream));
    if (elem_size == 8) return launch_transpose<double>(src, rows, cols, ld_src, dst, ld_dst, as_stream(stream));
    return set_error(AT_ERR_INVALID, "at_transpose: elem_size must be 4 or 8");
}

extern "C" int at_gather_rows(const int64_t* idx, int64_t n_out, int64_t n_src, const void* X,
                              int64_t ldx, void* Y, int64_t ldy, int64_t n_fields, int elem_size,
                              int32_t* err_flag, void* stream) {
    AT_REQUIRE(elem_size == 4 || elem_size == 8, "at_gather_rows: elem_size must be 4 or 8");
    AT_REQUIRE(n_out >= 0 && n_src >= 0 && n_fields >= 0 && ldx >= n_fields && ldy >= n_fields,
               "at_gather_rows: bad shape");
    if (n_out == 0 || n_fields == 0) return AT_OK;  // zero-length device arrays have null pointers
    AT_REQUIRE(idx != nullptr && X != nullptr && Y != nullptr, "at_gather_rows: null argument");
    cudaStream_t st = as_stream(stream);
    const int64_t per16 = 16 / elem_size;
    const bool vec16 = ldx % per16 == 0 && ldy % per16 == 0 &&
                       (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0;
    if (vec16) {
        // whole 16-byte chunks, including the padding columns inside ld
        const int64_t n_vec = (n_fields + per16 - 1) / per16;
        return launch_gather<uint4>(idx, n_out, n_src, X, ldx / per16, Y, ldy / per16, n_vec, err_flag, st);
    }
    if (elem_size == 4)
        return launch_gather<uint32_t>(idx, n_out, n_src, X, ldx, Y, ldy, n_fields, err_flag, st);
    return launch_gather<uint2>(idx, n_out, n_src, X, ldx, Y, ldy, n_fields, err_flag, st);
}

extern "C" int at_gather_cols(const int32_t* cols, int32_t n_out, int64_t n_rows, const void* X, int64_t ldx,
                              void* Y, int64_t ldy, int elem_size, void* stream) {
    AT_REQUIRE(cols != nullptr && X != nullptr && Y != nullptr, "at_gather_cols: null argument");
    AT_REQUIRE(elem_size == 4 || elem_size == 8, "at_gather_cols: elem_size must be 4 or 8");
    AT_REQUIRE(n_out >= 0 && n_rows >= 0 && ldy >= n_out, "at_gather_cols: bad shape");
    if (n_out == 0 || n_rows == 0) return AT_OK;
    const int64_t blocks = (n_rows + 7) / 8;
    AT_REQUIRE(blocks < (1ll << 31), "at_gather_cols: too many rows");
    if (elem_size == 4)
        gather_cols_kernel<float><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            cols, n_out, static_cast<const float*>(X), static_cast<size_t>(ldx), static_cast<float*>(Y),
            static_cast<size_t>(ldy), n_rows);
    else
        gather_cols_kernel<double><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            cols, n_out, static_cast<const double*>(X), static_cast<size_t>(ldx), static_cast<double*>(Y),
            static_cast<size_t>(ldy), n_rows);
    AT_LAUNCH_CHECK("gather_cols_kernel");
    return AT_OK;
}

extern "C" int at_compare_mask(const void* values, int dtype, int64_t stride, int64_t n, int op,
                               double threshold, uint8_t* mask, void* stream) {
    AT_REQUIRE(values != nullptr && mask != nullptr, "at_compare_mask: null argument");
    AT_REQUIRE(dtype == AT_F32 || dtype == AT_F64, "at_compare_mask: bad dtype code");
    AT_REQUIRE(op >= 0 && op <= 6, "at_compare_mask: unknown operator %d", op);
    AT_REQUIRE(n >= 0 && stride >= 1, "at_compare_mask: bad shape");
    if (n == 0) return AT_OK;
    const int64_t blocks = (n + 255) / 256;
    AT_REQUIRE(blocks < (1ll << 31), "at_compare_mask: too large");
    if (dtype == AT_F32)
        // numpy compares a float32 array with a Python scalar in float32 (NEP 50)
        compare_mask_kernel<float><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            static_cast<const float*>(values), static_cast<size_t>(stride), n, op, static_cast<float>(threshold), mask);
    else
        compare_mask_kernel<double><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            static_cast<const double*>(values), static_cast<size_t>(stride), n, op, threshold, mask);
    AT_LAUNCH_CHECK("compare_mask_kernel");
    return AT_OK;
}

extern "C" int at_sum_cols(const int32_t* cols, int32_t n_groups, int32_t n_terms, int64_t n_rows, const void* X,
                           int64_t ldx, void* Y, int64_t ldy, int dtype, void* stream) {
    AT_REQUIRE(cols != nullptr && X != nullptr && Y != nullptr, "at_sum_cols: null argument");
    AT_REQUIRE(dtype == AT_F32 || dtype == AT_F64, "at_sum_cols: bad dtype code");
    AT_REQUIRE(n_groups >= 0 && n_terms >= 1 && n_rows >= 0 && ldy >= n_groups, "at_sum_cols: bad shape");
    if (n_groups == 0 || n_rows == 0) return AT_OK;
    const int64_t blocks = (n_rows + 7) / 8;
    AT_REQUIRE(blocks < (1ll << 31), "at_sum_cols: too many rows");
    if (dtype == AT_F32)
        sum_cols_kernel<float><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            cols, n_groups, n_terms, static_cast<const float*>(X), static_cast<size_t>(ldx), static_cast<float*>(Y),
            static_cast<size_t>(ldy), n_rows);
    else
        sum_cols_kernel<double><<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
            cols, n_groups, n_terms, static_cast<const double*>(X), static_cast<size_t>(ldx), static_cast<double*>(Y),
            static_cast<size_t>(ldy), n_rows);
    AT_LAUNCH_CHECK("sum_cols_kernel");
    return AT_OK;
}

extern "C" int at_range_flags(const void* X, int64_t ldx, int64_t n_rows, int32_t first_col, int32_t n_cols, int dtype,
                              double lo, double hi, uint32_t* flags, void* stream) {
    AT_REQUIRE(X != nullptr && flags != nullptr, "at_range_flags: null argument");
    AT_REQUIRE(dtype == AT_F32 || dtype == AT_F64, "at_range_flags: bad dtype code");
    AT_REQUIRE(n_rows >= 0 && first_col >= 0 && n_cols >= 0 && ldx >= first_col + n_cols, "at_range_flags: bad shape");
    if (n_rows == 0 || n_cols == 0) return AT_OK;
    const unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n_rows + 7) / 8, 8 * sm_count()));
    if (dtype == AT_F32)
        // numpy compares a float32 array with a Python scalar in float32 (NEP 50)
        range_flags_kernel<float><<<blocks, 256, 0, as_stream(stream)>>>(
            static_cast<const float*>(X), static_cast<size_t>(ldx), n_rows, first_col, n_cols, static_cast<float>(lo),
            static_cast<float>(hi), flags);
    else
        range_flags_kernel<double><<<blocks, 256, 0, as_stream(stream)>>>(
            static_cast<const double*>(X), static_cast<size_t>(ldx), n_rows, first_col, n_cols, lo, hi, flags);
    AT_LAUNCH_CHECK("range_flags_kernel");
    return AT_OK;
}

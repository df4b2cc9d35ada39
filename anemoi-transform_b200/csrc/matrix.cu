// matrix.cu — interpolation-matrix construction on the device, replacing the external `mir`
// binary of `anemoi-transform make-regrid-file` (commands/make-regrid-file.py:142-160) and
// earthkit-regrid's matrix inventory (filters/fields/regrid.py:211-259) for the case that can
// be built without either: 4-point bilinear weights from a regular lat-lon source grid, and
// the structured bilinear (2 rows x 2 points) / bicubic (4 rows x 4 points) stencils on any
// global structured grid (rows of constant latitude, equally spaced longitudes: octahedral and
// classic reduced Gaussian, full Gaussian, regular lat-lon), and first-order conservative
// grid-box averages between two such grids (count, then fill at the scanned offsets).
//
// One thread per target point.  All arithmetic is float64 with separate multiplies and adds
// (the library is compiled with -fmad=false), in the order of the numpy restatement
// oracle/matrix.py::bilinear_matrix, so weights (rounded to float32 at the end) and column
// indices are bitwise those of the scipy-built matrix.
#include "common.cuh"

namespace at {

// numpy's float remainder (npy_divmod): fmod, then the sign of the divisor.
__device__ __forceinline__ double np_mod(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) {
        if ((b < 0.0) != (m < 0.0)) m += b;
    } else {
        m = copysign(0.0, b);
    }
    return m;
}

// Stable insertion sort of N (column, weight) pairs by column, in registers
// (numpy argsort(kind="stable")).
template <int N, typename C>
__device__ __forceinline__ void sort_by_column(C (&c)[N], double (&w)[N]) {
#pragma unroll
    for (int a = 1; a < N; ++a) {
#pragma unroll
        for (int b = a; b > 0; --b) {
            if (c[b - 1] > c[b]) {
                const C tc = c[b];
                c[b] = c[b - 1];
                c[b - 1] = tc;
                const double tw = w[b];
                w[b] = w[b - 1];
                w[b - 1] = tw;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
    bilinear_matrix_kernel(double lat0, double dlat, long long n_lat, double lon0, double dlon, long long n_lon,
                           const double* __restrict__ tlat, const double* __restrict__ tlon, long long n,
                           float* __restrict__ data, int* __restrict__ indices) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const double fy = (tlat[t] - lat0) / dlat;
    long long j = static_cast<long long>(floor(fy));
    j = j < 0 ? 0 : (j > n_lat - 2 ? n_lat - 2 : j);
    const double wy = fy - static_cast<double>(j);
    const double fx = np_mod(tlon[t] - lon0, 360.0) / dlon;
    long long i0 = static_cast<long long>(floor(fx));
    const double wx = fx - static_cast<double>(i0);
    i0 %= n_lon;
    const long long i1 = (i0 + 1) % n_lon;
    long long c[4] = {j * n_lon + i0, j * n_lon + i1, (j + 1) * n_lon + i0, (j + 1) * n_lon + i1};
    double w[4] = {(1.0 - wy) * (1.0 - wx), (1.0 - wy) * wx, wy * (1.0 - wx), wy * wx};
    sort_by_column(c, w);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        data[4 * t + a] = static_cast<float>(w[a]);
        indices[4 * t + a] = static_cast<int>(c[a]);
    }
}

// Structured-grid stencils, oracle/structured_matrix.py::structured_matrix.  Row tables north -> south.
// The stencil's rows are j, j+1 (S = 2) or j-1 .. j+2 (S = 4), j = the last row with latitude
// >= the target's (-1 north of every row); a row index beyond either end is that end's rows
// seen across the pole (latitude +-180 - lat_k, longitudes shifted by 180 degrees), the pole
// row itself not repeated.  Cubic Lagrange weights on points i-1 .. i+2 at offset t:
//   -t(t-1)(t-2)/6, (t+1)(t-1)(t-2)/2, -(t+1)t(t-2)/2, (t+1)t(t-1)/6
// (exactly 0 and 1 at t = 0); in latitude on the four rows' own latitudes.
template <int S>
__global__ void __launch_bounds__(256)
    structured_matrix_kernel(const double* __restrict__ row_lat, const double* __restrict__ row_lon0,
                             const int64_t* __restrict__ row_first, const int64_t* __restrict__ row_count,
                             int n_rows, const double* __restrict__ tlat, const double* __restrict__ tlon,
                             long long n, float* __restrict__ data, int* __restrict__ indices) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const double phi = tlat[t];
    const double lam = tlon[t];
    int lo = 0, hi = n_rows;  // number of rows with latitude >= phi (a prefix: latitudes descend)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (row_lat[mid] >= phi) lo = mid + 1;
        else hi = mid;
    }
    const int j = lo - 1;
    const int north_pole = row_lat[0] == 90.0 ? 1 : 0;
    const int south_pole = row_lat[n_rows - 1] == -90.0 ? 1 : 0;

    double y[S], lon0[S];
    int first[S], count[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int v = j + s - (S / 2 - 1);  // virtual row index
        int k = v < 0 ? -v - 1 + north_pole : (v >= n_rows ? 2 * n_rows - 1 - v - south_pole : v);
        k = k < 0 ? 0 : (k > n_rows - 1 ? n_rows - 1 : k);
        const double lat_k = row_lat[k];
        const double lon_k = row_lon0[k];
        y[s] = v < 0 ? 180.0 - lat_k : (v >= n_rows ? -180.0 - lat_k : lat_k);
        lon0[s] = (v < 0 || v >= n_rows) ? lon_k + 180.0 : lon_k;
        first[s] = static_cast<int>(row_first[k]);
        count[s] = static_cast<int>(row_count[k]);
    }

    double wlat[S];
    if constexpr (S == 2) {
        const double ty = (y[0] - phi) / (y[0] - y[1]);
        wlat[0] = 1.0 - ty;
        wlat[1] = ty;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double l = 1.0;
            bool started = false;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                if (m == k) continue;
                const double f = (phi - y[m]) / (y[k] - y[m]);
                l = started ? l * f : f;
                started = true;
            }
            wlat[k] = l;
        }
    }

    int c[S * S];
    double w[S * S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const long long nr = count[s];
        const double x = np_mod(lam - lon0[s], 360.0) / (360.0 / static_cast<double>(nr));
        const double fi = floor(x);
        const double tx = x - fi;
        const long long i = static_cast<long long>(fi) % nr;
        double wlon[S];
        if constexpr (S == 2) {
            wlon[0] = 1.0 - tx;
            wlon[1] = tx;
        } else {
            const double tp1 = tx + 1.0, tm1 = tx - 1.0, tm2 = tx - 2.0;
            wlon[0] = tx * tm1 * tm2 / -6.0;
            wlon[1] = tp1 * tm1 * tm2 / 2.0;
            wlon[2] = tp1 * tx * tm2 / -2.0;
            wlon[3] = tp1 * tx * tm1 / 6.0;
        }
#pragma unroll
        for (int p = 0; p < S; ++p) {
            const long long o = p - (S / 2 - 1);
            c[S * s + p] = first[s] + static_cast<int>((i + o + nr) % nr);
            w[S * s + p] = wlat[s] * wlon[p];
        }
    }
    sort_by_column(c, w);
#pragma unroll
    for (int a = 0; a < S * S; ++a) {
        data[S * S * t + a] = static_cast<float>(w[a]);
        indices[S * S * t + a] = c[a];
    }
}

// First-order conservative (area-weighted grid-box average) weights between two global
// structured grids, oracle/conservative_matrix.py::conservative_matrix.  A grid's boxes are a
// latitude band times a longitude interval: row k spans z = sin(latitude) in [zs[k], zn[k]]
// (edges halfway between row latitudes, +-90 at the ends; the host computes the sines, the
// device only compares and subtracts them) and its point i covers
// [lon0 + (i - 1/2) d, lon0 + (i + 1/2) d), d = 360 / n.  The overlap of two boxes is a product
// of intervals, so a target's weights are (dz / dz_T) * (piece / wc) over the source cells its
// interval touches, measured in source-cell units.
struct BoxRows {
    const double* zn;       // north edge, z = sin(latitude)
    const double* zs;       // south edge
    const double* lon0;     // longitude of the row's first point
    const int64_t* first;   // index of the row's first point as stored
    const int64_t* count;   // points in the row
    int n;                  // rows
};

// Length of source cell c inside [x, end), in cell units.
__device__ __forceinline__ double cell_piece(double x, double end, long long c) {
    const double c0 = static_cast<double>(c);
    const double hi = end < c0 + 1.0 ? end : c0 + 1.0;
    const double lo = x > c0 ? x : c0;
    return hi - lo;
}

// Calls emit(column, weight) for target t's entries in ascending column order.  The source
// table runs north -> south; the target table is in storage order (row_first ascending) so
// that a target finds its row by binary search.  Both kernels below walk the overlaps through
// this one function, so the count and the fill agree by construction.
template <class Emit>
__device__ __forceinline__ void conservative_visit(const BoxRows& src, const BoxRows& tgt, long long t, Emit&& emit) {
    int lo = 0, hi = tgt.n;  // rows whose first point is <= t
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tgt.first[mid] <= t) lo = mid + 1;
        else hi = mid;
    }
    const int r = lo - 1;
    const double zn_t = tgt.zn[r], zs_t = tgt.zs[r];
    const double dz_t = zn_t - zs_t;
    const long long n_t = tgt.count[r];
    const double d_t = 360.0 / static_cast<double>(n_t);
    const double start = tgt.lon0[r] + (static_cast<double>(t - tgt.first[r]) - 0.5) * d_t;

    // source rows k0 .. k1 overlap the band: zs[k] < zn_t and zn[k] > zs_t (both edges descend)
    lo = 0, hi = src.n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (src.zs[mid] >= zn_t) lo = mid + 1;
        else hi = mid;
    }
    const int k0 = lo;
    lo = k0, hi = src.n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (src.zn[mid] > zs_t) lo = mid + 1;
        else hi = mid;
    }
    const int k1 = lo - 1;
    // walk the rows in ascending row_first, so the columns ascend across rows
    const bool stored_north_first = src.first[0] < src.first[src.n - 1];
    for (int q = 0; q <= k1 - k0; ++q) {
        const int k = stored_north_first ? k0 + q : k1 - q;
        const double zn_s = src.zn[k], zs_s = src.zs[k];
        const double dz = (zn_t < zn_s ? zn_t : zn_s) - (zs_t > zs_s ? zs_t : zs_s);
        if (!(dz > 0.0)) continue;
        const long long n = src.count[k];
        const double nd = static_cast<double>(n);
        const double d_s = 360.0 / nd;
        double x = np_mod(start - (src.lon0[k] - d_s / 2.0), 360.0) / d_s;
        if (x >= nd) x = x - nd;  // a remainder rounded up to 360 is cell 0
        const double wc = nd / static_cast<double>(n_t);
        const double end = x + wc;
        const double a = dz / dz_t;
        const long long i0 = static_cast<long long>(floor(x));
        const long long last = static_cast<long long>(ceil(end)) - 1;
        // n + 1 cells touched: the first and the last are the same point, one entry
        const bool merge = last - i0 == n;
        const long long base = src.first[k];
        // cells at or past n wrap onto columns c - n: that run holds the lower columns
        for (long long c = i0 > n ? i0 : n; c <= last; ++c) {
            double p = cell_piece(x, end, c);
            if (merge && c == last) p = p + cell_piece(x, end, i0);
            if (p >= 1e-9) emit(base + c - n, a * (p / wc));
        }
        for (long long c = merge ? i0 + 1 : i0; c <= last && c < n; ++c) {
            const double p = cell_piece(x, end, c);
            if (p >= 1e-9) emit(base + c, a * (p / wc));
        }
    }
}

__global__ void __launch_bounds__(256)
    conservative_count_kernel(BoxRows src, BoxRows tgt, long long n, int* __restrict__ counts) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int nnz = 0;
    conservative_visit(src, tgt, t, [&](long long, double) { ++nnz; });
    counts[t] = nnz;
}

__global__ void __launch_bounds__(256)
    conservative_fill_kernel(BoxRows src, BoxRows tgt, long long n, const int* __restrict__ indptr,
                             float* __restrict__ data, int* __restrict__ indices) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int o = indptr[t];
    conservative_visit(src, tgt, t, [&](long long col, double w) {
        data[o] = static_cast<float>(w);
        indices[o] = static_cast<int>(col);
        ++o;
    });
}

}  // namespace at

using namespace at;

extern "C" int at_bilinear_matrix(double lat0, double dlat, int64_t n_lat, double lon0, double dlon, int64_t n_lon,
                                  const double* tgt_lat, const double* tgt_lon, int64_t n_tgt, float* data_out,
                                  int32_t* indices_out, void* stream) {
    AT_REQUIRE(n_lat >= 2 && n_lon >= 1 && dlat != 0.0 && dlon > 0.0, "at_bilinear_matrix: bad source grid");
    AT_REQUIRE(n_lat * n_lon < (1ll << 31), "at_bilinear_matrix: source grid too large for int32 columns");
    AT_REQUIRE(n_tgt >= 0 && 4 * n_tgt < (1ll << 31), "at_bilinear_matrix: bad target count");
    if (n_tgt == 0) return AT_OK;
    AT_REQUIRE(tgt_lat != nullptr && tgt_lon != nullptr && data_out != nullptr && indices_out != nullptr,
               "at_bilinear_matrix: null argument");
    const int64_t blocks = (n_tgt + 255) / 256;
    bilinear_matrix_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
        lat0, dlat, n_lat, lon0, dlon, n_lon, tgt_lat, tgt_lon, n_tgt, data_out, indices_out);
    AT_LAUNCH_CHECK("bilinear_matrix_kernel");
    return AT_OK;
}

extern "C" int at_structured_matrix(const double* row_lat, const double* row_lon0, const int64_t* row_first,
                                    const int64_t* row_count, int64_t n_rows, int64_t n_src, int32_t stencil,
                                    const double* tgt_lat, const double* tgt_lon, int64_t n_tgt, float* data_out,
                                    int32_t* indices_out, void* stream) {
    AT_REQUIRE(stencil == 2 || stencil == 4, "at_structured_matrix: stencil must be 2 or 4, not %d", stencil);
    AT_REQUIRE(n_rows >= 2 && n_rows >= stencil && n_rows < (1ll << 31),
               "at_structured_matrix: a %d-row stencil needs at least %d rows (got %lld)", stencil,
               stencil, static_cast<long long>(n_rows));
    AT_REQUIRE(n_src >= 1 && n_src < (1ll << 31), "at_structured_matrix: %lld source points do not fit int32 columns",
               static_cast<long long>(n_src));
    AT_REQUIRE(n_tgt >= 0 && n_tgt <= ((1ll << 31) - 1) / (stencil * stencil),
               "at_structured_matrix: %lld targets x %d entries do not fit int32 offsets",
               static_cast<long long>(n_tgt), stencil * stencil);
    AT_REQUIRE(row_lat != nullptr && row_lon0 != nullptr && row_first != nullptr && row_count != nullptr,
               "at_structured_matrix: null row table");
    if (n_tgt == 0) return AT_OK;
    AT_REQUIRE(tgt_lat != nullptr && tgt_lon != nullptr && data_out != nullptr && indices_out != nullptr,
               "at_structured_matrix: null argument");
    const unsigned blocks = static_cast<unsigned>((n_tgt + 255) / 256);
    const int rows = static_cast<int>(n_rows);
    cudaStream_t st = as_stream(stream);
    if (stencil == 2) {
        structured_matrix_kernel<2><<<blocks, 256, 0, st>>>(row_lat, row_lon0, row_first, row_count, rows, tgt_lat,
                                                             tgt_lon, n_tgt, data_out, indices_out);
        AT_LAUNCH_CHECK("structured_matrix_kernel<2>");
    } else {
        structured_matrix_kernel<4><<<blocks, 256, 0, st>>>(row_lat, row_lon0, row_first, row_count, rows, tgt_lat,
                                                             tgt_lon, n_tgt, data_out, indices_out);
        AT_LAUNCH_CHECK("structured_matrix_kernel<4>");
    }
    return AT_OK;
}

// The two conservative entries share their grid arguments and checks.
static int conservative_rows(const char* who, const double* zn, const double* zs, const double* lon0,
                             const int64_t* first, const int64_t* count, int64_t n_rows, int64_t n_points,
                             const char* grid, BoxRows* out) {
    AT_REQUIRE(n_rows >= 2 && n_rows <= n_points, "%s: the %s grid needs at least 2 rows and no more rows than points (got %lld rows)",
               who, grid, static_cast<long long>(n_rows));
    AT_REQUIRE(n_points < (1ll << 31), "%s: %lld %s points do not fit int32", who, static_cast<long long>(n_points), grid);
    AT_REQUIRE(zn != nullptr && zs != nullptr && lon0 != nullptr && first != nullptr && count != nullptr,
               "%s: null %s row table", who, grid);
    *out = BoxRows{zn, zs, lon0, first, count, static_cast<int>(n_rows)};
    return AT_OK;
}

extern "C" int at_conservative_matrix_count(const double* src_zn, const double* src_zs, const double* src_lon0,
                                            const int64_t* src_first, const int64_t* src_count, int64_t n_src_rows,
                                            int64_t n_src, const double* tgt_zn, const double* tgt_zs,
                                            const double* tgt_lon0, const int64_t* tgt_first, const int64_t* tgt_count,
                                            int64_t n_tgt_rows, int64_t n_tgt, int32_t* counts_out, void* stream) {
    const char* who = "at_conservative_matrix_count";
    BoxRows src, tgt;
    int rc = conservative_rows(who, src_zn, src_zs, src_lon0, src_first, src_count, n_src_rows, n_src, "source", &src);
    if (rc != AT_OK) return rc;
    rc = conservative_rows(who, tgt_zn, tgt_zs, tgt_lon0, tgt_first, tgt_count, n_tgt_rows, n_tgt, "target", &tgt);
    if (rc != AT_OK) return rc;
    AT_REQUIRE(counts_out != nullptr, "%s: null counts", who);
    conservative_count_kernel<<<static_cast<unsigned>((n_tgt + 255) / 256), 256, 0, as_stream(stream)>>>(src, tgt, n_tgt,
                                                                                                       counts_out);
    AT_LAUNCH_CHECK("conservative_count_kernel");
    return AT_OK;
}

extern "C" int at_conservative_matrix_fill(const double* src_zn, const double* src_zs, const double* src_lon0,
                                           const int64_t* src_first, const int64_t* src_count, int64_t n_src_rows,
                                           int64_t n_src, const double* tgt_zn, const double* tgt_zs,
                                           const double* tgt_lon0, const int64_t* tgt_first, const int64_t* tgt_count,
                                           int64_t n_tgt_rows, int64_t n_tgt, const int32_t* indptr, int64_t nnz,
                                           float* data_out, int32_t* indices_out, void* stream) {
    const char* who = "at_conservative_matrix_fill";
    BoxRows src, tgt;
    int rc = conservative_rows(who, src_zn, src_zs, src_lon0, src_first, src_count, n_src_rows, n_src, "source", &src);
    if (rc != AT_OK) return rc;
    rc = conservative_rows(who, tgt_zn, tgt_zs, tgt_lon0, tgt_first, tgt_count, n_tgt_rows, n_tgt, "target", &tgt);
    if (rc != AT_OK) return rc;
    AT_REQUIRE(nnz >= 0 && nnz < (1ll << 31), "%s: %lld entries do not fit int32 offsets", who, static_cast<long long>(nnz));
    AT_REQUIRE(indptr != nullptr && ((data_out != nullptr && indices_out != nullptr) || nnz == 0), "%s: null argument", who);
    conservative_fill_kernel<<<static_cast<unsigned>((n_tgt + 255) / 256), 256, 0, as_stream(stream)>>>(
        src, tgt, n_tgt, indptr, data_out, indices_out);
    AT_LAUNCH_CHECK("conservative_fill_kernel");
    return AT_OK;
}

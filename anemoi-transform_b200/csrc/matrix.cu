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

// ---------------------------------------------------------------------------- HEALPix ---
// HEALPix grids (Gorski et al. 2005) and pixel-exact conservative weights between a HEALPix
// grid and a HEALPix or global structured grid, oracle/healpix_conservative.py.  All geometry
// is in the plane of the HEALPix projection (Calabretta & Roukema 2007), scaled by 4/pi:
// X = longitude / 45 degrees in [0, 8) (periodic), Y in [-2, 2].  The projection is
// equal-area, so areas in this plane are proportional to areas on the sphere.  In it
//   - parallels are horizontal: Y = 1.5 z for |z| <= 2/3, +-(2 - s) in the caps,
//     s = sqrt(3 (1 - |z|));
//   - a meridian is X = Phi in the equatorial zone and X = Xc + (Phi - Xc) s inside the
//     polar facet k (Phi in [2k, 2k + 2], Xc = 2k + 1), a line through the facet's apex;
//   - pixel p of ring i (1 .. 4n - 1) at nside n is the diamond with centre
//     (xnum / n, (2n - i) / n) and half-diagonal 1 / n, area 2 / n^2 (xnum an integer below);
//   - a structured box (z in [zs, zn], longitude interval) is cut at Y = +-1 and, in the caps,
//     at the facet meridians Phi = 2k into convex pieces: rectangles in the equatorial zone,
//     trapezoids (a triangle at the pole) in the caps; its area is 1.5 dz dPhi = 12 dz / count.
// An overlap is a Sutherland-Hodgman clip of two convex polygons and a shoelace area, in
// coordinates relative to the target's centre.  float64, unfused, rounded to float32 last.
struct HpGrid {
    long long nside;  // > 0: HEALPix; 0: structured (rows)
    int nested;       // HEALPix pixel order: 1 nested, 0 ring
    BoxRows rows;     // structured: rows north -> south (source) or in storage order (target)
};

struct Poly {
    int n;
    double x[4], y[4];
};

__device__ __forceinline__ long long hp_isqrt(long long v) {
    long long r = static_cast<long long>(sqrt(static_cast<double>(v)));
    while (r * r > v) --r;
    while ((r + 1) * (r + 1) <= v) ++r;
    return r;
}

__device__ __forceinline__ long long floor_div(long long a, long long b) {
    const long long q = a / b;
    return (a % b != 0 && (a < 0) != (b < 0)) ? q - 1 : q;
}

__device__ __forceinline__ long long floor_mod(long long a, long long b) { return a - floor_div(a, b) * b; }

// Ring pixel r -> ring i (1 .. 4n - 1) and position p in the ring.
__device__ __forceinline__ void hp_ring_of(long long n, long long r, long long& i, long long& p) {
    const long long ncap = 2 * n * (n - 1), npix = 12 * n * n;
    if (r < ncap) {
        i = (1 + hp_isqrt(1 + 2 * r)) >> 1;
        p = r - 2 * i * (i - 1);
    } else if (r < npix - ncap) {
        const long long q = r - ncap;
        i = q / (4 * n) + n;
        p = q % (4 * n);
    } else {
        const long long q = npix - r;
        const long long ir = (1 + hp_isqrt(2 * q - 1)) >> 1;
        i = 4 * n - ir;
        p = 4 * ir - (q - 2 * ir * (ir - 1));
    }
}

// Pixels in ring i, index of its first pixel, and 1 / 0 for a polar-cap ring.
__device__ __forceinline__ long long hp_ring_size(long long n, long long i) {
    return i < n ? i : (i > 3 * n ? 4 * n - i : n);
}

__device__ __forceinline__ long long hp_ring_start(long long n, long long i) {
    if (i < n) return 2 * i * (i - 1);
    if (i <= 3 * n) return 2 * n * (n - 1) + (i - n) * 4 * n;
    const long long ir = 4 * n - i;
    return 12 * n * n - 2 * ir * (ir + 1);
}

// X numerator of pixel p' of ring i, p' unwrapped (any integer; p' + count is one turn east).
__device__ __forceinline__ long long hp_xnum(long long n, long long i, long long pp) {
    if (i < n || i > 3 * n) {
        const long long ir = i < n ? i : 4 * n - i;
        const long long k = floor_div(pp, ir);
        return (2 * k + 1) * n + 2 * (pp - k * ir) + 1 - ir;
    }
    return 2 * pp + ((i - n + 1) & 1);
}

__constant__ int kJrll[12] = {2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4};
__constant__ int kJpll[12] = {1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7};

__device__ __forceinline__ long long hp_spread(long long v) {  // bits of v to the even bits
    long long out = 0;
    for (int b = 0; b < 31; ++b) out |= ((v >> b) & 1ll) << (2 * b);
    return out;
}

__device__ __forceinline__ long long hp_compress(long long v) {  // even bits of v
    long long out = 0;
    for (int b = 0; b < 31; ++b) out |= ((v >> (2 * b)) & 1ll) << b;
    return out;
}

__device__ long long hp_nest2ring(long long n, long long pix) {
    const long long face = pix / (n * n), ipf = pix % (n * n);
    const long long ix = hp_compress(ipf), iy = hp_compress(ipf >> 1);
    const long long jr = kJrll[face] * n - ix - iy - 1;
    long long nr, start, kshift;
    if (jr < n) {
        nr = jr, start = 2 * jr * (jr - 1), kshift = 0;
    } else if (jr > 3 * n) {
        nr = 4 * n - jr, start = 12 * n * n - 2 * nr * (nr + 1), kshift = 0;
    } else {
        nr = n, start = 2 * n * (n - 1) + (jr - n) * 4 * n, kshift = (jr - n) & 1;
    }
    long long jp = (kJpll[face] * nr + ix - iy + 1 + kshift) / 2;
    if (jp > 4 * nr) jp -= 4 * nr;
    if (jp < 1) jp += 4 * nr;
    return start + jp - 1;
}

__device__ long long hp_ring2nest(long long n, long long pix) {
    long long i, p;
    hp_ring_of(n, pix, i, p);
    const long long iphi = p + 1;
    long long nr, kshift, face;
    if (i < n) {
        nr = i, kshift = 0, face = (iphi - 1) / nr;
    } else if (i <= 3 * n) {
        nr = n, kshift = (i + n) & 1;
        const long long tmp = i - n, ire = tmp + 1, irm = 2 * n + 1 - tmp;
        const long long ifm = (iphi - (ire >> 1) + n - 1) / n, ifp = (iphi - (irm >> 1) + n - 1) / n;
        face = ifp == ifm ? (ifp | 4) : (ifp < ifm ? ifp : ifm + 8);
    } else {
        nr = 4 * n - i, kshift = 0, face = (iphi - 1) / nr + 8;
    }
    const long long irt = i - (2 + (face >> 2)) * n + 1;
    long long ipt = 2 * iphi - kJpll[face] * nr - kshift - 1;
    if (ipt >= 2 * n) ipt -= 8 * n;
    const long long ix = (ipt - irt) >> 1, iy = (-ipt - irt) >> 1;
    return face * n * n + hp_spread(ix) + (hp_spread(iy) << 1);
}

// Y of a parallel z; z of a parallel Y.
__device__ __forceinline__ double hp_y_of_z(double z) {
    const double a = fabs(z);
    if (a <= 2.0 / 3.0) return 1.5 * z;
    const double y = 2.0 - sqrt(3.0 * (1.0 - a));
    return z < 0.0 ? -y : y;
}

__device__ __forceinline__ double hp_z_of_y(double y) {
    const double a = fabs(y);
    if (a <= 1.0) return y / 1.5;
    const double s = 2.0 - a;
    const double z = 1.0 - s * s / 3.0;
    return y < 0.0 ? -z : z;
}

// The diamond of pixel (i, p') at nside n, relative to (ox, oy).
__device__ __forceinline__ Poly hp_diamond(long long n, long long i, long long pp, double ox, double oy) {
    const double nd = static_cast<double>(n);
    const double x = static_cast<double>(hp_xnum(n, i, pp)) / nd - ox;
    const double y = static_cast<double>(2 * n - i) / nd - oy;
    const double h = 1.0 / nd;
    Poly d;
    d.n = 4;
    d.x[0] = x, d.y[0] = y - h;
    d.x[1] = x + h, d.y[1] = y;
    d.x[2] = x, d.y[2] = y + h;
    d.x[3] = x - h, d.y[3] = y;
    return d;
}

// Calls f(piece) for the convex pieces of the box Y in [ya, yb], Phi in [fa, fb] (Phi
// unwrapped), relative to (ox, oy): the equatorial rectangle, then the cap pieces facet by facet.
template <class F>
__device__ __forceinline__ void box_pieces(double ya, double yb, double fa, double fb, double ox, double oy, F&& f) {
    const double y0 = ya > -1.0 ? ya : -1.0, y1 = yb < 1.0 ? yb : 1.0;
    if (y1 > y0) {
        Poly r;
        r.n = 4;
        r.x[0] = fa - ox, r.y[0] = y0 - oy;
        r.x[1] = fb - ox, r.y[1] = y0 - oy;
        r.x[2] = fb - ox, r.y[2] = y1 - oy;
        r.x[3] = fa - ox, r.y[3] = y1 - oy;
        f(r);
    }
    for (int cap = 0; cap < 2; ++cap) {
        const double c0 = cap == 0 ? (ya > 1.0 ? ya : 1.0) : ya;
        const double c1 = cap == 0 ? yb : (yb < -1.0 ? yb : -1.0);
        if (!(c1 > c0)) continue;
        const double s0 = 2.0 - fabs(c0), s1 = 2.0 - fabs(c1);
        for (long long k = static_cast<long long>(floor(fa / 2.0)); 2.0 * static_cast<double>(k) < fb; ++k) {
            const double e0 = 2.0 * static_cast<double>(k);
            const double g0 = fa > e0 ? fa : e0, g1 = fb < e0 + 2.0 ? fb : e0 + 2.0;
            if (!(g1 > g0)) continue;
            const double xc = e0 + 1.0;
            Poly t;
            t.n = 0;
            t.x[t.n] = xc + (g0 - xc) * s0 - ox, t.y[t.n++] = c0 - oy;
            if (s0 != 0.0) t.x[t.n] = xc + (g1 - xc) * s0 - ox, t.y[t.n++] = c0 - oy;
            t.x[t.n] = xc + (g1 - xc) * s1 - ox, t.y[t.n++] = c1 - oy;
            if (s1 != 0.0) t.x[t.n] = xc + (g0 - xc) * s1 - ox, t.y[t.n++] = c1 - oy;
            f(t);
        }
    }
}

// Area of the convex polygons a and b's intersection (both counter-clockwise): a clipped by
// each edge of b, then the shoelace formula.
__device__ double clip_area(const Poly& a, const Poly& b) {
    double px[12], py[12], qx[12], qy[12];
    int m = a.n;
    for (int v = 0; v < m; ++v) px[v] = a.x[v], py[v] = a.y[v];
    for (int e = 0; e < b.n && m > 0; ++e) {
        const double ex = b.x[e], ey = b.y[e];
        const int e1 = e + 1 == b.n ? 0 : e + 1;
        const double dx = b.x[e1] - ex, dy = b.y[e1] - ey;
        int k = 0;
        for (int v = 0; v < m; ++v) {
            const int w = v + 1 == m ? 0 : v + 1;
            const double sp = dx * (py[v] - ey) - dy * (px[v] - ex);
            const double sq = dx * (py[w] - ey) - dy * (px[w] - ex);
            if (sp >= 0.0 && k < 12) qx[k] = px[v], qy[k] = py[v], ++k;
            if (((sp > 0.0 && sq < 0.0) || (sp < 0.0 && sq > 0.0)) && k < 12) {
                const double t = sp / (sp - sq);
                qx[k] = px[v] + (px[w] - px[v]) * t, qy[k] = py[v] + (py[w] - py[v]) * t, ++k;
            }
        }
        m = k;
        for (int v = 0; v < m; ++v) px[v] = qx[v], py[v] = qy[v];
    }
    double s = 0.0;
    for (int v = 0; v < m; ++v) {
        const int w = v + 1 == m ? 0 : v + 1;
        s = s + (px[v] * py[w] - px[w] * py[v]);
    }
    return 0.5 * s;
}

// Calls visit(c, pp) for the columns c (0 .. count - 1) of the unwrapped range [pa, pb] in
// ascending order (the run wrapped past count first), once per unwrapped index pp == c
// (mod count): a range longer than count meets a column twice, once at each end.
template <class V>
__device__ __forceinline__ void unwrapped_runs(long long pa, long long pb, long long count, V&& visit) {
    if (pb < pa) return;
    const long long len = pb - pa + 1, a = floor_mod(pa, count);
    auto one = [&](long long c) {
        for (long long pp = pa + floor_mod(c - a, count); pp <= pb; pp += count) visit(c, pp);
    };
    if (len >= count) {
        for (long long c = 0; c < count; ++c) one(c);
        return;
    }
    for (long long c = 0; c <= a + len - 1 - count; ++c) one(c);
    for (long long c = a; c < count && c <= a + len - 1; ++c) one(c);
}

// Calls emit(column, weight) for target t's entries: ring-ordered source columns ascending for
// a HEALPix source (the caller maps and sorts a nested one), storage order for a structured
// source.  Count and fill both walk this one function.
template <class Emit>
__device__ __forceinline__ void healpix_visit(const HpGrid& src, const HpGrid& tgt, long long t, Emit&& emit) {
    // the target: a diamond, or a structured box cut into pieces
    long long ti = 0, tp = 0;
    double ya, yb, fa = 0.0, fb = 0.0, ox, oy, area_t;
    const long long tn = tgt.nside;
    if (tn > 0) {
        hp_ring_of(tn, tgt.nested ? hp_nest2ring(tn, t) : t, ti, tp);
        const double nd = static_cast<double>(tn);
        ox = static_cast<double>(hp_xnum(tn, ti, tp)) / nd;
        oy = static_cast<double>(2 * tn - ti) / nd;
        ya = oy - 1.0 / nd, yb = oy + 1.0 / nd;
        area_t = 2.0 / (nd * nd);
    } else {
        const BoxRows& tr = tgt.rows;
        int lo = 0, hi = tr.n;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (tr.first[mid] <= t) lo = mid + 1;
            else hi = mid;
        }
        const int r = lo - 1;
        const double cnt = static_cast<double>(tr.count[r]);
        const double d = 360.0 / cnt;
        const double start = tr.lon0[r] + (static_cast<double>(t - tr.first[r]) - 0.5) * d;
        fa = start / 45.0, fb = (start + d) / 45.0;
        ya = hp_y_of_z(tr.zs[r]), yb = hp_y_of_z(tr.zn[r]);
        ox = 0.5 * (fa + fb), oy = 0.5 * (ya + yb);
        area_t = 12.0 * (tr.zn[r] - tr.zs[r]) / cnt;
    }
    auto target_pieces = [&](auto&& f) {
        if (tn > 0) f(hp_diamond(tn, ti, tp, ox, oy));
        else box_pieces(ya, yb, fa, fb, ox, oy, f);
    };

    if (src.nside > 0) {
        const long long n = src.nside;
        const double nd = static_cast<double>(n), h = 1.0 / nd;
        const double area_s = 2.0 / (nd * nd);
        const double keep = 1e-9 * (area_s < area_t ? area_s : area_t);
        long long i0 = static_cast<long long>(floor((2.0 - yb) * nd));
        long long i1 = static_cast<long long>(ceil((2.0 - ya) * nd));
        i0 = i0 < 1 ? 1 : i0;
        i1 = i1 > 4 * n - 1 ? 4 * n - 1 : i1;
        for (long long i = i0; i <= i1; ++i) {
            const double yc = static_cast<double>(2 * n - i) / nd;
            // the X extent of the target's pieces that reach the ring's band
            double xlo = 0.0, xhi = 0.0;
            bool any = false;
            target_pieces([&](const Poly& q) {
                double qlo = q.y[0], qhi = q.y[0], plo = q.x[0], phi = q.x[0];
                for (int v = 1; v < q.n; ++v) {
                    qlo = q.y[v] < qlo ? q.y[v] : qlo, qhi = q.y[v] > qhi ? q.y[v] : qhi;
                    plo = q.x[v] < plo ? q.x[v] : plo, phi = q.x[v] > phi ? q.x[v] : phi;
                }
                if (!(qlo + oy < yc + h && qhi + oy > yc - h)) return;
                plo = plo + ox, phi = phi + ox;
                xlo = !any || plo < xlo ? plo : xlo, xhi = !any || phi > xhi ? phi : xhi;
                any = true;
            });
            if (!any) continue;
            const long long ir = hp_ring_size(n, i);
            long long pa, pb, count;
            if (i < n || i > 3 * n) {
                const long long ka = static_cast<long long>(floor(xlo / 2.0)), kb = static_cast<long long>(floor(xhi / 2.0));
                long long ja = static_cast<long long>(floor(((xlo - 2.0 * static_cast<double>(ka) - 1.0) * nd + static_cast<double>(ir) - 2.0) / 2.0));
                long long jb = static_cast<long long>(ceil(((xhi - 2.0 * static_cast<double>(kb) - 1.0) * nd + static_cast<double>(ir)) / 2.0));
                ja = ja < 0 ? 0 : (ja > ir ? ir : ja);
                jb = jb < -1 ? -1 : (jb > ir - 1 ? ir - 1 : jb);
                pa = ka * ir + ja, pb = kb * ir + jb, count = 4 * ir;
            } else {
                const double s = static_cast<double>((i - n + 1) & 1);
                pa = static_cast<long long>(floor((xlo * nd - 1.0 - s) / 2.0));
                pb = static_cast<long long>(ceil((xhi * nd + 1.0 - s) / 2.0));
                count = 4 * n;
            }
            const long long base = hp_ring_start(n, i);
            long long col = -1;
            double acc = 0.0;
            unwrapped_runs(pa, pb, count, [&](long long c, long long pp) {
                if (c != col) {
                    if (col >= 0 && acc >= keep) emit(base + col, acc / area_t);
                    col = c, acc = 0.0;
                }
                const Poly d = hp_diamond(n, i, pp, ox, oy);
                target_pieces([&](const Poly& q) { acc = acc + clip_area(d, q); });
            });
            if (col >= 0 && acc >= keep) emit(base + col, acc / area_t);
        }
        return;
    }

    // structured source, HEALPix target: the diamond's longitude range from its vertices
    const double nd = static_cast<double>(tn), h = 1.0 / nd;
    const double xf = 2.0 * floor(ox / 2.0) + 1.0;  // centre of the facet holding the diamond
    double plo = 0.0, phi = 0.0;
    for (int v = 0; v < 4; ++v) {
        const double vx = ox + (v == 1 ? h : (v == 3 ? -h : 0.0));
        const double vy = oy + (v == 0 ? -h : (v == 2 ? h : 0.0));
        double lo_v, hi_v;
        if (fabs(vy) <= 1.0) {
            lo_v = hi_v = vx;
        } else {
            const double s = 2.0 - fabs(vy);
            if (s == 0.0) lo_v = xf - 1.0, hi_v = xf + 1.0;
            else lo_v = hi_v = xf + (vx - xf) / s;
        }
        plo = v == 0 || lo_v < plo ? lo_v : plo;
        phi = v == 0 || hi_v > phi ? hi_v : phi;
    }
    const BoxRows& sr = src.rows;
    const double zlo = hp_z_of_y(ya), zhi = hp_z_of_y(yb);
    int lo = 0, hi = sr.n;  // rows k0 .. k1 overlap [zlo, zhi]
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sr.zs[mid] >= zhi) lo = mid + 1;
        else hi = mid;
    }
    const int k0 = lo;
    lo = k0, hi = sr.n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sr.zn[mid] > zlo) lo = mid + 1;
        else hi = mid;
    }
    const int k1 = lo - 1;
    const bool stored_north_first = sr.first[0] < sr.first[sr.n - 1];
    const double start = plo * 45.0, width = (phi - plo) * 45.0;
    for (int q = 0; q <= k1 - k0; ++q) {
        const int k = stored_north_first ? k0 + q : k1 - q;
        const long long n = sr.count[k];
        const double cnt = static_cast<double>(n);
        const double d = 360.0 / cnt;
        double x = np_mod(start - (sr.lon0[k] - d / 2.0), 360.0) / d;
        if (x >= cnt) x = x - cnt;
        const double shift = start - x * d;  // west edge of cell 0, in the diamond's frame
        const long long ca = static_cast<long long>(floor(x));
        const long long cb = static_cast<long long>(ceil(x + width / d)) - 1;
        const double by0 = hp_y_of_z(sr.zs[k]), by1 = hp_y_of_z(sr.zn[k]);
        const double area_s = 12.0 * (sr.zn[k] - sr.zs[k]) / cnt;
        const double keep = 1e-9 * (area_s < area_t ? area_s : area_t);
        const Poly dia = hp_diamond(tn, ti, tp, ox, oy);
        long long col = -1;
        double acc = 0.0;
        unwrapped_runs(ca, cb, n, [&](long long c, long long cc) {
            if (c != col) {
                if (col >= 0 && acc >= keep) emit(sr.first[k] + col, acc / area_t);
                col = c, acc = 0.0;
            }
            const double ga = (shift + static_cast<double>(cc) * d) / 45.0;
            const double gb = (shift + static_cast<double>(cc + 1) * d) / 45.0;
            box_pieces(by0, by1, ga, gb, ox, oy, [&](const Poly& b) { acc = acc + clip_area(b, dia); });
        });
        if (col >= 0 && acc >= keep) emit(sr.first[k] + col, acc / area_t);
    }
}

__global__ void __launch_bounds__(128)
    healpix_count_kernel(HpGrid src, HpGrid tgt, long long n, int* __restrict__ counts) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int nnz = 0;
    healpix_visit(src, tgt, t, [&](long long, double) { ++nnz; });
    counts[t] = nnz;
}

__global__ void __launch_bounds__(128)
    healpix_fill_kernel(HpGrid src, HpGrid tgt, long long n, const int* __restrict__ indptr,
                        float* __restrict__ data, int* __restrict__ indices) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int o = indptr[t];
    healpix_visit(src, tgt, t, [&](long long col, double w) {
        data[o] = static_cast<float>(w);
        indices[o] = static_cast<int>(col);
        ++o;
    });
}

__global__ void __launch_bounds__(256)
    healpix_reorder_kernel(long long nside, int to_nested, const int* __restrict__ in, long long n,
                           int* __restrict__ out) {
    const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const long long p = in[t];
    out[t] = static_cast<int>(to_nested ? hp_ring2nest(nside, p) : hp_nest2ring(nside, p));
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

// The HEALPix entries share their grid arguments and checks: nside > 0 is a HEALPix grid of
// 12 nside^2 points (ordering 0 ring, 1 nested, nested needing a power of two) and ignores the
// row tables; nside == 0 is a structured grid given by its row tables, as above.
static int healpix_side(const char* who, int64_t nside, int32_t ordering, const double* zn, const double* zs,
                        const double* lon0, const int64_t* first, const int64_t* count, int64_t n_rows,
                        int64_t n_points, const char* grid, HpGrid* out) {
    *out = HpGrid{};
    if (nside == 0) {
        out->nside = 0;
        return conservative_rows(who, zn, zs, lon0, first, count, n_rows, n_points, grid, &out->rows);
    }
    AT_REQUIRE(nside > 0 && 12 * nside * nside < (1ll << 31), "%s: the %s grid's nside %lld is not in 1 .. 13376",
               who, grid, static_cast<long long>(nside));
    AT_REQUIRE(ordering == 0 || ordering == 1, "%s: the %s grid's ordering must be 0 (ring) or 1 (nested), not %d",
               who, grid, ordering);
    AT_REQUIRE(ordering == 0 || (nside & (nside - 1)) == 0, "%s: nested order needs a power-of-two nside, the %s grid has %lld",
               who, grid, static_cast<long long>(nside));
    AT_REQUIRE(n_points == 12 * nside * nside, "%s: the %s grid has %lld points, nside %lld has %lld", who, grid,
               static_cast<long long>(n_points), static_cast<long long>(nside), static_cast<long long>(12 * nside * nside));
    out->nside = nside;
    out->nested = ordering;
    return AT_OK;
}

#define AT_HEALPIX_SIDES(who)                                                                                     \
    HpGrid src, tgt;                                                                                              \
    int rc = healpix_side(who, src_nside, src_ordering, src_zn, src_zs, src_lon0, src_first, src_count,           \
                          n_src_rows, n_src, "source", &src);                                                     \
    if (rc != AT_OK) return rc;                                                                                   \
    rc = healpix_side(who, tgt_nside, tgt_ordering, tgt_zn, tgt_zs, tgt_lon0, tgt_first, tgt_count, n_tgt_rows,   \
                      n_tgt, "target", &tgt);                                                                     \
    if (rc != AT_OK) return rc;                                                                                   \
    AT_REQUIRE(src.nside > 0 || tgt.nside > 0, "%s: at least one grid must be HEALPix", who)

extern "C" int at_healpix_conservative_count(int64_t src_nside, int32_t src_ordering, const double* src_zn,
                                             const double* src_zs, const double* src_lon0, const int64_t* src_first,
                                             const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                                             int64_t tgt_nside, int32_t tgt_ordering, const double* tgt_zn,
                                             const double* tgt_zs, const double* tgt_lon0, const int64_t* tgt_first,
                                             const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                                             int32_t* counts_out, void* stream) {
    const char* who = "at_healpix_conservative_count";
    AT_HEALPIX_SIDES(who);
    AT_REQUIRE(counts_out != nullptr, "%s: null counts", who);
    healpix_count_kernel<<<static_cast<unsigned>((n_tgt + 127) / 128), 128, 0, as_stream(stream)>>>(src, tgt, n_tgt,
                                                                                                 counts_out);
    AT_LAUNCH_CHECK("healpix_count_kernel");
    return AT_OK;
}

extern "C" int at_healpix_conservative_fill(int64_t src_nside, int32_t src_ordering, const double* src_zn,
                                            const double* src_zs, const double* src_lon0, const int64_t* src_first,
                                            const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                                            int64_t tgt_nside, int32_t tgt_ordering, const double* tgt_zn,
                                            const double* tgt_zs, const double* tgt_lon0, const int64_t* tgt_first,
                                            const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                                            const int32_t* indptr, int64_t nnz, float* data_out, int32_t* indices_out,
                                            void* stream) {
    const char* who = "at_healpix_conservative_fill";
    AT_HEALPIX_SIDES(who);
    AT_REQUIRE(nnz >= 0 && nnz < (1ll << 31), "%s: %lld entries do not fit int32 offsets", who, static_cast<long long>(nnz));
    AT_REQUIRE(indptr != nullptr && ((data_out != nullptr && indices_out != nullptr) || nnz == 0), "%s: null argument", who);
    healpix_fill_kernel<<<static_cast<unsigned>((n_tgt + 127) / 128), 128, 0, as_stream(stream)>>>(
        src, tgt, n_tgt, indptr, data_out, indices_out);
    AT_LAUNCH_CHECK("healpix_fill_kernel");
    return AT_OK;
}

extern "C" int at_healpix_reorder(int64_t nside, int32_t to_nested, const int32_t* in, int64_t n, int32_t* out,
                                  void* stream) {
    AT_REQUIRE(nside > 0 && (nside & (nside - 1)) == 0 && 12 * nside * nside < (1ll << 31),
               "at_healpix_reorder: nside %lld is not a power of two in 1 .. 8192", static_cast<long long>(nside));
    AT_REQUIRE(to_nested == 0 || to_nested == 1, "at_healpix_reorder: to_nested must be 0 or 1, not %d", to_nested);
    AT_REQUIRE(n >= 0 && n < (1ll << 31), "at_healpix_reorder: bad count %lld", static_cast<long long>(n));
    if (n == 0) return AT_OK;
    AT_REQUIRE(in != nullptr && out != nullptr, "at_healpix_reorder: null argument");
    healpix_reorder_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(nside, to_nested, in,
                                                                                                   n, out);
    AT_LAUNCH_CHECK("healpix_reorder_kernel");
    return AT_OK;
}

/*
 * at_b200.h — C-ABI of libat_b200.so: the B200 (sm_100a) field-transform hot path.
 *
 * This is the drop-in boundary of the regrid / spatial / pointwise path of
 * ecmwf/anemoi-transform (reference v0.4.2).  The reference is pure Python; its native
 * arithmetic lives in scipy.sparse (csr_matvec), scipy.spatial (cKDTree) and numpy ufuncs.
 * Every entry point below names the reference call site (file:line under
 * src/anemoi/transform/) whose native work it replaces.  The Python host side
 * (anemoi_transform_b200/_cabi.py) binds these with ctypes; see INTEGRATION.md for the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns an int status (AT_OK == 0); at_last_error() gives the message
 *     of the last failure on the calling thread;
 *   - "host" / "device" in a parameter comment says where the pointer must live;
 *   - device buffers are caller-owned (torch tensors on the Python side); the library
 *     allocates device memory only inside opaque handles (at_csr_t, at_epilogue_t,
 *     at_knn_t, at_pipeline_t, at_hostio_t), released by the matching *_destroy;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no torch / numpy types appear in any signature.
 */
#ifndef AT_B200_H
#define AT_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define AT_API __attribute__((visibility("default")))
#else
#define AT_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- status / dtypes --- */
#define AT_OK 0
#define AT_ERR_INVALID 1     /* bad argument (shape, alignment, dtype, null pointer)   */
#define AT_ERR_CUDA 2        /* a CUDA runtime call or a kernel launch failed          */
#define AT_ERR_NOMEM 3       /* device / host allocation failed                        */
#define AT_ERR_UNSUPPORTED 4 /* valid request outside what the kernels implement       */
#define AT_ERR_INDEX 5       /* an index was out of range (numpy would raise IndexError) */

#define AT_F32 0
#define AT_F64 1
#define AT_I32 0
#define AT_I64 1

typedef struct at_csr at_csr_t;
typedef struct at_epilogue at_epilogue_t;
typedef struct at_knn at_knn_t;
typedef struct at_pipeline at_pipeline_t;
typedef struct at_hostio at_hostio_t;
typedef struct at_hostio_group at_hostio_group_t;

AT_API const char* at_last_error(void);
AT_API int at_version(void);
/* Number of CUDA devices visible; fails (AT_ERR_CUDA) when there is no usable GPU. */
AT_API int at_device_count(int* count);
AT_API int at_set_device(int device);
/* Pin / unpin an existing host allocation so the async copies of at_pipeline_* overlap. */
/* Return the library's cached device blocks (handles and temporaries recycle their memory
 * instead of calling cudaMalloc / cudaFree every time; AT_B200_DEVICE_CACHE_MB caps the cache,
 * default 4096) to the driver. */
AT_API int at_device_cache_trim(void);
AT_API int at_host_register(void* ptr, size_t bytes);
AT_API int at_host_unregister(void* ptr);

/* ------------------------------------------------------------------ CSR matrix ------ */
/*
 * Stage a CSR interpolation matrix once in HBM.
 * Replaces: MIRMatrix.__init__  filters/fields/regrid.py:281-285
 *           (np.load(npz) -> scipy.sparse.csr_array((data, indices, indptr), shape)).
 * indptr/indices/data are HOST pointers in the dtypes the .npz stores
 * (make-regrid-file.py:150-160); indices are range-checked here.
 * nnz must be < 2^31 and n_cols < 2^31 (device copies are int32).
 */
AT_API int at_csr_create(int64_t n_rows, int64_t n_cols, int64_t nnz,
                  const void* indptr, int indptr_dtype,   /* host, AT_I32 | AT_I64, n_rows+1 */
                  const void* indices, int indices_dtype, /* host, AT_I32 | AT_I64, nnz      */
                  const void* data, int data_dtype,       /* host, AT_F32 | AT_F64, nnz      */
                  at_csr_t** out);
AT_API int at_csr_destroy(at_csr_t* csr);
/*
 * A copy of a staged matrix on another device, made device to device (the host arrays are not
 * read again): one matrix per device of an at_hostio_group_t that regrids the FieldList of one
 * RegridFilter.forward (regrid.py:174-208) over several GPUs.  The copy is independent of
 * `src` (either may be destroyed first).
 */
AT_API int at_csr_replicate(const at_csr_t* src, int device, at_csr_t** out);
/* uniform_nnz = k when every row has exactly k stored entries, else 0. */
AT_API int at_csr_info(const at_csr_t* csr, int64_t* n_rows, int64_t* n_cols, int64_t* nnz,
                int* uniform_nnz, int* data_dtype);

/*
 * Y[n_rows, n_fields] = A · X[n_cols, n_fields]   (point-major, row-major, ld in elements).
 * Replaces: MIRMatrix.__call__ `self.matrix @ data`  filters/fields/regrid.py:309-310
 *           (scipy.sparse._sparsetools csr_matvec), batched over fields.
 * Semantics are scipy's, bit for bit: per (row, field) the products are accumulated
 * sequentially in storage order, starting from +0, with separate multiply and add (no FMA);
 * explicit zeros are not skipped (0·NaN = NaN); an empty row gives 0.
 * Result dtype follows numpy: y_dtype must be F64 if the matrix or X is F64, else F32.
 * The f32·f32 fast path needs ldx, ldy multiples of 4 and 16-byte aligned X, Y.
 * A matrix staged on another device than the current one is refused (AT_ERR_INVALID), here and
 * in at_spmm_fused / at_hostio_regrid (whose engine's device counts).
 * spmm_variant: 0 = default tuning; other values select kernel shapes (see DESIGN.md).
 */
AT_API int at_spmm(const at_csr_t* csr,
            const void* X, int x_dtype, int64_t ldx, /* device */
            void* Y, int y_dtype, int64_t ldy,       /* device */
            int64_t n_fields, int spmm_variant, void* stream);

/*
 * at_spmm for fields with missing values.  A source value is missing when it is NaN (Inf is
 * not).  Per target row and field, Σ′ sums over the entries whose x is not NaN, sequentially in
 * storage order from +0 in the result dtype, multiply and add unfused:
 *   AT_MISSING_PROPAGATE  y = Σ w·x: exactly at_spmm (default tuning), which it calls.
 *   AT_MISSING_ALL        no entry missing: y = Σ w·x, bit for bit at_spmm.  Otherwise
 *                         y = Σ′ w·x / Σ′ w (IEEE division), NaN when every entry is missing
 *                         or Σ′ w is not > 0.
 *   AT_MISSING_HEAVIEST   as AT_MISSING_ALL, and NaN whenever the row's heaviest entry (largest
 *                         weight, the first in storage order on ties) is missing.
 * Dtypes, alignment and devices are checked as in at_spmm; an unknown policy is AT_ERR_INVALID.
 */
#define AT_MISSING_PROPAGATE 0
#define AT_MISSING_ALL 1
#define AT_MISSING_HEAVIEST 2
AT_API int at_spmm_missing(const at_csr_t* csr,
            const void* X, int x_dtype, int64_t ldx, /* device */
            void* Y, int y_dtype, int64_t ldy,       /* device */
            int64_t n_fields, int policy, void* stream);

/* ------------------------------------------------------------ fused epilogue -------- */
/*
 * A pointwise program over the columns of a point-major batch, fused into the SpMM
 * epilogue (at_spmm_fused) or run on its own (at_pointwise).  Columns are described in
 * segments; within a segment the kind is uniform and partner columns are adjacent.
 *
 *   AT_EPI_PLAIN     in (a)        -> out (a)             clip / mask only
 *   AT_EPI_UV2DDFF   in (u, v)     -> out (ws, wdir)      uv_to_ddff.py:77-101
 *   AT_EPI_DDFF2UV   in (ws, wdir) -> out (u, v)          uv_to_ddff.py:103-127
 *   AT_EPI_QT2R      in (q, t)     -> out (r)             q_to_r.py:69-73
 *   AT_EPI_QT2QTR    in (q, t)     -> out (q, t, r)       q_to_r.py:69-73, return_inputs="all"
 *   AT_EPI_RT2Q      in (r, t)     -> out (q)             q_to_r.py:75-81
 *   AT_EPI_RT2RTQ    in (r, t)     -> out (r, t, q)       q_to_r.py:75-81, return_inputs="all"
 *   AT_EPI_AFFINE    in (x)        -> out (x*pa + pb)     rescale.py:25-26   (Rescale / Convert forward)
 *   AT_EPI_AFFINE_INV in (x)       -> out ((x-pb)/pa)     rescale.py:28-29   (backward)
 *   AT_EPI_EXP       in (x)        -> out (exp x)         lnsp_to_sp.py:47-49
 *   AT_EPI_LOG       in (x)        -> out (log x)         lnsp_to_sp.py:65-67
 *   AT_EPI_IMPUTE_NAN in (x)       -> out (isnan x ? pa : x)  impute_nans.py:52-54
 *   AT_EPI_COSSIN    in (x)        -> out (cos(x*pa), sin(x*pa))   cos_sin_from_rad.py:78-79 (pa = 1),
 *                                                          cos_sin_mean_wave_direction.py:71-74 (pa = deg2rad(1))
 *   AT_EPI_ATAN2     in (c, s)     -> out (atan2(s, c)*pa), wrapped into [0, 360) when pb != 0
 *                                                          cos_sin_from_rad.py:100, cos_sin_mean_wave_direction.py:96-98
 *   AT_EPI_RT2D      in (r, t)     -> out (td)            dewpoint.py:62-67 (r == 0 -> 1e-4 first)
 *   AT_EPI_RT2RTD    in (r, t)     -> out (r, t, td)      dewpoint.py, return_inputs="all"
 *   AT_EPI_DT2R      in (td, t)    -> out (r)             dewpoint.py:69-74
 *   AT_EPI_DT2DTR    in (td, t)    -> out (td, t, r)      dewpoint.py, return_inputs="all"
 * pa / pb are per-segment constants (a filter instance applies one scale / offset / value to
 * every field it selects); on the float32 path they are rounded to float32 (NEP 50).
 *
 * After the kind's conversion every OUTPUT column c applies, in this order,
 *   clip:  np.clip(x, lo, hi) with NaN passing through     clipper.py:67-70
 *   mask:  x = NaN where row_mask[row] != 0                 apply_mask.py:184-185
 * as selected by cols[c].flags.
 */
#define AT_EPI_PLAIN 0
#define AT_EPI_UV2DDFF 1
#define AT_EPI_DDFF2UV 2
#define AT_EPI_QT2R 3
#define AT_EPI_QT2QTR 4
#define AT_EPI_RT2Q 5
#define AT_EPI_RT2RTQ 6
#define AT_EPI_AFFINE 7
#define AT_EPI_AFFINE_INV 8
#define AT_EPI_EXP 9
#define AT_EPI_LOG 10
#define AT_EPI_IMPUTE_NAN 11
#define AT_EPI_COSSIN 12
#define AT_EPI_ATAN2 13
#define AT_EPI_RT2D 14
#define AT_EPI_RT2RTD 15
#define AT_EPI_DT2R 16
#define AT_EPI_DT2DTR 17
#define AT_EPI_KIND_COUNT 18

#define AT_COL_CLIP_LO 1u /* lo is set  */
#define AT_COL_CLIP_HI 2u /* hi is set  */
#define AT_COL_MASK 4u    /* apply row_mask to this column */

typedef struct {
    int32_t kind;    /* AT_EPI_*                                                        */
    int32_t in_col;  /* first input column; multiple of 4                               */
    int32_t n_in;    /* input columns in the segment (even for pair kinds)              */
    int32_t out_col; /* first output column; multiple of 2 (of 4 for 1:1 and 1:2 kinds) */
    double pa, pb;   /* per-segment constants of the kind (see the table above)         */
} at_epi_segment_t;

typedef struct {
    double lo, hi;    /* clip bounds (used when the flag is set); rounded to float32 on
                         the float32 path, as numpy rounds Python scalars (NEP 50)      */
    double pressure;  /* Pa; read on the humidity OUTPUT column of QT / RT kinds        */
    uint32_t flags;   /* AT_COL_*                                                       */
    uint32_t reserved;
} at_epi_col_t;

/* segments / cols are HOST arrays; cols has n_out_cols entries indexed by output column. */
AT_API int at_epilogue_create(const at_epi_segment_t* segments, int32_t n_segments,
                       const at_epi_col_t* cols, int32_t n_out_cols, at_epilogue_t** out);
AT_API int at_epilogue_destroy(at_epilogue_t* epi);

/* Y = epilogue(A · X).  f32 only.  row_mask: device uint8[n_rows] or NULL. */
AT_API int at_spmm_fused(const at_csr_t* csr, const at_epilogue_t* epi,
                  const float* X, int64_t n_src /* rows of X; must equal the matrix's n_cols */,
                  int64_t ldx, float* Y, int64_t ldy,
                  const uint8_t* row_mask, void* stream);
/* Y = epilogue(X) on a resident batch of n_rows points (the standalone pointwise filters).
 * dtype AT_F32 | AT_F64 is the type of X and Y (numpy keeps the dtype of the field). */
AT_API int at_pointwise(const at_epilogue_t* epi, int64_t n_rows,
                 const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype,
                 const uint8_t* row_mask, void* stream);

/* Y[r, :] = epilogue(X[idx[r], :]) for r < n_out: the nearest-neighbour / masked regrid
 * (`data[..., idx]`, regrid.py:380, 420) fused with the pointwise filters after it.
 * idx: device int64[n_out], every entry in [0, n_src) (validated by the caller: a kNN result
 * or a checked mask); values are copied exactly, as numpy indexing does. */
AT_API int at_gather_pointwise(const at_epilogue_t* epi, const int64_t* idx, int64_t n_out, int64_t n_src,
                        const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype,
                        const uint8_t* row_mask, void* stream);

/* --------------------------------------------------------------- layout ------------- */
/*
 * dst[c, r] = src[r, c]: field-major [n_fields, n_points] <-> point-major
 * [n_points, n_fields] (the FieldList delivers one array per field: regrid.py:309).
 * elem_size 4 or 8.  ld in elements.
 */
AT_API int at_transpose(const void* src, int64_t rows, int64_t cols, int64_t ld_src,
                 void* dst, int64_t ld_dst, int elem_size, void* stream);
/*
 * Y[i, :] = X[idx[i], :]  for i < n_out — the nearest-neighbour / masked regrid gather.
 * Replaces: `data[..., self.nearest_grid_points]` regrid.py:380 and
 *           `data[..., self.mask]` regrid.py:420 (numpy fancy indexing).
 * idx: device int64[n_out]; an index outside [0, n_src) sets *err_flag (device int32,
 * may be NULL) to 1 and writes nothing for that row (numpy raises IndexError).
 */
AT_API int at_gather_rows(const int64_t* idx, int64_t n_out, int64_t n_src,
                   const void* X, int64_t ldx, void* Y, int64_t ldy,
                   int64_t n_fields, int elem_size, int32_t* err_flag, void* stream);
/* Y[r, j] = X[r, cols[j]] for j < n_out: regroup the fields of a resident batch so partner
 * fields (u with v, q with t — GroupByParam, grouping/__init__.py:93-137) sit in adjacent
 * columns.  cols: device int32[n_out], every entry < ldx.  elem_size 4 or 8. */
AT_API int at_gather_cols(const int32_t* cols, int32_t n_out, int64_t n_rows, const void* X, int64_t ldx,
                   void* Y, int64_t ldy, int elem_size, void* stream);
/* mask[i] = OP(values[i], threshold) — MaskVariable._compute_mask apply_mask.py:160-163.
 * op: 0 ==, 1 !=, 2 >, 3 >=, 4 <, 5 <=, 6 "is not NaN" (threshold unused; `~np.isnan(data)`,
 * remove_nans.py:103).  values: device f32 / f64 (dtype) with element
 * stride `stride`; a float32 array is compared in float32, as numpy does (NEP 50). */
AT_API int at_compare_mask(const void* values, int dtype, int64_t stride, int64_t n, int op,
                    double threshold, uint8_t* mask, void* stream);
/* Y[r, g] = ((X[r, cols[g*n_terms]] + X[r, cols[g*n_terms+1]]) + ...) for g < n_groups: the
 * `sum` filter's `s += c` over its params in field order (sum.py:109-115), one output column
 * per group.  cols: device int32[n_groups * n_terms].  dtype AT_F32 | AT_F64. */
AT_API int at_sum_cols(const int32_t* cols, int32_t n_groups, int32_t n_terms, int64_t n_rows,
                const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype, void* stream);
/* flags[j] |= 1 if any X[r, first_col + j] < lo, 2 if any > hi, 4 if any is NaN, for
 * j < n_cols: the range validation of cos_sin_from_rad.py:74-77 without a host round trip.
 * flags: device uint32[n_cols], zeroed by the caller. */
AT_API int at_range_flags(const void* X, int64_t ldx, int64_t n_rows, int32_t first_col, int32_t n_cols,
                   int dtype, double lo, double hi, uint32_t* flags, void* stream);

/* ------------------------------------------------ end-to-end host pipeline ----------- */
/*
 * Regrid host-resident fields through the GPU: chunked H2D -> pack -> SpMM -> unpack ->
 * D2H on three streams with double buffering.  This is the call a FieldList-in /
 * FieldList-out RegridFilter.forward makes (regrid.py:174-208), batched.
 * fields_in[f] : host float32[n_cols], fields_out[f] : host float32[n_rows]
 * (pinned memory lets the copies overlap; pageable memory still works).
 */
AT_API int at_pipeline_create(const at_csr_t* csr, int32_t chunk_fields, at_pipeline_t** out);
AT_API int at_pipeline_destroy(at_pipeline_t* p);
AT_API int at_pipeline_regrid(at_pipeline_t* p, const float* const* fields_in,
                       float* const* fields_out, int64_t n_fields);

/* ---------------------------------------------------------- matrix construction ------ */
/*
 * 4-point bilinear interpolation weights from a regular, longitude-periodic lat-lon grid
 * (row k at latitude lat0 + k*dlat, column i at longitude lon0 + i*dlon, point k*n_lon + i)
 * to n_tgt arbitrary points: row t of the CSR matrix has the four entries
 * data_out[4t..4t+3] / indices_out[4t..4t+3], sorted by column, explicit zeros kept
 * (indptr is 4*t).  Replaces, for this scheme, the external `mir` binary behind
 * `make-regrid-file` (commands/make-regrid-file.py:142-160) and earthkit-regrid's matrix
 * inventory (filters/fields/regrid.py:246-255).  float64 arithmetic, unfused, weights rounded
 * to float32 last: bitwise the numpy restatement oracle/matrix.py.  All pointers device.
 */
AT_API int at_bilinear_matrix(double lat0, double dlat, int64_t n_lat, double lon0, double dlon, int64_t n_lon,
                       const double* tgt_lat, const double* tgt_lon, int64_t n_tgt,
                       float* data_out, int32_t* indices_out, void* stream);

/*
 * Structured bilinear (stencil 2: 2 rows x 2 points, nnz 4 per target) or bicubic (stencil 4:
 * 4 rows x 4 points, cubic Lagrange in longitude on each row, then in latitude on the rows'
 * latitudes; nnz 16) interpolation weights from a global structured grid (octahedral and
 * classic reduced Gaussian, full Gaussian, regular lat-lon) to n_tgt arbitrary points.  The grid
 * is n_rows rows north to south: row r at latitude row_lat[r] (strictly decreasing) holds
 * row_count[r] points at row_lon0[r] + i*360/row_count[r], stored as source points
 * row_first[r] .. row_first[r] + row_count[r] - 1; n_src is the total number of source points.
 * Rows beyond the outermost rows are those rows seen across the pole (latitude +-180 - lat,
 * longitudes shifted by 180 degrees); a row on the pole itself is not repeated.  Row t of the
 * CSR matrix is data_out / indices_out[S*S*t .. S*S*t + S*S - 1] (indptr is S*S*t), sorted by
 * column (stable), explicit zeros and duplicate columns kept.  Target latitudes must lie in
 * [-90, 90].  Replaces, for these schemes, the external `mir` binary behind `make-regrid-file`
 * (commands/make-regrid-file.py:142-160) and earthkit-regrid's matrix inventory
 * (filters/fields/regrid.py:246-255).  float64 arithmetic, unfused, weights rounded to float32
 * last: bitwise the numpy restatement oracle/structured_matrix.py::structured_matrix.  All pointers device.
 */
AT_API int at_structured_matrix(const double* row_lat, const double* row_lon0, const int64_t* row_first,
                       const int64_t* row_count, int64_t n_rows, int64_t n_src, int32_t stencil,
                       const double* tgt_lat, const double* tgt_lon, int64_t n_tgt,
                       float* data_out, int32_t* indices_out, void* stream);

/*
 * First-order conservative (area-weighted grid-box average) weights from one global
 * structured grid to another, in two passes: at_conservative_matrix_count writes each target's
 * number of entries to counts_out[n_tgt]; the caller scans them into indptr[n_tgt + 1] (nnz =
 * indptr[n_tgt]) and at_conservative_matrix_fill writes row t at data_out / indices_out
 * [indptr[t] ..], columns ascending and unique.  Each grid is given as per-row tables: the
 * row's north and south edge as z = sin(latitude) (zn, zs), the longitude of its first point
 * (lon0), the index of that point as stored (first) and the row's point count (count), point i
 * covering [lon0 + (i - 1/2) 360/count, lon0 + (i + 1/2) 360/count).  The source tables run
 * north to south; the target tables run in storage order (first ascending).  n_src and n_tgt
 * are the grids' point counts.  Weight = (dz / dz_target) * (piece / width) with both
 * fractions in float64, unfused, rounded to float32 last; overlaps with dz <= 0 or shorter than
 * 1e-9 of a source cell are dropped.  Replaces, for this scheme, the external `mir` binary
 * behind `make-regrid-file` (commands/make-regrid-file.py:142-160) and earthkit-regrid's
 * matrix inventory (filters/fields/regrid.py:246-255).  Bitwise the numpy restatement
 * oracle/conservative_matrix.py::conservative_matrix.  All pointers device.
 */
AT_API int at_conservative_matrix_count(const double* src_zn, const double* src_zs, const double* src_lon0,
                       const int64_t* src_first, const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                       const double* tgt_zn, const double* tgt_zs, const double* tgt_lon0,
                       const int64_t* tgt_first, const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                       int32_t* counts_out, void* stream);
AT_API int at_conservative_matrix_fill(const double* src_zn, const double* src_zs, const double* src_lon0,
                       const int64_t* src_first, const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                       const double* tgt_zn, const double* tgt_zs, const double* tgt_lon0,
                       const int64_t* tgt_first, const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                       const int32_t* indptr, int64_t nnz, float* data_out, int32_t* indices_out, void* stream);

/*
 * First-order conservative weights between a HEALPix grid and a HEALPix or global structured
 * grid, with the true HEALPix pixels (`method="healpix-conservative"`), in the same two passes
 * as at_conservative_matrix_count / _fill.  Each side is either HEALPix, nside > 0 with
 * ordering 0 (ring) or 1 (nested, nside a power of two) and 12 nside^2 points (its row-table
 * pointers are ignored and may be NULL), or structured, nside == 0 with the row tables of
 * at_conservative_matrix_count (source rows north to south, target rows in storage order); at
 * least one side is HEALPix.  Overlaps are exact polygon areas in the plane of the HEALPix
 * projection: weight = area(source cell and target cell) / area(target cell), float64,
 * unfused, rounded to float32 last; overlaps under 1e-9 of the smaller cell are dropped.
 * Columns are unique and ascending, except that a nested HEALPix source comes out with the
 * ring-order columns (the caller maps them with at_healpix_reorder and sorts each row).
 * Replaces, for this scheme, the external `mir` binary behind `make-regrid-file`
 * (commands/make-regrid-file.py:142-160) and earthkit-regrid's matrix inventory
 * (filters/fields/regrid.py:246-255).  Bitwise the numpy restatement
 * oracle/healpix_conservative.py.  All pointers device.
 */
AT_API int at_healpix_conservative_count(int64_t src_nside, int32_t src_ordering, const double* src_zn,
                       const double* src_zs, const double* src_lon0, const int64_t* src_first,
                       const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                       int64_t tgt_nside, int32_t tgt_ordering, const double* tgt_zn,
                       const double* tgt_zs, const double* tgt_lon0, const int64_t* tgt_first,
                       const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                       int32_t* counts_out, void* stream);
AT_API int at_healpix_conservative_fill(int64_t src_nside, int32_t src_ordering, const double* src_zn,
                       const double* src_zs, const double* src_lon0, const int64_t* src_first,
                       const int64_t* src_count, int64_t n_src_rows, int64_t n_src,
                       int64_t tgt_nside, int32_t tgt_ordering, const double* tgt_zn,
                       const double* tgt_zs, const double* tgt_lon0, const int64_t* tgt_first,
                       const int64_t* tgt_count, int64_t n_tgt_rows, int64_t n_tgt,
                       const int32_t* indptr, int64_t nnz, float* data_out, int32_t* indices_out, void* stream);

/*
 * HEALPix pixel indices from ring to nested order (to_nested = 1) or back (0), for a
 * power-of-two nside: out[t] = the index of pixel in[t] in the other order.  Used to build a
 * nested grid's matrices in ring order and map their columns, where earthkit-regrid reads
 * `{"grid": "H<nside>", "ordering": "nested"}` gridspecs (filters/fields/regrid.py:246-255).
 * All pointers device; in and out may be the same array.
 */
AT_API int at_healpix_reorder(int64_t nside, int32_t to_nested, const int32_t* in, int64_t n, int32_t* out,
                       void* stream);

/* ------------------------------------------------ field I/O engine (FieldList <-> HBM) --- */
/*
 * A caching allocator of page-locked host memory.  The numpy arrays the drop-in filters hand
 * back to the caller (`field.to_numpy()` of a regridded field, regrid.py:312 wraps a fresh
 * array per field) are blocks of this pool, so the device-to-host DMA writes the final array.
 * Blocks are recycled by size; at_pinned_trim returns unused slabs to the system.
 * AT_B200_PINNED_LIMIT_MB caps the pool (default: half of the physical memory); beyond it
 * at_pinned_alloc fails with AT_ERR_NOMEM and callers fall back to pageable destinations.
 */
AT_API int at_pinned_alloc(size_t bytes, void** out);
/* n blocks of `bytes` each into out[0..n); all or nothing. */
AT_API int at_pinned_alloc_many(size_t bytes, int64_t n, void** out);
AT_API int at_pinned_free(void* ptr);
AT_API int at_pinned_trim(void);
AT_API int at_pinned_stats(size_t* bytes_in_use, size_t* bytes_reserved);

/*
 * The engine: worker threads (n_threads = 0: one per available core, at most 16, or
 * AT_B200_COPY_THREADS), three pinned + three device staging slots per direction, its own
 * copy / compute streams.  One engine per device and process is enough.
 */
AT_API int at_hostio_create(int32_t n_threads, at_hostio_t** out);
AT_API int at_hostio_destroy(at_hostio_t* io);
AT_API int at_hostio_threads(const at_hostio_t* io, int32_t* n_threads, int32_t* nontemporal_copies);
/*
 * d_pm[p, f] = fields[f][p]: upload n_fields host arrays of n_points elements (4 or 8 bytes)
 * into columns [0, n_fields) of a point-major device batch with leading dimension ld.
 * Replaces: the per-field `field.to_numpy(flatten=True)` hand-over of regrid.py:309 /
 * matching.py:242-246.  Pageable arrays are staged by the worker threads; page-locked ones
 * are read in place.  Device work is ordered on `stream`; the call returns when every input
 * byte has been consumed (the caller may reuse its arrays).
 */
AT_API int at_hostio_upload(at_hostio_t* io, const void* const* fields, int64_t n_fields, int64_t n_points,
                     int elem_size, void* d_pm, int64_t ld, void* stream);
/*
 * dst[f][p] = d_pm[p, f] for f < n_fields (after the work already queued on `stream`).
 * Page-locked destinations (at_pinned_alloc blocks): returns at once, *ticket identifies the
 * transfer; at_hostio_wait(ticket) blocks until the arrays are complete.  Pageable
 * destinations: complete on return, *ticket = -1.
 */
AT_API int at_hostio_download(at_hostio_t* io, const void* d_pm, int64_t ld, int64_t n_fields, int64_t n_points,
                       int elem_size, void* const* dst, void* stream, int64_t* ticket);
AT_API int at_hostio_wait(at_hostio_t* io, int64_t ticket);
/*
 * One RegridFilter.forward over host fields (regrid.py:174-208), streamed: chunks of fields
 * are staged, uploaded, packed, transformed and sent back while the next chunk is staged.
 *   op = AT_HOSTIO_SPMM    y = csr @ x            (MIRMatrix.__call__, regrid.py:309-310)
 *   op = AT_HOSTIO_GATHER  y = x[gather_idx]      (regrid.py:380, 420); gather_idx device
 *                          int64[n_out_points], every entry in [0, n_src)
 *   op = AT_HOSTIO_SPMM_MISSING_ALL / AT_HOSTIO_SPMM_MISSING_HEAVIEST
 *                          y = csr @ x skipping missing (NaN) sources: at_spmm_missing with
 *                          AT_MISSING_ALL / AT_MISSING_HEAVIEST
 * fields_in[f]: host x_dtype[n_src].  d_Y (optional): device [n_tgt, ldy] point-major batch
 * that keeps the results resident for the next filter; work on `consumer_stream` queued after
 * the call sees it complete.  fields_out (optional): host destinations of the result dtype
 * (numpy's result_type of matrix and field), filled behind *ticket as in at_hostio_download.
 * Returns when the inputs have been consumed.
 */
#define AT_HOSTIO_SPMM 0
#define AT_HOSTIO_GATHER 1
#define AT_HOSTIO_SPMM_MISSING_ALL 2
#define AT_HOSTIO_SPMM_MISSING_HEAVIEST 3
AT_API int at_hostio_regrid(at_hostio_t* io, int op, const at_csr_t* csr, const int64_t* gather_idx,
                     int64_t n_out_points, const void* const* fields_in, int64_t n_fields, int64_t n_src,
                     int x_dtype, void* d_Y, int64_t ldy, void* const* fields_out, void* consumer_stream,
                     int64_t* ticket);

/* ------------------------------------------------ GRIB simple packing on the device --- */
/*
 * A GRIB-backed FieldList reaches RegridFilter.forward as earthkit-data GribFields; the
 * per-field `field.to_numpy(flatten=True)` of regrid.py:309 (matching.py:242-246 for the
 * pointwise filters) is where ecCodes decodes each message to float64 on one CPU core.  These
 * entry points move the packed octets instead (2 bytes per point at 16 bits rather than 8 bytes
 * of float64) and decode them on the device:
 *     Y = ((X * 2^E) + R) * 10^-D        (WMO FM 92, regulation 92.9.4; float64, unfused)
 * Supported: editions 1 and 2, grid-point simple packing (BDS flag 0 / template 5.0),
 * 0..32 bits per value, ECMWF's long edition-1 messages, bitmaps (a point whose bit is clear
 * decodes to NaN, which is what earthkit-data's to_numpy() hands to the filters), and edition-2
 * CCSDS packing (template 5.42, libaec's AEC stream of the same X): block size 8/16/32/64,
 * reference sample interval 1..4096, with or without AEC_DATA_PREPROCESS (8) and AEC_PAD_RSI
 * (32); AEC_DATA_3BYTE (2) and AEC_DATA_MSB (4) do not change the stream.  CCSDS fields are
 * decoded on the device in two kernels (RSI offsets, then one thread per RSI) into 32-bit
 * words that the simple-packing unpack then reads.  Edition-2 complex packing (templates 5.2
 * and 5.3, first- or second-order spatial differencing, missing value management 0) is decoded
 * the same way: a group pass (block-wide scans of the group lengths and bit counts), then a
 * value pass per tile of 2 048 values that undoes the differencing as a scan, into the same
 * 32-bit words.  Its integers X must lie in [0, 2^32).  A malformed AEC stream or complex
 * section 7, or a bitmap with more set bits than the message has values, makes the call
 * return AT_ERR_INVALID naming the message.  Anything else (GRIB1 second-order, complex with
 * missing value management 1 or 2, JPEG, PNG, spectral, signed or restricted AEC, several
 * fields per message, predefined bitmaps) is AT_ERR_UNSUPPORTED from at_grib_scan and the
 * caller decodes such fields itself.
 */
#define AT_GRIB_SIMPLE 0  /* template 5.0 / GRIB1 BDS flag 0 */
#define AT_GRIB_CCSDS 1   /* template 5.42 */
#define AT_GRIB_COMPLEX 2 /* templates 5.2 and 5.3 */
typedef struct at_grib_field {
    int32_t edition;        /* 1 | 2 */
    int32_t bits_per_value; /* 0 = constant field equal to reference_value */
    int32_t binary_scale;   /* E */
    int32_t decimal_scale;  /* D */
    int32_t has_bitmap;
    int32_t packing;        /* AT_GRIB_SIMPLE | AT_GRIB_CCSDS | AT_GRIB_COMPLEX (0 in a zero-initialised scan) */
    double reference_value; /* R (IEEE float32 in edition 2, IBM float32 in edition 1) */
    int64_t n_points;       /* grid points, -1 when the message does not say (edition 1) */
    int64_t n_values;       /* packed values, -1 when the message does not say */
    int64_t data_offset;    /* octet offset of the packed values inside the message */
    int64_t data_length;    /* octets of packed values (padding included) */
    int64_t bitmap_offset;  /* octet offset of the bitmap, -1 without one */
    int64_t message_length;
    int32_t ccsds_flags;      /* template 5.42 octet 22 (0 for simple packing) */
    int32_t ccsds_block_size; /* J, octet 23 */
    int32_t ccsds_rsi;        /* reference sample interval in blocks, octets 24-25 */
    int32_t ccsds_pad;
    /* complex packing (templates 5.2 / 5.3; all 0 otherwise).  bits_per_value is octet 20,
     * the width of a group reference.  Offsets are octets from the start of section 7's data. */
    int64_t complex_groups;         /* NG, octets 32-35 */
    int64_t complex_length_ref;     /* reference for group lengths, octets 38-41 */
    int64_t complex_last_length;    /* true length of the last group, octets 43-46 */
    int32_t complex_width_ref;      /* reference for group widths, octet 36 */
    int32_t complex_width_bits;     /* bits per group width, octet 37 */
    int32_t complex_length_incr;    /* length increment, octet 42 */
    int32_t complex_length_bits;    /* bits per scaled group length, octet 47 */
    int32_t complex_order;          /* spatial differencing: 0 (5.2), 1 or 2 (5.3, octet 48) */
    int32_t complex_ww;             /* octets per extra descriptor (5.3, octet 49) */
    int64_t complex_refs_offset;    /* the NG group references */
    int64_t complex_widths_offset;  /* the NG group widths */
    int64_t complex_lengths_offset; /* the NG scaled group lengths */
    int64_t complex_values_offset;  /* the packed values, group after group */
} at_grib_field_t;
/* Host only, no CUDA call: parse one message. */
AT_API int at_grib_scan(const void* message, size_t length, at_grib_field_t* out);
/* The same for n messages in one call: status[i] is what at_grib_scan returned for message i. */
AT_API int at_grib_scan_many(const void* const* messages, const size_t* lengths, int64_t n,
                      at_grib_field_t* out, int32_t* status);
/*
 * d_pm[p, f] = value p of field f, f < n_fields: decode packed values that are already in
 * device memory.  d_packed: device buffer; byte_offsets[f] (host): where field f's packed
 * values (message + data_offset) start inside it; fields (host): the scans.
 * out_dtype AT_F64 (what to_numpy gives) or AT_F32 (that value rounded to float32).
 * Messages with a bitmap are refused here (the packed values alone do not say where they go),
 * and so are CCSDS and complex messages (they need device scratch for the decoded words):
 * at_hostio_upload_grib / at_hostio_regrid_grib stage the bitmap as well and decode both.
 */
AT_API int at_grib_unpack(const void* d_packed, const int64_t* byte_offsets, const at_grib_field_t* fields,
                   int64_t n_fields, int64_t n_points, int out_dtype, void* d_pm, int64_t ld, void* stream);
/*
 * at_hostio_upload / at_hostio_regrid for packed fields: messages[f] is the host pointer to
 * message f (any memory), fields[f] its scan.  Only the packed values (the whole section 7 of
 * a CCSDS or complex field, and the bitmap, one bit per point, of a field that has one) are
 * staged and cross PCIe; the unpack kernel replaces the pack transposition.  A chunk may mix
 * simple, CCSDS and complex fields.  x_dtype: the dtype the values
 * are decoded to (the dtype of the [points x fields] batch the matrix is applied to).
 */
AT_API int at_hostio_upload_grib(at_hostio_t* io, const void* const* messages, const at_grib_field_t* fields,
                          int64_t n_fields, int64_t n_points, int x_dtype, void* d_pm, int64_t ld, void* stream);
AT_API int at_hostio_regrid_grib(at_hostio_t* io, int op, const at_csr_t* csr, const int64_t* gather_idx,
                          int64_t n_out_points, const void* const* messages, const at_grib_field_t* fields,
                          int64_t n_fields, int64_t n_src, int x_dtype, void* d_Y, int64_t ldy,
                          void* const* fields_out, void* consumer_stream, int64_t* ticket);

/*
 * One RegridFilter.forward (regrid.py:174-208) over several GPUs from one process.  A group is
 * n_engines engines, engine e on devices[e] (a device may appear more than once: one more
 * engine there), with their own slots, streams and events and ONE pool of staging threads
 * (n_threads as in at_hostio_create: host memory bandwidth, not the device count, bounds
 * staging).  Destroying the group waits for its devices.
 */
AT_API int at_hostio_group_create(int32_t n_engines, const int32_t* devices, int32_t n_threads,
                           at_hostio_group_t** out);
AT_API int at_hostio_group_destroy(at_hostio_group_t* group);
/*
 * at_hostio_regrid / at_hostio_regrid_grib with the chunks of fields dealt to the engines: each
 * chunk goes to the first engine (counting on from the last one used) whose next input slot is
 * free.  csrs[e] (the AT_HOSTIO_SPMM* ops) / gather_idx[e] (op AT_HOSTIO_GATHER) is engine e's copy,
 * staged on devices[e] (at_csr_replicate).  Results go to the host destinations fields_out only
 * (no resident result); *ticket (at_hostio_group_wait) says when they are complete, -1 when
 * they already are.  Results equal those of one engine bit for bit.
 */
AT_API int at_hostio_group_regrid(at_hostio_group_t* group, int op, const at_csr_t* const* csrs,
                           const int64_t* const* gather_idx, int64_t n_out_points,
                           const void* const* fields_in, int64_t n_fields, int64_t n_src, int x_dtype,
                           void* const* fields_out, int64_t* ticket);
AT_API int at_hostio_group_regrid_grib(at_hostio_group_t* group, int op, const at_csr_t* const* csrs,
                                const int64_t* const* gather_idx, int64_t n_out_points,
                                const void* const* messages, const at_grib_field_t* fields, int64_t n_fields,
                                int64_t n_src, int x_dtype, void* const* fields_out, int64_t* ticket);
AT_API int at_hostio_group_wait(at_hostio_group_t* group, int64_t ticket);

/* --------------------------------------------------------------- kNN / masks -------- */
/*
 * Build the bucketed search structure over source points (float64 xyz, SoA).
 * Replaces: scipy.spatial.cKDTree(points) construction
 *           spatial.py:96, 396, 501, 533, 628-632.
 * x, y, z: float64[n]; host pointers unless on_device != 0.
 * cell_size <= 0 picks the cell from the point density.
 */
AT_API int at_knn_create(const double* x, const double* y, const double* z, int64_t n,
                  int on_device, double cell_size, at_knn_t** out);
AT_API int at_knn_destroy(at_knn_t* knn);
/*
 * k nearest sources of each query, ascending by (d², index).
 * Replaces: cKDTree.query(points, k[, distance_upper_bound])  spatial.py:96,396,501,628-632.
 * d² = ((dx·dx)+(dy·dy))+(dz·dz) in float64, unfused (bitwise cKDTree's p=2 distance);
 * dist_out = sqrt(d²).  Candidates need d² < upper_bound² (strict; upper_bound = +inf for
 * none); unfilled slots get index n and distance +inf, as cKDTree pads.
 * idx_out int64[nq,k]; dist_out float64[nq,k] or NULL;
 * tie_out uint8[nq] or NULL: bit0 = two selected neighbours have equal d²,
 *                            bit1 = the k-th and the (k+1)-th candidates have equal d²
 * (the only queries on which cKDTree's traversal order may legitimately pick differently).
 * All pointers device.  k <= 32.
 */
AT_API int at_knn_query(const at_knn_t* knn, const double* qx, const double* qy, const double* qz,
                 int64_t nq, int k, double upper_bound,
                 int64_t* idx_out, double* dist_out, uint8_t* tie_out, void* stream);
/*
 * at_knn_query for a query set sharded over the GPUs of one box, with the all-gather of the
 * indices fused into the search: every rank's query kernels store each finished index into the
 * gather buffer of EVERY rank (P2P-mapped peer memory over NVLink / NVSwitch) at
 * [row_offset + q], then a one-warp kernel exchanges arrival flags (release / acquire at system
 * scope) so that work queued on `stream` after the call sees the complete [n_total, k] result in
 * gather_bufs[rank].  Replaces query + ncclAllGather (SURVEY §8e; spatial.py:628-632 run by
 * N ranks).  gather_bufs / flag_bufs: HOST arrays of `world` device pointers (own buffers from
 * at_peer_alloc, the others' from at_peer_open); flag_bufs[r] is uint64[world], zero at start;
 * `epoch` increases by one per call on every rank — or is 0, and the library counts the calls
 * itself in device memory (flag_bufs[r] is then uint64[world + 2]), which leaves the launch
 * without per-call arguments so that a step can be captured once and replayed as a CUDA graph.
 * A rank that does not arrive within 2 s
 * sets *error_flag (device int32) instead of hanging.  dist_out / tie_out are local
 * ([nq_local, k] / [nq_local]) or NULL.  world <= 16.
 * exchange: AT_EXCHANGE_INLINE — the search kernels store to the peers as they finish each
 * query; AT_EXCHANGE_BULK — the search writes this rank's slice only and one kernel after it
 * copies the slice to every peer with coalesced 16-byte stores, its last CTA running the flag
 * exchange (flag_bufs[r] must then be uint64[world + 1]: the CTA counter follows the flags).
 */
#define AT_EXCHANGE_INLINE 0
#define AT_EXCHANGE_BULK 1
AT_API int at_knn_query_gather(const at_knn_t* knn, const double* qx, const double* qy, const double* qz,
                        int64_t nq_local, int k, double upper_bound,
                        int64_t* const* gather_bufs, uint64_t* const* flag_bufs, int world, int rank,
                        int64_t row_offset, double* dist_out, uint8_t* tie_out, uint64_t epoch,
                        int32_t* error_flag, int exchange, void* stream);
/* Device memory that the other processes of the box can map: zero-filled, `handle` receives the
 * 64-byte inter-process handle to send to the peers; at_peer_open maps a peer's buffer. */
AT_API int at_peer_alloc(size_t bytes, void** ptr, void* handle);
AT_API int at_peer_free(void* ptr);
AT_API int at_peer_open(const void* handle, void** ptr);
AT_API int at_peer_close(void* ptr);
/*
 * mark[j] = 1 for every source j with d²(q, j) <= r·r for some query q (mark is OR-ed into;
 * zero it first).  Replaces: cKDTree.query_ball_point + Python set-union  spatial.py:533-534.
 */
AT_API int at_ball_mark(const at_knn_t* knn, const double* qx, const double* qy, const double* qz,
                 int64_t nq, double r, uint8_t* mark, void* stream);
/* out_host = min over sources [first, first+count) of the distance to their 2nd nearest
 * source (self included as the 1st) — `_resolution`  spatial.py:93-97; count < 0 means
 * "to the end" (ranks take sub-ranges and all-reduce MIN).  Synchronises the stream. */
AT_API int at_min_nn_distance(const at_knn_t* knn, int64_t first, int64_t count, double* out_host,
                       void* stream);
/* Sorted indices of the non-zero bytes of mark[n] (stream compaction):
 * `np.array(sorted(set(...)))` spatial.py:534 / boolean-mask selection.
 * out_idx: device int64[n] (capacity n); *count_host receives the count. Synchronises. */
AT_API int at_compact_mask(const uint8_t* mark, int64_t n, int64_t* out_idx, int64_t* count_host,
                    void* stream);
/* cropping_mask  spatial.py:236-275 — inclusive box with ±360 longitude wrap. */
AT_API int at_cropping_mask(const double* lats, const double* lons, int64_t n,
                     double north, double west, double south, double east,
                     uint8_t* mask, void* stream);
/*
 * Per cropped global point: inside | close | too_far  — the body of the Python loop of
 * cutout_mask spatial.py:404-424 with Triangle3D.intersect spatial.py:189-233.
 * lam xyz: float64[n_lam] SoA; global xyz: float64[nq] SoA; nbr_idx int64[nq,k] and
 * nbr_dist float64[nq,k] from at_knn_query (ascending).  max_distance < 0 means None.
 * dot_mode: 0 = unfused dot products, 1 = FMA-chain dot products (OpenBLAS ddot as numpy
 * calls it on x86-64 with FMA; np.cross is always unfused).
 * out uint8[nq].  All pointers device.
 */
AT_API int at_cutout_classify(const double* lx, const double* ly, const double* lz, int64_t n_lam,
                       const double* gx, const double* gy, const double* gz, int64_t nq,
                       const int64_t* nbr_idx, const double* nbr_dist, int k,
                       double min_distance, double max_distance, int dot_mode,
                       uint8_t* out, void* stream);
/*
 * outline  spatial.py:539-584 — out[i] = 1 when a ray from the Earth's centre through point i
 * hits one of the triangles (idx[j], idx[(j+1)%k], idx[(j+2)%k]), j = 1 … k-1, of the point's
 * own k nearest neighbours (nbr_idx / nbr_dist from a self-query; neighbour 0 is the point
 * itself).  The outline is the set of points with out[i] == 0.
 */
AT_API int at_outline_classify(const double* x, const double* y, const double* z, int64_t n,
                        const int64_t* nbr_idx, const double* nbr_dist, int k, int dot_mode,
                        uint8_t* inside, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AT_B200_H */

// grib.cuh — internal interface between grib.cu (parser + unpack kernel) and hostio.cu (the
// streamed upload of packed messages).
#pragma once

#include <cstdint>

#include "common.cuh"

namespace at {

// CCSDS flags (template 5.42 octet 22, libaec's AEC_* values)
constexpr int kAecSigned = 1, kAecPreprocess = 8, kAecRestricted = 16, kAecPadRsi = 32;

// One field of a packed chunk as the kernel sees it (device table, 200 bytes).  For a CCSDS or
// complex field the unpack reads the decoded integers: byte_offset then points at the scratch
// words (big-endian, nbits = 32) that ccsds_decode_kernel or complex_values_kernel writes from
// the staged section 7.
struct GribColumn {
    long long byte_offset;    // of the field's packed values inside the chunk's device buffer
    long long bitmap_offset;  // of its bitmap (one bit per grid point, MSB first), -1 without one
    long long rank_offset;    // of its rank table (uint32 per 256 points: values before the tile), device scratch
    double reference;         // R
    double binary;            // 2^E
    double decimal;           // 10^-D
    int nbits;
    int packing;              // AT_GRIB_SIMPLE | AT_GRIB_CCSDS | AT_GRIB_COMPLEX
    long long s7_offset;      // CCSDS, complex: the staged section 7, -1 for simple packing
    long long s7_length;      //                 its octets
    long long rsi_offset;     // CCSDS: device scratch: bit offset (uint64) of every RSI
    long long n_values;       // values the field packs (what a bitmap may reference)
    int aec_bits;             //        n, bits per sample
    int aec_flags;            //        CCSDS flags
    int aec_block;            //        J
    int aec_rsi;              //        blocks per RSI
    // complex packing (templates 5.2 / 5.3); offsets of parts are octets inside section 7
    long long cx_table;       // device scratch: group starts (uint32, NG + 1), group bit offsets
                              // (uint64, NG), per tile of values its sums and carry (4 x uint64)
    long long cx_groups, cx_length_ref, cx_last_length;
    long long cx_refs, cx_widths, cx_lengths, cx_values;
    int cx_nbits, cx_width_ref, cx_width_bits, cx_length_bits, cx_length_incr, cx_order, cx_ww, cx_pad;
};
static_assert(sizeof(GribColumn) == 200, "the device table layout");

// Octets a field occupies in a chunk buffer: packed values, bitmap, rank table, CCSDS scratch
// — each part starts on a 256-byte boundary; bitmap and ranks are 0 for a field without a
// bitmap, scratch is 0 for simple packing.
struct GribFootprint {
    size_t values = 0, bitmap = 0, ranks = 0, scratch = 0;
    size_t total() const { return values + bitmap + ranks + scratch; }
    size_t value_octets = 0, bitmap_octets = 0;  // what has to be copied from the message
};

// Per-field status words of the decode kernels (0 = decoded).
enum GribStatus : int32_t {
    kCcsdsOk = 0,
    kCcsdsTruncated = 1,   // the stream ends before value n_values - 1
    kCcsdsBadOption = 2,   // a split option with k >= n
    kCcsdsZeroRun = 3,     // a zero-block run leaves its RSI
    kCcsdsRange = 4,       // a sample (or mapped difference) above 2^n - 1
    kComplexLengths = 5,   // group lengths that do not sum to the value count
    kComplexOverrun = 6,   // value bits that run past section 7
    kComplexWidth = 7,     // a group width above 32
    kComplexRange = 8,     // a final X outside [0, 2^32)
    kBitmapCount = 9,      // a bitmap with more set bits than the field has values
};
const char* grib_status_text(int32_t code);

// Decode the CCSDS fields of a chunk into their scratch words (other fields are skipped):
// ccsds_rsi_scan_kernel, then ccsds_decode_kernel.  err[f]: status word of field f (zeroed by
// the caller), max_rsi: the most RSIs of any CCSDS field of the chunk (0: nothing is launched).
int ccsds_decode_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int32_t* d_err, long long max_rsi, cudaStream_t st);
// Decode the complex fields of a chunk into their scratch words (other fields are skipped):
// complex_groups_kernel, then for spatial differencing complex_tile_sums_kernel and
// complex_carry_kernel, then complex_values_kernel.  max_tiles: the most value tiles of any
// complex field of the chunk (0: no complex field, nothing is launched).
int complex_decode_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int32_t* d_err, long long max_tiles, cudaStream_t st);
GribFootprint grib_footprint(const at_grib_field_t& info, int64_t n_points);
// RSIs of a CCSDS field of n_values samples (0 for simple packing and constant fields).
int64_t ccsds_rsi_count(const at_grib_field_t& info, int64_t n_values);
// Value tiles of a complex field of n_values values.
int64_t complex_tile_count(int64_t n_values);

// Validate one scanned message against the batch (value count, section lengths) and fill its
// kernel parameters for a field region that starts at `byte_offset` of the chunk buffer.
int grib_column_of(const at_grib_field_t& info, int64_t n_points, int64_t byte_offset, GribColumn* out);

// out[p, f] = value p of field f for f < n_fields (out_dtype AT_F32 | AT_F64, leading dimension ld).
// `any_bitmap`: some field has one (the rank tables are then built first, inside d_packed, and
// a bitmap with more set bits than its field has values sets d_err[f] and is cleared).
int grib_unpack_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int64_t n_points, int out_dtype, void* d_pm,
                       int64_t ld, bool any_bitmap, int32_t* d_err, cudaStream_t st);

}  // namespace at

// grib.cuh — internal interface between grib.cu (parser + unpack kernel) and hostio.cu (the
// streamed upload of packed messages).
#pragma once

#include <cstdint>

#include "common.cuh"

namespace at {

// CCSDS flags (template 5.42 octet 22, libaec's AEC_* values)
constexpr int kAecSigned = 1, kAecPreprocess = 8, kAecRestricted = 16, kAecPadRsi = 32;

// One field of a packed chunk as the kernel sees it (device table, 104 bytes).  For a CCSDS
// field the unpack reads the decoded samples: byte_offset then points at the scratch words
// (big-endian, nbits = 32) that ccsds_decode_kernel writes from the staged AEC stream.
struct GribColumn {
    long long byte_offset;    // of the field's packed values inside the chunk's device buffer
    long long bitmap_offset;  // of its bitmap (one bit per grid point, MSB first), -1 without one
    long long rank_offset;    // of its rank table (uint32 per 256 points: values before the tile), device scratch
    double reference;         // R
    double binary;            // 2^E
    double decimal;           // 10^-D
    int nbits;
    int packing;              // AT_GRIB_SIMPLE | AT_GRIB_CCSDS
    long long aec_offset;     // CCSDS: the staged AEC stream (section 7), -1 for simple packing
    long long aec_length;     //        its octets
    long long rsi_offset;     //        device scratch: bit offset (uint64) of every RSI
    long long n_values;       //        samples in the stream
    int aec_bits;             //        n, bits per sample
    int aec_flags;            //        CCSDS flags
    int aec_block;            //        J
    int aec_rsi;              //        blocks per RSI
};

// Octets a field occupies in a chunk buffer: packed values, bitmap, rank table, CCSDS scratch
// — each part starts on a 256-byte boundary; bitmap and ranks are 0 for a field without a
// bitmap, scratch is 0 for simple packing.
struct GribFootprint {
    size_t values = 0, bitmap = 0, ranks = 0, scratch = 0;
    size_t total() const { return values + bitmap + ranks + scratch; }
    size_t value_octets = 0, bitmap_octets = 0;  // what has to be copied from the message
};

// Per-field status words of the CCSDS kernels (0 = decoded).
enum CcsdsError : int32_t {
    kCcsdsOk = 0,
    kCcsdsTruncated = 1,   // the stream ends before value n_values - 1
    kCcsdsBadOption = 2,   // a split option with k >= n
    kCcsdsZeroRun = 3,     // a zero-block run leaves its RSI
    kCcsdsRange = 4,       // a sample (or mapped difference) above 2^n - 1
};
const char* ccsds_error_text(int32_t code);

// Decode the CCSDS fields of a chunk into their scratch words (simple fields are skipped):
// ccsds_rsi_scan_kernel, then ccsds_decode_kernel.  err[f]: status word of field f (zeroed by
// the caller), max_rsi: the most RSIs of any CCSDS field of the chunk.
int ccsds_decode_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int32_t* d_err, long long max_rsi, cudaStream_t st);
GribFootprint grib_footprint(const at_grib_field_t& info, int64_t n_points);
// RSIs of a CCSDS field of n_values samples (0 for simple packing and constant fields).
int64_t ccsds_rsi_count(const at_grib_field_t& info, int64_t n_values);

// Validate one scanned message against the batch (value count, section lengths) and fill its
// kernel parameters for a field region that starts at `byte_offset` of the chunk buffer.
int grib_column_of(const at_grib_field_t& info, int64_t n_points, int64_t byte_offset, GribColumn* out);

// out[p, f] = value p of field f for f < n_fields (out_dtype AT_F32 | AT_F64, leading dimension ld).
// `any_bitmap`: some field has one (the rank tables are then built first, inside d_packed).
int grib_unpack_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int64_t n_points, int out_dtype, void* d_pm,
                       int64_t ld, bool any_bitmap, cudaStream_t st);

}  // namespace at

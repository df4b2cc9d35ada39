// grib.cu — GRIB simple packing decoded on the device, straight into the point-major batch.
//
// Where this sits: a GRIB-backed FieldList reaches RegridFilter.forward as earthkit-data
// GribFields, and the per-field `field.to_numpy(flatten=True)` of the reference
// (src/anemoi/transform/filters/fields/regrid.py:309, matching.py:242-246) is where ecCodes
// decodes each message to float64 on one CPU core.  Here the packed octets (2 bytes per point
// at 16 bits, instead of 8 bytes of decoded float64) cross PCIe and the kernel below unpacks
// them into columns of the [points x fields] batch the SpMM reads (SURVEY §8(f) rank 4).
//
//   at_grib_scan      host: locate packing parameters, the packed values and the bitmap of one
//                     message (editions 1 and 2, grid-point simple packing; edition 2 CCSDS
//                     packing, template 5.42, and complex packing, templates 5.2 / 5.3)
//   ccsds_*_kernel    device: a CCSDS field's AEC stream -> its integers X as 32-bit words
//   complex_*_kernel  device: a complex field's groups (and spatial differencing) -> the same
//   at_grib_unpack    device: Y = ((X · 2^E) + R) · 10^-D for a batch of fields, fused with the
//                     field-major -> point-major transposition
//
// Arithmetic: float64, one multiplication, one addition, one multiplication, never fused —
// the order ecCodes' data_simple_packing uses (restated in oracle/grib.py; parity with ecCodes
// itself is unpinned offline, see DESIGN.md).  For D = 0 the result is the correctly rounded
// R + X·2^E whatever the order.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "grib.cuh"

namespace at {

namespace {

// ---- host: message scan ----------------------------------------------------------------
inline uint64_t be(const uint8_t* p, int n) {
    uint64_t v = 0;
    for (int i = 0; i < n; ++i) v = (v << 8) | p[i];
    return v;
}

inline int sign_magnitude16(const uint8_t* p) {
    const int u = static_cast<int>(be(p, 2));
    return (u & 0x8000) ? -(u & 0x7fff) : (u & 0x7fff);
}

inline double ibm32(const uint8_t* p) {
    const uint32_t u = static_cast<uint32_t>(be(p, 4));
    const uint32_t mantissa = u & 0xffffffu;
    const int exponent = static_cast<int>((u >> 24) & 0x7f);
    if (mantissa == 0) return 0.0;
    const double v = std::ldexp(static_cast<double>(mantissa), 4 * (exponent - 64 - 6));  // 16^(e-70), exact
    return (u >> 31) ? -v : v;
}

inline double ieee32(const uint8_t* p) {
    const uint32_t u = static_cast<uint32_t>(be(p, 4));
    float f;
    std::memcpy(&f, &u, 4);
    return static_cast<double>(f);
}

#define GRIB_NEED(cond, ...)                                             \
    do {                                                                 \
        if (!(cond)) return set_error(AT_ERR_INVALID, __VA_ARGS__);      \
    } while (0)
#define GRIB_UNSUPPORTED(...) return set_error(AT_ERR_UNSUPPORTED, __VA_ARGS__)

// The AEC parameters the device decodes: unsigned samples, the full option set, J in
// {8, 16, 32, 64}, RSI in [1, 4096], n <= 32.  Flags 2 (3BYTE) and 4 (MSB) only describe
// libaec's sample layout in memory; PREPROCESS (8) and PAD_RSI (32) are handled.
int ccsds_check(const at_grib_field_t& o, const char* who) {
    if (o.ccsds_flags & kAecSigned) GRIB_UNSUPPORTED("%s: signed samples (CCSDS flags 0x%02x)", who, o.ccsds_flags);
    if ((o.ccsds_flags & kAecRestricted) && o.bits_per_value <= 4)
        GRIB_UNSUPPORTED("%s: restricted option set for %d-bit samples (CCSDS flags 0x%02x)", who, o.bits_per_value, o.ccsds_flags);
    const int J = o.ccsds_block_size;
    if (J != 8 && J != 16 && J != 32 && J != 64) GRIB_UNSUPPORTED("%s: block size %d (8, 16, 32 or 64)", who, J);
    if (o.ccsds_rsi < 1 || o.ccsds_rsi > 4096) GRIB_UNSUPPORTED("%s: reference sample interval %d (1 .. 4096)", who, o.ccsds_rsi);
    if (o.bits_per_value < 0 || o.bits_per_value > 32) GRIB_UNSUPPORTED("%s: %d bits per value", who, o.bits_per_value);
    return AT_OK;
}

// The octet offsets of the parts of a complex field's section 7, from NG and the bit counts
// alone: extra descriptors (5.3), group references, widths and scaled lengths (each padded to
// an octet), then the values.  The groups themselves are walked on the device.
int complex_parts(at_grib_field_t* o) {
    const int64_t ng = o->complex_groups;
    GRIB_NEED(ng > 0 || o->n_values == 0, "at_grib_scan: complex packing with no groups for %lld values", (long long)o->n_values);
    GRIB_NEED(ng <= o->n_values, "at_grib_scan: complex packing with %lld groups for %lld values", (long long)ng, (long long)o->n_values);
    o->complex_refs_offset = o->complex_order > 0 ? static_cast<int64_t>(o->complex_order + 1) * o->complex_ww : 0;
    o->complex_widths_offset = o->complex_refs_offset + (ng * o->bits_per_value + 7) / 8;
    o->complex_lengths_offset = o->complex_widths_offset + (ng * o->complex_width_bits + 7) / 8;
    o->complex_values_offset = o->complex_lengths_offset + (ng * o->complex_length_bits + 7) / 8;
    GRIB_NEED(o->complex_values_offset <= o->data_length, "at_grib_scan: complex packing: the group descriptors need %lld octets, section 7 holds %lld",
              (long long)o->complex_values_offset, (long long)o->data_length);
    return AT_OK;
}

int scan_edition2(const uint8_t* m, size_t len, at_grib_field_t* o) {
    GRIB_NEED(len >= 20, "at_grib_scan: truncated edition-2 message");
    const uint64_t total = be(m + 8, 8);
    GRIB_NEED(total <= len && total >= 20, "at_grib_scan: message length %llu exceeds the buffer (%zu)", (unsigned long long)total, len);
    GRIB_NEED(std::memcmp(m + total - 4, "7777", 4) == 0, "at_grib_scan: end section missing");
    o->edition = 2;
    o->message_length = static_cast<int64_t>(total);
    size_t pos = 16;
    int seen5 = 0, seen7 = 0, seen3 = 0;
    while (pos + 5 <= total - 4) {
        const uint64_t sl = be(m + pos, 4);
        const int number = m[pos + 4];
        GRIB_NEED(sl >= 5 && pos + sl <= total - 4, "at_grib_scan: section %d overruns the message", number);
        switch (number) {
            case 3:
                GRIB_NEED(sl >= 14, "at_grib_scan: section 3 too short");
                o->n_points = static_cast<int64_t>(be(m + pos + 6, 4));
                ++seen3;
                break;
            case 5: {
                GRIB_NEED(sl >= 11, "at_grib_scan: section 5 too short");
                o->n_values = static_cast<int64_t>(be(m + pos + 5, 4));
                const int tmpl = static_cast<int>(be(m + pos + 9, 2));
                if (tmpl != 0 && tmpl != 2 && tmpl != 3 && tmpl != 42)
                    GRIB_UNSUPPORTED("at_grib_scan: data representation template 5.%d (only 5.0, simple packing, 5.2 / 5.3, complex packing, and 5.42, CCSDS)", tmpl);
                // a 5.42 section without its CCSDS octets is not something the device decodes
                if (tmpl == 42 && sl < 25) GRIB_UNSUPPORTED("at_grib_scan: template 5.42 section of %llu octets (25 needed)", (unsigned long long)sl);
                if ((tmpl == 2 && sl < 47) || (tmpl == 3 && sl < 49))
                    GRIB_UNSUPPORTED("at_grib_scan: template 5.%d section of %llu octets (%d needed)", tmpl, (unsigned long long)sl, tmpl == 2 ? 47 : 49);
                GRIB_NEED(sl >= 20, "at_grib_scan: template 5.0 too short");
                o->reference_value = ieee32(m + pos + 11);
                o->binary_scale = sign_magnitude16(m + pos + 15);
                o->decimal_scale = sign_magnitude16(m + pos + 17);
                o->bits_per_value = m[pos + 19];
                if (tmpl == 42) {
                    o->packing = AT_GRIB_CCSDS;
                    o->ccsds_flags = m[pos + 21];
                    o->ccsds_block_size = m[pos + 22];
                    o->ccsds_rsi = static_cast<int32_t>(be(m + pos + 23, 2));
                    const int rc = ccsds_check(*o, "at_grib_scan: template 5.42");
                    if (rc != AT_OK) return rc;
                }
                if (tmpl == 2 || tmpl == 3) {
                    const uint8_t* q = m + pos - 1;  // q[k] = octet k of the section
                    o->packing = AT_GRIB_COMPLEX;
                    if (q[23] != 0) GRIB_UNSUPPORTED("at_grib_scan: template 5.%d with missing value management %d (only 0)", tmpl, q[23]);
                    o->complex_groups = static_cast<int64_t>(be(q + 32, 4));
                    o->complex_width_ref = q[36];
                    o->complex_width_bits = q[37];
                    o->complex_length_ref = static_cast<int64_t>(be(q + 38, 4));
                    o->complex_length_incr = q[42];
                    o->complex_last_length = static_cast<int64_t>(be(q + 43, 4));
                    o->complex_length_bits = q[47];
                    if (tmpl == 3) {
                        o->complex_order = q[48];
                        o->complex_ww = q[49];
                        if (o->complex_order != 1 && o->complex_order != 2)
                            GRIB_UNSUPPORTED("at_grib_scan: template 5.3 with spatial differencing of order %d (1 or 2)", o->complex_order);
                        if (o->complex_ww < 1 || o->complex_ww > 4)
                            GRIB_UNSUPPORTED("at_grib_scan: template 5.3 with %d octets per extra descriptor (1 .. 4)", o->complex_ww);
                    }
                    // wider fields cannot hold a 32-bit X or a group width up to 32
                    if (o->bits_per_value > 32 || o->complex_width_bits > 32 || o->complex_length_bits > 32)
                        GRIB_UNSUPPORTED("at_grib_scan: template 5.%d with %d / %d / %d bits per group reference / width / length (32 at most)", tmpl,
                                         o->bits_per_value, o->complex_width_bits, o->complex_length_bits);
                }
                ++seen5;
                break;
            }
            case 6: {
                GRIB_NEED(sl >= 6, "at_grib_scan: section 6 too short");
                const int indicator = m[pos + 5];
                if (indicator == 0) {
                    o->has_bitmap = 1;
                    o->bitmap_offset = static_cast<int64_t>(pos + 6);
                } else if (indicator != 255) {
                    GRIB_UNSUPPORTED("at_grib_scan: bitmap indicator %d", indicator);
                }
                break;
            }
            case 7:
                o->data_offset = static_cast<int64_t>(pos + 5);
                o->data_length = static_cast<int64_t>(sl - 5);
                ++seen7;
                break;
            default:
                break;
        }
        pos += sl;
    }
    if (seen7 != 1 || seen5 != 1 || seen3 != 1) GRIB_UNSUPPORTED("at_grib_scan: expected one field per message (sections 3/5/7 seen %d/%d/%d times)", seen3, seen5, seen7);
    if (o->packing == AT_GRIB_COMPLEX) return complex_parts(o);
    return AT_OK;
}

int scan_edition1(const uint8_t* m, size_t len, at_grib_field_t* o) {
    const uint32_t len3 = static_cast<uint32_t>(be(m + 4, 3));
    size_t pos = 8;
    GRIB_NEED(len >= pos + 28, "at_grib_scan: truncated edition-1 message");
    const size_t pds_len = be(m + pos, 3);
    GRIB_NEED(pds_len >= 28 && pos + pds_len <= len, "at_grib_scan: bad PDS length");
    const int flag = m[pos + 7];
    o->edition = 1;
    o->decimal_scale = sign_magnitude16(m + pos + 26);
    pos += pds_len;
    if (flag & 0x80) {
        GRIB_NEED(pos + 3 <= len, "at_grib_scan: truncated GDS");
        pos += be(m + pos, 3);
    }
    int64_t n_points = -1;
    if (flag & 0x40) {
        GRIB_NEED(pos + 6 <= len, "at_grib_scan: truncated BMS");
        const size_t bms_len = be(m + pos, 3);
        if (be(m + pos + 4, 2) != 0) GRIB_UNSUPPORTED("at_grib_scan: predefined bitmaps");
        o->has_bitmap = 1;
        o->bitmap_offset = static_cast<int64_t>(pos + 6);
        n_points = static_cast<int64_t>(bms_len - 6) * 8 - m[pos + 3];
        pos += bms_len;
    }
    GRIB_NEED(pos + 11 <= len, "at_grib_scan: truncated BDS");
    const uint64_t stored4 = be(m + pos, 3);
    uint64_t total, bds_len;
    const bool long_message = (len3 & 0x800000u) != 0;
    if (long_message) {  // ECMWF convention: units of 120 octets, stored section-4 length subtracted
        total = static_cast<uint64_t>(len3 & 0x7fffffu) * 120u - stored4;
        GRIB_NEED(total > pos + 15, "at_grib_scan: bad long-message length");
        bds_len = total - 4 - pos;
    } else {
        total = len3;
        bds_len = stored4;
    }
    GRIB_NEED(total <= len && bds_len >= 11 && pos + bds_len + 4 <= total, "at_grib_scan: message length %llu exceeds the buffer (%zu)", (unsigned long long)total, len);
    GRIB_NEED(std::memcmp(m + total - 4, "7777", 4) == 0, "at_grib_scan: end section missing");
    const int flags4 = m[pos + 3];
    if (flags4 & 0xf0) GRIB_UNSUPPORTED("at_grib_scan: BDS flags 0x%02x (only grid-point simple packing of float values)", flags4 & 0xf0);
    o->binary_scale = sign_magnitude16(m + pos + 4);
    o->reference_value = ibm32(m + pos + 6);
    o->bits_per_value = m[pos + 10];
    o->data_offset = static_cast<int64_t>(pos + 11);
    o->data_length = static_cast<int64_t>(bds_len - 11);
    // the value count is implied by the section length; a long message pads without recording it
    o->n_values = (o->bits_per_value > 0 && !long_message) ? (o->data_length * 8 - (flags4 & 0x0f)) / o->bits_per_value : -1;
    o->n_points = n_points >= 0 ? n_points : o->n_values;
    o->message_length = static_cast<int64_t>(total);
    return AT_OK;
}

// n^s by repeated multiplication / division from 1.0 (how ecCodes forms 2^E and 10^-D).
double repeated_power(long s, long n) {
    double v = 1.0;
    if (s == 0) return 1.0;
    if (s == 1) return static_cast<double>(n);
    while (s < 0) {
        v /= static_cast<double>(n);
        ++s;
    }
    while (s > 0) {
        v *= static_cast<double>(n);
        --s;
    }
    return v;
}

}  // namespace

// ---- device: unpack + transpose ---------------------------------------------------------
constexpr int kTileFields = 32;   // columns of a CTA tile (one warp-wide row segment)
constexpr int kTilePoints = 256;  // points of a CTA tile: 32 lanes x 8 values

__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }

// Field status words: the first failure of a field is kept.
__device__ __forceinline__ void fail_field(int32_t* err, int code) { atomicCAS(reinterpret_cast<int*>(err), 0, code); }

// The 8 values of point group g (points 8g .. 8g+7) of one field start on an octet boundary:
// 8·nbits bits = nbits octets.  `avail` = values of the group that exist (8 except at the end).
template <typename TOut>
__device__ __forceinline__ void unpack_group(const uint8_t* __restrict__ src, const GribColumn& c, int avail, TOut* __restrict__ dst) {
    const int nbits = c.nbits;
    if (nbits == 0) {
#pragma unroll
        for (int v = 0; v < 8; ++v)
            if (v < avail) dst[v] = static_cast<TOut>(c.reference);
        return;
    }
    uint32_t x[8];
    if (nbits == 16 && avail == 8 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(src));
        const uint32_t ws[4] = {bswap32(w.x), bswap32(w.y), bswap32(w.z), bswap32(w.w)};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            x[2 * j] = ws[j] >> 16;
            x[2 * j + 1] = ws[j] & 0xffffu;
        }
    } else if ((nbits & 3) == 0 && avail == 8 && (reinterpret_cast<uintptr_t>(src) & 3) == 0) {
        // whole 32-bit words: nbits / 4 of them hold the 8 values
        const uint32_t* w = reinterpret_cast<const uint32_t*>(src);
        const int n_words = nbits >> 2;
        unsigned long long acc = 0;
        int have = 0, next = 0;
        const uint32_t mask = nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u);
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            if (have < nbits) {
                acc = (acc << 32) | (next < n_words ? bswap32(__ldg(w + next)) : 0u);
                ++next;
                have += 32;
            }
            x[v] = static_cast<uint32_t>(acc >> (have - nbits)) & mask;
            have -= nbits;
        }
    } else {
        // any width, any alignment, partial last group: octet by octet
        const int n_octets = (avail * nbits + 7) >> 3;
        unsigned long long acc = 0;
        int have = 0, next = 0;
        const uint32_t mask = nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u);
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            x[v] = 0;
            if (v < avail) {
                while (have < nbits) {
                    acc = (acc << 8) | (next < n_octets ? __ldg(src + next) : 0u);
                    ++next;
                    have += 8;
                }
                x[v] = static_cast<uint32_t>(acc >> (have - nbits)) & mask;
                have -= nbits;
            }
        }
    }
#pragma unroll
    for (int v = 0; v < 8; ++v) {
        if (v < avail) {
            const double y = __dmul_rn(__dadd_rn(__dmul_rn(static_cast<double>(x[v]), c.binary), c.reference), c.decimal);
            dst[v] = static_cast<TOut>(y);
        }
    }
}

// ---- bitmaps: points without a value ------------------------------------------------------
// A field with a bitmap packs only the points whose bit is set; point p's value is number
// rank(p) = (set bits before p) of the stream.  grib_bitmap_rank_kernel writes, per field and per
// tile of 256 points, the rank of the tile's first point (one warp per field, 32 tiles per step,
// warp scan with carry); the unpack kernel adds the set bits of the lanes before it inside the
// tile.  A missing point decodes to NaN (what earthkit-data's to_numpy() hands to the filters).
//
// A bitmap with more set bits than the field has values would send the unpack past them: the
// kernel then clears the bitmap (nothing is read, every point decodes to NaN) and sets the
// field's status word, which fails the call.
__global__ void __launch_bounds__(32)
    grib_bitmap_rank_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, long long n_points, int32_t* __restrict__ err) {
    const GribColumn c = cols[blockIdx.x];
    if (c.bitmap_offset < 0) return;
    const int lane = threadIdx.x;
    const uint32_t* words = reinterpret_cast<const uint32_t*>(packed + c.bitmap_offset);  // 256-byte aligned
    uint32_t* rank = reinterpret_cast<uint32_t*>(packed + c.rank_offset);
    const long long n_tiles = (n_points + kTilePoints - 1) / kTilePoints;
    unsigned long long carry = 0;
    for (long long t0 = 0; t0 < n_tiles; t0 += 32) {
        const long long t = t0 + lane;
        uint32_t count = 0;
        if (t < n_tiles) {
            const long long first = t * kTilePoints;
            const int valid = static_cast<int>(min(static_cast<long long>(kTilePoints), n_points - first));
#pragma unroll
            for (int w = 0; w < kTilePoints / 32; ++w) {
                const int v = valid - 32 * w;  // points of this word that exist
                if (v <= 0) break;
                uint32_t word = words[t * (kTilePoints / 32) + w];
                if (v < 32) {
                    // point i of the word is bit 7 - i % 8 of octet i / 8; octet j is bits 8j .. 8j+7 of the little-endian word
                    const int whole = v >> 3, rest = v & 7;
                    uint32_t mask = whole >= 4 ? 0xffffffffu : ((1u << (8 * whole)) - 1u);
                    if (rest != 0) mask |= ((0xffu << (8 - rest)) & 0xffu) << (8 * whole);
                    word &= mask;
                }
                count += __popc(word);
            }
        }
        uint32_t inc = count;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (t < n_tiles) rank[t] = static_cast<uint32_t>(carry + inc - count);
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (carry > static_cast<unsigned long long>(c.n_values)) {
        uint32_t* bitmap = reinterpret_cast<uint32_t*>(packed + c.bitmap_offset);
        for (long long w = lane; w < (n_points + 31) / 32; w += 32) bitmap[w] = 0;
        if (lane == 0 && err != nullptr) fail_field(err + blockIdx.x, kBitmapCount);
    }
}

// Value number `index` of a stream of nbits-wide big-endian fields that starts at `values`.
__device__ __forceinline__ uint32_t extract_bits(const uint8_t* __restrict__ values, long long index, int nbits) {
    const long long bit = index * nbits;
    const uint8_t* b = values + (bit >> 3);
    const int shift = static_cast<int>(bit & 7);
    // shift + nbits <= 39 bits: five octets (the regions carry 16 octets of slack)
    unsigned long long acc = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) acc = (acc << 8) | __ldg(b + i);
    const uint32_t mask = nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u);
    return static_cast<uint32_t>(acc >> (40 - shift - nbits)) & mask;
}

template <typename TOut>
__device__ __forceinline__ void unpack_group_bitmap(const uint8_t* __restrict__ packed, const GribColumn& c, long long p0,
                                                    long long n_points, int lane, int avail, TOut* __restrict__ dst) {
    // this lane's octet of the bitmap: points p0 + 8·lane .. + 7, MSB first
    uint32_t bits = 0;
    if (avail > 0) {
        bits = __ldg(packed + c.bitmap_offset + ((p0 >> 3) + lane));
        if (avail < 8) bits &= (0xffu << (8 - avail)) & 0xffu;
    }
    uint32_t inc = __popc(bits);
    const uint32_t mine = inc;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    const uint32_t* rank = reinterpret_cast<const uint32_t*>(packed + c.rank_offset);
    long long index = static_cast<long long>(__ldg(rank + p0 / kTilePoints)) + (inc - mine);
    const uint8_t* values = packed + c.byte_offset;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (k >= avail) break;
        if (bits & (0x80u >> k)) {
            const uint32_t x = c.nbits == 0 ? 0u : extract_bits(values, index, c.nbits);
            ++index;
            const double y = c.nbits == 0 ? c.reference : __dmul_rn(__dadd_rn(__dmul_rn(static_cast<double>(x), c.binary), c.reference), c.decimal);
            dst[k] = static_cast<TOut>(y);
        } else {
            dst[k] = static_cast<TOut>(__longlong_as_double(0x7ff8000000000000ll));
        }
    }
}

// One CTA per (tile of 256 points, group of 32 fields).  Warp w unpacks fields w, w+8, w+16,
// w+24 of the group (every lane 8 consecutive points: coalesced reads of nbits octets per lane)
// into shared memory; then every warp writes rows of 32 adjacent columns of the batch.
template <typename TOut, bool BITMAPS>
__global__ void __launch_bounds__(256)
    grib_unpack_kernel(const uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int n_fields, long long n_points,
                       TOut* __restrict__ out, long long ld, unsigned n_field_groups) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TOut* tile = reinterpret_cast<TOut*>(smem_raw);  // [kTileFields][kTilePoints + 1]
    constexpr int kPitch = kTilePoints + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // field groups vary fastest: CTAs that run together write adjacent column segments of the
    // same rows, so whole rows of the batch reach DRAM together
    const long long p0 = static_cast<long long>(blockIdx.x / n_field_groups) * kTilePoints;
    const int f0 = static_cast<int>(blockIdx.x % n_field_groups) * kTileFields;
    const long long p = p0 + lane * 8;
    const int avail = static_cast<int>(max(0ll, min(8ll, n_points - p)));
#pragma unroll 1
    for (int j = warp; j < kTileFields; j += 8) {
        const int f = f0 + j;
        if (f >= n_fields) continue;  // warp-uniform
        const GribColumn c = cols[f];
        TOut v[8];
        if (BITMAPS && c.bitmap_offset >= 0) {  // warp-uniform: the whole warp takes part in the scan
            unpack_group_bitmap<TOut>(packed, c, p0, n_points, lane, avail, v);
        } else {
            if (avail <= 0) continue;
            unpack_group<TOut>(packed + c.byte_offset + (p >> 3) * c.nbits, c, avail, v);
        }
        // point 8·lane + k of the tile is kept at position 32·k + lane: consecutive lanes write
        // consecutive words (position 8·lane + k put 32 lanes on 2 banks: ncu counted 121 M
        // bank conflicts per launch and the kernel sat at 0.52 of the HBM peak)
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < avail) tile[j * kPitch + k * 32 + lane] = v[k];
    }
    __syncthreads();
    const int f = f0 + lane;
    const int rows = static_cast<int>(min(static_cast<long long>(kTilePoints), n_points - p0));
    if (f < n_fields)
        for (int r = warp; r < rows; r += 8) out[(p0 + r) * ld + f] = tile[lane * kPitch + (r & 7) * 32 + (r >> 3)];
}

// ---- CCSDS (template 5.42): AEC stream -> 32-bit words -----------------------------------
// The stream (CCSDS 121.0-B with libaec's conventions, restated in oracle/ccsds.py) is blocks of
// J samples, `rsi` blocks per reference sample interval.  Only RSI boundaries are points where
// decoding can start, and without AEC_PAD_RSI they are not octet-aligned: ccsds_rsi_scan_kernel
// walks the block headers once and records the bit offset of every RSI, then
// ccsds_decode_kernel decodes every RSI in its own thread.  Every read is bounded by the staged
// length (octets past it read as zero); a stream that runs out, or breaks a rule, sets the
// field's status word and the kernels stop on that field.
constexpr int kAecSegment = 64;  // blocks of a "remainder of segment" zero run
constexpr int kAecRos = 5;       // zero-block code z meaning "remainder of segment"
constexpr int kDecodeThreads = 64;

__device__ __forceinline__ int aec_id_length(int n) { return n > 16 ? 5 : (n > 8 ? 4 : 3); }

__device__ __forceinline__ uint32_t aec_byte(const uint8_t* __restrict__ s, long long len, long long i) {
    return i < len ? static_cast<uint32_t>(__ldg(s + i)) : 0u;
}

// 32 stream bits from bit `pos`, MSB first; zeros past the end.
__device__ __forceinline__ uint32_t aec_word(const uint8_t* __restrict__ s, long long len, long long pos) {
    const long long b = pos >> 3;
    unsigned long long acc = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) acc = (acc << 8) | aec_byte(s, len, b + i);
    return static_cast<uint32_t>(acc >> (8 - static_cast<int>(pos & 7)));
}

__device__ __forceinline__ uint32_t aec_bits(const uint8_t* __restrict__ s, long long len, long long pos, int w) {
    return w == 0 ? 0u : aec_word(s, len, pos) >> (32 - w);
}

// The position just past the count-th set bit at or after `pos` (the end of `count` FS codes),
// found by the whole warp over 1 024-bit windows: a popcount per lane and word, a warp scan,
// and __fns in the word that holds it.  -1 when the stream ends first.
__device__ long long warp_skip_fs(const uint8_t* __restrict__ s, long long len, long long pos, int count, int lane) {
    const long long limit = len * 8;
    int need = count;
    while (pos < limit) {
        const uint32_t w = aec_word(s, len, pos + 32ll * lane);
        const int c = __popc(w);
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        const int total = __shfl_sync(0xffffffffu, inc, 31);
        if (total >= need) {
            const int l = __ffs(__ballot_sync(0xffffffffu, inc >= need)) - 1;
            const int before = __shfl_sync(0xffffffffu, inc - c, l);
            const uint32_t wl = __shfl_sync(0xffffffffu, w, l);
            // stream bit i of the word is bit i of its reverse
            return pos + 32ll * l + static_cast<long long>(__fns(__brev(wl), 0, need - before)) + 1;
        }
        need -= total;
        pos += 1024;
    }
    return -1;
}


// One warp per field of the chunk (simple-packed fields return at once).  It walks RSIs
// 0 .. n_rsi - 2 (the last RSI's offset is known once the one before it is walked) and writes
// offsets[r] = bit offset of RSI r.
__global__ void __launch_bounds__(32)
    ccsds_rsi_scan_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (c.packing != AT_GRIB_CCSDS || c.aec_bits == 0 || c.n_values <= 0) return;
    const int lane = threadIdx.x;
    const uint8_t* s = packed + c.s7_offset;
    const long long len = c.s7_length, limit = len * 8;
    const int n = c.aec_bits, J = c.aec_block, rsi = c.aec_rsi, idlen = aec_id_length(n);
    const bool pre = (c.aec_flags & kAecPreprocess) != 0, pad = (c.aec_flags & kAecPadRsi) != 0;
    const long long n_blocks = (c.n_values + J - 1) / J, n_rsi = (n_blocks + rsi - 1) / rsi;
    unsigned long long* offsets = reinterpret_cast<unsigned long long*>(packed + c.rsi_offset);
    if (lane == 0) offsets[0] = 0;
    long long pos = 0;
    for (long long r = 0; r + 1 < n_rsi; ++r) {
        int b = 0;
        while (b < rsi) {
            const int ref = (pre && b == 0) ? 1 : 0;
            const uint32_t id = aec_bits(s, len, pos, idlen);
            pos += idlen;
            if (id == 0) {
                const uint32_t second = aec_bits(s, len, pos, 1);
                pos += 1 + ref * n;
                const long long next = warp_skip_fs(s, len, pos, second ? J / 2 : 1, lane);
                if (next < 0) {
                    if (lane == 0) fail_field(err + blockIdx.x, kCcsdsTruncated);
                    return;
                }
                if (!second) {
                    const long long z = next - pos;  // FS code m, z = m + 1
                    const long long run = z == kAecRos ? min(rsi - b, kAecSegment - b % kAecSegment) : (z > kAecRos ? z - 1 : z);
                    if (b + run > rsi) {
                        if (lane == 0) fail_field(err + blockIdx.x, kCcsdsZeroRun);
                        return;
                    }
                    pos = next;
                    b += static_cast<int>(run);
                    continue;
                }
                pos = next;
            } else if (id == (1u << idlen) - 1u) {
                pos += static_cast<long long>(J) * n;
            } else {
                const int k = static_cast<int>(id) - 1;
                if (k >= n) {
                    if (lane == 0) fail_field(err + blockIdx.x, kCcsdsBadOption);
                    return;
                }
                pos += ref * n;
                const long long next = warp_skip_fs(s, len, pos, J - ref, lane);
                if (next < 0) {
                    if (lane == 0) fail_field(err + blockIdx.x, kCcsdsTruncated);
                    return;
                }
                pos = next + static_cast<long long>(J - ref) * k;
            }
            if (pos > limit) {
                if (lane == 0) fail_field(err + blockIdx.x, kCcsdsTruncated);
                return;
            }
            ++b;
        }
        if (pad) pos = (pos + 7) & ~7ll;
        if (lane == 0) offsets[r + 1] = static_cast<unsigned long long>(pos);
    }
}

// Sequential reader of one thread: a 64-bit window, MSB first, refilled octet by octet.
struct AecReader {
    const uint8_t* s;
    long long len, next;
    unsigned long long acc;
    int have;

    __device__ __forceinline__ void start(const uint8_t* stream, long long length, long long bit) {
        s = stream;
        len = length;
        next = bit >> 3;
        acc = 0;
        have = 0;
        refill();
        const int drop = static_cast<int>(bit & 7);
        acc <<= drop;
        have -= drop;
    }
    __device__ __forceinline__ void refill() {
        while (have <= 56) {
            acc |= static_cast<unsigned long long>(aec_byte(s, len, next)) << (56 - have);
            ++next;
            have += 8;
        }
    }
    __device__ __forceinline__ long long pos() const { return next * 8 - have; }
    __device__ __forceinline__ uint32_t read(int w) {  // w <= 32
        refill();
        if (w == 0) return 0u;
        const uint32_t v = static_cast<uint32_t>(acc >> (64 - w));
        acc <<= w;
        have -= w;
        return v;
    }
    // one FS code: the count of zeros before the next one; ~0 when the stream ends first
    __device__ __forceinline__ unsigned long long fs() {
        unsigned long long m = 0;
        for (;;) {
            refill();
            if (acc == 0) {
                m += static_cast<unsigned long long>(have);
                have = 0;
                if (pos() > len * 8) return ~0ull;
                continue;
            }
            const int lz = __clzll(static_cast<long long>(acc));
            m += static_cast<unsigned long long>(lz);
            acc = (acc << lz) << 1;
            have -= lz + 1;
            return m;
        }
    }
};

// Where the decoded samples of one RSI go: postprocessing (inverse predictor mapping) and the
// big-endian 32-bit word of every sample below `end`.
struct AecSink {
    uint32_t* out;
    long long idx, end;
    uint32_t prev, xmax;
    bool pre;
    int error;

    __device__ __forceinline__ void put_reference(uint32_t x) {
        prev = x;
        if (idx < end) out[idx] = __byte_perm(x, 0, 0x0123);
        ++idx;
    }
    __device__ __forceinline__ void put(unsigned long long d) {
        if (d > xmax) {
            error = kCcsdsRange;
            return;
        }
        const uint32_t delta = static_cast<uint32_t>(d);
        uint32_t x = delta;
        if (pre) {
            const uint32_t theta = min(prev, xmax - prev);
            if (static_cast<unsigned long long>(delta) <= 2ull * theta)
                x = (delta & 1u) ? prev - ((delta >> 1) + 1u) : prev + (delta >> 1);
            else
                x = prev <= xmax - prev ? delta : xmax - delta;
            prev = x;
        }
        if (idx < end) out[idx] = __byte_perm(x, 0, 0x0123);
        ++idx;
    }
};

// One thread per (field, RSI): decode the RSI's blocks from its recorded offset.
__global__ void __launch_bounds__(kDecodeThreads)
    ccsds_decode_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (c.packing != AT_GRIB_CCSDS || c.aec_bits == 0 || c.n_values <= 0) return;
    if (*reinterpret_cast<volatile int32_t*>(err + blockIdx.x) != 0) return;  // the scan found the stream bad
    const int n = c.aec_bits, J = c.aec_block, rsi = c.aec_rsi, idlen = aec_id_length(n);
    const long long n_blocks = (c.n_values + J - 1) / J, n_rsi = (n_blocks + rsi - 1) / rsi;
    const long long limit = c.s7_length * 8;
    const unsigned long long* offsets = reinterpret_cast<const unsigned long long*>(packed + c.rsi_offset);
    for (long long r = static_cast<long long>(blockIdx.y) * kDecodeThreads + threadIdx.x; r < n_rsi;
         r += static_cast<long long>(gridDim.y) * kDecodeThreads) {
        AecReader rd;
        rd.start(packed + c.s7_offset, c.s7_length, static_cast<long long>(offsets[r]));
        AecSink out;
        out.out = reinterpret_cast<uint32_t*>(packed + c.byte_offset);
        out.idx = r * rsi * J;
        out.end = min(c.n_values, out.idx + static_cast<long long>(rsi) * J);
        out.prev = 0;
        out.xmax = n == 32 ? 0xffffffffu : ((1u << n) - 1u);
        out.pre = (c.aec_flags & kAecPreprocess) != 0;
        out.error = kCcsdsOk;
        int b = 0;
        while (out.idx < out.end && out.error == kCcsdsOk) {
            const int ref = (out.pre && b == 0) ? 1 : 0;
            const uint32_t id = rd.read(idlen);
            if (id == 0) {
                const uint32_t second = rd.read(1);
                if (ref) out.put_reference(rd.read(n));
                if (!second) {
                    const unsigned long long m = rd.fs();
                    if (m == ~0ull) {
                        out.error = kCcsdsTruncated;
                        break;
                    }
                    const long long z = static_cast<long long>(m) + 1;
                    const long long run = z == kAecRos ? min(rsi - b, kAecSegment - b % kAecSegment) : (z > kAecRos ? z - 1 : z);
                    if (b + run > rsi) {
                        out.error = kCcsdsZeroRun;
                        break;
                    }
                    const long long stop = min(out.end, out.idx + run * J - ref);
                    while (out.idx < stop) out.put(0);
                    b += static_cast<int>(run);
                    if (rd.pos() > limit) out.error = kCcsdsTruncated;
                    continue;
                }
                for (int i = 0; i < J / 2 && out.error == kCcsdsOk; ++i) {
                    const unsigned long long m = rd.fs();
                    if (m == ~0ull) {
                        out.error = kCcsdsTruncated;
                        break;
                    }
                    // m = s(s+1)/2 + b with s = a + b
                    long long sq = static_cast<long long>((sqrt(8.0 * static_cast<double>(m) + 1.0) - 1.0) * 0.5);
                    while (sq > 0 && static_cast<unsigned long long>(sq * (sq + 1) / 2) > m) --sq;
                    while (static_cast<unsigned long long>((sq + 1) * (sq + 2) / 2) <= m) ++sq;
                    const unsigned long long bb = m - static_cast<unsigned long long>(sq * (sq + 1) / 2);
                    if (!(ref && i == 0)) out.put(static_cast<unsigned long long>(sq) - bb);
                    out.put(bb);
                }
            } else if (id == (1u << idlen) - 1u) {
                if (ref) out.put_reference(rd.read(n));
                for (int i = ref; i < J; ++i) out.put(rd.read(n));
            } else {
                const int k = static_cast<int>(id) - 1;
                if (k >= n) {
                    out.error = kCcsdsBadOption;
                    break;
                }
                if (ref) out.put_reference(rd.read(n));
                // the k-bit LSBs follow all J - ref FS codes: a second reader walks the FS codes
                // while this one, moved past them, reads the LSBs
                AecReader lsb = rd;
                for (int i = ref; i < J; ++i)
                    if (lsb.fs() == ~0ull) {
                        out.error = kCcsdsTruncated;
                        break;
                    }
                if (out.error != kCcsdsOk) break;
                for (int i = ref; i < J; ++i) {
                    const unsigned long long fs = rd.fs();
                    const uint32_t low = lsb.read(k);
                    if (fs > (static_cast<unsigned long long>(out.xmax) >> k)) {
                        out.error = kCcsdsRange;
                        break;
                    }
                    out.put((fs << k) | low);
                }
                rd = lsb;
            }
            if (rd.pos() > limit) out.error = kCcsdsTruncated;
            ++b;
        }
        if (out.error != kCcsdsOk) fail_field(err + blockIdx.x, out.error);
    }
}

// ---- complex packing (templates 5.2 / 5.3): groups -> 32-bit words -------------------------
// Section 7 holds (5.3 only) the extra descriptors h1, [h2,] gmin, then NG group references,
// NG group widths and NG scaled group lengths (each part padded to an octet), then the values
// of every group back to back.  Nothing in it is serial: complex_groups_kernel turns lengths
// and widths into each group's first value and bit offset with block-wide scans, and
// complex_values_kernel gives every tile of kCxTile values its groups by binary search.
// Spatial differencing is a linear recurrence; with e_0 = h1, e_1 = h2 - 2·h1 and
// e_n = (X_n + gmin) after that, order 1 is X = prefix(e) and order 2 is X = prefix(prefix(e)).
// A tile acts on the incoming pair (D, X) = (last first difference, last value) as an affine
// map, so complex_tile_sums_kernel reduces every tile, complex_carry_kernel scans the tiles of
// a field, and complex_values_kernel applies each tile's carry.  All of it is two's-complement
// int64 arithmetic (unsigned here: the same bits), as in oracle/grib_complex.py.
constexpr int kCxGroupThreads = 1024;
constexpr int kCxThreads = 256;
constexpr int kCxPerThread = 8;
constexpr int kCxTile = kCxThreads * kCxPerThread;
constexpr int kCxTileWords = 4;  // per tile: sum of e, sum of inclusive prefixes of e, carry D, carry X

__host__ __device__ constexpr long long round256(long long n) { return (n + 255) / 256 * 256; }

struct CxTable {
    uint32_t* start;             // [NG + 1]: first value of every group, then the value count
    unsigned long long* bitoff;  // [NG]: bit offset of every group inside the values part
    unsigned long long* tiles;   // [kCxTileWords x tiles]
};

__device__ __forceinline__ CxTable cx_table(uint8_t* packed, const GribColumn& c) {
    uint8_t* t = packed + c.cx_table;
    CxTable tb;
    tb.start = reinterpret_cast<uint32_t*>(t);
    t += round256((c.cx_groups + 1) * 4);
    tb.bitoff = reinterpret_cast<unsigned long long*>(t);
    tb.tiles = reinterpret_cast<unsigned long long*>(t + round256(c.cx_groups * 8));
    return tb;
}

__device__ __forceinline__ bool cx_active(const GribColumn& c, const int32_t* err) {
    return c.packing == AT_GRIB_COMPLEX && c.n_values > 0 && *reinterpret_cast<const volatile int32_t*>(err + blockIdx.x) == 0;
}

// Extra descriptor k: ww octets, sign and magnitude.
__device__ __forceinline__ unsigned long long cx_descriptor(const uint8_t* s, long long len, int k, int ww) {
    unsigned long long u = 0;
    for (int i = 0; i < ww; ++i) u = (u << 8) | aec_byte(s, len, static_cast<long long>(k) * ww + i);
    const unsigned long long sign = 1ull << (8 * ww - 1);
    return (u & sign) ? 0ull - (u & (sign - 1)) : u;
}

// One block per field: every group's first value and bit offset, scanned kCxGroupThreads groups
// at a time with a carry.  The scan stops at the first group width above 32, or as soon as the
// lengths pass the value count or the bits pass section 7.
__global__ void __launch_bounds__(kCxGroupThreads)
    complex_groups_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (!cx_active(c, err)) return;
    __shared__ unsigned long long s_len[kCxGroupThreads / 32], s_bits[kCxGroupThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint8_t* s = packed + c.s7_offset;
    const long long len = c.s7_length, ng = c.cx_groups;
    const unsigned long long n = static_cast<unsigned long long>(c.n_values);
    const unsigned long long avail = static_cast<unsigned long long>(len - c.cx_values) * 8ull;
    const CxTable tb = cx_table(packed, c);
    unsigned long long carry_len = 0, carry_bits = 0;
    int status = kCcsdsOk;
    for (long long g0 = 0; g0 < ng; g0 += kCxGroupThreads) {
        const long long g = g0 + threadIdx.x;
        unsigned long long l = 0, b = 0;
        int bad = kCcsdsOk;
        if (g < ng) {
            const unsigned w = c.cx_width_ref + aec_bits(s, len, c.cx_widths * 8 + g * c.cx_width_bits, c.cx_width_bits);
            l = g == ng - 1 ? static_cast<unsigned long long>(c.cx_last_length)
                            : static_cast<unsigned long long>(c.cx_length_ref) +
                                  static_cast<unsigned long long>(c.cx_length_incr) * aec_bits(s, len, c.cx_lengths * 8 + g * c.cx_length_bits, c.cx_length_bits);
            if (w > 32) bad = kComplexWidth;
            else if (l > n) bad = kComplexLengths;
            if (bad != kCcsdsOk) {
                fail_field(err + blockIdx.x, bad);
                l = 0;
            }
            b = l * w;
        }
        unsigned long long il = l, ib = b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long ul = __shfl_up_sync(0xffffffffu, il, o), ub = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= o) {
                il += ul;
                ib += ub;
            }
        }
        if (lane == 31) {
            s_len[warp] = il;
            s_bits[warp] = ib;
        }
        const int any_bad = __syncthreads_or(bad);
        if (warp == 0) {
            unsigned long long wl = s_len[lane], wb = s_bits[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long ul = __shfl_up_sync(0xffffffffu, wl, o), ub = __shfl_up_sync(0xffffffffu, wb, o);
                if (lane >= o) {
                    wl += ul;
                    wb += ub;
                }
            }
            s_len[lane] = wl;
            s_bits[lane] = wb;
        }
        __syncthreads();
        const unsigned long long before_l = warp > 0 ? s_len[warp - 1] : 0ull, before_b = warp > 0 ? s_bits[warp - 1] : 0ull;
        if (g < ng) {
            tb.start[g] = static_cast<uint32_t>(carry_len + before_l + il - l);
            tb.bitoff[g] = carry_bits + before_b + ib - b;
        }
        carry_len += s_len[31];
        carry_bits += s_bits[31];
        __syncthreads();  // s_len / s_bits are rewritten by the next step
        if (any_bad) return;
        if (carry_len > n) {
            status = kComplexLengths;
            break;
        }
        if (carry_bits > avail) {
            status = kComplexOverrun;
            break;
        }
    }
    if (status == kCcsdsOk && carry_len != n) status = kComplexLengths;
    if (threadIdx.x == 0) {
        if (status != kCcsdsOk) fail_field(err + blockIdx.x, status);
        tb.start[ng] = static_cast<uint32_t>(n);
    }
}

// (sum of e, sum of its inclusive prefixes, count) of a run of values; `then` follows `first`.
struct CxSums {
    unsigned long long a, b, l;
};
__device__ __forceinline__ CxSums cx_combine(const CxSums& first, const CxSums& then) {
    return {first.a + then.a, first.b + then.b + then.l * first.a, first.l + then.l};
}

// Tile t of a complex field, one thread per kCxPerThread consecutive values: e (or X for 5.2)
// of every value, and the block's exclusive scan of the threads' sums.
struct CxTile {
    unsigned long long e[kCxPerThread];
    int count;
};

__device__ __forceinline__ void cx_load_tile(uint8_t* packed, const GribColumn& c, const CxTable& tb, long long t, CxTile& out) {
    const uint8_t* s = packed + c.s7_offset;
    const long long len = c.s7_length, ng = c.cx_groups;
    const long long i0 = t * kCxTile + static_cast<long long>(threadIdx.x) * kCxPerThread;
    out.count = static_cast<int>(max(0ll, min(static_cast<long long>(kCxPerThread), c.n_values - i0)));
    if (out.count == 0) return;
    // the last group that starts at or before i0 (empty groups start where the next one does)
    long long lo = 0, hi = ng - 1;
    while (lo < hi) {
        const long long mid = (lo + hi + 1) >> 1;
        if (static_cast<long long>(__ldg(tb.start + mid)) <= i0) lo = mid;
        else hi = mid - 1;
    }
    long long g = lo, first = __ldg(tb.start + g), next = __ldg(tb.start + g + 1);
    const int nbits = c.cx_nbits;
    unsigned long long ref = aec_bits(s, len, c.cx_refs * 8 + g * nbits, nbits);
    int width = c.cx_width_ref + static_cast<int>(aec_bits(s, len, c.cx_widths * 8 + g * c.cx_width_bits, c.cx_width_bits));
    AecReader rd;
    rd.start(s, len, c.cx_values * 8 + static_cast<long long>(__ldg(tb.bitoff + g)) + (i0 - first) * width);
    const int order = c.cx_order;
    unsigned long long h1 = 0, h2 = 0, gmin = 0;
    if (order > 0) {
        h1 = cx_descriptor(s, len, 0, c.cx_ww);
        if (order == 2) h2 = cx_descriptor(s, len, 1, c.cx_ww);
        gmin = cx_descriptor(s, len, order, c.cx_ww);
    }
#pragma unroll
    for (int k = 0; k < kCxPerThread; ++k) {
        const long long i = i0 + k;
        out.e[k] = 0;
        if (k >= out.count) continue;
        if (i >= next) {  // the next non-empty group
            do {
                ++g;
                first = next;
                next = __ldg(tb.start + g + 1);
            } while (i >= next);
            ref = aec_bits(s, len, c.cx_refs * 8 + g * nbits, nbits);
            width = c.cx_width_ref + static_cast<int>(aec_bits(s, len, c.cx_widths * 8 + g * c.cx_width_bits, c.cx_width_bits));
            rd.start(s, len, c.cx_values * 8 + static_cast<long long>(__ldg(tb.bitoff + g)));
        }
        const unsigned long long x = ref + rd.read(width);
        if (order == 0) out.e[k] = x;
        else if (i == 0) out.e[k] = h1;
        else if (i == 1 && order == 2) out.e[k] = h2 - 2ull * h1;
        else out.e[k] = x + gmin;
    }
}

// This thread's sums, and the block's exclusive scan of them (`total`: the whole tile's).
__device__ __forceinline__ CxSums cx_scan_tile(const CxTile& tl, CxSums& total) {
    __shared__ CxSums s_warp[kCxThreads / 32];
    CxSums mine{0, 0, static_cast<unsigned long long>(tl.count)};
#pragma unroll
    for (int k = 0; k < kCxPerThread; ++k) {
        mine.a += tl.e[k];
        mine.b += mine.a;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    CxSums inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const CxSums u{__shfl_up_sync(0xffffffffu, inc.a, o), __shfl_up_sync(0xffffffffu, inc.b, o), __shfl_up_sync(0xffffffffu, inc.l, o)};
        if (lane >= o) inc = cx_combine(u, inc);
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    CxSums before{0, 0, 0};
    for (int w = 0; w < warp; ++w) before = cx_combine(before, s_warp[w]);
    total = before;
    for (int w = warp; w < kCxThreads / 32; ++w) total = cx_combine(total, s_warp[w]);
    __syncthreads();  // s_warp is rewritten by the next tile
    CxSums ex{__shfl_up_sync(0xffffffffu, inc.a, 1), __shfl_up_sync(0xffffffffu, inc.b, 1), __shfl_up_sync(0xffffffffu, inc.l, 1)};
    if (lane == 0) ex = CxSums{0, 0, 0};
    return cx_combine(before, ex);
}

// Fields with spatial differencing: every tile's sums.  Grid (field, tiles strided).
__global__ void __launch_bounds__(kCxThreads)
    complex_tile_sums_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (!cx_active(c, err) || c.cx_order == 0) return;
    const CxTable tb = cx_table(packed, c);
    const long long n_tiles = (c.n_values + kCxTile - 1) / kCxTile;
    for (long long t = blockIdx.y; t < n_tiles; t += gridDim.y) {
        CxTile tl;
        cx_load_tile(packed, c, tb, t, tl);
        CxSums total;
        cx_scan_tile(tl, total);
        if (threadIdx.x == 0) {
            tb.tiles[kCxTileWords * t] = total.a;
            tb.tiles[kCxTileWords * t + 1] = total.b;
        }
    }
}

// One warp per field with spatial differencing: the pair (D, X) every tile starts from.
__global__ void __launch_bounds__(32)
    complex_carry_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (!cx_active(c, err) || c.cx_order == 0) return;
    const int lane = threadIdx.x;
    const CxTable tb = cx_table(packed, c);
    const long long n_tiles = (c.n_values + kCxTile - 1) / kCxTile;
    unsigned long long d = 0, x = 0;
    for (long long t0 = 0; t0 < n_tiles; t0 += 32) {
        const long long t = t0 + lane;
        CxSums mine{0, 0, 0};
        if (t < n_tiles)
            mine = CxSums{tb.tiles[kCxTileWords * t], tb.tiles[kCxTileWords * t + 1],
                          static_cast<unsigned long long>(min(static_cast<long long>(kCxTile), c.n_values - t * kCxTile))};
        CxSums inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const CxSums u{__shfl_up_sync(0xffffffffu, inc.a, o), __shfl_up_sync(0xffffffffu, inc.b, o), __shfl_up_sync(0xffffffffu, inc.l, o)};
            if (lane >= o) inc = cx_combine(u, inc);
        }
        CxSums ex{__shfl_up_sync(0xffffffffu, inc.a, 1), __shfl_up_sync(0xffffffffu, inc.b, 1), __shfl_up_sync(0xffffffffu, inc.l, 1)};
        if (lane == 0) ex = CxSums{0, 0, 0};
        if (t < n_tiles) {
            tb.tiles[kCxTileWords * t + 2] = d + ex.a;
            tb.tiles[kCxTileWords * t + 3] = x + ex.l * d + ex.b;
        }
        const CxSums all{__shfl_sync(0xffffffffu, inc.a, 31), __shfl_sync(0xffffffffu, inc.b, 31), __shfl_sync(0xffffffffu, inc.l, 31)};
        x += all.l * d + all.b;
        d += all.a;
    }
}

// Every value of every complex field as a big-endian 32-bit word in its scratch.  A final X
// outside [0, 2^32) sets the field's status word.  Grid (field, tiles strided).
__global__ void __launch_bounds__(kCxThreads)
    complex_values_kernel(uint8_t* __restrict__ packed, const GribColumn* __restrict__ cols, int32_t* __restrict__ err) {
    const GribColumn& c = cols[blockIdx.x];
    if (!cx_active(c, err)) return;
    const CxTable tb = cx_table(packed, c);
    uint32_t* out = reinterpret_cast<uint32_t*>(packed + c.byte_offset);
    const long long n_tiles = (c.n_values + kCxTile - 1) / kCxTile;
    const int order = c.cx_order;
    for (long long t = blockIdx.y; t < n_tiles; t += gridDim.y) {
        CxTile tl;
        cx_load_tile(packed, c, tb, t, tl);
        unsigned long long d = 0, x = 0;
        if (order > 0) {  // block-uniform
            CxSums total;
            const CxSums ex = cx_scan_tile(tl, total);
            const unsigned long long d_in = tb.tiles[kCxTileWords * t + 2], x_in = tb.tiles[kCxTileWords * t + 3];
            d = d_in + ex.a;
            x = x_in + ex.l * d_in + ex.b;
        }
        const long long i0 = t * kCxTile + static_cast<long long>(threadIdx.x) * kCxPerThread;
        bool bad = false;
#pragma unroll
        for (int k = 0; k < kCxPerThread; ++k) {
            if (k >= tl.count) break;
            d += tl.e[k];
            x += d;
            const unsigned long long v = order == 0 ? tl.e[k] : (order == 1 ? d : x);
            bad |= v > 0xffffffffull;  // as int64: negative or >= 2^32
            out[i0 + k] = bswap32(static_cast<uint32_t>(v));
        }
        if (bad) fail_field(err + blockIdx.x, kComplexRange);
    }
}

int complex_decode_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int32_t* d_err, long long max_tiles, cudaStream_t st) {
    if (n_fields == 0 || max_tiles <= 0) return AT_OK;
    const unsigned nf = static_cast<unsigned>(n_fields);
    const dim3 grid(nf, static_cast<unsigned>(std::min<long long>(max_tiles, 65535)));
    complex_groups_kernel<<<nf, kCxGroupThreads, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("complex_groups_kernel");
    complex_tile_sums_kernel<<<grid, kCxThreads, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("complex_tile_sums_kernel");
    complex_carry_kernel<<<nf, 32, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("complex_carry_kernel");
    complex_values_kernel<<<grid, kCxThreads, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("complex_values_kernel");
    return AT_OK;
}

const char* grib_status_text(int32_t code) {
    switch (code) {
        case kCcsdsTruncated: return "the AEC stream ends before the last value";
        case kCcsdsBadOption: return "a split-sample option with k >= bits per value";
        case kCcsdsZeroRun: return "a zero-block run leaves its reference sample interval";
        case kCcsdsRange: return "a decoded sample exceeds 2^bits - 1";
        case kComplexLengths: return "the group lengths do not add up to the value count";
        case kComplexOverrun: return "the packed values run past section 7";
        case kComplexWidth: return "a group width above 32 bits";
        case kComplexRange: return "a decoded integer outside [0, 2^32)";
        case kBitmapCount: return "the bitmap has more set bits than the message has values";
        default: return "malformed section 7";
    }
}

int ccsds_decode_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int32_t* d_err, long long max_rsi, cudaStream_t st) {
    if (n_fields == 0 || max_rsi <= 0) return AT_OK;
    ccsds_rsi_scan_kernel<<<static_cast<unsigned>(n_fields), 32, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("ccsds_rsi_scan_kernel");
    const long long per_field = (max_rsi + kDecodeThreads - 1) / kDecodeThreads;
    const dim3 grid(static_cast<unsigned>(n_fields), static_cast<unsigned>(std::min<long long>(per_field, 65535)));
    ccsds_decode_kernel<<<grid, kDecodeThreads, 0, st>>>(d_packed, d_cols, d_err);
    AT_LAUNCH_CHECK("ccsds_decode_kernel");
    return AT_OK;
}

template <typename TOut, bool BITMAPS>
static int launch_unpack(const uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int64_t n_points, TOut* out, int64_t ld,
                         unsigned grid, unsigned n_field_groups, cudaStream_t st) {
    const size_t smem = sizeof(TOut) * kTileFields * (kTilePoints + 1);
    if (smem > 48 * 1024) {  // above the default: opt in (idempotent)
        AT_CUDA_TRY(cudaFuncSetAttribute(grib_unpack_kernel<TOut, BITMAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    }
    grib_unpack_kernel<TOut, BITMAPS><<<grid, 256, smem, st>>>(d_packed, d_cols, n_fields, n_points, out, ld, n_field_groups);
    AT_LAUNCH_CHECK("grib_unpack_kernel");
    return AT_OK;
}

int grib_unpack_launch(uint8_t* d_packed, const GribColumn* d_cols, int n_fields, int64_t n_points, int out_dtype, void* d_pm,
                       int64_t ld, bool any_bitmap, int32_t* d_err, cudaStream_t st) {
    if (n_fields == 0 || n_points == 0) return AT_OK;
    const unsigned n_field_groups = static_cast<unsigned>((n_fields + kTileFields - 1) / kTileFields);
    const long long blocks = ((n_points + kTilePoints - 1) / kTilePoints) * n_field_groups;
    if (blocks >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "GRIB unpack: batch too large for one launch");
    const unsigned grid = static_cast<unsigned>(blocks);
    if (any_bitmap) {
        grib_bitmap_rank_kernel<<<static_cast<unsigned>(n_fields), 32, 0, st>>>(d_packed, d_cols, n_points, d_err);
        AT_LAUNCH_CHECK("grib_bitmap_rank_kernel");
        if (out_dtype == AT_F32) return launch_unpack<float, true>(d_packed, d_cols, n_fields, n_points, static_cast<float*>(d_pm), ld, grid, n_field_groups, st);
        return launch_unpack<double, true>(d_packed, d_cols, n_fields, n_points, static_cast<double*>(d_pm), ld, grid, n_field_groups, st);
    }
    if (out_dtype == AT_F32) return launch_unpack<float, false>(d_packed, d_cols, n_fields, n_points, static_cast<float*>(d_pm), ld, grid, n_field_groups, st);
    return launch_unpack<double, false>(d_packed, d_cols, n_fields, n_points, static_cast<double*>(d_pm), ld, grid, n_field_groups, st);
}

static size_t round_up_256(size_t n) { return (n + 255) / 256 * 256; }

static bool is_ccsds(const at_grib_field_t& info) { return info.packing == AT_GRIB_CCSDS && info.bits_per_value > 0; }
static bool is_complex(const at_grib_field_t& info) { return info.packing == AT_GRIB_COMPLEX; }

int64_t complex_tile_count(int64_t n_values) { return n_values > 0 ? (n_values + kCxTile - 1) / kCxTile : 0; }

int64_t ccsds_rsi_count(const at_grib_field_t& info, int64_t n_values) {
    if (!is_ccsds(info) || n_values <= 0 || info.ccsds_block_size <= 0 || info.ccsds_rsi <= 0) return 0;
    const int64_t blocks = (n_values + info.ccsds_block_size - 1) / info.ccsds_block_size;
    return (blocks + info.ccsds_rsi - 1) / info.ccsds_rsi;
}

GribFootprint grib_footprint(const at_grib_field_t& info, int64_t n_points) {
    GribFootprint fp;
    const int64_t n_values = info.has_bitmap ? (info.n_values >= 0 ? info.n_values : n_points) : n_points;
    int64_t octets = (n_values * std::max(info.bits_per_value, 0) + 7) / 8;
    if (info.has_bitmap && info.n_values < 0) octets = std::max<int64_t>(info.data_length, 0);  // count unknown: the whole section
    if (is_ccsds(info) || is_complex(info)) octets = std::max<int64_t>(info.data_length, 0);  // all of section 7
    fp.value_octets = static_cast<size_t>(std::min<int64_t>(octets, std::max<int64_t>(info.data_length, 0)));
    fp.values = round_up_256(fp.value_octets + 16);
    if (is_ccsds(info))  // device only: the decoded words (+ the unpack's 16 octets of slack) and the RSI offsets
        fp.scratch = round_up_256(static_cast<size_t>(std::max<int64_t>(n_values, 0)) * 4 + 16) +
                     round_up_256(static_cast<size_t>(ccsds_rsi_count(info, n_values)) * 8);
    if (is_complex(info))  // the decoded words, then the group starts and bit offsets and the tile sums
        fp.scratch = round_up_256(static_cast<size_t>(std::max<int64_t>(n_values, 0)) * 4 + 16) +
                     static_cast<size_t>(round256((info.complex_groups + 1) * 4) + round256(info.complex_groups * 8) +
                                         round256(complex_tile_count(n_values) * kCxTileWords * 8));
    if (info.has_bitmap) {
        fp.bitmap_octets = static_cast<size_t>((n_points + 7) / 8);
        fp.bitmap = round_up_256(fp.bitmap_octets + 32);
        fp.ranks = round_up_256(static_cast<size_t>((n_points + kTilePoints - 1) / kTilePoints + 1) * sizeof(uint32_t));
    }
    return fp;
}

int grib_column_of(const at_grib_field_t& info, int64_t n_points, int64_t byte_offset, GribColumn* out) {
    AT_REQUIRE(info.bits_per_value >= 0 && info.bits_per_value <= 32, "GRIB unpack: bitsPerValue %d out of range", info.bits_per_value);
    AT_REQUIRE(info.packing == AT_GRIB_SIMPLE || info.packing == AT_GRIB_CCSDS || info.packing == AT_GRIB_COMPLEX, "GRIB unpack: unknown packing %d",
               info.packing);
    const GribFootprint fp = grib_footprint(info, n_points);
    const bool ccsds = is_ccsds(info), cx = is_complex(info);
    *out = GribColumn{};
    if (info.packing == AT_GRIB_CCSDS) {
        const int rc = ccsds_check(info, "GRIB unpack: template 5.42");
        if (rc != AT_OK) return rc;
    }
    if (cx) {  // the host scan's checks, again: the table comes from the caller
        AT_REQUIRE(info.complex_groups >= 0 && info.complex_groups <= std::max<int64_t>(info.n_values, 0) && info.complex_width_bits >= 0 &&
                       info.complex_width_bits <= 32 && info.complex_length_bits >= 0 && info.complex_length_bits <= 32 &&
                       (info.complex_groups > 0 || info.n_values == 0) && info.complex_order >= 0 && info.complex_order <= 2 &&
                       (info.complex_order == 0 || (info.complex_ww >= 1 && info.complex_ww <= 4)),
                   "GRIB unpack: complex packing parameters out of range");
        AT_REQUIRE(info.complex_refs_offset >= 0 && info.complex_refs_offset <= info.complex_widths_offset &&
                       info.complex_widths_offset <= info.complex_lengths_offset && info.complex_lengths_offset <= info.complex_values_offset &&
                       info.complex_values_offset <= info.data_length,
                   "GRIB unpack: complex packing: the group descriptors do not fit section 7");
    }
    if (ccsds || cx) {  // the packed length says nothing about the value count: check the counts alone
        const int64_t n_values = info.has_bitmap ? info.n_values : n_points;
        AT_REQUIRE(info.n_values >= 0 && (info.has_bitmap ? info.n_values <= n_points : info.n_values == n_points),
                   "GRIB unpack: message holds %lld values, the batch has %lld points", (long long)info.n_values, (long long)n_points);
        if (info.has_bitmap)
            AT_REQUIRE((info.n_points < 0 || info.n_points == n_points) && info.bitmap_offset >= 0 &&
                           info.bitmap_offset + static_cast<int64_t>(fp.bitmap_octets) <= info.message_length,
                       "GRIB unpack: the bitmap does not fit the message or the batch");
        const int64_t scratch = byte_offset + static_cast<int64_t>(fp.values + fp.bitmap + fp.ranks);
        out->byte_offset = scratch;
        out->bitmap_offset = info.has_bitmap ? byte_offset + static_cast<int64_t>(fp.values) : -1;
        out->rank_offset = info.has_bitmap ? byte_offset + static_cast<int64_t>(fp.values + fp.bitmap) : -1;
        out->reference = info.reference_value;
        out->binary = repeated_power(info.binary_scale, 2);
        out->decimal = repeated_power(-info.decimal_scale, 10);
        out->nbits = 32;
        out->packing = info.packing;
        out->s7_offset = byte_offset;
        out->s7_length = static_cast<long long>(fp.value_octets);
        out->n_values = n_values;
        const int64_t tables = scratch + static_cast<int64_t>(round_up_256(static_cast<size_t>(n_values) * 4 + 16));
        if (ccsds) {
            out->rsi_offset = tables;
            out->aec_bits = info.bits_per_value;
            out->aec_flags = info.ccsds_flags;
            out->aec_block = info.ccsds_block_size;
            out->aec_rsi = info.ccsds_rsi;
            out->cx_table = -1;
            return AT_OK;
        }
        out->rsi_offset = -1;
        out->cx_table = tables;
        out->cx_groups = info.complex_groups;
        out->cx_length_ref = info.complex_length_ref;
        out->cx_last_length = info.complex_last_length;
        out->cx_refs = info.complex_refs_offset;
        out->cx_widths = info.complex_widths_offset;
        out->cx_lengths = info.complex_lengths_offset;
        out->cx_values = info.complex_values_offset;
        out->cx_nbits = info.bits_per_value;
        out->cx_width_ref = info.complex_width_ref;
        out->cx_width_bits = info.complex_width_bits;
        out->cx_length_bits = info.complex_length_bits;
        out->cx_length_incr = info.complex_length_incr;
        out->cx_order = info.complex_order;
        out->cx_ww = info.complex_ww;
        return AT_OK;
    }
    if (info.has_bitmap) {
        AT_REQUIRE(info.n_points < 0 || info.n_points == n_points, "GRIB unpack: the bitmap covers %lld points, the batch has %lld",
                   (long long)info.n_points, (long long)n_points);
        AT_REQUIRE(info.n_values <= n_points, "GRIB unpack: %lld values for %lld points", (long long)info.n_values, (long long)n_points);
        AT_REQUIRE(info.bitmap_offset >= 0 && info.bitmap_offset + static_cast<int64_t>(fp.bitmap_octets) <= info.message_length,
                   "GRIB unpack: the bitmap runs past the end of the message");
        if (info.n_values >= 0)
            AT_REQUIRE(info.data_length >= (info.n_values * info.bits_per_value + 7) / 8, "GRIB unpack: %lld octets of packed values, %lld needed",
                       (long long)info.data_length, (long long)((info.n_values * info.bits_per_value + 7) / 8));
    } else {
        AT_REQUIRE(info.n_values < 0 || info.n_values == n_points, "GRIB unpack: message holds %lld values, the batch has %lld points",
                   (long long)info.n_values, (long long)n_points);
        const int64_t need = (n_points * info.bits_per_value + 7) / 8;
        AT_REQUIRE(info.data_length >= need, "GRIB unpack: %lld octets of packed values, %lld needed", (long long)info.data_length, (long long)need);
    }
    out->byte_offset = byte_offset;
    out->bitmap_offset = info.has_bitmap ? byte_offset + static_cast<int64_t>(fp.values) : -1;
    out->rank_offset = info.has_bitmap ? byte_offset + static_cast<int64_t>(fp.values + fp.bitmap) : -1;
    out->reference = info.reference_value;
    out->binary = repeated_power(info.binary_scale, 2);
    out->decimal = repeated_power(-info.decimal_scale, 10);
    out->nbits = info.bits_per_value;
    out->packing = AT_GRIB_SIMPLE;  // a constant CCSDS field (0 bits) is decoded like simple packing
    out->s7_offset = out->s7_length = out->rsi_offset = -1;
    // the values the staged octets hold: a bitmap with more set bits is refused on the device
    out->n_values = n_points;
    if (info.has_bitmap && info.bits_per_value > 0)
        out->n_values = info.n_values >= 0 ? info.n_values : static_cast<int64_t>(fp.value_octets) * 8 / info.bits_per_value;
    out->aec_bits = out->aec_flags = out->aec_block = out->aec_rsi = 0;
    out->cx_table = -1;
    return AT_OK;
}

}  // namespace at

using namespace at;

extern "C" int at_grib_scan(const void* message, size_t length, at_grib_field_t* out) {
    AT_REQUIRE(message != nullptr && out != nullptr, "at_grib_scan: null argument");
    std::memset(out, 0, sizeof(*out));
    out->bitmap_offset = -1;
    out->n_points = out->n_values = -1;
    const uint8_t* m = static_cast<const uint8_t*>(message);
    AT_REQUIRE(length >= 8 && std::memcmp(m, "GRIB", 4) == 0, "at_grib_scan: not a GRIB message");
    const int edition = m[7];
    if (edition == 2) return scan_edition2(m, length, out);
    if (edition == 1) return scan_edition1(m, length, out);
    return set_error(AT_ERR_UNSUPPORTED, "at_grib_scan: GRIB edition %d", edition);
}

extern "C" int at_grib_scan_many(const void* const* messages, const size_t* lengths, int64_t n, at_grib_field_t* out, int32_t* status) {
    AT_REQUIRE(n >= 0, "at_grib_scan_many: negative count");
    if (n == 0) return AT_OK;
    AT_REQUIRE(messages != nullptr && lengths != nullptr && out != nullptr && status != nullptr, "at_grib_scan_many: null argument");
    for (int64_t i = 0; i < n; ++i) status[i] = messages[i] != nullptr ? at_grib_scan(messages[i], lengths[i], out + i) : AT_ERR_INVALID;
    return AT_OK;
}

extern "C" int at_grib_unpack(const void* d_packed, const int64_t* byte_offsets, const at_grib_field_t* fields, int64_t n_fields,
                              int64_t n_points, int out_dtype, void* d_pm, int64_t ld, void* stream) {
    AT_REQUIRE(n_fields >= 0 && n_points >= 0, "at_grib_unpack: negative size");
    AT_REQUIRE(out_dtype == AT_F32 || out_dtype == AT_F64, "at_grib_unpack: bad dtype code");
    if (n_fields == 0 || n_points == 0) return AT_OK;
    AT_REQUIRE(d_packed != nullptr && byte_offsets != nullptr && fields != nullptr && d_pm != nullptr, "at_grib_unpack: null argument");
    AT_REQUIRE(ld >= n_fields && n_fields < (1ll << 31), "at_grib_unpack: bad leading dimension");
    std::vector<GribColumn> cols(static_cast<size_t>(n_fields));
    for (int64_t f = 0; f < n_fields; ++f) {
        AT_REQUIRE(byte_offsets[f] >= 0, "at_grib_unpack: negative offset");
        AT_REQUIRE(fields[f].has_bitmap == 0, "at_grib_unpack: messages with a bitmap go through at_hostio_upload_grib / at_hostio_regrid_grib (they stage the bitmap too)");
        if (fields[f].packing == AT_GRIB_CCSDS)
            return set_error(AT_ERR_UNSUPPORTED, "at_grib_unpack: message %lld is CCSDS-packed (template 5.42): it goes through at_hostio_upload_grib / at_hostio_regrid_grib (they decode the AEC stream)", (long long)f);
        if (fields[f].packing == AT_GRIB_COMPLEX)
            return set_error(AT_ERR_UNSUPPORTED, "at_grib_unpack: message %lld uses complex packing (template 5.2 / 5.3): it goes through at_hostio_upload_grib / at_hostio_regrid_grib (they decode the groups)", (long long)f);
        const int rc = grib_column_of(fields[f], n_points, byte_offsets[f], &cols[static_cast<size_t>(f)]);
        if (rc != AT_OK) return rc;
    }
    GribColumn* d_cols = nullptr;
    AT_CUDA_TRY(device_alloc(reinterpret_cast<void**>(&d_cols), cols.size() * sizeof(GribColumn)));
    cudaStream_t st = as_stream(stream);
    cudaError_t e = cudaMemcpyAsync(d_cols, cols.data(), cols.size() * sizeof(GribColumn), cudaMemcpyHostToDevice, st);
    int rc = AT_OK;
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // `cols` is pageable and leaves scope
    if (e != cudaSuccess) rc = set_error(AT_ERR_CUDA, "at_grib_unpack: %s", cudaGetErrorString(e));
    if (rc == AT_OK)
        rc = grib_unpack_launch(const_cast<uint8_t*>(static_cast<const uint8_t*>(d_packed)), d_cols, static_cast<int>(n_fields), n_points, out_dtype, d_pm, ld, false, nullptr, st);
    device_free(d_cols);  // waits for the device, like cudaFree
    return rc;
}

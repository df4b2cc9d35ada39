// masks.cu — mask machinery of anemoi.transform.spatial that is not the neighbour search:
// the cropping box, the per-point classification of cutout_mask (Möller–Trumbore ray /
// triangle tests against the k nearest LAM points), and byte-mask -> sorted-index
// compaction.
//
// Reference (src/anemoi/transform/spatial.py):
//   cropping_mask            236-275
//   Triangle3D.intersect     189-233
//   cutout_mask loop body    404-424
//   np.array(sorted(set(…))) 534 (global_on_lam_mask), boolean selection 380-381, 487-488
#include <algorithm>

#include "common.cuh"

namespace at {

__global__ void cropping_mask_kernel(const double* __restrict__ lats, const double* __restrict__ lons,
                                     long long n, double north, double west, double south, double east,
                                     double west_p, double east_p, double west_m, double east_m,
                                     uint8_t* __restrict__ mask) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double la = lats[i], lo = lons[i];
    const bool in_lat = (la >= south) && (la <= north);
    const bool in_lon = ((lo >= west) && (lo <= east)) || ((lo >= west_p) && (lo <= east_p)) ||
                        ((lo >= west_m) && (lo <= east_m));
    mask[i] = (in_lat && in_lon) ? 1 : 0;
}

struct V3 {
    double x, y, z;
};

__device__ __forceinline__ V3 sub(V3 a, V3 b) {
    return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)};
}
// np.cross: each product rounded, then subtracted (never fused).
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
    return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)),
            __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
            __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
// np.dot on two float64 3-vectors goes to BLAS ddot.  FMA: OpenBLAS' x86-64 kernels
// accumulate fma(a2,b2, fma(a1,b1, a0*b0)); otherwise plain left-to-right.
template <bool FMA>
__device__ __forceinline__ double dot(V3 a, V3 b) {
    if (FMA) return __fma_rn(a.z, b.z, __fma_rn(a.y, b.y, __dmul_rn(a.x, b.x)));
    return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}

// Triangle3D(v0, v1, v2).intersect(ray_origin = 0, ray_direction = dir)
template <bool FMA>
__device__ __forceinline__ bool ray_hits(V3 v0, V3 v1, V3 v2, V3 dir) {
    const double eps = 0.0000001;
    const V3 e2 = sub(v2, v0);
    const V3 h = cross(dir, e2);
    const V3 e1 = sub(v1, v0);
    const double a = dot<FMA>(e1, h);
    if (-eps < a && a < eps) return false;
    const double f = __ddiv_rn(1.0, a);
    const V3 zero = {0.0, 0.0, 0.0};
    const V3 s = sub(zero, v0);
    const double u = __dmul_rn(f, dot<FMA>(s, h));
    if (u < 0.0 || u > 1.0) return false;
    const V3 q = cross(s, e1);
    const double v = __dmul_rn(f, dot<FMA>(dir, q));
    if (v < 0.0 || __dadd_rn(u, v) > 1.0) return false;
    const double t = __dmul_rn(f, dot<FMA>(e2, q));
    return t > eps;
}

template <bool FMA>
__global__ void __launch_bounds__(128)
    cutout_classify_kernel(const double* __restrict__ lx, const double* __restrict__ ly,
                           const double* __restrict__ lz, long long n_lam, const double* __restrict__ gx,
                           const double* __restrict__ gy, const double* __restrict__ gz, long long nq,
                           const long long* __restrict__ nbr_idx, const double* __restrict__ nbr_dist, int k,
                           double min_distance, double max_distance, int first_triangle,
                           uint8_t* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const V3 g = {gx[i], gy[i], gz[i]};
    const long long* idx = nbr_idx + i * k;
    const double* dist = nbr_dist + i * k;

    double dmin = dist[0];
    for (int j = 1; j < k; ++j) dmin = fmin(dmin, dist[j]);  // np.min (no NaN on this path)

    bool inside = false;
    for (int j = first_triangle; j < k && !inside; ++j) {
        const long long i0 = idx[j], i1 = idx[(j + 1) % k], i2 = idx[(j + 2) % k];
        if (i0 >= n_lam || i1 >= n_lam || i2 >= n_lam) continue;  // host raised IndexError already
        const V3 v0 = {lx[i0], ly[i0], lz[i0]};
        const V3 v1 = {lx[i1], ly[i1], lz[i1]};
        const V3 v2 = {lx[i2], ly[i2], lz[i2]};
        inside = ray_hits<FMA>(v0, v1, v2, g);
    }
    const bool close = dmin <= min_distance;
    const bool too_far = max_distance >= 0.0 && dmin > max_distance;
    out[i] = (inside || close || too_far) ? 1 : 0;
}

// ---- byte mask -> sorted indices -------------------------------------------------------
constexpr int kChunk = 4096;  // bytes per block: 256 threads x 16

__device__ __forceinline__ int count_nonzero_bytes(uint4 v) {
    auto nz = [](uint32_t w) {
        // number of non-zero bytes in w
        uint32_t t = (w | (w >> 4)) & 0x0f0f0f0fu;
        t = (t | (t >> 2)) & 0x03030303u;
        t = (t | (t >> 1)) & 0x01010101u;
        return __popc(t);
    };
    return nz(v.x) + nz(v.y) + nz(v.z) + nz(v.w);
}

__device__ __forceinline__ uint4 load_chunk16(const uint8_t* __restrict__ mark, long long n, long long base) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (base + 16 <= n && (reinterpret_cast<uintptr_t>(mark + base) & 15) == 0) {
        v = *reinterpret_cast<const uint4*>(mark + base);
    } else if (base < n) {
        uint8_t b[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) b[j] = base + j < n ? mark[base + j] : 0;
        memcpy(&v, b, 16);
    }
    return v;
}

__global__ void __launch_bounds__(256) compact_count_kernel(const uint8_t* __restrict__ mark, long long n,
                                                            int32_t* __restrict__ block_counts) {
    __shared__ int warp_tot[8];
    const long long base = static_cast<long long>(blockIdx.x) * kChunk + threadIdx.x * 16;
    int c = count_nonzero_bytes(load_chunk16(mark, n, base));
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < 8; ++w) t += warp_tot[w];
        block_counts[blockIdx.x] = t;
    }
}

// Single block: exclusive scan of block counts (int64 offsets), total to *total.
__global__ void __launch_bounds__(1024) compact_scan_kernel(const int32_t* __restrict__ counts, int n_blocks,
                                                            long long* __restrict__ offsets,
                                                            long long* __restrict__ total) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n_blocks; base += 1024) {
        const int i = base + threadIdx.x;
        const long long v = i < n_blocks ? counts[i] : 0;
        long long inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) warp_tot[warp] = inc;
        __syncthreads();
        long long woff = 0;
        for (int w = 0; w < warp; ++w) woff += warp_tot[w];
        const long long carry = carry_s;
        if (i < n_blocks) offsets[i] = carry + woff + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + woff + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry_s;
}

__global__ void __launch_bounds__(256) compact_write_kernel(const uint8_t* __restrict__ mark, long long n,
                                                            const long long* __restrict__ offsets,
                                                            long long* __restrict__ out_idx) {
    __shared__ int warp_tot[8];
    const long long base = static_cast<long long>(blockIdx.x) * kChunk + threadIdx.x * 16;
    const uint4 v = load_chunk16(mark, n, base);
    const int c = count_nonzero_bytes(v);
    int inc = c;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += warp_tot[w];
    long long pos = offsets[blockIdx.x] + woff + inc - c;
    if (c == 0) return;
    uint8_t b[16];
    memcpy(b, &v, 16);
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (b[j] != 0) out_idx[pos++] = base + j;
}

}  // namespace at

using namespace at;

extern "C" int at_cropping_mask(const double* lats, const double* lons, int64_t n, double north, double west,
                                double south, double east, uint8_t* mask, void* stream) {
    AT_REQUIRE(n >= 0, "at_cropping_mask: negative size");
    if (n == 0) return AT_OK;  // zero-length device arrays have null pointers
    AT_REQUIRE(lats != nullptr && lons != nullptr && mask != nullptr, "at_cropping_mask: null argument");
    const int64_t blocks = (n + 255) / 256;
    AT_REQUIRE(blocks < (1ll << 31), "at_cropping_mask: too large");
    // the ±360 bounds are formed on the host in float64 exactly as numpy evaluates west + 360 …
    cropping_mask_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(
        lats, lons, n, north, west, south, east, west + 360, east + 360, west - 360, east - 360, mask);
    AT_LAUNCH_CHECK("cropping_mask_kernel");
    return AT_OK;
}

extern "C" int at_cutout_classify(const double* lx, const double* ly, const double* lz, int64_t n_lam,
                                  const double* gx, const double* gy, const double* gz, int64_t nq,
                                  const int64_t* nbr_idx, const double* nbr_dist, int k, double min_distance,
                                  double max_distance, int dot_mode, uint8_t* out, void* stream) {
    AT_REQUIRE(k >= 1 && k <= 32, "at_cutout_classify: neighbours must be in [1, 32]");
    AT_REQUIRE(nq >= 0 && n_lam >= 1, "at_cutout_classify: bad sizes");
    AT_REQUIRE(dot_mode == 0 || dot_mode == 1, "at_cutout_classify: dot_mode must be 0 or 1");
    if (nq == 0) return AT_OK;  // zero-length device arrays have null pointers
    AT_REQUIRE(lx && ly && lz && gx && gy && gz && nbr_idx && nbr_dist && out, "at_cutout_classify: null argument");
    const int64_t blocks = (nq + 127) / 128;
    AT_REQUIRE(blocks < (1ll << 31), "at_cutout_classify: too large");
    const long long* idx = reinterpret_cast<const long long*>(nbr_idx);
    if (dot_mode == 1)
        cutout_classify_kernel<true><<<static_cast<unsigned>(blocks), 128, 0, as_stream(stream)>>>(
            lx, ly, lz, n_lam, gx, gy, gz, nq, idx, nbr_dist, k, min_distance, max_distance, 0, out);
    else
        cutout_classify_kernel<false><<<static_cast<unsigned>(blocks), 128, 0, as_stream(stream)>>>(
            lx, ly, lz, n_lam, gx, gy, gz, nq, idx, nbr_dist, k, min_distance, max_distance, 0, out);
    AT_LAUNCH_CHECK("cutout_classify_kernel");
    return AT_OK;
}

extern "C" int at_outline_classify(const double* x, const double* y, const double* z, int64_t n,
                                   const int64_t* nbr_idx, const double* nbr_dist, int k, int dot_mode, uint8_t* out,
                                   void* stream) {
    AT_REQUIRE(k >= 1 && k <= 32, "at_outline_classify: neighbours must be in [1, 32]");
    AT_REQUIRE(n >= 0, "at_outline_classify: bad size");
    AT_REQUIRE(dot_mode == 0 || dot_mode == 1, "at_outline_classify: dot_mode must be 0 or 1");
    if (n == 0) return AT_OK;
    AT_REQUIRE(x && y && z && nbr_idx && nbr_dist && out, "at_outline_classify: null argument");
    const int64_t blocks = (n + 127) / 128;
    AT_REQUIRE(blocks < (1ll << 31), "at_outline_classify: too large");
    const long long* idx = reinterpret_cast<const long long*>(nbr_idx);
    // the same triangle fan as cutout_mask over the point's own neighbours, starting at the second
    // neighbour (the first is the point itself) and with both distance tests switched off
    if (dot_mode == 1)
        cutout_classify_kernel<true><<<static_cast<unsigned>(blocks), 128, 0, as_stream(stream)>>>(
            x, y, z, n, x, y, z, n, idx, nbr_dist, k, -1.0, -1.0, 1, out);
    else
        cutout_classify_kernel<false><<<static_cast<unsigned>(blocks), 128, 0, as_stream(stream)>>>(
            x, y, z, n, x, y, z, n, idx, nbr_dist, k, -1.0, -1.0, 1, out);
    AT_LAUNCH_CHECK("cutout_classify_kernel");
    return AT_OK;
}

extern "C" int at_compact_mask(const uint8_t* mark, int64_t n, int64_t* out_idx, int64_t* count_host,
                               void* stream) {
    AT_REQUIRE(count_host != nullptr, "at_compact_mask: null argument");
    AT_REQUIRE(n >= 0, "at_compact_mask: negative size");
    *count_host = 0;
    if (n == 0) return AT_OK;  // zero-length device arrays have null pointers
    AT_REQUIRE(mark != nullptr && out_idx != nullptr, "at_compact_mask: null argument");
    cudaStream_t st = as_stream(stream);
    const int64_t blocks = (n + kChunk - 1) / kChunk;
    AT_REQUIRE(blocks < (1ll << 31), "at_compact_mask: too large");
    int32_t* d_counts = nullptr;
    long long* d_offsets = nullptr;
    AT_CUDA_TRY(device_alloc(reinterpret_cast<void**>(&d_counts), static_cast<size_t>(blocks) * 4));
    cudaError_t e = device_alloc(reinterpret_cast<void**>(&d_offsets), (static_cast<size_t>(blocks) + 1) * 8);
    if (e != cudaSuccess) {
        device_free(d_counts);
        return set_error(AT_ERR_NOMEM, "at_compact_mask: %s", cudaGetErrorString(e));
    }
    compact_count_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(mark, n, d_counts);
    compact_scan_kernel<<<1, 1024, 0, st>>>(d_counts, static_cast<int>(blocks), d_offsets, d_offsets + blocks);
    compact_write_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(mark, n, d_offsets,
                                                                       reinterpret_cast<long long*>(out_idx));
    e = cudaGetLastError();
    long long total = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, d_offsets + blocks, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    device_free(d_counts);
    device_free(d_offsets);
    if (e != cudaSuccess) return set_error(AT_ERR_CUDA, "at_compact_mask: %s", cudaGetErrorString(e));
    *count_host = total;
    return AT_OK;
}

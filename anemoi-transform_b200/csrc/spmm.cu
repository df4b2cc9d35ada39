// spmm.cu — the regrid hot loop: a CSR interpolation matrix staged once in HBM and applied
// to a point-major batch of fields, Y[n_tgt, F] = A · X[n_src, F].
//
// Replaces scipy.sparse csr_matvec behind `self.matrix @ data`
// (reference src/anemoi/transform/filters/fields/regrid.py:309-310), batched over the
// per-field Python loop of RegridFilter._interpolate (regrid.py:204-208).
//
// Layout / mapping (see DESIGN.md §3):
//   - X, Y row-major [points, fields]; one nonzero's weight multiplies a contiguous row
//     of fields, read as coalesced 16-byte vectors;
//   - one warp per target row per column tile (32·VPL float4 = 128·VPL fields);
//   - a CTA owns `rows_per_cta` consecutive target rows; their CSR segment (column indices
//     and weights, contiguous in memory) is staged in shared memory once per CTA — with a
//     1-D bulk async copy (TMA, cp.async.bulk + mbarrier) when the matrix has a uniform
//     row length, so the tile is regular and 16-byte aligned, else with cooperative loads;
//   - blockIdx.x = row_block * S + tile_in_supertile: CTAs that are resident together cover S
//     adjacent column tiles of neighbouring rows (long contiguous spans of each source row,
//     DRAM page locality) and the ~2x re-reference of each source row hits L2; S is sized from
//     the matrix's reuse working set; blockIdx.y walks the super-tiles;
//   - float64 results (float64 matrix and / or fields) run spmm_f64_kernel, same mapping with
//     16-byte units of X; the pointwise filters run in the epilogue (spmm_fused_kernel) or on
//     their own (pointwise_kernel), compiled per kind family (epilogue.cuh);
//   - accumulation is scipy's, bit for bit: sequential in storage order from +0 with
//     __fmul_rn / __fadd_rn (never contracted to FMA);
//   - Y is write-once: streaming stores (st.global.cs).
#include <algorithm>
#include <type_traits>
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "epilogue.cuh"

struct at_csr {
    int64_t n_rows = 0, n_cols = 0, nnz = 0;
    int data_dtype = AT_F32;
    int uniform_nnz = 0;
    int max_row_nnz = 0;
    int max_seg64 = 0;  // largest number of entries in any aligned block of 64 rows
    double live_cols = 0;  // average number of source columns between their first and last use
    int32_t* d_indptr = nullptr;   // n_rows + 1 (+ padding)
    int32_t* d_indices = nullptr;  // nnz (+ padding)
    void* d_data = nullptr;        // nnz float or double (+ padding)
    int device = 0;
};

namespace at {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / kWarp;
constexpr int kMaxRowsPerCta = 64;
constexpr int kSegCap = 1024;  // CSR entries staged per CTA (8 KB of smem)
constexpr int kPad = 64;       // padding entries behind the device CSR arrays
constexpr int kDefaultVPL = 2;  // float4 per lane per nonzero of variant 0 (and of at_spmm_missing)

// ---- mbarrier / bulk-copy (TMA 1-D) primitives --------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

struct SpmmArgs {
    const int32_t* __restrict__ indptr;
    const int32_t* __restrict__ indices;
    const float* __restrict__ data;
    const float4* __restrict__ X;
    float4* __restrict__ Y;
    size_t ldx4, ldy4;  // leading dimensions in float4
    int n_rows;
    int n_vec;          // F / 4 (float4 columns), rounded up
    int rows_per_cta;
    int super;          // column tiles per super-tile: blockIdx.x walks (row block, tile in super-tile)
};

// (Blackwell's packed mul.rn.f32x2 / add.rn.f32x2 would halve these instructions, but ptxas 12.9
// contracts the pair into one FFMA2 even with -fmad=false, which breaks bit-exactness with scipy's
// unfused accumulation; measured gain of the contracted form was 1 % — the kernel is HBM-bound.)
__device__ __forceinline__ float4 mul_add_rn(float4 acc, float w, float4 x) {
    acc.x = __fadd_rn(acc.x, __fmul_rn(w, x.x));
    acc.y = __fadd_rn(acc.y, __fmul_rn(w, x.y));
    acc.z = __fadd_rn(acc.z, __fmul_rn(w, x.z));
    acc.w = __fadd_rn(acc.w, __fmul_rn(w, x.w));
    return acc;
}

// ---- missing values (at_spmm_missing) --------------------------------------------------
// The kernels take the policy MP as a template argument: 0 is the plain SpMM (its code is
// untouched), AT_MISSING_ALL / AT_MISSING_HEAVIEST skip NaN sources.  Per lane and field a
// missing-aware row carries Σ′w·x in the accumulator, Σ′w beside it and a "some entry missing"
// bit.  The heaviest entry (largest weight, the first in storage order on ties: a strict `>`)
// depends on the weights only, so it is found once per row from the staged weights, outside the
// entry loop; after the row each lane reads its x at that entry's column again (the line the row
// has just read: an L1 / L2 hit, no HBM bytes) and sets a "heaviest missing" bit.  Following the
// maximum inside the loop cost 25 % on conservative rows (O1280 -> N320-like, float32).
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

template <typename T>
__device__ __forceinline__ void skip_add(T& acc, T& ws, uint32_t& miss, uint32_t bit, T w, T x) {
    const bool nan = isnan(x);
    if (!nan) {
        acc = add_rn(acc, mul_rn(w, x));
        ws = add_rn(ws, w);
    }
    if (nan) miss |= bit;
}

// y of one (row, field): the plain sum when nothing was missing, else Σ′w·x / Σ′w or NaN
template <typename T>
__device__ __forceinline__ T missing_result(T acc, T ws, uint32_t miss, uint32_t heavy, uint32_t bit) {
    if ((miss & bit) == 0) return acc;
    if ((heavy & bit) != 0 || !(ws > T(0))) return quiet_nan(T(0));
    return div_rn(acc, ws);
}

// Position of the heaviest of entries [p0, p1) (weight(p) reads entry p), -1 for an empty row.
template <typename WeightAt>
__device__ __forceinline__ int heaviest_entry(int p0, int p1, WeightAt weight) {
    int best = -1;
    double wmax = 0.0;  // float weights widen exactly: the same order
    for (int p = p0; p < p1; ++p) {
        const double w = static_cast<double>(weight(p));
        if (best < 0 || w > wmax) wmax = w, best = p;
    }
    return best;
}

template <int VPL>
struct MissF4 {
    float4 ws[VPL];
    uint32_t miss, heavy;  // bit 4v + e: float4 v, component e
    __device__ __forceinline__ MissF4() : miss(0), heavy(0) {
#pragma unroll
        for (int v = 0; v < VPL; ++v) ws[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __device__ __forceinline__ void add(float4& acc, int v, float w, const float4& x) {
        skip_add(acc.x, ws[v].x, miss, 1u << (4 * v), w, x.x);
        skip_add(acc.y, ws[v].y, miss, 2u << (4 * v), w, x.y);
        skip_add(acc.z, ws[v].z, miss, 4u << (4 * v), w, x.z);
        skip_add(acc.w, ws[v].w, miss, 8u << (4 * v), w, x.w);
    }
    // the row's heaviest entry reads source row `col` (-1: empty row)
    __device__ __forceinline__ void mark_heaviest(const float4* __restrict__ X, size_t ldx4, int col, const int (&vcol)[VPL], const bool (&vok)[VPL]) {
        if (col < 0) return;
        const float4* xr = X + static_cast<size_t>(col) * ldx4;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            if (!vok[v]) continue;
            const float4 x = ld_ro_f4(xr + vcol[v]);
            heavy |= (isnan(x.x) ? 1u : 0u) << (4 * v) | (isnan(x.y) ? 2u : 0u) << (4 * v) | (isnan(x.z) ? 4u : 0u) << (4 * v) | (isnan(x.w) ? 8u : 0u) << (4 * v);
        }
    }
    __device__ __forceinline__ float4 result(const float4& acc, int v) const {
        return make_float4(missing_result(acc.x, ws[v].x, miss, heavy, 1u << (4 * v)), missing_result(acc.y, ws[v].y, miss, heavy, 2u << (4 * v)),
                           missing_result(acc.z, ws[v].z, miss, heavy, 4u << (4 * v)), missing_result(acc.w, ws[v].w, miss, heavy, 8u << (4 * v)));
    }
};

// Stage the CTA's CSR segment in shared memory.  Returns the base entry (segment start).
// UNNZ > 0: uniform row length, regular tile -> bulk async copy when BULK.
template <int UNNZ, bool BULK, bool FALLBACK>
__device__ __forceinline__ void stage_segment(const SpmmArgs& a, int r0, int nrows, int* s_ptr,
                                              int* s_idx, float* s_w, uint64_t* s_bar,
                                              int& seg_base, bool& in_smem) {
    const int tid = threadIdx.x;
    if (UNNZ > 0) {
        seg_base = r0 * UNNZ;
        const int len = nrows * UNNZ;
        in_smem = true;  // host guarantees rows_per_cta * UNNZ <= kSegCap
        if (BULK) {
            // Regular tile: base is a multiple of 4 entries (rows_per_cta % 4 == 0), length is
            // rounded up to 16 bytes (arrays are padded), so both copies are 16-byte aligned.
            const uint32_t bytes = static_cast<uint32_t>((len * 4 + 15) & ~15);
            if (tid == 0) {
                mbar_init(s_bar, 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncthreads();
            if (tid == 0) {
                mbar_expect_tx(s_bar, 2 * bytes);
                bulk_g2s(s_idx, a.indices + seg_base, bytes, s_bar);
                bulk_g2s(s_w, a.data + seg_base, bytes, s_bar);
            }
            mbar_wait(s_bar, 0);
        } else {
            for (int i = tid; i < len; i += kThreads) {
                s_idx[i] = __ldg(a.indices + seg_base + i);
                s_w[i] = __ldg(a.data + seg_base + i);
            }
            __syncthreads();
        }
    } else {
        for (int i = tid; i <= nrows; i += kThreads) s_ptr[i] = __ldg(a.indptr + r0 + i);
        __syncthreads();
        seg_base = s_ptr[0];
        const int len = s_ptr[nrows] - seg_base;
        // without FALLBACK the host has checked that every CTA's segment fits (max_seg64)
        in_smem = !FALLBACK || len <= kSegCap;
        if (in_smem) {
            for (int i = tid; i < len; i += kThreads) {
                s_idx[i] = __ldg(a.indices + seg_base + i);
                s_w[i] = __ldg(a.data + seg_base + i);
            }
        }
        __syncthreads();
    }
}

// Accumulate one target row for this lane's VPL float4 columns.
// (p0, p1) are entry offsets relative to the staged segment when IN_SMEM, absolute otherwise.
// MP != 0: missing-aware (Σ′), with the rest of the lane's state in *m.
template <int VPL, int U, bool IN_SMEM, int MP = 0>
__device__ __forceinline__ void accumulate_row(const SpmmArgs& a, int p0, int p1,
                                               const int* s_idx, const float* s_w,
                                               const int (&vcol)[VPL], const bool (&vok)[VPL],
                                               float4 (&acc)[VPL], MissF4<VPL>* m = nullptr) {
    for (int p = p0; p < p1; p += U) {
        int c[U];
        float w[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const bool ok = p + j < p1;
            if (IN_SMEM) {
                c[j] = ok ? s_idx[p + j] : 0;
                w[j] = ok ? s_w[p + j] : 0.0f;
            } else {
                c[j] = ok ? __ldg(a.indices + p + j) : 0;
                w[j] = ok ? __ldg(a.data + p + j) : 0.0f;
            }
        }
        float4 x[U][VPL];
        // Issue every gather of the chunk before the first dependent add.
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const float4* xr = a.X + static_cast<size_t>(c[j]) * a.ldx4;
#pragma unroll
            for (int v = 0; v < VPL; ++v)
                if (vok[v] && p + j < p1) x[j][v] = ld_ro_f4(xr + vcol[v]);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (p + j < p1) {
                if constexpr (MP == 0) {
#pragma unroll
                    for (int v = 0; v < VPL; ++v) acc[v] = mul_add_rn(acc[v], w[j], x[j][v]);
                } else {
#pragma unroll
                    for (int v = 0; v < VPL; ++v) m->add(acc[v], v, w[j], x[j][v]);
                }
            }
        }
    }
}

template <int VPL, int UNNZ, bool BULK, bool FALLBACK, int MP>
__global__ void __launch_bounds__(kThreads) spmm_f32_kernel(const SpmmArgs a) {
    __shared__ __align__(16) int s_idx[kSegCap];
    __shared__ __align__(16) float s_w[kSegCap];
    __shared__ int s_ptr[kMaxRowsPerCta + 1];
    __shared__ __align__(8) uint64_t s_bar;

    // blockIdx.x = row_block * super + tile_in_super: CTAs that run together cover `super`
    // adjacent column tiles of the same rows, i.e. super·VPL·512 contiguous bytes per source row.
    const int tile = blockIdx.y * a.super + static_cast<int>(blockIdx.x % a.super);
    const int r0 = static_cast<int>(blockIdx.x / a.super) * a.rows_per_cta;
    const int nrows = min(a.rows_per_cta, a.n_rows - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (tile * (kWarp * VPL) >= a.n_vec) return;

    int vcol[VPL];
    bool vok[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        vcol[v] = tile * (kWarp * VPL) + v * kWarp + lane;
        vok[v] = vcol[v] < a.n_vec;
    }

    int seg_base;
    bool in_smem;
    stage_segment<UNNZ, BULK, FALLBACK>(a, r0, nrows, s_ptr, s_idx, s_w, &s_bar, seg_base, in_smem);

    // AT_MISSING_HEAVIEST: the column of each row's heaviest entry, one thread per row, once per CTA
    int* s_hcol = nullptr;
    if constexpr (MP == AT_MISSING_HEAVIEST) {
        __shared__ int s_heavy_col[kMaxRowsPerCta];
        s_hcol = s_heavy_col;
        for (int lr = threadIdx.x; lr < nrows; lr += kThreads) {
            int col = -1;
            if (UNNZ > 0 || !FALLBACK || in_smem) {
                const int p0 = UNNZ > 0 ? lr * UNNZ : s_ptr[lr] - seg_base, p1 = UNNZ > 0 ? (lr + 1) * UNNZ : s_ptr[lr + 1] - seg_base;
                const int h = heaviest_entry(p0, p1, [&](int p) { return s_w[p]; });
                if (h >= 0) col = s_idx[h];
            } else {
                const int h = heaviest_entry(s_ptr[lr], s_ptr[lr + 1], [&](int p) { return __ldg(a.data + p); });
                if (h >= 0) col = __ldg(a.indices + h);
            }
            s_hcol[lr] = col;
        }
        __syncthreads();
    }

    // The ragged last tile of a batch (3120 fields are twelve tiles of 64 float4 and one of 12):
    // when it fills half a warp or less, several target rows share the warp — lane -> (float4
    // column v, row sub), every lane walking the CSR entries of its own row — instead of leaving
    // most lanes idle for the whole row block.  Full tiles keep the warp-uniform loop below.
    // (Config 3 at 1560 fields: 1.440 -> 1.422 ms; 3120 fields: 2.880 -> 2.876 ms.  The same
    // change in spmm_f64_kernel measured slower — 1.256 -> 1.34 ms for float64 weights on 780
    // float32 fields — and was not kept.)
    const int nv_here = min(kWarp * VPL, a.n_vec - tile * (kWarp * VPL));
    if (nv_here <= kWarp / 2) {
        int vbits = 4;
        while (vbits > 0 && (1 << (vbits - 1)) >= nv_here) --vbits;
        const int rpw = kWarp >> vbits;
        const int pcol[1] = {tile * (kWarp * VPL) + (lane & ((1 << vbits) - 1))};
        const bool pok[1] = {(lane & ((1 << vbits) - 1)) < nv_here};
        for (int lr = warp * rpw + (lane >> vbits); lr < nrows; lr += kWarps * rpw) {
            float4 acc[1] = {make_float4(0.f, 0.f, 0.f, 0.f)};
            MissF4<1> m;
            if constexpr (UNNZ > 0) {
                accumulate_row<1, (UNNZ < 4 ? UNNZ : 4), true, MP>(a, lr * UNNZ, (lr + 1) * UNNZ, s_idx, s_w, pcol, pok, acc, &m);
            } else if (!FALLBACK || in_smem) {
                accumulate_row<1, 4, true, MP>(a, s_ptr[lr] - seg_base, s_ptr[lr + 1] - seg_base, s_idx, s_w, pcol, pok, acc, &m);
            } else {
                accumulate_row<1, 4, false, MP>(a, s_ptr[lr], s_ptr[lr + 1], s_idx, s_w, pcol, pok, acc, &m);
            }
            if constexpr (MP == AT_MISSING_HEAVIEST) m.mark_heaviest(a.X, a.ldx4, s_hcol[lr], pcol, pok);
            if constexpr (MP != 0) acc[0] = m.result(acc[0], 0);
            if (pok[0]) st_stream_f4(a.Y + static_cast<size_t>(r0 + lr) * a.ldy4 + pcol[0], acc[0]);
        }
        return;
    }

    for (int lr = warp; lr < nrows; lr += kWarps) {
        float4 acc[VPL];
#pragma unroll
        for (int v = 0; v < VPL; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        MissF4<VPL> m;

        if constexpr (UNNZ > 0) {
            accumulate_row<VPL, (UNNZ < 4 ? UNNZ : 4), true, MP>(a, lr * UNNZ, (lr + 1) * UNNZ, s_idx,
                                                                 s_w, vcol, vok, acc, &m);
        } else if (!FALLBACK || in_smem) {
            accumulate_row<VPL, 4, true, MP>(a, s_ptr[lr] - seg_base, s_ptr[lr + 1] - seg_base, s_idx,
                                             s_w, vcol, vok, acc, &m);
        } else {
            accumulate_row<VPL, 4, false, MP>(a, s_ptr[lr], s_ptr[lr + 1], s_idx, s_w, vcol, vok, acc, &m);
        }
        if constexpr (MP == AT_MISSING_HEAVIEST) m.mark_heaviest(a.X, a.ldx4, s_hcol[lr], vcol, vok);
        if constexpr (MP != 0) {
#pragma unroll
            for (int v = 0; v < VPL; ++v) acc[v] = m.result(acc[v], v);
        }

        float4* yr = a.Y + static_cast<size_t>(r0 + lr) * a.ldy4;
#pragma unroll
        for (int v = 0; v < VPL; ++v)
            if (vok[v]) st_stream_f4(yr + vcol[v], acc[v]);
    }
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- fused epilogue variant: general CSR, one float4 per lane, tile table ------------
struct FusedArgs {
    SpmmArgs s;
    const EpiTile* __restrict__ tiles;
    const ColF32* __restrict__ cols;
    const uint8_t* __restrict__ row_mask;
    float* __restrict__ Yf;
    size_t ldy;  // in floats
};

// One warp per target row, one entry of the tile table per CTA (32 lanes x 4 input columns,
// CTA-uniform kind), 64 registers so 4 CTAs stay resident per SM.  Measured alternatives on
// config 4 (fused uv_to_ddff / q_to_r / clip / mask, 4.2 ms): two table entries per CTA (epilogue
// inlined twice, 116 registers, 2 CTAs / SM) 5.0 ms; two rows per warp step with one epilogue
// copy (8 gathers in flight, spills at 64 registers) 5.9 ms, 4.3 ms at 80 registers / 3 CTAs.
template <int UNNZ, bool FALLBACK, uint32_t FAM>
__global__ void __launch_bounds__(kThreads, 4) spmm_fused_kernel(const FusedArgs f) {
    __shared__ __align__(16) int s_idx[kSegCap];
    __shared__ __align__(16) float s_w[kSegCap];
    __shared__ int s_ptr[kMaxRowsPerCta + 1];
    __shared__ __align__(8) uint64_t s_bar;

    // Same grid order as spmm_f32_kernel.
    const SpmmArgs& a = f.s;
    const int t_index = blockIdx.y * a.super + static_cast<int>(blockIdx.x % a.super);
    const int r0 = static_cast<int>(blockIdx.x / a.super) * a.rows_per_cta;
    const int nrows = min(a.rows_per_cta, a.n_rows - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (t_index >= a.n_vec) return;  // n_vec = number of tile-table entries here

    const EpiTile tile = f.tiles[t_index];
    // A tile narrower than half a warp (the ragged end of a segment) packs several target rows
    // into the warp, lane -> (column group v, row sub), instead of idling its lanes; every lane
    // then walks the CSR entries of its own row.
    int vbits = 5;
    while (vbits > 0 && (1 << (vbits - 1)) >= tile.n_vec) --vbits;
    const int v = lane & ((1 << vbits) - 1), rpw = kWarp >> vbits;
    const int rfirst = warp * rpw + (lane >> vbits), rstep = kWarps * rpw;  // this lane's rows
    int vcol[1] = {tile.in_vec0 + v};
    bool vok[1] = {v < tile.n_vec};

    int seg_base;
    bool in_smem;
    stage_segment<UNNZ, UNNZ != 0, FALLBACK>(a, r0, nrows, s_ptr, s_idx, s_w, &s_bar, seg_base, in_smem);

    const EpiLane<float> lane_prm = epilogue_prepare<float>(tile, v, f.cols);
    const bool any_mask = (tile.flags_any & AT_COL_MASK) != 0 && f.row_mask != nullptr;

    // The kind is CTA-uniform: dispatch it once, outside the row loop, so each loop is compiled for
    // its kind (no switch per row, row-invariant tests hoisted); every kind's code exists once.
    auto rows = [&](auto kind_c) {
        EpiTile tk = tile;
        if constexpr (decltype(kind_c)::value >= 0) tk.kind = decltype(kind_c)::value;
        // Clip bounds and mask bits of the lane's outputs in registers (the kind is known here, so
        // only its outputs' bounds stay live) instead of a read of the per-column table per row and
        // output: 2.91 -> 2.44 ms on a program with flags on every column.  The 12-nonzero
        // instantiation has no registers to spare (it spills more and loses 1 %): it keeps the reads.
        constexpr bool kHoist = UNNZ < 8;
        EpiClip<float> clip;
        if constexpr (kHoist) clip = epilogue_prepare_clip<float>(tk, v, f.cols);
        float* yrow = f.Yf + static_cast<size_t>(r0 + rfirst) * f.ldy;
        const size_t ystep = static_cast<size_t>(rstep) * f.ldy;
        for (int lr = rfirst; lr < nrows; lr += rstep, yrow += ystep) {
            float4 acc[1] = {make_float4(0.f, 0.f, 0.f, 0.f)};
            if constexpr (UNNZ > 0) {
                accumulate_row<1, 4, true>(a, lr * UNNZ, (lr + 1) * UNNZ, s_idx, s_w, vcol, vok, acc);
            } else if (!FALLBACK || in_smem) {
                accumulate_row<1, 4, true>(a, s_ptr[lr] - seg_base, s_ptr[lr + 1] - seg_base, s_idx, s_w, vcol, vok, acc);
            } else {
                accumulate_row<1, 4, false>(a, s_ptr[lr], s_ptr[lr + 1], s_idx, s_w, vcol, vok, acc);
            }
            const bool masked = any_mask && f.row_mask[r0 + lr] != 0;
            // The warp has no gather in flight while it runs the epilogue (the 64-register cap
            // leaves no room for a second row of loads).  Rows of many nonzeros scattered over a
            // large source grid (config 4: 12 per row over 6.6 M points) wait on DRAM for every
            // gather: ask L2 for the source rows of the warp's next target row now.  Measured:
            // config 4 fused 4.05 -> 3.85 ms (the plain SpMM takes 3.81); on 4-nonzero bilinear rows,
            // whose re-referenced source rows already sit in L2, the extra instructions cost
            // 5 % (3.19 -> 3.34 ms on a 2/3-transcendental program), so those do not prefetch.
            if constexpr (UNNZ >= 8) {
                if (lr + rstep < nrows && vok[0]) {
#pragma unroll
                    for (int j = 0; j < UNNZ; ++j) prefetch_l2(a.X + static_cast<size_t>(s_idx[(lr + rstep) * UNNZ + j]) * a.ldx4 + vcol[0]);
                }
            }
            if (vok[0]) epilogue_store<float, kHoist, FAM>(tk, v, acc[0].x, acc[0].y, acc[0].z, acc[0].w, lane_prm, f.cols, masked, yrow, &clip);
        }
    };
#define AT_FUSED_KIND(K)                                                       \
    case K:                                                                    \
        if constexpr ((FAM & kind_bit(K)) != 0) rows(std::integral_constant<int, K>{}); \
        break;
    switch (tile.kind) {
        AT_FUSED_KIND(AT_EPI_PLAIN)
        AT_FUSED_KIND(AT_EPI_UV2DDFF)
        AT_FUSED_KIND(AT_EPI_DDFF2UV)
        AT_FUSED_KIND(AT_EPI_QT2R)
        AT_FUSED_KIND(AT_EPI_QT2QTR)
        AT_FUSED_KIND(AT_EPI_RT2Q)
        AT_FUSED_KIND(AT_EPI_RT2RTQ)
        AT_FUSED_KIND(AT_EPI_COSSIN)
        AT_FUSED_KIND(AT_EPI_ATAN2)
        AT_FUSED_KIND(AT_EPI_RT2D)
        AT_FUSED_KIND(AT_EPI_RT2RTD)
        AT_FUSED_KIND(AT_EPI_DT2R)
        AT_FUSED_KIND(AT_EPI_DT2DTR)
        default:  // the unary kinds share one loop (their switch is four selects)
            rows(std::integral_constant<int, -1>{});
            break;
    }
#undef AT_FUSED_KIND
}

// ---- pointwise on a resident batch (identity "matrix") --------------------------------
template <typename T>
struct PointwiseArgs {
    const EpiTile* __restrict__ tiles;
    const typename ColStore<T>::type* __restrict__ cols;
    const uint8_t* __restrict__ row_mask;
    const T* __restrict__ X;
    T* __restrict__ Y;
    const long long* __restrict__ row_index;  // output row r reads input row row_index[r] (NULL: r)
    size_t ldx, ldy;
    long long n_rows;
    int rows_per_cta;
    int n_tiles;
    int uses_es;  // the program has a (q, t) <-> r kind: stage the es(T) table in shared memory
};

__device__ __forceinline__ void load4(const float* p, float& a, float& b, float& c, float& d) {
    const float4 v = ld_ro_f4(reinterpret_cast<const float4*>(p));
    a = v.x, b = v.y, c = v.z, d = v.w;
}
__device__ __forceinline__ void load4(const double* p, double& a, double& b, double& c, double& d) {
    const double2 v0 = __ldg(reinterpret_cast<const double2*>(p));
    const double2 v1 = __ldg(reinterpret_cast<const double2*>(p) + 1);
    a = v0.x, b = v0.y, c = v1.x, d = v1.y;
}

// Warp w of a CTA owns tile-table entry blockIdx.y * 8 + w (32 lanes x 4 input columns, one
// kind) for all of the CTA's rows: the 8 warps together read 4 KB of contiguous columns per row
// (DRAM page locality), and everything row-invariant (pressures, clip bounds, mask bits) lives
// in registers.  Both paths are bound by bytes in flight before anything else (HBM latency x
// bandwidth is ~35 KB per SM): copy-like tiles (clip / mask, affine, impute) keep kPwRows rows
// of loads in flight in registers; transcendental tiles, which have no registers to spare at the
// 64-register cap (4 CTAs per SM), keep kPwAhead rows in flight in shared memory instead —
// cp.async (LDGSTS) into a per-lane ring, 16 bytes per lane and row, read back by the lane that
// copied them (no barrier, no bank conflict) — behind a row loop compiled once per kind.
// (Measured, profiles/r02_pw_ring_depth_sweep.log: 1 / 2 / 4 rows in flight -> uv_to_ddff 0.60 /
// 0.81 / 0.87 of the HBM peak, 6 and 8 add nothing; the per-kind loops then reach 1.00.)
constexpr int kPwRows = 4;
constexpr int kPwCtaRows = 32;  // rows per CTA (launch_pointwise)
#ifndef AT_PW_AHEAD
#define AT_PW_AHEAD 4
#endif
constexpr int kPwAhead = AT_PW_AHEAD;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
// a lane's 4 columns of one row: global -> its ring slot (asynchronously), ring slot -> registers
__device__ __forceinline__ void ring_fetch(uint32_t slot, const float* p) { cp_async16(slot, p); }
__device__ __forceinline__ void ring_fetch(uint32_t slot, const double* p) {
    cp_async16(slot, p);
    cp_async16(slot + 16, p + 2);
}
__device__ __forceinline__ void ring_read(uint32_t slot, float& a, float& b, float& c, float& d) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "r"(slot) : "memory");
}
__device__ __forceinline__ void ring_read(uint32_t slot, double& a, double& b, double& c, double& d) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(slot) : "memory");
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(c), "=d"(d) : "r"(slot + 16) : "memory");
}

template <typename T, uint32_t FAM>
__global__ void __launch_bounds__(kThreads, sizeof(T) == 4 ? 4 : 2) pointwise_kernel(const PointwiseArgs<T> f) {
    constexpr int kSlot = 4 * sizeof(T);  // bytes a lane owns per row
    constexpr int kAhead = sizeof(T) == 4 ? kPwAhead : (kPwAhead < 4 ? kPwAhead : 4);  // float64: 2 CTAs per SM of twice the bytes
    __shared__ __align__(16) unsigned char s_ring[kWarps * kAhead * kWarp * kSlot];
    __shared__ uint8_t s_mask[kPwCtaRows];
    // es(T) cubics of the float32 humidity fast paths (epilogue.cuh): 32 lanes look up 32 different
    // entries, which costs the L1 up to 32 sectors per warp load and shared memory a few wavefronts
    __shared__ __align__(16) float4 s_es[sizeof(T) == 4 ? kEsTableN : 1];
    const long long r0 = static_cast<long long>(blockIdx.x) * kPwCtaRows;
    const int nrows = static_cast<int>(min(static_cast<long long>(kPwCtaRows), f.n_rows - r0));
    // the CTA's slice of the row mask and the table, once (before any warp leaves: every thread reaches the barrier)
    const bool stage_es = sizeof(T) == 4 && f.uses_es != 0;
    if (f.row_mask != nullptr || stage_es) {
        if (f.row_mask != nullptr && threadIdx.x < nrows) s_mask[threadIdx.x] = f.row_mask[r0 + threadIdx.x];
        if (stage_es)
            for (int i = threadIdx.x; i < kEsTableN; i += kThreads) s_es[i] = g_es_mixed_table[i];
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // A CTA covers up to 8 table entries; when fewer are left (narrow batches) the spare warps
    // take a share of the rows instead of idling: warp w -> entry w % t_here, row group w / t_here.
    const int t_here = min(kWarps, f.n_tiles - static_cast<int>(blockIdx.y) * kWarps);
    const int groups = kWarps / t_here, group = warp / t_here;
    if (group >= groups) return;
    const EpiTile tile = f.tiles[blockIdx.y * kWarps + warp % t_here];
    // A tile narrower than half a warp (the ragged end of a segment: 520 columns are four full
    // tiles and one of 2 lanes) packs several rows into the warp instead of idling its lanes:
    // lane -> (column group v, row sub) with `rpw` rows per warp step.
    int vbits = 5;
    while (vbits > 0 && (1 << (vbits - 1)) >= tile.n_vec) --vbits;
    const int v = lane & ((1 << vbits) - 1), sub = lane >> vbits, rpw = kWarp >> vbits;
    if (v >= tile.n_vec) return;
    const int rfirst = group * rpw + sub, rstep = groups * rpw;  // this lane's rows: rfirst, rfirst + rstep, ...
    const bool any_mask = f.row_mask != nullptr && (tile.flags_any & AT_COL_MASK) != 0;
    const T* xcol = f.X + 4 * static_cast<size_t>(tile.in_vec0 + v);
    const EpiClip<T> clip = epilogue_prepare_clip<T>(tile, v, f.cols);
    // nearest-neighbour / masked regrid fused with the pointwise program: a row gather on the way in
    const long long* __restrict__ rix = f.row_index;
    auto src_row = [rix](long long r) { return rix != nullptr ? __ldg(rix + r) : r; };

    // one-in / one-out kinds with next to no arithmetic (clip / mask only, affine, impute) are
    // latency-bound copies: kPwRows rows of loads in flight, the small switch inlined once per row
    constexpr uint32_t kCopyLike = kind_bit(AT_EPI_PLAIN) | kind_bit(AT_EPI_AFFINE) | kind_bit(AT_EPI_AFFINE_INV) | kind_bit(AT_EPI_IMPUTE_NAN);
    if ((kind_bit(tile.kind) & kCopyLike) != 0) {
        const EpiLane<T> none = {T(0), T(0)};
        for (int lr = rfirst; lr < nrows; lr += rstep * kPwRows) {
            T a[kPwRows][4];
            bool masked[kPwRows];
#pragma unroll
            for (int j = 0; j < kPwRows; ++j) {
                masked[j] = false;
                if (lr + j * rstep < nrows) {
                    load4(xcol + static_cast<size_t>(src_row(r0 + lr + j * rstep)) * f.ldx, a[j][0], a[j][1], a[j][2], a[j][3]);
                    if (any_mask) masked[j] = s_mask[lr + j * rstep] != 0;
                }
            }
#pragma unroll
            for (int j = 0; j < kPwRows; ++j)
                if (lr + j * rstep < nrows)
                    epilogue_store<T, true, FAM & kCopyLike>(tile, v, a[j][0], a[j][1], a[j][2], a[j][3], none, f.cols, masked[j],
                                                            f.Y + static_cast<size_t>(r0 + lr + j * rstep) * f.ldy, &clip);
        }
        return;
    }

    const EpiLane<T> lane_prm = epilogue_prepare<T>(tile, v, f.cols);
    if (rfirst >= nrows) return;
    // Transcendental kinds: a ring of kAhead rows in flight behind the epilogue.  The kind is
    // dispatched once per warp, outside the row loop, so each loop is compiled for its kind (no
    // switch per row, row-invariant range tests hoisted) and every kind's code still exists once.
    // Addresses advance by additions; slot k of a lane is refilled only after the epilogue has
    // consumed the values read from it.
    const uint32_t ring0 = static_cast<uint32_t>(__cvta_generic_to_shared(s_ring)) + (warp * kAhead * kWarp + lane) * kSlot;
    const uint32_t ring_end = ring0 + kAhead * (kWarp * kSlot);
    const uint32_t smask0 = static_cast<uint32_t>(__cvta_generic_to_shared(s_mask)) + rfirst;
    auto rows = [&](auto kind_c) {
        EpiTile tk = tile;
        tk.kind = decltype(kind_c)::value;
        EpiLane<T> lp = lane_prm;
        constexpr int K = decltype(kind_c)::value;
        if constexpr (sizeof(T) == 4 && (K == AT_EPI_QT2R || K == AT_EPI_QT2QTR || K == AT_EPI_RT2Q || K == AT_EPI_RT2RTQ)) lp.es_table = s_es;
#pragma unroll
        for (int j = 0; j < kAhead; ++j) {
            const int lr = rfirst + j * rstep;
            if (lr < nrows) ring_fetch(ring0 + j * (kWarp * kSlot), xcol + static_cast<size_t>(src_row(r0 + lr)) * f.ldx);
            cp_async_commit();  // one group per row, empty or not, so the wait below counts rows
        }
        uint32_t slot = ring0, smask = smask0;
        const size_t xstep = static_cast<size_t>(rstep) * f.ldx, ystep = static_cast<size_t>(rstep) * f.ldy;
        const T* xnext = xcol + static_cast<size_t>(r0 + rfirst + kAhead * rstep) * f.ldx;  // the row the ring asks for next (no gather)
        T* yrow = f.Y + static_cast<size_t>(r0 + rfirst) * f.ldy;
#pragma unroll 1
        for (int lr = rfirst; lr < nrows; lr += rstep) {
            T a0, a1, a2, a3;
            cp_async_wait<kAhead - 1>();
            ring_read(slot, a0, a1, a2, a3);
            bool masked = false;
            if (any_mask) {
                uint32_t m;
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(m) : "r"(smask));
                masked = m != 0;
            }
            epilogue_store<T, true, FAM>(tk, v, a0, a1, a2, a3, lp, f.cols, masked, yrow, &clip);
            const int nxt = lr + kAhead * rstep;
            if (nxt < nrows) ring_fetch(slot, rix != nullptr ? xcol + static_cast<size_t>(__ldg(rix + r0 + nxt)) * f.ldx : xnext);
            cp_async_commit();
            xnext += xstep, yrow += ystep, smask += rstep;
            slot += kWarp * kSlot;
            if (slot == ring_end) slot = ring0;
        }
    };
#define AT_PW_KIND(K)                                                          \
    case K:                                                                    \
        if constexpr ((FAM & kind_bit(K)) != 0) rows(std::integral_constant<int, K>{}); \
        break;
    switch (tile.kind) {
        AT_PW_KIND(AT_EPI_UV2DDFF)
        AT_PW_KIND(AT_EPI_DDFF2UV)
        AT_PW_KIND(AT_EPI_QT2R)
        AT_PW_KIND(AT_EPI_QT2QTR)
        AT_PW_KIND(AT_EPI_RT2Q)
        AT_PW_KIND(AT_EPI_RT2RTQ)
        AT_PW_KIND(AT_EPI_EXP)
        AT_PW_KIND(AT_EPI_LOG)
        AT_PW_KIND(AT_EPI_COSSIN)
        AT_PW_KIND(AT_EPI_ATAN2)
        AT_PW_KIND(AT_EPI_RT2D)
        AT_PW_KIND(AT_EPI_RT2RTD)
        AT_PW_KIND(AT_EPI_DT2R)
        AT_PW_KIND(AT_EPI_DT2DTR)
        default:
            break;
    }
#undef AT_PW_KIND
}

// ---- generic dtypes (float64 matrix and / or float64 fields): scalar columns ----------
template <typename TW, typename TX, typename TY, int MP>
__global__ void __launch_bounds__(kThreads)
    spmm_generic_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                        const TW* __restrict__ data, const TX* __restrict__ X, size_t ldx,
                        TY* __restrict__ Y, size_t ldy, int n_rows, int n_fields) {
    const int row = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    const int p0 = __ldg(indptr + row), p1 = __ldg(indptr + row + 1);
    for (int col = blockIdx.y * 128 + lane; col < min(n_fields, (int)(blockIdx.y + 1) * 128);
         col += kWarp) {
        TY acc = TY(0);
        TY ws = TY(0);
        uint32_t miss = 0, heavy = 0;
        for (int p = p0; p < p1; ++p) {
            const TY w = static_cast<TY>(__ldg(data + p));
            const TY x = static_cast<TY>(__ldg(X + static_cast<size_t>(__ldg(indices + p)) * ldx + col));
            if constexpr (MP != 0) {
                skip_add(acc, ws, miss, 1u, w, x);
            } else if (sizeof(TY) == 8) {
                acc = __dadd_rn(acc, __dmul_rn(w, x));
            } else {
                acc = __fadd_rn(acc, __fmul_rn(w, x));
            }
        }
        if constexpr (MP == AT_MISSING_HEAVIEST) {
            const int h = heaviest_entry(p0, p1, [&](int p) { return __ldg(data + p); });
            if (h >= 0 && isnan(static_cast<TY>(__ldg(X + static_cast<size_t>(__ldg(indices + h)) * ldx + col)))) heavy = 1u;
        }
        if constexpr (MP != 0) acc = missing_result(acc, ws, miss, heavy, 1u);
        Y[static_cast<size_t>(row) * ldy + col] = acc;
    }
}

// ---- float64 results (float64 matrix and / or float64 fields), vectorised ---------------
// What MIR writes (float64 weights) applied to what GRIB decodes to (float64 values), and
// the two mixed cases numpy promotes to float64.  Same mapping as spmm_f32_kernel: one warp
// per target row per column tile, a lane owns VPL groups of 4 adjacent fields (16 bytes of
// float32 or 2 x 16 bytes of float64 per nonzero), the CTA's CSR segment is staged in
// shared memory (weights converted to float64 once, while staging), super-tiled grid order.
// Accumulation is scipy's csr_matvec<double> bit for bit: x is promoted to float64 exactly,
// acc = acc + w*x unfused, storage order, from +0.
// A lane's unit of work per nonzero is 16 bytes of X: 4 float32 fields or 2 float64 fields, so a
// warp-wide load always covers 512 contiguous bytes of the source row.
template <typename TX>
struct WideUnit;
template <>
struct WideUnit<float> {
    static constexpr int N = 4;
    using Raw = float4;
    static __device__ __forceinline__ Raw load(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
    static __device__ __forceinline__ void widen(const Raw& r, double (&x)[4]) {
        x[0] = r.x, x[1] = r.y, x[2] = r.z, x[3] = r.w;
    }
    static __device__ __forceinline__ uint32_t nan_bits(const Raw& r) {
        return (isnan(r.x) ? 1u : 0u) | (isnan(r.y) ? 2u : 0u) | (isnan(r.z) ? 4u : 0u) | (isnan(r.w) ? 8u : 0u);
    }
    static __device__ __forceinline__ void store(double* p, const double (&y)[4]) {
        __stcs(reinterpret_cast<double2*>(p), make_double2(y[0], y[1]));
        __stcs(reinterpret_cast<double2*>(p) + 1, make_double2(y[2], y[3]));
    }
};
template <>
struct WideUnit<double> {
    static constexpr int N = 2;
    using Raw = double2;
    static __device__ __forceinline__ Raw load(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
    static __device__ __forceinline__ void widen(const Raw& r, double (&x)[2]) { x[0] = r.x, x[1] = r.y; }
    static __device__ __forceinline__ uint32_t nan_bits(const Raw& r) { return (isnan(r.x) ? 1u : 0u) | (isnan(r.y) ? 2u : 0u); }
    static __device__ __forceinline__ void store(double* p, const double (&y)[2]) {
        __stcs(reinterpret_cast<double2*>(p), make_double2(y[0], y[1]));
    }
};

template <typename TW, typename TX>
struct WideArgs {
    const int32_t* __restrict__ indptr;
    const int32_t* __restrict__ indices;
    const TW* __restrict__ data;
    const TX* __restrict__ X;
    double* __restrict__ Y;
    size_t ldx, ldy;  // in elements
    int n_rows;
    int n_units;  // 16-byte units of X per row: ceil(F / (16 / sizeof(TX)))
    int rows_per_cta;
    int super;
};

constexpr int kWideSegCap = 1024;  // 4 KB of indices + 8 KB of float64 weights
// 16-byte units per lane of the missing-aware float64 kernels (at_spmm_missing has no variant)
constexpr int kMissingNV = 1;

template <typename TW, typename TX, int NV, bool FALLBACK, int MIN_CTAS, int MP>
__global__ void __launch_bounds__(kThreads, MIN_CTAS) spmm_f64_kernel(const WideArgs<TW, TX> a) {
    using Unit = WideUnit<TX>;
    constexpr int N = Unit::N;
    __shared__ int s_idx[kWideSegCap];
    __shared__ double s_w[kWideSegCap];
    __shared__ int s_ptr[kMaxRowsPerCta + 1];

    const int tile = blockIdx.y * a.super + static_cast<int>(blockIdx.x % a.super);
    const int r0 = static_cast<int>(blockIdx.x / a.super) * a.rows_per_cta;
    const int nrows = min(a.rows_per_cta, a.n_rows - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    if (tile * (kWarp * NV) >= a.n_units) return;

    int ucol[NV];
    bool uok[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        ucol[v] = tile * (kWarp * NV) + v * kWarp + lane;
        uok[v] = ucol[v] < a.n_units;
    }

    for (int i = tid; i <= nrows; i += kThreads) s_ptr[i] = __ldg(a.indptr + r0 + i);
    __syncthreads();
    const int seg_base = s_ptr[0];
    const int seg_len = s_ptr[nrows] - seg_base;
    const bool in_smem = !FALLBACK || seg_len <= kWideSegCap;
    if (in_smem) {
        for (int i = tid; i < seg_len; i += kThreads) {
            s_idx[i] = __ldg(a.indices + seg_base + i);
            s_w[i] = static_cast<double>(__ldg(a.data + seg_base + i));
        }
    }
    __syncthreads();

    constexpr int U = 4;
    for (int lr = warp; lr < nrows; lr += kWarps) {
        double acc[NV][N];
#pragma unroll
        for (int v = 0; v < NV; ++v)
#pragma unroll
            for (int e = 0; e < N; ++e) acc[v][e] = 0.0;
        double ws[MP != 0 ? NV : 1][N];  // missing-aware state, bit v * N + e
        uint32_t miss = 0, heavy = 0;
        if constexpr (MP != 0) {
#pragma unroll
            for (int v = 0; v < NV; ++v)
#pragma unroll
                for (int e = 0; e < N; ++e) ws[v][e] = 0.0;
        }
        const int p0 = s_ptr[lr], p1 = s_ptr[lr + 1];
        // AT_MISSING_HEAVIEST: the heaviest entry's position, found by the warp from the staged
        // weights before the gathers (a per-CTA table of columns, as in spmm_f32_kernel, spills in
        // the FALLBACK instantiation at this kernel's 64-register cap; one int does not)
        int ph = -1;
        if constexpr (MP == AT_MISSING_HEAVIEST) {
            if (!FALLBACK || in_smem)
                ph = heaviest_entry(p0 - seg_base, p1 - seg_base, [&](int p) { return s_w[p]; });
            else
                ph = heaviest_entry(p0, p1, [&](int p) { return __ldg(a.data + p); });
        }
        for (int p = p0; p < p1; p += U) {
            int c[U];
            double w[U];
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const bool ok = p + j < p1;
                if (!FALLBACK || in_smem) {
                    c[j] = ok ? s_idx[p + j - seg_base] : 0;
                    w[j] = ok ? s_w[p + j - seg_base] : 0.0;
                } else {
                    c[j] = ok ? __ldg(a.indices + p + j) : 0;
                    w[j] = ok ? static_cast<double>(__ldg(a.data + p + j)) : 0.0;
                }
            }
            typename Unit::Raw x[U][NV];  // gathers of the chunk in flight before the first add
#pragma unroll
            for (int j = 0; j < U; ++j) {
                const TX* xr = a.X + static_cast<size_t>(c[j]) * a.ldx;
#pragma unroll
                for (int v = 0; v < NV; ++v)
                    if (uok[v] && p + j < p1) x[j][v] = Unit::load(xr + N * static_cast<size_t>(ucol[v]));
            }
#pragma unroll
            for (int j = 0; j < U; ++j) {
                if (p + j < p1) {
#pragma unroll
                    for (int v = 0; v < NV; ++v) {
                        double xd[N];
                        Unit::widen(x[j][v], xd);
#pragma unroll
                        for (int e = 0; e < N; ++e) {
                            if constexpr (MP == 0)
                                acc[v][e] = __dadd_rn(acc[v][e], __dmul_rn(w[j], xd[e]));
                            else
                                skip_add(acc[v][e], ws[v][e], miss, 1u << (v * N + e), w[j], xd[e]);
                        }
                    }
                }
            }
        }
        if constexpr (MP == AT_MISSING_HEAVIEST) {  // the row's heaviest entry, read again
            if (ph >= 0) {
                const int col = (!FALLBACK || in_smem) ? s_idx[ph] : __ldg(a.indices + ph);
                const TX* xr = a.X + static_cast<size_t>(col) * a.ldx;
#pragma unroll
                for (int v = 0; v < NV; ++v)
                    if (uok[v]) heavy |= Unit::nan_bits(Unit::load(xr + N * static_cast<size_t>(ucol[v]))) << (v * N);
            }
        }
        if constexpr (MP != 0) {
#pragma unroll
            for (int v = 0; v < NV; ++v)
#pragma unroll
                for (int e = 0; e < N; ++e) acc[v][e] = missing_result(acc[v][e], ws[v][e], miss, heavy, 1u << (v * N + e));
        }
        double* yr = a.Y + static_cast<size_t>(r0 + lr) * a.ldy;
#pragma unroll
        for (int v = 0; v < NV; ++v)
            if (uok[v]) Unit::store(yr + N * static_cast<size_t>(ucol[v]), acc[v]);
    }
}

template <typename TW, typename TX, int NV, int MIN_CTAS, int MP>
static int launch_wide_nv(const at_csr* csr, const void* X, int64_t ldx, void* Y, int64_t ldy,
                          int64_t n_fields, int rows_per_warp, int super, cudaStream_t st) {
    constexpr int N = WideUnit<TX>::N;
    WideArgs<TW, TX> a;
    a.indptr = csr->d_indptr;
    a.indices = csr->d_indices;
    a.data = static_cast<const TW*>(csr->d_data);
    a.X = static_cast<const TX*>(X);
    a.Y = static_cast<double*>(Y);
    a.ldx = static_cast<size_t>(ldx);
    a.ldy = static_cast<size_t>(ldy);
    a.n_rows = static_cast<int>(csr->n_rows);
    a.n_units = static_cast<int>((n_fields + N - 1) / N);
    a.rows_per_cta = rows_per_warp * kWarps;
    const int tiles = (a.n_units + kWarp * NV - 1) / (kWarp * NV);
    if (super == 0) {
        const double tile_bytes = 16.0 * kWarp * NV;
        super = static_cast<int>(64.0e6 / (2.0 * std::max(1.0, csr->live_cols) * tile_bytes));
    }
    a.super = std::max(1, std::min({super, tiles, 63}));
    const int64_t row_blocks = (csr->n_rows + a.rows_per_cta - 1) / a.rows_per_cta;
    const int64_t gx64 = row_blocks * a.super, gy64 = (tiles + a.super - 1) / a.super;
    if (gy64 > 65535 || gx64 >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "grid too large");
    dim3 grid(static_cast<unsigned>(gx64), static_cast<unsigned>(gy64));
    if (csr->max_seg64 <= kWideSegCap)
        spmm_f64_kernel<TW, TX, NV, false, MIN_CTAS, MP><<<grid, kThreads, 0, st>>>(a);
    else
        spmm_f64_kernel<TW, TX, NV, true, MIN_CTAS, MP><<<grid, kThreads, 0, st>>>(a);
    AT_LAUNCH_CHECK("spmm_f64_kernel");
    return AT_OK;
}

template <typename TW, typename TX, int MP>
static int launch_wide(const at_csr* csr, const void* X, int64_t ldx, void* Y, int64_t ldy,
                       int64_t n_fields, int variant, cudaStream_t st) {
    // variant bits as in at_spmm: 0-2 16-byte units of X per lane per nonzero (1, 2, 4; default 2),
    // 4-7 rows per warp, 12-17 super-tile width.  Measured on config 3 (1560 fields): occupancy
    // decides — 2 units at 64 registers (4 CTAs / SM) 3.04 ms, uncapped (3 CTAs) 3.21 ms,
    // 4 units (2 CTAs) 3.30 ms, 1 unit 3.78 ms.
    int nv = variant & 7, rpw = (variant >> 4) & 15;
    const int super = (variant >> 12) & 63;
    if (nv == 0) nv = 2;
    if (rpw == 0) rpw = 8;
    if (rpw * kWarps > kMaxRowsPerCta) return set_error(AT_ERR_INVALID, "at_spmm: variant selects %d rows per warp", rpw);
    if constexpr (MP != 0) return launch_wide_nv<TW, TX, kMissingNV, 4, MP>(csr, X, ldx, Y, ldy, n_fields, rpw, super, st);
    if (nv == 1) return launch_wide_nv<TW, TX, 1, 4, 0>(csr, X, ldx, Y, ldy, n_fields, rpw, super, st);
    if (nv == 2) return launch_wide_nv<TW, TX, 2, 4, 0>(csr, X, ldx, Y, ldy, n_fields, rpw, super, st);
    if (nv == 4) return launch_wide_nv<TW, TX, 4, 2, 0>(csr, X, ldx, Y, ldy, n_fields, rpw, super, st);
    return set_error(AT_ERR_INVALID, "at_spmm: float64 results support 1, 2 or 4 units per lane, not %d", nv);
}

template <typename TW, typename TX, typename TY, int MP>
static int launch_generic(const at_csr* csr, const void* X, int64_t ldx, void* Y, int64_t ldy,
                          int64_t n_fields, cudaStream_t st) {
    dim3 grid(static_cast<unsigned>((csr->n_rows + kWarps - 1) / kWarps),
              static_cast<unsigned>((n_fields + 127) / 128));
    spmm_generic_kernel<TW, TX, TY, MP><<<grid, kThreads, 0, st>>>(
        csr->d_indptr, csr->d_indices, static_cast<const TW*>(csr->d_data),
        static_cast<const TX*>(X), static_cast<size_t>(ldx), static_cast<TY*>(Y),
        static_cast<size_t>(ldy), static_cast<int>(csr->n_rows), static_cast<int>(n_fields));
    AT_LAUNCH_CHECK("spmm_generic_kernel");
    return AT_OK;
}

template <int VPL, int MP>
static int launch_f32(const at_csr* csr, const SpmmArgs& args, bool bulk, bool force_general,
                      cudaStream_t st) {
    const int64_t row_blocks = (csr->n_rows + args.rows_per_cta - 1) / args.rows_per_cta;
    const int64_t tiles = (args.n_vec + kWarp * VPL - 1) / (kWarp * VPL);
    const int64_t gx64 = row_blocks * args.super, gy64 = (tiles + args.super - 1) / args.super;
    if (gy64 > 65535 || gx64 >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "grid too large");
    dim3 grid(static_cast<unsigned>(gx64), static_cast<unsigned>(gy64));
    const int u = force_general ? 0 : csr->uniform_nnz;
    const bool fits = csr->max_seg64 <= kSegCap;
    if (u == 4 && bulk)
        spmm_f32_kernel<VPL, 4, true, false, MP><<<grid, kThreads, 0, st>>>(args);
    else if (u == 4)
        spmm_f32_kernel<VPL, 4, false, false, MP><<<grid, kThreads, 0, st>>>(args);
    else if (u == 12 && VPL <= 2 && bulk)
        spmm_f32_kernel<(VPL <= 2 ? VPL : 1), 12, true, false, MP><<<grid, kThreads, 0, st>>>(args);
    else if (u == 12 && VPL <= 2)
        spmm_f32_kernel<(VPL <= 2 ? VPL : 1), 12, false, false, MP><<<grid, kThreads, 0, st>>>(args);
    else if (fits)
        spmm_f32_kernel<VPL, 0, false, false, MP><<<grid, kThreads, 0, st>>>(args);
    else
        spmm_f32_kernel<VPL, 0, false, true, MP><<<grid, kThreads, 0, st>>>(args);
    AT_LAUNCH_CHECK("spmm_f32_kernel");
    return AT_OK;
}

// first[c] / last[c] = first / last row whose segment references column c (live-column span)
__global__ void col_span_kernel(const int* __restrict__ indptr, const int* __restrict__ indices, int n_rows,
                                int* __restrict__ first, int* __restrict__ last) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    for (int p = indptr[r]; p < indptr[r + 1]; ++p) {
        const int col = indices[p];
        atomicMin(first + col, r);
        atomicMax(last + col, r);
    }
}
__global__ void col_span_sum_kernel(const int* __restrict__ first, const int* __restrict__ last, long long n_cols,
                                    unsigned long long* __restrict__ sum) {
    unsigned long long local = 0;
    for (long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x; c < n_cols; c += (long long)gridDim.x * blockDim.x)
        if (last[c] >= 0) local += static_cast<unsigned long long>(last[c] - first[c] + 1);
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(sum, local);
}

template <typename T>
static bool copy_index_array(const void* src, int dtype, int64_t n, std::vector<int32_t>& dst,
                             int64_t limit, const char* what, bool monotone) {
    dst.resize(static_cast<size_t>(n));
    int64_t prev = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t v = dtype == AT_I32 ? static_cast<const int32_t*>(src)[i]
                                          : static_cast<const int64_t*>(src)[i];
        if (v < 0 || v > limit) {
            set_error(AT_ERR_INVALID, "%s[%lld] = %lld out of range [0, %lld]", what,
                      (long long)i, (long long)v, (long long)limit);
            return false;
        }
        if (monotone && v < prev) {
            set_error(AT_ERR_INVALID, "%s is not non-decreasing at %lld", what, (long long)i);
            return false;
        }
        prev = v;
        dst[static_cast<size_t>(i)] = static_cast<int32_t>(v);
    }
    return true;
}

}  // namespace at

using namespace at;

extern "C" int at_csr_create(int64_t n_rows, int64_t n_cols, int64_t nnz, const void* indptr,
                             int indptr_dtype, const void* indices, int indices_dtype,
                             const void* data, int data_dtype, at_csr_t** out) {
    AT_REQUIRE(out != nullptr, "at_csr_create: out is null");
    *out = nullptr;
    AT_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0, "at_csr_create: negative size");
    AT_REQUIRE(n_rows < (1ll << 31) - 64 && n_cols < (1ll << 31) && nnz < (1ll << 31) - 64,
               "at_csr_create: sizes must be < 2^31 (n_rows=%lld n_cols=%lld nnz=%lld)",
               (long long)n_rows, (long long)n_cols, (long long)nnz);
    AT_REQUIRE(indptr != nullptr && (nnz == 0 || (indices != nullptr && data != nullptr)),
               "at_csr_create: null array");
    AT_REQUIRE((indptr_dtype == AT_I32 || indptr_dtype == AT_I64) &&
                   (indices_dtype == AT_I32 || indices_dtype == AT_I64) &&
                   (data_dtype == AT_F32 || data_dtype == AT_F64),
               "at_csr_create: bad dtype code");

    std::vector<int32_t> h_ptr, h_idx;
    if (!copy_index_array<int32_t>(indptr, indptr_dtype, n_rows + 1, h_ptr, nnz, "indptr", true))
        return AT_ERR_INVALID;
    AT_REQUIRE(h_ptr[0] == 0 && h_ptr[static_cast<size_t>(n_rows)] == nnz,
               "at_csr_create: indptr must start at 0 and end at nnz");
    if (!copy_index_array<int32_t>(indices, indices_dtype, nnz, h_idx, n_cols - 1, "indices", false))
        return AT_ERR_INVALID;

    at_csr* c = new at_csr();
    c->n_rows = n_rows;
    c->n_cols = n_cols;
    c->nnz = nnz;
    c->data_dtype = data_dtype;
    int uniform = n_rows > 0 ? h_ptr[1] - h_ptr[0] : 0, max_nnz = 0;
    for (int64_t r = 0; r < n_rows; ++r) {
        const int len = h_ptr[static_cast<size_t>(r + 1)] - h_ptr[static_cast<size_t>(r)];
        if (len != uniform) uniform = 0;
        max_nnz = std::max(max_nnz, len);
    }
    c->uniform_nnz = uniform;
    c->max_row_nnz = max_nnz;
    for (int64_t r = 0; r < n_rows; r += kMaxRowsPerCta) {
        const int64_t e = std::min<int64_t>(n_rows, r + kMaxRowsPerCta);
        c->max_seg64 = std::max(c->max_seg64, h_ptr[static_cast<size_t>(e)] - h_ptr[static_cast<size_t>(r)]);
    }
    cudaGetDevice(&c->device);

    const size_t esz = data_dtype == AT_F32 ? 4 : 8;
    auto fail = [&](int code) {
        at_csr_destroy(c);
        return code;
    };
    cudaError_t e;
    if ((e = device_alloc(reinterpret_cast<void**>(&c->d_indptr), (static_cast<size_t>(n_rows) + 1 + kPad) * 4)) != cudaSuccess ||
        (e = device_alloc(reinterpret_cast<void**>(&c->d_indices), (static_cast<size_t>(nnz) + kPad) * 4)) != cudaSuccess ||
        (e = device_alloc(reinterpret_cast<void**>(&c->d_data), (static_cast<size_t>(nnz) + kPad) * esz)) != cudaSuccess) {
        set_error(e == cudaErrorMemoryAllocation ? AT_ERR_NOMEM : AT_ERR_CUDA,
                  "at_csr_create: cudaMalloc failed: %s", cudaGetErrorString(e));
        return fail(e == cudaErrorMemoryAllocation ? AT_ERR_NOMEM : AT_ERR_CUDA);
    }
    if ((e = cudaMemset(c->d_indptr, 0, (static_cast<size_t>(n_rows) + 1 + kPad) * 4)) != cudaSuccess ||
        (e = cudaMemset(c->d_indices, 0, (static_cast<size_t>(nnz) + kPad) * 4)) != cudaSuccess ||
        (e = cudaMemset(c->d_data, 0, (static_cast<size_t>(nnz) + kPad) * esz)) != cudaSuccess ||
        (e = cudaMemcpy(c->d_indptr, h_ptr.data(), (static_cast<size_t>(n_rows) + 1) * 4,
                        cudaMemcpyHostToDevice)) != cudaSuccess ||
        (nnz > 0 && (e = cudaMemcpy(c->d_indices, h_idx.data(), static_cast<size_t>(nnz) * 4,
                                    cudaMemcpyHostToDevice)) != cudaSuccess) ||
        (nnz > 0 && (e = cudaMemcpy(c->d_data, data, static_cast<size_t>(nnz) * esz,
                                    cudaMemcpyHostToDevice)) != cudaSuccess)) {
        set_error(AT_ERR_CUDA, "at_csr_create: staging the matrix failed: %s", cudaGetErrorString(e));
        return fail(AT_ERR_CUDA);
    }
    {
        // Reuse working set: a source column is "live" between the first and the last target
        // row that references it; the mean number of live columns while the rows are walked in
        // order is sum(span) / n_rows.  at_spmm sizes its column super-tile so that the live
        // source rows of the CTAs in flight stay in L2.  Computed on the device from the staged
        // arrays (the scattered first / last updates were the slowest part of the host set-up
        // for matrices with millions of nonzeros).
        int32_t *d_first = nullptr, *d_last = nullptr;
        unsigned long long* d_sum = nullptr;
        c->live_cols = 0.0;
        if (n_rows > 0 && n_cols > 0 && nnz > 0) {
            const size_t cb = static_cast<size_t>(n_cols) * 4;
            unsigned long long h_sum = 0;
            if ((e = device_alloc(reinterpret_cast<void**>(&d_first), cb)) == cudaSuccess && (e = device_alloc(reinterpret_cast<void**>(&d_last), cb)) == cudaSuccess &&
                (e = device_alloc(reinterpret_cast<void**>(&d_sum), 8)) == cudaSuccess && (e = cudaMemset(d_first, 0x7f, cb)) == cudaSuccess &&
                (e = cudaMemset(d_last, 0xff, cb)) == cudaSuccess && (e = cudaMemset(d_sum, 0, 8)) == cudaSuccess) {
                col_span_kernel<<<static_cast<unsigned>((n_rows + 255) / 256), 256>>>(c->d_indptr, c->d_indices, static_cast<int>(n_rows), d_first, d_last);
                col_span_sum_kernel<<<static_cast<unsigned>(std::min<int64_t>((n_cols + 255) / 256, 1024)), 256>>>(d_first, d_last, n_cols, d_sum);
                e = cudaGetLastError();
                if (e == cudaSuccess) e = cudaMemcpy(&h_sum, d_sum, 8, cudaMemcpyDeviceToHost);
            }
            device_free(d_first);
            device_free(d_last);
            device_free(d_sum);
            if (e != cudaSuccess) {
                set_error(AT_ERR_CUDA, "at_csr_create: column-span scan failed: %s", cudaGetErrorString(e));
                return fail(AT_ERR_CUDA);
            }
            c->live_cols = static_cast<double>(h_sum) / static_cast<double>(n_rows);
        }
    }
    *out = c;
    return AT_OK;
}

extern "C" int at_csr_destroy(at_csr_t* c) {
    if (c == nullptr) return AT_OK;
    device_free(c->d_indptr);
    device_free(c->d_indices);
    device_free(c->d_data);
    delete c;
    return AT_OK;
}

// Copy a staged matrix to another device, device to device: the host arrays are not read again
// and the row statistics travel with the copy.
extern "C" int at_csr_replicate(const at_csr_t* src, int device, at_csr_t** out) {
    AT_REQUIRE(src != nullptr && out != nullptr, "at_csr_replicate: null argument");
    *out = nullptr;
    int n_dev = 0;
    AT_CUDA_TRY(cudaGetDeviceCount(&n_dev));
    AT_REQUIRE(device >= 0 && device < n_dev, "at_csr_replicate: device %d out of range (%d visible)", device, n_dev);
    int prev = 0;
    AT_CUDA_TRY(cudaGetDevice(&prev));
    AT_CUDA_TRY(cudaSetDevice(device));
    at_csr* c = new at_csr(*src);
    c->d_indptr = nullptr;
    c->d_indices = nullptr;
    c->d_data = nullptr;
    c->device = device;
    const size_t esz = src->data_dtype == AT_F32 ? 4 : 8;
    const size_t b_ptr = (static_cast<size_t>(src->n_rows) + 1 + kPad) * 4, b_idx = (static_cast<size_t>(src->nnz) + kPad) * 4,
                 b_data = (static_cast<size_t>(src->nnz) + kPad) * esz;
    cudaError_t e;
    if ((e = device_alloc(reinterpret_cast<void**>(&c->d_indptr), b_ptr)) != cudaSuccess ||
        (e = device_alloc(reinterpret_cast<void**>(&c->d_indices), b_idx)) != cudaSuccess ||
        (e = device_alloc(&c->d_data, b_data)) != cudaSuccess ||
        (e = cudaMemcpyPeerAsync(c->d_indptr, device, src->d_indptr, src->device, b_ptr, nullptr)) != cudaSuccess ||
        (e = cudaMemcpyPeerAsync(c->d_indices, device, src->d_indices, src->device, b_idx, nullptr)) != cudaSuccess ||
        (e = cudaMemcpyPeerAsync(c->d_data, device, src->d_data, src->device, b_data, nullptr)) != cudaSuccess ||
        (e = cudaStreamSynchronize(nullptr)) != cudaSuccess) {
        at_csr_destroy(c);
        cudaSetDevice(prev);
        return set_error(e == cudaErrorMemoryAllocation ? AT_ERR_NOMEM : AT_ERR_CUDA, "at_csr_replicate: %s", cudaGetErrorString(e));
    }
    cudaSetDevice(prev);
    *out = c;
    return AT_OK;
}

namespace at {
// A matrix lives in the memory of the device it was staged on; a kernel launched on another
// device would read that device's memory through whatever mapping happens to exist.
int check_csr_device(const at_csr_t* c, int device, const char* who) {
    AT_REQUIRE(c->device == device, "%s: the matrix is staged on device %d, the call runs on device %d", who, c->device, device);
    return AT_OK;
}
int check_csr_on_current_device(const at_csr_t* c, const char* who) {
    int dev = 0;
    AT_CUDA_TRY(cudaGetDevice(&dev));
    return check_csr_device(c, dev, who);
}
}  // namespace at

extern "C" int at_csr_info(const at_csr_t* c, int64_t* n_rows, int64_t* n_cols, int64_t* nnz,
                           int* uniform_nnz, int* data_dtype) {
    AT_REQUIRE(c != nullptr, "at_csr_info: null handle");
    if (n_rows) *n_rows = c->n_rows;
    if (n_cols) *n_cols = c->n_cols;
    if (nnz) *nnz = c->nnz;
    if (uniform_nnz) *uniform_nnz = c->uniform_nnz;
    if (data_dtype) *data_dtype = c->data_dtype;
    return AT_OK;
}

static int decode_variant(int variant, int& vpl, int& rows_per_warp, bool& bulk, bool& general, int& super) {
    // bits 0-2: float4 per lane per nonzero (1, 2, 4); bits 4-7: rows per warp;
    // bit 8: bulk-copy (TMA) staging off; bit 9: force the general-CSR kernel;
    // bits 12-17: column tiles per super-tile.
    vpl = variant & 7;
    rows_per_warp = (variant >> 4) & 15;
    bulk = ((variant >> 8) & 1) == 0;
    general = ((variant >> 9) & 1) != 0;
    super = (variant >> 12) & 63;  // 0: chosen from the matrix's reuse working set
    if (vpl == 0) vpl = kDefaultVPL;
    if (rows_per_warp == 0) rows_per_warp = 8;
    if (vpl != 1 && vpl != 2 && vpl != 4)
        return set_error(AT_ERR_INVALID, "at_spmm: variant selects %d float4 per lane", vpl);
    if (rows_per_warp * kWarps > kMaxRowsPerCta)
        return set_error(AT_ERR_INVALID, "at_spmm: variant selects %d rows per warp", rows_per_warp);
    return AT_OK;
}

// at_spmm (MP = 0) and at_spmm_missing (MP = the policy): the same checks, shapes and dispatch.
// The missing-aware kernels exist for the default shape only (at_spmm_missing takes no variant).
template <int MP>
static int spmm_impl(const char* who, const at_csr_t* csr, const void* X, int x_dtype, int64_t ldx, void* Y,
                     int y_dtype, int64_t ldy, int64_t n_fields, int spmm_variant, void* stream) {
    AT_REQUIRE(csr != nullptr && X != nullptr && Y != nullptr, "%s: null argument", who);
    AT_REQUIRE(n_fields >= 0 && ldx >= n_fields && ldy >= n_fields,
               "%s: leading dimensions (%lld, %lld) smaller than n_fields %lld", who,
               (long long)ldx, (long long)ldy, (long long)n_fields);
    int rc = check_csr_on_current_device(csr, who);
    if (rc != AT_OK) return rc;
    const int want_y = (csr->data_dtype == AT_F64 || x_dtype == AT_F64) ? AT_F64 : AT_F32;
    AT_REQUIRE(y_dtype == want_y, "%s: result dtype must be %s (numpy result_type)", who,
               want_y == AT_F64 ? "float64" : "float32");
    if (n_fields == 0 || csr->n_rows == 0) return AT_OK;
    cudaStream_t st = as_stream(stream);

    if (csr->data_dtype == AT_F32 && x_dtype == AT_F32) {
        AT_REQUIRE(ldx % 4 == 0 && ldy % 4 == 0, "%s: ldx, ldy must be multiples of 4", who);
        AT_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0,
                   "%s: X and Y must be 16-byte aligned", who);
        int vpl, rpw, super;
        bool bulk, general;
        rc = decode_variant(spmm_variant, vpl, rpw, bulk, general, super);
        if (rc != AT_OK) return rc;
        if constexpr (MP != 0) vpl = kDefaultVPL;  // the only shape of the missing-aware kernels: tiling and kernel agree
        SpmmArgs a;
        a.indptr = csr->d_indptr;
        a.indices = csr->d_indices;
        a.data = static_cast<const float*>(csr->d_data);
        a.X = static_cast<const float4*>(X);
        a.Y = static_cast<float4*>(Y);
        a.ldx4 = static_cast<size_t>(ldx / 4);
        a.ldy4 = static_cast<size_t>(ldy / 4);
        a.n_rows = static_cast<int>(csr->n_rows);
        // Columns beyond n_fields up to the next multiple of 4 are padding inside ld.
        a.n_vec = static_cast<int>((n_fields + 3) / 4);
        a.rows_per_cta = rpw * kWarps;
        if (csr->uniform_nnz > 0 && !general)  // the staged segment of a CTA must fit
            a.rows_per_cta = std::max(kWarps, std::min(a.rows_per_cta, kSegCap / csr->uniform_nnz / kWarps * kWarps));
        const int tiles = (a.n_vec + kWarp * vpl - 1) / (kWarp * vpl);
        if (super == 0) {
            // Widest super-tile (most contiguous bytes per source row, best DRAM page locality)
            // whose live source rows stay in L2.  Rows being streamed by the resident CTAs
            // roughly double the set that has to survive until its last use; 64 MB is half of
            // the B200's L2.
            const double l2_budget = 64.0e6;
            const double tile_bytes = 512.0 * vpl;
            super = static_cast<int>(l2_budget / (2.0 * std::max(1.0, csr->live_cols) * tile_bytes));
        }
        a.super = std::max(1, std::min({super, tiles, 63}));
        if constexpr (MP != 0) {
            return launch_f32<kDefaultVPL, MP>(csr, a, bulk, general, st);
        } else {
            switch (vpl) {
                case 1: return launch_f32<1, 0>(csr, a, bulk, general, st);
                case 2: return launch_f32<2, 0>(csr, a, bulk, general, st);
                default: return launch_f32<4, 0>(csr, a, bulk, general, st);
            }
        }
    }
    // float64 results: the vectorised kernel needs 4-field groups (ld % 4 == 0, 16-byte aligned
    // bases — what DeviceBatch provides); other layouts take the scalar-column kernel.
    const bool wide = ldx % 4 == 0 && ldy % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(Y) & 15) == 0 && ((spmm_variant >> 9) & 1) == 0;
    if (wide) {
        if (csr->data_dtype == AT_F64 && x_dtype == AT_F32) return launch_wide<double, float, MP>(csr, X, ldx, Y, ldy, n_fields, spmm_variant, st);
        if (csr->data_dtype == AT_F64 && x_dtype == AT_F64) return launch_wide<double, double, MP>(csr, X, ldx, Y, ldy, n_fields, spmm_variant, st);
        if (csr->data_dtype == AT_F32 && x_dtype == AT_F64) return launch_wide<float, double, MP>(csr, X, ldx, Y, ldy, n_fields, spmm_variant, st);
    }
    if (csr->data_dtype == AT_F64 && x_dtype == AT_F32)
        return launch_generic<double, float, double, MP>(csr, X, ldx, Y, ldy, n_fields, st);
    if (csr->data_dtype == AT_F64 && x_dtype == AT_F64)
        return launch_generic<double, double, double, MP>(csr, X, ldx, Y, ldy, n_fields, st);
    if (csr->data_dtype == AT_F32 && x_dtype == AT_F64)
        return launch_generic<float, double, double, MP>(csr, X, ldx, Y, ldy, n_fields, st);
    return set_error(AT_ERR_INVALID, "%s: bad dtype codes", who);
}

extern "C" int at_spmm(const at_csr_t* csr, const void* X, int x_dtype, int64_t ldx, void* Y,
                       int y_dtype, int64_t ldy, int64_t n_fields, int spmm_variant,
                       void* stream) {
    return spmm_impl<0>("at_spmm", csr, X, x_dtype, ldx, Y, y_dtype, ldy, n_fields, spmm_variant, stream);
}

extern "C" int at_spmm_missing(const at_csr_t* csr, const void* X, int x_dtype, int64_t ldx, void* Y,
                               int y_dtype, int64_t ldy, int64_t n_fields, int policy, void* stream) {
    switch (policy) {
        case AT_MISSING_PROPAGATE: return at_spmm(csr, X, x_dtype, ldx, Y, y_dtype, ldy, n_fields, 0, stream);
        case AT_MISSING_ALL: return spmm_impl<AT_MISSING_ALL>("at_spmm_missing", csr, X, x_dtype, ldx, Y, y_dtype, ldy, n_fields, 0, stream);
        case AT_MISSING_HEAVIEST: return spmm_impl<AT_MISSING_HEAVIEST>("at_spmm_missing", csr, X, x_dtype, ldx, Y, y_dtype, ldy, n_fields, 0, stream);
        default:
            return set_error(AT_ERR_INVALID, "at_spmm_missing: unknown policy %d (AT_MISSING_PROPAGATE %d, AT_MISSING_ALL %d, AT_MISSING_HEAVIEST %d)",
                             policy, AT_MISSING_PROPAGATE, AT_MISSING_ALL, AT_MISSING_HEAVIEST);
    }
}

// ---- epilogue handle --------------------------------------------------------------------
// The cubic table of es(T) (epilogue.cuh): the float64 formula sampled at four Chebyshev points of
// every 0.5 K interval, interpolating cubic in f = (t - node) / 0.5, rounded to float32.  Once per
// device and process.
namespace {

double es_mixed_f64(double t) {
    // thresholds as the float32 numbers numpy compares a float32 field with (NEP 50)
    const double t0 = static_cast<double>(273.16f), ti = static_cast<double>(250.16f);
    const double es_w = 611.21 * std::exp(17.502 * (t - 273.16) / (t - 32.19));
    const double es_i = 611.21 * std::exp(22.587 * (t - 273.16) / (t + 0.7));
    if (t <= ti) return es_i;
    if (t >= t0) return es_w;
    const double a = (t - 250.16) / 23.0;
    return a * a * es_w + (1.0 - a * a) * es_i;
}

void fit_es_table(double (*fn)(double), float4* out) {
    const double pi = 3.14159265358979323846;
    double f[4];
    for (int k = 0; k < 4; ++k) f[k] = 0.5 * (1.0 - std::cos((2 * k + 1) * pi / 8.0));
    for (int j = 0; j < kEsTableN; ++j) {
        const double node = static_cast<double>(kEsTableT) + 0.5 * (j - kEsTableZero);
        // Newton divided differences through the four points, expanded to monomials in f
        double dd[4];
        for (int k = 0; k < 4; ++k) dd[k] = fn(node + 0.5 * f[k]);
        for (int level = 1; level < 4; ++level)
            for (int k = 3; k >= level; --k) dd[k] = (dd[k] - dd[k - 1]) / (f[k] - f[k - level]);
        // p(x) = dd0 + dd1 (x-f0) + dd2 (x-f0)(x-f1) + dd3 (x-f0)(x-f1)(x-f2)
        double c[4] = {dd[3], 0, 0, 0};  // Horner from the top: coefficients of the running polynomial, highest first
        int deg = 0;
        for (int k = 2; k >= 0; --k) {  // poly = poly * (x - f[k]) + dd[k]
            double nc[4] = {0, 0, 0, 0};
            for (int i = 0; i <= deg; ++i) {
                nc[i] += c[i];
                nc[i + 1] -= c[i] * f[k];
            }
            ++deg;
            nc[deg] += dd[k];
            for (int i = 0; i < 4; ++i) c[i] = nc[i];
        }
        // c[0..3] = coefficients of x^3, x^2, x^1, x^0
        out[j] = make_float4(static_cast<float>(c[3]), static_cast<float>(c[2]), static_cast<float>(c[1]), static_cast<float>(c[0]));
    }
}

int ensure_es_tables() {
    static std::mutex mu;
    static std::vector<int> ready;  // devices whose tables are loaded
    int dev = 0;
    AT_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    if (std::find(ready.begin(), ready.end(), dev) != ready.end()) return AT_OK;
    std::vector<float4> mixed(kEsTableN);
    fit_es_table(es_mixed_f64, mixed.data());
    AT_CUDA_TRY(cudaMemcpyToSymbol(g_es_mixed_table, mixed.data(), sizeof(float4) * kEsTableN));
    ready.push_back(dev);
    return AT_OK;
}

}  // namespace

extern "C" int at_epilogue_create(const at_epi_segment_t* segments, int32_t n_segments,
                                  const at_epi_col_t* cols, int32_t n_out_cols,
                                  at_epilogue_t** out) {
    AT_REQUIRE(out != nullptr, "at_epilogue_create: out is null");
    *out = nullptr;
    AT_REQUIRE(segments != nullptr && n_segments > 0 && cols != nullptr && n_out_cols > 0,
               "at_epilogue_create: empty program");
    {
        const int rc = ensure_es_tables();
        if (rc != AT_OK) return rc;
    }
    std::vector<EpiTile> tiles;
    int n_in_cols = 0;
    for (int s = 0; s < n_segments; ++s) {
        const at_epi_segment_t& g = segments[s];
        AT_REQUIRE(g.kind >= AT_EPI_PLAIN && g.kind < AT_EPI_KIND_COUNT,
                   "at_epilogue_create: segment %d has unknown kind %d", s, g.kind);
        AT_REQUIRE(g.in_col >= 0 && g.in_col % 4 == 0 && g.n_in > 0 && g.n_in % 4 == 0,
                   "at_epilogue_create: segment %d: in_col and n_in must be multiples of 4", s);
        AT_REQUIRE(g.kind != AT_EPI_AFFINE_INV || g.pa != 0.0, "at_epilogue_create: segment %d: zero scale", s);
        int out_per_vec = 4;  // outputs per 4 input columns
        switch (g.kind) {
            case AT_EPI_QT2R: case AT_EPI_RT2Q: case AT_EPI_ATAN2: case AT_EPI_RT2D: case AT_EPI_DT2R: out_per_vec = 2; break;
            case AT_EPI_QT2QTR: case AT_EPI_RT2RTQ: case AT_EPI_RT2RTD: case AT_EPI_DT2DTR: out_per_vec = 6; break;
            case AT_EPI_COSSIN: out_per_vec = 8; break;
            default: break;
        }
        const int align = out_per_vec == 2 || out_per_vec == 6 ? 2 : 4;
        AT_REQUIRE(g.out_col >= 0 && g.out_col % align == 0,
                   "at_epilogue_create: segment %d: out_col must be a multiple of %d", s, align);
        const int n_vec = g.n_in / 4;
        AT_REQUIRE(g.out_col + n_vec * out_per_vec <= n_out_cols,
                   "at_epilogue_create: segment %d writes past n_out_cols", s);
        for (int v0 = 0; v0 < n_vec; v0 += kWarp) {
            EpiTile t;
            t.kind = g.kind;
            t.in_vec0 = g.in_col / 4 + v0;
            t.n_vec = std::min(kWarp, n_vec - v0);
            t.out_col0 = g.out_col + v0 * out_per_vec;
            t.flags_any = 0;
            t.reserved = 0;
            t.pa = g.pa;
            t.pb = g.pb;
            for (int c = t.out_col0; c < t.out_col0 + t.n_vec * out_per_vec; ++c)
                t.flags_any |= static_cast<int32_t>(cols[c].flags & (AT_COL_CLIP_LO | AT_COL_CLIP_HI | AT_COL_MASK));
            tiles.push_back(t);
        }
        n_in_cols = std::max(n_in_cols, g.in_col + g.n_in);
    }
    AT_REQUIRE(tiles.size() <= 65535, "at_epilogue_create: too many column tiles");
    std::vector<ColF32> h32(static_cast<size_t>(n_out_cols));
    std::vector<ColF64> h64(static_cast<size_t>(n_out_cols));
    for (int c = 0; c < n_out_cols; ++c) {
        // an absent bound becomes -inf / +inf: the kernels clip unconditionally (NaN still passes)
        const double lo = (cols[c].flags & AT_COL_CLIP_LO) ? cols[c].lo : -HUGE_VAL;
        const double hi = (cols[c].flags & AT_COL_CLIP_HI) ? cols[c].hi : HUGE_VAL;
        h32[static_cast<size_t>(c)] = {static_cast<float>(lo), static_cast<float>(hi),
                                       static_cast<float>(cols[c].pressure), cols[c].flags};
        h64[static_cast<size_t>(c)] = {lo, hi, cols[c].pressure, cols[c].flags};
    }
    at_epilogue* e = new at_epilogue();
    for (int sgm = 0; sgm < n_segments; ++sgm) e->kinds_mask |= kind_bit(segments[sgm].kind);
    e->n_tiles = static_cast<int32_t>(tiles.size());
    e->n_in_cols = n_in_cols;
    e->n_out_cols = n_out_cols;
    cudaGetDevice(&e->device);
    cudaError_t ce;
    if ((ce = device_alloc(reinterpret_cast<void**>(&e->d_tiles), tiles.size() * sizeof(EpiTile))) != cudaSuccess ||
        (ce = device_alloc(reinterpret_cast<void**>(&e->d_cols32), h32.size() * sizeof(ColF32))) != cudaSuccess ||
        (ce = device_alloc(reinterpret_cast<void**>(&e->d_cols64), h64.size() * sizeof(ColF64))) != cudaSuccess ||
        (ce = cudaMemcpy(e->d_tiles, tiles.data(), tiles.size() * sizeof(EpiTile), cudaMemcpyHostToDevice)) !=
            cudaSuccess ||
        (ce = cudaMemcpy(e->d_cols32, h32.data(), h32.size() * sizeof(ColF32), cudaMemcpyHostToDevice)) !=
            cudaSuccess ||
        (ce = cudaMemcpy(e->d_cols64, h64.data(), h64.size() * sizeof(ColF64), cudaMemcpyHostToDevice)) !=
            cudaSuccess) {
        at_epilogue_destroy(e);
        return set_error(AT_ERR_CUDA, "at_epilogue_create: %s", cudaGetErrorString(ce));
    }
    *out = e;
    return AT_OK;
}

extern "C" int at_epilogue_destroy(at_epilogue_t* e) {
    if (e == nullptr) return AT_OK;
    device_free(e->d_tiles);
    device_free(e->d_cols32);
    device_free(e->d_cols64);
    delete e;
    return AT_OK;
}

extern "C" int at_spmm_fused(const at_csr_t* csr, const at_epilogue_t* epi, const float* X,
                             int64_t n_src, int64_t ldx, float* Y, int64_t ldy, const uint8_t* row_mask,
                             void* stream) {
    AT_REQUIRE(csr != nullptr && epi != nullptr && X != nullptr && Y != nullptr,
               "at_spmm_fused: null argument");
    const int dev_rc = check_csr_on_current_device(csr, "at_spmm_fused");
    if (dev_rc != AT_OK) return dev_rc;
    AT_REQUIRE(n_src == csr->n_cols, "at_spmm_fused: dimension mismatch: matrix has %lld columns, X has %lld rows",
               (long long)csr->n_cols, (long long)n_src);
    AT_REQUIRE(csr->data_dtype == AT_F32, "at_spmm_fused: float32 matrices only");
    AT_REQUIRE(ldx % 4 == 0 && ldx >= epi->n_in_cols, "at_spmm_fused: ldx %lld too small or not a multiple of 4",
               (long long)ldx);
    AT_REQUIRE(ldy % 2 == 0 && ldy >= epi->n_out_cols, "at_spmm_fused: ldy %lld too small or odd", (long long)ldy);
    AT_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0,
               "at_spmm_fused: X and Y must be 16-byte aligned");
    AT_REQUIRE(ldy % 4 == 0, "at_spmm_fused: ldy must be a multiple of 4");
    if (csr->n_rows == 0) return AT_OK;
    FusedArgs f;
    f.s.indptr = csr->d_indptr;
    f.s.indices = csr->d_indices;
    f.s.data = static_cast<const float*>(csr->d_data);
    f.s.X = reinterpret_cast<const float4*>(X);
    f.s.Y = nullptr;
    f.s.ldx4 = static_cast<size_t>(ldx / 4);
    f.s.ldy4 = 0;
    f.s.n_rows = static_cast<int>(csr->n_rows);
    f.s.n_vec = epi->n_tiles;
    f.s.rows_per_cta = kMaxRowsPerCta;
    if (csr->uniform_nnz > 0)  // the staged segment of a CTA must fit
        f.s.rows_per_cta = std::max(kWarps, std::min(f.s.rows_per_cta, kSegCap / csr->uniform_nnz / kWarps * kWarps));
    f.tiles = epi->d_tiles;
    f.cols = epi->d_cols32;
    f.row_mask = row_mask;
    f.Yf = Y;
    f.ldy = static_cast<size_t>(ldy);
    const int groups = epi->n_tiles;
    // widest super-tile whose live source rows stay in L2 (see at_spmm)
    const int super_fit = static_cast<int>(64.0e6 / (2.0 * std::max(1.0, csr->live_cols) * 512.0));
    f.s.super = std::max(1, std::min({super_fit, groups, 63}));
    const int64_t row_blocks = (csr->n_rows + f.s.rows_per_cta - 1) / f.s.rows_per_cta;
    const int64_t gx64 = row_blocks * f.s.super, gy64 = (groups + f.s.super - 1) / f.s.super;
    if (gy64 > 65535 || gx64 >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "at_spmm_fused: grid too large");
    dim3 grid(static_cast<unsigned>(gx64), static_cast<unsigned>(gy64));
#define AT_FUSED_LAUNCH(FAM)                                                                       \
    do {                                                                                           \
        if (csr->uniform_nnz == 4)                                                                 \
            spmm_fused_kernel<4, false, FAM><<<grid, kThreads, 0, as_stream(stream)>>>(f);    \
        else if (csr->uniform_nnz == 12)                                                           \
            spmm_fused_kernel<12, false, FAM><<<grid, kThreads, 0, as_stream(stream)>>>(f);   \
        else if (csr->max_seg64 <= kSegCap)                                                        \
            spmm_fused_kernel<0, false, FAM><<<grid, kThreads, 0, as_stream(stream)>>>(f);    \
        else                                                                                       \
            spmm_fused_kernel<0, true, FAM><<<grid, kThreads, 0, as_stream(stream)>>>(f);     \
    } while (0)
    // the smallest kind family that holds the program (epilogue.cuh)
    if ((epi->kinds_mask & ~FAM_BASIC) == 0)
        AT_FUSED_LAUNCH(FAM_BASIC);
    else if ((epi->kinds_mask & ~FAM_UNARY) == 0)
        AT_FUSED_LAUNCH(FAM_UNARY);
    else if ((epi->kinds_mask & ~FAM_TRIG) == 0)
        AT_FUSED_LAUNCH(FAM_TRIG);
    else
        AT_FUSED_LAUNCH(FAM_ALL);
#undef AT_FUSED_LAUNCH
    AT_LAUNCH_CHECK("spmm_fused_kernel");
    return AT_OK;
}

template <typename T>
static int launch_pointwise(const at_epilogue_t* epi, int64_t n_rows, const void* X, int64_t ldx, void* Y,
                            int64_t ldy, const typename ColStore<T>::type* cols, const uint8_t* row_mask,
                            const int64_t* row_index, cudaStream_t st) {
    PointwiseArgs<T> f;
    f.tiles = epi->d_tiles;
    f.cols = cols;
    f.row_mask = row_mask;
    f.X = static_cast<const T*>(X);
    f.Y = static_cast<T*>(Y);
    f.row_index = reinterpret_cast<const long long*>(row_index);
    f.ldx = static_cast<size_t>(ldx);
    f.ldy = static_cast<size_t>(ldy);
    f.n_rows = n_rows;
    f.rows_per_cta = kPwCtaRows;
    f.n_tiles = epi->n_tiles;
    f.uses_es = (epi->kinds_mask & (kind_bit(AT_EPI_QT2R) | kind_bit(AT_EPI_QT2QTR) | kind_bit(AT_EPI_RT2Q) | kind_bit(AT_EPI_RT2RTQ))) != 0;
    const int64_t gx = (n_rows + kPwCtaRows - 1) / kPwCtaRows;
    if (gx >= (1ll << 31)) return set_error(AT_ERR_UNSUPPORTED, "at_pointwise: too many rows");
    dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>((epi->n_tiles + kWarps - 1) / kWarps));
    if ((epi->kinds_mask & ~FAM_BASIC) == 0)
        pointwise_kernel<T, FAM_BASIC><<<grid, kThreads, 0, st>>>(f);
    else if ((epi->kinds_mask & ~FAM_UNARY) == 0)
        pointwise_kernel<T, FAM_UNARY><<<grid, kThreads, 0, st>>>(f);
    else if ((epi->kinds_mask & ~FAM_TRIG) == 0)
        pointwise_kernel<T, FAM_TRIG><<<grid, kThreads, 0, st>>>(f);
    else
        pointwise_kernel<T, FAM_ALL><<<grid, kThreads, 0, st>>>(f);
    AT_LAUNCH_CHECK("pointwise_kernel");
    return AT_OK;
}

extern "C" int at_pointwise(const at_epilogue_t* epi, int64_t n_rows, const void* X, int64_t ldx, void* Y,
                            int64_t ldy, int dtype, const uint8_t* row_mask, void* stream) {
    AT_REQUIRE(epi != nullptr && X != nullptr && Y != nullptr, "at_pointwise: null argument");
    AT_REQUIRE(n_rows >= 0, "at_pointwise: negative n_rows");
    AT_REQUIRE(dtype == AT_F32 || dtype == AT_F64, "at_pointwise: bad dtype code");
    AT_REQUIRE(ldx % 4 == 0 && ldx >= epi->n_in_cols, "at_pointwise: ldx %lld too small or not a multiple of 4",
               (long long)ldx);
    AT_REQUIRE(ldy % 4 == 0 && ldy >= epi->n_out_cols, "at_pointwise: ldy %lld too small or not a multiple of 4",
               (long long)ldy);
    AT_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0,
               "at_pointwise: X and Y must be 16-byte aligned");
    if (n_rows == 0) return AT_OK;
    if (dtype == AT_F32)
        return launch_pointwise<float>(epi, n_rows, X, ldx, Y, ldy, epi->d_cols32, row_mask, nullptr, as_stream(stream));
    return launch_pointwise<double>(epi, n_rows, X, ldx, Y, ldy, epi->d_cols64, row_mask, nullptr, as_stream(stream));
}

// Y[r, :] = epilogue(X[idx[r], :]): the nearest-neighbour / masked regrid (a row gather,
// regrid.py:380, 420) fused with the pointwise filters that follow it — one read of the source
// rows, one write of the results.  The gather copies values exactly (numpy indexing: -0.0 stays
// -0.0), unlike a one-nonzero-per-row matrix, which would add them to +0.
extern "C" int at_gather_pointwise(const at_epilogue_t* epi, const int64_t* idx, int64_t n_out, int64_t n_src,
                                   const void* X, int64_t ldx, void* Y, int64_t ldy, int dtype,
                                   const uint8_t* row_mask, void* stream) {
    AT_REQUIRE(epi != nullptr && X != nullptr && Y != nullptr, "at_gather_pointwise: null argument");
    AT_REQUIRE(n_out >= 0 && n_src >= 0, "at_gather_pointwise: negative size");
    AT_REQUIRE(dtype == AT_F32 || dtype == AT_F64, "at_gather_pointwise: bad dtype code");
    AT_REQUIRE(ldx % 4 == 0 && ldx >= epi->n_in_cols, "at_gather_pointwise: ldx %lld too small or not a multiple of 4",
               (long long)ldx);
    AT_REQUIRE(ldy % 4 == 0 && ldy >= epi->n_out_cols, "at_gather_pointwise: ldy %lld too small or not a multiple of 4",
               (long long)ldy);
    AT_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0,
               "at_gather_pointwise: X and Y must be 16-byte aligned");
    if (n_out == 0) return AT_OK;
    AT_REQUIRE(idx != nullptr, "at_gather_pointwise: null index");
    if (dtype == AT_F32)
        return launch_pointwise<float>(epi, n_out, X, ldx, Y, ldy, epi->d_cols32, row_mask, idx, as_stream(stream));
    return launch_pointwise<double>(epi, n_out, X, ldx, Y, ldy, epi->d_cols64, row_mask, idx, as_stream(stream));
}

// hostio.cu — the field I/O engine behind the drop-in filters: moves FieldList values between
// ordinary host arrays (one array per field, reference filters/fields/regrid.py:204-208,
// 309) and point-major device batches, and streams a whole regrid through the GPU.
//
//   pinned pool   at_pinned_alloc/free: a caching allocator of page-locked host memory.  The
//                 arrays a filter hands back to the caller are pool blocks, so the D2H DMA
//                 writes the final array directly — no staging copy, no page faults of fresh
//                 memory on the way out.
//   upload        pageable fields -> (worker threads, non-temporal copy) -> pinned slot ->
//                 H2D per piece -> at_transpose into the batch's columns.  Fields that are
//                 already page-locked (pool blocks, registered memory) are DMA-ed in place.
//   download      at_transpose -> field-major device slot -> D2H straight into pinned
//                 destinations (asynchronous; a ticket says when), or through a pinned slot
//                 and worker copies for pageable destinations.
//   regrid        chunked upload -> SpMM / row gather -> download with three slots per
//                 direction, so staging, H2D, compute and D2H of consecutive chunks overlap
//                 (PCIe is full duplex).  Returns when every input byte has been consumed;
//                 the results keep arriving behind the ticket.
//   group         several engines, one per device (a device may appear twice), sharing one
//                 worker pool: a streamed regrid deals its chunks to whichever engine has a
//                 free input slot, so one process drives several PCIe links.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <sched.h>
#include <sys/mman.h>
#include <unistd.h>

#include "common.cuh"
#include "grib.cuh"
#include "hostcopy.h"

using namespace at;

// ------------------------------------------------------------------ pinned pool -------
namespace {

struct PinnedPool {
    struct Slab {
        char* base;
        size_t bytes, used;
        int64_t live;
        bool registered;  // mmap + cudaHostRegister (else cudaHostAlloc)
    };
    std::mutex mu;
    std::vector<Slab> slabs;
    std::unordered_map<size_t, std::vector<void*>> free_lists;              // size class -> blocks
    struct Block {
        size_t cls;
        int slab;
        bool live;
    };
    std::unordered_map<void*, Block> blocks;
    std::map<uintptr_t, uintptr_t> ranges;                                  // slab base -> end
    size_t reserved = 0, in_use = 0, limit = 0;

    static constexpr size_t kPage = 4096, kSlab = 64u << 20;

    size_t limit_bytes() {
        if (limit == 0) {
            const char* e = std::getenv("AT_B200_PINNED_LIMIT_MB");
            if (e != nullptr && std::atoll(e) > 0) {
                limit = static_cast<size_t>(std::atoll(e)) << 20;
            } else {
                const long pages = sysconf(_SC_PHYS_PAGES), psz = sysconf(_SC_PAGE_SIZE);
                limit = pages > 0 && psz > 0 ? static_cast<size_t>(pages) * static_cast<size_t>(psz) / 2 : (size_t(16) << 30);
            }
        }
        return limit;
    }

    // A slab of page-locked memory.  Anonymous memory backed by transparent huge pages and then
    // registered pins ~9x faster than cudaHostAlloc (measured on the gpurun hosts,
    // benchmarks/pin_rate_bench.cu: 16.8 GB/s from 4 threads against 1.8 GB/s), which is what a
    // cold pool costs the first large call; cudaHostAlloc remains the fallback.
    static bool make_slab(size_t bytes, Slab* out) {
        static const bool use_mmap = [] {
            const char* e = std::getenv("AT_B200_PINNED_MMAP");
            return !(e != nullptr && e[0] == '0');
        }();
        constexpr size_t kHuge = size_t(2) << 20;
        if (use_mmap) {
            const size_t span = bytes + kHuge;
            void* raw = mmap(nullptr, span, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
            if (raw != MAP_FAILED) {
                const uintptr_t lo = reinterpret_cast<uintptr_t>(raw), base = (lo + kHuge - 1) / kHuge * kHuge;
                if (base > lo) munmap(raw, base - lo);
                if (base + bytes < lo + span) munmap(reinterpret_cast<void*>(base + bytes), lo + span - (base + bytes));
                char* m = reinterpret_cast<char*>(base);
                madvise(m, bytes, MADV_HUGEPAGE);
                for (size_t o = 0; o < bytes; o += kPage) reinterpret_cast<volatile char*>(m)[o] = 0;  // fault the pages in
                if (cudaHostRegister(m, bytes, cudaHostRegisterPortable) == cudaSuccess) {
                    *out = Slab{m, bytes, 0, 0, true};
                    return true;
                }
                cudaGetLastError();
                munmap(m, bytes);
            }
        }
        void* base = nullptr;
        if (cudaHostAlloc(&base, bytes, cudaHostAllocPortable) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        *out = Slab{static_cast<char*>(base), bytes, 0, 0, false};
        return true;
    }

    void adopt_slab_locked(const Slab& slab) {
        slabs.push_back(slab);
        ranges[reinterpret_cast<uintptr_t>(slab.base)] = reinterpret_cast<uintptr_t>(slab.base) + slab.bytes;
        reserved += slab.bytes;
    }

    // Grow the pool ahead of `n` allocations of `bytes` each, new slabs pinned in parallel.
    void reserve(size_t bytes, int64_t n) {
        const size_t cls = (std::max<size_t>(bytes, 1) + kPage - 1) / kPage * kPage;
        const size_t slab_bytes = std::max(cls, kSlab), per_slab = slab_bytes / cls;
        int64_t missing = n;
        {
            std::lock_guard<std::mutex> lk(mu);
            auto it = free_lists.find(cls);
            if (it != free_lists.end()) missing -= static_cast<int64_t>(it->second.size());
            if (!slabs.empty() && slabs.back().base != nullptr) missing -= static_cast<int64_t>((slabs.back().bytes - slabs.back().used) / cls);
            if (missing <= 0) return;
            const size_t room = limit_bytes() > reserved ? (limit_bytes() - reserved) / slab_bytes : 0;
            missing = std::min<int64_t>((missing + static_cast<int64_t>(per_slab) - 1) / static_cast<int64_t>(per_slab), static_cast<int64_t>(room));
        }
        if (missing <= 1) return;  // a single slab is made by alloc() itself
        std::vector<Slab> made(static_cast<size_t>(missing));
        std::vector<uint8_t> ok(static_cast<size_t>(missing), 0);
        const int threads = static_cast<int>(std::min<int64_t>(4, missing));
        std::vector<std::thread> ts;
        for (int t = 0; t < threads; ++t)
            ts.emplace_back([&, t] {
                for (int64_t i = t; i < missing; i += threads) ok[static_cast<size_t>(i)] = make_slab(slab_bytes, &made[static_cast<size_t>(i)]);
            });
        for (auto& th : ts) th.join();
        std::lock_guard<std::mutex> lk(mu);
        // the partly used last slab keeps serving small requests: put the fresh ones after it
        for (int64_t i = 0; i < missing; ++i)
            if (ok[static_cast<size_t>(i)]) adopt_slab_locked(made[static_cast<size_t>(i)]);
    }

    int alloc(size_t bytes, void** out) {
        const size_t cls = (std::max<size_t>(bytes, 1) + kPage - 1) / kPage * kPage;
        std::lock_guard<std::mutex> lk(mu);
        auto it = free_lists.find(cls);
        if (it != free_lists.end() && !it->second.empty()) {
            void* p = it->second.back();
            it->second.pop_back();
            Block& b = blocks[p];
            b.live = true;
            slabs[static_cast<size_t>(b.slab)].live++;
            in_use += cls;
            *out = p;
            return AT_OK;
        }
        // any slab with room (reserve() may have added several at once), newest first
        int s = -1;
        for (int i = static_cast<int>(slabs.size()) - 1; i >= 0; --i) {
            const Slab& c = slabs[static_cast<size_t>(i)];
            if (c.base != nullptr && c.bytes - c.used >= cls) {
                s = i;
                break;
            }
        }
        if (s < 0) {
            const size_t want = std::max(cls, kSlab);
            if (reserved + want > limit_bytes())
                return set_error(AT_ERR_NOMEM, "at_pinned_alloc: pinned-memory limit of %zu MB reached (AT_B200_PINNED_LIMIT_MB)",
                                 limit_bytes() >> 20);
            Slab fresh;
            if (!make_slab(want, &fresh)) return set_error(AT_ERR_NOMEM, "at_pinned_alloc: could not pin %zu bytes of host memory", want);
            adopt_slab_locked(fresh);
            s = static_cast<int>(slabs.size()) - 1;
        }
        Slab& slab = slabs[static_cast<size_t>(s)];
        void* p = slab.base + slab.used;
        slab.used += cls;
        slab.live++;
        blocks[p] = Block{cls, s, true};
        in_use += cls;
        *out = p;
        return AT_OK;
    }

    int release(void* p) {
        std::lock_guard<std::mutex> lk(mu);
        auto it = blocks.find(p);
        if (it == blocks.end()) return set_error(AT_ERR_INVALID, "at_pinned_free: %p is not a live pool block", p);
        if (!it->second.live) return set_error(AT_ERR_INVALID, "at_pinned_free: double free of %p", p);
        it->second.live = false;
        free_lists[it->second.cls].push_back(p);
        slabs[static_cast<size_t>(it->second.slab)].live--;
        in_use -= it->second.cls;
        return AT_OK;
    }

    // Give slabs without live blocks back to the system.
    void trim() {
        std::lock_guard<std::mutex> lk(mu);
        for (size_t s = 0; s < slabs.size(); ++s) {
            Slab& slab = slabs[s];
            if (slab.base == nullptr || slab.live != 0) continue;
            for (auto it = blocks.begin(); it != blocks.end();) {
                if (it->second.slab == static_cast<int>(s)) {
                    auto& fl = free_lists[it->second.cls];
                    fl.erase(std::remove(fl.begin(), fl.end(), it->first), fl.end());
                    it = blocks.erase(it);
                } else {
                    ++it;
                }
            }
            ranges.erase(reinterpret_cast<uintptr_t>(slab.base));
            if (slab.registered) {
                cudaHostUnregister(slab.base);
                munmap(slab.base, slab.bytes);
            } else {
                cudaFreeHost(slab.base);
            }
            reserved -= slab.bytes;
            slab.base = nullptr;
            slab.used = slab.bytes;  // never carve from it again
        }
    }

    bool owns(const void* p) {
        std::lock_guard<std::mutex> lk(mu);
        const uintptr_t a = reinterpret_cast<uintptr_t>(p);
        auto it = ranges.upper_bound(a);
        if (it == ranges.begin()) return false;
        --it;
        return a < it->second;
    }
};

PinnedPool& pool() {
    static PinnedPool* p = new PinnedPool();  // leaked on purpose: blocks may outlive static destructors
    return *p;
}

// Is [p, p + bytes) page-locked memory the DMA engines can read / write in place?
bool is_page_locked(const void* p) {
    if (pool().owns(p)) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

constexpr int kSlots = 3;
constexpr size_t kPiece = 8u << 20;        // staging / DMA granularity: every cudaMemcpyAsync costs microseconds
                                           // under the driver's lock, so pieces are whole fields as a rule
constexpr size_t kMaxSlotBytes = 256u << 20;
constexpr size_t kAlign = 256;

size_t round_up(size_t n, size_t m) { return (n + m - 1) / m * m; }

// The workers of a group serve every device of the group: a copy for a device's stream is
// issued with that device current.
void use_device(int dev) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != dev) cudaSetDevice(dev);
}

}  // namespace

extern "C" int at_pinned_alloc(size_t bytes, void** out) {
    AT_REQUIRE(out != nullptr, "at_pinned_alloc: out is null");
    *out = nullptr;
    return pool().alloc(bytes, out);
}

extern "C" int at_pinned_alloc_many(size_t bytes, int64_t n, void** out) {
    AT_REQUIRE(out != nullptr && n >= 0, "at_pinned_alloc_many: bad arguments");
    for (int64_t i = 0; i < n; ++i) out[i] = nullptr;
    pool().reserve(bytes, n);
    for (int64_t i = 0; i < n; ++i) {
        const int rc = pool().alloc(bytes, &out[i]);
        if (rc != AT_OK) {  // all or nothing
            for (int64_t j = 0; j < i; ++j) {
                pool().release(out[j]);
                out[j] = nullptr;
            }
            return rc;
        }
    }
    return AT_OK;
}

extern "C" int at_pinned_free(void* ptr) {
    if (ptr == nullptr) return AT_OK;
    return pool().release(ptr);
}

extern "C" int at_pinned_trim(void) {
    pool().trim();
    return AT_OK;
}

extern "C" int at_pinned_stats(size_t* in_use, size_t* reserved) {
    std::lock_guard<std::mutex> lk(pool().mu);
    if (in_use) *in_use = pool().in_use;
    if (reserved) *reserved = pool().reserved;
    return AT_OK;
}

// ------------------------------------------------------------------ engine ------------
struct at_hostio {
    int device = 0;
    std::shared_ptr<WorkerPool> workers;  // shared by the engines of a group
    std::mutex mu;  // one operation at a time

    size_t in_slot_bytes = 0, out_slot_bytes = 0, hout_slot_bytes = 0;
    char* h_in[kSlots] = {nullptr, nullptr, nullptr};
    char* d_in[kSlots] = {nullptr, nullptr, nullptr};
    char* d_out[kSlots] = {nullptr, nullptr, nullptr};
    char* h_out[kSlots] = {nullptr, nullptr, nullptr};
    cudaEvent_t in_free[kSlots] = {}, h2d_done[kSlots] = {}, out_free[kSlots] = {}, unpacked[kSlots] = {};
    uint64_t in_seq = 0, out_seq = 0;
    cudaStream_t s_in = nullptr, s_out = nullptr, s_compute = nullptr;
    cudaEvent_t ev_sync = nullptr;
    // GRIB chunks whose per-field decode status words (copied back into h_in[slot] behind the
    // table) have not been read yet: the chunk's field count and the call's index of its first
    int status_nf[kSlots] = {0, 0, 0};
    int64_t status_first[kSlots] = {0, 0, 0};

    char* d_x = nullptr;
    char* d_y = nullptr;
    size_t d_x_bytes = 0, d_y_bytes = 0;

    std::mutex ticket_mu;
    std::vector<cudaEvent_t> tickets;
    std::vector<int64_t> free_tickets;
    std::vector<uint8_t> ticket_live;
};

namespace {

int ensure_device_buffer(char** buf, size_t* have, size_t want) {
    if (*have >= want) return AT_OK;
    if (*buf != nullptr) {
        AT_CUDA_TRY(cudaDeviceSynchronize());
        cudaFree(*buf);
        *buf = nullptr;
        *have = 0;
    }
    AT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(buf), want));
    *have = want;
    return AT_OK;
}

int ensure_in_slots(at_hostio* io, size_t bytes, bool need_host) {
    if (io->in_slot_bytes < bytes) {
        AT_CUDA_TRY(cudaDeviceSynchronize());
        for (int s = 0; s < kSlots; ++s) {
            if (io->h_in[s]) pool().release(io->h_in[s]);
            if (io->d_in[s]) cudaFree(io->d_in[s]);
            io->h_in[s] = io->d_in[s] = nullptr;
        }
        io->in_slot_bytes = 0;
        for (int s = 0; s < kSlots; ++s) AT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&io->d_in[s]), bytes));
        io->in_slot_bytes = bytes;
    }
    if (need_host)
        for (int s = 0; s < kSlots; ++s)
            if (io->h_in[s] == nullptr) {  // staging slots are blocks of the pinned pool (it pins fast, §3.7)
                const int rc = pool().alloc(io->in_slot_bytes, reinterpret_cast<void**>(&io->h_in[s]));
                if (rc != AT_OK) return rc;
            }
    return AT_OK;
}

int ensure_out_slots(at_hostio* io, size_t bytes, bool need_host) {
    if (io->out_slot_bytes < bytes) {
        AT_CUDA_TRY(cudaDeviceSynchronize());
        for (int s = 0; s < kSlots; ++s) {
            if (io->d_out[s]) cudaFree(io->d_out[s]);
            if (io->h_out[s]) pool().release(io->h_out[s]);
            io->d_out[s] = io->h_out[s] = nullptr;
        }
        io->out_slot_bytes = io->hout_slot_bytes = 0;
        for (int s = 0; s < kSlots; ++s) AT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&io->d_out[s]), bytes));
        io->out_slot_bytes = bytes;
    }
    if (need_host && io->hout_slot_bytes < io->out_slot_bytes) {
        for (int s = 0; s < kSlots; ++s) {
            if (io->h_out[s]) pool().release(io->h_out[s]);
            io->h_out[s] = nullptr;
            const int rc = pool().alloc(io->out_slot_bytes, reinterpret_cast<void**>(&io->h_out[s]));
            if (rc != AT_OK) return rc;
        }
        io->hout_slot_bytes = io->out_slot_bytes;
    }
    return AT_OK;
}

// Fields per chunk: at most kMaxSlotBytes per slot, at least `min_chunks` chunks (four per
// engine) for jobs worth pipelining, a multiple of `multiple` (4 when the chunk becomes a
// point-major batch).
int64_t chunk_fields(int64_t n_fields, size_t stride, int64_t multiple, int64_t min_chunks = 4) {
    int64_t by_slot = std::max<int64_t>(1, static_cast<int64_t>(kMaxSlotBytes / std::max<size_t>(stride, 1)));
    int64_t chunk = std::min<int64_t>(n_fields, by_slot);
    const size_t total = stride * static_cast<size_t>(n_fields);
    if (total > (size_t(64) << 20)) chunk = std::min<int64_t>(chunk, (n_fields + min_chunks - 1) / min_chunks);
    chunk = std::max<int64_t>(multiple, chunk / multiple * multiple);
    return chunk;
}

// Bytes per staging task.  The tasks of a chunk are handed out dynamically and the chunk ends
// with a barrier, so the last round of tasks should be short against the whole: at least four
// tasks per thread when the fields are large enough (pieces stay >= 1 MB — every H2D copy costs
// microseconds under the driver's lock — and <= kPiece).
size_t piece_bytes(size_t field_bytes, int n_fields, int n_threads) {
    size_t pieces = (field_bytes + kPiece - 1) / kPiece;
    const size_t want_tasks = static_cast<size_t>(4 * std::max(1, n_threads));
    while (pieces * static_cast<size_t>(n_fields) < want_tasks && field_bytes / (pieces + 1) >= (size_t(1) << 20)) ++pieces;
    if (n_threads > 1 && (pieces * static_cast<size_t>(n_fields)) % static_cast<size_t>(n_threads) != 0) {
        // one more split when it makes the task count a multiple of the thread count
        for (size_t p = pieces; p <= pieces + 8; ++p)
            if ((p * static_cast<size_t>(n_fields)) % static_cast<size_t>(n_threads) == 0 && field_bytes / p >= (size_t(1) << 20)) {
                pieces = p;
                break;
            }
    }
    const size_t piece = (field_bytes + pieces - 1) / pieces;
    return std::max<size_t>(round_up(piece, 4096), 4096);
}

struct Classified {
    std::vector<uint8_t> pinned;
    bool any_pinned = false, all_pinned = true;
};

Classified classify(const void* const* ptrs, int64_t n) {
    Classified c;
    c.pinned.resize(static_cast<size_t>(n));
    for (int64_t f = 0; f < n; ++f) {
        const bool p = is_page_locked(ptrs[f]);
        c.pinned[static_cast<size_t>(f)] = p;
        c.any_pinned |= p;
        c.all_pinned &= p;
    }
    return c;
}

// Stage + H2D + pack one chunk of fields into columns [0, nf) of the point-major buffer d_pm.
int upload_chunk(at_hostio* io, const void* const* fields, const uint8_t* pinned, int nf, int64_t n_points, int elem,
                 size_t stride, void* d_pm, int64_t ld, cudaStream_t st) {
    const int slot = static_cast<int>(io->in_seq++ % kSlots);
    AT_CUDA_TRY(cudaEventSynchronize(io->in_free[slot]));  // the pack that last read this slot
    const size_t fb = static_cast<size_t>(n_points) * static_cast<size_t>(elem);
    const size_t piece = piece_bytes(fb, nf, io->workers->size());
    const int64_t ppf = static_cast<int64_t>((fb + piece - 1) / piece);
    std::atomic<int> err{static_cast<int>(cudaSuccess)};
    char* const h = io->h_in[slot];
    char* const d = io->d_in[slot];
    cudaStream_t s_in = io->s_in;
    const int dev = io->device;
    io->workers->parallel_for(static_cast<int64_t>(nf) * ppf, [&](int64_t i) {
        use_device(dev);
        const int64_t f = i / ppf;
        const size_t off = static_cast<size_t>(i % ppf) * piece, len = std::min(piece, fb - off);
        const char* src = static_cast<const char*>(fields[f]) + off;
        char* dev = d + static_cast<size_t>(f) * stride + off;
        cudaError_t e;
        if (pinned[f]) {
            e = cudaMemcpyAsync(dev, src, len, cudaMemcpyHostToDevice, s_in);
        } else {
            char* stg = h + static_cast<size_t>(f) * stride + off;
            copy_streaming(stg, src, len);
            e = cudaMemcpyAsync(dev, stg, len, cudaMemcpyHostToDevice, s_in);
        }
        if (e != cudaSuccess) err.store(static_cast<int>(e));
    });
    if (err.load() != static_cast<int>(cudaSuccess))
        return set_error(AT_ERR_CUDA, "hostio upload: %s", cudaGetErrorString(static_cast<cudaError_t>(err.load())));
    AT_CUDA_TRY(cudaEventRecord(io->h2d_done[slot], s_in));
    AT_CUDA_TRY(cudaStreamWaitEvent(st, io->h2d_done[slot], 0));
    int rc = at_transpose(d, nf, n_points, static_cast<int64_t>(stride / static_cast<size_t>(elem)), d_pm, ld, elem, st);
    if (rc != AT_OK) return rc;
    AT_CUDA_TRY(cudaEventRecord(io->in_free[slot], st));
    return AT_OK;
}

// The packed-message variant of upload_chunk: only the packed values of each field (data_length
// octets, 2 bytes per point at 16 bits) are staged and cross PCIe; the slot starts with the
// table of kernel parameters, and grib_unpack_kernel takes the place of the pack transposition.
// The table is followed by one int32 status word per field (CCSDS and complex decode, bitmap
// count; zero when the field decoded).
size_t grib_table_bytes(int nf) { return round_up(static_cast<size_t>(nf) * (sizeof(GribColumn) + sizeof(int32_t)), 4096); }

// Largest footprint of a field in a chunk buffer (+ its share of the parameter table).
size_t grib_packed_stride(const at_grib_field_t* infos, int64_t n_fields, int64_t n_points) {
    size_t stride = 0;
    for (int64_t f = 0; f < n_fields; ++f)
        stride = std::max(stride, grib_footprint(infos[f], n_points).total() + sizeof(GribColumn) + sizeof(int32_t));
    return stride;
}

// Read the status words of the chunk that last used `slot` (waits for its decode).  A
// malformed field is AT_ERR_INVALID naming the message by its index in the call.
int status_check_slot(at_hostio* io, int slot) {
    const int nf = io->status_nf[slot];
    if (nf == 0) return AT_OK;
    io->status_nf[slot] = 0;
    AT_CUDA_TRY(cudaEventSynchronize(io->in_free[slot]));
    const int32_t* status = reinterpret_cast<const int32_t*>(io->h_in[slot] + static_cast<size_t>(nf) * sizeof(GribColumn));
    for (int f = 0; f < nf; ++f)
        if (status[f] != 0)
            return set_error(AT_ERR_INVALID, "GRIB decode: message %lld: %s", (long long)(io->status_first[slot] + f), grib_status_text(status[f]));
    return AT_OK;
}

// Every slot's status words; all are read (and cleared) even after the first error.
int status_check_all(at_hostio* io) {
    int rc = AT_OK;
    for (int s = 0; s < kSlots; ++s) {
        const int r = status_check_slot(io, s);
        if (rc == AT_OK) rc = r;
    }
    return rc;
}

// A call that fails leaves the engine idle: whatever it queued has run when it returns, and
// status words of its chunks are not reported by the next call.
void quiesce(at_hostio* io) {
    cudaStreamSynchronize(io->s_in);
    cudaStreamSynchronize(io->s_compute);
    cudaStreamSynchronize(io->s_out);
    for (int s = 0; s < kSlots; ++s) io->status_nf[s] = 0;
}

int upload_chunk_grib(at_hostio* io, const void* const* messages, const at_grib_field_t* infos, int nf, int64_t n_points,
                      int x_dtype, void* d_pm, int64_t ld, cudaStream_t st, int64_t first) {
    const int slot = static_cast<int>(io->in_seq++ % kSlots);
    AT_CUDA_TRY(cudaEventSynchronize(io->in_free[slot]));  // the unpack that last read this slot
    int rc0 = status_check_slot(io, slot);
    if (rc0 != AT_OK) return rc0;
    char* const h = io->h_in[slot];
    char* const d = io->d_in[slot];
    GribColumn* table = reinterpret_cast<GribColumn*>(h);
    int32_t* status = reinterpret_cast<int32_t*>(h + static_cast<size_t>(nf) * sizeof(GribColumn));
    struct Task {
        const char* src;
        size_t at, len;
    };
    std::vector<Task> tasks;
    size_t cursor = grib_table_bytes(nf);
    bool any_bitmap = false;
    int64_t max_rsi = 0, max_tiles = 0;
    for (int f = 0; f < nf; ++f) {
        const int rc = grib_column_of(infos[f], n_points, static_cast<int64_t>(cursor), &table[f]);
        if (rc != AT_OK) return rc;
        status[f] = 0;
        if (table[f].packing == AT_GRIB_CCSDS) max_rsi = std::max(max_rsi, ccsds_rsi_count(infos[f], table[f].n_values));
        if (table[f].packing == AT_GRIB_COMPLEX) max_tiles = std::max(max_tiles, complex_tile_count(table[f].n_values));
        const GribFootprint fp = grib_footprint(infos[f], n_points);
        // what the kernel reads: the packed values (the section may be padded), and the bitmap
        const char* msg = static_cast<const char*>(messages[f]);
        for (size_t o = 0; o < fp.value_octets; o += kPiece) tasks.push_back({msg + infos[f].data_offset + o, cursor + o, std::min(kPiece, fp.value_octets - o)});
        if (infos[f].has_bitmap) {
            any_bitmap = true;
            for (size_t o = 0; o < fp.bitmap_octets; o += kPiece)
                tasks.push_back({msg + infos[f].bitmap_offset + o, cursor + fp.values + o, std::min(kPiece, fp.bitmap_octets - o)});
        }
        cursor += fp.total();
    }
    if (cursor > io->in_slot_bytes) return set_error(AT_ERR_INVALID, "hostio grib upload: chunk of %zu bytes exceeds the slot (%zu)", cursor, io->in_slot_bytes);
    cudaStream_t s_in = io->s_in;
    const bool with_status = max_rsi > 0 || max_tiles > 0 || any_bitmap;
    const size_t table_octets = static_cast<size_t>(nf) * (sizeof(GribColumn) + (with_status ? sizeof(int32_t) : 0));
    AT_CUDA_TRY(cudaMemcpyAsync(d, h, table_octets, cudaMemcpyHostToDevice, s_in));
    std::atomic<int> err{static_cast<int>(cudaSuccess)};
    const int dev = io->device;
    io->workers->parallel_for(static_cast<int64_t>(tasks.size()), [&](int64_t i) {
        use_device(dev);
        const Task& t = tasks[static_cast<size_t>(i)];
        copy_streaming(h + t.at, t.src, t.len);
        const cudaError_t e = cudaMemcpyAsync(d + t.at, h + t.at, t.len, cudaMemcpyHostToDevice, s_in);
        if (e != cudaSuccess) err.store(static_cast<int>(e));
    });
    if (err.load() != static_cast<int>(cudaSuccess))
        return set_error(AT_ERR_CUDA, "hostio grib upload: %s", cudaGetErrorString(static_cast<cudaError_t>(err.load())));
    AT_CUDA_TRY(cudaEventRecord(io->h2d_done[slot], s_in));
    AT_CUDA_TRY(cudaStreamWaitEvent(st, io->h2d_done[slot], 0));
    int32_t* d_status = with_status ? reinterpret_cast<int32_t*>(d + static_cast<size_t>(nf) * sizeof(GribColumn)) : nullptr;
    const GribColumn* d_table = reinterpret_cast<const GribColumn*>(d);
    // CCSDS and complex fields: section 7 -> 32-bit words in their scratch
    int rc = ccsds_decode_launch(reinterpret_cast<uint8_t*>(d), d_table, nf, d_status, max_rsi, st);
    if (rc == AT_OK) rc = complex_decode_launch(reinterpret_cast<uint8_t*>(d), d_table, nf, d_status, max_tiles, st);
    if (rc == AT_OK) rc = grib_unpack_launch(reinterpret_cast<uint8_t*>(d), d_table, nf, n_points, x_dtype, d_pm, ld, any_bitmap, d_status, st);
    if (rc != AT_OK) return rc;
    if (with_status) {  // status words back to the host, read when the slot is reused or the call ends
        AT_CUDA_TRY(cudaMemcpyAsync(status, d_status, static_cast<size_t>(nf) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        io->status_nf[slot] = nf;
        io->status_first[slot] = first;
    }
    AT_CUDA_TRY(cudaEventRecord(io->in_free[slot], st));
    return AT_OK;
}

struct PendingHostCopy {
    int slot = -1, nf = 0;
    void* const* dst = nullptr;
};

// Host half of a download into pageable destinations: wait for the slot's D2H, copy out.
int finish_host_copy(at_hostio* io, const PendingHostCopy& p, size_t fb, size_t stride) {
    if (p.slot < 0) return AT_OK;
    AT_CUDA_TRY(cudaEventSynchronize(io->out_free[p.slot]));
    const int64_t ppf = static_cast<int64_t>((fb + kPiece - 1) / kPiece);
    const char* h = io->h_out[p.slot];
    io->workers->parallel_for(static_cast<int64_t>(p.nf) * ppf, [&](int64_t i) {
        const int64_t f = i / ppf;
        const size_t off = static_cast<size_t>(i % ppf) * kPiece, len = std::min(kPiece, fb - off);
        std::memcpy(static_cast<char*>(p.dst[f]) + off, h + static_cast<size_t>(f) * stride + off, len);
    });
    return AT_OK;
}

// Unpack + D2H of columns [0, nf) of d_pm.  Pinned destinations: fully asynchronous.
// Pageable destinations: the D2H lands in a pinned slot; `pending` carries the host copy,
// which the caller finishes one chunk later (so it overlaps the next chunk's DMA).
int download_chunk(at_hostio* io, const void* d_pm, int64_t ld, int nf, int64_t n_points, int elem, size_t stride,
                   void* const* dst, bool all_pinned, cudaStream_t st, PendingHostCopy* pending) {
    const int slot = static_cast<int>(io->out_seq++ % kSlots);
    AT_CUDA_TRY(cudaStreamWaitEvent(st, io->out_free[slot], 0));  // the D2H that last read this slot
    int rc = at_transpose(d_pm, n_points, nf, ld, io->d_out[slot], static_cast<int64_t>(stride / static_cast<size_t>(elem)), elem, st);
    if (rc != AT_OK) return rc;
    AT_CUDA_TRY(cudaEventRecord(io->unpacked[slot], st));
    AT_CUDA_TRY(cudaStreamWaitEvent(io->s_out, io->unpacked[slot], 0));
    const size_t fb = static_cast<size_t>(n_points) * static_cast<size_t>(elem);
    if (all_pinned) {
        for (int f = 0; f < nf;) {
            int g = f + 1;
            if (stride == fb)  // adjacent destinations (one [F, n] array) go in one copy
                while (g < nf && static_cast<char*>(dst[g]) == static_cast<char*>(dst[g - 1]) + fb) ++g;
            AT_CUDA_TRY(cudaMemcpyAsync(dst[f], io->d_out[slot] + static_cast<size_t>(f) * stride,
                                        g - f == 1 ? fb : fb * static_cast<size_t>(g - f), cudaMemcpyDeviceToHost, io->s_out));
            f = g;
        }
    } else {
        AT_CUDA_TRY(cudaMemcpyAsync(io->h_out[slot], io->d_out[slot], static_cast<size_t>(nf) * stride, cudaMemcpyDeviceToHost, io->s_out));
        pending->slot = slot;
        pending->nf = nf;
        pending->dst = dst;
    }
    AT_CUDA_TRY(cudaEventRecord(io->out_free[slot], io->s_out));
    return AT_OK;
}

int new_ticket(at_hostio* io, cudaStream_t after, int64_t* ticket) {
    std::lock_guard<std::mutex> lk(io->ticket_mu);
    int64_t t;
    if (!io->free_tickets.empty()) {
        t = io->free_tickets.back();
        io->free_tickets.pop_back();
    } else {
        cudaEvent_t e;
        AT_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        io->tickets.push_back(e);
        io->ticket_live.push_back(0);
        t = static_cast<int64_t>(io->tickets.size()) - 1;
    }
    cudaError_t e = cudaEventRecord(io->tickets[static_cast<size_t>(t)], after);
    if (e != cudaSuccess) {
        io->free_tickets.push_back(t);
        return set_error(AT_ERR_CUDA, "hostio: cudaEventRecord failed: %s", cudaGetErrorString(e));
    }
    io->ticket_live[static_cast<size_t>(t)] = 1;
    *ticket = t;
    return AT_OK;
}

// Cores (not hardware threads) this process may run on: memory copies do not speed up when two
// staging threads share a core.
int physical_cores() {
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) != 0) return std::max(1u, std::thread::hardware_concurrency() / 2);
    std::vector<std::string> groups;
    int cpus = 0;
    for (int c = 0; c < CPU_SETSIZE; ++c) {
        if (!CPU_ISSET(c, &set)) continue;
        ++cpus;
        char path[128], line[256] = {0};
        snprintf(path, sizeof(path), "/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list", c);
        FILE* f = fopen(path, "r");
        if (f == nullptr) continue;
        if (fgets(line, sizeof(line), f) != nullptr && std::find(groups.begin(), groups.end(), line) == groups.end()) groups.push_back(line);
        fclose(f);
    }
    if (groups.empty()) return std::max(1, cpus / 2);
    return static_cast<int>(groups.size());
}

// Makes `dev` current; the caller's device is current again at the end of the scope, also when
// the scope switched devices in between (the engines of a group).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && (cudaGetDevice(&cur) != cudaSuccess || cur != prev)) cudaSetDevice(prev);
    }
};

int default_copy_threads(int n_threads) {
    if (n_threads > 0) return n_threads;
    const char* e = std::getenv("AT_B200_COPY_THREADS");
    if (e != nullptr && std::atoi(e) > 0) return std::min(256, std::atoi(e));
    // ~50 GB/s of staging saturates a PCIe Gen5 x16 link; measured on a 16-core host, 6-10
    // threads do that and more only contend for memory bandwidth with the DMA engines
    return std::max(1, std::min(8, physical_cores() / 2));
}

}  // namespace

extern "C" int at_hostio_destroy(at_hostio_t* io) {
    if (io == nullptr) return AT_OK;
    cudaSetDevice(io->device);
    cudaDeviceSynchronize();
    io->workers.reset();
    for (int s = 0; s < kSlots; ++s) {
        if (io->h_in[s]) pool().release(io->h_in[s]);
        if (io->h_out[s]) pool().release(io->h_out[s]);
        if (io->d_in[s]) cudaFree(io->d_in[s]);
        if (io->d_out[s]) cudaFree(io->d_out[s]);
        if (io->in_free[s]) cudaEventDestroy(io->in_free[s]);
        if (io->h2d_done[s]) cudaEventDestroy(io->h2d_done[s]);
        if (io->out_free[s]) cudaEventDestroy(io->out_free[s]);
        if (io->unpacked[s]) cudaEventDestroy(io->unpacked[s]);
    }
    for (cudaEvent_t e : io->tickets) cudaEventDestroy(e);
    if (io->ev_sync) cudaEventDestroy(io->ev_sync);
    if (io->d_x) cudaFree(io->d_x);
    if (io->d_y) cudaFree(io->d_y);
    if (io->s_in) cudaStreamDestroy(io->s_in);
    if (io->s_out) cudaStreamDestroy(io->s_out);
    if (io->s_compute) cudaStreamDestroy(io->s_compute);
    delete io;
    return AT_OK;
}

// An engine on `dev` (the current device) staging with `workers`.
static int make_engine(int dev, std::shared_ptr<WorkerPool> workers, at_hostio** out) {
    at_hostio* io = new at_hostio();
    io->device = dev;
    io->workers = std::move(workers);
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) {
        if (e == cudaSuccess) e = r;
    };
    for (int s = 0; s < kSlots; ++s) {
        ok(cudaEventCreateWithFlags(&io->in_free[s], cudaEventDisableTiming));
        ok(cudaEventCreateWithFlags(&io->h2d_done[s], cudaEventDisableTiming));
        ok(cudaEventCreateWithFlags(&io->out_free[s], cudaEventDisableTiming));
        ok(cudaEventCreateWithFlags(&io->unpacked[s], cudaEventDisableTiming));
    }
    ok(cudaEventCreateWithFlags(&io->ev_sync, cudaEventDisableTiming));
    ok(cudaStreamCreateWithFlags(&io->s_in, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&io->s_out, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&io->s_compute, cudaStreamNonBlocking));
    if (e != cudaSuccess) {
        at_hostio_destroy(io);
        return set_error(AT_ERR_CUDA, "at_hostio_create: %s", cudaGetErrorString(e));
    }
    *out = io;
    return AT_OK;
}

extern "C" int at_hostio_create(int32_t n_threads, at_hostio_t** out) {
    AT_REQUIRE(out != nullptr, "at_hostio_create: out is null");
    *out = nullptr;
    AT_REQUIRE(n_threads >= 0 && n_threads <= 256, "at_hostio_create: n_threads must be in [0, 256]");
    int dev = 0;
    AT_CUDA_TRY(cudaGetDevice(&dev));
    return make_engine(dev, std::make_shared<WorkerPool>(default_copy_threads(n_threads), [dev] { cudaSetDevice(dev); }), out);
}

extern "C" int at_hostio_threads(const at_hostio_t* io, int32_t* n_threads, int32_t* nontemporal) {
    AT_REQUIRE(io != nullptr, "at_hostio_threads: null engine");
    if (n_threads) *n_threads = io->workers->size();
    if (nontemporal) *nontemporal = copy_streaming_is_nontemporal() ? 1 : 0;
    return AT_OK;
}

extern "C" int at_hostio_upload(at_hostio_t* io, const void* const* fields, int64_t n_fields, int64_t n_points,
                                int elem_size, void* d_pm, int64_t ld, void* stream) {
    AT_REQUIRE(io != nullptr && fields != nullptr && d_pm != nullptr, "at_hostio_upload: null argument");
    AT_REQUIRE(elem_size == 4 || elem_size == 8, "at_hostio_upload: elem_size must be 4 or 8");
    AT_REQUIRE(n_fields >= 0 && n_points >= 0 && ld >= n_fields, "at_hostio_upload: bad sizes");
    if (n_fields == 0 || n_points == 0) return AT_OK;
    for (int64_t f = 0; f < n_fields; ++f) AT_REQUIRE(fields[f] != nullptr, "at_hostio_upload: field %lld is null", (long long)f);
    std::lock_guard<std::mutex> lk(io->mu);
    DeviceGuard guard(io->device);
    const size_t fb = static_cast<size_t>(n_points) * static_cast<size_t>(elem_size), stride = round_up(fb, kAlign);
    const int64_t chunk = chunk_fields(n_fields, stride, 1);
    const Classified cls = classify(fields, n_fields);
    int rc = ensure_in_slots(io, static_cast<size_t>(chunk) * stride, !cls.all_pinned);
    if (rc != AT_OK) return rc;
    cudaStream_t st = as_stream(stream);
    for (int64_t c0 = 0; c0 < n_fields; c0 += chunk) {
        const int nf = static_cast<int>(std::min<int64_t>(chunk, n_fields - c0));
        rc = upload_chunk(io, fields + c0, cls.pinned.data() + c0, nf, n_points, elem_size, stride,
                          static_cast<char*>(d_pm) + static_cast<size_t>(c0) * static_cast<size_t>(elem_size), ld, st);
        if (rc != AT_OK) return rc;
    }
    // page-locked inputs were read in place: they belong to the caller again only after the DMA
    if (cls.any_pinned) AT_CUDA_TRY(cudaStreamSynchronize(io->s_in));
    return AT_OK;
}

extern "C" int at_hostio_download(at_hostio_t* io, const void* d_pm, int64_t ld, int64_t n_fields, int64_t n_points,
                                  int elem_size, void* const* dst, void* stream, int64_t* ticket) {
    AT_REQUIRE(io != nullptr && d_pm != nullptr && dst != nullptr && ticket != nullptr, "at_hostio_download: null argument");
    AT_REQUIRE(elem_size == 4 || elem_size == 8, "at_hostio_download: elem_size must be 4 or 8");
    AT_REQUIRE(n_fields >= 0 && n_points >= 0 && ld >= n_fields, "at_hostio_download: bad sizes");
    *ticket = -1;
    if (n_fields == 0 || n_points == 0) return AT_OK;
    for (int64_t f = 0; f < n_fields; ++f) AT_REQUIRE(dst[f] != nullptr, "at_hostio_download: destination %lld is null", (long long)f);
    std::lock_guard<std::mutex> lk(io->mu);
    DeviceGuard guard(io->device);
    const size_t fb = static_cast<size_t>(n_points) * static_cast<size_t>(elem_size), stride = round_up(fb, kAlign);
    const int64_t chunk = chunk_fields(n_fields, stride, 1);
    const Classified cls = classify(dst, n_fields);
    int rc = ensure_out_slots(io, static_cast<size_t>(chunk) * stride, !cls.all_pinned);
    if (rc != AT_OK) return rc;
    cudaStream_t st = as_stream(stream);
    PendingHostCopy pending, next;
    for (int64_t c0 = 0; c0 < n_fields; c0 += chunk) {
        const int nf = static_cast<int>(std::min<int64_t>(chunk, n_fields - c0));
        next = PendingHostCopy();
        rc = download_chunk(io, static_cast<const char*>(d_pm) + static_cast<size_t>(c0) * static_cast<size_t>(elem_size), ld, nf,
                            n_points, elem_size, stride, dst + c0, cls.all_pinned, st, &next);
        if (rc != AT_OK) return rc;
        rc = finish_host_copy(io, pending, fb, stride);
        if (rc != AT_OK) return rc;
        pending = next;
    }
    rc = finish_host_copy(io, pending, fb, stride);
    if (rc != AT_OK) return rc;
    if (cls.all_pinned) return new_ticket(io, io->s_out, ticket);
    return AT_OK;  // pageable destinations are complete on return
}

extern "C" int at_hostio_wait(at_hostio_t* io, int64_t ticket) {
    AT_REQUIRE(io != nullptr, "at_hostio_wait: null engine");
    if (ticket < 0) return AT_OK;
    cudaEvent_t e;
    {
        std::lock_guard<std::mutex> lk(io->ticket_mu);
        AT_REQUIRE(ticket < static_cast<int64_t>(io->tickets.size()) && io->ticket_live[static_cast<size_t>(ticket)],
                   "at_hostio_wait: ticket %lld is not outstanding", (long long)ticket);
        e = io->tickets[static_cast<size_t>(ticket)];
    }
    const cudaError_t r = cudaEventSynchronize(e);
    {
        std::lock_guard<std::mutex> lk(io->ticket_mu);
        io->ticket_live[static_cast<size_t>(ticket)] = 0;
        io->free_tickets.push_back(ticket);
    }
    if (r != cudaSuccess) return set_error(AT_ERR_CUDA, "at_hostio_wait: %s", cudaGetErrorString(r));
    return AT_OK;
}

namespace {

// The ops that apply a matrix: the plain SpMM and the missing-aware ones (at_spmm_missing).
bool is_matrix_op(int op) { return op == AT_HOSTIO_SPMM || op == AT_HOSTIO_SPMM_MISSING_ALL || op == AT_HOSTIO_SPMM_MISSING_HEAVIEST; }
// First check of every streamed-regrid entry point: an unknown op is refused before anything else.
int check_op(int op, const char* who) {
    AT_REQUIRE(is_matrix_op(op) || op == AT_HOSTIO_GATHER, "%s: unknown op %d (AT_HOSTIO_SPMM, AT_HOSTIO_GATHER, AT_HOSTIO_SPMM_MISSING_ALL, AT_HOSTIO_SPMM_MISSING_HEAVIEST)", who, op);
    return AT_OK;
}

// What every chunk of one streamed regrid shares, whichever engine runs it.
struct RegridJob {
    int op, x_dtype, y_dtype, xe, ye;
    const void* const* fields_in;
    const at_grib_field_t* grib;  // != nullptr: fields_in are whole GRIB messages, grib[f] their scans
    int64_t n_src, n_tgt, chunk;
    size_t in_stride, out_fb, out_stride;
    void* d_Y;  // optional resident result [n_tgt, ldy] (single engine only)
    int64_t ldy;
    void* const* fields_out;
    Classified cin, cout;
};

// Fields [c0, c0 + nf) on engine `io` (its device current): stage + H2D + pack (or unpack),
// SpMM or row gather, unpack + D2H.  The pageable host copy of the engine's previous chunk
// (`pending`) is finished behind this chunk's DMA.
int regrid_chunk(at_hostio* io, const RegridJob& j, const at_csr_t* csr, const int64_t* gather_idx, int64_t c0, int nf,
                 PendingHostCopy* pending) {
    cudaStream_t sc = io->s_compute;
    int rc = j.grib != nullptr ? upload_chunk_grib(io, j.fields_in + c0, j.grib + c0, nf, j.n_src, j.x_dtype, io->d_x, j.chunk, sc, c0)
                               : upload_chunk(io, j.fields_in + c0, j.cin.pinned.data() + c0, nf, j.n_src, j.xe, j.in_stride, io->d_x, j.chunk, sc);
    if (rc != AT_OK) return rc;
    char* y = j.d_Y != nullptr ? static_cast<char*>(j.d_Y) + static_cast<size_t>(c0) * j.ye : io->d_y;
    const int64_t y_ld = j.d_Y != nullptr ? j.ldy : j.chunk;
    if (j.n_tgt > 0) {
        if (j.op == AT_HOSTIO_SPMM)
            rc = at_spmm(csr, io->d_x, j.x_dtype, j.chunk, y, j.y_dtype, y_ld, nf, 0, sc);
        else if (j.op == AT_HOSTIO_SPMM_MISSING_ALL || j.op == AT_HOSTIO_SPMM_MISSING_HEAVIEST)
            rc = at_spmm_missing(csr, io->d_x, j.x_dtype, j.chunk, y, j.y_dtype, y_ld, nf,
                                 j.op == AT_HOSTIO_SPMM_MISSING_ALL ? AT_MISSING_ALL : AT_MISSING_HEAVIEST, sc);
        else
            rc = at_gather_rows(gather_idx, j.n_tgt, j.n_src, io->d_x, j.chunk, y, y_ld, nf, j.xe, nullptr, sc);
        if (rc != AT_OK) return rc;
    }
    if (j.fields_out != nullptr && j.n_tgt > 0) {
        PendingHostCopy next;
        rc = download_chunk(io, y, y_ld, nf, j.n_tgt, j.ye, j.out_stride, j.fields_out + c0, j.cout.all_pinned, sc, &next);
        if (rc != AT_OK) return rc;
        rc = finish_host_copy(io, *pending, j.out_fb, j.out_stride);
        if (rc != AT_OK) return rc;
        *pending = next;
    }
    return AT_OK;
}

// The engine for the next chunk: the first one, counting on from the one after `last`, whose
// next input slot is free (the pack that last read the slot has run).  While every device keeps
// up this deals the chunks round robin; a device that falls behind is skipped.
int next_engine(at_hostio* const* engines, int n, int last, int* pick) {
    for (;;) {
        for (int k = 1; k <= n; ++k) {
            const int e = (last + k) % n;
            const at_hostio* io = engines[e];
            const cudaError_t q = cudaEventQuery(io->in_free[io->in_seq % kSlots]);
            if (q == cudaSuccess) {
                *pick = e;
                return AT_OK;
            }
            if (q != cudaErrorNotReady) return set_error(AT_ERR_CUDA, "at_hostio_group_regrid: %s", cudaGetErrorString(q));
        }
        cudaGetLastError();  // "not ready" is not an error
        std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
}

// One streamed regrid over n_eng engines (one for at_hostio_regrid, all of a group's for
// at_hostio_group_regrid); engine e applies csrs[e] / gather_idx[e], staged on its device.
// lane_tickets[e] receives engine e's ticket (-1: nothing outstanding there).
int regrid_impl(at_hostio* const* engines, int n_eng, std::mutex& mu, int op, const at_csr_t* const* csrs,
                const int64_t* const* gather_idx, int64_t n_out_points, const void* const* fields_in, const at_grib_field_t* grib,
                int64_t n_fields, int64_t n_src, int x_dtype, void* d_Y, int64_t ldy, void* const* fields_out, void* consumer_stream,
                int64_t* lane_tickets) {
    AT_REQUIRE(fields_in != nullptr, "at_hostio_regrid: null argument");
    AT_REQUIRE(x_dtype == AT_F32 || x_dtype == AT_F64, "at_hostio_regrid: bad dtype code");
    AT_REQUIRE(d_Y != nullptr || fields_out != nullptr, "at_hostio_regrid: neither a resident result nor host destinations");
    AT_REQUIRE(d_Y == nullptr || n_eng == 1, "at_hostio_regrid: a resident result needs a single engine");
    AT_REQUIRE(n_fields >= 0 && n_src >= 0, "at_hostio_regrid: negative size");
    if (lane_tickets)
        for (int e = 0; e < n_eng; ++e) lane_tickets[e] = -1;
    int y_dtype = x_dtype;
    int64_t n_tgt = n_out_points;
    if (is_matrix_op(op)) {
        for (int e = 0; e < n_eng; ++e) {
            AT_REQUIRE(csrs[e] != nullptr, "at_hostio_regrid: null matrix");
            int64_t n_rows, n_cols, nnz;
            int uniform, wdtype;
            int rc = at_csr_info(csrs[e], &n_rows, &n_cols, &nnz, &uniform, &wdtype);
            if (rc != AT_OK) return rc;
            AT_REQUIRE(n_cols == n_src, "at_hostio_regrid: dimension mismatch: matrix has %lld columns, fields have %lld points",
                       (long long)n_cols, (long long)n_src);
            AT_REQUIRE(e == 0 || (n_rows == n_tgt && (wdtype == AT_F64 ? AT_F64 : x_dtype) == y_dtype),
                       "at_hostio_regrid: the engines' matrices differ in shape or dtype");
            rc = check_csr_device(csrs[e], engines[e]->device, "at_hostio_regrid");
            if (rc != AT_OK) return rc;
            n_tgt = n_rows;
            y_dtype = (wdtype == AT_F64 || x_dtype == AT_F64) ? AT_F64 : AT_F32;
        }
    } else {
        for (int e = 0; e < n_eng; ++e) AT_REQUIRE(gather_idx[e] != nullptr && n_out_points >= 0, "at_hostio_regrid: gather needs an index");
    }
    AT_REQUIRE(fields_out == nullptr || lane_tickets != nullptr, "at_hostio_regrid: ticket is null");
    AT_REQUIRE(d_Y == nullptr || (ldy % 4 == 0 && ldy >= n_fields), "at_hostio_regrid: ldy must be a multiple of 4 and >= n_fields");
    if (n_fields == 0) return AT_OK;
    for (int64_t f = 0; f < n_fields; ++f) {
        AT_REQUIRE(fields_in[f] != nullptr, "at_hostio_regrid: input field %lld is null", (long long)f);
        AT_REQUIRE(fields_out == nullptr || fields_out[f] != nullptr, "at_hostio_regrid: output field %lld is null", (long long)f);
    }
    std::lock_guard<std::mutex> lk(mu);
    DeviceGuard guard(engines[0]->device);
    RegridJob j;
    j.op = op;
    j.x_dtype = x_dtype;
    j.y_dtype = y_dtype;
    j.xe = x_dtype == AT_F32 ? 4 : 8;
    j.ye = y_dtype == AT_F32 ? 4 : 8;
    j.fields_in = fields_in;
    j.grib = grib;
    j.n_src = n_src;
    j.n_tgt = n_tgt;
    j.d_Y = d_Y;
    j.ldy = ldy;
    j.fields_out = fields_out;
    const size_t in_fb = static_cast<size_t>(n_src) * j.xe;
    j.in_stride = round_up(std::max<size_t>(in_fb, 1), kAlign);
    j.out_fb = static_cast<size_t>(n_tgt) * j.ye;
    j.out_stride = round_up(std::max<size_t>(j.out_fb, 1), kAlign);
    // largest packed field (+ its share of the parameter table)
    const size_t packed_stride = grib != nullptr ? grib_packed_stride(grib, n_fields, n_src) : 0;
    // a chunk is bounded by the slots (what crosses PCIe) and by its decoded [points x fields] batch
    const size_t bound_stride = grib != nullptr ? std::max({packed_stride, j.out_stride, j.in_stride / 4}) : std::max(j.in_stride, j.out_stride);
    j.chunk = chunk_fields(n_fields, bound_stride, 4, 4 * static_cast<int64_t>(n_eng));
    if (grib == nullptr) j.cin = classify(fields_in, n_fields);
    if (fields_out) j.cout = classify(fields_out, n_fields);
    for (int e = 0; e < n_eng; ++e) {
        at_hostio* io = engines[e];
        AT_CUDA_TRY(cudaSetDevice(io->device));
        for (int s = 0; s < kSlots; ++s) io->status_nf[s] = 0;  // nothing of an earlier call is reported
        int rc = grib != nullptr ? ensure_in_slots(io, static_cast<size_t>(j.chunk) * packed_stride + 8192, true)
                                 : ensure_in_slots(io, static_cast<size_t>(j.chunk) * j.in_stride, !j.cin.all_pinned);
        if (rc != AT_OK) return rc;
        if (fields_out) {
            rc = ensure_out_slots(io, static_cast<size_t>(j.chunk) * j.out_stride, !j.cout.all_pinned);
            if (rc != AT_OK) return rc;
        }
        rc = ensure_device_buffer(&io->d_x, &io->d_x_bytes, std::max<size_t>(static_cast<size_t>(n_src) * static_cast<size_t>(j.chunk) * j.xe, 16));
        if (rc != AT_OK) return rc;
        if (d_Y == nullptr) {
            rc = ensure_device_buffer(&io->d_y, &io->d_y_bytes, std::max<size_t>(static_cast<size_t>(n_tgt) * static_cast<size_t>(j.chunk) * j.ye, 16));
            if (rc != AT_OK) return rc;
        }
    }
    AT_CUDA_TRY(cudaSetDevice(engines[0]->device));
    cudaStream_t consumer = as_stream(consumer_stream);
    if (d_Y != nullptr) {  // the resident result was allocated on the consumer's stream
        AT_CUDA_TRY(cudaEventRecord(engines[0]->ev_sync, consumer));
        AT_CUDA_TRY(cudaStreamWaitEvent(engines[0]->s_compute, engines[0]->ev_sync, 0));
    }
    std::vector<PendingHostCopy> pending(static_cast<size_t>(n_eng));
    std::vector<uint8_t> used(static_cast<size_t>(n_eng), 0);
    int e = n_eng - 1;
    for (int64_t c0 = 0; c0 < n_fields; c0 += j.chunk) {
        const int nf = static_cast<int>(std::min<int64_t>(j.chunk, n_fields - c0));
        if (n_eng > 1) {
            int rc = next_engine(engines, n_eng, e, &e);
            if (rc != AT_OK) return rc;
            AT_CUDA_TRY(cudaSetDevice(engines[e]->device));
        } else {
            e = 0;
        }
        used[static_cast<size_t>(e)] = 1;
        const int rc = regrid_chunk(engines[e], j, is_matrix_op(op) ? csrs[e] : nullptr, op == AT_HOSTIO_GATHER ? gather_idx[e] : nullptr,
                                    c0, nf, &pending[static_cast<size_t>(e)]);
        if (rc != AT_OK) {
            if (grib != nullptr)
                for (int k = 0; k < n_eng; ++k) {
                    cudaSetDevice(engines[k]->device);
                    quiesce(engines[k]);
                }
            return rc;
        }
    }
    if (grib != nullptr) {  // a malformed field fails the call (each engine waits for its last decode)
        int rc = AT_OK;
        for (int k = 0; k < n_eng && rc == AT_OK; ++k) {
            if (!used[static_cast<size_t>(k)]) continue;
            AT_CUDA_TRY(cudaSetDevice(engines[k]->device));
            rc = status_check_all(engines[k]);
        }
        if (rc != AT_OK) {
            for (int k = 0; k < n_eng; ++k) {
                cudaSetDevice(engines[k]->device);
                quiesce(engines[k]);
            }
            return rc;
        }
    }
    for (int k = 0; k < n_eng; ++k) {
        if (!used[static_cast<size_t>(k)]) continue;
        at_hostio* io = engines[k];
        AT_CUDA_TRY(cudaSetDevice(io->device));
        int rc = finish_host_copy(io, pending[static_cast<size_t>(k)], j.out_fb, j.out_stride);
        if (rc != AT_OK) return rc;
        if (d_Y != nullptr) {  // whoever reads the resident result on `consumer` waits for the last SpMM
            AT_CUDA_TRY(cudaEventRecord(io->ev_sync, io->s_compute));
            AT_CUDA_TRY(cudaStreamWaitEvent(consumer, io->ev_sync, 0));
        }
        // page-locked inputs were read in place: they belong to the caller again only after the DMA
        if (j.cin.any_pinned) AT_CUDA_TRY(cudaStreamSynchronize(io->s_in));
        if (fields_out != nullptr && j.cout.all_pinned && n_tgt > 0) {
            rc = new_ticket(io, io->s_out, &lane_tickets[k]);
            if (rc != AT_OK) return rc;
        }
    }
    return AT_OK;
}

}  // namespace

extern "C" int at_hostio_regrid(at_hostio_t* io, int op, const at_csr_t* csr, const int64_t* gather_idx,
                                int64_t n_out_points, const void* const* fields_in, int64_t n_fields, int64_t n_src,
                                int x_dtype, void* d_Y, int64_t ldy, void* const* fields_out, void* consumer_stream,
                                int64_t* ticket) {
    const int rc = check_op(op, "at_hostio_regrid");
    if (rc != AT_OK) return rc;
    AT_REQUIRE(io != nullptr, "at_hostio_regrid: null argument");
    return regrid_impl(&io, 1, io->mu, op, &csr, &gather_idx, n_out_points, fields_in, nullptr, n_fields, n_src, x_dtype, d_Y, ldy,
                       fields_out, consumer_stream, ticket);
}

extern "C" int at_hostio_regrid_grib(at_hostio_t* io, int op, const at_csr_t* csr, const int64_t* gather_idx,
                                     int64_t n_out_points, const void* const* messages, const at_grib_field_t* fields,
                                     int64_t n_fields, int64_t n_src, int x_dtype, void* d_Y, int64_t ldy,
                                     void* const* fields_out, void* consumer_stream, int64_t* ticket) {
    const int rc = check_op(op, "at_hostio_regrid_grib");
    if (rc != AT_OK) return rc;
    AT_REQUIRE(io != nullptr, "at_hostio_regrid_grib: null argument");
    AT_REQUIRE(fields != nullptr || n_fields == 0, "at_hostio_regrid_grib: null scans");
    return regrid_impl(&io, 1, io->mu, op, &csr, &gather_idx, n_out_points, messages, fields, n_fields, n_src, x_dtype, d_Y, ldy,
                       fields_out, consumer_stream, ticket);
}

extern "C" int at_hostio_upload_grib(at_hostio_t* io, const void* const* messages, const at_grib_field_t* fields,
                                     int64_t n_fields, int64_t n_points, int x_dtype, void* d_pm, int64_t ld, void* stream) {
    AT_REQUIRE(io != nullptr && d_pm != nullptr, "at_hostio_upload_grib: null argument");
    AT_REQUIRE(x_dtype == AT_F32 || x_dtype == AT_F64, "at_hostio_upload_grib: bad dtype code");
    AT_REQUIRE(n_fields >= 0 && n_points >= 0 && ld >= n_fields, "at_hostio_upload_grib: bad sizes");
    if (n_fields == 0 || n_points == 0) return AT_OK;
    AT_REQUIRE(messages != nullptr && fields != nullptr, "at_hostio_upload_grib: null argument");
    for (int64_t f = 0; f < n_fields; ++f) AT_REQUIRE(messages[f] != nullptr, "at_hostio_upload_grib: message %lld is null", (long long)f);
    std::lock_guard<std::mutex> lk(io->mu);
    DeviceGuard guard(io->device);
    const size_t packed_stride = grib_packed_stride(fields, n_fields, n_points);
    const int64_t chunk = chunk_fields(n_fields, packed_stride, 1);
    int rc = ensure_in_slots(io, static_cast<size_t>(chunk) * packed_stride + 8192, true);
    if (rc != AT_OK) return rc;
    cudaStream_t st = as_stream(stream);
    const size_t elem = x_dtype == AT_F32 ? 4 : 8;
    for (int s = 0; s < kSlots; ++s) io->status_nf[s] = 0;  // nothing of an earlier call is reported
    for (int64_t c0 = 0; c0 < n_fields; c0 += chunk) {
        const int nf = static_cast<int>(std::min<int64_t>(chunk, n_fields - c0));
        rc = upload_chunk_grib(io, messages + c0, fields + c0, nf, n_points, x_dtype, static_cast<char*>(d_pm) + static_cast<size_t>(c0) * elem, ld, st, c0);
        if (rc != AT_OK) {
            quiesce(io);
            return rc;
        }
    }
    rc = status_check_all(io);  // a malformed field fails the call
    if (rc != AT_OK) quiesce(io);
    return rc;
}

// ------------------------------------------------------------------ group -------------
struct at_hostio_group {
    std::vector<at_hostio*> engines;
    std::mutex mu;  // one operation at a time
    std::mutex ticket_mu;
    std::vector<std::vector<int64_t>> tickets;  // group ticket -> the engines' tickets
    std::vector<int64_t> free_tickets;
};

extern "C" int at_hostio_group_destroy(at_hostio_group_t* g) {
    if (g == nullptr) return AT_OK;
    int prev = -1;
    cudaGetDevice(&prev);
    for (at_hostio* io : g->engines) at_hostio_destroy(io);
    if (prev >= 0) cudaSetDevice(prev);
    delete g;
    return AT_OK;
}

extern "C" int at_hostio_group_create(int32_t n_engines, const int32_t* devices, int32_t n_threads, at_hostio_group_t** out) {
    AT_REQUIRE(out != nullptr && devices != nullptr, "at_hostio_group_create: null argument");
    *out = nullptr;
    AT_REQUIRE(n_engines >= 1 && n_engines <= 64, "at_hostio_group_create: n_engines must be in [1, 64]");
    AT_REQUIRE(n_threads >= 0 && n_threads <= 256, "at_hostio_group_create: n_threads must be in [0, 256]");
    int n_dev = 0;
    AT_CUDA_TRY(cudaGetDeviceCount(&n_dev));
    for (int32_t e = 0; e < n_engines; ++e)
        AT_REQUIRE(devices[e] >= 0 && devices[e] < n_dev, "at_hostio_group_create: device %d out of range (%d visible)", devices[e], n_dev);
    DeviceGuard guard(devices[0]);
    // one pool for the whole group: host memory bandwidth, not the device count, bounds staging
    const int dev0 = devices[0];
    auto workers = std::make_shared<WorkerPool>(default_copy_threads(n_threads), [dev0] { cudaSetDevice(dev0); });
    at_hostio_group* g = new at_hostio_group();
    for (int32_t e = 0; e < n_engines; ++e) {
        at_hostio* io = nullptr;
        cudaError_t r = cudaSetDevice(devices[e]);
        int rc = r == cudaSuccess ? make_engine(devices[e], workers, &io) : set_error(AT_ERR_CUDA, "at_hostio_group_create: %s", cudaGetErrorString(r));
        if (rc != AT_OK) {
            at_hostio_group_destroy(g);
            return rc;
        }
        g->engines.push_back(io);
    }
    *out = g;
    return AT_OK;
}

static int group_regrid(at_hostio_group_t* g, int op, const at_csr_t* const* csrs, const int64_t* const* gather_idx,
                        int64_t n_out_points, const void* const* fields_in, const at_grib_field_t* grib, int64_t n_fields, int64_t n_src,
                        int x_dtype, void* const* fields_out, int64_t* ticket) {
    if (ticket != nullptr) *ticket = -1;
    const int op_rc = check_op(op, "at_hostio_group_regrid");
    if (op_rc != AT_OK) return op_rc;
    AT_REQUIRE(g != nullptr && fields_out != nullptr && ticket != nullptr, "at_hostio_group_regrid: null argument");
    AT_REQUIRE(!is_matrix_op(op) || csrs != nullptr, "at_hostio_group_regrid: null matrices");
    AT_REQUIRE(op != AT_HOSTIO_GATHER || gather_idx != nullptr, "at_hostio_group_regrid: null indices");
    const int n = static_cast<int>(g->engines.size());
    std::vector<const at_csr_t*> cs(static_cast<size_t>(n), nullptr);
    std::vector<const int64_t*> gi(static_cast<size_t>(n), nullptr);
    for (int e = 0; e < n; ++e) {
        if (csrs != nullptr) cs[static_cast<size_t>(e)] = csrs[e];
        if (gather_idx != nullptr) gi[static_cast<size_t>(e)] = gather_idx[e];
    }
    std::vector<int64_t> lanes(static_cast<size_t>(n), -1);
    const int rc = regrid_impl(g->engines.data(), n, g->mu, op, cs.data(), gi.data(), n_out_points, fields_in, grib, n_fields, n_src,
                               x_dtype, nullptr, 0, fields_out, nullptr, lanes.data());
    if (rc != AT_OK) {  // destinations must not be handed back while a DMA still writes them
        for (int e = 0; e < n; ++e) at_hostio_wait(g->engines[static_cast<size_t>(e)], lanes[static_cast<size_t>(e)]);
        return rc;
    }
    if (std::all_of(lanes.begin(), lanes.end(), [](int64_t t) { return t < 0; })) return AT_OK;
    std::lock_guard<std::mutex> lk(g->ticket_mu);
    if (!g->free_tickets.empty()) {
        *ticket = g->free_tickets.back();
        g->free_tickets.pop_back();
        g->tickets[static_cast<size_t>(*ticket)] = std::move(lanes);
    } else {
        *ticket = static_cast<int64_t>(g->tickets.size());
        g->tickets.push_back(std::move(lanes));
    }
    return AT_OK;
}

extern "C" int at_hostio_group_regrid(at_hostio_group_t* g, int op, const at_csr_t* const* csrs, const int64_t* const* gather_idx,
                                      int64_t n_out_points, const void* const* fields_in, int64_t n_fields, int64_t n_src, int x_dtype,
                                      void* const* fields_out, int64_t* ticket) {
    return group_regrid(g, op, csrs, gather_idx, n_out_points, fields_in, nullptr, n_fields, n_src, x_dtype, fields_out, ticket);
}

extern "C" int at_hostio_group_regrid_grib(at_hostio_group_t* g, int op, const at_csr_t* const* csrs, const int64_t* const* gather_idx,
                                           int64_t n_out_points, const void* const* messages, const at_grib_field_t* fields,
                                           int64_t n_fields, int64_t n_src, int x_dtype, void* const* fields_out, int64_t* ticket) {
    AT_REQUIRE(fields != nullptr || n_fields == 0, "at_hostio_group_regrid_grib: null scans");
    return group_regrid(g, op, csrs, gather_idx, n_out_points, messages, fields, n_fields, n_src, x_dtype, fields_out, ticket);
}

extern "C" int at_hostio_group_wait(at_hostio_group_t* g, int64_t ticket) {
    AT_REQUIRE(g != nullptr, "at_hostio_group_wait: null group");
    if (ticket < 0) return AT_OK;
    std::vector<int64_t> lanes;
    {
        std::lock_guard<std::mutex> lk(g->ticket_mu);
        AT_REQUIRE(ticket < static_cast<int64_t>(g->tickets.size()) && !g->tickets[static_cast<size_t>(ticket)].empty(),
                   "at_hostio_group_wait: ticket %lld is not outstanding", (long long)ticket);
        lanes.swap(g->tickets[static_cast<size_t>(ticket)]);
        g->free_tickets.push_back(ticket);
    }
    int rc = AT_OK;
    for (size_t e = 0; e < lanes.size(); ++e) {
        const int r = at_hostio_wait(g->engines[e], lanes[e]);
        if (rc == AT_OK) rc = r;
    }
    return rc;
}

// alac_abi.cu -- the C ABI of include/alac_b200.h over the kernels in alac_kernels.cuh and alac_planar.cuh.
//
// Host-side plumbing only: handles, device buffers, the chunked H2D -> decode kernel -> D2H pipeline over four slots (a
// CUDA stream and its buffers each), the multi-track / multi-device front end, pinned memory, error text. No decode
// arithmetic lives here and there is no CPU fallback: if CUDA is unusable every decode entry point fails.
#include "alac_kernels.cuh"
#include "alac_planar.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/alac_b200.h"

using namespace alacb200;

namespace {

thread_local std::string g_last_error;

bool cuda_ok(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return true;
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
}
#define CU(call)                                       \
    do {                                               \
        if (!cuda_ok((call), #call)) return ALACB200_E_CUDA; \
    } while (0)

#ifndef ALACB200_SLOTS
#define ALACB200_SLOTS 4
#endif
#ifndef ALACB200_CHUNK_PACKETS
#define ALACB200_CHUNK_PACKETS 4096
#endif
constexpr int kSlots = ALACB200_SLOTS;                         // pipeline depth of the host-buffer path
constexpr uint32_t kMaxChunkPackets = ALACB200_CHUNK_PACKETS;  // packets per pipeline chunk (c3 end to end: 93.7 ms at 16384, 90.2 ms at ~3500;
                                                               // round 2, one box: 4 slots x 4096 90.5 ms, 6 x 4096 91.1, 4 x 2048 90.0, 8 x 2048 91.1: the box's copy rate, not the schedule)
constexpr uint64_t kMaxChunkPcm = 512ull << 20;   // PCM bytes per pipeline chunk

// Device memory of every decoder of the process comes from one stream-ordered pool per device that KEEPS what is freed
// (up to kPoolKeepBytes) instead of handing it back to the driver at the next synchronisation, which is what the
// device's default pool does: a caller that opens one decoder per file (NewDecoder, decode.go:50-75) would otherwise pay
// the physical allocation of its staging and scratch -- tens of milliseconds -- for every file.
constexpr uint64_t kPoolKeepBytes = 8ull << 30;
cudaMemPool_t device_pool() {  // of the current device; nullptr: use the device's default pool
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {};
    static bool tried[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!tried[dev]) {
        tried[dev] = true;
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t pool = nullptr;
        if (cudaMemPoolCreate(&pool, &props) == cudaSuccess) {
            uint64_t keep = kPoolKeepBytes;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            pools[dev] = pool;  // never destroyed: lives as long as the process
        }
        cudaGetLastError();
    }
    return pools[dev];
}
cudaError_t pool_alloc(void **p, size_t bytes, cudaStream_t stream) {
    cudaMemPool_t pool = device_pool();
    return pool ? cudaMallocFromPoolAsync(p, bytes, pool, stream) : cudaMallocAsync(p, bytes, stream);
}

// Stream-ordered device buffer: growing frees and allocates on the owning stream, so nothing in flight loses its
// memory and the device is never synchronised. Contents are not preserved.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool reserve(size_t bytes, cudaStream_t stream) {
        if (bytes <= cap) return true;
        release(stream);
        const size_t want = bytes + bytes / 8 + 256;
        if (pool_alloc(&p, want, stream) != cudaSuccess) {
            g_last_error = "cudaMallocAsync failed";
            cudaGetLastError();
            p = nullptr;
            return false;
        }
        cap = want;
        return true;
    }
    void release(cudaStream_t stream) {
        if (p) cudaFreeAsync(p, stream);
        p = nullptr;
        cap = 0;
    }
};
// Page-locking host memory costs milliseconds per call, which is most of what NewDecoder / NewPacketDecoder would cost
// a caller that opens one decoder per file. Released staging buffers are therefore kept (up to a bound) and handed to the
// next decoder of the process; portable pinned memory serves every device.
struct PinPool {
    static constexpr size_t kMaxCached = 3ull << 30;
    std::mutex mu;
    std::vector<std::pair<void *, size_t>> cached;
    size_t cached_bytes = 0;
    void *take(size_t bytes, size_t &cap) {
        std::lock_guard<std::mutex> lock(mu);
        size_t best = cached.size();
        for (size_t i = 0; i < cached.size(); i++)
            if (cached[i].second >= bytes && cached[i].second <= 4 * bytes + (1u << 20) && (best == cached.size() || cached[i].second < cached[best].second))
                best = i;
        if (best == cached.size()) return nullptr;
        void *p = cached[best].first;
        cap = cached[best].second;
        cached_bytes -= cap;
        cached.erase(cached.begin() + (ptrdiff_t)best);
        return p;
    }
    void give(void *p, size_t cap) {
        {
            std::lock_guard<std::mutex> lock(mu);
            if (cached_bytes + cap <= kMaxCached && cached.size() < 256) {
                cached.emplace_back(p, cap);
                cached_bytes += cap;
                return;
            }
        }
        cudaFreeHost(p);
    }
};
PinPool &pin_pool() {
    static PinPool *pool = new PinPool();  // never destroyed: the CUDA runtime may be gone before static destructors run
    return *pool;
}

struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool reserve(size_t bytes) {
        if (bytes <= cap) return true;
        release();
        const size_t want = bytes + bytes / 8 + 256;
        if ((p = pin_pool().take(want, cap)) != nullptr) return true;
        if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess) {
            g_last_error = "cudaHostAlloc failed";
            cudaGetLastError();
            p = nullptr;
            return false;
        }
        cap = want;
        return true;
    }
    void release() {
        if (p) pin_pool().give(p, cap);
        p = nullptr;
        cap = 0;
    }
};

// What a launch needs besides its inputs and outputs: one slot of parked samples and element lists per RESIDENT CTA (the
// kernel's CTAs are persistent and pull packet groups from a counter), so its size does not depend on the batch.
struct Work {
    DevBuf scratch;                // int32 [ctas][channels][frame_length][32]
    DevBuf descs;                  // PacketDesc [ctas][32]
    uint32_t *counters = nullptr;  // {next group, CTAs done}; zero between launches (the kernel's last CTA re-zeroes them)
    bool reserve(uint32_t ctas, size_t per_cta_scratch, cudaStream_t stream) {
        if (!scratch.reserve((size_t)ctas * per_cta_scratch, stream) || !descs.reserve((size_t)ctas * 32u * sizeof(PacketDesc), stream))
            return false;
        if (!counters) {
            if (pool_alloc((void **)&counters, 2 * sizeof(uint32_t), stream) != cudaSuccess ||
                cudaMemsetAsync(counters, 0, 2 * sizeof(uint32_t), stream) != cudaSuccess) {
                g_last_error = "cudaMallocAsync failed (group counters)";
                cudaGetLastError();
                counters = nullptr;
                return false;
            }
        }
        return true;
    }
    void release(cudaStream_t stream) {
        scratch.release(stream);
        descs.release(stream);
        if (counters) cudaFreeAsync(counters, stream);
        counters = nullptr;
    }
};

// The scratch of the device entry points, which enqueue on the caller's stream. It is stream-ordered memory: moving to
// another stream first waits for the work of the previous one (the only host synchronisation of those entry points).
struct DevicePathWork {
    Work work;
    cudaStream_t stream = nullptr;  // stream `work` was last used (and is owned) on
    int32_t use(cudaStream_t st) {
        if (st != stream && work.scratch.p) {
            CU(cudaStreamSynchronize(stream));
            work.release(stream);
        }
        stream = st;
        return ALACB200_OK;
    }
};

// Pinned staging of the small tables the device entry points upload (the planar path's track table). A buffer is
// written again only once the copy that read it has completed, and a call never waits for that: it takes a buffer
// whose copy is done, or adds one.
struct TableStaging {
    struct Buf {
        PinBuf pin;
        cudaEvent_t copied = nullptr;
    };
    std::vector<std::unique_ptr<Buf>> bufs;
    int32_t upload(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
        Buf *b = nullptr;
        for (auto &x : bufs)
            if (cudaEventQuery(x->copied) == cudaSuccess) {
                b = x.get();
                break;
            }
        if (!b) {
            bufs.emplace_back(new Buf());
            b = bufs.back().get();
            CU(cudaEventCreateWithFlags(&b->copied, cudaEventDisableTiming));
        }
        if (!b->pin.reserve(bytes)) return ALACB200_E_NOMEM;
        std::memcpy(b->pin.p, src, bytes);
        CU(cudaMemcpyAsync(dst, b->pin.p, bytes, cudaMemcpyHostToDevice, stream));
        CU(cudaEventRecord(b->copied, stream));
        return ALACB200_OK;
    }
    void release() {  // call with the device current and idle
        for (auto &x : bufs) {
            x->pin.release();
            if (x->copied) cudaEventDestroy(x->copied);
        }
        bufs.clear();
    }
};

// A run of packets of one track inside a pipeline chunk.
struct Segment {
    const uint8_t *src;  // host bytes the offsets are relative to (packed packets or a whole file image)
    uint64_t src_len;    // bytes readable at src
    const uint64_t *offsets;
    const uint32_t *sizes;
    uint32_t n;
    uint8_t *pcm_out;  // host; packet i at pcm_out + i * out_stride
    uint32_t *out_bytes;
    int32_t *status;
};

// Where the per-packet results of a retired chunk go (caller arrays may be pageable: copying into them straight from
// the stream would make every chunk synchronous).
struct Scatter {
    uint32_t *out_bytes;
    int32_t *status;
    uint32_t first, n;          // rows [first, first + n) of the chunk
    std::vector<uint32_t> bad;  // rows whose packet lies outside the source bytes
};

struct Slot {
    cudaStream_t stream = nullptr;
    Work work;
    DevBuf packed, meta, pcm, results;
    PinBuf h_in;   // pinned staging of this chunk's rebased offsets (u64) + sizes (u32)
    PinBuf h_out;  // pinned staging of this chunk's out_bytes (u32) + status (i32)
    cudaEvent_t done = nullptr;
    std::vector<Scatter> scatter;
    uint32_t pending = 0;
    uint64_t pcm_stride = 0, pcm_frame_bytes = 0;  // what the gaps of `pcm` were last zeroed for
};

struct ProfEvents {
    cudaEvent_t e0, e1;
};

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cuda_ok(cudaSetDevice(dev), "cudaSetDevice");
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int32_t check_config(const alacb200_config *cfg) {
    if (alacb200_bytes_per_sample(cfg->bit_depth) == 0) return ALACB200_ST_BIT_DEPTH;  // decoder.go:91-93
    if (cfg->num_channels < 1 || cfg->num_channels > 8) return ALACB200_ST_UNSUPPORTED_CONFIG;
    if (cfg->frame_length < 1 || cfg->frame_length > 65536) return ALACB200_ST_UNSUPPORTED_CONFIG;
    return ALACB200_ST_OK;
}

// The part of a cookie the kernel needs, and the size of a decoded packet.
struct Shape {
    DevConfig dev;
    uint64_t frame_bytes;
    bool same_kernel_config(const Shape &o) const {
        return dev.frame_length == o.dev.frame_length && dev.bit_depth == o.dev.bit_depth && dev.num_channels == o.dev.num_channels &&
               dev.pb == o.dev.pb && dev.mb == o.dev.mb && dev.kb == o.dev.kb;
    }
};
Shape make_shape(const alacb200_config &cfg, uint32_t num_sms) {
    Shape s;
    s.dev.frame_length = cfg.frame_length;
    s.dev.bit_depth = cfg.bit_depth;
    s.dev.num_channels = cfg.num_channels;
    s.dev.bps = (uint32_t)alacb200_bytes_per_sample(cfg.bit_depth);
    s.dev.pb = cfg.pb;
    s.dev.mb = cfg.mb;
    s.dev.kb = cfg.kb;
    s.dev.num_sms = num_sms;
    s.frame_bytes = (uint64_t)cfg.frame_length * cfg.num_channels * s.dev.bps;
    return s;
}

// One device: streams, staging and scratch of the chunked host path, shared by whatever configs are decoded on it.
struct Pipeline {
    int device = -1;
    uint32_t num_sms = 148;
    uint32_t max_ctas = 0;  // CTAs the device keeps resident (SMs x CTAs per SM): the grid never needs more
    uint32_t max_ctas_lat = 0;  // the same for the register-rich build that small batches run
    Slot slots[kSlots];
    uint32_t next_slot = 0;
    DevicePathWork device_path;  // scratch of the device entry points
    TableStaging tables;         // pinned staging of their track tables
    bool profiling = false;
    std::vector<ProfEvents> prof_events;
    alacb200_profile prof{};

    int32_t init(int dev) {
        device = dev;
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        num_sms = (uint32_t)sms;
        CU(cudaFuncSetAttribute(alac_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecShared)));
        CU(cudaFuncSetAttribute(alac_decode_kernel_lat, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecShared)));
        int per_sm = 0, per_sm_lat = 0;  // persistent CTAs: as many as the device keeps resident
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, alac_decode_kernel, DEC_THREADS, sizeof(DecShared)));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_lat, alac_decode_kernel_lat, DEC_THREADS, sizeof(DecShared)));
        if (per_sm <= 0 || per_sm_lat <= 0) {
            g_last_error = "alac_decode_kernel does not fit on this device";
            return ALACB200_E_CUDA;
        }
        max_ctas = (uint32_t)(per_sm * sms);
        max_ctas_lat = (uint32_t)(per_sm_lat * sms);
        if (std::getenv("ALACB200_VERBOSE"))
            std::fprintf(stderr, "alacb200: device %d, %d SMs x %d resident CTAs of %d threads, %zu B shared each\n", dev, sms, per_sm,
                         DEC_THREADS, sizeof(DecShared));
        for (auto &s : slots) {
            CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        }
        return ALACB200_OK;
    }
    void destroy() {  // call with the device current
        cudaDeviceSynchronize();
        for (auto &pe : prof_events) {
            cudaEventDestroy(pe.e0);
            cudaEventDestroy(pe.e1);
        }
        prof_events.clear();
        device_path.work.release(nullptr);
        tables.release();
        for (auto &s : slots) {
            s.work.release(s.stream);
            s.packed.release(s.stream);
            s.meta.release(s.stream);
            s.pcm.release(s.stream);
            s.results.release(s.stream);
            s.h_in.release();
            s.h_out.release();
            if (s.done) cudaEventDestroy(s.done);
            if (s.stream) cudaStreamDestroy(s.stream);
            s.done = nullptr;
            s.stream = nullptr;
        }
    }

    // Enqueue the decode kernel for n device-resident packets on `stream`: ONE launch whatever n is.
    int32_t launch(Work &work, const Shape &shape, const uint8_t *d_packed, const uint64_t *d_offsets, const uint32_t *d_sizes,
                   uint32_t n, uint8_t *d_pcm, uint64_t out_stride, uint32_t *d_out_bytes, int32_t *d_status, cudaStream_t stream) {
        if (n == 0) return ALACB200_OK;
        const DevConfig &c = shape.dev;
        const uint32_t groups = (n + 31u) / 32u;
        // one scratch slot per CTA; very long frames (up to 65536 x 8 channels = 64 MB per slot) get fewer CTAs
        const uint64_t per_cta = (uint64_t)c.num_channels * c.frame_length * 32u * sizeof(int32_t);
        const uint32_t budget_ctas = (uint32_t)std::max<uint64_t>(8, (4ull << 30) / per_cta);
        // A batch that fits the register-rich build in one wave runs that build. (Giving every CTA two groups when a batch
        // is between one and two waves was measured and is slower -- a quarter of c3: 3.70 vs 3.36 ms -- because the few
        // CTAs of a sparse second round run almost twice as fast as those of a full one.)
        const uint32_t want = groups;
        const bool lat = want <= max_ctas_lat && !std::getenv("ALACB200_NO_LAT_BUILD");
        const uint32_t grid = std::min(want, std::min(lat ? max_ctas_lat : max_ctas, budget_ctas));
        if (!work.reserve(grid, (size_t)per_cta, stream)) return ALACB200_E_NOMEM;
        ProfEvents pe{};
        if (profiling) {
            CU(cudaEventCreate(&pe.e0));
            CU(cudaEventCreate(&pe.e1));
            CU(cudaEventRecord(pe.e0, stream));
        }
        auto *kernel = lat ? alac_decode_kernel_lat : alac_decode_kernel;
        kernel<<<grid, DEC_THREADS, sizeof(DecShared), stream>>>(d_packed, d_offsets, d_sizes, n, c, (int32_t *)work.scratch.p,
                                                                 (PacketDesc *)work.descs.p, d_pcm, out_stride, d_out_bytes, d_status,
                                                                 work.counters);
        CU(cudaGetLastError());
        if (profiling) {
            CU(cudaEventRecord(pe.e1, stream));
            prof_events.push_back(pe);
            prof.launches_decode++;
        }
        return ALACB200_OK;
    }

    int32_t drain_profile() {
        for (auto &pe : prof_events) {
            CU(cudaEventSynchronize(pe.e1));
            float a = 0;
            CU(cudaEventElapsedTime(&a, pe.e0, pe.e1));
            prof.ms_decode += a;
            cudaEventDestroy(pe.e0);
            cudaEventDestroy(pe.e1);
        }
        prof_events.clear();
        return ALACB200_OK;
    }

    // Wait for the slot's chunk and hand its per-packet results to the caller.
    int32_t retire(Slot &s) {
        if (!s.pending) return ALACB200_OK;
        CU(cudaEventSynchronize(s.done));
        const uint32_t *ob = (const uint32_t *)s.h_out.p;
        const int32_t *st = (const int32_t *)(ob + s.pending);
        for (auto &sc : s.scatter) {
            std::memcpy(sc.out_bytes, ob + sc.first, (size_t)sc.n * 4);
            std::memcpy(sc.status, st + sc.first, (size_t)sc.n * 4);
            for (uint32_t r : sc.bad) {  // the packet lies outside the source bytes: the reference's reader fails before decoding
                sc.out_bytes[r] = 0;
                sc.status[r] = ALACB200_ST_IO_TRUNCATED;
            }
        }
        s.scatter.clear();
        s.pending = 0;
        return ALACB200_OK;
    }
    int32_t drain() {
        for (auto &s : slots) {
            const int32_t rc = retire(s);
            if (rc != ALACB200_OK) return rc;
        }
        return ALACB200_OK;
    }
    // After a failed call: nothing may still be copying into the caller's buffers, no slot may keep pointers into them.
    void abort_all() {
        for (auto &s : slots) {
            if (s.stream) cudaStreamSynchronize(s.stream);
            s.pending = 0;
            s.scatter.clear();
        }
    }

    // One pipeline chunk: H2D of every segment's byte span, the kernel, D2H of PCM and per-packet results. All segments
    // share the kernel config and out_stride. Returns as soon as the work is enqueued.
    int32_t submit_chunk(const Shape &shape, uint64_t out_stride, const Segment *segs, size_t nsegs) {
        Slot &s = slots[next_slot];
        next_slot = (next_slot + 1) % kSlots;
        int32_t rc = retire(s);  // the slot's previous chunk (and its staging) is finished
        if (rc != ALACB200_OK) return rc;
        uint32_t m = 0;
        for (size_t k = 0; k < nsegs; k++) m += segs[k].n;
        if (m == 0) return ALACB200_OK;
        // byte span of every segment inside its source, and where it lands in the device staging (alignment mod 16 kept)
        struct Span {
            uint64_t lo, hi, dev_pos;
        };
        std::vector<Span> spans(nsegs);
        uint64_t pos = 0;
        for (size_t k = 0; k < nsegs; k++) {
            const Segment &g = segs[k];
            uint64_t lo = UINT64_MAX, hi = 0;
            for (uint32_t i = 0; i < g.n; i++) {
                const uint64_t off = g.offsets[i], sz = g.sizes[i];
                if (off > g.src_len || sz > g.src_len - off) continue;  // outside the source: not copied, not decoded
                lo = std::min(lo, off);
                hi = std::max(hi, off + sz);
            }
            if (hi < lo) lo = hi = 0;
            pos = (pos + 15u) / 16u * 16u + (lo & 15u);
            spans[k] = Span{lo, hi, pos};
            pos += hi - lo;
        }
        if (!s.packed.reserve(pos + 64, s.stream) || !s.meta.reserve((size_t)m * 12, s.stream) || !s.results.reserve((size_t)m * 8, s.stream) ||
            !s.h_in.reserve((size_t)m * 12) || !s.h_out.reserve((size_t)m * 8))
            return ALACB200_E_NOMEM;
        const bool has_gap = out_stride > shape.frame_bytes;
        if ((size_t)m * out_stride > s.pcm.cap || (has_gap && (s.pcm_stride != out_stride || s.pcm_frame_bytes != shape.frame_bytes))) {
            if (!s.pcm.reserve((size_t)m * out_stride, s.stream)) return ALACB200_E_NOMEM;
            // the kernel never touches the gap between frame_bytes and out_stride, and the gap travels back with the
            // slot: define it once per buffer and per shape (PCM of an earlier call must not show up in it)
            if (has_gap) CU(cudaMemsetAsync(s.pcm.p, 0, s.pcm.cap, s.stream));
            s.pcm_stride = out_stride;
            s.pcm_frame_bytes = shape.frame_bytes;
        }
        uint64_t *ho = (uint64_t *)s.h_in.p;
        uint32_t *hs = (uint32_t *)(ho + m);
        uint32_t row = 0;
        for (size_t k = 0; k < nsegs; k++) {
            const Segment &g = segs[k];
            Scatter sc{g.out_bytes, g.status, row, g.n, {}};
            for (uint32_t i = 0; i < g.n; i++, row++) {
                const uint64_t off = g.offsets[i], sz = g.sizes[i];
                if (off > g.src_len || sz > g.src_len - off) {
                    ho[row] = 0;
                    hs[row] = 0;
                    sc.bad.push_back(i);
                } else {
                    ho[row] = off - spans[k].lo + spans[k].dev_pos;
                    hs[row] = g.sizes[i];
                }
            }
            s.scatter.push_back(std::move(sc));
            if (spans[k].hi > spans[k].lo)
                CU(cudaMemcpyAsync((uint8_t *)s.packed.p + spans[k].dev_pos, g.src + spans[k].lo, spans[k].hi - spans[k].lo,
                                   cudaMemcpyHostToDevice, s.stream));
        }
        CU(cudaMemcpyAsync(s.meta.p, ho, (size_t)m * 12, cudaMemcpyHostToDevice, s.stream));  // offsets[m] then sizes[m]
        const uint64_t *d_off = (const uint64_t *)s.meta.p;
        const uint32_t *d_sz = (const uint32_t *)(d_off + m);
        uint32_t *d_ob = (uint32_t *)s.results.p;  // out_bytes[m] then status[m], one D2H copy
        int32_t *d_st = (int32_t *)(d_ob + m);
        rc = launch(s.work, shape, (const uint8_t *)s.packed.p, d_off, d_sz, m, (uint8_t *)s.pcm.p, out_stride, d_ob, d_st, s.stream);
        if (rc != ALACB200_OK) return rc;
        row = 0;
        for (size_t k = 0; k < nsegs; k++) {
            const Segment &g = segs[k];
            if (g.n)
                CU(cudaMemcpyAsync(g.pcm_out, (const uint8_t *)s.pcm.p + (size_t)row * out_stride,
                                   (size_t)(g.n - 1) * out_stride + shape.frame_bytes, cudaMemcpyDeviceToHost, s.stream));
            row += g.n;
        }
        CU(cudaMemcpyAsync(s.h_out.p, d_ob, (size_t)m * 8, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaEventRecord(s.done, s.stream));
        s.pending = m;
        return ALACB200_OK;
    }
};

uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

bool stride_ok(uint64_t out_stride, uint64_t frame_bytes) { return out_stride >= frame_bytes && (out_stride & 3u) == 0; }

// Packets per chunk so that copies of chunk k+1 / k-1 overlap the kernel of chunk k.
uint32_t chunk_packets(uint64_t n, uint64_t out_stride) {
    uint32_t nchunks_target = 6;
    if (const char *env = std::getenv("ALACB200_CHUNKS")) nchunks_target = (uint32_t)std::max(1, std::atoi(env));  // tuning knob
    uint64_t chunk = (n + nchunks_target - 1u) / nchunks_target;
    chunk = std::min<uint64_t>(std::max<uint64_t>(chunk, 512u), kMaxChunkPackets);
    while (chunk > 32u && chunk * out_stride > kMaxChunkPcm) chunk /= 2u;
    return (uint32_t)((chunk + 31u) & ~31ull);
}

}  // namespace

struct alacb200_decoder {
    alacb200_config cfg;
    Shape shape;
    Pipeline pipe;
    PinBuf arena_in, arena_out;  // alacb200_arena: decoder-owned pinned staging for the host wrappers
};

// Decoders of several tracks (any mix of cookies) on one or more devices of this process.
struct alacb200_library {
    std::vector<std::unique_ptr<Pipeline>> devs;
};

namespace {

size_t sample_type_bytes(int32_t sample_type) {
    return sample_type == ALACB200_SAMPLES_S16 ? 2 : (sample_type == ALACB200_SAMPLES_S32 || sample_type == ALACB200_SAMPLES_F32) ? 4 : 0;
}

// One planar launch set on `st` for rows [row0, row0 + rows) of the packet table, all of kernel config `shape`: the decode
// kernel into a stream-ordered intermediate (freed on the stream at the end), the frame scan of the ntracks tracks at
// d_tracks (device), the planar pass.
int32_t enqueue_planar(Pipeline &pipe, const Shape &shape, int32_t sample_type, const uint8_t *d_packed, const uint64_t *d_offsets,
                       const uint32_t *d_sizes, int32_t *d_status, uint64_t *d_frame_start, const PlanarTrack *d_tracks,
                       uint32_t ntracks, uint64_t row0, uint32_t rows, cudaStream_t st) {
    const uint32_t ch = shape.dev.num_channels, bps = shape.dev.bps, bpf = ch * bps, fl = shape.dev.frame_length;
    // the interleaved intermediate: packet slots of frame_bytes rounded up to 16, then out_bytes[rows]
    const uint64_t slot = (shape.frame_bytes + 15u) / 16u * 16u;
    uint8_t *inter = nullptr;
    if (rows && pool_alloc((void **)&inter, (size_t)(rows * slot + (uint64_t)rows * 4u), st) != cudaSuccess) {
        g_last_error = "cudaMallocAsync failed (planar intermediate)";
        cudaGetLastError();
        return ALACB200_E_NOMEM;
    }
    uint32_t *d_out_bytes = rows ? (uint32_t *)(inter + rows * slot) : nullptr;
    int32_t rc = pipe.launch(pipe.device_path.work, shape, d_packed, d_offsets + row0, d_sizes + row0, rows, inter, slot, d_out_bytes,
                             d_status + row0, st);
    if (rc == ALACB200_OK) {
        alac_frame_scan_kernel<<<ntracks, SCAN_THREADS, 0, st>>>(d_out_bytes, d_status, d_tracks, row0, bpf, d_frame_start);
        if (rows) {
            const uint32_t tile = planar_tile_frames(bpf, fl);
            const dim3 grid(rows, (fl + tile - 1) / tile);
            if (sample_type == ALACB200_SAMPLES_S16)
                alac_planar_kernel<int16_t><<<grid, PLANAR_THREADS, 0, st>>>(inter, slot, d_frame_start, d_tracks, ntracks, row0, ch, bps, tile);
            else if (sample_type == ALACB200_SAMPLES_S32)
                alac_planar_kernel<int32_t><<<grid, PLANAR_THREADS, 0, st>>>(inter, slot, d_frame_start, d_tracks, ntracks, row0, ch, bps, tile);
            else
                alac_planar_kernel<float><<<grid, PLANAR_THREADS, 0, st>>>(inter, slot, d_frame_start, d_tracks, ntracks, row0, ch, bps, tile);
        }
        if (!cuda_ok(cudaGetLastError(), "alac_planar_kernel")) rc = ALACB200_E_CUDA;
    }
    if (inter) cudaFreeAsync(inter, st);
    return rc;
}

// The track table of a planar call, uploaded through the pipeline's pinned staging into stream-ordered memory that is
// freed on the stream after the call's launches.
struct DeviceTracks {
    PlanarTrack *p = nullptr;
    int32_t upload(Pipeline &pipe, const std::vector<PlanarTrack> &host, cudaStream_t st) {
        const size_t bytes = host.size() * sizeof(PlanarTrack);
        if (pool_alloc((void **)&p, bytes, st) != cudaSuccess) {
            g_last_error = "cudaMallocAsync failed (planar track table)";
            cudaGetLastError();
            p = nullptr;
            return ALACB200_E_NOMEM;
        }
        return pipe.tables.upload(p, host.data(), bytes, st);
    }
    void release(cudaStream_t st) {
        if (p) cudaFreeAsync(p, st);
        p = nullptr;
    }
};

// The tracks `order` on one device: already grouped by kernel config (so every launch is depth-homogeneous, SURVEY.md
// 8e), cut into pipeline chunks that may span several tracks.
int32_t decode_tracks_on(Pipeline &pipe, alacb200_track_desc *tracks, const std::vector<Shape> &shapes, const std::vector<uint32_t> &order) {
    DeviceGuard guard(pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    int32_t rc = ALACB200_OK;
    std::vector<Segment> segs;
    uint32_t in_chunk = 0;
    const Shape *cur = nullptr;
    uint64_t cur_stride = 0;
    auto flush = [&]() -> int32_t {
        int32_t r = ALACB200_OK;
        if (in_chunk) r = pipe.submit_chunk(*cur, cur_stride, segs.data(), segs.size());
        segs.clear();
        in_chunk = 0;
        return r;
    };
    for (uint32_t t : order) {
        alacb200_track_desc &tr = tracks[t];
        const Shape &sh = shapes[t];
        if (cur && (!cur->same_kernel_config(sh) || cur_stride != tr.out_stride)) {
            if ((rc = flush()) != ALACB200_OK) break;
        }
        cur = &sh;
        cur_stride = tr.out_stride;
        uint32_t limit = kMaxChunkPackets;
        while (limit > 32u && (uint64_t)limit * tr.out_stride > kMaxChunkPcm) limit /= 2u;
        for (uint32_t a = 0; a < tr.n && rc == ALACB200_OK;) {
            const uint32_t take = std::min(tr.n - a, limit - std::min(limit, in_chunk));
            if (take == 0) {
                rc = flush();
                continue;
            }
            segs.push_back(Segment{tr.data, tr.data_len, tr.offsets + a, tr.sizes + a, take, tr.pcm_out + (size_t)a * tr.out_stride,
                                   tr.out_bytes + a, tr.status + a});
            in_chunk += take;
            a += take;
        }
        if (rc != ALACB200_OK) break;
    }
    if (rc == ALACB200_OK) rc = flush();
    if (rc == ALACB200_OK) rc = pipe.drain();
    if (rc != ALACB200_OK) pipe.abort_all();
    return rc;
}

}  // namespace

extern "C" {

int32_t alacb200_parse_cookie(const uint8_t *cookie, size_t len, alacb200_config *out) {
    if (!out) return ALACB200_ST_INVALID_COOKIE;
    std::memset(out, 0, sizeof(*out));
    const uint8_t *d = cookie;
    if (!d) len = 0;
    // optional 'frma' and 'alac' atom wrappers, config.go:50-58
    if (len >= 12 && std::memcmp(d + 4, "frma", 4) == 0) { d += 12; len -= 12; }
    if (len >= 12 && std::memcmp(d + 4, "alac", 4) == 0) { d += 12; len -= 12; }
    if (len < 24) return ALACB200_ST_INVALID_COOKIE;       // config.go:60-62
    if (d[4] > 0) return ALACB200_ST_UNSUPPORTED_VERSION;  // config.go:64-67
    out->frame_length = be32(d);
    out->bit_depth = d[5];
    out->pb = d[6];
    out->mb = d[7];
    out->kb = d[8];
    out->num_channels = d[9];
    out->max_run = (uint16_t)((d[10] << 8) | d[11]);
    out->max_frame_bytes = be32(d + 12);
    out->avg_bit_rate = be32(d + 16);
    out->sample_rate = be32(d + 20);
    return ALACB200_ST_OK;
}

int32_t alacb200_bytes_per_sample(uint8_t bit_depth) {
    switch (bit_depth) {
    case 16: return 2;
    case 20:
    case 24: return 3;
    case 32: return 4;
    default: return 0;
    }
}

int32_t alacb200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t alacb200_create(const alacb200_config *cfg, int device, alacb200_decoder **out, int32_t *status_out) {
    if (status_out) *status_out = ALACB200_ST_OK;
    if (!cfg || !out) return ALACB200_E_ARG;
    *out = nullptr;
    int32_t st = check_config(cfg);
    if (st != ALACB200_ST_OK) {
        if (status_out) *status_out = st;
        return ALACB200_E_CONFIG;
    }
    int ndev = alacb200_device_count();
    if (ndev <= 0 || device < 0 || device >= ndev) {
        g_last_error = "no usable CUDA device (this library has no CPU fallback)";
        return ALACB200_E_NO_DEVICE;
    }
    DeviceGuard guard(device);
    if (!guard.ok) return ALACB200_E_CUDA;
    auto *dec = new alacb200_decoder();
    dec->cfg = *cfg;
    const int32_t rc = dec->pipe.init(device);
    if (rc != ALACB200_OK) {
        dec->pipe.destroy();
        delete dec;
        return rc;
    }
    dec->shape = make_shape(*cfg, dec->pipe.num_sms);
    *out = dec;
    return ALACB200_OK;
}

void alacb200_destroy(alacb200_decoder *dec) {
    if (!dec) return;
    DeviceGuard guard(dec->pipe.device);
    dec->pipe.destroy();  // synchronises the device first
    dec->arena_in.release();
    dec->arena_out.release();
    delete dec;
}

int32_t alacb200_format(const alacb200_decoder *dec, alacb200_pcm_format *out) {
    if (!dec || !out) return ALACB200_E_ARG;
    out->sample_rate = (int32_t)dec->cfg.sample_rate;  // decoder.go:99-103
    out->bit_depth = dec->cfg.bit_depth;
    out->channels = dec->cfg.num_channels;
    return ALACB200_OK;
}

int32_t alacb200_get_config(const alacb200_decoder *dec, alacb200_config *out) {
    if (!dec || !out) return ALACB200_E_ARG;
    *out = dec->cfg;
    return ALACB200_OK;
}

uint64_t alacb200_max_packet_pcm_bytes(const alacb200_decoder *dec) { return dec ? dec->shape.frame_bytes : 0; }

int32_t alacb200_decode_packets_device(alacb200_decoder *dec, const uint8_t *d_packed, uint64_t packed_bytes,
                                       const uint64_t *d_offsets, const uint32_t *d_sizes, uint32_t n,
                                       uint8_t *d_pcm_out, uint64_t out_stride, uint32_t *d_out_bytes,
                                       int32_t *d_status, void *stream) {
    (void)packed_bytes;
    if (!dec) return ALACB200_E_ARG;
    if (n == 0) return ALACB200_OK;
    if (!d_packed || !d_offsets || !d_sizes || !d_pcm_out || !d_out_bytes || !d_status) return ALACB200_E_ARG;
    if (!stride_ok(out_stride, dec->shape.frame_bytes) || (((uintptr_t)d_pcm_out) & 3u) || (((uintptr_t)d_packed) & 15u)) {
        g_last_error = "out_stride must be >= max_packet_pcm_bytes and a multiple of 4; d_packed 16-byte aligned";
        return ALACB200_E_ARG;
    }
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t rc = dec->pipe.device_path.use(st);
    if (rc != ALACB200_OK) return rc;
    return dec->pipe.launch(dec->pipe.device_path.work, dec->shape, d_packed, d_offsets, d_sizes, n, d_pcm_out, out_stride, d_out_bytes,
                            d_status, st);
}

int32_t alacb200_decode_planar_device(alacb200_decoder *dec, const uint8_t *d_packed, uint64_t packed_bytes,
                                      const uint64_t *d_offsets, const uint32_t *d_sizes, uint32_t n, int32_t sample_type,
                                      void *d_out, uint64_t channel_stride, uint64_t *d_frame_start, int32_t *d_status,
                                      void *stream) {
    (void)packed_bytes;
    if (!dec) return ALACB200_E_ARG;
    const size_t esz = sample_type_bytes(sample_type);
    if (esz == 0 || (sample_type == ALACB200_SAMPLES_S16 && dec->cfg.bit_depth != 16)) {
        g_last_error = "sample_type must be S16 (16-bit streams only), S32 or F32";
        return ALACB200_E_ARG;
    }
    if (!d_frame_start) return ALACB200_E_ARG;
    const uint32_t fl = dec->cfg.frame_length;
    if (n && (!d_packed || !d_offsets || !d_sizes || !d_out || !d_status)) return ALACB200_E_ARG;
    if (channel_stride < (uint64_t)n * fl || (((uintptr_t)d_out) % esz) || (((uintptr_t)d_packed) & 15u)) {
        g_last_error = "channel_stride must be >= n * frame_length; d_out aligned to its element size; d_packed 16-byte aligned";
        return ALACB200_E_ARG;
    }
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        CU(cudaMemsetAsync(d_frame_start, 0, sizeof(uint64_t), st));
        return ALACB200_OK;
    }
    int32_t rc = dec->pipe.device_path.use(st);
    if (rc != ALACB200_OK) return rc;
    DeviceTracks tracks;  // the one-track case of the library's planar path
    rc = tracks.upload(dec->pipe, {PlanarTrack{0, 0, d_out, channel_stride, n, 0}}, st);
    if (rc == ALACB200_OK)
        rc = enqueue_planar(dec->pipe, dec->shape, sample_type, d_packed, d_offsets, d_sizes, d_status, d_frame_start, tracks.p, 1, 0, n, st);
    tracks.release(st);
    return rc;
}

int32_t alacb200_decode_packets(alacb200_decoder *dec, const uint8_t *packed, uint64_t packed_bytes, const uint64_t *offsets,
                                const uint32_t *sizes, uint32_t n, uint8_t *pcm_out, uint64_t out_stride,
                                uint32_t *out_bytes, int32_t *status) {
    if (!dec) return ALACB200_E_ARG;
    if (n == 0) return ALACB200_OK;
    if (!packed || !offsets || !sizes || !pcm_out || !out_bytes || !status) return ALACB200_E_ARG;
    if (!stride_ok(out_stride, dec->shape.frame_bytes)) {
        g_last_error = "out_stride must be >= max_packet_pcm_bytes and a multiple of 4";
        return ALACB200_E_ARG;
    }
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    // Chunk schedule: small chunks first and last. Nothing can overlap the upload + decode of the first chunk or the
    // download of the last one, so those are kept short; the chunks in between are as large as the slots allow.
    const uint32_t chunk = chunk_packets(n, out_stride);
    std::vector<uint32_t> plan;
    {
        uint32_t left = n, cur = std::max(512u, (chunk / 8u + 31u) & ~31u);
        while (left) {
            const uint32_t m = std::min(left, cur);
            plan.push_back(m);
            left -= m;
            cur = std::min(chunk, cur * 2u);
        }
        if (plan.size() > 3 && plan.back() >= 4096u) {  // ramp down: ... X/2, X/4, X/8, X/8
            uint32_t x = plan.back();
            plan.pop_back();
            for (int k = 0; k < 3; k++) {
                const uint32_t h = ((x / 2u) + 31u) & ~31u;
                plan.push_back(h);
                x -= h;
            }
            plan.push_back(x);
        }
    }
    int32_t rc = ALACB200_OK;
    uint32_t a = 0;
    for (size_t k = 0; k < plan.size() && rc == ALACB200_OK; a += plan[k], k++) {
        const uint32_t m = plan[k];
        const Segment seg{packed, packed_bytes, offsets + a, sizes + a, m, pcm_out + (size_t)a * out_stride, out_bytes + a, status + a};
        rc = dec->pipe.submit_chunk(dec->shape, out_stride, &seg, 1);
    }
    if (rc == ALACB200_OK) rc = dec->pipe.drain();
    if (rc != ALACB200_OK) dec->pipe.abort_all();
    return rc;
}

int32_t alacb200_arena(alacb200_decoder *dec, uint64_t in_bytes, uint64_t out_bytes, uint8_t **in, uint8_t **out) {
    if (!dec || !in || !out) return ALACB200_E_ARG;
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    if (!dec->arena_in.reserve((size_t)in_bytes + 64) || !dec->arena_out.reserve((size_t)out_bytes + 64)) return ALACB200_E_NOMEM;
    *in = (uint8_t *)dec->arena_in.p;
    *out = (uint8_t *)dec->arena_out.p;
    return ALACB200_OK;
}

// ---- several tracks, several devices ----------------------------------------------------------------------------
int32_t alacb200_library_create(const int *devices, int ndevices, alacb200_library **out) {
    if (!out || ndevices < 1 || !devices) return ALACB200_E_ARG;
    *out = nullptr;
    const int ndev = alacb200_device_count();
    auto lib = std::unique_ptr<alacb200_library>(new alacb200_library());
    int32_t rc = ALACB200_OK;
    for (int k = 0; k < ndevices && rc == ALACB200_OK; k++) {
        if (ndev <= 0 || devices[k] < 0 || devices[k] >= ndev) {
            g_last_error = "no usable CUDA device (this library has no CPU fallback)";
            rc = ALACB200_E_NO_DEVICE;
            break;
        }
        DeviceGuard guard(devices[k]);
        if (!guard.ok) {
            rc = ALACB200_E_CUDA;
            break;
        }
        lib->devs.emplace_back(new Pipeline());
        rc = lib->devs.back()->init(devices[k]);
    }
    if (rc != ALACB200_OK) {
        alacb200_library_destroy(lib.release());
        return rc;
    }
    *out = lib.release();
    return ALACB200_OK;
}

void alacb200_library_destroy(alacb200_library *lib) {
    if (!lib) return;
    for (auto &p : lib->devs) {
        DeviceGuard guard(p->device);
        p->destroy();
    }
    delete lib;
}

int32_t alacb200_library_devices(const alacb200_library *lib) { return lib ? (int32_t)lib->devs.size() : 0; }

int32_t alacb200_library_decode_tracks(alacb200_library *lib, alacb200_track_desc *tracks, uint32_t ntracks) {
    if (!lib || (!tracks && ntracks)) return ALACB200_E_ARG;
    // per track: ParseMagicCookie + NewPacketDecoder's checks (config.go:47-81, decoder.go:90-110)
    std::vector<Shape> shapes(ntracks);
    std::vector<uint64_t> weight(ntracks, 0);
    std::vector<uint32_t> good;
    for (uint32_t t = 0; t < ntracks; t++) {
        alacb200_track_desc &tr = tracks[t];
        tr.result = ALACB200_OK;
        tr.device = -1;
        tr.track_status = alacb200_parse_cookie(tr.cookie, tr.cookie_len, &tr.config);
        if (tr.track_status == ALACB200_ST_OK) tr.track_status = check_config(&tr.config);
        if (tr.track_status != ALACB200_ST_OK) {
            tr.result = ALACB200_E_CONFIG;
            continue;
        }
        shapes[t] = make_shape(tr.config, 0);
        if (tr.n == 0) continue;
        if (!tr.data || !tr.offsets || !tr.sizes || !tr.pcm_out || !tr.out_bytes || !tr.status || !stride_ok(tr.out_stride, shapes[t].frame_bytes)) {
            tr.result = ALACB200_E_ARG;
            continue;
        }
        for (uint32_t i = 0; i < tr.n; i++) weight[t] += tr.sizes[i];
        good.push_back(t);
    }
    // contiguous track ranges per device, balanced by compressed bytes; inside a device, tracks grouped by config
    const size_t nd = lib->devs.size();
    uint64_t total = 0;
    for (uint32_t t : good) total += weight[t];
    std::vector<std::vector<uint32_t>> per_dev(nd);
    uint64_t acc = 0;
    for (uint32_t t : good) {
        size_t d = total ? (size_t)(((long double)acc + weight[t] / 2.0L) * nd / (long double)total) : 0;
        d = std::min(d, nd - 1);
        per_dev[d].push_back(t);
        tracks[t].device = lib->devs[d]->device;
        acc += weight[t];
    }
    for (size_t d = 0; d < nd; d++) {
        for (uint32_t t : per_dev[d]) shapes[t].dev.num_sms = lib->devs[d]->num_sms;
        std::stable_sort(per_dev[d].begin(), per_dev[d].end(), [&](uint32_t a, uint32_t b) {
            const DevConfig &x = shapes[a].dev, &y = shapes[b].dev;
            if (x.bit_depth != y.bit_depth) return x.bit_depth < y.bit_depth;
            if (x.num_channels != y.num_channels) return x.num_channels < y.num_channels;
            if (x.frame_length != y.frame_length) return x.frame_length < y.frame_length;
            if (x.pb != y.pb) return x.pb < y.pb;
            if (x.mb != y.mb) return x.mb < y.mb;
            return x.kb < y.kb;
        });
    }
    std::vector<int32_t> rcs(nd, ALACB200_OK);
    std::vector<std::string> errs(nd);
    auto run = [&](size_t d) {
        rcs[d] = decode_tracks_on(*lib->devs[d], tracks, shapes, per_dev[d]);
        if (rcs[d] != ALACB200_OK) errs[d] = g_last_error;
    };
    if (nd == 1) {
        run(0);
    } else {  // one submitting host thread per device
        std::vector<std::thread> th;
        for (size_t d = 0; d < nd; d++) th.emplace_back(run, d);
        for (auto &x : th) x.join();
    }
    int32_t rc = ALACB200_OK;
    for (size_t d = 0; d < nd; d++)
        if (rcs[d] != ALACB200_OK) {
            if (rc == ALACB200_OK) {
                g_last_error = errs[d];
                rc = rcs[d];
            }
            for (uint32_t t : per_dev[d]) tracks[t].result = rcs[d];
        }
    return rc;
}

int32_t alacb200_library_decode_planar_device(alacb200_library *lib, int device, const uint8_t *d_packed, uint64_t packed_bytes,
                                              const uint64_t *d_offsets, const uint32_t *d_sizes, alacb200_planar_track *tracks,
                                              uint32_t ntracks, int32_t sample_type, uint64_t *d_frame_start, int32_t *d_status,
                                              void *stream) {
    (void)packed_bytes;
    if (!lib || (!tracks && ntracks) || (!d_frame_start && ntracks)) return ALACB200_E_ARG;
    Pipeline *pipe = nullptr;
    for (auto &p : lib->devs)
        if (p->device == device) pipe = p.get();
    const size_t esz = sample_type_bytes(sample_type);
    if (!pipe || esz == 0) {
        g_last_error = "device must be one of the library's devices; sample_type S16, S32 or F32";
        return ALACB200_E_ARG;
    }
    // per track: ParseMagicCookie + NewPacketDecoder's checks (config.go:47-81, decoder.go:90-110), then the arguments
    std::vector<Shape> shapes(ntracks);
    uint64_t rows = 0;
    for (uint32_t t = 0; t < ntracks; t++) {
        alacb200_planar_track &tr = tracks[t];
        tr.result = ALACB200_OK;
        tr.track_status = alacb200_parse_cookie(tr.cookie, tr.cookie_len, &tr.config);
        if (tr.track_status == ALACB200_ST_OK) tr.track_status = check_config(&tr.config);
        rows += tr.n;
        if (tr.track_status != ALACB200_ST_OK) {
            tr.result = ALACB200_E_CONFIG;
            continue;
        }
        shapes[t] = make_shape(tr.config, pipe->num_sms);
        if (sample_type == ALACB200_SAMPLES_S16 && tr.config.bit_depth != 16) {
            g_last_error = "sample_type S16 holds 16-bit streams only";
            return ALACB200_E_ARG;
        }
        if (tr.n && (!tr.d_out || ((uintptr_t)tr.d_out) % esz || tr.channel_stride < (uint64_t)tr.n * tr.config.frame_length)) {
            g_last_error = "every track's d_out must be aligned to its element size and channel_stride >= n * frame_length";
            return ALACB200_E_ARG;
        }
    }
    if (rows > UINT32_MAX) {
        g_last_error = "more than 2^32 - 1 packets in one call";
        return ALACB200_E_ARG;
    }
    if (rows && (!d_packed || !d_offsets || !d_sizes || !d_status || (((uintptr_t)d_packed) & 15u))) {
        g_last_error = "d_packed (16-byte aligned), d_offsets, d_sizes and d_status must be set";
        return ALACB200_E_ARG;
    }
    DeviceGuard guard(pipe->device);
    if (!guard.ok) return ALACB200_E_CUDA;
    cudaStream_t st = (cudaStream_t)stream;
    if (rows == 0) {
        if (ntracks) CU(cudaMemsetAsync(d_frame_start, 0, (size_t)ntracks * sizeof(uint64_t), st));
        return ALACB200_OK;
    }
    int32_t rc = pipe->device_path.use(st);
    if (rc != ALACB200_OK) return rc;
    // the device table: the runs' tracks in order (a run: adjacent decodable tracks of one kernel config), then the tracks
    // without a decoder
    struct Run {
        uint32_t first, count;  // entries of the table
        uint32_t track;         // its first track (for the shape)
        uint64_t row0, rows;
    };
    std::vector<PlanarTrack> table;
    std::vector<Run> runs;
    std::vector<PlanarTrack> failed;
    uint64_t row = 0;
    bool open = false;
    for (uint32_t t = 0; t < ntracks; t++) {
        const alacb200_planar_track &tr = tracks[t];
        const PlanarTrack e{row, row + t, tr.d_out, tr.channel_stride, tr.n, tr.result == ALACB200_OK ? 0 : tr.track_status};
        row += tr.n;
        if (e.fail) {
            failed.push_back(e);
            open = false;
            continue;
        }
        if (!open || !shapes[runs.back().track].same_kernel_config(shapes[t])) runs.push_back(Run{(uint32_t)table.size(), 0, t, e.row, 0});
        open = true;
        runs.back().count++;
        runs.back().rows += e.n;
        table.push_back(e);
    }
    const uint32_t first_failed = (uint32_t)table.size();
    table.insert(table.end(), failed.begin(), failed.end());
    DeviceTracks dt;
    rc = dt.upload(*pipe, table, st);
    for (size_t k = 0; k < runs.size() && rc == ALACB200_OK; k++) {
        const Run &r = runs[k];
        rc = enqueue_planar(*pipe, shapes[r.track], sample_type, d_packed, d_offsets, d_sizes, d_status, d_frame_start, dt.p + r.first,
                            r.count, r.row0, (uint32_t)r.rows, st);
    }
    if (rc == ALACB200_OK && !failed.empty()) {
        alac_frame_scan_kernel<<<(uint32_t)failed.size(), SCAN_THREADS, 0, st>>>(nullptr, d_status, dt.p + first_failed, 0, 1, d_frame_start);
        if (!cuda_ok(cudaGetLastError(), "alac_frame_scan_kernel")) rc = ALACB200_E_CUDA;
    }
    dt.release(st);
    return rc;
}

// The public pinned allocator goes through the same pool; the capacity of a block is kept in a small table.
namespace {
std::mutex g_pin_mu;
std::vector<std::pair<void *, size_t>> g_pin_caps;
}  // namespace
void *alacb200_pinned_alloc(size_t bytes) {
    PinBuf b;
    if (!b.reserve(bytes ? bytes : 1)) return nullptr;
    std::lock_guard<std::mutex> lock(g_pin_mu);
    g_pin_caps.emplace_back(b.p, b.cap);
    return b.p;
}
void alacb200_pinned_free(void *p) {
    if (!p) return;
    size_t cap = 0;
    {
        std::lock_guard<std::mutex> lock(g_pin_mu);
        for (size_t i = 0; i < g_pin_caps.size(); i++)
            if (g_pin_caps[i].first == p) {
                cap = g_pin_caps[i].second;
                g_pin_caps.erase(g_pin_caps.begin() + (ptrdiff_t)i);
                break;
            }
    }
    if (cap) pin_pool().give(p, cap);
    else cudaFreeHost(p);
}

const char *alacb200_strerror(int32_t status) {
    switch (ALACB200_ST_CODE(status)) {  // strings of internal/alac/errors.go:24-33
    case ALACB200_ST_OK: return "ok";
    case ALACB200_ST_INVALID_COOKIE: return "alac: invalid magic cookie";
    case ALACB200_ST_UNSUPPORTED_VERSION: return "alac: unsupported compatible version";
    case ALACB200_ST_UNSUPPORTED_ELEMENT: return "alac: unsupported element type (CCE/PCE)";
    case ALACB200_ST_INVALID_HEADER: return "alac: invalid frame header";
    case ALACB200_ST_INVALID_SHIFT: return "alac: invalid bytesShifted value";
    case ALACB200_ST_BITSTREAM_OVERRUN: return "alac: bitstream overrun";
    case ALACB200_ST_SAMPLE_OVERRUN: return "alac: sample count exceeds buffer";
    case ALACB200_ST_BIT_DEPTH: return "alac: unsupported bit depth";
    case ALACB200_ST_REF_PANIC: return "alac: malformed packet (the reference decoder would panic)";
    case ALACB200_ST_UNSUPPORTED_CONFIG: return "alac: unsupported channel count or frame length";
    case ALACB200_ST_IO_TRUNCATED: return "unexpected EOF";
    default: return "alac: unknown status";
    }
}

size_t alacb200_format_error(int32_t status, char *buf, size_t cap) {
    if (!buf || cap == 0) return 0;
    const int code = ALACB200_ST_CODE(status);
    if (code == ALACB200_ST_OK) return (size_t)std::snprintf(buf, cap, "ok");
    if (code == ALACB200_ST_IO_TRUNCATED) return (size_t)std::snprintf(buf, cap, "unexpected EOF");  // io.ReadFull, decode.go:172-174
    const bool is_config = code == ALACB200_ST_INVALID_COOKIE || code == ALACB200_ST_UNSUPPORTED_VERSION ||
                           code == ALACB200_ST_BIT_DEPTH || code == ALACB200_ST_UNSUPPORTED_CONFIG;
    static const char *ctx[] = {"", "SCE/LFE: ", "CPE: ", "DSE: ", "FIL: "};
    static const char *ent[] = {"", "entropy decode: ", "entropy decode U: ", "entropy decode V: "};
    const int c = ALACB200_ST_CTX(status), e = ALACB200_ST_ENT(status);
    int w = std::snprintf(buf, cap, "%s: %s%s%s", is_config ? "invalid configuration" : "decode failed",
                          c <= 4 ? ctx[c] : "", ent[e], alacb200_strerror(status));
    return w < 0 ? 0 : (size_t)w;
}

const char *alacb200_last_error(void) { return g_last_error.c_str(); }

#ifdef ALACB200_DEV
// Developer hooks (only in the `make dev` build, not part of include/alac_b200.h): point the decode kernel's per-role
// clock64 counters at a device buffer of n_ctas*16 u64 (or NULL to switch them off). Used by tools/role_cycles.py.
int32_t alacb200_debug_flags(unsigned int flags) {
    CU(cudaMemcpyToSymbol(g_debug_flags, &flags, sizeof(flags)));
    return ALACB200_OK;
}

int32_t alacb200_debug_role_cycles(unsigned long long *d_buf) {
    CU(cudaMemcpyToSymbol(g_role_cycles, &d_buf, sizeof(d_buf)));
    return ALACB200_OK;
}
#endif

int32_t alacb200_set_profiling(alacb200_decoder *dec, int enable) {
    if (!dec) return ALACB200_E_ARG;
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    int32_t rc = dec->pipe.drain_profile();
    if (rc != ALACB200_OK) return rc;
    dec->pipe.profiling = enable != 0;
    if (enable) dec->pipe.prof = alacb200_profile{};
    return ALACB200_OK;
}

int32_t alacb200_get_profile(alacb200_decoder *dec, alacb200_profile *out) {
    if (!dec || !out) return ALACB200_E_ARG;
    DeviceGuard guard(dec->pipe.device);
    if (!guard.ok) return ALACB200_E_CUDA;
    int32_t rc = dec->pipe.drain_profile();
    if (rc != ALACB200_OK) return rc;
    *out = dec->pipe.prof;
    return ALACB200_OK;
}

}  // extern "C"

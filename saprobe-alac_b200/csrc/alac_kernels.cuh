// alac_kernels.cuh -- the hand-written sm_100a kernel of the ALAC packet-decode hot path.
//
// One kernel body, decode_cta (built twice: alac_decode_kernel for big batches, alac_decode_kernel_lat with a larger
// register budget for batches of at most one wave), parallel ACROSS packets (packets are independent, decoder.go:79-87)
// and across STAGES. A CTA is persistent, pulls groups of 32 packets from a counter and works on a group with two role
// warps, lane = packet:
//
//   ENTROPY     walks the element grammar of decodePacketInto (decoder.go:133-207) and the adaptive Golomb-Rice
//               stream (DynDecomp, golomb.go:148-253) in branch-free batches of 16 samples (decode_batch) and hands
//               the codes through a shared-memory ring (mbarrier full/empty pairs) to the predictor warp. Compressed
//               bytes are staged into shared memory with 128-bit cp.async (zero-fill past the packet end) one
//               period ahead of their use.
//   PREDICTOR   sign-LMS filter (UnpcBlock, predictor.go:45-684) of every stream of the group in bitstream order. Mono /
//               U streams are parked as int32 in a lane-interleaved scratch of the CTA ([slot][sample][32 lanes]: every
//               warp store is one 128-byte line). For the V stream of a 2-channel pair it emits PCM itself, ring slot
//               by ring slot: un-mix + shift-merge + interleaved little-endian bytes (WriteStereo*, matrix.go:30-215),
//               128-bit stores to the packet's own output slot.
//
// Whatever is not emitted live (mono, multi-channel, escape pairs, short or failed packets) is written by both warps
// after the group's barrier, from the parked samples (emit_group: WriteStereo*/WriteMono*, matrix.go:30-301).
//
// Integer semantics are the Go reference's: wrap-around int32/uint32, shifts >= 32 give 0 / sign
// fill (PTX shl/shr clamp exactly like that), int32 coefficients for orders 4/5/6/8 and int16-wrapping
// coefficients otherwise (predictor.go:107-110 vs :664). Where the reference would panic the packet
// gets ST_REF_PANIC.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace alacb200 {

enum : int32_t {
    ST_OK = 0,
    ST_UNSUPPORTED_ELEMENT = 3,
    ST_INVALID_HEADER = 4,
    ST_INVALID_SHIFT = 5,
    ST_BITSTREAM_OVERRUN = 6,
    ST_SAMPLE_OVERRUN = 7,
    ST_REF_PANIC = 9,
};
enum : int32_t { CTX_SCE = 1, CTX_CPE = 2, CTX_DSE = 3, CTX_FIL = 4 };
enum : int32_t { ENT_MONO = 1, ENT_U = 2, ENT_V = 3 };

struct DevConfig {
    uint32_t frame_length;
    uint32_t bit_depth;
    uint32_t num_channels;
    uint32_t bps;
    uint32_t pb, mb, kb;
    uint32_t num_sms;  // for spreading the role warps of co-resident CTAs over the SM sub-partitions
};

// What stage 1+2 hands to stage 3 for one decoded element (one "write op" of matrix.go).
struct OpDesc {
    uint32_t n;             // samples this element wrote
    uint32_t shift_bitpos;  // absolute bit position of the shift data inside the packet
    uint8_t kind;           // 1 = WriteMono*, 2 = WriteStereo*
    uint8_t out_chan;       // output channel index (channelLayoutOffsets, decoder.go:55-64)
    uint8_t slot;           // scratch slot of U (V = slot+1)
    uint8_t shift;          // bytesShifted seen by the writer (0 for escape elements)
    uint8_t mix_bits;
    int8_t mix_res;
    uint16_t pad_;          // 1: the element was emitted live by the predictor warp
};
struct PacketDesc {
    int32_t status;
    uint32_t n_final;
    uint32_t nops;
    uint32_t pad_;          // frames already covered by live emission (multiple of 32)
    OpDesc ops[8];
};

// ---- Go shift semantics: PTX shl/shr clamp the shift amount to 32 ------------------------------
__device__ __forceinline__ uint32_t shl_go(uint32_t x, uint32_t s) {
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(s));
    return r;
}
__device__ __forceinline__ uint32_t shr_go(uint32_t x, uint32_t s) {
    uint32_t r;
    asm("shr.u32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(s));
    return r;
}
__device__ __forceinline__ int32_t sar_go(int32_t x, uint32_t s) {
    int32_t r;
    asm("shr.s32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(s));
    return r;
}
// (del << chanShift) >> chanShift, predictor.go:69
__device__ __forceinline__ int32_t sext_go(int32_t x, uint32_t cs) { return sar_go((int32_t)shl_go((uint32_t)x, cs), cs); }
// signOfInt, predictor.go:35-39
__device__ __forceinline__ int32_t sign_of(int32_t v) { return (int32_t)((uint32_t)(-v) >> 31) | (v >> 31); }

// ---- slow bit reads straight from global memory (element headers; BitBuffer.Read*, bitbuffer.go:55-96)
struct Packet {
    const uint8_t *p;  // first byte of the packet
    uint32_t size;     // unpadded size; bytes [size, size+4) read as zero (bitbuffer.go:36-51)
};
__device__ __forceinline__ uint32_t pk_byte(const Packet &pk, uint32_t idx) { return idx < pk.size ? (uint32_t)__ldg(pk.p + idx) : 0u; }
// nb <= 16 bits at absolute bit position bp (the 24-bit window of Read)
__device__ __forceinline__ uint32_t pk_bits(const Packet &pk, uint32_t bp, uint32_t nb) {
    uint32_t b = bp >> 3;
    uint32_t w = (pk_byte(pk, b) << 16) | (pk_byte(pk, b + 1) << 8) | pk_byte(pk, b + 2);
    w = (w << (bp & 7)) & 0x00FFFFFFu;
    return shr_go(w, 24u - nb);
}
// read32bit, golomb.go:80 (big endian), zero pad semantics
__device__ __forceinline__ uint32_t pk_be32(const Packet &pk, uint32_t b) {
    return (pk_byte(pk, b) << 24) | (pk_byte(pk, b + 1) << 16) | (pk_byte(pk, b + 2) << 8) | pk_byte(pk, b + 3);
}

// Header cursor: absolute bit position + sticky "the reference would have panicked" flag.
struct Cursor {
    uint32_t bp;
    bool panic;
};
__device__ __forceinline__ uint32_t cur_read(const Packet &pk, Cursor &c, uint32_t nb) {  // Read, needs Pos+3 <= cap
    if ((c.bp >> 3) + 3u > pk.size + 4u) c.panic = true;
    uint32_t v = pk_bits(pk, c.bp, nb);
    c.bp += nb;
    return v;
}
__device__ __forceinline__ uint32_t cur_read_small(const Packet &pk, Cursor &c, uint32_t nb) {  // ReadSmall, Pos+2 <= cap
    if ((c.bp >> 3) + 2u > pk.size + 4u) c.panic = true;
    uint32_t v = pk_bits(pk, c.bp, nb);
    c.bp += nb;
    return v;
}
__device__ __forceinline__ uint32_t cur_read_one(const Packet &pk, Cursor &c) {  // ReadOne, Pos < cap
    if ((c.bp >> 3) >= pk.size + 4u) c.panic = true;
    uint32_t v = pk_bits(pk, c.bp, 1);
    c.bp += 1;
    return v;
}

// ---- mbarrier (shared-memory producer/consumer barriers between the role warps) -----------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sts32(uint32_t addr, int32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v)); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
// A waiting role warp must not eat the issue slots of the entropy warps that share its SM sub-partition (a ring chunk
// takes ~8000 cycles to produce, a whole stream ~1 M): mbarrier.try_wait with a suspend-time hint parks the warp in
// hardware until the phase completes or the hint expires, so the poll loop issues a handful of instructions per wait
// instead of one poll every ~20 cycles (__nanosleep returned almost at once in the round-1 captures: 90 M polls on c2).
// `long_wait`: a warp that waits for a whole ring slot to be produced may stay suspended longer per try.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity, bool long_wait = false) {
    const uint32_t addr = smem_u32(bar);
    const uint32_t hint = long_wait ? 100000u : 2000u;  // ns the hardware may keep the warp suspended per try
    uint32_t done;
    for (;;) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(hint)
            : "memory");
        if (done) break;
    }
}

__device__ unsigned int g_sm_ticket[256];        // per-SM CTA counter (monotonic; only its value mod 4 is used)
__device__ unsigned int g_sm_entropy_load[256];  // per SM: four 8-bit counts of resident entropy warps, by sub-partition
// Developer build only (-DALACB200_DEV, `make dev`): per-role clock64 counters, [cta][16] (0..2 E total / wait-empty /
// top-up, 3..4 predictor total / wait-full, 8..9 emit tail per warp), enabled by pointing g_role_cycles at a buffer
// (alacb200_debug_role_cycles), and g_debug_flags (bit 0: no live emission). The product library carries none of it.
#ifdef ALACB200_DEV
__device__ unsigned long long *g_role_cycles = nullptr;
__device__ unsigned int g_debug_flags = 0;
struct RoleTimer {
    unsigned long long *slot;
    unsigned long long acc[3] = {0, 0, 0};
    __device__ __forceinline__ RoleTimer(uint32_t lane, int base) {
        unsigned long long *b = g_role_cycles;
        slot = (b != nullptr && lane == 0) ? b + (size_t)blockIdx.x * 16 + base : nullptr;
    }
    __device__ __forceinline__ unsigned long long now() const { return slot ? clock64() : 0ull; }
    __device__ __forceinline__ void add(int k, unsigned long long t0) { if (slot) acc[k] += clock64() - t0; }
    __device__ __forceinline__ void flush(int n) { if (slot) for (int k = 0; k < n; k++) slot[k] = acc[k]; }
};
#else
struct RoleTimer {
    static constexpr unsigned long long *slot = nullptr;
    __device__ __forceinline__ RoleTimer(uint32_t, int) {}
    __device__ __forceinline__ unsigned long long now() const { return 0ull; }
    __device__ __forceinline__ void add(int, unsigned long long) {}
    __device__ __forceinline__ void flush(int) {}
};
#endif

// ---- geometry of one decode CTA ---------------------------------------------------------------------
// A CTA is TWO warps working on one group of 32 packets at a time (lane = packet); it is persistent and pulls group after
// group from a counter. The ENTROPY warp hands residual codes, 32 samples at a time, through a two-slot shared-memory
// ring to the PREDICTOR warp. The streams of a packet follow each other in the bitstream (V starts where U's last code
// ends), so one ring and one predictor warp serve them all in turn; for a 2-channel pair the predictor warp also turns
// every finished V slot (plus the parked U samples and the shift bytes) into PCM right away.
// Why two warps: every role warp is one dependent chain per lane and issues about once every 4.5 cycles, so a scheduler
// wants ~4.5 BUSY warps. The four-warp form of this kernel (entropy, predictor, emit, spare: profiles/r02a) kept only
// ~2.4 of its 4 warps per scheduler busy (issue slots 55 %); with two always-busy warps per group, 64 threads x 128
// registers and ~27 KB of shared memory, EIGHT groups are resident per SM instead of four.
constexpr int DEC_THREADS = 64;
constexpr int CTAS_PER_SM = 8;        // throughput build of the kernel: 128 registers per thread
// Batches that cannot fill eight CTAs per SM anyway run a second build of the same kernel with the register budget of
// six (168 registers: the spills of the 128-register build are gone, and with 222 KB of the SM's 228 KB carved out as
// shared memory a spill reload is an L1 miss): c2 1.72 -> 1.58 ms, c4 10.7 -> 9.8 ms; c3 is the same at either budget,
// the 93 k-packet batch 5 % slower at six.
#ifndef ALACB200_CTAS_PER_SM_LAT
#define ALACB200_CTAS_PER_SM_LAT 6
#endif
constexpr int CTAS_PER_SM_LAT = ALACB200_CTAS_PER_SM_LAT;
constexpr int DEC_WARPS = DEC_THREADS / 32;
constexpr int RING_SLOTS = 2;    // ring depth
constexpr int CHUNK = 32;        // samples per ring slot
constexpr int FIFO_CHUNKS = 16;  // 16-byte chunks of compressed bytes staged per lane (256 B window)
constexpr int LIVE_SHIFT_CHUNKS = 10;  // 16-byte chunks covering 32 frames x 2 channels x 2 shift bytes at any alignment
constexpr int JOB_WORDS = 6;     // per lane and stream: n, meta, coefficient bit position, nmax, live-emit word, shift bit position

struct DecShared {
    // Compressed bytes staged by cp.async: a 256-byte window per lane, [lane][chunk ^ (lane & 7)]. The window of a lane
    // starts on a 256-byte boundary of the shared address space (the struct sits at a 1024-byte aligned base), so the
    // address of a word is one LOP3: (byte offset & 0xfc) ^ window base; the XOR spreads the lanes over the banks.
    uint4 fifo[32][FIFO_CHUNKS];
    int32_t ring[RING_SLOTS][CHUNK][32];     // residual codes (then, for a live pair, decoded V samples), [slot][sample][lane]
    uint32_t job[RING_SLOTS][JOB_WORDS][32];  // what the stream is, with its first slot
    // live emission (2-channel streams): the parked U samples and the shift bytes of the current 32-frame chunk
    int32_t live_u[CHUNK][32];
    uint4 live_shift[32][LIVE_SHIFT_CHUNKS + 1];
    // per lane, of the live pair being emitted: sample count / live word (bit 31: lane is live) | (packet address & 15) << 18 /
    // bit position of the shift bytes. In shared memory because the predictor loop has no registers to spare for them and
    // local memory does not stay in L1 behind the streaming stores (profiles/r02g_c2: 17 % of the predictor warp's time)
    uint32_t live_ctx[3][32];
    // barriers last: stage 3 reuses everything in front of them as its transpose tiles
    uint64_t full_bar[RING_SLOTS];
    uint64_t empty_bar[RING_SLOTS];
    uint32_t group;                     // packet group this CTA works on
    uint32_t next_group;                // the one after it, fetched by the entropy warp while the group is decoded
    uint32_t entropy_smsp;              // sub-partition of this CTA's entropy warp
    uint32_t warp_smsp[DEC_WARPS];      // sub-partition every warp reports
    uint32_t role_of_warp[DEC_WARPS];
};
static_assert(offsetof(DecShared, fifo) == 0 && (FIFO_CHUNKS & (FIFO_CHUNKS - 1)) == 0 && FIFO_CHUNKS >= 16, "lane windows must be aligned to their size");
static_assert(offsetof(DecShared, ring) % 16 == 0 && offsetof(DecShared, live_shift) % 16 == 0 && offsetof(DecShared, full_bar) % 8 == 0, "alignment");
static_assert(sizeof(DecShared) + 1024 <= (228 * 1024) / CTAS_PER_SM, "eight CTAs per SM");

// ---- hand-over between the two role warps ------------------------------------------------------------------------
//   full[slot]   entropy -> predictor: the ring slot holds 32 codes per lane
//   empty[slot]  predictor -> entropy: the slot may be refilled
// mbarriers in shared memory. A waiting warp polls -- try_wait comes back within ~10 cycles whatever suspend hint or
// nanosleep it is given -- but the polls are free: the same protocol on hardware named barriers (bar.arrive / bar.sync),
// where a waiting warp issues nothing at all, was bit-identical and 0.5-1.5 % SLOWER when measured on the four-warp form
// of this kernel (profiles/r02a). The issue slots were never the limit; the dependent chains of the role warps are.
// Every lane arrives (32 arrivals per hand-over). One arrival by one lane after a __syncwarp() was bit-identical and
// measured at +-0.4 % on every workload: the waiter's polls (a tenth of the instructions the kernel issues) are not caused
// by the per-lane arrivals and cost nothing anybody else wanted.
// `seq` is the ring sequence number of the slot (slot = seq % RING_SLOTS, phase = seq / RING_SLOTS)
constexpr uint32_t BAR_ARRIVALS = 32u;
__device__ __forceinline__ void wait_full(DecShared &sm, uint32_t seq) { mbar_wait(&sm.full_bar[seq % RING_SLOTS], (seq / RING_SLOTS) & 1u, true); }
__device__ __forceinline__ void arrive_full(DecShared &sm, uint32_t seq) { mbar_arrive(&sm.full_bar[seq % RING_SLOTS]); }
__device__ __forceinline__ void wait_empty(DecShared &sm, uint32_t seq) { mbar_wait(&sm.empty_bar[seq % RING_SLOTS], ((seq / RING_SLOTS) & 1u) ^ 1u); }
__device__ __forceinline__ void arrive_empty(DecShared &sm, uint32_t seq) { mbar_arrive(&sm.empty_bar[seq % RING_SLOTS]); }

// job meta word
enum : uint32_t { JOB_INACTIVE = 0, JOB_REG = 1, JOB_GENERIC = 2, JOB_EXIT = 3 };  // JOB_EXIT: the group is finished
// warp-uniform flag in the meta word of a job: the two halves of an interleaved escape pair arrive in alternating slots
// (this job is the first half's, the next slot carries the second half's)
enum : uint32_t { JOBF_PAIR = 1u << 25 };
__device__ __forceinline__ uint32_t job_meta(uint32_t kind, uint32_t order, uint32_t den, uint32_t mode, uint32_t chan_bits,
                                             uint32_t slot) {
    return kind | (order << 2) | (den << 7) | ((mode != 0 ? 1u : 0u) << 11) | (chan_bits << 12) | (slot << 18);
}

// ---- bit reader of the entropy warp -----------------------------------------------------------------
// The compressed packet is staged into shared memory with 128-bit cp.async (zero-filled past the packet
// end = the reference's zero padding, bitbuffer.go:36-51) at least one half-chunk period ahead of its use;
// the hot loop then needs one LDS per sample, issued at the top of the iteration, and a branch-free refill.

// clz(x) for x != 0 in ONE instruction (FLO.U32.SH); 0xffffffff for x == 0
__device__ __forceinline__ uint32_t clz_nz(uint32_t x) {
    uint32_t r;
    asm("bfind.shiftamt.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}

// index of the highest set bit (31 - clz) in one instruction (FLO.U32); x != 0
__device__ __forceinline__ uint32_t bit_index(uint32_t x) {
    uint32_t r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}

struct BitReader {
    const uint8_t *gbase;  // 16-byte aligned global address at or below the packet start
    uint32_t end_rel;      // packet end, bytes from gbase
    uint32_t fifo;         // shared address of this lane's window, XORed with the lane's bank swizzle
    uint32_t req;          // next 16-byte chunk to request
    uint32_t landed;       // chunks below this one have landed (requested before the last wait)
    uint32_t qo;           // byte offset from gbase (multiple of 4) of the next word to load; hi, lo are the two before it
    uint32_t hi, lo;       // big-endian-converted words
    uint32_t sh;           // bits of hi already consumed (0..31)

    __device__ __forceinline__ void request(uint32_t c) {
        const uint32_t b0 = c << 4;
        const uint32_t nbytes = b0 >= end_rel ? 0u : min(16u, end_rel - b0);
        const uint8_t *src = gbase + (nbytes ? b0 : 0u);
        const uint32_t dst = fifo ^ (b0 & (FIFO_CHUNKS * 16 - 16));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
    }
    __device__ __forceinline__ static void wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
    // the word at byte offset `off` (multiple of 4) from gbase
    __device__ __forceinline__ uint32_t load(uint32_t off) const {
        const uint32_t a = (off & (FIFO_CHUNKS * 16 - 4)) ^ fifo;
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
        return __byte_perm(v, 0, 0x0123);
    }
    // land what was requested a period ago, request up to a full window ahead of the reader. 16 samples eat at most
    // 16 x 67 bits = 134 bytes (+ the two words in hand): if a run of maximal codes has brought the reader that close to
    // what had landed, wait for the new requests as well (never the case on real streams).
    __device__ __forceinline__ void top_up() {
        wait_all();
        landed = req;
        const uint32_t lim = (qo >> 4) + FIFO_CHUNKS;
        while (req < lim) request(req++);
        if (qo + 160u > (landed << 4)) {
            wait_all();
            landed = req;
        }
    }
    __device__ __forceinline__ void init(const Packet &pk, uint32_t bp, uint32_t fifo_addr) {
        const uintptr_t a = (uintptr_t)pk.p;
        const uint32_t mis = (uint32_t)(a & 15u);
        gbase = pk.p - mis;
        end_rel = mis + pk.size;
        fifo = fifo_addr;
        const uint32_t abp = bp + mis * 8u;
        const uint32_t q = (abp >> 5) << 2;
        sh = abp & 31u;
        wait_all();  // nothing of a previous element may still be landing in the window
        req = q >> 4;
        const uint32_t lim = req + FIFO_CHUNKS;
        while (req < lim) request(req++);
        wait_all();
        landed = req;
        hi = load(q);
        lo = load(q + 4u);
        qo = q + 8u;
    }
    __device__ __forceinline__ uint32_t window() const { return __funnelshift_l(lo, hi, sh); }
    // branch-free consume of nb <= 32 bits; `next` is the word after lo. Returns whether a word was taken.
    __device__ __forceinline__ bool advance(uint32_t nb, uint32_t next) {
        const uint32_t sh2 = sh + nb;
        const bool need = sh2 >= 32u;
        hi = need ? lo : hi;
        lo = need ? next : lo;
        if (need) qo += 4u;
        sh = sh2 & 31u;
        return need;
    }
    // any other consume: reloads as it goes
    __device__ __forceinline__ void consume_slow(uint32_t nb) {
        sh += nb;
        while (sh >= 32u) {
            hi = lo;
            lo = load(qo);
            qo += 4u;
            sh -= 32u;
        }
    }
};

// Special registers re-read at the point of use (volatile: never hoisted, so nothing derived from them is carried across
// the hot loops -- or spilled: with 222 of the SM's 228 KB carved out as shared memory a spill reload is an L1 miss).
__device__ __forceinline__ uint32_t lane_now() {
    uint32_t v;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(v));
    return v;
}
__device__ __forceinline__ uint32_t cta_now() {
    uint32_t v;
    asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(v));
    return v;
}

// The ring carries residuals as the sign-folded codes the entropy stage decodes (golomb.go:207-214: odd -> negative),
// so the fold is undone by the predictor warp (the result doubles as the sign mask of the LMS ladder there).
__device__ __forceinline__ int32_t code_to_residual(uint32_t nd) { return (int32_t)((nd >> 1) ^ (0u - (nd & 1u))); }
__device__ __forceinline__ int32_t residual_to_code(int32_t r) { return (int32_t)(((uint32_t)r << 1) ^ (uint32_t)(r >> 31)); }

// ---- adaptive Golomb-Rice state (DynDecomp, golomb.go:148-253) --------------------------------------
struct Entropy {
    uint32_t mean, zmode, zrun;
    uint32_t pb, kb, wb;
    uint32_t max_size;  // escape width = chanBits
    uint32_t size8;     // packet size in bits
};

// After a decoded code: does the decoder enter zero-run mode (golomb.go:220)?
__device__ __forceinline__ bool zero_run_due(uint32_t mean, uint32_t i, uint32_t n) { return (mean << 2) < 512u && i + 1u < n; }

// Zero run: dynGet, golomb.go:112-144 and :221-245. Returns false and sets st on error.
__device__ __forceinline__ bool zero_run_start(const Packet &pk, BitReader &br, uint32_t &bp, Entropy &e, uint32_t i,
                                               uint32_t n, int32_t &st) {
    e.zmode = 1;
    int32_t k32 = __clz((int32_t)e.mean) - 24 + (int32_t)((e.mean + 16u) >> 6);
    if (k32 < 0) k32 = 0;
    const uint32_t mz = (shl_go(1u, (uint32_t)k32) - 1u) & e.wb;
    if ((bp >> 3) > pk.size) { st = ST_REF_PANIC; return false; }
    const uint32_t w2 = br.window();
    const uint32_t pre = (uint32_t)__clz((int32_t)~w2);
    uint32_t run, nb;
    if (pre >= 9u) {
        run = (w2 << 9) >> 16;
        nb = 25u;
    } else {
        nb = pre + 1u;
        const uint32_t s = shl_go(w2, nb);
        const uint32_t val = shr_go(s, 32u - (uint32_t)k32);
        nb += (uint32_t)k32;
        if (val < 2u) {
            run = pre * mz;
            nb -= 1u;
        } else {
            run = pre * mz + val - 1u;
        }
    }
    bp += nb;
    br.consume_slow(nb);
    if (i + 1u + run > n) {  // golomb.go:232-234
        st = ST_SAMPLE_OVERRUN;
        return false;
    }
    e.zrun = run;
    if (run >= 65535u) e.zmode = 0;
    e.mean = 0;
    return true;
}

// The general (cold) step of DynDecomp for sample index i of n: zero-run continuation, overrun, escape
// codes, oversized codes. Returns false and sets st on error.
__device__ __forceinline__ bool entropy_next(const Packet &pk, BitReader &br, uint32_t &bp, Entropy &e, uint32_t i,
                                             uint32_t n, int32_t &res, int32_t &st) {
    if (e.zrun > 0) {  // inside a zero run (clear(predCoefs[count:end]), golomb.go:237)
        e.zrun--;
        res = 0;
        return true;
    }
    if (bp >= e.size8) {  // golomb.go:168-170
        st = ST_BITSTREAM_OVERRUN;
        return false;
    }
    uint32_t m = e.mean >> 9;
    uint32_t k = 31u - (uint32_t)__clz((int32_t)(m + 3u));
    k = min(k, e.kb);
    m = shl_go(1u, k) - 1u;
    const uint32_t w = br.window();
    uint32_t r = (uint32_t)__clz((int32_t)~w);
    if (r >= 9u) {
        // getStreamBits(input, bitPos+9, maxSize), golomb.go:86-108
        const uint32_t bo = bp + 9u;
        const uint32_t byte_off = bo >> 3;
        if (byte_off > pk.size) { st = ST_REF_PANIC; return false; }
        const uint32_t load1 = pk_be32(pk, byte_off);
        const uint32_t nb = e.max_size;
        if (nb + (bo & 7u) > 32u) {
            if (byte_off >= pk.size) { st = ST_REF_PANIC; return false; }
            uint32_t v = load1 << (bo & 7u);
            uint32_t load2 = pk_byte(pk, byte_off + 4u);
            load2 = shr_go(load2, 8u - (nb + (bo & 7u) - 32u));
            v = shr_go(v, 32u - nb);
            r = v | load2;
        } else {
            uint32_t v = shr_go(load1, 32u - nb - (bo & 7u));
            if (nb < 32u) v &= shl_go(1u, nb) - 1u;
            r = v;
        }
        bp += 9u + nb;
        br.consume_slow(9u + nb);
    } else {
        // prefix r, then a k-bit suffix v; v < 2 means "no suffix value" and gives one bit back. k == 1 and
        // k == 0 fall out of the same formula (golomb.go:188-201): m = 1 / 0 and v < 2 always.
        const uint32_t s = w << (r + 1u);
        const uint32_t v = shr_go(s, 32u - k);
        const bool big = v >= 2u;
        const uint32_t nb = r + k + (big ? 1u : 0u);
        r = r * m + (big ? v - 1u : 0u);
        bp += nb;
        br.consume_slow(nb);
    }
    const uint32_t nd = r + e.zmode;
    const int32_t mag = (int32_t)((nd + 1u) >> 1);
    res = (nd & 1u) ? -mag : mag;
    e.mean = e.pb * nd + e.mean - ((e.pb * e.mean) >> 9);
    if (r > 0xffffu) e.mean = 0xffffu;
    e.zmode = 0;
    if (zero_run_due(e.mean, i, n)) return zero_run_start(pk, br, bp, e, i, n, st);
    return true;
}

// decodeSCEEscape / decodeCPEEscape, decoder.go:326-345, :504-535
__device__ __forceinline__ int32_t escape_sample(BitReader &br, uint32_t chan_bits) {
    const uint32_t shift = 32u - chan_bits;
    if (chan_bits <= 16u) {
        const int32_t val = (int32_t)shr_go(br.window(), 32u - chan_bits);
        br.consume_slow(chan_bits);
        return sext_go(val, shift);
    }
    const uint32_t extra = chan_bits - 16u;
    int32_t val = (int32_t)(br.window() >> 16);
    br.consume_slow(16u);
    val = sar_go((int32_t)((uint32_t)val << 16), shift);
    const int32_t lo = (int32_t)shr_go(br.window(), 32u - extra);
    br.consume_slow(extra);
    return val | lo;
}

__constant__ int8_t k_layout[8][8] = {{0, 0, 0, 0, 0, 0, 0, 0}, {0, 1, 0, 0, 0, 0, 0, 0}, {2, 0, 1, 0, 0, 0, 0, 0},
                                      {2, 0, 1, 3, 0, 0, 0, 0}, {2, 0, 1, 3, 4, 0, 0, 0}, {2, 0, 1, 4, 5, 3, 0, 0},
                                      {2, 0, 1, 4, 5, 6, 3, 0}, {2, 6, 7, 0, 1, 4, 5, 3}};

// ====================================================================================================
// ENTROPY warp
// ====================================================================================================
constexpr uint32_t FULL_MASK = 0xffffffffu;

enum : uint32_t { BUSY_ESCAPE = 2, BUSY_LONG_CODES = 4, BUSY_DEAD = 8, BUSY_PARTIAL = 16 };
// pseudo zero runs: a lane in one consumes nothing, like a lane inside a real run (those are < 2^20 long)
constexpr uint32_t ZRUN_PARKED = 0x40000000u;      // nothing (left) to decode
constexpr uint32_t ZRUN_REDO = 0x20000000u;        // frozen at a sample that is not decoded yet
constexpr uint32_t ZRUN_OWES_RUN = 0x10000000u;    // frozen after a decoded sample whose run-length code is not
constexpr uint32_t ZRUN_FROZEN_MIN = 0x0fff0000u;

// What one lane needs to produce one stream (a channel of a compressed element, or the raw samples of an
// escape element).
struct StreamSpec {
    bool active;      // this lane takes part
    bool escape;      // raw samples instead of Golomb codes
    uint32_t n;
    uint32_t chan_bits;
    uint32_t pb_factor;
    uint32_t meta;         // job meta word for the consumer
    uint32_t coef_bitpos;  // where the consumer finds the 16-bit coefficients
    uint32_t live;         // V of a pair in a 2-channel stream: bit 31 set, mixBits | mixRes<<8 | bytesShifted<<16
    uint32_t shift_bitpos;
};

// ---- 16 samples without a branch ------------------------------------------------------------------------------
// Every lane runs the same instructions: one ordinary code (golomb.go:172-201) and -- in the QUIET flavour -- the
// run-length code that may follow it (dynGet, golomb.go:112-144, :220-245), each committed or not by selects. A lane
// inside a zero run (clear(predCoefs[count:end]), golomb.go:237) consumes nothing and produces 0. A lane that meets
// anything else (escape code, packet overrun, a saturating mean, a run that does not fit, a run-length code in the
// other flavour, ...) FREEZES: it is put into a pseudo zero run whose length counts the samples it sits out, and
// catches up in the general code after the batch. The QUIET flavour has the longer dependency chain (two codes per
// sample) and is only used while run-length codes keep appearing; it returns whether this lane saw one.
#ifndef ALACB200_EUNROLL
#define ALACB200_EUNROLL 2  // was 4 while four groups shared an SM; with eight, the loop's footprint in the L0 I-cache counts more
#endif
constexpr int E_UNROLL = ALACB200_EUNROLL;
#ifndef ALACB200_PUNROLL
#define ALACB200_PUNROLL 2
#endif
constexpr int P_UNROLL = ALACB200_PUNROLL;
#ifndef ALACB200_QUNROLL
#define ALACB200_QUNROLL 2
#endif
constexpr int Q_UNROLL = ALACB200_QUNROLL;
template <bool QUIET>
__device__ __forceinline__ bool decode_batch(BitReader &br, Entropy &e, uint32_t &bp, uint32_t pk_size, uint32_t lim,
                                             uint32_t a0, uint32_t a_last) {
    bool saw_run = false;
    const uint32_t a_end = a0 + (CHUNK / 2) * 128u;
#pragma unroll (QUIET ? Q_UNROLL : E_UNROLL)
    for (uint32_t aj = a0; aj != a_end; aj += 128u) {
        const uint32_t n0 = br.load(br.qo);  // the word after lo
        const uint32_t w = br.window();
        const uint32_t pre = clz_nz(~w);  // leading ones; 0xffffffff when all 32 are ones
        const uint32_t k = min(bit_index((e.mean >> 9) + 3u), e.kb);
        const uint32_t pre1 = pre + 1u;
        const uint32_t v = __funnelshift_l(shl_go(w, pre1), 0u, k);  // the k bits after the prefix; k == 0 -> 0
        // prefix * (2^k - 1) + (v >= 2 ? v - 1 : 0): v < 2 means "no suffix value" and gives one bit back
        const uint32_t r = shl_go(pre, k) - pre1 + max(v, 1u);
        const uint32_t nb0 = pre + k + (min(v, 2u) >> 1);  // kb <= 22 on this path: <= 31 bits, one refill
        const bool hold = e.zrun != 0u;
        const bool take = !hold & (bp < lim) & (pre < 9u) & (r <= 0xffffu);
        const uint32_t nb = take ? nb0 : 0u;
        const uint32_t nd = take ? r + e.zmode : 0u;
        const uint32_t n1 = QUIET ? br.load(br.qo + 4u) : 0u;
        const bool adv = br.advance(nb, n0);
        bp += nb;
        const uint32_t mean2 = e.pb * nd + e.mean - ((e.pb * e.mean) >> 9);
        sts32(aj, (int32_t)nd);  // the consumer undoes the sign fold (code_to_residual)
        // the run-length code: due after a code that leaves a small mean, unless it was the last sample (golomb.go:220)
        const bool zdue = take & ((mean2 << 2) < 512u) & (aj != a_last);
        // a real or pseudo zero run loses one sample; a lane that is not in one and did not take its code freezes
        if (hold) e.zrun -= 1u;
        if (!hold & !take) e.zrun = ZRUN_REDO;
        if (!QUIET) {
            e.mean = take ? mean2 : e.mean;
            e.zmode = take ? 0u : e.zmode;
            if (zdue) e.zrun = ZRUN_OWES_RUN;
        } else {
            saw_run |= zdue;
            int32_t k32 = __clz((int32_t)mean2) - 24 + (int32_t)((mean2 + 16u) >> 6);  // <= 10 when due
            k32 = max(k32, 0);
            const uint32_t mz = ((1u << (k32 & 31)) - 1u) & e.wb;
            const uint32_t w2 = br.window();
            const uint32_t pre2 = clz_nz(~w2);
            const uint32_t val = __funnelshift_l(shl_go(w2, pre2 + 1u), 0u, (uint32_t)k32);
            const uint32_t run = pre2 * mz + max(val, 1u) - 1u;
            const uint32_t nb2 = pre2 + (uint32_t)k32 + (min(val, 2u) >> 1);  // <= 20 bits
            // escape-coded runs, a position past the packet and runs past the stream end (golomb.go:232) go the long way
            const bool go = zdue & (pre2 < 9u) & ((bp >> 3) <= pk_size) & (run <= ((a_last - aj) >> 7));
            const uint32_t nbb = go ? nb2 : 0u;
            (void)br.advance(nbb, adv ? n1 : n0);
            bp += nbb;
            e.mean = go ? 0u : take ? mean2 : e.mean;
            e.zmode = go ? 1u : take ? 0u : e.zmode;
            if (zdue) e.zrun = go ? run : ZRUN_OWES_RUN;
        }
    }
    return saw_run;
}

// Produce one stream: ceil(nmax/32) ring slots (at least one: it carries the job). The two halves of an interleaved
// escape pair are filled in the same pass and go out in alternating slots (first half, second half, first half, ...).
__device__ __forceinline__ void produce_stream(DecShared &sm, uint32_t lane, uint32_t &seq, const Packet &pk,
                                               const DevConfig &cfg, BitReader &br, uint32_t &bp, int32_t &st,
                                               const StreamSpec &sp, const StreamSpec &sp2, bool pair, bool &quiet,
                                               RoleTimer &rt) {
    bool active = sp.active && st == ST_OK;
    const uint32_t nmax = __reduce_max_sync(FULL_MASK, active ? sp.n : 0u);
    const uint32_t nchunks = max(1u, (nmax + CHUNK - 1) / CHUNK);
    Entropy e;
    e.mean = cfg.mb;
    e.zmode = 0;
    e.zrun = 0;
    e.pb = (cfg.pb * sp.pb_factor) / 4u;  // SetAGParams, decoder.go:296-300
    e.kb = cfg.kb;
    e.wb = shl_go(1u, cfg.kb) - 1u;
    e.max_size = sp.chan_bits;
    e.size8 = pk.size * 8u;
    // per-lane reasons to stay out of the straight-line path
    uint32_t busy = (sp.escape ? BUSY_ESCAPE : 0u) | (cfg.kb > 22u ? BUSY_LONG_CODES : 0u) | (active ? 0u : BUSY_DEAD);
#pragma unroll 1
    for (uint32_t c = 0; c < nchunks; c++) {
        const uint32_t slot = seq % RING_SLOTS, slot2 = (seq + 1u) % RING_SLOTS;
        const unsigned long long tw = rt.now();
        wait_empty(sm, seq);
        if (pair) wait_empty(sm, seq + 1u);
        rt.add(1, tw);
        if (c == 0) {
            sm.job[slot][0][lane] = sp.n;
            sm.job[slot][1][lane] = (active ? sp.meta : (uint32_t)JOB_INACTIVE) | (pair ? (uint32_t)JOBF_PAIR : 0u);
            sm.job[slot][2][lane] = sp.coef_bitpos;
            sm.job[slot][3][lane] = nmax;
            sm.job[slot][4][lane] = active ? sp.live : 0u;
            sm.job[slot][5][lane] = sp.shift_bitpos;
            if (pair) {
                sm.job[slot2][0][lane] = sp2.n;
                sm.job[slot2][1][lane] = active ? sp2.meta : (uint32_t)JOB_INACTIVE;
                sm.job[slot2][2][lane] = sp2.coef_bitpos;
                sm.job[slot2][3][lane] = nmax;
                sm.job[slot2][4][lane] = 0u;  // escape pairs arrive interleaved: not emitted live
            }
        }
        const uint32_t a_dst = smem_u32(&sm.ring[slot][0][lane]);
        const uint32_t a_pair = smem_u32(&sm.ring[slot2][0][lane]) - a_dst;
        // samples of this lane inside this chunk
        const uint32_t base_i = c * CHUNK;
        const uint32_t cnt = (active && sp.n > base_i) ? min((uint32_t)CHUNK, sp.n - base_i) : 0u;
        const uint32_t a_last = a_dst + (sp.n - 1u - base_i) * 128u;  // ring address of the stream's last sample, if it is in this chunk
        // a lane with a short last chunk stops in the middle of it: it takes the general step for this chunk
        busy = (busy & ~BUSY_PARTIAL) | ((cnt != 0u && cnt != (uint32_t)CHUNK) ? BUSY_PARTIAL : 0u);
        if (cnt == 0u) e.zrun = ZRUN_PARKED;  // nothing (left) to decode: idle without touching bp
        // a lane that cannot use the straight-line decode at all (escape element, long codes, short chunk) fails
        // the packet-overrun test of every sample instead
        const uint32_t lim = busy ? 0u : e.size8;
#pragma unroll 1
        for (uint32_t half = 0; half < 2; half++) {
            // keep the staged window ahead of the reader: 16 samples eat at most 16 x 67 bits = 9 chunks of 16
            // bytes, and what is consumed now was requested at least one such period ago
            if (active) {
                const unsigned long long tt = rt.now();
                br.top_up();
                rt.add(2, tt);
            }
            const uint32_t a0 = a_dst + half * (CHUNK / 2) * 128u;  // ring address of the lane's sample: a_dst + 128 j
            // 16 samples without a branch (decode_batch), in the flavour the previous batches call for
            if (quiet) {
                const bool saw_run = decode_batch<true>(br, e, bp, pk.size, lim, a0, a_last);
                quiet = __any_sync(FULL_MASK, saw_run);
            } else {
                (void)decode_batch<false>(br, e, bp, pk.size, lim, a0, a_last);
            }
            // ---- frozen lanes catch up: general step (DynDecomp as written) for the samples they sat out ------------
            const bool frozen = e.zrun >= ZRUN_FROZEN_MIN && e.zrun < ZRUN_PARKED - 0x10000u;
            if (__any_sync(FULL_MASK, frozen)) {
                // run-length codes have started to appear: the next batch decodes them in line
                quiet = quiet | __any_sync(FULL_MASK, frozen && e.zrun <= ZRUN_OWES_RUN);
                if (frozen) {
                    const bool owes = e.zrun <= ZRUN_OWES_RUN;
                    const uint32_t since = (owes ? ZRUN_OWES_RUN : ZRUN_REDO) - e.zrun;  // samples after the one it froze at
                    const uint32_t jend = (half + 1u) * (CHUNK / 2);
                    uint32_t j = jend - 1u - since;
                    e.zrun = 0;
                    bool alive = true;
                    if (owes) {  // sample j is decoded, its run-length code is not
                        alive = zero_run_start(pk, br, bp, e, base_i + j, sp.n, st);
                        j++;
                    }
#pragma unroll 1
                    for (; j < jend; j++) {
                        int32_t res = 0, res2 = 0;
                        if (alive && j < cnt) {
                            if (sp.escape) {
                                res = escape_sample(br, sp.chan_bits);
                                if (pair) res2 = escape_sample(br, sp.chan_bits);
                            } else if (!entropy_next(pk, br, bp, e, base_i + j, sp.n, res, st)) {
                                alive = false;
                                res = 0;
                            }
                        }
                        sts32(a_dst + j * 128u, residual_to_code(res));
                        if (pair) sts32(a_dst + j * 128u + a_pair, residual_to_code(res2));
                    }
                    if (!alive) {  // a failed lane idles through the rest of the stream
                        active = false;
                        busy |= BUSY_DEAD;
                        e.zrun = ZRUN_PARKED;
                    }
                }
            }
        }
        arrive_full(sm, seq);
        seq++;
        if (pair) {
            arrive_full(sm, seq);
            seq++;
        }
    }
}

// Parsed element header of one lane (decodeSCE/decodeCPE up to the entropy stage, decoder.go:210-300, :348-460).
struct ElemHdr {
    bool have;    // an audio element is ready to be streamed
    bool stereo;
    bool escape;
    uint32_t n, chan_bits, shift, mix_bits, shift_bitpos, chan_idx;
    int32_t mix_res;
    uint32_t mode[2], den[2], pbf[2], num[2], coef_bitpos[2];
};

// One channel header: mode/denShift, pbFactor/num, num x 16-bit coefficients (decoder.go:275-286). The
// coefficients are not copied: the predictor warp reads them from the packet itself.
__device__ __forceinline__ void read_chan_hdr(const Packet &pk, Cursor &c, ElemHdr &h, int ch) {
    uint32_t hb = cur_read(pk, c, 8);
    h.mode[ch] = hb >> 4;
    h.den[ch] = hb & 0xfu;
    hb = cur_read(pk, c, 8);
    h.pbf[ch] = hb >> 5;
    h.num[ch] = hb & 0x1fu;
    h.coef_bitpos[ch] = c.bp;
    if (h.num[ch] > 0) {  // every Read(16) needs Pos+3 <= cap; the last one binds
        const uint32_t last = c.bp + 16u * (h.num[ch] - 1u);
        if ((last >> 3) + 3u > pk.size + 4u) c.panic = true;
        c.bp += 16u * h.num[ch];
    }
}

// Advance one lane through DSE/FIL/END until the next SCE/LFE/CPE header is parsed (decodePacketInto,
// decoder.go:142-203, and the header part of decodeSCE/decodeCPE). Sets h.have, or finishes the lane
// (parsing = false) with st.
__device__ __forceinline__ void parse_to_next_element(const Packet &pk, const DevConfig &cfg, Cursor &cur, uint32_t chan_idx,
                                                      uint32_t ns, bool &parsing, int32_t &st, ElemHdr &h) {
    h.have = false;
#pragma unroll 1
    while (parsing) {
        if ((cur.bp >> 3) >= pk.size) {  // PastEnd, decoder.go:143-145
            st = ST_BITSTREAM_OVERRUN;
            parsing = false;
            break;
        }
        const uint32_t tag = cur_read_small(pk, cur, 3);
        if (cur.panic) { st = ST_REF_PANIC; parsing = false; break; }
        if (tag == 0 || tag == 3 || tag == 1) {
            const bool stereo = tag == 1;
            if (stereo && chan_idx + 2 > cfg.num_channels) { parsing = false; break; }  // decoder.go:163-165
            const int32_t ctx = (stereo ? CTX_CPE : CTX_SCE) << 8;
            (void)cur_read_small(pk, cur, 4);
            const uint32_t unused = cur_read(pk, cur, 12);
            if (cur.panic) { st = ST_REF_PANIC | ctx; parsing = false; break; }
            if (unused != 0) { st = ST_INVALID_HEADER | ctx; parsing = false; break; }
            const uint32_t hb = cur_read(pk, cur, 4);
            if (cur.panic) { st = ST_REF_PANIC | ctx; parsing = false; break; }
            const uint32_t partial = hb >> 3;
            h.shift = (hb >> 1) & 3u;
            if (h.shift == 3u) { st = ST_INVALID_SHIFT | ctx; parsing = false; break; }
            h.escape = (hb & 1u) != 0;
            h.stereo = stereo;
            h.chan_idx = chan_idx;
            h.chan_bits = cfg.bit_depth - h.shift * 8u + (stereo ? 1u : 0u);
            h.n = ns;
            if (partial) {
                h.n = cur_read(pk, cur, 16) << 16;
                h.n |= cur_read(pk, cur, 16);
                if (cur.panic) { st = ST_REF_PANIC | ctx; parsing = false; break; }
            }
            h.mix_bits = 0;
            h.mix_res = 0;
            h.shift_bitpos = 0;
            // numSamples > frame_length: every later path re-slices a frame_length buffer and panics
            // (golomb.go:155, decoder.go:328, :506)
            const bool n_too_big = h.n > cfg.frame_length;
            if (!h.escape) {
                h.mix_bits = cur_read(pk, cur, 8);
                h.mix_res = (int32_t)(int8_t)cur_read(pk, cur, 8);
                read_chan_hdr(pk, cur, h, 0);
                if (stereo) read_chan_hdr(pk, cur, h, 1);
                if (cur.panic) { st = ST_REF_PANIC | ctx; parsing = false; break; }
                h.shift_bitpos = cur.bp;
                if (h.shift != 0) cur.bp += h.shift * 8u * h.n * (stereo ? 2u : 1u);
                if (n_too_big) { st = ST_REF_PANIC | ctx; parsing = false; break; }
            } else {
                if (stereo) h.chan_bits = cfg.bit_depth;  // decoder.go:388
                if (n_too_big) { st = ST_REF_PANIC | ctx; parsing = false; break; }
                if (h.n > 0) {
                    // every Read needs Pos+3 <= cap; positions only grow, so checking the last one is enough
                    const uint32_t per = h.chan_bits * (stereo ? 2u : 1u);
                    const uint32_t last_nb = h.chan_bits <= 16u ? h.chan_bits : h.chan_bits - 16u;
                    const uint32_t bp_last = cur.bp + h.n * per - last_nb;
                    if ((bp_last >> 3) + 3u > pk.size + 4u) { st = ST_REF_PANIC | ctx; parsing = false; break; }
                }
            }
            h.have = true;
            break;
        } else if (tag == 2 || tag == 5) {
            st = ST_UNSUPPORTED_ELEMENT;
            parsing = false;
        } else if (tag == 4) {  // skipDSE, decoder.go:553-574
            (void)cur_read_small(pk, cur, 4);
            const uint32_t align = cur_read_one(pk, cur);
            uint32_t count = cur_read_small(pk, cur, 8);
            if (count == 255) count += cur_read_small(pk, cur, 8);
            if (cur.panic) { st = ST_REF_PANIC | (CTX_DSE << 8); parsing = false; break; }
            if (align) cur.bp = (cur.bp + 7u) & ~7u;
            cur.bp += count * 8u;
            if ((cur.bp >> 3) >= pk.size) { st = ST_BITSTREAM_OVERRUN | (CTX_DSE << 8); parsing = false; }
        } else if (tag == 6) {  // skipFIL, decoder.go:538-551
            uint32_t count = cur_read_small(pk, cur, 4);
            if (count == 15) count += cur_read_small(pk, cur, 8) - 1u;
            if (cur.panic) { st = ST_REF_PANIC | (CTX_FIL << 8); parsing = false; break; }
            cur.bp += count * 8u;
            if ((cur.bp >> 3) >= pk.size) { st = ST_BITSTREAM_OVERRUN | (CTX_FIL << 8); parsing = false; }
        } else {  // END, decoder.go:192-195
            parsing = false;
        }
    }
}

// One group of 32 packets. `seq` (ring sequence number) lives across the groups of a persistent CTA; `descs` are the
// CTA's own 32 descriptors.
__device__ __forceinline__ void entropy_warp(DecShared &sm, uint32_t lane, const uint8_t *__restrict__ packed,
                                             const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ sizes,
                                             uint32_t npackets, const DevConfig &cfg, PacketDesc *__restrict__ descs,
                                             uint32_t *__restrict__ out_bytes, int32_t *__restrict__ status, uint32_t group,
                                             uint32_t &seq, uint32_t *__restrict__ counters) {
    // the group after this one: fetched now, read by the whole CTA after the group's barrier
    if (lane == 0) sm.next_group = atomicAdd(&counters[0], 1u);
    const uint32_t pidx = group * 32u + lane;
    const bool valid = pidx < npackets;
    Packet pk{packed, 0};
    if (valid) pk = Packet{packed + offsets[pidx], sizes[pidx]};
    PacketDesc *desc = descs + lane;
    const uint32_t fifo_addr = smem_u32(&sm.fifo[lane][0]) ^ ((lane & 7u) << 4);

    Cursor cur{0, false};
    uint32_t ns = cfg.frame_length, chan_idx = 0, nops = 0;
    int32_t st = ST_OK;
    bool parsing = valid;
    if (valid && pk.size > 0x0FFFFFFFu) { st = ST_REF_PANIC; parsing = false; }  // bit positions are 32-bit here
    bool quiet = false;      // warp-uniform: run-length codes keep appearing, decode them in line (decode_batch<true>)
    BitReader br;
    br.fifo = fifo_addr;
    RoleTimer rt(lane, 0);
    const unsigned long long t_start = rt.now();

#pragma unroll 1
    for (;;) {
        ElemHdr h;
        h.have = false;
        if (parsing) parse_to_next_element(pk, cfg, cur, chan_idx, ns, parsing, st, h);
        if (!__any_sync(FULL_MASK, h.have)) break;
        const int32_t ctx = (h.stereo ? CTX_CPE : CTX_SCE) << 8;
        StreamSpec s0, s1;
        s0.live = s1.live = 0;
        s0.shift_bitpos = s1.shift_bitpos = 0;
        // 2-channel streams whose 32 packets all carry one compressed pair: the predictor warp emits PCM itself
        #ifdef ALACB200_DEV
        const bool live_allowed = !(g_debug_flags & 1u);
#else
        const bool live_allowed = true;
#endif
        const bool live_round = cfg.num_channels == 2u && live_allowed &&
                                __all_sync(FULL_MASK, !valid || (h.have && h.stereo && !h.escape && st == ST_OK &&
                                                                 (h.num[1] == 0 || h.num[1] == 31 || h.num[1] == 8 ||
                                                                  (h.num[1] >= 4 && h.num[1] <= 6))));
        s0.active = h.have;
        s1.active = h.have && h.stereo;
        s0.escape = s1.escape = h.escape;
        s0.n = s1.n = h.n;
        s0.chan_bits = s1.chan_bits = h.chan_bits;
        if (h.have) {
            if (!h.escape) {
                // DynDecomp entry: input := Buf[Pos:] (golomb.go:149) and the first read32bit when Pos > Size
                const uint32_t pos = cur.bp >> 3;
                if (pos > pk.size + 4u || (h.n > 0 && pos > pk.size)) st = ST_REF_PANIC | ctx;
                for (int c = 0; c < 2; c++) {
                    StreamSpec &s = c ? s1 : s0;
                    const uint32_t ord = h.num[c];
                    const bool reg_path = ord == 0 || ord == 31 || (ord >= 4 && ord <= 6) || ord == 8;
                    s.pb_factor = h.pbf[c];
                    s.meta = job_meta(reg_path ? JOB_REG : JOB_GENERIC, ord, h.den[c], h.mode[c], h.chan_bits, h.chan_idx + c);
                    s.coef_bitpos = h.coef_bitpos[c];
                }
            } else {
                s0.pb_factor = s1.pb_factor = 0;
                s0.meta = job_meta(JOB_REG, 0, 0, 0, h.chan_bits, h.chan_idx);      // pass-through
                s1.meta = job_meta(JOB_REG, 0, 0, 0, h.chan_bits, h.chan_idx + 1);
                s0.coef_bitpos = s1.coef_bitpos = 0;
            }
            if (st == ST_OK) br.init(pk, cur.bp, fifo_addr);
        }
        // compressed elements: pass 0 = U (or mono), pass 1 = V; escape pairs: pass 2, one interleaved sweep
        // feeding both consumers (decoder.go:513-533)
        uint32_t bp = cur.bp;
#pragma unroll 1
        for (int pass = 0; pass < 3; pass++) {
            const bool esc_pair = h.have && h.stereo && h.escape;
            const bool act = pass == 0 ? (h.have && !esc_pair) : pass == 1 ? (h.have && h.stereo && !h.escape) : esc_pair;
            if (!__any_sync(FULL_MASK, act)) continue;
            StreamSpec a = pass == 1 ? s1 : s0;
            a.active = act;
            if (pass == 1 && act && st == ST_OK) {
                // U's predictor warm-up indexes [1..numActive] of frame_length-long slices (predictor.go:76-79),
                // then V's DynDecomp entry: bitBuf.Buf[bitBuf.Pos:] (golomb.go:149)
                const uint32_t pos = bp >> 3;
                if ((h.num[0] != 0 && h.num[0] != 31 && h.num[0] >= cfg.frame_length) || pos > pk.size + 4u ||
                    (h.n > 0 && pos > pk.size))
                    st = ST_REF_PANIC | ctx;
            }
            const int32_t before = st;
            if (pass == 1 && live_round) {
                a.live = 0x80000000u | (h.mix_bits & 0xffu) | (((uint32_t)h.mix_res & 0xffu) << 8) | (h.shift << 16);
                a.shift_bitpos = h.shift_bitpos;
            }
            produce_stream(sm, lane, seq, pk, cfg, br, bp, st, a, s1, pass == 2, quiet, rt);
            if (act && before == ST_OK && st != ST_OK) {  // an entropy error of this stream: tag it (decoder.go:303, :463, :478)
                if ((st & 0xff) == ST_REF_PANIC) st |= ctx;
                else st |= ctx | ((pass == 1 ? ENT_V : h.stereo ? ENT_U : ENT_MONO) << 12);
            }
        }
        // ---- per-lane epilogue of the element: position, panics of the predictor/writer, op record ----
        if (h.have) {
            if (st != ST_OK) {
                parsing = false;
            } else {
                if (!h.escape) cur.bp = bp;
                else cur.bp += h.n * h.chan_bits * (h.stereo ? 2u : 1u);
                // warm-up indexes [1..numActive] of frame_length-long slices (predictor.go:76-79)
                const uint32_t last = h.stereo ? 1u : 0u;
                if (!h.escape && h.num[last] != 0 && h.num[last] != 31 && h.num[last] >= cfg.frame_length) st = ST_REF_PANIC | ctx;
                const uint32_t out_chan = (uint32_t)k_layout[cfg.num_channels - 1][h.chan_idx];
                // dst := out[off:off+W:off+W] past cap(out), matrix.go:44 (a pair mapped onto the last channel)
                if (st == ST_OK && h.n > 0 && out_chan + (h.stereo ? 2u : 1u) > cfg.num_channels && h.n == cfg.frame_length)
                    st = ST_REF_PANIC | ctx;
                if (st != ST_OK) {
                    parsing = false;
                } else {
                    OpDesc op;
                    op.n = h.n;
                    op.shift_bitpos = h.shift_bitpos;
                    op.kind = h.stereo ? 2 : 1;
                    op.out_chan = (uint8_t)out_chan;
                    op.slot = (uint8_t)h.chan_idx;
                    op.shift = (uint8_t)(h.escape ? 0u : h.shift);
                    op.mix_bits = (uint8_t)h.mix_bits;
                    op.mix_res = (int8_t)h.mix_res;
                    op.pad_ = live_round ? 1 : 0;  // already written to pcm_out by the predictor warp
                    desc->ops[nops++] = op;
                    ns = h.n;
                    chan_idx += h.stereo ? 2u : 1u;
                    if (chan_idx >= cfg.num_channels) parsing = false;  // decoder.go:200-202
                }
            }
        }
    }
    BitReader::wait_all();
    rt.add(0, t_start);
    rt.flush(3);
#ifdef ALACB200_DEV
    if (rt.slot) {
        uint32_t smid, wid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
        rt.slot[11] = ((unsigned long long)smid << 8) | wid;
    }
#endif
    // the group is finished: tell the predictor warp
    wait_empty(sm, seq);
    sm.job[seq % RING_SLOTS][1][lane] = JOB_EXIT;
    arrive_full(sm, seq);
    seq++;
    if (valid) {
        desc->status = st;
        desc->n_final = ns;
        desc->nops = nops;
        status[pidx] = st;
        out_bytes[pidx] = st == ST_OK ? ns * cfg.num_channels * cfg.bps : 0u;
    }
}

// ====================================================================================================
// PREDICTOR warp
// ====================================================================================================
// Order-31 pre-pass (mode != 0: UnpcBlock(pred, pred, n, nil, 31, chanBits, 0), decoder.go:306-308)
__device__ __forceinline__ int32_t delta_step(bool on, int32_t &prev, int32_t r, uint32_t i, uint32_t cs) {
    if (!on) return r;
    prev = (i == 0) ? r : sext_go(r + prev, cs);
    return prev;
}

struct Job {
    uint32_t kind, order, den, mode, chan_bits, slot, n, coef_bitpos, nmax, live, shift_bitpos;
};

// sb (8 or 16) bits at bit offset `rel` of a staged shift row (bytes in stream order, 32-bit words as loaded)
__device__ __forceinline__ uint32_t shift_field(const uint32_t *row_words, uint32_t rel, uint32_t sb) {
    const uint32_t b = rel >> 3;
    const uint32_t w0 = __byte_perm(row_words[b >> 2], 0, 0x0123);
    const uint32_t w1 = __byte_perm(row_words[(b >> 2) + 1u], 0, 0x0123);
    const uint32_t win = __funnelshift_l(w1, w0, (b & 3u) * 8u + (rel & 7u));  // < 32
    return win >> (32u - sb);
}

// ---- the writer rules of stage 3 (WriteStereo*/WriteMono*, matrix.go:30-301), one copy for every emit path -----------
// One frame: un-mix (matrix.go:40-41), 20-bit samples moved up by 4, then the shift buffer merge (matrix.go:132-135,
// :270-272: BitBuffer.Read of sb bits at bit `rel` of the staged shift row). A mono frame leaves `right` alone.
__device__ __forceinline__ void writer_frame(int32_t &left, int32_t &right, bool stereo, int32_t mix_res, uint32_t mix_bits,
                                             bool depth20, uint32_t sb, const uint32_t *shift_row, uint32_t rel) {
    if (stereo && mix_res != 0) {
        const int32_t v = right;
        left = left + v - sar_go(mix_res * v, mix_bits);
        right = left - v;
    }
    if (depth20) {
        left = (int32_t)((uint32_t)left << 4);
        right = (int32_t)((uint32_t)right << 4);
    }
    if (sb) {
        left = (int32_t)shl_go((uint32_t)left, sb) | (int32_t)shift_field(shift_row, rel, sb);
        if (stereo) right = (int32_t)shl_go((uint32_t)right, sb) | (int32_t)shift_field(shift_row, rel + sb, sb);
    }
}

// OR frame q of a batch -- the BPS little-endian bytes of `left`, then, for WIDTH 2, those of `right` -- into the packed
// words ow[] of the batch; a frame that is not kept (past the sample count, decoder.go:120, :127) stays zero.
template <int BPS, int WIDTH>
__device__ __forceinline__ void pack_frame(uint32_t *ow, int q, int32_t left, int32_t right, bool keep) {
    constexpr int FB = BPS * WIDTH;
    constexpr uint64_t lmask = BPS == 4 ? 0xffffffffull : ((1ull << (8 * BPS)) - 1ull);
    uint64_t v = (uint64_t)(uint32_t)left & lmask;
    if (WIDTH == 2) v |= ((uint64_t)(uint32_t)right & lmask) << (8 * BPS);
    if (!keep) v = 0;
    const int bit = q * FB * 8;  // static after unrolling
    const int wi = bit / 32, sh = bit % 32;
    ow[wi] |= (uint32_t)(v << sh);
    if (sh + FB * 8 > 32) ow[wi + 1] |= (uint32_t)(v >> (32 - sh));
    if (sh + FB * 8 > 64) ow[wi + 2] |= (uint32_t)(v >> (64 - sh));
}

// Store the packed words of FRAMES frames (NW4 x 16 bytes) from frame f0 on to a packet slot: 128-bit stores when the
// batch is whole and the slot 16-byte aligned, else 32-bit stores and the bytes of a last partial word (the last, short
// batch of a frame length that is not a multiple of FRAMES; 24-bit pairs are a multiple of 4 bytes only for an even
// number of frames).
template <int NW4, int FRAMES>
__device__ __forceinline__ void store_words(uint8_t *slot, uint32_t f0, uint32_t frame_bytes, uint32_t frame_length,
                                            bool vec_ok, const uint32_t *ow) {
    uint8_t *dst = slot + (size_t)f0 * frame_bytes;
    const uint32_t frames_here = min((uint32_t)FRAMES, frame_length - f0);
    if (frames_here == (uint32_t)FRAMES && vec_ok) {
#pragma unroll
        for (int k = 0; k < NW4; k++)
            reinterpret_cast<uint4 *>(dst)[k] = make_uint4(ow[4 * k], ow[4 * k + 1], ow[4 * k + 2], ow[4 * k + 3]);
    } else {
        const uint32_t nb = frames_here * frame_bytes;
#pragma unroll
        for (int k = 0; k < 4 * NW4; k++) {
            if ((uint32_t)(4 * k + 4) <= nb) reinterpret_cast<uint32_t *>(dst)[k] = ow[k];
            else
                for (int j = 0; j < 4; j++)
                    if ((uint32_t)(4 * k + j) < nb) dst[4 * k + j] = (uint8_t)(ow[k] >> (8 * j));
        }
    }
}

// Word k of a shift row staged from packet byte rel_pk on (gsrc: the row's 4-byte aligned global address): one aligned
// load, or, where the word runs past the packet end, its bytes one by one with those outside the packet read as zero
// (bitbuffer.go:36-51).
__device__ __forceinline__ uint32_t shift_word(const Packet &pk, int64_t rel_pk, uint32_t k, const uint32_t *gsrc) {
    const int64_t b_first = rel_pk + 4 * (int64_t)k;
    if (b_first + 4 <= (int64_t)pk.size) return __ldg(gsrc + k);
    uint32_t w = 0;
    for (int j = 0; j < 4; j++)
        if (b_first + j >= 0 && b_first + j < (int64_t)pk.size) w |= (uint32_t)__ldg(pk.p + (b_first + j)) << (8 * j);
    return w;
}

// What the predictor warp needs to emit PCM itself (2-channel streams), apart from the per-lane words in
// DecShared::live_ctx: launch facts that rematerialise from the kernel's parameter bank. Only ever handed to inlined
// code, so it never has an address.
struct LiveEnv {
    const int32_t *scratch;  // the kernel's scratch parameter: CTA b owns [b][channel][sample][lane]
    uint32_t num_channels;
    uint8_t *pcm_out;
    uint64_t out_stride;
    PacketDesc *descs;      // the kernel's descriptor parameter: CTA b owns [b][32]
    uint32_t frame_length, bps, bit_depth;
    bool enabled;
};
// this CTA's slot of parked samples, rebuilt from the launch parameters where it is needed
__device__ __forceinline__ const int32_t *cta_scratch(const LiveEnv &lc) {
    return lc.scratch + (size_t)cta_now() * lc.num_channels * lc.frame_length * 32u;
}
__device__ __forceinline__ uint32_t live_shift_bits(uint32_t bit_depth, uint32_t live_word) {
    return (bit_depth == 24 || bit_depth == 32) ? ((live_word >> 16) & 3u) * 8u : 0u;
}
// bit offset, inside the staged shift row, of the first shift field of chunk `ck` (the row starts at the 16-byte aligned
// address at or below the field's byte)
__device__ __forceinline__ uint32_t live_rel0(uint32_t live_word, uint32_t shift_bitpos, uint32_t sb, uint32_t ck) {
    const uint32_t first_bit = shift_bitpos + ck * CHUNK * 2u * sb;
    const uint32_t lead = (((live_word >> 18) & 15u) + (first_bit >> 3)) & 15u;
    return lead * 8u + (first_bit & 7u);
}

// Start fetching what the emission of chunk `ck` needs: the parked U samples of the 32 frames (one 4 KB block,
// cooperative) and this lane's shift bytes, all by cp.async so they land while the predictor runs.
__device__ __forceinline__ void live_prefetch(DecShared &sm, uint32_t lane, const LiveEnv &lc, const Packet &pk, uint32_t ck) {
    const uint32_t n_lane = sm.live_ctx[0][lane], live_word = sm.live_ctx[1][lane];
    const uint32_t sb = live_shift_bits(lc.bit_depth, live_word);
    const uint32_t shift_bitpos = sm.live_ctx[2][lane];
    const bool live_lane = (live_word >> 31) != 0u;
    const uint32_t base_i = ck * CHUNK;
    const uint8_t *ug = reinterpret_cast<const uint8_t *>(cta_scratch(lc) + (size_t)base_i * 32u);  // channel 0: U
    const uint32_t frames_left = lc.frame_length > base_i ? lc.frame_length - base_i : 0u;
    const uint32_t ubase = smem_u32(&sm.live_u[0][0]);
#pragma unroll
    for (uint32_t k = 0; k < 8; k++) {
        const uint32_t piece = k * 32u + lane;                  // 16-byte piece of the 4 KB block: frame = piece / 8
        const uint32_t nb = (piece >> 3) < frames_left ? 16u : 0u;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ubase + piece * 16u),
                     "l"(ug + (nb ? (size_t)piece * 16u : 0)), "r"(nb)
                     : "memory");
    }
    const uint32_t cnt = (live_lane && n_lane > base_i) ? min((uint32_t)CHUNK, n_lane - base_i) : 0u;
    if (sb && cnt) {
        const uint32_t first_bit = shift_bitpos + base_i * 2u * sb;
        const uint32_t nbytes = ((first_bit & 7u) + cnt * 2u * sb + 7u) / 8u + 2u;  // +2: the 24-bit window of BitBuffer.Read
        const uint8_t *g0 = pk.p + (first_bit >> 3);
        const uint8_t *ga = reinterpret_cast<const uint8_t *>(((uintptr_t)g0) & ~(uintptr_t)15);
        const uint32_t lead = (uint32_t)(g0 - ga);
        const uint32_t nchunks = (lead + nbytes + 15u) / 16u;  // <= LIVE_SHIFT_CHUNKS
        const uint8_t *pend = pk.p + pk.size;
        const uint32_t sbase = smem_u32(&sm.live_shift[lane][0]);
#pragma unroll
        for (uint32_t c = 0; c < LIVE_SHIFT_CHUNKS; c++) {
            if (c < nchunks) {
                const uint8_t *src = ga + c * 16u;
                // bytes at or past the packet end arrive as zeros (bitbuffer.go:36-51)
                const uint32_t nb = src >= pend ? 0u : (uint32_t)min((ptrdiff_t)16, pend - src);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sbase + c * 16u), "l"(nb ? src : ga), "r"(nb)
                             : "memory");
            }
        }
    }
}

// Where and in which shape a live pair's PCM leaves (built inside live_chunk_emit from by-value arguments).
struct LiveOut {
    uint8_t *slot;  // this lane's packet slot in pcm_out
    uint32_t frame_length, bit_depth;
    bool vec_ok;
};

// Generic (any depth / shift) emission of the 32 frames of chunk `ck` of a live pair: V from the ring slot, U from live_u,
// shift bytes from live_shift; two batches of 16 frames, each leaving as 2*BPS 128-bit stores to the lane's own packet
// slot (matrix.go:30-215).
template <int BPS>
__device__ __noinline__ void live_emit_generic(DecShared &sm, uint32_t lane, const LiveOut lc, uint32_t ck, bool live_lane,
                                          uint32_t n_lane, uint32_t live_word, uint32_t sb, uint32_t rel0,
                                          const int32_t *vsrc) {
    constexpr int FB = 2 * BPS;
    constexpr int EB = 16;
    const int32_t mix_res = (int32_t)(int8_t)((live_word >> 8) & 0xffu);
    const uint32_t mix_bits = live_word & 0xffu;
    const bool depth20 = lc.bit_depth == 20;
    const uint32_t *shrow = reinterpret_cast<const uint32_t *>(&sm.live_shift[lane][0]);
#pragma unroll 1
    for (uint32_t half = 0; half < 2; half++) {
        const uint32_t f0 = ck * CHUNK + half * EB;
        if (f0 >= lc.frame_length) break;
        const uint32_t cnt = n_lane > f0 ? min((uint32_t)EB, n_lane - f0) : 0u;
        uint32_t ow[4 * FB];
#pragma unroll
        for (int k = 0; k < 4 * FB; k++) ow[k] = 0;
#pragma unroll
        for (int q = 0; q < EB; q++) {
            const uint32_t jq = half * EB + (uint32_t)q;
            int32_t left = sm.live_u[jq][lane], right = vsrc[jq * 32u];
            writer_frame(left, right, true, mix_res, mix_bits, depth20, sb, shrow, rel0 + jq * 2u * sb);
            pack_frame<BPS, 2>(ow, q, left, right, (uint32_t)q < cnt);
        }
        if (live_lane) store_words<FB, EB>(lc.slot, f0, FB, lc.frame_length, lc.vec_ok, ow);
    }
}

// un-mix of one frame (matrix.go:40-41; mixRes == 0 means plain L/R)
__device__ __forceinline__ void unmix(int32_t u, int32_t v, int32_t mix_res, uint32_t mix_bits, int32_t &left, int32_t &right) {
    const int32_t l = u + v - sar_go(mix_res * v, mix_bits);
    left = mix_res != 0 ? l : u;
    right = mix_res != 0 ? l - v : v;
}

// Emit the 32 frames of chunk `ck` of a live pair: V from the ring slot, U from live_u, shift bytes from live_shift; four
// batches of 8 frames, each leaving as 128-bit stores to the lane's own packet slot (WriteStereo16/24, matrix.go:30-142).
// The two shapes real streams have -- 16-bit, and 24-bit with one shifted byte -- are packed with byte permutes
// (3 PRMT per 2 frames); everything else takes the generic path. The batch loop is NOT unrolled: this code runs once per
// ring slot between two stretches of the predictor loop, and what it evicts from the instruction cache costs more than
// the loop overhead.
template <int BPS>
__device__ __forceinline__ void live_emit(DecShared &sm, uint32_t lane, const LiveOut &lc, uint32_t ck, bool live_lane,
                                          uint32_t n_lane, uint32_t live_word, uint32_t sb, uint32_t rel0,
                                          const int32_t *vsrc) {
    const bool fast = (BPS == 2 && lc.bit_depth == 16) || (BPS == 3 && lc.bit_depth == 24 && sb == 8u);
    if (!__all_sync(FULL_MASK, fast)) {
        live_emit_generic<BPS>(sm, lane, lc, ck, live_lane, n_lane, live_word, sb, rel0, vsrc);
        return;
    }
    const int32_t mix_res = (int32_t)(int8_t)((live_word >> 8) & 0xffu);
    const uint32_t mix_bits = live_word & 0xffu;
    const uint32_t *shrow = reinterpret_cast<const uint32_t *>(&sm.live_shift[lane][0]);
#pragma unroll 1
    for (uint32_t b8 = 0; b8 < CHUNK / 8; b8++) {
        const uint32_t f0 = ck * CHUNK + b8 * 8u;
        if (f0 >= lc.frame_length) break;
        const uint32_t cnt = n_lane > f0 ? min(8u, n_lane - f0) : 0u;
        if (BPS == 3) {
            // 8 frames x (1 byte L + 1 byte R) of shift data: 4 windows of 32 bits, two frames each
            const uint32_t rel = rel0 + b8 * 128u;
            const uint32_t wb = rel >> 5, bo = rel & 31u;
            uint32_t W[5], S[4];
#pragma unroll
            for (int k = 0; k < 5; k++) W[k] = __byte_perm(shrow[wb + k], 0, 0x0123);
#pragma unroll
            for (int k = 0; k < 4; k++) S[k] = __funnelshift_l(W[k + 1], W[k], bo);
            uint32_t ow[12];
#pragma unroll
            for (int pr = 0; pr < 4; pr++) {
                uint32_t x24[4];
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int q = 2 * pr + e;
                    const uint32_t jq = b8 * 8u + (uint32_t)q;
                    int32_t left, right;
                    unmix(sm.live_u[jq][lane], vsrc[jq * 32u], mix_res, mix_bits, left, right);
                    // (x << 8) | shift byte (matrix.go:132-135): frame 2k sits in the upper half of S[k], 2k+1 in the lower
                    uint32_t l24 = __byte_perm(S[pr], (uint32_t)left, e == 0 ? 0x6543 : 0x6541);
                    uint32_t r24 = __byte_perm(S[pr], (uint32_t)right, e == 0 ? 0x6542 : 0x6540);
                    if ((uint32_t)q >= cnt) l24 = r24 = 0;  // frames past the sample count stay zero
                    x24[2 * e] = l24;
                    x24[2 * e + 1] = r24;
                }
                ow[3 * pr] = __byte_perm(x24[0], x24[1], 0x4210);      // L0 L0 L0 R0
                ow[3 * pr + 1] = __byte_perm(x24[1], x24[2], 0x5421);  // R0 R0 L1 L1
                ow[3 * pr + 2] = __byte_perm(x24[2], x24[3], 0x6542);  // L1 R1 R1 R1
            }
            if (live_lane) store_words<3, 8>(lc.slot, f0, 6u, lc.frame_length, lc.vec_ok, ow);
        } else {
            uint32_t ow[8];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t jq = b8 * 8u + (uint32_t)q;
                int32_t left, right;
                unmix(sm.live_u[jq][lane], vsrc[jq * 32u], mix_res, mix_bits, left, right);
                uint32_t w = __byte_perm((uint32_t)left, (uint32_t)right, 0x5410);
                if ((uint32_t)q >= cnt) w = 0;
                ow[q] = w;
            }
            if (live_lane) store_words<2, 8>(lc.slot, f0, 4u, lc.frame_length, lc.vec_ok, ow);
        }
    }
}

// Stage 3 of one ring slot of a live pair, by the predictor warp itself: the slot holds the decoded V samples, live_u /
// live_shift were requested (live_prefetch) before the slot was predicted. One copy of the packing code for every
// instantiation of the predictor loop.
// Arguments by value, per-lane stream facts from DecShared::live_ctx: nothing here lives in local memory.
// `shape` = bytes per sample | bit depth << 8 | (slots 16-byte aligned) << 16.
__device__ __noinline__ void live_chunk_emit(DecShared &sm, uint32_t lane, uint8_t *slot, uint32_t frame_length, uint32_t shape,
                                             uint32_t ck, const int32_t *vsrc) {
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();  // live_u is fetched cooperatively
    LiveOut lo;
    lo.slot = slot;
    lo.frame_length = frame_length;
    lo.bit_depth = (shape >> 8) & 0xffu;
    lo.vec_ok = ((shape >> 16) & 1u) != 0;
    const uint32_t bps = shape & 0xffu;
    const uint32_t n_lane = sm.live_ctx[0][lane], live_word = sm.live_ctx[1][lane], shift_bitpos = sm.live_ctx[2][lane];
    const bool live_lane = (live_word >> 31) != 0u;
    const uint32_t sb = live_shift_bits(lo.bit_depth, live_word);
    const uint32_t rel0 = sb ? live_rel0(live_word, shift_bitpos, sb, ck) : 0u;
    if (bps == 3) live_emit<3>(sm, lane, lo, ck, live_lane, n_lane, live_word, sb, rel0, vsrc);
    else if (bps == 2) live_emit<2>(sm, lane, lo, ck, live_lane, n_lane, live_word, sb, rel0, vsrc);
    else live_emit<4>(sm, lane, lo, ck, live_lane, n_lane, live_word, sb, rel0, vsrc);
    __syncwarp();  // live_u / live_shift are free for the next slot's requests
}

// sign-extend the low `bits` (1..32) of v: (v << (32 - bits)) >> (32 - bits) in one SGXT (szext; bfe.s32 cost four instructions)
__device__ __forceinline__ int32_t sext_bits(int32_t v, uint32_t bits) {
    int32_t r;
    asm("szext.clamp.s32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(bits));
    return r;
}
__device__ __forceinline__ int32_t lds32(uint32_t addr) {
    int32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
// if (p) c += a * b, as one predicated IMAD
__device__ __forceinline__ void mad_if(int32_t &c, int32_t a, int32_t b, bool p) {
    asm("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q mad.lo.s32 %0, %1, %2, %0;\n\t}" : "+r"(c) : "r"(a), "r"(b), "r"((uint32_t)p));
}

// Register predictor: orders 4/5/6/8 with int32 coefficients (unpcBlock4/5/6/8, predictor.go:99-618), plus
// order 0 (copy, also escape pass-through) and order 31 (running sum), predictor.go:55-72. T = taps kept;
// a lane whose order is below T runs with its upper taps' history differences forced to zero, which keeps
// their coefficients at zero and their LMS terms at zero. The body is branch-free. The decoded samples replace the codes
// in the ring slot; when the slot is done they leave as PCM (`live`: the V stream of a 2-channel pair, live_chunk_emit)
// or are parked in the scratch. One loop body for both kinds of stream: the U and V streams of a packet alternate in
// this warp, and every KB of hot code less is instruction-cache hits for the 16 role warps of the SM (the 6 KB L0 of a
// scheduler holds the loops of its entropy and predictor warps or it does not: profiles/r02b, stall_no_inst).
template <int T, bool MODE>
__device__ __forceinline__ void stream_reg(DecShared &sm, uint32_t lane, uint32_t &seq, const Packet &pk,
                                           const Job &jb, bool active, RoleTimer &rt, const LiveEnv &lc, bool live) {
    const uint32_t cs = 32u - jb.chan_bits;
    const uint32_t den = jb.den;
    const int32_t den_half = den > 0 ? (int32_t)(1u << (den - 1)) : 0;
    const int32_t order = (int32_t)jb.order;
    const bool fir_order = order == 4 || order == 5 || order == 6 || order == 8;
    const uint32_t fir_from = fir_order ? (uint32_t)order + 1u : 0xffffffffu;
    const bool copy = order == 0;  // order 0 copies; warm-up and order 31 accumulate
    const bool mode = MODE && jb.mode != 0;
    const uint32_t n_lane = active ? jb.n : 0u;
    const bool sel4 = order == 4, sel5 = order == 5, sel6 = order == 6;
    int32_t c[T], h[T + 1], nwgt[T];  // nwgt = -(order - t): both ladders ADD weight * term (one IMAD per tap, no negation)
    uint32_t tmask[T];
#pragma unroll
    for (int t = 0; t < T; t++) {
        const bool in = fir_order && t < order;
        c[t] = (active && in) ? (int32_t)(int16_t)pk_bits(pk, jb.coef_bitpos + 16u * (uint32_t)t, 16) : 0;
        nwgt[t] = in ? t - order : 0;
        tmask[t] = in ? 0xffffffffu : 0u;
    }
#pragma unroll
    for (int t = 0; t <= T; t++) h[t] = 0;
    int32_t dprev = 0;
    const uint32_t nchunks = max(1u, (jb.nmax + CHUNK - 1) / CHUNK);
    // From the second ring slot on every FIR lane is past its warm-up (order <= 8 < 32). If the warp carries nothing but
    // such lanes, with samples of at most 31 bits (so a history difference never is INT_MIN) and no pre-pass, the
    // steady-state body below runs instead of the general one: no warm-up arithmetic, and the early-exit ladder of
    // predictor.go:137-185 in a sign-folded form -- with E = del0 for a positive residual and ~del0 for a negative one,
    // both ladders are "E -= weight * q; go on while E >= thr", q = |diff| >> denShift rounded down / up, thr = 1 / 0.
    const bool steady_ok = !MODE && __all_sync(FULL_MASK, !active || (fir_order && jb.chan_bits <= 31u));
    const uint32_t den_mask = (1u << den) - 1u;
    // One ring slot = wait for it, start the fetches its emission needs, run a sample loop over it, emit or park it, hand
    // it back. Two loops over the slots instead of one with both bodies in it: the general body takes the first slot of
    // every stream (warm-up) and every slot of a warp the steady body cannot serve, the steady body all others -- so the
    // invariants of the general body (order, warm-up bounds, pre-pass state) are dead while the steady loop runs and do
    // not compete with it for the 128 registers.
    auto slot_begin = [&](uint32_t ck) -> uint32_t {
        const uint32_t slot = seq % RING_SLOTS;
        if (ck > 0) {
            const unsigned long long tw = rt.now();
            wait_full(sm, seq);
            rt.add(1, tw);
        }
        if (live) live_prefetch(sm, lane, lc, pk, ck);  // lands while the slot is predicted
        return slot;
    };
    auto slot_end = [&](uint32_t ck, uint32_t slot) {
        // everything below is rebuilt from the launch parameters and re-read special registers: nothing of it is live
        // (or spilled) across the sample loop
        const uint32_t lane_v = lane_now();
        int32_t *vdst = &sm.ring[slot][0][lane_v];
        if (live) {
            const bool vec_ok = ((((uintptr_t)lc.pcm_out) | lc.out_stride) & 15u) == 0;
            const uint32_t pidx = (uint32_t)lds32(smem_u32(&sm.group)) * 32u + lane_v;
            live_chunk_emit(sm, lane_v, lc.pcm_out + (size_t)pidx * lc.out_stride, lc.frame_length,
                            lc.bps | (lc.bit_depth << 8) | ((vec_ok ? 1u : 0u) << 16), ck, vdst);
        } else {  // park the lane's column of the slot: [sample][lane], one 128-byte line per warp store
            const uint32_t base_i = ck * CHUNK;
            const uint32_t cnt = n_lane > base_i ? min((uint32_t)CHUNK, n_lane - base_i) : 0u;
            int32_t *outp = const_cast<int32_t *>(cta_scratch(lc)) + ((size_t)jb.slot * lc.frame_length + base_i) * 32u + lane_v;
#pragma unroll 8
            for (uint32_t j = 0; j < CHUNK; j++)
                if (j < cnt) outp[j * 32u] = vdst[j * 32];
        }
        arrive_empty(sm, seq);
        seq++;
    };
    uint32_t ck = 0;
#pragma unroll 1
    do {
        const uint32_t slot = slot_begin(ck);
        const int32_t *src = &sm.ring[slot][0][lane_now()];
// unroll 2, not more: the entropy warps sharing the SM pay for every extra KB of hot code in instruction fetch
#pragma unroll 2
        for (uint32_t j = 0; j < CHUNK; j++) {
            const uint32_t i = ck * CHUNK + j;
            int32_t r = code_to_residual((uint32_t)src[j * 32]);
            if (MODE) {  // order-31 pre-pass on the residuals (decoder.go:306-308)
                const int32_t dn = (i == 0) ? r : sext_go(r + dprev, cs);
                r = mode ? dn : r;
                dprev = r;
            }
            int32_t top;
            if (T == 8) top = sel4 ? h[4] : sel5 ? h[5] : sel6 ? h[6] : h[8];
            else top = sel4 ? h[4] : sel5 ? h[5] : h[6];
            int32_t d[T];
            int32_t sum = den_half;
#pragma unroll
            for (int t = 0; t < T; t++) {
                d[t] = top - h[t];
                if (t >= 4) d[t] &= (int32_t)tmask[t];  // orders start at 4: taps 0..3 always live
                sum -= c[t] * d[t];
            }
            const int32_t fir = sext_go(r + top + (sum >> den), cs);
            const int32_t warm = (i == 0 || copy) ? r : sext_go(r + h[0], cs);
            const bool is_fir = i >= fir_from;
            const int32_t x = is_fir ? fir : warm;
            // sign-LMS adaptation on the residual's sign: walk the taps from the oldest sample, stop once the
            // running residual has changed sign or reached zero (predictor.go:137-185)
            bool alive = is_fir && (r != 0);
            const int32_t smask = r >> 31;           // 0 / -1
            const int32_t sone = smask | 1;          // +1 / -1
            const int32_t thr = 1 + smask;           // continue while (D ^ smask) >= thr <=> D > 0 (r>0) / D < 0 (r<0)
            int32_t D = r;
#pragma unroll
            for (int t = T - 1; t >= 0; t--) {
                const int32_t sg = max(min(d[t], 1), -1);  // signOfInt
                const int32_t sgn = sg * sone;             // sign for r > 0, -sign for r < 0
                if (alive) c[t] -= sgn;
                if (t > 0) {
                    const int32_t term = (sgn * d[t]) >> den;
                    D += nwgt[t] * term;
                    alive = alive && ((D ^ smask) >= thr);  // masked taps: term 0, D still r: stays alive
                }
            }
#pragma unroll
            for (int t = T; t > 0; t--) h[t] = h[t - 1];
            h[0] = x;
            const_cast<int32_t *>(src)[j * 32] = x;
        }
        slot_end(ck, slot);
        ck++;
    } while (ck < nchunks && !steady_ok);
#pragma unroll 1
    for (; ck < nchunks; ck++) {
        const uint32_t slot = slot_begin(ck);
        {
            // the lane's column of the slot by shared address: one add per unrolled body instead of an index rebuilt from
            // the thread id (which is what the 128-register budget makes of src[j * 32])
            const uint32_t a_begin = smem_u32(&sm.ring[slot][0][lane_now()]), a_end = a_begin + CHUNK * 128u;
#pragma unroll P_UNROLL
            for (uint32_t a = a_begin; a != a_end; a += 128u) {
                const uint32_t code = (uint32_t)lds32(a);
                const int32_t r = code_to_residual(code);
                int32_t top;
                if (T == 8) top = sel4 ? h[4] : sel5 ? h[5] : sel6 ? h[6] : h[8];
                else top = sel4 ? h[4] : sel5 ? h[5] : h[6];
                int32_t d[T];
                int32_t sum = den_half;
                int32_t sum_b = 0;  // two accumulators: the dependent IMAD chain of the FIR is half as long (wrap-around sums commute)
#pragma unroll
                for (int t = 0; t < T; t++) {
                    d[t] = top - h[t];
                    if (t >= 4) d[t] &= (int32_t)tmask[t];  // orders start at 4: taps 0..3 always live
                    if (t & 1) sum_b -= c[t] * d[t];
                    else sum -= c[t] * d[t];
                }
                sum += sum_b;
                const int32_t x = sext_bits(r + top + (sum >> den), jb.chan_bits);
                const int32_t smask = r >> 31;                       // 0 / -1
                const int32_t nsone = -(smask | 1);                  // -1 for r > 0, +1 for r < 0: coef -= sign(diff) * sign(r)
                const uint32_t bias = (uint32_t)smask & den_mask;    // round |diff| >> den up for r < 0
                const int32_t thr = smask + 1;
                int32_t E = r ^ smask;
                bool alive = r != 0;
#pragma unroll
                for (int t = T - 1; t >= 0; t--) {
                    const int32_t sg = max(min(d[t], 1), -1);        // signOfInt
                    mad_if(c[t], sg, nsone, alive);
                    if (t > 0) {
                        const uint32_t q = ((uint32_t)(sg * d[t]) + bias) >> den;  // |diff| < 2^31: no wrap
                        E += nwgt[t] * (int32_t)q;
                        alive = alive && (E >= thr);                 // masked taps: q = 0, E unchanged
                    }
                }
#pragma unroll
                for (int t = T; t > 0; t--) h[t] = h[t - 1];
                h[0] = x;
                sts32(a, x);
            }
            asm volatile("" ::: "memory");  // the slot is re-read through vdst below
        }
        slot_end(ck, slot);
    }
}

// Any mix of orders in the warp, including the int16-wrapping ones: unpcBlockGeneral, predictor.go:623-684,
// with per-lane coefficient width (int32 kept for 4/5/6/8 as the reference's specialised loops do).
__device__ __noinline__ void stream_generic(DecShared &sm, uint32_t lane, uint32_t &seq, const Packet &pk,
                                            const Job &jb, bool active, int32_t *__restrict__ dst, RoleTimer &rt) {
    const uint32_t cs = 32u - jb.chan_bits;
    const uint32_t den = jb.den;
    const int32_t den_half = den > 0 ? (int32_t)(1u << (den - 1)) : 0;
    const int32_t order = (int32_t)jb.order;
    const bool wrap16 = jb.kind == JOB_GENERIC;
    const bool mode = jb.mode != 0;
    int32_t coef[32];
    int32_t hist[32];  // ring: out[i] at hist[i & 31]
#pragma unroll 1
    for (int k = 0; k < 32; k++) {
        coef[k] = (active && k < order && order != 31) ? (int32_t)(int16_t)pk_bits(pk, jb.coef_bitpos + 16u * (uint32_t)k, 16) : 0;
        hist[k] = 0;
    }
    int32_t dprev = 0;
    const uint32_t nchunks = max(1u, (jb.nmax + CHUNK - 1) / CHUNK);
#pragma unroll 1
    for (uint32_t ck = 0; ck < nchunks; ck++) {
        const uint32_t slot = seq % RING_SLOTS;
        if (ck > 0) {
            const unsigned long long tw = rt.now();
            wait_full(sm, seq);
            rt.add(1, tw);
        }
        const int32_t *src = &sm.ring[slot][0][lane];
#pragma unroll 1
        for (uint32_t j = 0; j < CHUNK; j++) {
            const uint32_t i = ck * CHUNK + j;
            int32_t r = code_to_residual((uint32_t)src[j * 32]);
            if (active && i < jb.n) {
                r = delta_step(mode, dprev, r, i, cs);
                int32_t x;
                if (i == 0 || order == 0) x = r;
                else if (order == 31 || (int32_t)i <= order) x = sext_go(r + hist[(i - 1) & 31u], cs);
                else {
                    const int32_t top = hist[(i - (uint32_t)order - 1u) & 31u];
                    int32_t sum1 = 0;
#pragma unroll 1
                    for (int32_t k = 0; k < order; k++) sum1 += coef[k] * (hist[(i - 1u - (uint32_t)k) & 31u] - top);
                    x = sext_go(r + top + ((sum1 + den_half) >> den), cs);
                    int32_t del0 = r;
                    if (r != 0) {
                        const int32_t s = r > 0 ? 1 : -1;
#pragma unroll 1
                        for (int32_t k = order - 1; k >= 0; k--) {
                            const int32_t dd = top - hist[(i - 1u - (uint32_t)k) & 31u];
                            const int32_t sgn = s * sign_of(dd);
                            int32_t nc = coef[k] - sgn;
                            if (wrap16) nc = (int32_t)(int16_t)nc;
                            coef[k] = nc;
                            del0 -= (order - k) * ((sgn * dd) >> den);
                            if (s > 0 ? del0 <= 0 : del0 >= 0) break;
                        }
                    }
                }
                hist[i & 31u] = x;
                dst[(size_t)i * 32u] = x;
            }
        }
        arrive_empty(sm, seq);
        seq++;
    }
}

// The two halves of an interleaved escape pair (decoder.go:513-533) arrive in alternating ring slots; the raw samples are
// only parked (order 0, no pre-pass). The first slot (first half, chunk 0) is already full.
__device__ __forceinline__ void stream_escape_pair(DecShared &sm, uint32_t lane, uint32_t &seq, const Job &j0, bool act0,
                                                   int32_t *__restrict__ dst0, bool valid, const DevConfig &cfg,
                                                   int32_t *__restrict__ scratch_lane, RoleTimer &rt) {
    const uint32_t nchunks = max(1u, (j0.nmax + CHUNK - 1) / CHUNK);
    const uint32_t n0 = act0 ? j0.n : 0u;
    uint32_t n1 = 0;
    int32_t *dst1 = scratch_lane;
#pragma unroll 1
    for (uint32_t ck = 0; ck < nchunks; ck++) {
#pragma unroll 1
        for (uint32_t half = 0; half < 2; half++) {
            const uint32_t slot = seq % RING_SLOTS;
            if (ck > 0 || half > 0) {
                const unsigned long long tw = rt.now();
                wait_full(sm, seq);
                rt.add(1, tw);
            }
            if (ck == 0 && half == 1) {  // the job of the pair's second half
                const uint32_t meta = sm.job[slot][1][lane];
                const bool act1 = valid && (meta & 3u) != JOB_INACTIVE;
                n1 = act1 ? sm.job[slot][0][lane] : 0u;
                dst1 = scratch_lane + (size_t)((meta >> 18) & 7u) * cfg.frame_length * 32u;
            }
            const int32_t *src = &sm.ring[slot][0][lane];
            const uint32_t nn = half ? n1 : n0;
            int32_t *dd = half ? dst1 : dst0;
#pragma unroll 4
            for (uint32_t j = 0; j < CHUNK; j++) {
                const uint32_t i = ck * CHUNK + j;
                if (i < nn) dd[(size_t)i * 32u] = code_to_residual((uint32_t)src[j * 32]);
            }
            arrive_empty(sm, seq);
            seq++;
        }
    }
}

// The first slot of the next stream is full: read its job. Returns the meta word.
__device__ __forceinline__ uint32_t read_job(DecShared &sm, uint32_t slot, uint32_t lane, Job &jb) {
    jb.n = sm.job[slot][0][lane];
    const uint32_t meta = sm.job[slot][1][lane];
    jb.coef_bitpos = sm.job[slot][2][lane];
    jb.nmax = __shfl_sync(FULL_MASK, sm.job[slot][3][lane], 0);
    jb.live = sm.job[slot][4][lane];
    jb.shift_bitpos = sm.job[slot][5][lane];
    jb.kind = meta & 3u;
    jb.order = (meta >> 2) & 31u;
    jb.den = (meta >> 7) & 15u;
    jb.mode = (meta >> 11) & 1u;
    jb.chan_bits = (meta >> 12) & 63u;
    jb.slot = (meta >> 18) & 7u;
    return meta;
}

// One stream, by the loop that fits the orders / modes the warp's lanes carry.
__device__ __forceinline__ void run_stream(DecShared &sm, uint32_t lane, uint32_t &seq, const Packet &pk, const Job &jb,
                                           bool active, int32_t *__restrict__ dst, RoleTimer &rt, const LiveEnv &lc,
                                           const DevConfig &cfg) {
    const bool any_generic = __any_sync(FULL_MASK, active && jb.kind == JOB_GENERIC);
    const bool any8 = __any_sync(FULL_MASK, active && jb.order == 8);
    const bool any_mode = __any_sync(FULL_MASK, active && jb.mode != 0);
    // live emission (2-channel streams, V): decided per stream by the entropy warp, uniform over the warp (it only
    // marks pairs whose orders the register loops take, so a live stream never goes to stream_generic)
    const bool live_lane = active && (jb.live >> 31) != 0u;
    const bool live = lc.enabled && !any_generic && __any_sync(FULL_MASK, live_lane);
    if (live) {
        sm.live_ctx[0][lane] = live_lane ? jb.n : 0u;
        sm.live_ctx[1][lane] = live_lane ? (jb.live | ((uint32_t)((uintptr_t)pk.p & 15u) << 18)) : 0u;  // bit 31: this lane is live
        sm.live_ctx[2][lane] = jb.shift_bitpos;
        // the U samples of this pair were parked by this warp's own lanes: order them before the cooperative fetches
        __threadfence_block();
        __syncwarp();
    }
    if (any_generic) stream_generic(sm, lane, seq, pk, jb, active, dst, rt);
    else if (any_mode) {  // rare: the order-31 pre-pass is on for some lane
        if (any8) stream_reg<8, true>(sm, lane, seq, pk, jb, active, rt, lc, live);
        else stream_reg<6, true>(sm, lane, seq, pk, jb, active, rt, lc, live);
    } else if (any8) stream_reg<8, false>(sm, lane, seq, pk, jb, active, rt, lc, live);
    else stream_reg<6, false>(sm, lane, seq, pk, jb, active, rt, lc, live);
    if (live && live_lane)
        (lc.descs + (size_t)cta_now() * 32u + lane_now())->pad_ = max(1u, (jb.nmax + CHUNK - 1) / CHUNK) * CHUNK;  // frames written so far (zeros past the sample count)
}

// PREDICTOR warp, one group of 32 packets: every stream the entropy warp produces, in order, until the group's end
// marker. `seq` lives across the groups of the CTA.
__device__ __forceinline__ void predictor_warp(DecShared &sm, uint32_t lane, const uint8_t *__restrict__ packed,
                                               const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ sizes,
                                               uint32_t npackets, const DevConfig &cfg, PacketDesc *__restrict__ descs_all,
                                               uint8_t *__restrict__ pcm_out, uint64_t out_stride, uint32_t group,
                                               uint32_t &seq, const int32_t *__restrict__ scratch_all) {
    const uint32_t pidx = group * 32u + lane;
    const bool valid = pidx < npackets;
    Packet pk{packed, 0};
    if (valid) pk = Packet{packed + offsets[pidx], sizes[pidx]};
    LiveEnv lc;
    lc.scratch = scratch_all;  // the kernel parameters: this CTA's parts are rebuilt where they are needed
    lc.descs = descs_all;
    lc.num_channels = cfg.num_channels;
    lc.pcm_out = pcm_out;
    lc.out_stride = out_stride;
    lc.frame_length = cfg.frame_length;
    lc.bps = cfg.bps;
    lc.bit_depth = cfg.bit_depth;
    lc.enabled = cfg.num_channels == 2u;
    RoleTimer rt(lane, 3);
    const unsigned long long t_start = rt.now();
#pragma unroll 1
    for (;;) {
        const uint32_t slot = seq % RING_SLOTS;
        const unsigned long long tw = rt.now();
        wait_full(sm, seq);
        rt.add(1, tw);
        Job jb;
        const uint32_t meta = read_job(sm, slot, lane, jb);
        if (jb.kind == JOB_EXIT) {  // written for every lane: the group is finished
            arrive_empty(sm, seq);
            seq++;
            break;
        }
        const bool active = valid && jb.kind != JOB_INACTIVE;
        int32_t *scratch_lane = const_cast<int32_t *>(cta_scratch(lc)) + lane_now();  // the CTA's own scratch, [slot][sample][lane]
        int32_t *dst = scratch_lane + (size_t)jb.slot * cfg.frame_length * 32u;
        if (meta & JOBF_PAIR) stream_escape_pair(sm, lane, seq, jb, active, dst, valid, cfg, scratch_lane, rt);
        else run_stream(sm, lane, seq, pk, jb, active, dst, rt, lc, cfg);
    }
    rt.add(0, t_start);
    rt.flush(3);
}

// ---- stage 3 ---------------------------------------------------------------------------------------
// WriteStereo16/20/24/32 + WriteMono16/20/24/32 (matrix.go:30-301) for the 32 packets of one group, run by
// the whole CTA once its role warps are done. Lane = packet reads the parked samples coalesced, un-mixes,
// merges the shift bytes, writes the little-endian bytes into a shared-memory tile (odd word stride:
// conflict-free transpose); then each warp flushes packet rows with 128-bit stores. The element ops are
// replayed in element order with a barrier in between, so later elements overwrite earlier ones exactly as
// the sequential reference does (a pair mapped onto the last channel spills into the next frame,
// matrix.go:44-48). Bytes past output[:n] (decoder.go:127) and failed packets are written as zeros.
struct EmitArgs {
    const uint8_t *packed;
    const uint64_t *offsets;
    const uint32_t *sizes;
    uint32_t npackets;
    const int32_t *scratch;   // the CTA's own parked samples, [slot][sample][lane]
    const PacketDesc *descs;  // the CTA's own 32 descriptors
    uint8_t *pcm_out;
    uint64_t out_stride;
};

__device__ __forceinline__ void tile_put(uint8_t *row, int32_t lo_byte, int32_t hi_byte, int32_t off, int32_t v, int bps) {
    // store the bps little-endian bytes of v at packet byte offset `off`, clipped to the tile [lo_byte, hi_byte)
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (k < bps) {
            int32_t o = off + k;
            if (o >= lo_byte && o < hi_byte) row[o - lo_byte] = (uint8_t)((uint32_t)v >> (8 * k));
        }
    }
}

// the little-endian bytes of one mono sample / one stereo pair into the transpose tile, widest aligned stores
template <int BPS>
__device__ __forceinline__ void tile_store(uint8_t *dst, int32_t left, int32_t right, bool stereo) {
    const uint64_t lmask = BPS == 4 ? 0xffffffffull : ((1ull << (8 * BPS)) - 1ull);
    uint64_t v = (uint64_t)(uint32_t)left & lmask;
    if (stereo) v |= ((uint64_t)(uint32_t)right & lmask) << (8 * BPS);
    const uint32_t nbytes = stereo ? 2u * BPS : (uint32_t)BPS;
    const uint32_t a = (uint32_t)(uintptr_t)dst;
    if ((a & 3u) == 0 && nbytes == 4u) {
        *reinterpret_cast<uint32_t *>(dst) = (uint32_t)v;
    } else if ((a & 3u) == 0 && nbytes == 8u) {
        *reinterpret_cast<uint32_t *>(dst) = (uint32_t)v;
        *reinterpret_cast<uint32_t *>(dst + 4) = (uint32_t)(v >> 32);
    } else if ((a & 1u) == 0 && (nbytes & 1u) == 0) {
#pragma unroll
        for (int k = 0; k < BPS; k++)
            if (2u * (uint32_t)k < nbytes) *reinterpret_cast<uint16_t *>(dst + 2 * k) = (uint16_t)(v >> (16 * k));
    } else {
#pragma unroll
        for (int k = 0; k < 2 * BPS; k++)
            if ((uint32_t)k < nbytes) dst[k] = (uint8_t)(v >> (8 * k));
    }
}

struct EmitOp {
    const int32_t *su, *sv;
    int32_t i_lo, i_hi, s0, mix_res;
    uint32_t mix_bits, sb, rel0, width, fb, out_off;
    bool stereo, depth20;
};

// frames [i_lo, i_hi) of one element, all inside the tile: batched parked-sample loads, un-mix, shift merge, store
template <int BPS>
__device__ __forceinline__ void emit_frames(const EmitOp &o, uint8_t *row, const uint32_t *shrow_words) {
    constexpr int EB = 8;  // frames per batch: all parked-sample loads of a batch are issued together
#pragma unroll 1
    for (int32_t ib = o.i_lo; ib < o.i_hi; ib += EB) {
        int32_t lu[EB], lv[EB];
#pragma unroll
        for (int q = 0; q < EB; q++) {
            const int32_t i = min(ib + q, o.i_hi - 1);
            lu[q] = __ldcs(o.su + (size_t)i * 32u);  // parked samples are read exactly once
            lv[q] = __ldcs(o.sv + (size_t)i * 32u);
        }
#pragma unroll
        for (int q = 0; q < EB; q++) {
            const int32_t i = ib + q;
            if (i < o.i_hi) {
                int32_t left = lu[q], right = o.stereo ? lv[q] : 0;
                writer_frame(left, right, o.stereo, o.mix_res, o.mix_bits, o.depth20, o.sb, shrow_words,
                             o.rel0 + (uint32_t)(i - o.i_lo) * o.width * o.sb);
                tile_store<BPS>(row + (uint32_t)(i - o.s0) * o.fb + o.out_off, left, right, o.stereo);
            }
        }
    }
}

// ---- stage 3, direct path: the element covers the whole frame (mono in a 1-channel stream, a pair in a
// 2-channel stream). Each lane then owns contiguous output: 16 frames are un-mixed, shift-merged and packed into
// registers and leave as FB 128-bit stores to the lane's own packet slot -- no transpose tile, no barrier. All
// parked-sample and shift-word loads of a batch are issued together (32 + ~10 per lane) so that the sixteen warps of an SM
// keep enough bytes in flight. Frames past the element's sample count are written as zeros (decoder.go:120, :127).
template <int BPS, int WIDTH>
__device__ __forceinline__ void emit_direct(const EmitArgs &x, const DevConfig &cfg, uint32_t group, uint8_t *smem,
                                            bool valid, const Packet &pk, const OpDesc &op, uint32_t n_final,
                                            uint32_t first_frame) {
    constexpr int FB = BPS * WIDTH;  // bytes per frame
    constexpr int EB = 16;           // frames per batch: 16*FB bytes = FB 128-bit stores
    constexpr uint32_t SROW = 21;    // shift words staged per lane and batch: 16 frames x 2 x 2 bytes + window + slack, odd
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    constexpr uint32_t NW = DEC_WARPS;
    uint32_t *myrow = reinterpret_cast<uint32_t *>(smem) + ((size_t)warp * 32u + lane) * SROW;
    const uint32_t pidx = group * 32u + lane;
    const bool stereo = WIDTH == 2;
    const bool depth20 = cfg.bit_depth == 20;
    const bool merges_shift = cfg.bit_depth == 24 || cfg.bit_depth == 32;
    const uint32_t sb = (merges_shift ? (uint32_t)op.shift : 0u) * 8u;
    const uint32_t n_op = min(op.n, n_final);  // output[:n] cuts what an earlier, longer element wrote
    const int32_t *su = x.scratch + lane;
    const int32_t *sv = stereo ? su + (size_t)cfg.frame_length * 32u : su;
    uint8_t *slot = x.pcm_out + (size_t)pidx * x.out_stride;
    const bool vec_ok = ((((uintptr_t)x.pcm_out) | x.out_stride) & 15u) == 0;
    const uint32_t nbatches = (cfg.frame_length + EB - 1) / EB;
    const int32_t mix_res = op.mix_res;
    const uint32_t mix_bits = op.mix_bits;
#pragma unroll 1
    for (uint32_t b = warp; b < nbatches; b += NW) {
        const uint32_t f0 = b * EB;
        const uint32_t cnt = n_op > f0 ? min((uint32_t)EB, n_op - f0) : 0u;
        // ---- issue every load of the batch -----------------------------------------------------------------
        int32_t lu[EB], lv[EB];
        const uint32_t last = n_op > 0 ? n_op - 1u : 0u;
#pragma unroll
        for (int q = 0; q < EB; q++) {
            const uint32_t i = min(f0 + (uint32_t)q, last);
            lu[q] = __ldcs(su + (size_t)i * 32u);
            lv[q] = __ldcs(sv + (size_t)i * 32u);
        }
        uint32_t rel0 = 0;
        if (sb && cnt) {
            const uint32_t first_bit = op.shift_bitpos + f0 * WIDTH * sb;
            const uint32_t nbits = cnt * WIDTH * sb;
            const uint32_t byte0 = first_bit >> 3;
            const uint32_t nbytes = ((first_bit & 7u) + nbits + 7u) / 8u + 2u;  // +2: the 24-bit window of BitBuffer.Read
            const uintptr_t ga = ((uintptr_t)(pk.p + byte0)) & ~(uintptr_t)3;
            const uint32_t lead_bytes = (uint32_t)((uintptr_t)(pk.p + byte0) - ga);
            const int64_t rel_pk = (int64_t)byte0 - (int64_t)lead_bytes;
            const uint32_t nw = (lead_bytes + nbytes + 3u) / 4u;  // <= 18
            const uint32_t *gsrc = reinterpret_cast<const uint32_t *>(ga);
            uint32_t wbuf[SROW - 2];
#pragma unroll
            for (uint32_t k = 0; k < SROW - 2; k++) wbuf[k] = k < nw ? shift_word(pk, rel_pk, k, gsrc) : 0u;
#pragma unroll
            for (uint32_t k = 0; k < SROW - 2; k++) myrow[k] = wbuf[k];
            myrow[SROW - 2] = 0;
            myrow[SROW - 1] = 0;
            rel0 = lead_bytes * 8u + (first_bit & 7u);
        }
        // ---- un-mix, merge, pack ------------------------------------------------------------------------------
        uint32_t ow[4 * FB];
#pragma unroll
        for (int k = 0; k < 4 * FB; k++) ow[k] = 0;
#pragma unroll
        for (int q = 0; q < EB; q++) {
            int32_t left = lu[q], right = stereo ? lv[q] : 0;
            writer_frame(left, right, stereo, mix_res, mix_bits, depth20, sb, myrow, rel0 + (uint32_t)q * WIDTH * sb);
            pack_frame<BPS, WIDTH>(ow, q, left, right, (uint32_t)q < cnt);
        }
        // ---- store: FB x 16 bytes to the lane's own packet slot ---------------------------------------------------
        if (valid && f0 >= first_frame)  // frames below first_frame were emitted live by the predictor warp
            store_words<FB, EB>(slot, f0, FB, cfg.frame_length, vec_ok, ow);
    }
}

// ---- stage 3, row path: canonical multi-element packets (every element as long as the packet, the elements cover
// every channel once, nothing spills). No transpose: each lane builds FR frames of ITS packet in a private shared-memory
// row (element after element: batched parked-sample loads, un-mix, shift merge, byte placement at the element's
// channel offset) and stores the row to its own packet slot with 128-bit stores. Frames past the packet's sample count
// are written as zeros (decoder.go:120, :127). Two warps x 32 lanes x 16 parked-sample loads in flight per element and CTA
// keep enough bytes in flight for the copy to be bandwidth- rather than latency-bound.
// 32-bit words of shift data staged per lane and element: FR frames x 2 channels x 2 bytes + the 24-bit window of
// BitBuffer.Read, fetched as whole 16-byte pieces
__host__ __device__ constexpr uint32_t row_shift_words(uint32_t fr) { return ((fr * 4u + 2u + 15u + 15u) / 16u) * 4u; }

template <int BPS, int FR, int NWARPS>
__device__ __forceinline__ void emit_rows(const EmitArgs &x, const DevConfig &cfg, uint32_t group, uint8_t *smem, bool valid,
                                          const Packet &pk, const PacketDesc *desc, uint32_t nops, uint32_t n_final,
                                          uint32_t max_ops) {
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t fb = cfg.num_channels * BPS;            // bytes per frame
    const uint32_t row_words = ((FR * fb) / 4u) | 1u;      // FR * fb is a multiple of 16; odd stride: conflict-free rows
    constexpr uint32_t SHIFT_WORDS = row_shift_words(FR);
    constexpr uint32_t SHIFT_ROW = SHIFT_WORDS | 1u;
    uint32_t *wbase = reinterpret_cast<uint32_t *>(smem) + (size_t)warp * 32u * (row_words + SHIFT_ROW);
    uint32_t *roww = wbase + (size_t)lane * row_words;
    uint8_t *row = reinterpret_cast<uint8_t *>(roww);
    uint32_t *shrow = wbase + 32u * row_words + (size_t)lane * SHIFT_ROW;
    const uint32_t pidx = group * 32u + lane;
    const int32_t *sbase = x.scratch + lane;
    uint8_t *slot = x.pcm_out + (size_t)pidx * x.out_stride;
    const bool depth20 = cfg.bit_depth == 20;
    const bool merges_shift = cfg.bit_depth == 24 || cfg.bit_depth == 32;  // 16/20-bit writers ignore the shift buffer
    const uint32_t nbatches = cfg.frame_length / FR;
    const uint32_t nvec = (FR * fb) / 16u;
#pragma unroll 1
    for (uint32_t b = warp; b < nbatches; b += NWARPS) {
        const uint32_t f0 = b * FR;
#pragma unroll 1
        for (uint32_t e = 0; e < max_ops; e++) {
            if (e < nops) {
                const OpDesc op = desc->ops[e];
                const bool stereo = op.kind == 2;
                const uint32_t width = stereo ? 2u : 1u;
                const uint32_t sb = (merges_shift ? (uint32_t)op.shift : 0u) * 8u;
                const uint32_t cnt = op.n > f0 ? min((uint32_t)FR, op.n - f0) : 0u;
                // ---- every load of this element's FR frames is issued before anything waits: parked samples ...
                const int32_t *su = sbase + (size_t)op.slot * cfg.frame_length * 32u;
                const int32_t *sv = stereo ? su + (size_t)cfg.frame_length * 32u : su;
                const uint32_t last = op.n > 0 ? op.n - 1u : 0u;
                int32_t lu[FR], lv[FR];
#pragma unroll
                for (int q = 0; q < FR; q++) {
                    const uint32_t i = min(f0 + (uint32_t)q, last);
                    lu[q] = __ldcs(su + (size_t)i * 32u);  // parked samples are read exactly once
                    lv[q] = __ldcs(sv + (size_t)i * 32u);
                }
                // ... and the shift bytes of these frames (zeros at or past the packet end, bitbuffer.go:36-51)
                uint32_t rel0 = 0;
                if (sb && cnt) {
                    const uint32_t first_bit = op.shift_bitpos + f0 * width * sb;
                    const uint32_t nbits = cnt * width * sb;
                    const uint32_t byte0 = first_bit >> 3;
                    const uint32_t nbytes = ((first_bit & 7u) + nbits + 7u) / 8u + 2u;  // +2: the 24-bit window of BitBuffer.Read
                    const uintptr_t ga = ((uintptr_t)(pk.p + byte0)) & ~(uintptr_t)15;  // 16-byte pieces: few requests per lane
                    const uint32_t lead_bytes = (uint32_t)((uintptr_t)(pk.p + byte0) - ga);
                    const int64_t rel_pk = (int64_t)byte0 - (int64_t)lead_bytes;
                    const uint32_t nw = (lead_bytes + nbytes + 3u) / 4u;  // <= SHIFT_WORDS - 2
                    uint32_t wbuf[SHIFT_WORDS];
                    if (rel_pk >= 0 && rel_pk + 4 * (int64_t)SHIFT_WORDS <= (int64_t)pk.size) {  // the whole window lies inside the packet
                        const uint4 *g4 = reinterpret_cast<const uint4 *>(ga);
#pragma unroll
                        for (uint32_t k = 0; k < SHIFT_WORDS / 4; k++) {
                            const uint4 v = __ldg(g4 + k);
                            wbuf[4 * k] = v.x; wbuf[4 * k + 1] = v.y; wbuf[4 * k + 2] = v.z; wbuf[4 * k + 3] = v.w;
                        }
                    } else {
                        const uint32_t *gsrc = reinterpret_cast<const uint32_t *>(ga);
#pragma unroll 1
                        for (uint32_t k = 0; k < SHIFT_WORDS; k++) shrow[k] = k < nw ? shift_word(pk, rel_pk, k, gsrc) : 0u;
#pragma unroll
                        for (uint32_t k = 0; k < SHIFT_WORDS; k++) wbuf[k] = shrow[k];
                    }
#pragma unroll
                    for (uint32_t k = 0; k < SHIFT_WORDS; k++) shrow[k] = wbuf[k];
                    rel0 = lead_bytes * 8u + (first_bit & 7u);
                }
                // ---- un-mix, merge, place the bytes at the element's channel offset of every frame ----
                const int32_t mix_res = op.mix_res;
                const uint32_t mix_bits = op.mix_bits;
                uint8_t *dstb = row + (uint32_t)op.out_chan * BPS;
#pragma unroll
                for (int q = 0; q < FR; q++) {
                    if ((uint32_t)q < cnt) {
                        int32_t left = lu[q], right = stereo ? lv[q] : 0;
                        writer_frame(left, right, stereo, mix_res, mix_bits, depth20, sb, shrow, rel0 + (uint32_t)q * width * sb);
                        tile_store<BPS>(dstb + (uint32_t)q * fb, left, right, stereo);
                    }
                }
            }
        }
        // the lane's own row -> its packet slot; bytes at or past n_final frames are zeros, and so is a packet
        // without any element (END first, or failed)
        const uint32_t n_rows = nops ? n_final : 0u;
        const uint32_t nvalid = n_rows > f0 ? min((n_rows - f0) * fb, FR * fb) : 0u;
        if (valid) {
            uint4 *dst = reinterpret_cast<uint4 *>(slot + (size_t)f0 * fb);
#pragma unroll 4
            for (uint32_t k = 0; k < nvec; k++) {
                uint32_t w[4];
#pragma unroll
                for (uint32_t j = 0; j < 4; j++) {
                    const uint32_t byte = (4u * k + j) * 4u;
                    uint32_t v = roww[4u * k + j];
                    if (byte + 4u > nvalid) v = byte >= nvalid ? 0u : v & (0xffffffffu >> (8u * (byte + 4u - nvalid)));
                    w[j] = v;
                }
                dst[k] = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
}

// ---- stage 3, packed row path: the shapes real multi-channel files have -- canonical packets of full-length elements,
// 16-bit, or 24-bit with zero or one shifted byte per element, every shift byte inside the packet. Like emit_rows each lane
// builds FR frames of ITS packet in a private shared-memory row, but one 32-bit word per sample: the element pass is
// loads (parked samples + five words of shift bytes), un-mix, ONE byte permute per sample for `(x << 8) | shift byte`
// (matrix.go:132-135, :270-272) and one STS; the flush packs 16 samples into 3 (24-bit) or 2 (16-bit) 128-bit stores with
// byte permutes. ~10 instructions per sample instead of ~50 (profiles/r02c_c4: the tail was 22 % of the 7.1 workload's
// instructions and 43 % of its stall samples).
template <int BPS, int FR, int NWARPS>
__device__ __forceinline__ void emit_rows_packed(const EmitArgs &x, const DevConfig &cfg, uint32_t group, uint8_t *smem,
                                                 bool valid, const Packet &pk, const PacketDesc *desc, uint32_t nops,
                                                 uint32_t max_ops) {
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t nch = cfg.num_channels;
    const uint32_t fb = nch * BPS;
    const uint32_t row_words = (FR * nch) | 1u;  // odd stride: the lanes' rows are conflict-free
    uint32_t *roww = reinterpret_cast<uint32_t *>(smem) + ((size_t)warp * 32u + lane) * row_words;
    const uint32_t pidx = group * 32u + lane;
    const int32_t *sbase = x.scratch + lane;
    uint8_t *slot = x.pcm_out + (size_t)pidx * x.out_stride;
    const uint32_t nbatches = cfg.frame_length / FR;
    const uint32_t ngroups16 = (FR * nch) / 16u;  // 16 samples -> BPS 128-bit stores
#pragma unroll 1
    for (uint32_t b = warp; b < nbatches; b += NWARPS) {
        const uint32_t f0 = b * FR;
#pragma unroll 1
        for (uint32_t e = 0; e < max_ops; e++) {
            if (e < nops) {
                const OpDesc op = desc->ops[e];
                const bool stereo = op.kind == 2;
                const uint32_t width = stereo ? 2u : 1u;
                const bool merge = BPS == 3 && op.shift != 0;
                const int32_t *su = sbase + ((size_t)op.slot * cfg.frame_length + f0) * 32u;
                const int32_t *sv = su + (size_t)cfg.frame_length * 32u;
                int32_t lu[FR], lv[FR];
#pragma unroll
                for (int q = 0; q < FR; q++) lu[q] = __ldcs(su + (size_t)q * 32u);  // parked samples are read exactly once
#pragma unroll
                for (int q = 0; q < FR; q++) lv[q] = stereo ? __ldcs(sv + (size_t)q * 32u) : 0;
                // FR x width shift bytes from bit `first_bit` of the packet: aligned words, big-endian, one funnel shift each
                constexpr int NS = FR / 2;  // 32-bit windows a stereo element needs (two frames each); a mono one needs FR / 4
                uint32_t S[NS];
#pragma unroll
                for (int k = 0; k < NS; k++) S[k] = 0;
                if (merge) {
                    const uint32_t first_bit = op.shift_bitpos + f0 * width * 8u;
                    const uint8_t *g0 = pk.p + (first_bit >> 3);
                    const uint32_t *ga = reinterpret_cast<const uint32_t *>(((uintptr_t)g0) & ~(uintptr_t)3);
                    const uint32_t bo = (uint32_t)(((uintptr_t)g0) & 3u) * 8u + (first_bit & 7u);
                    uint32_t W[NS + 1];
#pragma unroll
                    for (int k = 0; k <= NS; k++) W[k] = (stereo || k <= NS / 2) ? __byte_perm(__ldg(ga + k), 0, 0x0123) : 0u;
#pragma unroll
                    for (int k = 0; k < NS; k++) S[k] = __funnelshift_l(W[k + 1], W[k], bo);
                }
                const int32_t mix_res = op.mix_res;
                const uint32_t mix_bits = op.mix_bits;
                uint32_t *dstw = roww + op.out_chan;
#pragma unroll
                for (int q = 0; q < FR; q++) {
                    int32_t left = lu[q], right = lv[q];
                    if (stereo) unmix(lu[q], lv[q], mix_res, mix_bits, left, right);
                    uint32_t xl = (uint32_t)left, xr = (uint32_t)right;
                    if (BPS == 3) {
                        // (x << 8) | shift byte: a pair's bytes sit L R L R in its windows, a mono element's four to a window
                        const uint32_t ws = S[q >> 1], wm = S[q >> 2];
                        const uint32_t ml = __byte_perm(stereo ? ws : wm, xl, stereo ? ((q & 1) ? 0x6541 : 0x6543) : 0x6540 + (3 - (q & 3)));
                        const uint32_t mr = __byte_perm(ws, xr, (q & 1) ? 0x6540 : 0x6542);
                        xl = merge ? ml : xl;
                        xr = merge ? mr : xr;
                    }
                    dstw[q * nch] = xl;
                    if (stereo) dstw[q * nch + 1u] = xr;
                }
            }
        }
        // the lane's row -> its packet slot
        if (valid) {
            uint4 *dst = reinterpret_cast<uint4 *>(slot + (size_t)f0 * fb);
#pragma unroll 1
            for (uint32_t g = 0; g < ngroups16; g++) {
                uint32_t v[16];
#pragma unroll
                for (int k = 0; k < 16; k++) v[k] = roww[g * 16u + k];
                if (BPS == 3) {
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t w0 = __byte_perm(v[4 * k], v[4 * k + 1], 0x4210);
                        const uint32_t w1 = __byte_perm(v[4 * k + 1], v[4 * k + 2], 0x5421);
                        const uint32_t w2 = __byte_perm(v[4 * k + 2], v[4 * k + 3], 0x6542);
                        v[3 * k] = w0; v[3 * k + 1] = w1; v[3 * k + 2] = w2;  // 3k+2 < 4(k+1): nothing unread is overwritten
                    }
#pragma unroll
                    for (int k = 0; k < 3; k++) dst[g * 3u + k] = make_uint4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
                } else {
#pragma unroll
                    for (int k = 0; k < 8; k++) v[k] = __byte_perm(v[2 * k], v[2 * k + 1], 0x5410);
#pragma unroll
                    for (int k = 0; k < 2; k++) dst[g * 2u + k] = make_uint4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
                }
            }
        }
    }
}

// Stage 3 runs warp-local: every warp owns a transpose tile of 32 packet rows x TL frames (+ a staging row for
// the shift bytes) inside the shared memory the decode stage leaves behind, and walks the tiles w, w+NWARPS, ...
// of the group on its own -- no block barrier, one tile in flight per warp.
__host__ __device__ inline uint32_t emit_tile_frames(uint32_t frame_bytes, uint32_t nwarps, uint32_t smem_bytes) {
    // per packet row: TL*fb + 4 bytes of tile (odd word stride) and 4*TL + 12 bytes of shift staging
    // (TL frames x 2 channels x 2 shift bytes, + the 24-bit window of BitBuffer.Read, odd word stride)
    const uint32_t per_row = smem_bytes / (nwarps * 32u);
    uint32_t tl = (per_row - 28u) / (frame_bytes + 4u);
    tl = tl > 64u ? 64u : tl;
    return tl >= 16u ? (tl & ~15u) : (tl & ~3u);  // keep TL*fb a multiple of 16 where possible (128-bit stores)
}

// Inlined into decode_cta: an out-of-line tail was measured and made no difference.
template <int NWARPS>
__device__ __forceinline__ void emit_group(const EmitArgs &x, const DevConfig &cfg, uint32_t group, uint8_t *smem,
                                           uint32_t smem_bytes) {
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t fb = cfg.num_channels * cfg.bps;  // bytes per frame
    const uint32_t TL = emit_tile_frames(fb, NWARPS, smem_bytes);
    const uint32_t row_words = (TL * fb) / 4u + 1u;  // odd => conflict-free lane-per-row access
    const uint32_t EMIT_SHIFT_ROW_WORDS = TL + 5u;   // TL is a multiple of 4: odd; +2 words so a 64-bit window never runs off
    const uint32_t warp_words = 32u * (row_words + EMIT_SHIFT_ROW_WORDS);
    uint32_t *sw = reinterpret_cast<uint32_t *>(smem) + (size_t)warp * warp_words;  // this warp's tile
    uint32_t *shw = sw + 32u * row_words;                                             // this warp's shift rows
    const uint32_t pidx = group * 32u + lane;
    const bool valid = pidx < x.npackets;
    const PacketDesc *desc = x.descs + lane;
    int32_t st = ST_REF_PANIC;
    uint32_t nops = 0, n_final = 0;
    Packet pk{x.packed, 0};
    if (valid) {
        st = desc->status;
        nops = st == ST_OK ? desc->nops : 0;
        n_final = st == ST_OK ? desc->n_final : 0;
        pk = Packet{x.packed + x.offsets[pidx], x.sizes[pidx]};
    }
    const uint32_t max_ops = __reduce_max_sync(FULL_MASK, nops);
    // direct path when, for every packet of the group, one element covers the whole frame (or nothing is written)
    {
        // cleared field by field, pad_ left out (it is only read when nops == 1): `OpDesc op0{}` makes ptxas spill more
        // in both kernel builds
        OpDesc op0;
        op0.n = 0; op0.shift_bitpos = 0; op0.kind = 0; op0.out_chan = 0; op0.slot = 0; op0.shift = 0; op0.mix_bits = 0; op0.mix_res = 0;
        if (nops == 1) op0 = desc->ops[0];
        const bool whole = cfg.num_channels <= 2u && (nops == 0 || (nops == 1 && op0.kind == cfg.num_channels && op0.out_chan == 0));
        uint32_t first_frame = 0;
        if (nops == 1 && op0.pad_ != 0) {  // emitted live: only frames the V warp did not reach are left (zeros)
            first_frame = desc->pad_;
            op0.n = 0;
        }
        if (__all_sync(FULL_MASK, !valid || first_frame >= cfg.frame_length)) return;  // nothing left to write
        if (__all_sync(FULL_MASK, whole)) {
            if (cfg.num_channels == 2u) {
                if (cfg.bps == 3) emit_direct<3, 2>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
                else if (cfg.bps == 2) emit_direct<2, 2>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
                else emit_direct<4, 2>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
            } else {
                if (cfg.bps == 3) emit_direct<3, 1>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
                else if (cfg.bps == 2) emit_direct<2, 1>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
                else emit_direct<4, 1>(x, cfg, group, smem, valid, pk, op0, n_final, first_frame);
            }
            return;
        }
    }
    // row path when every packet of the group is canonical: all elements as long as the packet, every channel covered
    // once, no pair spilling past the last channel; and the shapes allow whole 128-bit row stores
    {
        bool canon = true;
        uint32_t chans = 0;  // channels written so far
        for (uint32_t e = 0; e < nops; e++) {
            const OpDesc op = desc->ops[e];
            const uint32_t w = op.kind == 2 ? 2u : 1u;
            const uint32_t m = ((1u << w) - 1u) << op.out_chan;
            canon = canon && op.n == n_final && (uint32_t)op.out_chan + w <= cfg.num_channels && (chans & m) == 0u;
            chans |= m;
        }
        bool packed_ok = canon && chans == (1u << cfg.num_channels) - 1u && nops > 0 && n_final == cfg.frame_length;
        canon = !valid || nops == 0 || (canon && chans == (1u << cfg.num_channels) - 1u);
        const uint32_t FR = (fb & 1u) ? 16u : 8u;  // frames per row: FR * fb must be a multiple of 16
        const uint32_t need = NWARPS * 32u * 4u * ((((FR * fb) / 4u) | 1u) + (row_shift_words(FR) | 1u));
        const bool vec_ok = ((((uintptr_t)x.pcm_out) | x.out_stride) & 15u) == 0;
        // packed row path: 16-bit, or 24-bit with at most one shifted byte per element and every shift byte (plus the
        // words the aligned window loads touch) inside the packet
        {
            const bool depth_ok = (cfg.bps == 3 && cfg.bit_depth == 24) || (cfg.bps == 2 && cfg.bit_depth == 16);
            if (cfg.bps == 3)
                for (uint32_t e = 0; e < nops; e++) {
                    const OpDesc op = desc->ops[e];
                    const uint32_t w = op.kind == 2 ? 2u : 1u;
                    packed_ok = packed_ok && (op.shift == 0 || (op.shift == 1 && (op.shift_bitpos >> 3) >= 4u &&
                                                                (op.shift_bitpos >> 3) + op.n * w + 8u <= pk.size));
                }
            const uint32_t FRP = (cfg.num_channels & 1u) ? 16u : 8u;  // FRP * channels samples: a multiple of 16
            const uint32_t need_p = NWARPS * 32u * 4u * ((FRP * cfg.num_channels) | 1u);
            if (depth_ok && vec_ok && __all_sync(FULL_MASK, !valid || packed_ok) && cfg.frame_length % FRP == 0 && need_p <= smem_bytes) {
                if (cfg.bps == 3) {
                    if (FRP == 8u) emit_rows_packed<3, 8, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, max_ops);
                    else emit_rows_packed<3, 16, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, max_ops);
                } else {
                    if (FRP == 8u) emit_rows_packed<2, 8, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, max_ops);
                    else emit_rows_packed<2, 16, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, max_ops);
                }
                return;
            }
        }
        if (__all_sync(FULL_MASK, canon) && vec_ok && cfg.frame_length % FR == 0 && need <= smem_bytes) {
            if (FR == 8u) {
                if (cfg.bps == 3) emit_rows<3, 8, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, n_final, max_ops);
                else if (cfg.bps == 2) emit_rows<2, 8, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, n_final, max_ops);
                else emit_rows<4, 8, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, n_final, max_ops);
            } else {
                emit_rows<3, 16, NWARPS>(x, cfg, group, smem, valid, pk, desc, nops, n_final, max_ops);  // odd frame size: 24-bit only
            }
            return;
        }
    }
    uint8_t *row = reinterpret_cast<uint8_t *>(sw) + (size_t)lane * row_words * 4u;
    const int32_t *sbase = x.scratch + lane;
    const int bps = (int)cfg.bps;
    const bool depth20 = cfg.bit_depth == 20;
    const bool merges_shift = cfg.bit_depth == 24 || cfg.bit_depth == 32;  // 16/20-bit writers ignore the shift buffer
    const uint32_t ntiles = (cfg.frame_length + TL - 1u) / TL;

#pragma unroll 1
    for (uint32_t tile = warp; tile < ntiles; tile += NWARPS) {
        const int32_t s0 = (int32_t)(tile * TL);
        const int32_t lo_byte = s0 * (int32_t)fb, hi_byte = (s0 + (int32_t)TL) * (int32_t)fb;
        __syncwarp();  // previous tile flushed
        for (uint32_t i = lane; i < row_words * 32u; i += 32u) sw[i] = 0;  // fresh make(), decoder.go:120
        __syncwarp();
#pragma unroll 1
        for (uint32_t e = 0; e < max_ops; e++) {
            OpDesc op{};
            if (e < nops) op = desc->ops[e];
            const bool stereo = op.kind == 2;
            const uint32_t sb = (merges_shift ? (uint32_t)op.shift : 0u) * 8u;
            // a pair mapped onto the last channel spills R into the next frame (matrix.go:44-48)
            const bool spills = op.kind != 0 && (uint32_t)op.out_chan + (stereo ? 2u : 1u) > cfg.num_channels;
            int32_t i_lo = spills ? s0 - 1 : s0;
            i_lo = max(i_lo, 0);
            const int32_t i_hi = min(s0 + (int32_t)TL, (int32_t)min(op.n, 0x7fffffffu));
            // ---- stage the shift bytes of this lane's (op, tile) into its own shared row: 32-bit loads, 8 in flight ----
            const uint32_t width = stereo ? 2u : 1u;
            const uint32_t first_bit = op.shift_bitpos + (uint32_t)i_lo * width * sb;  // of frame i_lo
            const uint32_t nbits = (i_hi > i_lo && sb) ? (uint32_t)(i_hi - i_lo) * width * sb : 0u;
            uint32_t rel0 = 0;  // bit offset of frame i_lo's first field inside the staged row
            if (nbits) {
                const uint32_t byte0 = first_bit >> 3;
                const uint32_t nbytes = ((first_bit & 7u) + nbits + 7u) / 8u + 2u;  // +2: the 24-bit window of BitBuffer.Read
                const uintptr_t ga = ((uintptr_t)(pk.p + byte0)) & ~(uintptr_t)3;
                const uint32_t lead_bytes = (uint32_t)((uintptr_t)(pk.p + byte0) - ga);
                const int64_t rel_pk = (int64_t)byte0 - (int64_t)lead_bytes;  // packet byte index of staged byte 0
                const uint32_t nw = (lead_bytes + nbytes + 3u) / 4u;           // <= TL + 3
                uint32_t *myrow = shw + (size_t)lane * EMIT_SHIFT_ROW_WORDS;
                const uint32_t *gsrc = reinterpret_cast<const uint32_t *>(ga);
#pragma unroll 8
                for (uint32_t k = 0; k < nw; k++) myrow[k] = shift_word(pk, rel_pk, k, gsrc);
                myrow[nw] = 0;
                myrow[nw + 1u] = 0;
                rel0 = lead_bytes * 8u + (first_bit & 7u);
            }
            if (op.kind != 0) {
                const int32_t *su = sbase + (size_t)op.slot * cfg.frame_length * 32u;
                const int32_t *sv = stereo ? su + (size_t)cfg.frame_length * 32u : su;
                if (!spills) {  // every byte of these frames lies inside the tile: no clipping
                    EmitOp eo;
                    eo.su = su; eo.sv = sv; eo.i_lo = i_lo; eo.i_hi = i_hi; eo.s0 = s0; eo.mix_res = op.mix_res;
                    eo.mix_bits = op.mix_bits; eo.sb = sb; eo.rel0 = rel0; eo.width = width; eo.fb = fb;
                    eo.out_off = (uint32_t)op.out_chan * cfg.bps; eo.stereo = stereo; eo.depth20 = depth20;
                    const uint32_t *shrow_words = shw + (size_t)lane * EMIT_SHIFT_ROW_WORDS;
                    if (bps == 3) emit_frames<3>(eo, row, shrow_words);
                    else if (bps == 2) emit_frames<2>(eo, row, shrow_words);
                    else emit_frames<4>(eo, row, shrow_words);
                } else {  // a pair spilling over the frame end (non-canonical element order): clip byte by byte
                    const uint32_t *shrow_words = shw + (size_t)lane * EMIT_SHIFT_ROW_WORDS;
#pragma unroll 1
                    for (int32_t i = i_lo; i < i_hi; i++) {
                        int32_t left = su[(size_t)i * 32u], right = stereo ? sv[(size_t)i * 32u] : 0;
                        writer_frame(left, right, stereo, op.mix_res, op.mix_bits, depth20, sb, shrow_words,
                                     rel0 + (uint32_t)(i - i_lo) * width * sb);
                        const int32_t off = i * (int32_t)fb + (int32_t)op.out_chan * bps;
                        tile_put(row, lo_byte, hi_byte, off, left, bps);
                        if (stereo) tile_put(row, lo_byte, hi_byte, off + bps, right, bps);
                    }
                }
            }
            __syncwarp();
        }
        // flush: the warp walks the 32 packet rows; the whole tile is written so the packet's slot is fully defined
        const uint32_t tile_frames = min(TL, cfg.frame_length - (uint32_t)s0);
        const uint32_t limit = tile_frames * fb;  // a multiple of 4 except, for odd frame sizes, in the packet's last tile
        for (uint32_t r = 0; r < 32u; r++) {
            const uint32_t p = group * 32u + r;
            if (p >= x.npackets) break;
            const uint32_t r_nfinal = __shfl_sync(FULL_MASK, n_final, r);
            int64_t nvalid = (int64_t)r_nfinal * fb - lo_byte;
            nvalid = nvalid < 0 ? 0 : (nvalid > (int64_t)limit ? (int64_t)limit : nvalid);
            uint32_t *src = sw + (size_t)r * row_words;
            if ((uint32_t)nvalid < limit) {
                uint8_t *srcb = reinterpret_cast<uint8_t *>(src);
                for (uint32_t b2 = (uint32_t)nvalid + lane; b2 < limit; b2 += 32u) srcb[b2] = 0;
                __syncwarp();
            }
            uint8_t *dst = x.pcm_out + (size_t)p * x.out_stride + (size_t)lo_byte;
            const uint32_t nvec = limit >> 4;
            if ((((uintptr_t)dst) & 15u) == 0) {
                for (uint32_t v = lane; v < nvec; v += 32u) {
                    uint4 q = make_uint4(src[v * 4u], src[v * 4u + 1u], src[v * 4u + 2u], src[v * 4u + 3u]);
                    reinterpret_cast<uint4 *>(dst)[v] = q;
                }
            } else {
                for (uint32_t w = lane; w < nvec * 4u; w += 32u) reinterpret_cast<uint32_t *>(dst)[w] = src[w];
            }
            for (uint32_t w = nvec * 4u + lane; w < (limit >> 2); w += 32u) reinterpret_cast<uint32_t *>(dst)[w] = src[w];
            if (lane < (limit & 3u)) dst[(limit & ~3u) + lane] = reinterpret_cast<const uint8_t *>(src)[(limit & ~3u) + lane];
        }
    }
}

// decodePacketInto (decoder.go:133-207) for groups of 32 packets: persistent two-warp CTAs pull group after group from
// counters[0]; per group the two role warps run stages 1+2 (and stage 3 of live pairs), then both emit what is left.
// scratch / descs hold one slot per CTA (gridDim.x), not per group. counters = {next group, CTAs done}: both zero at
// launch, and the last CTA to leave zeroes them again for the next launch on the same stream.
__device__ __forceinline__ void decode_cta(
    const uint8_t *__restrict__ packed, const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ sizes,
    uint32_t npackets, const DevConfig &cfg, int32_t *__restrict__ scratch, PacketDesc *__restrict__ descs,
    uint8_t *__restrict__ pcm_out, uint64_t out_stride, uint32_t *__restrict__ out_bytes, int32_t *__restrict__ status,
    uint32_t *__restrict__ counters) {
    extern __shared__ __align__(1024) uint8_t dec_smem[];
    DecShared &sm = *reinterpret_cast<DecShared *>(dec_smem);
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t ngroups = (npackets + 31u) / 32u;
    uint32_t smid, hw_warp;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_warp));
    if (threadIdx.x == 0) {
        for (int s = 0; s < RING_SLOTS; s++) {
            mbar_init(&sm.full_bar[s], BAR_ARRIVALS);
            mbar_init(&sm.empty_bar[s], BAR_ARRIVALS);
        }
        sm.group = atomicAdd(&counters[0], 1u);
    }
    if (lane == 0) sm.warp_smsp[warp] = hw_warp & 3u;  // %warpid is a hint, but any assignment of roles is correct
    __syncthreads();
    if (threadIdx.x == 0) {
        // The entropy warp is the one that should not share a scheduler with other entropy warps (it has the least
        // instruction-level parallelism). Per SM, a packed word counts the resident entropy warps of every
        // sub-partition; the CTA gives the role to its warp on the less loaded one.
        unsigned int *word = &g_sm_entropy_load[smid & 255u];
        const uint32_t first = atomicAdd(&g_sm_ticket[smid & 255u], 1u) % DEC_WARPS;  // rotates the tie-break
        unsigned int seen = *reinterpret_cast<volatile unsigned int *>(word), assumed;
        uint32_t best;
        do {
            assumed = seen;
            best = first;
            for (uint32_t k = 1; k < DEC_WARPS; k++) {
                const uint32_t w = (first + k) % DEC_WARPS;
                if (((assumed >> (8 * sm.warp_smsp[w])) & 0xffu) < ((assumed >> (8 * sm.warp_smsp[best])) & 0xffu)) best = w;
            }
            seen = atomicCAS(word, assumed, assumed + (1u << (8 * sm.warp_smsp[best])));
        } while (seen != assumed);
        sm.entropy_smsp = sm.warp_smsp[best];
        for (uint32_t k = 0; k < DEC_WARPS; k++) sm.role_of_warp[(best + k) % DEC_WARPS] = k;
    }
    __syncthreads();
    const uint32_t role = sm.role_of_warp[warp];
#ifdef ALACB200_DEV
    if (g_role_cycles != nullptr && lane == 0) {  // developer aid: hardware warp slot of every warp of the CTA, by CTA warp index
        reinterpret_cast<volatile uint8_t *>(g_role_cycles + (size_t)blockIdx.x * 16 + 14)[warp] = (uint8_t)hw_warp;
        if (warp == 0) {
            reinterpret_cast<volatile uint8_t *>(g_role_cycles + (size_t)blockIdx.x * 16 + 14)[4] = (uint8_t)(sm.entropy_smsp & 3u);
            g_role_cycles[(size_t)blockIdx.x * 16 + 15] = clock64();
        }
    }
#endif
    // the CTA's own slot of parked samples and element lists
    // (rebuilt from the launch parameters at every use: a pointer kept across the role phases is a spilled pointer)
#define ALACB200_SCRATCH_CTA (scratch + (size_t)cta_now() * cfg.num_channels * cfg.frame_length * 32u)
#define ALACB200_DESCS_CTA (descs + (size_t)cta_now() * 32u)
    uint32_t seq = 0;  // ring sequence number of this warp's role
    uint32_t group = sm.group;
#pragma unroll 1
    while (group < ngroups) {
        if (role == 0) entropy_warp(sm, lane, packed, offsets, sizes, npackets, cfg, ALACB200_DESCS_CTA, out_bytes, status, group, seq, counters);
        else predictor_warp(sm, lane, packed, offsets, sizes, npackets, cfg, descs, pcm_out, out_stride, group, seq, scratch);
        __syncthreads();  // scratch + descriptors of this group are complete and visible to the CTA
        // stage 3 of whatever was not emitted live reuses the window / ring / job memory as its transpose tiles
        EmitArgs ea{packed, offsets, sizes, npackets, ALACB200_SCRATCH_CTA, ALACB200_DESCS_CTA, pcm_out, out_stride};
        RoleTimer rt(lane, 8 + (int)(warp % 3u));
        const unsigned long long t_emit = rt.now();
        emit_group<DEC_WARPS>(ea, cfg, group, dec_smem, (uint32_t)offsetof(DecShared, full_bar));
        rt.add(0, t_emit);
        rt.flush(1);
        group = sm.next_group;
        if (threadIdx.x == 0) sm.group = group;  // the predictor warp re-reads it where it needs the packet index
        __syncthreads();  // the tiles are free again; nobody reads next_group after this point
    }
    if (threadIdx.x == 0) {
        uint32_t smid_end;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid_end));  // a CTA never migrates: same value as at the start
        atomicSub(&g_sm_entropy_load[smid_end & 255u], 1u << (8 * sm.entropy_smsp));
        __threadfence();
        if (atomicAdd(&counters[1], 1u) == gridDim.x - 1u) {  // last CTA out: every fetch has been made
            counters[0] = 0;
            counters[1] = 0;
        }
    }
}

#define ALACB200_KERNEL_PARAMS                                                                                              \
    const uint8_t *__restrict__ packed, const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ sizes,          \
        uint32_t npackets, DevConfig cfg, int32_t *__restrict__ scratch, PacketDesc *__restrict__ descs,                   \
        uint8_t *__restrict__ pcm_out, uint64_t out_stride, uint32_t *__restrict__ out_bytes,                              \
        int32_t *__restrict__ status, uint32_t *__restrict__ counters
// The throughput build (big batches) ...
__global__ void __launch_bounds__(DEC_THREADS, CTAS_PER_SM) alac_decode_kernel(ALACB200_KERNEL_PARAMS) {
    decode_cta(packed, offsets, sizes, npackets, cfg, scratch, descs, pcm_out, out_stride, out_bytes, status, counters);
}
// ... and the register-rich build for batches of at most one wave of it.
__global__ void __launch_bounds__(DEC_THREADS, CTAS_PER_SM_LAT) alac_decode_kernel_lat(ALACB200_KERNEL_PARAMS) {
    decode_cta(packed, offsets, sizes, npackets, cfg, scratch, descs, pcm_out, out_stride, out_bytes, status, counters);
}

}  // namespace alacb200

// alac_planar.cuh -- channel-planar typed samples from the decode kernel's interleaved packet slots.
//
// A planar launch serves a run of tracks that share one kernel config (one track for alacb200_decode_planar_device, a run
// of adjacent tracks for alacb200_library_decode_planar_device). The rows of all tracks form one packet table, track
// after track; a device-resident PlanarTrack per track says where its rows, frame starts and output are. The decode
// kernel fills a stream-ordered intermediate of per-packet slots for the run's rows (stride frame_bytes rounded up to 16,
// so every slot is 16-byte aligned), then two passes of this file run:
//
//   alac_frame_scan_kernel  one CTA per track: frames[i] = out_bytes[i] / (channels * bps) (0 for a failed packet) and
//                           its exclusive prefix sum, the track's frame_start[0..n]. Off the hot path.
//   alac_planar_kernel      packet i of track t, frame f, channel c -> out_t[c * channel_stride_t + frame_start[i] + f]. A
//                           CTA takes one tile of frames of one packet and finds the packet's track by a binary search
//                           over the tracks' first rows: 128-bit loads stage the tile's interleaved bytes in shared
//                           memory, then each thread converts a run of frames of one channel row and stores it, 16-byte
//                           vector stores where the element address allows and scalar stores at the row's two ends.
//
// The conversions are defined on the container value, the sign-extended bps-byte little-endian sample (a 20-bit sample is
// the stored value, i.e. << 4): S16 (16-bit streams only) and S32 store it, F32 stores (float)value * 2^-(8*bps-1) with
// round-to-nearest-even int-to-float, so 16/20/24-bit values are exact and full scale maps to [-1, 1).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace alacb200 {

constexpr int SCAN_THREADS = 1024;
constexpr int PLANAR_THREADS = 256;
constexpr uint32_t PLANAR_TILE_BYTES = 16384;  // interleaved bytes a CTA stages: a power-of-two number of frames

// Frames per planar tile: the largest power of two whose interleaved bytes fit PLANAR_TILE_BYTES (512 for 8 x 32-bit,
// so at least 16 and every tile starts 16-byte aligned inside its slot), capped at the frame length.
inline uint32_t planar_tile_frames(uint32_t frame_bytes_per_frame, uint32_t frame_length) {
    uint32_t t = 16;
    while (2 * t * frame_bytes_per_frame <= PLANAR_TILE_BYTES && t < frame_length) t *= 2;
    return t;
}

// One track of a planar launch. Its rows are [row, row + n) of the shared packet table, its frame starts
// frame_start[fs .. fs + n] (n + 1 entries, [n] is its total), and channel c of its samples starts at
// out + c * channel_stride elements.
struct PlanarTrack {
    uint64_t row;
    uint64_t fs;
    void *out;
    uint64_t channel_stride;
    uint32_t n;
    int32_t fail;  // 0, or the status word of a track without a decoder: every row gets it and every frame start is 0
};

// One CTA per track (grid = the run's tracks): each thread owns a contiguous range of the track's packets, sums it, the
// CTA scans the per-thread sums, and each thread writes its range's prefixes. out_bytes holds the run's rows from
// row0 on; status is the whole table.
__global__ void __launch_bounds__(SCAN_THREADS) alac_frame_scan_kernel(const uint32_t *__restrict__ out_bytes,
                                                                     int32_t *__restrict__ status,
                                                                     const PlanarTrack *__restrict__ tracks, uint64_t row0,
                                                                     uint32_t bytes_per_frame,
                                                                     uint64_t *__restrict__ frame_start) {
    __shared__ uint64_t warp_sums[SCAN_THREADS / 32];
    const PlanarTrack tr = tracks[blockIdx.x];
    const uint32_t n = tr.n;
    if (tr.fail) {
        for (uint32_t i = threadIdx.x; i <= n; i += SCAN_THREADS) {
            if (i < n) status[tr.row + i] = tr.fail;
            frame_start[tr.fs + i] = 0;
        }
        return;
    }
    out_bytes += tr.row - row0;
    status += tr.row;
    frame_start += tr.fs;
    const uint32_t t = threadIdx.x, per = (n + SCAN_THREADS - 1) / SCAN_THREADS;
    const uint32_t lo = min(n, t * per), hi = min(n, lo + per);
    auto frames = [&](uint32_t i) -> uint64_t { return status[i] == 0 ? out_bytes[i] / bytes_per_frame : 0u; };
    uint64_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += frames(i);
    // inclusive scan of the per-thread sums: shuffles inside a warp, then over the warp totals
    const uint32_t lane = t & 31u, warp = t >> 5;
    uint64_t incl = sum;
    for (int d = 1; d < 32; d *= 2) {
        const uint64_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += v;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = warp_sums[lane];
        for (int d = 1; d < 32; d *= 2) {
            const uint64_t v = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= (uint32_t)d) w += v;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    uint64_t run = incl - sum + (warp ? warp_sums[warp - 1] : 0);
    for (uint32_t i = lo; i < hi; i++) {
        frame_start[i] = run;
        run += frames(i);
    }
    if (t == SCAN_THREADS - 1) frame_start[n] = run;
}

// int16_t / int32_t: the container value; float: the container value * scale.
template <typename T> __device__ __forceinline__ T planar_convert(int32_t v, float scale) {
    if constexpr (std::is_same<T, float>::value) return __fmul_rn(__int2float_rn(v), scale);
    else return (T)v;
}
// The bits of planar_convert's result, zero-extended to 32 (what one lane of a vector store carries).
template <typename T> __device__ __forceinline__ uint32_t planar_bits(int32_t v, float scale) {
    if constexpr (std::is_same<T, float>::value) return __float_as_uint(planar_convert<T>(v, scale));
    else return (uint32_t)(std::make_unsigned_t<T>)planar_convert<T>(v, scale);
}

// The container sample at byte `off` of the staged tile (words: the tile, 4 bytes of padding after it).
__device__ __forceinline__ int32_t planar_sample(const uint32_t *words, uint32_t off, uint32_t bps) {
    const uint32_t w = off >> 2;
    const uint32_t v = __funnelshift_r(words[w], words[w + 1], (off & 3u) * 8u);
    const uint32_t drop = 32u - 8u * bps;
    return (int32_t)(v << drop) >> drop;
}

// grid (the run's rows, tiles per packet), PLANAR_THREADS threads; slots: the decode kernel's output, the run's row
// row0 + i at slots + i * slot_stride (16-byte aligned); tracks: the run's ntracks tracks in row order; frame_start from
// alac_frame_scan_kernel.
template <typename T>
__global__ void __launch_bounds__(PLANAR_THREADS) alac_planar_kernel(const uint8_t *__restrict__ slots, uint64_t slot_stride,
                                                                   const uint64_t *__restrict__ frame_start,
                                                                   const PlanarTrack *__restrict__ tracks, uint32_t ntracks,
                                                                   uint64_t row0, uint32_t channels, uint32_t bps,
                                                                   uint32_t tile_frames) {
    constexpr uint32_t V = 16 / sizeof(T);  // elements per 16-byte store
    __shared__ uint4 tile[PLANAR_TILE_BYTES / 16 + 1];
    const uint32_t pkt = blockIdx.x;
    // the packet's track: the last one whose first row is at or before it (a track without rows shares its first row
    // with the next one, so it is never picked for a row)
    const uint64_t row = row0 + pkt;
    uint32_t lo = 0, hi = ntracks - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) / 2;
        if (tracks[mid].row <= row) lo = mid;
        else hi = mid - 1;
    }
    const PlanarTrack &tr = tracks[lo];
    const uint64_t k0 = tr.fs + (row - tr.row);
    T *const out = static_cast<T *>(tr.out);
    const uint64_t channel_stride = tr.channel_stride;
    const uint64_t fs = frame_start[k0];
    const uint32_t frames = (uint32_t)(frame_start[k0 + 1] - fs);
    const uint32_t f0 = blockIdx.y * tile_frames;
    if (f0 >= frames) return;  // a failed or short packet: nothing in this tile
    const uint32_t cnt = min(tile_frames, frames - f0);
    const uint32_t bpf = channels * bps;

    // stage: tile_frames is a multiple of 16, so the tile starts 16-byte aligned inside its 16-byte aligned slot, and
    // rounding its length up to 16 stays inside the slot (slot_stride >= frame_bytes rounded up to 16)
    const uint4 *src = reinterpret_cast<const uint4 *>(slots + pkt * slot_stride + (uint64_t)f0 * bpf);
    const uint32_t nvec = (cnt * bpf + 15u) / 16u;
#pragma unroll
    for (uint32_t r = 0; r < PLANAR_TILE_BYTES / 16 / PLANAR_THREADS; r++) {
        const uint32_t k = threadIdx.x + r * PLANAR_THREADS;
        if (k < nvec) tile[k] = __ldcs(src + k);
    }
    __syncthreads();
    const uint32_t *words = reinterpret_cast<const uint32_t *>(tile);

    // Row c of the tile is cnt elements from out + c * channel_stride + fs + f0. Work item (c, k) is the k-th 16-byte
    // block the row touches: a whole block is one vector store, the partial blocks at the row's ends are scalar stores.
    const float scale = __int_as_float((127 - (int)(8 * bps - 1)) << 23);  // 2^-(8*bps-1)
    const uint32_t blocks = cnt / V + 2;
    for (uint32_t item = threadIdx.x; item < channels * blocks; item += PLANAR_THREADS) {
        const uint32_t c = item / blocks, k = item - c * blocks;
        T *row = out + c * channel_stride + fs + f0;
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(row) / sizeof(T)) & (V - 1);
        const int32_t first = (int32_t)(k * V) - (int32_t)mis;  // row-local frame of the block's first element
        const int32_t a = max(first, 0), b = min(first + (int32_t)V, (int32_t)cnt);
        if (a >= b) continue;
        if (b - a == (int32_t)V) {
            const uint32_t off = (a * channels + c) * bps, step = channels * bps;
            uint32_t w[4];
#pragma unroll
            for (uint32_t j = 0; j < 4; j++) {
                if constexpr (sizeof(T) == 4) {
                    w[j] = planar_bits<T>(planar_sample(words, off + j * step, bps), scale);
                } else {
                    w[j] = planar_bits<T>(planar_sample(words, off + 2 * j * step, bps), scale) |
                           planar_bits<T>(planar_sample(words, off + (2 * j + 1) * step, bps), scale) << 16;
                }
            }
            *reinterpret_cast<uint4 *>(row + a) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {
            for (int32_t f = a; f < b; f++) row[f] = planar_convert<T>(planar_sample(words, (f * channels + c) * bps, bps), scale);
        }
    }
}

}  // namespace alacb200

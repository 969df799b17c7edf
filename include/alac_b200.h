/*
 * alac_b200.h -- C ABI of the B200-native ALAC packet decoder (libalacb200.so).
 *
 * This is the drop-in boundary for saprobe-alac's packet-decode path. The reference has no FFI
 * of its own (pure Go); these entry points are exactly what a cgo shim behind its exported Go API
 * binds (see INTEGRATION.md). Each declaration cites the reference interface it replaces
 * (paths under /root/reference).
 *
 * Plain pointers and sizes only; no exceptions or panics cross this boundary. Functions return an
 * API result (ALACB200_OK or a negative ALACB200_E_*); per-packet outcomes are STATUS WORDS written
 * to the `status` arrays.
 *
 * There is NO CPU fallback: every decode call runs the CUDA kernels in csrc/alac_kernels.cuh and
 * fails with ALACB200_E_CUDA / ALACB200_E_NO_DEVICE when no device is usable.
 */
#ifndef ALAC_B200_H
#define ALAC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- API results ------------------------------------------------------------------------------ */
enum {
    ALACB200_OK = 0,
    ALACB200_E_ARG = -1,       /* NULL pointer, bad stride/alignment, n too large */
    ALACB200_E_CUDA = -2,      /* a CUDA runtime call failed; see alacb200_last_error() */
    ALACB200_E_NO_DEVICE = -3, /* no CUDA device / bad device index */
    ALACB200_E_NOMEM = -4,
    ALACB200_E_CONFIG = -5,    /* config rejected; the status word is returned via *status_out */
    ALACB200_E_IO = -6,        /* container reader: short read / seek failure */
    ALACB200_E_NO_TRACK = -7   /* container reader: no ALAC track (ErrNoTrack, errors.go:28) */
};

/* ---- per-packet status word --------------------------------------------------------------------
 * low byte  = sentinel, 1:1 with internal/alac/errors.go:24-33 (so Go can rebuild the %w chain)
 * bits 8-11 = element context of decoder.go's wrapping ("SCE/LFE:" :156, "CPE:" :172, "DSE:" :184,
 *             "FIL:" :189)
 * bits 12-13 = entropy context ("entropy decode:" :303, "entropy decode U:" :463, "... V:" :478) */
enum {
    ALACB200_ST_OK = 0,
    ALACB200_ST_INVALID_COOKIE = 1,      /* ErrInvalidCookie      errors.go:25 -> wrapped in ErrConfig */
    ALACB200_ST_UNSUPPORTED_VERSION = 2, /* ErrUnsupportedVersion errors.go:26 -> ErrConfig */
    ALACB200_ST_UNSUPPORTED_ELEMENT = 3, /* ErrUnsupportedElement errors.go:27 -> ErrDecode */
    ALACB200_ST_INVALID_HEADER = 4,      /* ErrInvalidHeader      errors.go:28 -> ErrDecode */
    ALACB200_ST_INVALID_SHIFT = 5,       /* ErrInvalidShift       errors.go:29 -> ErrDecode */
    ALACB200_ST_BITSTREAM_OVERRUN = 6,   /* ErrBitstreamOverrun   errors.go:30 -> ErrDecode */
    ALACB200_ST_SAMPLE_OVERRUN = 7,      /* ErrSampleOverrun      errors.go:31 -> ErrDecode */
    ALACB200_ST_BIT_DEPTH = 8,           /* ErrBitDepth           errors.go:32 -> ErrConfig */
    /* Deviations (documented in DESIGN.md): */
    ALACB200_ST_REF_PANIC = 9,           /* the Go reference would PANIC on this packet (slice/index out of
                                            range, SURVEY.md appendix B7); reported as a decode error */
    ALACB200_ST_UNSUPPORTED_CONFIG = 10, /* channels not in 1..8 or frame length not in 1..65536 */
    /* Not a decode error: the packet's (offset, size) lies outside the bytes handed over, so nothing was read or
     * decoded. The reference fails at this point in its READER (io.ReadFull -> "reading sample N: unexpected EOF",
     * decode.go:172-174), before the packet decoder is involved; the host wrappers raise that error. */
    ALACB200_ST_IO_TRUNCATED = 11
};
enum { ALACB200_CTX_NONE = 0, ALACB200_CTX_SCE = 1, ALACB200_CTX_CPE = 2, ALACB200_CTX_DSE = 3, ALACB200_CTX_FIL = 4 };
enum { ALACB200_ENT_NONE = 0, ALACB200_ENT_MONO = 1, ALACB200_ENT_U = 2, ALACB200_ENT_V = 3 };
#define ALACB200_ST_CODE(s) ((s) & 0xff)
#define ALACB200_ST_CTX(s) (((s) >> 8) & 0xf)
#define ALACB200_ST_ENT(s) (((s) >> 12) & 0x3)

/* PacketConfig, config.go:27-38 (field for field). */
typedef struct alacb200_config {
    uint32_t frame_length;
    uint8_t bit_depth;
    uint8_t num_channels;
    uint8_t pb;
    uint8_t mb;
    uint8_t kb;
    uint8_t reserved;
    uint16_t max_run;
    uint32_t max_frame_bytes;
    uint32_t avg_bit_rate;
    uint32_t sample_rate;
} alacb200_config;

/* PCMFormat, format.go:20-24. */
typedef struct alacb200_pcm_format {
    int32_t sample_rate;
    int32_t bit_depth;
    int32_t channels;
} alacb200_pcm_format;

typedef struct alacb200_decoder alacb200_decoder; /* PacketDecoder, decoder.go:79-87 */

/* ParseMagicCookie, config.go:47-81. Returns a status word (OK / INVALID_COOKIE / UNSUPPORTED_VERSION). */
int32_t alacb200_parse_cookie(const uint8_t *cookie, size_t len, alacb200_config *out);

/* BytesPerSample, internal/alac/format.go:23-34; 0 for an unsupported depth (the reference panics). */
int32_t alacb200_bytes_per_sample(uint8_t bit_depth);

/* NewPacketDecoder, decoder.go:90-110, bound to CUDA device `device`. On ALACB200_E_CONFIG
 * *status_out (may be NULL) holds BIT_DEPTH or UNSUPPORTED_CONFIG. */
int32_t alacb200_create(const alacb200_config *cfg, int device, alacb200_decoder **out, int32_t *status_out);
void alacb200_destroy(alacb200_decoder *dec);

/* PacketDecoder.Format, decoder.go:112-114. */
int32_t alacb200_format(const alacb200_decoder *dec, alacb200_pcm_format *out);
int32_t alacb200_get_config(const alacb200_decoder *dec, alacb200_config *out);
/* frame_length * num_channels * bytes_per_sample: the size of DecodePacket's output buffer, decoder.go:118-120 */
uint64_t alacb200_max_packet_pcm_bytes(const alacb200_decoder *dec);

/* DecodePackets (new, north star) == n x PacketDecoder.DecodePacket, decoder.go:117-128, on HOST buffers.
 *   packed            the bytes the packets live in: a packed buffer, or a whole M4A file image with the
 *                     sample table (internal/mp4 SampleInfo, mp4.go:28-31) as offsets/sizes -- no re-packing
 *   packed_bytes      bytes readable at `packed`; a packet with offsets[i]+sizes[i] > packed_bytes is not
 *                     read and gets ALACB200_ST_IO_TRUNCATED
 *   packet i          packed[offsets[i] .. offsets[i]+sizes[i]), any alignment, any order
 *   pcm_out           packet i's PCM goes to pcm_out + i*out_stride; out_stride >= max_packet_pcm_bytes
 *                     and a multiple of 4
 *   out_bytes[i]      numSamples*numChannels*bps on success (partial last packet => shorter), else 0
 *   status[i]         status word
 * Host buffers may be pageable or pinned (alacb200_pinned_alloc / alacb200_arena); pinned buffers are
 * copied asynchronously and overlap with the kernels. Inputs are borrowed for the call only
 * (bits.Reset copies, bitbuffer.go:44). One call at a time per decoder; several decoders per
 * device are fine. */
int32_t alacb200_decode_packets(alacb200_decoder *dec, const uint8_t *packed, uint64_t packed_bytes,
                                const uint64_t *offsets, const uint32_t *sizes, uint32_t n, uint8_t *pcm_out,
                                uint64_t out_stride, uint32_t *out_bytes, int32_t *status);

/* Decoder-owned pinned staging for the host wrappers (the Go shim's DecodePackets packs [][]byte into *in and
 * reads the PCM from *out): grow-only, valid until the next alacb200_arena call or alacb200_destroy, so a
 * steady stream of DecodePacket / DecodePackets calls allocates nothing (decoder.go:79-87 keeps its scratch
 * the same way). */
int32_t alacb200_arena(alacb200_decoder *dec, uint64_t in_bytes, uint64_t out_bytes, uint8_t **in, uint8_t **out);

/* Same on DEVICE buffers (everything already resident in HBM), enqueued on `stream` (a cudaStream_t,
 * NULL = default stream) as ONE kernel launch without synchronising (the scratch is stream-ordered
 * memory sized by the resident CTAs, not by n). d_packed must be 16-byte aligned and readable for
 * packed_bytes rounded up to 16. The decoder's scratch is shared, so calls on one decoder must be
 * stream-ordered; passing a different stream than the previous call first waits for that one. */
int32_t alacb200_decode_packets_device(alacb200_decoder *dec, const uint8_t *d_packed, uint64_t packed_bytes,
                                       const uint64_t *d_offsets, const uint32_t *d_sizes, uint32_t n,
                                       uint8_t *d_pcm_out, uint64_t out_stride, uint32_t *d_out_bytes,
                                       int32_t *d_status, void *stream);

/* Channel-planar typed samples on DEVICE buffers (alacb200_decode_planar_device). Every type is defined on the container
 * value, the sign-extended bps-byte little-endian sample of the interleaved PCM (a 20-bit sample is the stored value,
 * i.e. << 4):
 *   S16  int16, the container value; 16-bit streams only
 *   S32  int32, the container value
 *   F32  float, value * 2^-(8*bps-1), int-to-float rounded to nearest even: 16/20/24-bit values are exact and full
 *        scale maps to [-1, 1) */
enum { ALACB200_SAMPLES_S16 = 1, ALACB200_SAMPLES_S32 = 2, ALACB200_SAMPLES_F32 = 3 };

/* DecodePackets on DEVICE buffers into channel-planar samples. Packet i's frames land in
 * d_out[c*channel_stride + frame_start[i] .. frame_start[i+1]) of every channel c. A failed packet
 * contributes no frames. d_frame_start has n+1 entries, and [n] is the total. channel_stride
 * >= n*frame_length (elements). Frames between the total and channel_stride are not written.
 * Same contract as alacb200_decode_packets_device for d_packed (16-byte aligned, readable for packed_bytes rounded
 * up to 16, packets inside it), the stream and the decoder's scratch; d_status[n] gets the status words; d_out must
 * be aligned to its element size. Enqueued on `stream` without synchronising: the decode kernel into an interleaved
 * intermediate, the frame scan, the planar pass. The intermediate (n slots of max_packet_pcm_bytes rounded up to 16,
 * plus n*4 bytes) comes from the device's stream-ordered pool and is freed on `stream` at the end of the call: it is at
 * most the size of the output, and the decoder keeps no memory that grows with n between calls. n == 0 writes
 * d_frame_start[0] = 0. ALACB200_E_ARG for an unknown sample_type, S16 on a stream that is not 16-bit, a NULL pointer
 * (only d_frame_start when n == 0), channel_stride < n*frame_length, or a misaligned d_out or d_packed. */
int32_t alacb200_decode_planar_device(alacb200_decoder *dec, const uint8_t *d_packed, uint64_t packed_bytes,
                                      const uint64_t *d_offsets, const uint32_t *d_sizes, uint32_t n,
                                      int32_t sample_type, void *d_out, uint64_t channel_stride,
                                      uint64_t *d_frame_start, int32_t *d_status, void *stream);

/* ---- several tracks, several devices (BASELINE configs[4]: a library of mixed 16/24-bit tracks) -----------
 * A PacketDecoder holds ONE cookie (decoder.go:79-87); a library batch mixes cookies. A library handle owns one
 * pipeline per device and decodes any mix of tracks in one call: every track is checked like
 * ParseMagicCookie + NewPacketDecoder, tracks are split into contiguous ranges balanced by compressed bytes
 * over the devices (one submitting host thread per device, no collective), grouped by config inside a device
 * so every kernel launch is depth-homogeneous, and cut into pipeline chunks that may span tracks. The bytes
 * of a track are read in place (`data` = packed packets or the M4A file image, offsets/sizes = its sample
 * table); pin them (alacb200_pinned_alloc) for asynchronous copies. */
typedef struct alacb200_track_desc {
    /* in */
    const uint8_t *cookie;   /* magic cookie of the track (with or without the frma/alac wrappers) */
    size_t cookie_len;
    const uint8_t *data;     /* bytes the packets live in */
    uint64_t data_len;
    const uint64_t *offsets; /* sample table, n entries */
    const uint32_t *sizes;
    uint32_t n;
    uint32_t reserved;
    uint8_t *pcm_out;        /* packet i -> pcm_out + i*out_stride */
    uint64_t out_stride;     /* >= frame_length*channels*bps of THIS track, multiple of 4 */
    uint32_t *out_bytes;     /* n entries */
    int32_t *status;         /* n entries */
    /* out */
    alacb200_config config;  /* the parsed cookie */
    int32_t track_status;    /* ALACB200_ST_OK, or why the track has no decoder (INVALID_COOKIE ... BIT_DEPTH) */
    int32_t result;          /* ALACB200_OK, ALACB200_E_CONFIG (see track_status), ALACB200_E_ARG, or a device error */
    int32_t device;          /* CUDA device the track was decoded on (-1: not decoded) */
    int32_t reserved2;
} alacb200_track_desc;
typedef struct alacb200_library alacb200_library;
int32_t alacb200_library_create(const int *devices, int ndevices, alacb200_library **out);
void alacb200_library_destroy(alacb200_library *lib);
int32_t alacb200_library_devices(const alacb200_library *lib);
/* Returns ALACB200_OK when every decodable track was decoded (per-track outcomes are in the descriptors), or
 * the first device error. One call at a time per library. */
int32_t alacb200_library_decode_tracks(alacb200_library *lib, alacb200_track_desc *tracks, uint32_t ntracks);

/* Many tracks of any mix of cookies on DEVICE buffers into channel-planar samples, on one device of the library
 * (alacb200_library_decode_planar_device): the multi-track form of alacb200_decode_planar_device. */
typedef struct alacb200_planar_track {
    /* in */
    const uint8_t *cookie;   /* magic cookie of the track (with or without the frma/alac wrappers) */
    size_t cookie_len;
    uint32_t n;              /* this track's rows of the shared packet table: rows follow track order, track 0 first */
    uint32_t reserved;
    void *d_out;             /* num_channels rows of channel_stride elements of the sample type */
    uint64_t channel_stride; /* >= n*frame_length of THIS track (elements) */
    /* out */
    alacb200_config config;  /* the parsed cookie */
    int32_t track_status;    /* ALACB200_ST_OK, or why the track has no decoder (INVALID_COOKIE ... UNSUPPORTED_CONFIG) */
    int32_t result;          /* ALACB200_OK or ALACB200_E_CONFIG (see track_status) */
} alacb200_planar_track;
/* The packet table (d_offsets, d_sizes, d_status) has N = sum of n rows, track after track; offsets are absolute in
 * d_packed, which follows the rules of alacb200_decode_packets_device (16-byte aligned, readable for packed_bytes rounded
 * up to 16). Track t's rows are [r_t, r_t + n_t) with r_t the sum of the earlier n; packet r_t + i lands in
 * d_out_t[c*channel_stride_t + fs[i] .. fs[i+1]) of every channel c, where fs = d_frame_start + r_t + t holds the
 * track's n_t + 1 frame starts ([n_t] is its total). d_frame_start therefore has N + ntracks entries. A failed packet
 * contributes no frames; frames between a track's total and its channel_stride are not written.
 *
 * A track whose cookie fails ParseMagicCookie + NewPacketDecoder's checks gets result ALACB200_E_CONFIG: its rows get
 * track_status as their status word, its frame starts are 0 and nothing is written to its d_out. The other tracks are
 * cut into maximal runs of adjacent tracks of one kernel config (frame length, depth, channels, pb/mb/kb), and every
 * run is one decode launch, one frame scan and one planar pass; a table ordered by config is one decode launch per
 * config. Enqueued on `stream` without synchronising the host (except the stream switch of the device scratch, as
 * for alacb200_decode_packets_device). A run's interleaved intermediate (its rows of max_packet_pcm_bytes rounded up to
 * 16, plus 4 bytes a row) comes from the device's stream-ordered pool and is freed on the stream after the run, so the
 * peak is the largest run's. The track table goes through pinned staging that is not written again before its copy
 * has completed.
 *
 * ntracks == 0 or N == 0 writes only the frame starts, all 0. ALACB200_E_ARG, with nothing enqueued, for an unknown
 * sample_type, S16 with a decodable track that is not 16-bit, a decodable track with n > 0 whose channel_stride is
 * below n*frame_length or whose d_out is NULL or not aligned to its element size, a misaligned d_packed, a NULL
 * pointer (d_packed, d_offsets, d_sizes and d_status may be NULL when N == 0), more than 2^32-1 rows, or a device that
 * is not one of the library's. One call at a time per library. */
int32_t alacb200_library_decode_planar_device(alacb200_library *lib, int device, const uint8_t *d_packed,
                                              uint64_t packed_bytes, const uint64_t *d_offsets,
                                              const uint32_t *d_sizes, alacb200_planar_track *tracks,
                                              uint32_t ntracks, int32_t sample_type, uint64_t *d_frame_start,
                                              int32_t *d_status, void *stream);

/* Pinned (page-locked) host memory for packed input / PCM output. */
void *alacb200_pinned_alloc(size_t bytes);
void alacb200_pinned_free(void *p);

/* Sentinel text of a status word, identical to the Go error strings (errors.go:24-33). */
const char *alacb200_strerror(int32_t status);
/* Full message the Go shim rebuilds for a status word, e.g.
 * "decode failed: CPE: entropy decode U: alac: bitstream overrun". Writes at most cap bytes. */
size_t alacb200_format_error(int32_t status, char *buf, size_t cap);
/* Text of the last failing CUDA call on this thread. */
const char *alacb200_last_error(void);
int32_t alacb200_device_count(void);

/* Per-kernel device timing (CUDA events on the launch stream), for bench.py's roofline line. */
typedef struct alacb200_profile {
    uint64_t launches_decode;   /* alac_decode_kernel launches since enable (stages 1-3 are one kernel) */
    double ms_decode;           /* summed event time of alac_decode_kernel */
} alacb200_profile;
int32_t alacb200_set_profiling(alacb200_decoder *dec, int enable); /* enabling resets the counters */
int32_t alacb200_get_profile(alacb200_decoder *dec, alacb200_profile *out); /* synchronises the recorded events */

/* ---- container side: internal/mp4 (SURVEY.md section 8f-1) --------------------------------------
 * FindALACTrack, internal/mp4/mp4.go:233-300 over an in-memory M4A/MP4 image. Returns the raw
 * cookie (stsd payload after the sample entry) and the sample table (stco|co64 x stsc x stsz). */
typedef struct alacb200_sample_info { /* SampleInfo, mp4.go:28-31 */
    uint64_t offset;
    uint32_t size;
    uint32_t reserved;
} alacb200_sample_info;
typedef struct alacb200_track alacb200_track;
/* Returns ALACB200_OK or ALACB200_E_NO_TRACK. *out always receives a track object (free it with
 * alacb200_mp4_free_track); on failure alacb200_mp4_error(*out) is the reference's error text. */
int32_t alacb200_mp4_find_alac_track(const uint8_t *file, uint64_t file_len, alacb200_track **out);
void alacb200_mp4_free_track(alacb200_track *t);
const uint8_t *alacb200_mp4_cookie(const alacb200_track *t, size_t *len);
const alacb200_sample_info *alacb200_mp4_samples(const alacb200_track *t, uint64_t *count);
const char *alacb200_mp4_error(const alacb200_track *t);

#ifdef __cplusplus
}
#endif
#endif
